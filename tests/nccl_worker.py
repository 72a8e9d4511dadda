"""Worker of tests/test_dist_gpu.py::test_in_library_nccl_window (launched with torch.distributed.run,
one process per GPU): the landmark-sharded window driven INSIDE the library -- svs_ba_comm_init,
svs_ba_set_problem_sharded, svs_ba_optimize with its per-trial ncclAllReduce -- against the CPU oracle
on the whole window.  The same handle also re-sends a window with the same structure and new numbers, and runs the
one-call API (a whole window, no collectives) before and after the sharded loads.  Prints 'NCCL_WORKER_OK' on success."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from scavislam_b200 import capi, synth
    from oracle import pyoracle as po
    ids = [capi.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    pb = synth.make_window(40, 3000, seed=77)
    ba = capi.BundleAdjuster(device=local)
    ba.comm_init(world, rank, ids[0])
    rel = lambda a, b: np.abs(a - b).max() / np.abs(b).max()

    def one_call(window):
        """The one-call API on a handle that has a communicator: a whole window, solved by this rank alone."""
        it1, T1, psi1, st1 = ba.optimise_inner_and_outer_window(window, 2)
        T1_o, psi1_o, st1_o = po.optimize(window, 2)
        assert it1 == st1_o["iterations"] and st1["trials_iter"] == st1_o["trials_iter"]
        np.testing.assert_allclose(st1["chi2_iter"], st1_o["chi2_iter"], rtol=1e-7)
        assert rel(T1, T1_o) < 1e-6 and rel(psi1, psi1_o) < 1e-6

    # before the first points_all() (which sizes its own device buffer) and again at the end
    one_call(pb)
    ba.set_problem_sharded(pb)
    it, st = ba.optimize(5)
    poses, psi = ba.poses(), ba.points_all()
    p_o, s_o, st_o = po.optimize(pb, 5)
    assert it == st_o["iterations"], (it, st_o["iterations"])
    assert st["trials_iter"] == st_o["trials_iter"]
    np.testing.assert_allclose(st["chi2_iter"], st_o["chi2_iter"], rtol=1e-7)
    assert rel(poses, p_o) < 1e-6, rel(poses, p_o)
    assert rel(psi, s_o) < 1e-6, rel(psi, s_o)
    # a second call on the same communicator: the one-call path of a back-end tick
    ba.set_problem_sharded(pb)
    it2, st2 = ba.optimize(2)
    assert it2 == 2 and st2["trials_iter"] == st_o["trials_iter"][:2]
    # the same structure with other landmarks and observations: only the numbers are sent again
    pbn = pb.copy()
    rng = np.random.default_rng(3)
    pbn.psi = pb.psi * (1 + rng.normal(0, 0.02, pb.psi.shape))
    pbn.e_obs = pb.e_obs + rng.normal(0, 0.4, pb.e_obs.shape)
    ba.set_problem_sharded(pbn)
    itn, stn = ba.optimize(4)
    p_n, s_n, st_n = po.optimize(pbn, 4)
    assert abs(st_n["chi2_final"] - st_o["chi2_iter"][3]) > 1e-5 * st_n["chi2_final"]   # stale numbers would not pass
    assert itn == st_n["iterations"] and stn["trials_iter"] == st_n["trials_iter"]
    np.testing.assert_allclose(stn["chi2_iter"], st_n["chi2_iter"], rtol=1e-7)
    assert rel(ba.poses(), p_n) < 1e-6 and rel(ba.points_all(), s_n) < 1e-6
    # tracks with visibility drop-outs: every rank completes ITS tracks with zero-weight edges, so the block pattern all
    # ranks agree on must contain the pose pairs of every rank's padding (svs_ba_set_problem_sharded derives it from the
    # whole window with the same rule) -- a mismatch would sum different blocks in the all-reduce
    pbd = synth.with_dropouts(pb, 0.2, seed=5)
    ba.set_problem_sharded(pbd)
    itd, std = ba.optimize(4)
    p_d, s_d, st_d = po.optimize(pbd, 4)
    assert itd == st_d["iterations"] and std["trials_iter"] == st_d["trials_iter"]
    np.testing.assert_allclose(std["chi2_iter"], st_d["chi2_iter"], rtol=1e-7)
    assert rel(ba.poses(), p_d) < 1e-6 and rel(ba.points_all(), s_d) < 1e-6
    one_call(pbn)
    ba.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print(f"NCCL_WORKER_OK world={world} pose_rel={rel(poses, p_o):.2e} psi_rel={rel(psi, s_o):.2e}")


if __name__ == "__main__":
    main()
