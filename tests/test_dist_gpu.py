"""GPU tests of the landmark-sharded window (SURVEY.md 8e / BASELINE config C5 shape).
Single GPU: several shards on one device, partial reduced systems summed in place -- exercises
exactly the arithmetic the NCCL path uses.  Two GPUs (skipped otherwise): real torch.distributed
NCCL all-reduce, one process per GPU."""
import os

import numpy as np
import pytest

from scavislam_b200 import dist as sdist
from scavislam_b200 import synth

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


@pytest.mark.parametrize("nshards", [2, 3])
def test_sharded_window_equals_whole_window(svs, oracle, nshards):
    pb = synth.make_config("C1")
    whole = svs.BundleAdjuster()
    whole.set_problem(pb)
    it_w, st_w = whole.optimize(4)
    handles = [svs.BundleAdjuster() for _ in range(nshards)]
    sw = sdist.ShardedWindow(handles, pb)
    it_s, st_s = sw.optimize(4)
    assert it_s == it_w == 4
    assert st_s["trials_iter"] == st_w["trials_iter"]
    np.testing.assert_allclose(st_s["chi2_iter"], st_w["chi2_iter"], rtol=1e-9)
    assert _rel(sw.poses(), whole.poses()) < 1e-9
    psi = np.zeros((pb.L, 3))
    for idx, p in sw.points_local():
        psi[idx] = p
    assert _rel(psi, whole.points()) < 1e-9
    p_o, s_o, _ = oracle.optimize(pb, 4)
    assert _rel(sw.poses(), p_o) < 1e-6 and _rel(psi, s_o) < 1e-6
    for h in handles + [whole]:
        h.close()


def test_sharded_window_with_track_dropouts(svs, oracle):
    """Shards with a prescribed block pattern (svs_ba_set_structure) must not pad their tracks (a shard's padding would
    add pose pairs the other shards' layouts lack); the whole-window handle does pad -- both give the oracle's result."""
    pb = synth.with_dropouts(synth.make_window(40, 3000, seed=78), 0.2, seed=2)
    whole = svs.BundleAdjuster()
    whole.set_problem(pb)
    it_w, st_w = whole.optimize(4)
    handles = [svs.BundleAdjuster() for _ in range(3)]
    sw = sdist.ShardedWindow(handles, pb)
    it_s, st_s = sw.optimize(4)
    assert it_s == it_w == 4 and st_s["trials_iter"] == st_w["trials_iter"]
    np.testing.assert_allclose(st_s["chi2_iter"], st_w["chi2_iter"], rtol=1e-9)
    assert _rel(sw.poses(), whole.poses()) < 1e-9
    p_o, s_o, _ = oracle.optimize(pb, 4)
    assert _rel(sw.poses(), p_o) < 1e-6 and _rel(whole.poses(), p_o) < 1e-6
    for h in handles + [whole]:
        h.close()


def _nccl_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from scavislam_b200 import capi
    pb = synth.make_window(40, 3000, seed=77)
    ba = capi.BundleAdjuster(device=rank)
    sw = sdist.ShardedWindow([ba], pb, rank=rank, world=world, dist=dist, device=rank)
    it, st = sw.optimize(5)
    q.put((rank, it, st["chi2_iter"], sw.poses(), sw.points_local()[0]))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_nccl_sharded_window(svs, oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 1000
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    pb = synth.make_window(40, 3000, seed=77)
    p_o, s_o, st_o = oracle.optimize(pb, 5)
    psi = np.zeros((pb.L, 3))
    for rank, it, chi, poses, (idx, p) in res:
        assert it == st_o["iterations"]
        np.testing.assert_allclose(chi, st_o["chi2_iter"], rtol=1e-7)
        assert _rel(poses, p_o) < 1e-6
        psi[idx] = p
    assert _rel(psi, s_o) < 1e-6


def test_in_library_nccl_window(svs, oracle):
    """The sharded window driven inside the library (C ABI: svs_ba_comm_init / svs_ba_set_problem_sharded /
    svs_ba_optimize with one ncclAllReduce of S|bp|bc per trial), one process per visible GPU (two when the
    box has them, else a one-rank communicator: same code path, collectives degenerate)."""
    import subprocess
    import sys
    import torch
    n = min(2, torch.cuda.device_count())
    port = 29700 + os.getpid() % 1000
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(os.path.dirname(os.path.abspath(__file__)), "nccl_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "NCCL_WORKER_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
