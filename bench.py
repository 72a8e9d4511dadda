#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native ScaViSLAM BA hot path.

Metric (BASELINE.json): Gauss-Newton/LM iterations per second on the 200-keyframe /
20k-landmark synthetic double window (config C2), 10 iterations per step.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one svs_ba_optimize(num_iters=10) over the whole window, starting from the same
initial state (svs_ba_reset_state, device-to-device).  `value` counts iterations with the
problem already resident in HBM; `e2e` goes through svs_optimiseInnerAndOuterWindow with HOST
buffers (H2D of the problem, symbolic analysis, all iterations, D2H of poses and points inside
the timed region).  N > 1 (torchrun): every rank owns an independent window (config C4,
replicas, no data-path collective), value = total iterations / max-over-ranks time.

--impl reference times the CPU oracle (oracle/ba_oracle.c, the restatement of the reference's
g2o path; the reference itself cannot be built here, see DESIGN.md) on the host cores.

--dump-outputs DIR writes what the last timed step of rank 0 returned, after the timed region, as
float64 arrays: DIR/poses.npy (P x 7, [q|t]), DIR/psi.npy (L x 3, inverse depth) and DIR/chi2_iter.npy
(chi2 after every LM iteration).  The inputs are seeded, so two builds can be compared output for output;
both arms write the same names.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NUM_ITERS = 10
WORKLOAD = "C2: 200-keyframe / 20k-landmark synthetic inner+outer window, 10 LM iterations per step"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed regions run.  NVML is initialised in the
    constructor (round 1 initialised it inside the thread and the 80 ms region was over before the first sample)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self._nv = self._h = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self._nv, self._h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
        except Exception as e:  # NVML missing: report that instead of inventing numbers
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def run(self):
        nv, h = self._nv, self._h
        if nv is None:
            return
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        try:
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.005)
        except Exception as e:
            self.reasons.add(f"nvml_error:{type(e).__name__}")

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "samples": len(self.samples), "reasons": sorted(self.reasons)}


def schur_kernel_bytes(st, pb):
    """Algorithmic bytes of one fused linearise+Schur launch (BASELINE.md / SURVEY.md 8d):
    reads 40 B/edge + 24 B/landmark + 56 B/pose, writes the Hpl spill 144 B/edge, 96 B/landmark
    (Hll, b_l) and 288 B per block of the reduced system."""
    return 184 * pb.E + 120 * pb.L + 288 * st["nnzb_S"] + 56 * pb.P


def solve_kernel_bytes(st, pb):
    """Algorithmic bytes of one k_solve launch (DESIGN.md 4): read the blocks of the reduced system in the
    factor pattern, write the folded factor N = L_ij L_jj^-1, read it again in the backward solve (288 B per
    block each), and the right-hand side / z / solution (3 x 48 B per pose)."""
    return 288 * 3 * st["nnzb_L"] + 144 * pb.P


def dump_outputs(out_dir, poses, psi, chi2_iter):
    """The arrays a caller of the timed step receives, as float64 .npy files (about 0.5 MB for C2)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("poses", poses), ("psi", psi), ("chi2_iter", chi2_iter)):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def cpu_mt_sample(po, pb, seconds=4.0):
    """The oracle's multi-threaded timing variant (landmark loops of the build and the Schur complement on OpenMP
    threads; the reduced solve stays serial).  The reference's own back-end runs g2o on ONE thread, so this is extra
    information beside the single-thread figure, not the reference's behaviour."""
    n = max(1, min(16, (os.cpu_count() or 1)))
    po.set_threads(n)
    try:
        po.optimize(pb, NUM_ITERS)
        c0, it, runs = time.perf_counter(), 0, 0
        while time.perf_counter() - c0 < seconds and runs < 40:
            it += po.optimize(pb, NUM_ITERS)[2]["iterations"]
            runs += 1
        dt = time.perf_counter() - c0
    finally:
        po.set_threads(1)
    return {"value": it / dt, "unit": "iterations/s", "cores": n, "kind": "port",
            "sample": f"{runs} runs x {NUM_ITERS} LM iterations, oracle/ba_oracle.c with oba_set_threads({n})"}


def run_reference(args):
    from oracle import pyoracle as po
    from scavislam_b200 import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pb = synth.make_config("C2")
    for _ in range(max(args.warmup, 1)):
        po.optimize(pb, NUM_ITERS)
    t0 = time.perf_counter()
    iters = 0
    for _ in range(args.steps):
        poses, psi, st = po.optimize(pb, NUM_ITERS)
        iters += st["iterations"]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, poses, psi, st["chi2_iter"])
    v = iters / dt
    mt = cpu_mt_sample(po, pb)
    line = {
        "impl": "reference", "metric": "GN iterations/sec on 200KF/20k-pt window", "value": v, "unit": "iterations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "P": pb.P, "L": pb.L, "E": pb.E, "C": pb.C, "iters_per_step": NUM_ITERS},
        "cpu_baseline": {"value": v, "unit": "iterations/s", "cores": 1, "kind": "port",
                         "sample": f"{args.steps} steps x {NUM_ITERS} LM iterations of the full C2 window, "
                                   "oracle/ba_oracle.c (single thread, as the reference's backend thread runs g2o)",
                         "multi_thread": mt},
        "e2e": {"value": v, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_ours(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    seq = None
    if rank == 0 and args.frames > 1:
        # the synthetic 640x480 stereo sequence of config C3, rendered by a process pool BEFORE torch / CUDA exist in
        # this process (input generation, untimed)
        from scavislam_b200 import synth_images as si
        seq = si.sequence(args.frames, workers=min(32, os.cpu_count() or 1))
    import torch
    from scavislam_b200 import capi, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # every rank: the C2 window (rank 0: the C2 seed itself, others: same structure, independent noise)
    from scavislam_b200 import dist as sdist
    pb = sdist.window_for_rank(rank)
    ba = capi.BundleAdjuster(device=local)
    ba.set_problem(pb)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        ba.reset_state()
        flush.zero_()                       # evict the window from L2 between steps (untimed)
        torch.cuda.synchronize()
        it, st = ba.optimize(NUM_ITERS)     # device time measured by CUDA events on the library stream
        return it, st

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local)
    if not os.environ.get("SVS_BENCH_NO_SAMPLER"):      # developer knob
        sampler.start()
    barrier()
    wall0 = time.perf_counter()
    ms = 0.0
    iters = 0
    launches = 0
    agg = {"ms_build": 0.0, "ms_solve": 0.0, "ms_update": 0.0, "ms_control": 0.0}
    trials = 0
    st = None
    for _ in range(args.steps):
        it, st = step()
        ms += st["ms_total"]
        iters += it
        launches += st["launches"]
        trials += st["trials_total"]
        for k in agg:
            agg[k] += st[k]
    barrier()
    wall = time.perf_counter() - wall0
    if args.dump_outputs and rank == 0:     # the state the last timed step left on the device, before anything else runs
        dump_outputs(args.dump_outputs, ba.poses(), ba.points(), st["chi2_iter"])

    # end to end through the reference-facing call with host buffers
    e2e_iters = 0
    for _ in range(2):
        ba.optimise_inner_and_outer_window(pb, NUM_ITERS)
    barrier()
    e2e_s = 0.0
    for _ in range(args.steps):
        flush.zero_()                       # L2 eviction between steps, untimed like in the resident loop
        torch.cuda.synchronize()
        t0 = time.perf_counter()            # the call returns with poses and points back in host memory
        it, poses, psi, _ = ba.optimise_inner_and_outer_window(pb, NUM_ITERS)
        e2e_s += time.perf_counter() - t0
        e2e_iters += it
    h2d = sum(getattr(pb, k).nbytes for k in ("pose_qt", "fixed", "psi", "e_point", "e_pose", "e_anchor", "e_obs",
                                               "e_info", "c_i", "c_j", "c_T", "c_Lambda"))
    d2h = pb.pose_qt.nbytes + pb.psi.nbytes

    # the callers' operating point: OptParams(2, true, 3) on a NEW window every back-end tick (backend.cpp:186-187,
    # 196-197, 215-217) -- two LM iterations per call, so the problem definition is not amortised over ten
    CALLER_ITERS = 2
    # consecutive ticks see DIFFERENT windows: alternate between the window and a copy with 2 % of the observations
    # dropped (another edge list, other track shapes), so no call finds its own structure on the device
    pb_alt = synth.with_dropouts(pb, 0.02, seed=5 + rank)
    pair = (pb, pb_alt)
    for k in range(4):
        ba.optimise_inner_and_outer_window(pair[k & 1], CALLER_ITERS)
    e2e2_s, e2e2_iters = 0.0, 0
    for k in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        it, _, _, _ = ba.optimise_inner_and_outer_window(pair[k & 1], CALLER_ITERS)
        e2e2_s += time.perf_counter() - t0
        e2e2_iters += it
    same_s, same_it = 0.0, 0                    # the second optimize() of a tick: same window again (backend.cpp:196-197)
    ba.optimise_inner_and_outer_window(pb, CALLER_ITERS)
    for k in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        it, _, _, _ = ba.optimise_inner_and_outer_window(pb, CALLER_ITERS)
        same_s += time.perf_counter() - t0
        same_it += it
    sp_ms = []                                  # host time of svs_ba_set_problem alone (returns with the uploads enqueued)
    for k in range(max(args.steps, 6)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ba.set_problem(pair[k & 1])
        sp_ms.append(1e3 * (time.perf_counter() - t0))
        torch.cuda.synchronize()
    ba.set_problem(pb)

    # structure variants of the same window, device-resident like `value` (rank 0 only; parity at this size is in
    # tests/test_ba_gpu.py): 20 % visibility drop-outs, and 10 loop-closure constraints that break the band
    variants = {}
    if rank == 0:
        for name, vpb in (("dropouts20", synth.with_dropouts(pb, 0.2, seed=1)), ("loops10", synth.with_loop_closures(pb, 10, seed=1))):
            ba.set_problem(vpb)
            v_ms, v_it, v_agg = 0.0, 0, {"ms_build": 0.0, "ms_solve": 0.0, "ms_update": 0.0}
            for k in range(3 + max(args.steps // 2, 3)):
                ba.reset_state()
                flush.zero_()
                torch.cuda.synchronize()
                it, vst = ba.optimize(NUM_ITERS)
                if k >= 3:
                    v_ms += vst["ms_total"]; v_it += it
                    for q in v_agg:
                        v_agg[q] += vst[q] / max(vst["trials_total"], 1)
            n = max(args.steps // 2, 3)
            variants[name] = {"it_s": v_it / (v_ms * 1e-3), "E": vpb.E, "C": vpb.C, "nnzb_L": vst["nnzb_L"],
                              "kernel_ms_per_trial": {q: v / n for q, v in v_agg.items()}}
    c5 = c5_sharded_block(args, torch, dist, rank, world, local, flush)
    clocks = sampler.stop()

    # max over ranks / sums
    (ms_max, e2e_max, e2e2_max), (tot_iters, tot_e2e, tot_launch, tot_e2e2) = sdist.reduce_job_totals(
        [ms, e2e_s, e2e2_s], [iters, e2e_iters, launches, e2e2_iters], dist, device="cuda")
    tot_launch = int(tot_launch)
    fe = frontend_bench(local, seq) if (rank == 0 and seq is not None) else None

    if rank == 0:
        peak, peak_src = load_peaks()
        traffic = {}
        tp = os.path.join(ROOT, "profiles", "kernel_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f)

        def roof(kernel, key, nbytes, ms_kernel, note):
            k_ms = ms_kernel / max(trials, 1)
            ach = nbytes / (k_ms * 1e-3) / 1e9
            return {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic.get(key), "peak_source": peak_src, "algorithmic_bytes_per_launch": nbytes,
                    "avg_launch_ms": k_ms, "share_of_step": ms_kernel / ms, "note": note}

        roofs = {
            "k_solve": roof("k_solve (block-sparse Cholesky + forward/backward solve, 2-CTA cluster)", "k_solve",
                            solve_kernel_bytes(st, pb), agg["ms_solve"],
                            "a dependent chain of P/2 + w block pivots per CTA: bounded by instruction latency, neither "
                            "HBM nor tensor throughput applies (DESIGN.md 4)"),
            "k_build": roof("k_build_wave (fused linearise + J^T W J + Schur elimination)", "k_build_wave",
                            schur_kernel_bytes(st, pb), agg["ms_build"],
                            "the kernel north_star names for HBM utilisation; FP64 issue/latency-bound at this window "
                            "size: 25 MB per launch, L2-resident between iterations (DESIGN.md 4)"),
        }
        dominant = "k_solve" if agg["ms_solve"] >= agg["ms_build"] else "k_build"
        # bounded CPU baseline sample on this box's host cores
        from oracle import pyoracle as po
        po.optimize(pb, NUM_ITERS)
        c0 = time.perf_counter()
        cit = 0
        nrun = 0
        while time.perf_counter() - c0 < 10.0 and nrun < 40:
            _, _, so = po.optimize(pb, NUM_ITERS)
            cit += so["iterations"]
            nrun += 1
        cdt = time.perf_counter() - c0
        cpu_mt = cpu_mt_sample(po, pb)
        line = {
            "metric": "GN iterations/sec on 200KF/20k-pt window", "value": tot_iters / (ms_max * 1e-3),
            "unit": "iterations/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "P": pb.P, "L": pb.L, "E": pb.E, "C": pb.C,
                       "iters_per_step": NUM_ITERS, "parallelism": f"replicas x{world} (independent windows)",
                       "l2": "flushed between steps (256 MiB write, untimed); iterations inside a step reuse L2 "
                             "as the real workload does",
                       "timing": "sum of per-step CUDA-event times on the library stream, max over ranks",
                       "wall_s_timed_region": wall},
            "e2e": {"value": tot_e2e / e2e_max, "unit": "iterations/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_max / args.steps},
            "e2e_2iter": {"value": tot_e2e2 / e2e2_max, "unit": "iterations/s", "iters_per_call": CALLER_ITERS,
                          "ms_per_call": 1e3 * e2e2_max / args.steps,
                          "set_problem_host_ms_median": float(np.median(sp_ms)),
                          "same_window_again": {"value": same_it / same_s, "ms_per_call": 1e3 * same_s / args.steps},
                          "note": "the callers' operating point, OptParams(2,true,3) (backend.cpp:186-187): host buffers in, poses "
                                  "and points back on the host; consecutive calls alternate between two windows with "
                                  "different edge lists, same_window_again repeats one window (backend.cpp:196-197)"},
            "variants": {k: dict(v, ratio_to_c2=v["it_s"] / (tot_iters / world / (ms_max * 1e-3))) for k, v in variants.items()},
            "c5_sharded": c5,
            "gpu_launches": tot_launch,
            "roofline": roofs[dominant],            # the dominant kernel of the step by measured device time
            "roofline_schur": roofs["k_build"],     # the Schur-elimination kernel, whatever its share
            "kernel_ms_per_step": {k: v / args.steps for k, v in agg.items()},
            "cpu_baseline": {"value": cit / cdt, "unit": "iterations/s", "cores": 1, "kind": "port",
                             "sample": f"{nrun} runs x {NUM_ITERS} LM iterations of the full C2 window "
                                       f"({cdt:.1f} s), oracle/ba_oracle.c single thread",
                             "multi_thread": cpu_mt},
            "clocks": clocks,
            "trials_per_step": trials / args.steps,
            "frontend": fe,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()



def c5_sharded_block(args, torch, dist, rank, world, local, flush):
    """BASELINE config C5: ONE 1000-keyframe / 100k-landmark window whose landmarks are split over all ranks
    (SURVEY.md 8e), driven inside the library: per Levenberg trial one ncclAllReduce of S|bp|bc, a replicated solve
    and one 3-scalar all-reduce, all on the library stream (svs_ba_set_problem_sharded / svs_ba_optimize).
    Strong scaling: the window is fixed, N grows.  Device-resident timing like `value`, max over ranks."""
    from scavislam_b200 import capi, synth
    try:
        pb5 = synth.make_config("C5")
        ba5 = capi.BundleAdjuster(device=local)
        if rank == 0:
            uid = torch.tensor(list(capi.comm_unique_id()), dtype=torch.uint8, device="cuda")
        else:
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if dist is not None:
            dist.broadcast(uid, src=0)
        ba5.comm_init(world, rank, bytes(uid.cpu().numpy().tobytes()))
        ba5.set_problem_sharded(pb5)
        steps = max(3, args.steps // 4)
        ms, iters, agg = 0.0, 0, {"ms_build": 0.0, "ms_solve": 0.0, "ms_update": 0.0, "ms_control": 0.0}
        trials = 0
        for k in range(2 + steps):
            ba5.reset_state()
            flush.zero_()
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            it, st = ba5.optimize(NUM_ITERS)
            if k >= 2:
                ms += st["ms_total"]; iters += it; trials += st["trials_total"]
                for q in agg:
                    agg[q] += st[q]
        t = torch.tensor([ms] + [agg[q] for q in ("ms_build", "ms_solve", "ms_update", "ms_control")], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = [float(x) for x in t]
        out = {"workload": "C5: 1000-keyframe / 100k-landmark single window, landmarks l % N == rank, 10 LM iterations per step",
               "P": pb5.P, "L": pb5.L, "E": pb5.E, "C": pb5.C, "n_gpus": world, "scaling": "strong", "steps": steps,
               "it_s": iters / (t[0] * 1e-3), "ms_per_iteration": t[0] / max(iters, 1),
               "ms_build": t[1] / max(trials, 1), "ms_solve": t[2] / max(trials, 1), "ms_update": t[3] / max(trials, 1),
               "ms_allreduce": t[4] / max(trials, 1), "nnzb_L": st["nnzb_L"],
               "allreduce_bytes_per_trial": 8 * (36 * st["nnzb_L"] + 12 * pb5.P + 3),
               "limiter": "the replicated reduced-system solve (identical on every rank): build and update shrink "
                          "with N, ms_solve does not"}
        ba5.close()
        if rank == 0 and world > 1:   # the same window on one GPU, no collective, beside it
            b1 = capi.BundleAdjuster(device=local)
            b1.set_problem(pb5)
            m1, i1 = 0.0, 0
            for k in range(2 + steps):
                b1.reset_state(); flush.zero_(); torch.cuda.synchronize()
                it, s1 = b1.optimize(NUM_ITERS)
                if k >= 2:
                    m1 += s1["ms_total"]; i1 += it
            out["single_gpu_it_s"] = i1 / (m1 * 1e-3)
            b1.close()
        elif world == 1:
            out["single_gpu_it_s"] = out["it_s"]
        return out
    except Exception as e:   # report, never hide: the main metric above stands on its own
        return {"error": f"{type(e).__name__}: {e}"}


def frontend_bench(device, seq):
    """Second half of the BASELINE metric: front-end frames/sec at 640x480 (config C3, SURVEY.md 8d: a 200-frame synthetic
    stereo sequence, 2 cm / 0.2 deg per frame) -- preprocessing (pyramids, gradients) + grid FAST (2 levels, adaptive) +
    dense tracking (3 levels) + dense point cloud + guided matching against the previous frame + motion-only LM, through the
    C ABI.  `fps_e2e` takes the raw left image and the disparity map from host memory every frame; `fps_resident` re-runs
    the kernels of the last frame pair on data already on the device."""
    import numpy as np
    import torch
    from oracle import pyoracle as po
    from scavislam_b200 import capi, frontend_inputs as fi
    cams = fi.level_cams()
    I7 = np.array([0, 0, 0, 1, 0, 0, 0.0])
    lv2 = [(640 >> l, 480 >> l, cams[l][0], cams[l][1], cams[l][2]) for l in range(2)]
    n_frames = len(seq) - 1
    grids = [capi.FastGrid(640, 480, 222, 74, 25, 3, 3, device=device), capi.FastGrid(320, 240, 55, 18, 25, 3, 3, device=device)]
    dt = capi.DenseTracker(640, 480, 3, device=device)
    for l in range(3):
        dt.set_intrinsics(l, cams[l][0], cams[l][1], cams[l][2])
    mt = capi.GuidedMatcher(lv2, device=device)

    def make_points(prev, kxy):
        d = prev["disp"][kxy[:, 1], kxy[:, 0]]
        ok = d > 0
        kxy, d = kxy[ok], d[ok]
        z = cams[0][0] * cams[0][3] / d
        p = np.zeros(len(kxy), capi.MATCH_POINT_DTYPE)
        p["xyz_anchor"] = np.stack([(kxy[:, 0] - cams[0][1]) / cams[0][0] * z, (kxy[:, 1] - cams[0][2]) / cams[0][0] * z, z], 1)
        p["anchor_obs_pyr"] = kxy
        return p

    pose = capi.PoseOptimizer(device=device)
    pps = [capi.FramePreprocessor(640, 480, 3, device=device) for _ in range(2)]
    state = {"k": 0}

    def one_frame(prev, cur, prev_xy, upload=True):
        """upload=True: the per-frame host inputs are the raw left image and the disparity maps; pyramids and gradients
        are made on the device (svs_prep_*) and handed over by pointer; the FAST corners go to the matcher on the device."""
        if upload:
            state["k"] ^= 1
            pp, pq = pps[state["k"]], pps[state["k"] ^ 1]       # pp: current frame, pq: previous frame
            pp.process(cur["img"])
            lv = [pp.level(l) for l in range(3)]
        xy0 = None
        for l in range(2):
            if upload:
                grids[l].set_image_device(lv[l]["u8"], lv[l]["pitch_u8"], lv[l]["w"], lv[l]["h"])
            xy, off = grids[l].detect_adaptively(6)
            if l == 0:
                xy0 = xy
            if upload:
                mt.set_features_from_fast(l, grids[l])
        if upload:
            dt.set_disparity(prev["disp"])
            dt.swap_prev_cur()                                   # FrameData::nextFrame
            for l in range(3):
                dt.set_images_device(l, None, lv[l]["f32"], lv[l]["dx"], lv[l]["dy"], lv[l]["stride_f32"])
        dt.compute_point_cloud(I7, cams)
        T, st = dt.track(I7)
        if upload:
            lq = [pq.level(l) for l in range(2)]
            mt.set_pyramid_device(0, [x["u8"] for x in lq], [x["pitch_u8"] for x in lq], I7)
            mt.set_pyramid_device(-1, [x["u8"] for x in lv[:2]], [x["pitch_u8"] for x in lv[:2]])
            mt.set_current_disparity(cur["disp"])
        res = mt.match(T, I7, make_points(prev, prev_xy), 4, 22, 10)
        nm = int(res["matched"].sum())
        if nm >= 20:                                             # stereo_frontend.cpp:1053-1063
            T, _ = pose.calc_fast_motion_only_matched(mt, cams[0][:4], T, True, 2.0, 15)
        return xy0, T, nm, st

    pps[0].process(seq[0]["img"])                # prime: frame 0 is "previous"
    for l in range(3):
        lv0 = pps[0].level(l)
        dt.set_images_device(l, lv0["f32"], lv0["f32"], lv0["dx"], lv0["dy"], lv0["stride_f32"])
    prev_xy = one_frame(seq[0], seq[1], np.zeros((0, 2), np.int32))[0]
    for i in range(1, min(4, n_frames)):         # warm-up on the first frames
        prev_xy = one_frame(seq[i], seq[i + 1], prev_xy)[0]
    # timed: the whole sequence once more from its start
    pps[state["k"]].process(seq[0]["img"])
    for l in range(3):
        lv0 = pps[state["k"]].level(l)
        dt.set_images_device(l, None, lv0["f32"], lv0["dx"], lv0["dy"], lv0["stride_f32"])
    prev_xy = one_frame(seq[0], seq[1], np.zeros((0, 2), np.int32))[0]
    torch.cuda.synchronize()
    frame_ms, matched, passes, dt_ms, dt_bytes = [], 0, np.zeros(3), 0.0, 0.0
    t0 = time.perf_counter()
    for i in range(1, n_frames):
        tf = time.perf_counter()
        prev_xy, T, m, st = one_frame(seq[i], seq[i + 1], prev_xy)
        frame_ms.append((time.perf_counter() - tf) * 1e3)
        matched += m
        passes += np.asarray(st["passes"][:3])
        dt_ms += st["ms_total"]
        dt_bytes += sum(36.0 * st["passes"][l] * (640 >> l) * (480 >> l) for l in range(3))
    e2e = time.perf_counter() - t0
    timed = n_frames - 1
    a, b = seq[n_frames - 1], seq[n_frames]
    t0 = time.perf_counter()
    nres = min(timed, 50)
    for i in range(nres):
        one_frame(a, b, prev_xy, upload=False)
    res_s = time.perf_counter() - t0
    # CPU oracle on frames of the same sequence (1 thread), bounded sample: >= 20 frames
    ncpu = min(20, n_frames)
    cpu_frames = []
    for f in seq[:ncpu + 1]:                    # host pyramids/gradients (OpenCV) feed the CPU baseline only
        fp = fi.float_pyramid(f["img"])
        cpu_frames.append(dict(u8=fi.uint8_pyramid(f["img"], 2), f32=fp, grad=[fi.gradients(x) for x in fp], disp=f["disp"]))
    c0 = time.perf_counter()
    for i in range(ncpu):
        fa, fb = cpu_frames[i], cpu_frames[i + 1]
        for l in range(2):
            g = po.fast_grid(640 >> l, 480 >> l, 222 if l == 0 else 55, 74 if l == 0 else 18, 25, 3, 3)
            po.fast_detect_adaptively(fb["u8"][l], g, 6)
        lv = [dict(prev=fa["f32"][l], cur=fb["f32"][l], dx=fb["grad"][l][0], dy=fb["grad"][l][1], f=cams[l][0], px=cams[l][1],
                   py=cams[l][2], cloud=po.dt_point_cloud(I7, cams[l], fa["disp"], l, 640 >> l, 480 >> l)) for l in range(3)]
        po.dt_track(lv, I7)
    cpu_s = time.perf_counter() - c0
    peak, peak_src = load_peaks()
    dt_gbs = dt_bytes / max(dt_ms * 1e-3, 1e-12) / 1e9
    out = {"workload": f"C3: 640x480 synthetic stereo stream, {len(seq)} frames (2 cm / 0.2 deg per frame); preprocessing (pyramids, "
                       "gradients) + FAST grid (2 levels, 6 trials) + dense tracking (3 levels) + point cloud + guided matching "
                       "(radius 4, corners handed over on the device) + motion-only LM (15 it)",
           "fps_e2e": timed / e2e, "fps_resident": nres / res_s, "frames": timed,
           "frame_ms_median": float(np.median(frame_ms)), "frame_ms_max": float(np.max(frame_ms)),
           "timing": "wall clock over the whole sequence, one pass",
           "matched_per_frame": matched / timed, "dense_tracking_passes_per_frame": (passes / timed).tolist(),
           "dense_tracking_ms_per_frame": dt_ms / timed,
           "roofline": {"bound": "hbm", "kernel": "k_dt_track_level (fused chi2 + J^T J + J^T r pass, whole LM loop on the device)",
                        "achieved": dt_gbs, "peak": peak, "unit": "GB/s", "frac": dt_gbs / peak, "traffic": None,
                        "peak_source": peak_src, "algorithmic_bytes_per_frame": dt_bytes / timed,
                        "note": "36 B per pixel and pass (SURVEY.md 8d); latency-bound: one grid-wide rendezvous, a 28-value "
                                "reduction and a 6x6 solve per pass, independent of the image size"},
           "cpu_baseline_fps": ncpu / cpu_s, "cpu_baseline": "oracle FAST + dense tracking (GPU semantics), 1 thread, "
                                                               f"{ncpu} frames of the sequence (matcher excluded: <5 ms)"}
    for g in grids + pps + [pose]:
        g.close()
    dt.close()
    mt.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=200, help="frames of the synthetic C3 sequence (0: skip the front-end part)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the poses, landmarks and chi2 trace of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
