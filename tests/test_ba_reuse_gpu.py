"""GPU parity tests of a BundleAdjuster handle that is reused across problems.

svs_ba_set_problem has three ways in: the full structure analysis; the same-structure re-send (index arrays, sizes,
`fixed` and flags equal to the problem on the device: only the numbers travel); and the cached symbolic
factorisation (the P x P co-visibility pattern is unchanged, the edge list is new).  The back-end runs the last two on
every tick.  Whatever a handle did before, a call must give what a fresh handle gives on THAT call's problem, so every
check here is against the oracle on the problem just loaded.  Every case also checks that it has teeth: the oracle's
answer for the problem loaded before differs from the current one by far more than the bar, so a number left over
from the earlier problem cannot pass.

Which path a call took is read from the library's SVS_HOST_TIMING lines on stderr.
"""
import dataclasses
import sys

import numpy as np
import pytest

from scavislam_b200 import synth, synth_graph

pytestmark = pytest.mark.gpu

POSE_RTOL = 1e-6
REUSED = "set_problem: structure reused"
SYMBOLIC = "set_problem: symbolic factorisation reused"
ITEMS = ("e_obs", "e_info", "psi", "pose_qt", "c_T", "c_Lambda", "cam")


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


@pytest.fixture
def timing(monkeypatch, capfd):
    """Switches the library's host-timing lines on; returns a function that gives the lines written since its last call."""
    monkeypatch.setenv("SVS_HOST_TIMING", "1")
    capfd.readouterr()

    def lines():
        err = capfd.readouterr().err
        with capfd.disabled():                 # the path lines go to the test log as well
            for ln in err.splitlines():
                if "reused" in ln:
                    sys.stderr.write(ln + "\n")
        return err
    return lines


def _paths(err):
    return REUSED in err, SYMBOLIC in err


def _perturb(pb, item, seed=0):
    """A copy of `pb` with one number class changed (same index arrays, sizes and `fixed`)."""
    from oracle import pyoracle as po
    rng = np.random.default_rng(seed)
    out = pb.copy()
    if item == "e_obs":
        out.e_obs = pb.e_obs + rng.normal(0, 0.4, pb.e_obs.shape)
    elif item == "e_info":
        out.e_info = pb.e_info * rng.uniform(0.3, 3.0, pb.e_info.shape)
    elif item == "psi":
        out.psi = pb.psi.copy()
        out.psi[:, :2] += rng.normal(0, 2e-3, (pb.L, 2))
        out.psi[:, 2] *= 1 + rng.normal(0, 0.05, pb.L)
    elif item == "pose_qt":
        out.pose_qt = pb.pose_qt.copy()
        for p in np.nonzero(pb.fixed == 0)[0]:
            d = np.concatenate([rng.normal(0, 0.01, 3), rng.normal(0, 0.003, 3)])
            out.pose_qt[p] = po.se3_mul(po.se3_exp(d), pb.pose_qt[p])
    elif item == "c_T":
        out.c_T = np.stack([po.se3_mul(po.se3_exp(np.concatenate([rng.normal(0, 0.01, 3), rng.normal(0, 0.003, 3)])), T)
                            for T in pb.c_T])
    elif item == "c_Lambda":
        out.c_Lambda = pb.c_Lambda * rng.uniform(0.2, 5.0, (pb.C, 1))
    elif item == "cam":
        out.cam = pb.cam * np.array([1.01, 1.0, 1.0, 1.03]) + np.array([0.0, 2.5, -1.5, 0.0])
    else:
        raise ValueError(item)
    return out


def _reference(oracle, pb, iters=4):
    """What a fresh handle must produce on `pb`: chi2, the reduced system at lambda 50, and an `iters` trajectory."""
    S, bs, chi = oracle.reduced_system(pb, True, 1.0, 50.0)
    return dict(chi2=oracle.chi2(pb, True, 1.0), S=S, bs=bs, chi=chi, iters=iters, traj=oracle.optimize(pb, iters))


def _moved(chi_new, chi_old):
    """Final chi2 of two trajectories 100 times further apart than the trajectory bar."""
    return abs(chi_new - chi_old) > 1e-5 * abs(chi_old)


def _has_teeth(ref_new, ref_old):
    """The reference moved by far more than the bars of _check: a value left over from the old problem fails."""
    assert (abs(ref_new["chi2"] - ref_old["chi2"]) > 1e-6 * abs(ref_old["chi2"]) or _rel(ref_new["S"], ref_old["S"]) > 1e-6
            or _rel(ref_new["bs"], ref_old["bs"]) > 1e-6), "the two problems have the same reference"
    assert _moved(ref_new["traj"][2]["chi2_final"], ref_old["traj"][2]["chi2_final"]), "the two problems optimise alike"


def _check(ba, ref):
    """The problem loaded in `ba` against its reference; returns the GPU trajectory's stats."""
    g = ba.chi2(True, 1.0)
    assert abs(g - ref["chi2"]) <= 1e-11 * abs(ref["chi2"]), (g, ref["chi2"])
    S, bs, chi = ba.reduced_system(True, 1.0, 50.0)
    assert abs(chi - ref["chi"]) <= 1e-11 * abs(ref["chi"])
    assert _rel(S, ref["S"]) < 1e-11, _rel(S, ref["S"])
    assert _rel(bs, ref["bs"]) < 1e-10, _rel(bs, ref["bs"])
    it, st = ba.optimize(ref["iters"])
    po_, ps_, sto = ref["traj"]
    assert it == sto["iterations"] and st["trials_iter"] == sto["trials_iter"], (it, st["trials_iter"], sto["trials_iter"])
    np.testing.assert_allclose(st["chi2_iter"], sto["chi2_iter"], rtol=1e-7)
    np.testing.assert_allclose(st["lambda_iter"], sto["lambda_iter"], rtol=1e-6)
    assert _rel(ba.poses(), po_) < POSE_RTOL and _rel(ba.points(), ps_) < POSE_RTOL
    return st


@pytest.fixture(scope="module")
def padded_window():
    """40 frames with 20 % drop-outs (tracks completed with zero-weight padding edges) and one fixed frame."""
    pb = synth.with_dropouts(synth.make_window(40, 3000, seed=41), 0.2, seed=3)
    pb.fixed[0] = 1
    return pb


@pytest.fixture(scope="module")
def padded_ref(oracle, padded_window):
    return _reference(oracle, padded_window)


# ---------------------------------------------------------------- (a) one number class at a time, same structure

@pytest.mark.parametrize("item", ITEMS)
def test_same_structure_resend_of_one_number_class(svs, oracle, timing, padded_window, padded_ref, item):
    A = padded_window
    B = _perturb(A, item, seed=ITEMS.index(item))
    ref_b = _reference(oracle, B)
    _has_teeth(ref_b, padded_ref)
    ba = svs.BundleAdjuster()
    ba.set_problem(A)
    ba.optimize(2)                                   # the control block, the state buffers and S are no longer fresh
    timing()
    ba.set_problem(B)
    assert _paths(timing())[0], "the same-structure path was not taken"
    _check(ba, ref_b)
    ba.close()


# ---------------------------------------------------------------- (b) the same on windows that reach the other build kernels

def _two_loads(svs, oracle, timing, A, B, iters=4):
    ref_a, ref_b = _reference(oracle, A, iters), _reference(oracle, B, iters)
    _has_teeth(ref_b, ref_a)
    ba = svs.BundleAdjuster()
    ba.set_problem(A)
    timing()
    st_a = _check(ba, ref_a)
    ba.set_problem(B)
    assert _paths(timing())[0], "the same-structure path was not taken"
    st_b = _check(ba, ref_b)
    ba.close()
    return st_a, st_b


def test_same_structure_resend_long_tracks(svs, oracle, timing):
    """Tracks of 9-32 slots (k_build) and of more than 32 (k_build_long): their landmark permutations."""
    A = synth.make_window(70, 900, seed=36, T=50)
    B = _perturb(_perturb(_perturb(A, "psi", 1), "e_obs", 2), "e_info", 3)
    _, st = _two_loads(svs, oracle, timing, A, B)
    assert st["max_track"] > 33


def test_same_structure_resend_full_size_c2(svs, oracle, timing):
    """C2 is the size at which k_build_wave runs its persistent grid."""
    A = synth.make_config("C2")
    B = _perturb(_perturb(A, "psi", 4), "e_obs", 5)
    _two_loads(svs, oracle, timing, A, B)


# ---------------------------------------------------------------- (c) `fixed` is part of the structure

def test_changed_fixed_frames_are_not_reused(svs, oracle, timing, padded_window, padded_ref):
    B = padded_window.copy()
    B.fixed[[5, 17, 30]] = 1
    ref_b = _reference(oracle, B)
    _has_teeth(ref_b, padded_ref)
    ba = svs.BundleAdjuster()
    ba.set_problem(padded_window)
    ba.optimize(2)
    timing()
    ba.set_problem(B)
    assert not _paths(timing())[0], "a change of `fixed` took the same-structure path"
    _check(ba, ref_b)
    g = ba.poses()
    assert np.array_equal(g[[0, 5, 17, 30]], B.pose_qt[[0, 5, 17, 30]])
    ba.close()


# ---------------------------------------------------------------- (d) the cached symbolic factorisation

def _add_constraints(pb, pairs, seed=0):
    """Pose-pose constraints (both orders) between far-apart keyframes, measured from the truth."""
    from oracle import pyoracle as po
    rng = np.random.default_rng(seed)
    ci, cj, cT, cL = list(pb.c_i), list(pb.c_j), list(pb.c_T), list(pb.c_Lambda)
    for (i, j) in pairs:
        for (a, b) in ((i, j), (j, i)):
            T = po.se3_mul(po.se3_exp(rng.normal(0, 1e-3, 6)), po.se3_mul(pb.truth_pose_qt[b], po.se3_inv(pb.truth_pose_qt[a])))
            ci.append(a); cj.append(b); cT.append(T); cL.append(np.diag([4e4] * 3 + [1e5] * 3).reshape(36))
    out = pb.copy()
    out.c_i, out.c_j = np.asarray(ci, np.int32), np.asarray(cj, np.int32)
    out.c_T, out.c_Lambda = np.asarray(cT, np.float64).reshape(-1, 7), np.asarray(cL, np.float64).reshape(-1, 36)
    out.C = len(ci)
    return out


@pytest.mark.parametrize("window", ["two_ended_split", "loop_closures"])
def test_symbolic_factorisation_cache(svs, oracle, timing, window):
    """A -> A with 2 % drop-outs (new edge list, same pattern: the cached factorisation, its branch split and separator
    are reused) -> A plus a loop closure (new pattern: nothing reused) -> A again (nothing reused: the cache holds the
    loop-closure pattern)."""
    A = synth.make_window(90, 4000, seed=34)
    if window == "loop_closures":             # both ends coupled: the coupled frames join the separator of the split
        A = _add_constraints(A, [(3, 84), (10, 77)], seed=1)
    steps = [(A, (False, False)), (synth.with_dropouts(A, 0.02, seed=7), (False, True)),
             (_add_constraints(A, [(20, 70)], seed=2), (False, False)), (A, (False, False))]
    refs = [_reference(oracle, pb) for pb, _ in steps]
    for k in range(1, len(steps)):
        _has_teeth(refs[k], refs[k - 1])
    ba = svs.BundleAdjuster()
    timing()
    for (pb, want), ref in zip(steps, refs):
        ba.set_problem(pb)
        assert _paths(timing()) == want, (pb.name, want)
        _check(ba, ref)
    ba.close()


# ---------------------------------------------------------------- (e) size and build-kernel mix on one handle

def test_size_and_kernel_mix_transitions(svs, oracle):
    """C2 (persistent k_build_wave grid) -> C1 (the arena shrinks, one task per warp) -> long tracks (k_build_long) ->
    C2 again (the arena grows back)."""
    c2 = synth.make_config("C2")
    seq = [c2, synth.make_config("C1"), synth.make_window(70, 900, seed=36, T=50), c2]
    refs = {}
    ba = svs.BundleAdjuster()
    for pb in seq:
        if id(pb) not in refs:
            refs[id(pb)] = _reference(oracle, pb)
        ba.set_problem(pb)
        _check(ba, refs[id(pb)])
    ba.close()


# ---------------------------------------------------------------- (f) map-assembled and host problems on one handle

def _assembled(pb, g):
    return dataclasses.replace(pb, E=len(g["e_point"]), pose_qt=g["pose_qt"], psi=g["psi"], e_point=g["e_point"],
                               e_pose=g["e_pose"], e_anchor=g["e_anchor"], e_obs=g["e_obs"], e_info=g["e_info"])


@pytest.fixture(scope="module")
def map_window():
    pb = synth.make_window(30, 3000, seed=6)
    pb.fixed[0] = 1
    m, win, act = synth_graph.make_map(pb, seed=6)
    return pb, m, win, act


def _load_map(dm, m):
    dm.set(m["poses"], m["point_anchor"], m["xyz_anchor"], m["vis_ptr"], m["vis_pose"], m["feat_center"], m["feat_level"])


def _map_problem(dm, ba, pb, win, act):
    return dm.set_problem(ba, win, act, pb.cam, fixed=pb.fixed, c_i=pb.c_i, c_j=pb.c_j, c_T=pb.c_T, c_Lambda=pb.c_Lambda)


def test_map_then_host_with_the_same_window(svs, oracle, timing, map_window):
    """The map path keeps observations on the device and never sized the handle's host staging buffer: the host call
    that follows with the same index arrays must still send its own observations and weights."""
    pb, m, win, act = map_window
    pa = _assembled(pb, oracle.copy_data_to_g2o(m, win, act))
    host = _perturb(_perturb(pa, "e_obs", 11), "e_info", 12)
    ref_m, ref_h = _reference(oracle, pa), _reference(oracle, host)
    _has_teeth(ref_h, ref_m)
    dm, ba = svs.DeviceMap(), svs.BundleAdjuster()
    _load_map(dm, m)
    timing()
    _map_problem(dm, ba, pb, win, act)
    assert _paths(timing()) == (False, False)
    _check(ba, ref_m)
    ba.set_problem(host)
    assert _paths(timing())[0], "the same-structure path was not taken"
    _check(ba, ref_h)
    dm.close(); ba.close()


def test_host_then_map_and_map_then_map(svs, oracle, timing, map_window):
    pb, m, win, act = map_window
    pa = _assembled(pb, oracle.copy_data_to_g2o(m, win, act))
    host = _perturb(_perturb(pa, "e_obs", 13), "psi", 14)
    m2 = dict(m)
    m2["feat_center"] = m["feat_center"] + np.random.default_rng(15).normal(0, 0.4, m["feat_center"].shape)
    pa2 = _assembled(pb, oracle.copy_data_to_g2o(m2, win, act))
    assert np.array_equal(pa2.e_point, pa.e_point) and np.array_equal(pa2.e_pose, pa.e_pose)
    refs = [_reference(oracle, x) for x in (host, pa, pa2)]
    _has_teeth(refs[1], refs[0])
    _has_teeth(refs[2], refs[1])
    dm, ba = svs.DeviceMap(), svs.BundleAdjuster()
    _load_map(dm, m)
    ba.set_problem(host)
    timing()
    _check(ba, refs[0])
    _map_problem(dm, ba, pb, win, act)                     # host -> map
    assert _paths(timing())[0], "the same-structure path was not taken"
    _check(ba, refs[1])
    _load_map(dm, m2)                                      # map -> map: the same edges with new observations
    _map_problem(dm, ba, pb, win, act)
    assert _paths(timing())[0], "the same-structure path was not taken"
    _check(ba, refs[2])
    dm.close(); ba.close()


# ---------------------------------------------------------------- (g) the back-end's tick

def test_one_call_ticks(svs, oracle, timing):
    """optimise_inner_and_outer_window twice on a window (the second call starts from the first call's write-back), then
    the window alternating with a 2 %-drop-out copy of it, as the end-to-end benchmark runs it."""
    pb = synth.make_window(40, 3000, seed=52)
    ba = svs.BundleAdjuster()
    timing()
    it, poses, psi, st = ba.optimise_inner_and_outer_window(pb, 2)
    p_o, s_o, st_o = oracle.optimize(pb, 2)
    assert it == st_o["iterations"] and st["trials_iter"] == st_o["trials_iter"]
    assert _rel(poses, p_o) < POSE_RTOL and _rel(psi, s_o) < POSE_RTOL
    upd = pb.copy()
    upd.pose_qt, upd.psi = poses.copy(), psi.copy()
    p_u, s_u, st_u = oracle.optimize(upd, 2)
    assert _moved(st_u["chi2_iter"][0], st_o["chi2_iter"][0])   # a stale initial state would repeat the first call
    it, poses2, psi2, st = ba.optimise_inner_and_outer_window(upd, 2)
    assert _paths(timing())[0], "the same-structure path was not taken"
    assert it == st_u["iterations"] and st["trials_iter"] == st_u["trials_iter"]
    np.testing.assert_allclose(st["chi2_iter"], st_u["chi2_iter"], rtol=1e-7)
    np.testing.assert_allclose(st["lambda_iter"], st_u["lambda_iter"], rtol=1e-6)
    assert _rel(poses2, p_u) < POSE_RTOL and _rel(psi2, s_u) < POSE_RTOL
    assert np.array_equal(poses2, ba.poses()) and np.array_equal(psi2, ba.points())
    drop = synth.with_dropouts(pb, 0.02, seed=9)
    prev = None
    for tick in (drop, pb, drop, pb):
        it, poses, psi, st = ba.optimise_inner_and_outer_window(tick, 2)
        assert _paths(timing()) == (False, True), tick.name
        p_t, s_t, st_t = oracle.optimize(tick, 2)
        if prev is not None:
            assert _moved(st_t["chi2_final"], prev)
        prev = st_t["chi2_final"]
        assert it == st_t["iterations"] and st["trials_iter"] == st_t["trials_iter"]
        np.testing.assert_allclose(st["chi2_iter"], st_t["chi2_iter"], rtol=1e-7)
        assert _rel(poses, p_t) < POSE_RTOL and _rel(psi, s_t) < POSE_RTOL
    ba.close()


# ---------------------------------------------------------------- (h) control: the re-send equals the full analysis

def test_resend_equals_full_analysis(svs, timing, monkeypatch, padded_window):
    """Every number class changed at once, loaded through the same-structure path and, on a second handle with the same
    history, through the full analysis (SVS_NO_STRUCT_REUSE=1): the results agree to the FP64-atomics level."""
    B = padded_window
    for k, item in enumerate(ITEMS):
        B = _perturb(B, item, seed=20 + k)
    out = []
    for reuse in (True, False):
        ba = svs.BundleAdjuster()
        ba.set_problem(padded_window)
        ba.optimize(2)
        timing()
        if not reuse:
            monkeypatch.setenv("SVS_NO_STRUCT_REUSE", "1")
        ba.set_problem(B)
        monkeypatch.delenv("SVS_NO_STRUCT_REUSE", raising=False)
        assert _paths(timing())[0] == reuse
        S, bs, chi = ba.reduced_system(True, 1.0, 50.0)
        it, st = ba.optimize(4)
        out.append((S, bs, chi, it, st, ba.poses(), ba.points()))
        ba.close()
    (S1, b1, c1, it1, st1, p1, s1), (S2, b2, c2, it2, st2, p2, s2) = out
    assert _rel(S1, S2) < 1e-10 and _rel(b1, b2) < 1e-10 and abs(c1 - c2) <= 1e-10 * abs(c2)
    assert it1 == it2 and st1["trials_iter"] == st2["trials_iter"]
    np.testing.assert_allclose(st1["chi2_iter"], st2["chi2_iter"], rtol=1e-10)
    assert _rel(p1, p2) < 1e-10 and _rel(s1, s2) < 1e-10
