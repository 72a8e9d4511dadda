"""The C++ host layer (include/svs_b200.hpp): compiles with plain g++ against the C ABI (CPU), and on
the GPU box reproduces the oracle through the id-based SlamGraph-like interface."""
import os
import subprocess

import numpy as np
import pytest

from scavislam_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bin_dir(tmp_path_factory):
    """The test programs are built outside the repository tree, which may be read-only."""
    return tmp_path_factory.mktemp("cpp")


def _compile(name, bin_dir):
    src = os.path.join(ROOT, "tests", "cpp", name + ".cpp")
    exe = str(bin_dir / name)
    if not os.path.exists(exe):
        lib_dir = os.path.join(ROOT, "scavislam_b200")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                               "-L", lib_dir, "-lsvsb200", f"-Wl,-rpath,{lib_dir}"])
    return exe


def _dump(pb, path):
    xyz = np.stack([pb.psi[:, 0] / pb.psi[:, 2], pb.psi[:, 1] / pb.psi[:, 2], 1.0 / pb.psi[:, 2]], 1)
    with open(path, "wb") as f:
        np.array([pb.P, pb.L, pb.E, pb.C], np.int32).tofile(f)
        np.asarray(pb.cam, np.float64).tofile(f)
        for a in (pb.pose_qt, xyz):
            np.ascontiguousarray(a, np.float64).tofile(f)
        for a in (pb.e_point, pb.e_pose, pb.e_anchor):
            np.ascontiguousarray(a, np.int32).tofile(f)
        for a in (pb.e_obs, pb.e_info):
            np.ascontiguousarray(a, np.float64).tofile(f)
        for a in (pb.c_i, pb.c_j):
            np.ascontiguousarray(a, np.int32).tofile(f)
        for a in (pb.c_T, pb.c_Lambda):
            np.ascontiguousarray(a, np.float64).tofile(f)


def test_cpp_layer_compiles_and_fails_loudly_without_gpu(svs, tmp_path, bin_dir):
    import torch
    exe = _compile("shim_main", bin_dir)
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    pb = synth.make_window(4, 30, seed=2)
    _dump(pb, tmp_path / "in.bin")
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin"), "1"], capture_output=True, text=True)
    assert r.returncode == 3 and "NO_GPU" in r.stdout        # no CPU fallback


@pytest.mark.gpu
def test_cpp_layer_matches_oracle(svs, oracle, tmp_path, bin_dir):
    exe = _compile("shim_main", bin_dir)
    pb = synth.make_config("C1")
    _dump(pb, tmp_path / "in.bin")
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin"), "2"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "OK iterations=2" in r.stdout and f"point_edges={pb.E}" in r.stdout
    out = np.fromfile(tmp_path / "out.bin", np.float64)
    poses = out[:7 * pb.P].reshape(pb.P, 7)
    xyz = out[7 * pb.P:].reshape(pb.L, 3)
    p_o, s_o, _ = oracle.optimize(pb, 2)     # huber delta stays 1 like the reference (SURVEY B1)
    xyz_o = np.stack([s_o[:, 0] / s_o[:, 2], s_o[:, 1] / s_o[:, 2], 1.0 / s_o[:, 2]], 1)
    assert np.abs(poses - p_o).max() <= 1e-6 * np.abs(p_o).max()
    assert np.abs(xyz - xyz_o).max() <= 1e-6 * np.abs(xyz_o).max()


def test_cpp_frontend_layer_compiles(svs, bin_dir):
    _compile("frontend_main", bin_dir)


@pytest.mark.gpu
def test_cpp_frontend_and_map_wrappers_equal_the_c_abi(svs, tmp_path, bin_dir):
    """FramePreprocessor, FastGrid, DenseTracker, GuidedMatcher (corners handed over on the device),
    BA_SE3_XYZ_STEREO and DeviceMap of include/svs_b200.hpp, driven from C++ with the reference's method names, give
    what the same calls through the C ABI give (made here from Python): every wrapper is exercised, none is a shell."""
    from scavislam_b200 import frontend_inputs as fi, synth_graph, synth_images as si
    exe = _compile("frontend_main", bin_dir)
    seq = si.sequence(2)
    cams = fi.level_cams()
    pb = synth.make_window(12, 600, seed=9)
    m, win, act = synth_graph.make_map(pb, seed=9)
    W, H = 640, 480
    with open(tmp_path / "in.bin", "wb") as f:
        np.array([W, H, len(m["poses"]), len(m["point_anchor"]), len(m["vis_pose"]), len(win), len(act), 3], np.int32).tofile(f)
        np.asarray(cams[:3], np.float64).tofile(f)
        for k in (0, 1):
            np.ascontiguousarray(seq[k]["img"], np.uint8).tofile(f)
        for k in (0, 1):
            np.ascontiguousarray(seq[k]["disp"], np.float32).tofile(f)
        np.ascontiguousarray(m["poses"], np.float64).tofile(f)
        np.ascontiguousarray(m["point_anchor"], np.int32).tofile(f)
        np.ascontiguousarray(m["xyz_anchor"], np.float64).tofile(f)
        np.ascontiguousarray(m["vis_ptr"], np.int32).tofile(f)
        np.ascontiguousarray(m["vis_pose"], np.int32).tofile(f)
        np.ascontiguousarray(m["feat_center"], np.float64).tofile(f)
        np.ascontiguousarray(m["feat_level"], np.int32).tofile(f)
        np.ascontiguousarray(win, np.int32).tofile(f)
        np.ascontiguousarray(act, np.int32).tofile(f)
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr

    # the same through the C ABI from Python
    I7 = np.array([0, 0, 0, 1, 0, 0, 0.0])
    pps = [svs.FramePreprocessor(W, H, 3) for _ in range(2)]
    for k in (0, 1):
        pps[k].process(seq[k]["img"])
    l0, l1 = [pps[0].level(l) for l in range(3)], [pps[1].level(l) for l in range(3)]
    fg0, fc0 = svs.FastGrid(W, H, 222, 74, 25, 3, 3), svs.FastGrid(W, H, 222, 74, 25, 3, 3)
    fg1 = svs.FastGrid(W // 2, H // 2, 55, 18, 25, 3, 3)
    fg0.set_image_device(l0[0]["u8"], l0[0]["pitch_u8"], W, H)
    kxy0, _ = fg0.detect_adaptively(6)
    fc0.set_image_device(l1[0]["u8"], l1[0]["pitch_u8"], W, H)
    xy0, _ = fc0.detect_adaptively(6)
    fg1.set_image_device(l1[1]["u8"], l1[1]["pitch_u8"], W // 2, H // 2)
    xy1, _ = fg1.detect_adaptively(6)
    dt = svs.DenseTracker(W, H, 3)
    for l in range(3):
        dt.set_intrinsics(l, cams[l][0], cams[l][1], cams[l][2])
        dt.set_images_device(l, l0[l]["f32"], l1[l]["f32"], l1[l]["dx"], l1[l]["dy"], l1[l]["stride_f32"])
    dt.set_disparity(seq[0]["disp"])
    dt.compute_point_cloud(I7, cams)
    T_track, _ = dt.track(I7)
    lv = [(W >> l, H >> l, cams[l][0], cams[l][1], cams[l][2]) for l in range(2)]
    gm = svs.GuidedMatcher(lv)
    gm.set_pyramid_device(0, [x["u8"] for x in l0[:2]], [x["pitch_u8"] for x in l0[:2]], I7)
    gm.set_pyramid_device(-1, [x["u8"] for x in l1[:2]], [x["pitch_u8"] for x in l1[:2]])
    gm.set_current_disparity(seq[1]["disp"])
    gm.set_features_from_fast(0, fc0)
    gm.set_features_from_fast(1, fg1)
    d = seq[0]["disp"][kxy0[:, 1], kxy0[:, 0]]
    ok = d > 0
    kk, dd = kxy0[ok], d[ok].astype(np.float64)
    z = cams[0][0] * cams[0][3] / dd
    pts = np.zeros(len(kk), svs.MATCH_POINT_DTYPE)
    pts["xyz_anchor"] = np.stack([(kk[:, 0] - cams[0][1]) / cams[0][0] * z, (kk[:, 1] - cams[0][2]) / cams[0][0] * z, z], 1)
    pts["anchor_obs_pyr"] = kk
    res = gm.match(T_track, I7, pts, 4, 22, 10)
    po = svs.PoseOptimizer()
    T_pose, pst = po.calc_fast_motion_only_matched(gm, cams[0][:4], T_track, True, 2.0, 15)
    dm, ba = svs.DeviceMap(), svs.BundleAdjuster()
    dm.set(m["poses"], m["point_anchor"], m["xyz_anchor"], m["vis_ptr"], m["vis_pose"], m["feat_center"], m["feat_level"])
    E = dm.set_problem(ba, win, act, cams[0][:4])
    assert ba.optimize(2)[0] == 2
    dm.absorb(ba)
    mp, mx = dm.get()
    Vm = len(m["poses"])
    ring = np.stack([(np.arange(Vm) + 1) % Vm, (np.arange(Vm) + Vm - 1) % Vm], 1).astype(np.int32)
    dm.set_graph(np.arange(0, 2 * Vm + 1, 2, dtype=np.int32), ring.reshape(-1))
    sel = dm.select_window(int(win[0]), 3, 6)
    newv, _ = dm.add_keyframe(int(win[1]), [0, 0, 0, 1, 0.25, -0.5, 0.125], track_point=[0, 1, 2, 3, 4],
                              track_center=np.full((5, 3), 100.0), track_level=[0, 1, 0, 1, 0])
    new_pose = dm.get()[0][-1]

    with open(tmp_path / "out.bin", "rb") as f:
        cnt = np.fromfile(f, np.int32, 6)
        c_xy0 = np.fromfile(f, np.int32, 2 * cnt[0]).reshape(-1, 2)
        c_xy1 = np.fromfile(f, np.int32, 2 * cnt[1]).reshape(-1, 2)
        c_midx = np.fromfile(f, np.int32, cnt[2])
        c_track, c_pose = np.fromfile(f, np.float64, 7), np.fromfile(f, np.float64, 7)
        c_mp = np.fromfile(f, np.float64, mp.size).reshape(mp.shape)
        c_mx = np.fromfile(f, np.float64, mx.size).reshape(mx.shape)
        cnt2 = np.fromfile(f, np.int32, 4)
        c_win, c_inner, c_act = np.fromfile(f, np.int32, cnt2[0]), np.fromfile(f, np.int32, cnt2[0]), np.fromfile(f, np.int32, cnt2[1])
        c_ci, c_cj = np.fromfile(f, np.int32, cnt2[2]), np.fromfile(f, np.int32, cnt2[2])
        c_new_pose = np.fromfile(f, np.float64, 7)
    np.testing.assert_array_equal(c_xy0, xy0); np.testing.assert_array_equal(c_xy1, xy1)
    assert cnt[2] == len(pts) and cnt[3] == int(res["matched"].sum()) and cnt[4] == E and cnt[3] > 50
    np.testing.assert_array_equal(c_midx, np.where(res["matched"] == 1, res["index"], -1))
    np.testing.assert_array_equal(c_track, T_track)
    np.testing.assert_array_equal(c_pose, T_pose)
    np.testing.assert_allclose(c_mp, mp, rtol=1e-9, atol=1e-12)     # FP64 atomics in the Schur scatter
    np.testing.assert_allclose(c_mx, mx, rtol=1e-9, atol=1e-12)
    np.testing.assert_array_equal(c_win, sel["window_vertex"]); np.testing.assert_array_equal(c_inner, sel["inner"])
    np.testing.assert_array_equal(c_act, sel["active_point"])
    np.testing.assert_array_equal(c_ci, sel["c_i"]); np.testing.assert_array_equal(c_cj, sel["c_j"])
    assert cnt2[3] == newv == Vm and len(c_win) >= 6 and len(c_ci) > 0
    np.testing.assert_allclose(c_new_pose, new_pose, rtol=1e-9, atol=1e-12)   # composed from the absorbed pose of win[1]
