"""-m gpu: parity of the CUDA tracker path (through the C ABI) against
   (1) the CPU oracle (oracle/tracker.c) and
   (2) the reference's own CUDA kernels compiled for sm_100a, through their outputs on the same inputs
       (tests/golden/tracker_ref_cases_sm100a.npz, made by tests/golden/make_ref_cases.py).

Tolerances (north_star: 1e-4 relative on float buffers, bit-exact on integer/index work):
  - integer outputs (grey, gradients, u8 pyramids, correspondence flags/counts): bit-exact vs oracle
  - image-prep floats computed without FMA contraction: bit-exact vs oracle
  - normal maps (rsqrtf) and reference-kernel comparisons (--prec-div=false etc.): <= 2e-6 abs
  - reduction sums A, b: <= 1e-4 relative (f32 tree sums vs f64 oracle sums)
  - poses: <= 1e-4 absolute on R and t
"""
import os

import numpy as np
import pytest

import orc
import scenes

pytestmark = pytest.mark.gpu

ANGLE = float(np.sin(np.deg2rad(20.0)))
REF_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tracker_ref_cases_sm100a.npz")


@pytest.fixture(scope="module")
def gu():
    import gpu_util
    return gpu_util


@pytest.fixture(scope="module")
def ref_golden():
    return dict(np.load(REF_GOLDEN))


def _ref_outputs(ref_golden, case):
    """the reference kernels' outputs for this case, keyed by name"""
    p = "c%dx%d_" % (case["W"], case["H"])
    assert str(ref_golden[p + "inputs"]) == scenes.case_digest(case), (
        "room_pair(%d, %d) no longer renders the inputs the stored reference outputs were computed from: "
        "regenerate them with tests/golden/make_ref_cases.py" % (case["W"], case["H"]))
    return {k[len(p):]: v for k, v in ref_golden.items() if k.startswith(p)}


def _check_sampled(r, name, x, planes, tol, scaled=True):
    """planar image x against the reference's: NaN pattern of the first plane, then every plane at the stored
    pixels within tol (times max(1, max |value|) of the reference's plane when scaled)"""
    h = x.shape[0] // planes
    assert scenes.nan_digest(x[:h]) == str(r[name + "_nan"]), "%s: NaN pattern differs from the reference" % name
    idx = r[name + "_idx"]
    for k in range(planes):
        d = np.abs(x[k * h:(k + 1) * h].reshape(-1)[idx] - r[name + "_val"][k]).max()
        lim = tol * (max(1.0, float(r[name + "_absmax"][k])) if scaled else 1.0)
        assert d <= lim, "%s plane %d: max abs diff %g > %g" % (name, k, d, lim)


@pytest.fixture(scope="module", params=[(640, 480), (160, 120), (72, 52)], ids=["640x480", "160x120", "72x52"])
def case(request):
    W, H = request.param
    return scenes.room_pair(W, H)


def test_image_preparation_matches_oracle(gu, case):
    K, W, H = case["K"], case["W"], case["H"]
    d1, rgb1 = case["d1"], case["rgb1"]
    # a1 bilateral: bit exact (deterministic exp, no FMA)
    df_o = orc.bilateral(d1, 5.0)
    df_g = gu.bilateral(d1, 5.0)
    assert np.array_equal(df_o, df_g), np.abs(df_o - df_g).max()
    # a2 depth pyramid: bit exact
    p1_o, p1_g = orc.pyr_down_f(df_o), gu.pyr_down_f(df_o)
    assert np.array_equal(p1_o, p1_g, equal_nan=True)
    # a5 grey + u8 pyramid: bit exact
    g_o, g_g = orc.rgb_to_intensity(rgb1), gu.rgb_to_intensity(rgb1)
    assert np.array_equal(g_o, g_g)
    assert np.array_equal(orc.pyr_down_u8(g_o), gu.pyr_down_u8(g_o))
    # a6 gradients: bit exact
    dx_o, dy_o = orc.derivative_images(g_o)
    dx_g, dy_g = gu.derivative_images(g_o)
    assert np.array_equal(dx_o, dx_g) and np.array_equal(dy_o, dy_g)
    # a4 vertex map: bit exact; normal map: rsqrtf -> tolerance
    v_o, v_g = orc.create_vmap(df_o, K, 20.0), gu.create_vmap(df_o, K, 20.0)
    ok, msg = scenes.nan_equal(v_g, v_o)
    assert ok, msg
    n_o, n_g = orc.create_nmap(v_o), gu.create_nmap(v_o)
    ok, msg = scenes.nan_equal(n_g, n_o, tol=2e-6)
    assert ok, msg
    # a3 copy / resize / transform
    cv_o, cn_o = orc.copy_maps(case["v4"], case["n4"])
    cv_g, cn_g = gu.copy_maps(case["v4"], case["n4"])
    assert scenes.nan_equal(cv_g, cv_o)[0] and scenes.nan_equal(cn_g, cn_o)[0]
    assert scenes.nan_equal(gu.resize_map(cv_o, False), orc.resize_map(cv_o, False))[0]
    ok, msg = scenes.nan_equal(gu.resize_map(cn_o, True), orc.resize_map(cn_o, True), tol=2e-6)
    assert ok, msg
    R, t = case["T0"][:3, :3], case["T0"][:3, 3]
    tv_o, tn_o = orc.transform_maps(cv_o, cn_o, R, t)
    tv_g, tn_g = gu.transform_maps(cv_o, cn_o, R, t)
    assert scenes.nan_equal(tv_g, tv_o, tol=2e-6)[0] and scenes.nan_equal(tn_g, tn_o, tol=2e-6)[0]
    # a5 depth from vertices, a6 cloud
    assert np.array_equal(orc.vertices_to_depth(case["v4"], 6.0), gu.vertices_to_depth(case["v4"], 6.0),
                          equal_nan=True)
    vd = orc.vertices_to_depth(case["v4"], 6.0)
    assert np.array_equal(orc.project_cloud(vd, K), gu.project_cloud(vd, K), equal_nan=True)


def test_image_preparation_matches_reference_kernels(gu, case, ref_golden):
    r = _ref_outputs(ref_golden, case)
    K = case["K"]
    df = orc.bilateral(case["d1"], 5.0)
    # the reference build contracts to FMA and uses approximate division: last-ulp differences
    _check_sampled(r, "pyr_f", gu.pyr_down_f(df), 1, 2e-6)
    g = orc.rgb_to_intensity(case["rgb1"])
    assert scenes.digest(gu.pyr_down_u8(g)) == str(r["pyr_u8"])
    # the reference's gradients are stored as the pixels where they differ from the oracle's
    dx_r, dy_r = orc.derivative_images(g)
    dx_r.reshape(-1)[r["dx_idx"]] = r["dx_val"]
    dy_r.reshape(-1)[r["dy_idx"]] = r["dy_val"]
    dx_g, dy_g = gu.derivative_images(g)
    # the reference build contracts a*b+c into FMA: a 1-LSB flip at an exact .0 boundary is possible
    assert np.abs(dx_r.astype(int) - dx_g.astype(int)).max() <= 1 and (dx_r != dx_g).mean() < 1e-3
    assert np.abs(dy_r.astype(int) - dy_g.astype(int)).max() <= 1 and (dy_r != dy_g).mean() < 1e-3
    v_g = gu.create_vmap(df, K, 20.0)
    _check_sampled(r, "vmap", v_g, 3, 2e-6)
    _check_sampled(r, "nmap", gu.create_nmap(v_g), 3, 5e-6, scaled=False)
    cv_g, cn_g = gu.copy_maps(case["v4"], case["n4"])
    assert scenes.digest(cv_g) == str(r["copy_v"]) and scenes.digest(cn_g) == str(r["copy_n"])
    _check_sampled(r, "resize_v", gu.resize_map(cv_g, False), 3, 2e-6)
    assert scenes.digest(gu.vertices_to_depth(case["v4"], 6.0)) == str(r["v2d"])


def _step_inputs(case, level, perturb=True):
    """pyramid data of one level from the oracle + a slightly wrong pose (so that b != 0)"""
    od, df = scenes.oracle_odometry(case)
    Kl = scenes.level_K(case["K"], level)
    views = {k: od.view(k, level) for k in range(11)}
    dx, dy = orc.derivative_images(views[7])
    cloud = orc.project_cloud(views[4], Kl)
    T0 = case["T0"].astype(np.float64)
    T = T0.copy()
    if perturb:
        T = T0 @ np.array(scenes.synth.make_pose(scenes.synth.rot_y(0.004) @ scenes.synth.rot_x(-0.002),
                                                 [0.003, -0.002, 0.004]))
    return od, Kl, views, dx, dy, cloud, T0, T


@pytest.mark.parametrize("level", [0, 1, 2])
def test_reduction_steps_match_oracle_and_reference(gu, case, level, ref_golden):
    if case["W"] < 160 and level > 0:
        pytest.skip("tiny case: level 0 only")
    od, Kl, v, dx, dy, cloud, T0, T = _step_inputs(case, level)
    r = _ref_outputs(ref_golden, case)
    q = "L%d_" % level
    Rpi = np.linalg.inv(T0[:3, :3]).astype(np.float32)
    args = (T[:3, :3], T[:3, 3], v[0], v[1], Rpi, T0[:3, 3], Kl, v[2], v[3], 0.10, ANGLE)
    # ---- ICP
    A_o, b_o, r_o, e_o = orc.icp_step(*args, want_error=True)
    A_g, b_g, r_g, e_g = gu.icp_step(*args, want_error=True)
    assert r_o[1] > 0.05 * v[0].shape[1] * (v[0].shape[0] // 3), "scene should have inliers"
    assert abs(r_g[1] - r_o[1]) <= max(2, 2e-4 * r_o[1]), (r_g, r_o)
    assert scenes.relerr(A_g, A_o) < 1e-4 and scenes.relerr(b_g, b_o) < 1e-4
    assert abs(r_g[0] - r_o[0]) <= 1e-4 * r_o[0]
    assert np.allclose(A_g, A_g.T)
    diff = np.abs(e_g - e_o)
    assert (diff > 1e-5).mean() < 1e-3  # borderline association flips only
    A_r, b_r, r_r = r[q + "icp_A"], r[q + "icp_b"], r[q + "icp_res"]
    assert abs(r_g[1] - r_r[1]) <= max(2, 2e-4 * r_r[1])
    assert scenes.relerr(A_g, A_r) < 1e-4 and scenes.relerr(b_g, b_r) < 1e-4
    # ---- RGB residual
    T_rel = np.linalg.inv(T) @ T0  # any small relative motion
    krk, kt = scenes.warp_for(Kl, T_rel)
    minScale = float((5, 3, 1)[level]) ** 2 / 0.125 ** 2
    c_o, s_o, n_o = orc.rgb_residual(minScale, dx, dy, v[4], v[5], v[6], v[7], 0.07, kt, krk)
    c_g, s_g, n_g = gu.rgb_residual(minScale, dx, dy, v[4], v[5], v[6], v[7], 0.07, kt, krk)
    assert n_o > 50
    vo, zxo, zyo, do = orc.corres_valid(c_o)
    vg, zxg, zyg, dg = orc.corres_valid(c_g)
    mism = (vo != vg).sum()
    assert mism <= max(2, 1e-3 * n_o), "valid-flag mismatches %d of %d" % (mism, n_o)
    both = vo & vg
    assert ((zxo[both] != zxg[both]) | (zyo[both] != zyg[both])).mean() < 1e-3
    assert abs(n_g - n_o) <= max(2, 1e-3 * n_o) and abs(s_g - s_o) <= max(2000, 2e-3 * abs(s_o))
    s_r, n_r = int(r[q + "res_sigma"]), int(r[q + "res_count"])
    assert abs(n_g - n_r) <= max(2, 1e-3 * n_r) and abs(s_g - s_r) <= max(2000, 2e-3 * abs(s_r))
    # ---- RGB step on identical correspondences
    sigma = float(n_o)
    A_o, b_o = orc.rgb_step(c_o, sigma, cloud, Kl, dx, dy, 0.125)
    A_g, b_g = gu.rgb_step(c_o, sigma, cloud, Kl, dx, dy, 0.125)
    assert scenes.relerr(A_g, A_o) < 1e-4 and scenes.relerr(b_g, b_o) < 1e-4
    A_r, b_r = r[q + "rgb_A"], r[q + "rgb_b"]
    assert scenes.relerr(A_g, A_r) < 1e-4 and scenes.relerr(b_g, b_r) < 1e-4
    # rgbOnly signalling (sigma == -1 -> unit weights)
    A_o1, b_o1 = orc.rgb_step(c_o, -1.0, cloud, Kl, dx, dy, 0.125)
    A_g1, b_g1 = gu.rgb_step(c_o, -1.0, cloud, Kl, dx, dy, 0.125)
    assert scenes.relerr(A_g1, A_o1) < 1e-4 and scenes.relerr(b_g1, b_o1) < 1e-4


def test_so3_step_matches_oracle_and_reference(gu, case, ref_golden):
    if case["W"] < 160:
        pytest.skip("so3 runs on level 2")
    od, df = scenes.oracle_odometry(case)
    L = 2
    last, nxt = od.view(10, L), od.view(7, L)
    fx, fy, cx, cy = [float(k) for k in scenes.level_K(case["K"], L)]
    Km = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]])
    R = scenes.synth.rot_y(0.01) @ scenes.synth.rot_x(0.004)
    H_, Kinv, KR = Km @ R @ np.linalg.inv(Km), np.linalg.inv(Km), Km @ R
    A_o, b_o, r_o = orc.so3_step(last, nxt, H_, Kinv, KR)
    A_g, b_g, r_g = gu.so3_step(last, nxt, H_, Kinv, KR)
    assert r_o[1] > 100 and r_g[1] == r_o[1]
    assert scenes.relerr(A_g, A_o) < 1e-4 and scenes.relerr(b_g, b_o) < 1e-4 and abs(r_g[0] - r_o[0]) <= 1e-4 * r_o[0]
    r = _ref_outputs(ref_golden, case)
    A_r, b_r, r_r = r["so3_A"], r["so3_b"], r["so3_res"]
    assert r_g[1] == r_r[1] and scenes.relerr(A_g, A_r) < 1e-4 and scenes.relerr(b_g, b_r) < 1e-4


def _cuda_odometry(gu, case, cutoff=20.0, maxD=5.0):
    import cofusion_b200 as cfb
    od = cfb.Odometry(case["W"], case["H"], case["K"])
    od.init_first_rgb(gu.dev(case["rgb0"]))
    od.init_icp_model(gu.dev(case["v4"]), gu.dev(case["n4"]), cutoff, case["T0"])
    od.init_rgb_model(gu.dev(case["img"]))
    df = gu.bilateral(case["d1"], maxD)
    pyr = [gu.dev(df)]
    for _ in range(2):
        pyr.append(gu.dev(gu.pyr_down_f(gu.host(pyr[-1]))))
    od.init_icp(pyr, cutoff)
    od.init_rgb(gu.dev(case["rgb1"]))
    return od


@pytest.mark.parametrize("variant", ["persistent", "host_loop"])
def test_full_tracking_matches_oracle(gu, case, variant, ref_golden):
    host_loop = variant == "host_loop"
    if case["W"] < 160:
        pytest.skip("pyramid needs >= 160x120")
    oo, _ = scenes.oracle_odometry(case)
    # pyramids built by the CUDA init path equal the oracle's
    co = _cuda_odometry(gu, case)
    for which, tol in ((0, 0.0), (2, 3e-6), (4, 0.0), (6, 0.0), (7, 0.0), (10, 0.0)):
        for lvl in range(3):
            a, b = co.view(which, lvl), oo.view(which, lvl)
            if a.dtype == np.float32:
                ok, msg = scenes.nan_equal(a, b, tol=tol)
                assert ok, (which, lvl, msg)
            else:
                assert np.array_equal(a, b), (which, lvl)
    p_o, st_o, err_o, _ = oo.track(case["T0"], want_error=True)
    import torch
    err_g = torch.zeros((case["H"], case["W"]), dtype=torch.float32, device="cuda")
    p_g, st_g = co.track(case["T0"], error_map=err_g, force_host_loop=host_loop)
    assert np.abs(p_g - p_o).max() < 1e-4, (p_g, p_o)
    # tracking actually moved the pose towards ground truth
    assert np.abs(p_g - case["T1"]).max() < 0.5 * np.abs(case["T0"] - case["T1"]).max() + 2e-3
    assert st_g.so3_iterations == st_o.so3_iterations
    assert abs(st_g.lastICPCount - st_o.lastICPCount) <= max(3, 1e-3 * st_o.lastICPCount)
    assert abs(st_g.lastRGBCount - st_o.lastRGBCount) <= max(3, 2e-3 * st_o.lastRGBCount)
    assert abs(st_g.lastICPError - st_o.lastICPError) <= 1e-3 * st_o.lastICPError + 1e-9
    assert scenes.relerr(np.array(st_g.lastA), np.array(st_o.lastA)) < 2e-3
    eg = err_g.cpu().numpy()
    assert (np.abs(eg - err_o) > 1e-4).mean() < 2e-3
    # reference kernels driven through the same loop agree as well
    p_r = _ref_outputs(ref_golden, case)["track_pose"]
    assert np.abs(p_g - p_r).max() < 1e-4, (p_g, p_r)


def test_tracking_is_deterministic_and_flag_variants_agree(gu):
    case = scenes.room_pair(160, 120)
    outs = []
    for _ in range(2):
        co = _cuda_odometry(gu, case)
        p, st = co.track(case["T0"])
        outs.append((p.copy(), np.array(st.lastA)))
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    # non-default flags agree with the oracle: rgb_only and icp_weight=100 run the generic host loop, so3=False,
    # fast_odom=True and pyramid=False the persistent kernel
    for kw in (dict(rgb_only=True), dict(icp_weight=100.0), dict(so3=False), dict(fast_odom=True),
               dict(pyramid=False)):
        oo, _ = scenes.oracle_odometry(case)
        p_o, _, _, _ = oo.track(case["T0"], **kw)
        co = _cuda_odometry(gu, case)
        p_g, _ = co.track(case["T0"], **kw)
        assert np.abs(p_g - p_o).max() < 2e-4, (kw, p_g, p_o)


def test_edge_cases_empty_depth_and_lost_tracking(gu):
    case = dict(scenes.room_pair(160, 120))
    case["d1"] = np.zeros_like(case["d1"])  # no valid depth at all
    co = _cuda_odometry(gu, case)
    p, st = co.track(case["T0"])
    oo, _ = scenes.oracle_odometry(case)
    p_o, _, _, _ = oo.track(case["T0"])
    # no inlier -> zero normal equations -> zero update: the pose is the SO(3) pre-alignment alone; its
    # stopping rule compares float sums (RGBDOdometry.cpp:285-292), so allow one iteration of difference
    assert st.lastICPCount == 0 and np.isfinite(p).all() and np.abs(p - p_o).max() < 2e-3
    # photometric sanity reset: a pose jump > 0.3 m is rejected (RGBDOdometry.cpp:464-467)
    case = scenes.room_pair(160, 120)
    oo, _ = scenes.oracle_odometry(case)
    far = case["T0"].copy()
    p_o, _, _, _ = oo.track(far)
    co = _cuda_odometry(gu, case)
    p_g, _ = co.track(far)
    assert np.abs(p_g - p_o).max() < 1e-4
