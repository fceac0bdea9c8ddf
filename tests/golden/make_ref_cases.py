"""Generates tests/golden/tracker_ref_cases_sm100a.npz on a B200:

    make -C oracle ref          (compiles the reference's own CUDA kernels into oracle/_ref/libcfref.so)
    python tests/golden/make_ref_cases.py [OUT.npz]

Outputs of the REFERENCE's kernels for the inputs of the room_pair cases of tests/test_tracker_gpu.py
(640x480, 160x120, 72x52), so that the GPU tests compare the CUDA path against the reference without the
reference being present.  Images are stored compactly:
  - exact comparisons: SHA-256 of the output (scenes.digest);
  - float images: SHA-256 of the NaN pattern of the first plane, the values of every plane at up to
    N_SAMPLE seeded valid pixels, and the per-plane maximum |value| the tolerances scale with;
  - gradient images: the pixels where the reference differs from the oracle (usually none).
Small outputs (normal equations, residuals, counts, poses) are stored whole."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import orc  # noqa: E402
import scenes  # noqa: E402

CASES = ((640, 480), (160, 120), (72, 52))
N_SAMPLE = 1024
ANGLE = float(np.sin(np.deg2rad(20.0)))


def case_key(W, H):
    return "c%dx%d_" % (W, H)


def sampled(out, key, x, planes, seed):
    """first-plane NaN digest + values at seeded valid pixels of every plane + per-plane max |value|"""
    h = x.shape[0] // planes
    valid = ~np.isnan(x[:h])
    pos = np.flatnonzero(valid)
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(pos, min(N_SAMPLE, pos.size), replace=False)).astype(np.int64)
    out[key + "_nan"] = np.array(scenes.nan_digest(x[:h]))
    out[key + "_idx"] = idx.astype(np.int32)
    out[key + "_val"] = np.stack([x[k * h:(k + 1) * h].reshape(-1)[idx] for k in range(planes)]).astype(np.float32)
    out[key + "_absmax"] = np.array([np.abs(x[k * h:(k + 1) * h][valid]).max() for k in range(planes)], np.float32)


def patch(out, key, ref_img, orc_img):
    """pixels where the reference differs from the oracle"""
    idx = np.flatnonzero(ref_img != orc_img)
    out[key + "_idx"] = idx.astype(np.int32)
    out[key + "_val"] = ref_img.reshape(-1)[idx]


def make_case(out, W, H, ref, gu, step_inputs):
    case = scenes.room_pair(W, H)
    p = case_key(W, H)
    K = case["K"]
    out[p + "inputs"] = np.array(scenes.case_digest(case))
    seed = W * 100003 + H
    # image preparation, as test_image_preparation_matches_reference_kernels computes it
    df = orc.bilateral(case["d1"], 5.0)
    sampled(out, p + "pyr_f", orc.pyr_down_f(df, ref), 1, seed + 1)
    g = orc.rgb_to_intensity(case["rgb1"])
    out[p + "pyr_u8"] = np.array(scenes.digest(orc.pyr_down_u8(g, ref)))
    dx_r, dy_r = orc.derivative_images(g, ref)
    dx_o, dy_o = orc.derivative_images(g)
    patch(out, p + "dx", dx_r, dx_o)
    patch(out, p + "dy", dy_r, dy_o)
    sampled(out, p + "vmap", orc.create_vmap(df, K, 20.0, ref), 3, seed + 2)
    sampled(out, p + "nmap", orc.create_nmap(gu.create_vmap(df, K, 20.0), ref), 3, seed + 3)
    cv_r, cn_r = orc.copy_maps(case["v4"], case["n4"], ref)
    out[p + "copy_v"], out[p + "copy_n"] = np.array(scenes.digest(cv_r)), np.array(scenes.digest(cn_r))
    sampled(out, p + "resize_v", orc.resize_map(cv_r, False, ref), 3, seed + 4)
    out[p + "v2d"] = np.array(scenes.digest(orc.vertices_to_depth(case["v4"], 6.0, ref)))
    # reduction steps, as test_reduction_steps_match_oracle_and_reference computes them
    for level in range(3):
        if W < 160 and level > 0:
            continue
        q = p + "L%d_" % level
        od, Kl, v, dx, dy, cloud, T0, T = step_inputs(case, level)
        Rpi = np.linalg.inv(T0[:3, :3]).astype(np.float32)
        args = (T[:3, :3], T[:3, 3], v[0], v[1], Rpi, T0[:3, 3], Kl, v[2], v[3], 0.10, ANGLE)
        out[q + "icp_A"], out[q + "icp_b"], out[q + "icp_res"], _ = orc.icp_step(*args, lib=ref)
        krk, kt = scenes.warp_for(Kl, np.linalg.inv(T) @ T0)
        minScale = float((5, 3, 1)[level]) ** 2 / 0.125 ** 2
        c_o, _, n_o = orc.rgb_residual(minScale, dx, dy, v[4], v[5], v[6], v[7], 0.07, kt, krk)
        _, s_r, n_r = orc.rgb_residual(minScale, dx, dy, v[4], v[5], v[6], v[7], 0.07, kt, krk, lib=ref)
        out[q + "res_sigma"], out[q + "res_count"] = np.int64(s_r), np.int64(n_r)
        out[q + "rgb_A"], out[q + "rgb_b"] = orc.rgb_step(c_o, float(n_o), cloud, Kl, dx, dy, 0.125, lib=ref)
    if W < 160:
        return
    # SO(3) pre-alignment step, as test_so3_step_matches_oracle_and_reference computes it
    od, _ = scenes.oracle_odometry(case)
    last, nxt = od.view(10, 2), od.view(7, 2)
    fx, fy, cx, cy = [float(k) for k in scenes.level_K(K, 2)]
    Km = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]])
    R = scenes.synth.rot_y(0.01) @ scenes.synth.rot_x(0.004)
    out[p + "so3_A"], out[p + "so3_b"], out[p + "so3_res"] = orc.so3_step(
        last, nxt, Km @ R @ np.linalg.inv(Km), np.linalg.inv(Km), Km @ R, lib=ref)
    # the whole tracker loop through the reference kernels
    oo, _ = scenes.oracle_odometry(case)
    out[p + "track_pose"], _, _, _ = oo.track(case["T0"], use_ref=True)


def main():
    import gpu_util as gu
    from test_tracker_gpu import _step_inputs
    ref = orc.ref()
    assert ref is not None and ref.ref_device_ok(), "needs oracle/_ref/libcfref.so and a GPU"
    out = {}
    for W, H in CASES:
        make_case(out, W, H, ref, gu, _step_inputs)
        print("case %dx%d inputs %s" % (W, H, out[case_key(W, H) + "inputs"]))
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "tracker_ref_cases_sm100a.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
