"""Seeded tracker test cases shared by CPU and GPU tests."""
import functools
import hashlib

import numpy as np

import orc
from cofusion_b200 import synth


def scaled_K(W):
    s = W / 640.0
    fx, fy, cx, cy = synth.K_DEFAULT
    return (fx * s, fy * s, cx * s, cy * s)


@functools.lru_cache(maxsize=8)
def room_pair(W=640, H=480, noise=True, frame=3, holes=True):
    """Two consecutive room frames + the 'model prediction' made from the first one."""
    K = scaled_K(W)
    seq = list(synth.room_sequence(frame + 2, W, H, K, noise=noise, seed=1234))
    (_, rgb0, d0, T0, _), (_, rgb1, d1, T1, _) = seq[frame], seq[frame + 1]
    if holes:  # invalid-depth blocks exercise the NaN paths
        d1 = d1.copy()
        d1[H // 4:H // 4 + H // 10, W // 3:W // 3 + W // 8] = 0
        d0 = d0.copy()
        d0[H // 2:H // 2 + H // 12, W // 5:W // 5 + W // 9] = 0
    v4, n4, img = synth.prediction_from_depth(d0, rgb0, K)
    return dict(W=W, H=H, K=K, rgb0=rgb0, d0=d0, T0=T0.astype(np.float32), rgb1=rgb1, d1=d1,
                T1=T1.astype(np.float32), v4=v4, n4=n4, img=img)


def oracle_odometry(case, cutoff=20.0, maxD=5.0):
    """OrcOdometry initialised like CoFusion::processFrame does before tracking."""
    od = orc.OrcOdometry(case["W"], case["H"], case["K"])
    od.init_first_rgb(case["rgb0"])
    od.init_model(case["v4"], case["n4"], case["img"], case["T0"])
    df = orc.bilateral(case["d1"], maxD)
    od.init_frame(df, case["rgb1"], cutoff)
    return od, df


def level_K(K, level):
    d = np.float32(1 << level)
    return tuple(np.float32(k) / d for k in K)


def warp_for(K, T_rel):
    """krkinv / kt as RGBDOdometry.cpp:348-358 for resultRt = T_rel (4x4 f64)."""
    fx, fy, cx, cy = [float(k) for k in K]
    Km = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], dtype=np.float64)
    Rt = np.linalg.inv(T_rel)
    krk = Km @ Rt[:3, :3] @ np.linalg.inv(Km)
    kt = Km @ Rt[:3, 3]
    return krk.astype(np.float32), kt.astype(np.float32)


def relerr(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def nan_equal(a, b, tol=0.0, ref_plane_rows=None):
    """compare planar maps: NaN pattern of the x plane must agree; valid entries within tol"""
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return False, "NaN pattern differs (%d vs %d)" % (na.sum(), nb.sum())
    m = ~na
    if tol == 0.0:
        ok = np.array_equal(a[m], b[m])
        return ok, "max abs diff %g" % (np.abs(a[m] - b[m]).max() if m.any() else 0)
    d = np.abs(a[m] - b[m]).max() if m.any() else 0.0
    return d <= tol, "max abs diff %g" % d


def digest(a):
    """SHA-256 of an array's bytes, every NaN replaced by one canonical NaN (equal_nan semantics)"""
    a = np.ascontiguousarray(a).copy()
    if a.dtype.kind == "f":
        a[np.isnan(a)] = np.nan
    return hashlib.sha256(a.tobytes()).hexdigest()


def nan_digest(a):
    """SHA-256 of an array's NaN pattern"""
    return hashlib.sha256(np.packbits(np.isnan(a)).tobytes()).hexdigest()


def case_digest(case):
    """fingerprint of the inputs of a room_pair case"""
    h = hashlib.sha256()
    for k in ("d0", "rgb0", "T0", "d1", "rgb1", "v4", "n4", "img"):
        h.update(np.ascontiguousarray(case[k]).tobytes())
    return h.hexdigest()
