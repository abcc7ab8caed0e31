"""NumPy restatement of fbus_marker_project and fbus_synth_corners (include/fbus_ekf.h), used by the corner-synthesis tests.

  philox4x32_10, normal2   the counter-based generator of fbus_kernels.cuh (Philox4x32-10, Box-Muller on two 53-bit uniforms)
  project_poses            the forward model: marker poses [7][n] -> stereo corners [16][n] and valid [n], in float64, built on
                           synth.forward_project (underwater) and the pinhole geometry of synth.marker_corners_inair (in air)
  synth_corners            the per-filter corner streams of frames [w0, w1) from the noise-free corners of each (frame, slot)
"""
from __future__ import annotations

import numpy as np

from fbus_ekf_b200 import synth

MASK = np.uint64(0xFFFFFFFF)
CORNER_STREAM0, CORNER_STREAM_STRIDE = 64, 32


def _u32(x):
    return np.asarray(x, dtype=np.uint64) & MASK


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counter (c0, c1, c2, c3) and key (k0, k1), element-wise over arrays -> four uint64 arrays < 2^32"""
    c0, c1, c2, c3, k0, k1 = (_u32(v) for v in (c0, c1, c2, c3, k0, k1))
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(c0, c1, c2, c3, k0, k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0 = (k0 + np.uint64(0x9E3779B9)) & MASK
        k1 = (k1 + np.uint64(0xBB67AE85)) & MASK
    return c0, c1, c2, c3


def _counter(seed, filt, idx, stream):
    filt = np.asarray(filt, dtype=np.uint64)
    seed = np.uint64(seed)
    return philox4x32_10(filt & MASK, filt >> np.uint64(32), idx, stream, seed & MASK, seed >> np.uint64(32))


def uniform53(hi, lo):
    """[0, 1) from the top 53 bits of (hi << 32) | lo"""
    return (((hi << np.uint64(32)) | lo) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def normal2(seed, filt, idx, stream):
    """two N(0,1) per counter, as normal2 of fbus_kernels.cuh: u1 in (0,1], u2 in [0,1), Box-Muller"""
    r = _counter(seed, filt, idx, stream)
    a = (r[0] << np.uint64(32)) | r[1]
    bb = (r[2] << np.uint64(32)) | r[3]
    u1 = ((a >> np.uint64(11)).astype(np.float64) + 1.0) * (1.0 / 9007199254740992.0)
    u2 = (bb >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    rad = np.sqrt(-2.0 * np.log(u1))
    return rad * np.cos(np.pi * (2.0 * u2)), rad * np.sin(np.pi * (2.0 * u2))


def project_poses(cfg, pose, underwater: bool = True):
    """poses float64 [7][n] -> (corners float64 [16][n], valid int32 [n]); invalid items (a corner at or behind the port) are NaN.
    The arithmetic of synth.board_base_corners (underwater) and synth.marker_corners_inair (in air), item by item."""
    pose = np.asarray(pose, dtype=np.float64)
    n = pose.shape[1]
    p_all = np.ascontiguousarray(pose[0:3].T)
    R_all = np.zeros((n, 3, 3))
    for k in range(n):
        q = pose[3:7, k]
        R_all[k] = synth._q2R(q / np.linalg.norm(q))
    size = cfg.marker_size
    cm = np.array([[0, 0, 0], [size, 0, 0], [size, size, 0], [0, size, 0]], dtype=np.float64)
    flip = np.array([-1.0, -1.0, 1.0])
    out = np.zeros((16, n))
    valid = np.ones(n, dtype=bool)
    if underwater:
        R_RL, P_LR = synth.stereo_extrinsics(cfg)
        Ri = np.linalg.inv(R_RL)
        zmin = cfg.d_air + cfg.d_glass
    else:
        TL = np.array(cfg.tsc_left, dtype=np.float64).reshape(4, 4)
        TR = np.array(cfg.tsc_right, dtype=np.float64).reshape(4, 4)
        Rr = TR[:3, :3] @ TL[:3, :3].T
        t = TL[:3, 3] - Rr @ TR[:3, 3]
        zmin = 0.0
    for i in range(4):
        XL = (p_all + np.einsum("nij,j->ni", R_all, cm[i])) * flip
        XR = (XL - P_LR) @ Ri.T if underwater else XL @ Rr.T + t
        valid &= (XL[:, 2] > zmin) & (XR[:, 2] > zmin)
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            if underwater:
                uvL, uvR = synth.forward_project(cfg, XL), synth.forward_project(cfg, XR)
            else:
                uvL, uvR = XL[:, :2] / XL[:, 2:3], XR[:, :2] / XR[:, 2:3]
        out[2 * i], out[2 * i + 1] = uvL[:, 0], uvL[:, 1]
        out[8 + 2 * i], out[9 + 2 * i] = uvR[:, 0], uvR[:, 1]
    out[:, ~valid] = np.nan
    return out, valid.astype(np.int32)


def synth_corners(base, base_id, B: int, m: int, w0: int, seed: int, filter_offset: int = 0, sigma_corner: float = 0.0,
                  p_drop: float = 0.0, p_outlier: float = 0.0, sigma_outlier: float = 0.0):
    """fbus_synth_corners over frames [w0, w0 + nws / m) from the noise-free corners base [16][nws] of each (frame, slot) and
    base_id [nws] (-1 where the slot is empty or its projection invalid) -> (corners float32 [16][nws * B], ids int32 [nws / m][m][B])"""
    base = np.asarray(base, dtype=np.float64)
    nws = base.shape[1]
    n = nws * B
    i = np.arange(n, dtype=np.uint64)
    ws = i // np.uint64(B)
    b = i % np.uint64(B)
    w = np.uint64(w0) + ws // np.uint64(m)
    st = np.uint64(CORNER_STREAM0) + np.uint64(CORNER_STREAM_STRIDE) * (ws % np.uint64(m))
    gf = np.uint64(filter_offset) + b
    ids = np.asarray(base_id, dtype=np.int32)[ws.astype(np.int64)].copy()
    r = _counter(seed, gf, w, st + np.uint64(8))
    u_drop, u_out = uniform53(r[0], r[1]), uniform53(r[2], r[3])
    live = ids >= 0
    drop = live & (u_drop < p_drop)
    outlier = live & ~drop & (u_out < p_outlier)
    ids[drop] = -1
    wsi = ws.astype(np.int64)
    c = np.zeros((16, n))
    for d in range(8):
        z0, z1 = normal2(seed, gf, w, st + np.uint64(d))
        c[2 * d] = base[2 * d, wsi] + sigma_corner * z0
        c[2 * d + 1] = base[2 * d + 1, wsi] + sigma_corner * z1
    if outlier.any():
        for d in range(8):
            z0, z1 = normal2(seed, gf, w, st + np.uint64(9 + d))
            c[2 * d] = np.where(outlier, c[2 * d] + sigma_outlier * z0, c[2 * d])
            c[2 * d + 1] = np.where(outlier, c[2 * d + 1] + sigma_outlier * z1, c[2 * d + 1])
    c[:, ids < 0] = 0.0
    return np.ascontiguousarray(c.astype(np.float32)), ids.reshape(nws // m, m, B), drop, outlier
