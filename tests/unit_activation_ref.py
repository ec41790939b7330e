"""NumPy restatement of the sampled-point rules of unit activation (ScalableTSDFVolume, SURVEY.md A.3 step 7) and of the
clip count, evaluated in float64 in the kernels' order of operations (no FMA), so that it agrees with `unit_mark_kernel` and
`orc_scalable_integrate` bit for bit:
  * every stride-th pixel (rows and columns 0, s, 2s, ... < H, W) with depth p > 0 is back-projected,
    x = ((j - cx) * z) / fx, y = ((i - cy) * z) / fy, z = p, and taken to the world with the cofactor inverse of the extrinsic;
  * a point whose world coordinate is not finite activates nothing and counts as outside the box;
  * otherwise the units floor((w - trunc) / unit_len) .. floor((w + trunc) / unit_len) per axis that lie in the box are
    activated; the point is outside when none does, partly outside when some of its range is cut.
Dense mode (the clip check without units) compares w -+ trunc with the box [origin, origin + n * vl) per axis: outside
when w + trunc < origin or w - trunc >= the far face on some axis.  Those comparisons are false for NaN, so a point with a
NaN coordinate (and no infinite one) counts as neither outside nor partly outside there."""
import numpy as np

import oracle

CLAMP = float(2 ** 40)


def cam_to_world(E):
    """camera -> world 3 x 4 rows of the cofactor inverse (what the kernel and the oracle use)"""
    from oracle.o3d import _ptr, lib
    E = np.ascontiguousarray(E, dtype=np.float64)
    M = np.zeros(16)
    lib().orc_invert4x4(_ptr(E), _ptr(M))
    return M.reshape(4, 4)[:3]


def sampled_world_points(depth, K, E, stride):
    """-> (world [n, 3] f64, finite [n] bool) of the sampled pixels with depth > 0, row-major"""
    d = np.asarray(depth, np.float32)
    H, W = d.shape
    ii, jj = np.meshgrid(np.arange(0, H, stride), np.arange(0, W, stride), indexing="ij")
    p = d[ii, jj]
    keep = p > 0
    i, j, z = ii[keep].astype(np.float64), jj[keep].astype(np.float64), p[keep].astype(np.float64)
    fx, fy, cx, cy = (float(k) for k in K)
    M = cam_to_world(E)
    with np.errstate(invalid="ignore", over="ignore"):
        x = ((j - cx) * z) / fx
        y = ((i - cy) * z) / fy
        w = np.stack([((M[r, 0] * x + M[r, 1] * y) + M[r, 2] * z) + M[r, 3] for r in range(3)], axis=1)
    return w, np.isfinite(w).all(axis=1)


def unit_ranges(w, finite, trunc, unit_len, u0):
    """-> (lo, hi) int64 [n, 3] of the units relative to u0; rows of non-finite points are meaningless"""
    with np.errstate(invalid="ignore"):
        ww = np.where(finite[:, None], w, 0.0)
        lo = np.clip(np.floor((ww - trunc) / unit_len), -CLAMP, CLAMP).astype(np.int64) - np.asarray(u0, np.int64)
        hi = np.clip(np.floor((ww + trunc) / unit_len), -CLAMP, CLAMP).astype(np.int64) - np.asarray(u0, np.int64)
    return lo, hi


def unit_activation(depth, K, E, dims, vl, trunc, origin, unit_res, stride):
    """-> dict(touched [nux, nuy, nuz] bool, points, outside, partly_outside) of one frame in unit mode"""
    nu = np.asarray(dims, np.int64) // unit_res
    ul = float(vl) * unit_res
    u0 = np.rint(np.asarray(origin, np.float64) / ul).astype(np.int64)
    w, finite = sampled_world_points(depth, K, E, stride)
    lo, hi = unit_ranges(w, finite, float(trunc), ul, u0)
    clo, chi = np.maximum(lo, 0), np.minimum(hi, nu - 1)
    empty = ~finite | (clo > chi).any(axis=1)
    part = ~empty & ((lo < 0) | (hi > nu - 1)).any(axis=1)
    touched = np.zeros(tuple(nu), bool)
    for r in np.unique(np.concatenate([clo, chi], axis=1)[~empty], axis=0):
        touched[r[0]:r[3] + 1, r[1]:r[4] + 1, r[2]:r[5] + 1] = True
    return dict(touched=touched, points=int(len(w)), outside=int(empty.sum()), partly_outside=int(part.sum()))


def dense_clip(depth, K, E, dims, vl, trunc, origin, stride):
    """-> dict(points, outside, partly_outside) of one frame in dense mode (dims: the whole grid, z = z_total planes)"""
    w, finite = sampled_world_points(depth, K, E, stride)
    length = np.asarray(dims, np.float64) * float(np.float32(vl))
    with np.errstate(invalid="ignore"):
        wo = w - np.asarray(origin, np.float64)
        empty = ((wo + trunc < 0.0) | (wo - trunc >= length)).any(axis=1)
        part = ~empty & ((wo - trunc < 0.0) | (wo + trunc >= length)).any(axis=1)
    return dict(points=int(len(w)), outside=int(empty.sum()), partly_outside=int(part.sum()))
