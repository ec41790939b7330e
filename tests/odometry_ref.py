"""ctypes front-end of the odometry's CPU reference, tests/odometry_ref.c (TEST INFRASTRUCTURE, like oracle/).

Compiled on first use with the oracle's flags (gcc, -ffp-contract=off, OpenMP) into the temporary directory, under a
name that carries the source's hash, so nothing is written into the repository tree.  Frames are prepared into the
library's prepared-frame layout, so the GPU's buffer can be compared with `prepare`'s output as is."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "odometry_ref.c")
_CFLAGS = ["-O3", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden", "-Wall", "-Wextra", "-shared"]
_lib = None
PLANES = ("depth", "intensity", "vx", "vy", "vz", "nx", "ny", "nz", "ddx", "ddy", "dix", "diy")
POINT_TO_PLANE, INTENSITY, HYBRID = 0, 1, 2


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src + " ".join(_CFLAGS).encode()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"bslam_odometry_ref_{os.getuid()}_{tag}.so")
        if not os.path.exists(path):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run([cc, *_CFLAGS, "-o", tmp, _SRC, "-lm"], check=True, capture_output=True)
            os.replace(tmp, path)      # atomic: concurrent test processes never load a half-written file
        L = C.CDLL(path)
        p, i, f = C.c_void_p, C.c_int, C.c_float
        L.ref_odom_frame_floats.restype = C.c_int64
        L.ref_odom_frame_floats.argtypes = [i, i, i]
        L.ref_odom_prepare.restype = None
        L.ref_odom_prepare.argtypes = [p, i, p, i, i, i, i, i, p, f, f, f, p]
        L.ref_odom_linearize.restype = None
        L.ref_odom_linearize.argtypes = [p, i, i, i, i, i, i, p, i, f, f, f, p, p]
        L.ref_odom_pixel.restype = i
        L.ref_odom_pixel.argtypes = [p, i, i, i, i, i, i, p, i, f, p, i, i, p, p]
        L.ref_odom_track.restype = i
        L.ref_odom_track.argtypes = [p, i, i, i, i, i, p, i, p, p, p, f, f, f, p, p, p]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _np(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)


class Frames:
    """prepared frames: `data` [F, frame_floats] f32 in the library's layout"""

    def __init__(self, depth, color, K, levels, depth_scale=1000.0, depth_max=3.0, depth_outlier_trunc=0.07):
        d = np.ascontiguousarray(_np(depth))
        if d.ndim == 2:
            d = d[None]
        c = None if color is None else np.ascontiguousarray(_np(color)).reshape(d.shape + (3,))
        if d.dtype not in (np.uint16, np.float32) or (c is not None and c.dtype not in (np.uint8, np.float32)):
            raise ValueError("depth uint16 / float32, colour uint8 / float32")
        self.F, self.H, self.W = d.shape
        self.levels, self.K = levels, np.asarray(K, np.float64).reshape(4)
        self.data = np.empty((self.F, lib().ref_odom_frame_floats(self.H, self.W, levels)), np.float32)
        lib().ref_odom_prepare(_ptr(d), int(d.dtype == np.float32), _ptr(c), int(c is not None and c.dtype == np.float32), self.F, self.H, self.W,
                               levels, _ptr(self.K), depth_scale, depth_max, depth_outlier_trunc, _ptr(self.data))

    def level_shape(self, l):
        return self.H >> l, self.W >> l

    def planes(self, f, l):
        """dict plane name -> [H_l, W_l] view of frame f, level l"""
        off = sum(12 * (self.H >> k) * (self.W >> k) for k in range(l))
        h, w = self.level_shape(l)
        blk = self.data[f, off:off + 12 * h * w].reshape(12, h, w)
        return dict(zip(PLANES, blk))

    def linearize(self, src, tgt, level, T, method, params=(0.07, 0.05, 0.1)):
        out = np.empty(29, np.float64)
        T = np.ascontiguousarray(T, np.float64).reshape(16)
        lib().ref_odom_linearize(_ptr(self.data), src, tgt, self.H, self.W, self.levels, level, _ptr(self.K), method, *params, _ptr(T), _ptr(out))
        return out

    def pixel(self, src, tgt, level, T, method, x, y, trunc=0.07):
        J, r = np.zeros(12, np.float32), np.zeros(2, np.float32)
        T = np.ascontiguousarray(T, np.float64).reshape(16)
        n = lib().ref_odom_pixel(_ptr(self.data), src, tgt, self.H, self.W, self.levels, level, _ptr(self.K), method, trunc, _ptr(T), x, y,
                                 _ptr(J), _ptr(r))
        return n, J.reshape(2, 6)[:n], r[:n]

    def track(self, src, tgt, method, criteria=((10, 1e-6, 1e-6), (5, 1e-6, 1e-6), (3, 1e-6, 1e-6)), init=np.eye(4), params=(0.07, 0.05, 0.1)):
        """criteria: (max_iteration, relative_rmse, relative_fitness) per level, coarsest first (len = levels) ->
        dict(T, rmse, fitness, iters, status)"""
        assert len(criteria) == self.levels
        mi = np.array([c[0] for c in criteria], np.int32)
        rr = np.array([c[1] for c in criteria], np.float64)
        rf = np.array([c[2] for c in criteria], np.float64)
        T = np.ascontiguousarray(init, np.float64).reshape(16).copy()
        out, iters = np.empty(2, np.float64), np.empty(self.levels, np.int32)
        st = lib().ref_odom_track(_ptr(self.data), src, tgt, self.H, self.W, self.levels, _ptr(self.K), method, _ptr(mi), _ptr(rf), _ptr(rr), *params,
                                  _ptr(T), _ptr(out), _ptr(iters))
        return dict(T=T.reshape(4, 4), rmse=float(out[0]), fitness=float(out[1]), iters=iters, status=int(st))


def level_dims(H, W, levels):
    return [(H >> l, W >> l) for l in range(levels)]


# ------------------------------------------------------------------------------------------------ float64 linearisation
# An independent restatement of a linearisation (the 29 sums of ref_odom_linearize / bslam_odom_linearize): the same
# decisions and formulas evaluated per pixel in float64 with NumPy instead of float32 in C, for checking the mirror's
# Huber terms, projection and rejection rules against arithmetic it does not share.  Only T is rounded to float32 first,
# as the kernel uses it; the prepared maps and the level's fx, fy, cx, cy are float32 in both.
#
# Error bound.  Every J, r and decision quantity q of the float32 code is a chain of at most 16 rounded +, -, x, / (the
# longest: the hybrid depth row of J through vs, invz and d2).  Running error analysis (Higham, Accuracy and Stability
# of Numerical Algorithms, 2nd ed., section 3.3) bounds |fl(q) - q| <= gamma_k |q|_abs with u = 2^-24, where |q|_abs is
# q evaluated with every operand replaced by its magnitude (a - b by |a| + |b|, a / b by |a|_abs / |b| (1 + |b|_abs / |b|)
# to first order).  K_OPS = 24 > 16 absorbs the second-order terms.  The products and sums of the 29 entries are exact or
# float64 in both, so an entry's difference is bounded by the propagated J / r / huber errors of its inliers, plus the
# whole contribution of every pixel one of whose decisions (vs_z > 0, the projection's range tests, roundf's half-way
# point, the truncation test) lies within the bound of its threshold: those may land on either side in float32.  The
# Huber terms need no such margin: huber and huber' are continuous at |r| = delta, so a branch flip moves them by at most
# the error of r.
U32 = 2.0 ** -24
K_OPS = 24
_GAMMA = K_OPS * U32


def _c(x):
    """exact operand: (value, magnitude)"""
    x = np.asarray(x, np.float64)
    return x, np.abs(x)


def _add(a, b):
    return a[0] + b[0], a[1] + b[1]


def _sub(a, b):
    return a[0] - b[0], a[1] + b[1]


def _mul(a, b):
    return a[0] * b[0], a[1] * b[1]


def _div(a, b):
    ab = np.abs(b[0])
    return a[0] / b[0], a[1] / ab * (1.0 + b[1] / ab)


def _neg(a):
    return -a[0], a[1]


def _round_away(x):
    """roundf: half-way cases away from zero"""
    return np.sign(x) * np.floor(np.abs(x) + 0.5)


def _huber(r, d):
    a = np.abs(r)
    return np.where(a <= d, 0.5 * r * r, d * (a - 0.5 * d))


def _huber_deriv(r, d):
    return np.where(np.abs(r) <= d, r, np.where(r > 0, d, -d))


def _terms(fr, src, tgt, level, vs, u, w, method, trunc, sel=slice(None)):
    """residuals and Jacobians of source pixels `sel` projected to target pixels (u, w), in float64 with magnitudes:
    -> ok (accepted under these float64 decisions), amb (the truncation test is within its error bound), nres,
    J [n,2,6], eJ, r [n,2], er (error bounds)"""
    Hl, Wl = fr.level_shape(level)
    s, t = fr.planes(src, level), fr.planes(tgt, level)
    fx, fy = (np.float64(np.float32(fr.K[k]) * np.float32(1.0 / (1 << level))) for k in (0, 1))
    inside = (u >= 0) & (u < Wl) & (w >= 0) & (w < Hl)
    j = np.where(inside, np.clip(w, 0, Hl - 1) * Wl + np.clip(u, 0, Wl - 1), 0).astype(np.int64)
    g = {k: v.reshape(-1)[j].astype(np.float64) for k, v in t.items()}
    n = u.shape[0]
    J, mJ, r, mr = np.zeros((n, 2, 6)), np.zeros((n, 2, 6)), np.zeros((n, 2)), np.zeros((n, 2))
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        if method == POINT_TO_PLANE:
            vt = [_c(g[k]) for k in ("vx", "vy", "vz")]
            nt = [_c(g[k]) for k in ("nx", "ny", "nz")]
            ok = inside & ~np.isnan(g["vz"]) & ~np.isnan(g["nx"]) & ~np.isnan(g["ny"]) & ~np.isnan(g["nz"])
            res = _add(_add(_mul(_sub(vs[0], vt[0]), nt[0]), _mul(_sub(vs[1], vt[1]), nt[1])), _mul(_sub(vs[2], vt[2]), nt[2]))
            amb = ok & (np.abs(np.abs(res[0]) - trunc) <= _GAMMA * res[1])
            ok &= ~(np.abs(res[0]) > trunc)
            rows = [_sub(_mul(vs[1], nt[2]), _mul(vs[2], nt[1])), _sub(_mul(vs[2], nt[0]), _mul(vs[0], nt[2])),
                    _sub(_mul(vs[0], nt[1]), _mul(vs[1], nt[0])), nt[0], nt[1], nt[2]]
            for a, q in enumerate(rows):
                J[:, 0, a], mJ[:, 0, a] = q
            r[:, 0], mr[:, 0] = res
            return ok, amb, 1, J, _GAMMA * mJ, r, _GAMMA * mr
        Is = _c(s["intensity"].reshape(-1)[sel].astype(np.float64))
        Dt = _c(g["depth"])
        dz = _sub(Dt, vs[2])
        ok = inside & ~np.isnan(g["depth"]) & ~np.isnan(g["dix"]) & ~np.isnan(g["diy"])
        if method == HYBRID:
            ok &= ~np.isnan(g["ddx"]) & ~np.isnan(g["ddy"])
        amb = ok & (np.abs(np.abs(dz[0]) - trunc) <= _GAMMA * dz[1])
        ok &= np.abs(dz[0]) <= trunc
        invz = _div(_c(1.0), vs[2])
        FX, FY = _c(fx), _c(fy)

        def grad_rows(dx, dy):
            c0 = _mul(_mul(_mul(_c(0.125), _c(dx)), FX), invz)
            c1 = _mul(_mul(_mul(_c(0.125), _c(dy)), FY), invz)
            c2 = _neg(_mul(_add(_mul(c0, vs[0]), _mul(c1, vs[1])), invz))
            return c0, c1, c2

        c0, c1, c2 = grad_rows(g["dix"], g["diy"])
        wI = _c(np.float64(np.float32(0.17888544)) if method == HYBRID else 1.0)
        rows = [_sub(_mul(vs[1], c2), _mul(vs[2], c1)), _sub(_mul(vs[2], c0), _mul(vs[0], c2)), _sub(_mul(vs[0], c1), _mul(vs[1], c0)),
                c0, c1, c2]
        for a, q in enumerate(rows):
            J[:, 0, a], mJ[:, 0, a] = _mul(wI, q)
        r[:, 0], mr[:, 0] = _mul(wI, _sub(_c(g["intensity"]), Is))
        if method != HYBRID:
            return ok, amb, 1, J, _GAMMA * mJ, r, _GAMMA * mr
        d0, d1, d2 = grad_rows(g["ddx"], g["ddy"])
        wD = _c(np.float64(np.float32(0.98386991)))
        rows = [_sub(_sub(_mul(vs[1], d2), _mul(vs[2], d1)), vs[1]), _add(_sub(_mul(vs[2], d0), _mul(vs[0], d2)), vs[0]),
                _sub(_mul(vs[0], d1), _mul(vs[1], d0)), d0, d1, _sub(d2, _c(1.0))]
        for a, q in enumerate(rows):
            J[:, 1, a], mJ[:, 1, a] = _mul(wD, q)
        r[:, 1], mr[:, 1] = _mul(wD, dz)
        return ok, amb, 2, J, _GAMMA * mJ, r, _GAMMA * mr


def _contrib(J, eJ, r, er, nres, deltas, exact):
    """per-pixel terms of the 29 sums [n,29], and with exact=False their error bounds"""
    iu = np.triu_indices(6)
    out = np.zeros((J.shape[0], 29))
    for k in range(nres):
        Jk, eJk, rk, erk, d = J[:, k], eJ[:, k], r[:, k], er[:, k], deltas[k]
        if exact:
            hp, loss = _huber_deriv(rk, d), _huber(rk, d)
            out[:, :21] += (Jk[:, :, None] * Jk[:, None, :])[:, iu[0], iu[1]]
            out[:, 21:27] += Jk * hp[:, None]
            out[:, 27] += loss
        else:
            aJ = np.abs(Jk)
            ahp = np.minimum(np.abs(rk), d)
            ehp = np.where(np.abs(rk) <= d + erk, erk, 0.0)
            out[:, :21] += (eJk[:, :, None] * aJ[:, None, :] + aJ[:, :, None] * eJk[:, None, :] + eJk[:, :, None] * eJk[:, None, :])[:, iu[0], iu[1]]
            out[:, 21:27] += eJk * ahp[:, None] + aJ * ehp[:, None] + eJk * ehp[:, None]
            # |huber'| <= |r|, and huber itself is rounded twice in float32
            out[:, 27] += (np.abs(rk) + erk) * erk + 4 * U32 * _huber(np.abs(rk) + erk, d)
    out[:, 28] = 0.0 if not exact else 1.0
    return out


def _bound(J, eJ, r, er, nres, deltas):
    """upper bound of the magnitude of every term a pixel can add to the 29 sums"""
    return np.abs(_contrib(np.abs(J) + eJ, eJ, np.abs(r) + er, er, nres, deltas, True))


def linearize_f64(fr, src, tgt, level, T, method, params=(0.07, 0.05, 0.1)):
    """the 29 sums of pair (src, tgt) of Frames `fr` at `level` under the 4x4 T, in float64 (see above) ->
    dict(sums [29], tol [29]: the bound on |ref_odom_linearize - sums| derived above, ambiguous: pixels with a decision
    within its bound, branches: {residual: (inliers with |r| <= delta, inliers with |r| > delta)}, inliers)"""
    trunc, dhd, ihd = (np.float64(np.float32(p)) for p in params)
    deltas = (dhd,) if method == POINT_TO_PLANE else ((ihd,) if method == INTENSITY else (ihd, dhd))
    names = ("depth",) if method == POINT_TO_PLANE else (("intensity",) if method == INTENSITY else ("intensity", "depth"))
    Hl, Wl = fr.level_shape(level)
    s = fr.planes(src, level)
    fx, fy, cx, cy = (np.float64(np.float32(fr.K[k]) * np.float32(1.0 / (1 << level))) for k in range(4))
    Tf = np.asarray(T, np.float64).reshape(4, 4)[:3].astype(np.float32).astype(np.float64)
    v = [_c(s[k].reshape(-1).astype(np.float64)) for k in ("vx", "vy", "vz")]
    src_ok = ~np.isnan(v[2][0])
    if method != POINT_TO_PLANE:
        src_ok &= ~np.isnan(s["intensity"].reshape(-1))
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        vs = [_add(_add(_add(_mul(_c(Tf[q, 0]), v[0]), _mul(_c(Tf[q, 1]), v[1])), _mul(_c(Tf[q, 2]), v[2])), _c(Tf[q, 3])) for q in range(3)]
        front = vs[2][0] > 0
        amb_front = np.abs(vs[2][0]) <= _GAMMA * vs[2][1]
        uf = _add(_div(_mul(_c(fx), vs[0]), vs[2]), _c(cx))
        vf = _add(_div(_mul(_c(fy), vs[1]), vs[2]), _c(cy))
        eu, ev = _GAMMA * uf[1], _GAMMA * vf[1]
        proj = (uf[0] > -1) & (uf[0] < Wl) & (vf[0] > -1) & (vf[0] < Hl)
        amb_proj = (np.abs(uf[0] + 1) <= eu) | (np.abs(uf[0] - Wl) <= eu) | (np.abs(vf[0] + 1) <= ev) | (np.abs(vf[0] - Hl) <= ev)
        big = ~(np.abs(uf[0]) < 1e9) | ~(np.abs(vf[0]) < 1e9)
        ru = lambda x: np.where(big, -2, _round_away(np.where(big, 0, x))).astype(np.int64)
        u, w = ru(uf[0]), ru(vf[0])
        u_lo, u_hi, w_lo, w_hi = ru(uf[0] - eu), ru(uf[0] + eu), ru(vf[0] - ev), ru(vf[0] + ev)
        amb_round = (u_lo != u_hi) | (w_lo != w_hi)
        ok, amb_t, nres, J, eJ, r, er = _terms(fr, src, tgt, level, vs, u, w, method, trunc)
    pre = src_ok & front & proj
    inl = pre & ok
    rejected = ~src_ok | (~front & ~amb_front) | (~proj & ~amb_proj & ~amb_front) | (~amb_round & ~ok & ~amb_t)
    amb = ~rejected & (amb_front | amb_proj | amb_round | amb_t)
    clean = inl & ~amb
    sums = _contrib(J[inl], eJ[inl], r[inl], er[inl], nres, deltas, True).sum(0)
    tol = _contrib(J[clean], eJ[clean], r[clean], er[clean], nres, deltas, False).sum(0)
    tol += 1e-12 * np.abs(_contrib(J[inl], eJ[inl], r[inl], er[inl], nres, deltas, True)).sum(0)      # float64 summation
    if amb.any():
        # an ambiguous pixel may be in or out in float32, and roundf may pick either neighbour: its own terms plus the
        # largest terms any candidate target pixel gives
        own = np.where(inl[amb, None], _bound(J[amb], eJ[amb], r[amb], er[amb], nres, deltas), 0.0)
        worst = np.zeros_like(own)
        idx = np.nonzero(amb)[0]
        vsa = [(q[0][idx], q[1][idx]) for q in vs]
        for uu in (u_lo[idx], u_hi[idx]):
            for ww in (w_lo[idx], w_hi[idx]):
                with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
                    ok_c, amb_c, _, Jc, eJc, rc, erc = _terms(fr, src, tgt, level, vsa, uu, ww, method, trunc, idx)
                b = np.where((ok_c | amb_c)[:, None], _bound(Jc, eJc, rc, erc, nres, deltas), 0.0)
                worst = np.maximum(worst, np.nan_to_num(b, nan=0.0, posinf=0.0))
        tol += own.sum(0) + worst.sum(0)
    tol[28] = float(amb.sum())
    branches = {}
    for k, name in enumerate(names):
        a = np.abs(r[inl, k])
        branches[name] = (int((a <= deltas[k]).sum()), int((a > deltas[k]).sum()))
    return dict(sums=sums, tol=tol, ambiguous=int(amb.sum()), branches=branches, inliers=int(inl.sum()))
