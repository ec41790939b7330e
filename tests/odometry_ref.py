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
