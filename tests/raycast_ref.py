"""ctypes front-end of the ray cast's CPU reference, tests/raycast_ref.c (TEST INFRASTRUCTURE, like oracle/).

The shared object is compiled on first use with the oracle's flags (gcc, -ffp-contract=off, OpenMP) into the temporary
directory, under a name that carries the source's hash, so nothing is written into the repository tree.  The functions
read the grids of an `oracle.o3d.Volume` (or any object with the same attributes)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "raycast_ref.c")
_CFLAGS = ["-O3", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden", "-Wall", "-Wextra", "-shared"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src + " ".join(_CFLAGS).encode()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"bslam_raycast_ref_{os.getuid()}_{tag}.so")
        if not os.path.exists(path):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run([cc, *_CFLAGS, "-o", tmp, _SRC, "-lm"], check=True, capture_output=True)
            os.replace(tmp, path)      # atomic: concurrent test processes never load a half-written file
        L = C.CDLL(path)
        p = C.c_void_p
        L.ref_raycast.restype = C.c_int64
        L.ref_raycast.argtypes = [p, p, p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, p, C.c_int, p, p, C.c_int, C.c_int, p, p,
                                  C.c_double, C.c_double, C.c_double, C.c_double, p, p, p, p]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _cast(V, flavour, K, M, W, H, depth_scale, depth_min, depth_max, weight_threshold, normals, colors, sdf_trunc, allocated=None,
          range_blocks=None):
    Kd = np.ascontiguousarray(K, dtype=np.float64)
    M = np.ascontiguousarray(M, dtype=np.float64).reshape(4, 4)
    a = None if allocated is None else np.ascontiguousarray(allocated, dtype=np.uint8)
    r = None if range_blocks is None else np.ascontiguousarray(range_blocks, dtype=np.uint8)
    grids = [np.ascontiguousarray(g, dtype=np.float32) for g in (V.tsdf, V.weight)]
    color = None if (V.color is None or not colors) else np.ascontiguousarray(V.color, dtype=np.float32)
    out = {"depth": np.empty((H, W), np.float32), "vertex": np.empty((H, W, 3), np.float32)}
    if normals:
        out["normal"] = np.empty((H, W, 3), np.float32)
    if colors:
        out["color"] = np.empty((H, W, 3), np.float32)
    out["samples"] = lib().ref_raycast(_ptr(grids[0]), _ptr(grids[1]), _ptr(color), V.nx, V.ny, V.nz, V.voxel_length, float(sdf_trunc),
                                       _ptr(np.ascontiguousarray(V.origin, dtype=np.float64)), int(flavour), _ptr(a), _ptr(r), int(W), int(H),
                                       _ptr(Kd), _ptr(M), float(depth_scale), float(depth_min), float(depth_max), float(weight_threshold),
                                       _ptr(out["depth"]), _ptr(out["vertex"]), _ptr(out.get("normal")), _ptr(out.get("color")))
    return out


def raycast(V, K, extrinsics, W, H, depth_min=0.0, depth_max=3.0, depth_scale=1.0, weight_threshold=0.0, normals=True, colors=None):
    """legacy flavour (`DenseTSDFVolume.raycast`): extrinsics [F,4,4] or one 4x4 world -> camera; V.sdf_trunc is the
    truncation.  -> dict of f32 arrays depth [F,H,W], vertex / normal / color [F,H,W,3] and `samples` (voxel samples the
    marches read)."""
    if getattr(V, "gz0", 0) or any(n % 8 for n in (V.nx, V.ny, V.nz)):
        raise ValueError("the ray cast needs a single box of whole 8^3 bricks")
    colors = V.color is not None if colors is None else bool(colors)
    E = np.asarray(extrinsics, dtype=np.float64).reshape(-1, 4, 4)
    frames = [_cast(V, 0, K, e, W, H, depth_scale, depth_min, depth_max, weight_threshold, normals, colors, V.sdf_trunc) for e in E]
    out = {k: np.stack([f[k] for f in frames]) for k in frames[0] if k != "samples"}
    out["samples"] = sum(f["samples"] for f in frames)
    return out


def raycast_vbg(V, K, pose, W, H, allocated, range_blocks, depth_scale=1000.0, depth_min=0.1, depth_max=3.0, weight_threshold=3.0,
                trunc_voxel_multiplier=8.0, normals=True, colors=None):
    """tensor flavour (`MAP.synthesize_model_frame`) from `pose` (camera -> world 4x4).  allocated / range_blocks:
    [nbx,nby,nbz] bool, the 16^3 blocks activated by any frame so far / by the last frame (`Volume.integrate_vbg`'s
    `touched`).  Same result layout as `raycast` with F = 1."""
    if any(n % 16 for n in (V.nx, V.ny, V.nz)):
        raise ValueError("the box must consist of whole 16^3 blocks")
    colors = V.color is not None if colors is None else bool(colors)
    out = _cast(V, 1, K, pose, W, H, depth_scale, depth_min, depth_max, weight_threshold, normals, colors, float(trunc_voxel_multiplier),
                allocated, range_blocks)
    return {k: (v if k == "samples" else v[None]) for k, v in out.items()}
