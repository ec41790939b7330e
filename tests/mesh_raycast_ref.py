"""ctypes front-end of the mesh ray cast's brute-force CPU reference, tests/mesh_raycast_ref.c (TEST INFRASTRUCTURE, like
oracle/).

The shared object is compiled on first use (gcc, -ffp-contract=off, OpenMP) into the temporary directory, under a name
that carries the source's hash, so nothing is written into the repository tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mesh_raycast_ref.c")
_CFLAGS = ["-O3", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden", "-Wall", "-Wextra", "-shared"]
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src + " ".join(_CFLAGS).encode()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"bslam_mesh_raycast_ref_{os.getuid()}_{tag}.so")
        if not os.path.exists(path):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run([cc, *_CFLAGS, "-o", tmp, _SRC, "-lm"], check=True, capture_output=True)
            os.replace(tmp, path)      # atomic: concurrent test processes never load a half-written file
        L = C.CDLL(path)
        p = C.c_void_p
        L.ref_mesh_cast.restype = None
        L.ref_mesh_cast.argtypes = [p, p, p, C.c_int, p, C.c_int64, p, p, p, p, p]
        L.ref_mesh_rays_pinhole.restype = None
        L.ref_mesh_rays_pinhole.argtypes = [p, p, C.c_int, C.c_int, p]
        L.ref_mesh_traverse.restype = None
        L.ref_mesh_traverse.argtypes = [p, p, C.c_int64, p, p, p, p]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def scene(geometries):
    """[(vertices [V,3], triangles [T,3]), ...] -> (verts f32, tris i32, geom [G+1,2] i64) as the library takes them"""
    vs, ts, geom = [], [], [[0, 0]]
    for v, t in geometries:
        v = np.ascontiguousarray(v, dtype=np.float32).reshape(-1, 3)
        t = np.asarray(t).reshape(-1, 3).astype(np.int64)
        if t.size and (t.min() < 0 or t.max() >= len(v)):
            raise ValueError("triangle index out of range")
        vs.append(v)
        ts.append(t.astype(np.int32))
        geom.append([geom[-1][0] + len(t), geom[-1][1] + len(v)])
    verts = np.concatenate(vs) if vs else np.zeros((0, 3), np.float32)
    tris = np.concatenate(ts) if ts else np.zeros((0, 3), np.int32)
    return np.ascontiguousarray(verts), np.ascontiguousarray(tris), np.ascontiguousarray(geom, dtype=np.int64)


def cast_rays(geometries, rays):
    """brute force: every ray against every triangle -> dict of numpy arrays with the rays' leading shape (Open3D keys)"""
    verts, tris, geom = scene(geometries)
    r = np.ascontiguousarray(rays, dtype=np.float32)
    lead = r.shape[:-1]
    n = r.size // 6
    out = {"t_hit": np.empty(n, np.float32), "geometry_ids": np.empty(n, np.uint32), "primitive_ids": np.empty(n, np.uint32),
           "primitive_uvs": np.empty((n, 2), np.float32), "primitive_normals": np.empty((n, 3), np.float32)}
    lib().ref_mesh_cast(_ptr(verts), _ptr(tris), _ptr(geom), len(geom) - 1, _ptr(r), n, *(_ptr(out[k]) for k in out))
    return {k: v.reshape(lead + v.shape[1:]) for k, v in out.items()}


def rays_pinhole(K, extrinsic, W, H):
    """[H, W, 6] f32 rays of one pinhole camera (K 3x3, extrinsic 4x4 world -> camera)"""
    Kd = np.ascontiguousarray(K, dtype=np.float64).reshape(3, 3)
    E = np.ascontiguousarray(extrinsic, dtype=np.float64).reshape(4, 4)
    out = np.empty((H, W, 6), np.float32)
    lib().ref_mesh_rays_pinhole(_ptr(Kd), _ptr(E), int(W), int(H), _ptr(out))
    return out


def traverse(bvh_bytes, rays):
    """replay of the GPU traversal over a host copy of the BVH -> (dict t_hit / geometry_ids / primitive_ids, inner
    nodes read, leaf triangles read)"""
    b = np.ascontiguousarray(bvh_bytes, dtype=np.uint8)
    r = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
    n = len(r)
    out = {"t_hit": np.empty(n, np.float32), "geometry_ids": np.empty(n, np.uint32), "primitive_ids": np.empty(n, np.uint32)}
    counts = np.zeros(2, np.int64)
    lib().ref_mesh_traverse(_ptr(b), _ptr(r), n, _ptr(out["t_hit"]), _ptr(out["geometry_ids"]), _ptr(out["primitive_ids"]), _ptr(counts))
    return out, int(counts[0]), int(counts[1])
