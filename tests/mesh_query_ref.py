"""ctypes front-end of the brute-force CPU reference of the mesh point and ray queries, tests/mesh_query_ref.c (TEST
INFRASTRUCTURE, like oracle/).  Scenes are built as for the cast's reference (mesh_raycast_ref.scene).

The shared object is compiled on first use (gcc, -ffp-contract=off, OpenMP) into the temporary directory, under a name
that carries the hash of its sources, so nothing is written into the repository tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from mesh_raycast_ref import _CFLAGS, _ptr, scene

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRCS = [os.path.join(_HERE, "mesh_query_ref.c"), os.path.join(_HERE, "mesh_raycast_ref.c"),
         os.path.join(os.path.dirname(_HERE), "bodyslam_b200", "csrc", "bslam_mesh_dirs.h")]
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = b"".join(open(p, "rb").read() for p in _SRCS)
        tag = hashlib.sha256(src + " ".join(_CFLAGS).encode()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"bslam_mesh_query_ref_{os.getuid()}_{tag}.so")
        if not os.path.exists(path):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run([cc, *_CFLAGS, "-o", tmp, _SRCS[0], "-lm"], check=True, capture_output=True)
            os.replace(tmp, path)      # atomic: concurrent test processes never load a half-written file
        L = C.CDLL(path)
        p = C.c_void_p
        L.ref_mesh_closest.restype = None
        L.ref_mesh_closest.argtypes = [p, p, p, C.c_int, p, C.c_int64, p, p, p, p, p, p]
        L.ref_mesh_count.restype = None
        L.ref_mesh_count.argtypes = [p, p, p, C.c_int, p, C.c_int64, C.c_float, C.c_float, p]
        L.ref_mesh_directions.restype = None
        L.ref_mesh_directions.argtypes = [C.c_int, p]
        L.ref_mesh_occupancy.restype = C.c_int
        L.ref_mesh_occupancy.argtypes = [p, p, p, C.c_int, p, C.c_int64, C.c_int, p, p]
        L.ref_mesh_traverse_closest.restype = None
        L.ref_mesh_traverse_closest.argtypes = [p, p, C.c_int64, p, p, p, p]
        L.ref_mesh_traverse_count.restype = None
        L.ref_mesh_traverse_count.argtypes = [p, p, C.c_int64, C.c_float, C.c_float, C.c_int, p, p]
        _lib = L
    return _lib


MAX_SAMPLES = 31     # BSLAM_MESH_MAX_SAMPLES


def _queries(x, width):
    q = np.ascontiguousarray(x, dtype=np.float32)
    if q.ndim < 1 or q.shape[-1] != width:
        raise ValueError(f"queries must be [..., {width}] (got {q.shape})")
    return q, q.shape[:-1], q.size // width


def closest_points(geometries, points):
    """brute force: every point against every triangle -> dict (Open3D keys of compute_closest_points, plus "distance")"""
    verts, tris, geom = scene(geometries)
    q, lead, n = _queries(points, 3)
    out = {"points": np.empty((n, 3), np.float32), "geometry_ids": np.empty(n, np.uint32), "primitive_ids": np.empty(n, np.uint32),
           "primitive_uvs": np.empty((n, 2), np.float32), "primitive_normals": np.empty((n, 3), np.float32), "distance": np.empty(n, np.float32)}
    lib().ref_mesh_closest(_ptr(verts), _ptr(tris), _ptr(geom), len(geom) - 1, _ptr(q), n, _ptr(out["distance"]), _ptr(out["points"]),
                           _ptr(out["geometry_ids"]), _ptr(out["primitive_ids"]), _ptr(out["primitive_uvs"]), _ptr(out["primitive_normals"]))
    return {k: v.reshape(lead + v.shape[1:]) for k, v in out.items()}


def count_intersections(geometries, rays, tnear=0.0, tfar=np.inf):
    """brute force: int32 number of accepted hits with tnear <= t <= tfar per ray"""
    verts, tris, geom = scene(geometries)
    r, lead, n = _queries(rays, 6)
    out = np.empty(n, np.int32)
    lib().ref_mesh_count(_ptr(verts), _ptr(tris), _ptr(geom), len(geom) - 1, _ptr(r), n, float(tnear), float(tfar), _ptr(out))
    return out.reshape(lead)


def test_occlusions(geometries, rays, tnear=0.0, tfar=np.inf):
    """brute force: bool, some accepted hit with tnear <= t <= tfar (tnear >= 0, no NaN bound)"""
    if not (tnear >= 0.0) or np.isnan(tfar):
        raise ValueError(f"bad bounds tnear={tnear} tfar={tfar}")
    return count_intersections(geometries, rays, tnear, tfar) > 0


test_occlusions.__test__ = False        # a reference function, not a pytest test


def directions(n=MAX_SAMPLES):
    """[n, 3] float32 occupancy ray directions (bslam_mesh_dirs.h)"""
    out = np.empty((n, 3), np.float32)
    lib().ref_mesh_directions(int(n), _ptr(out))
    return out


def occupancy(geometries, points, nsamples=1):
    """brute force -> (occupancy float32 0 / 1, signed distance float32)"""
    verts, tris, geom = scene(geometries)
    q, lead, n = _queries(points, 3)
    occ, sd = np.empty(n, np.float32), np.empty(n, np.float32)
    if lib().ref_mesh_occupancy(_ptr(verts), _ptr(tris), _ptr(geom), len(geom) - 1, _ptr(q), n, int(nsamples), _ptr(occ), _ptr(sd)) != 0:
        raise ValueError(f"nsamples must be odd and in [1, {MAX_SAMPLES}] (got {nsamples})")
    return occ.reshape(lead), sd.reshape(lead)


def traverse_closest(bvh_bytes, points):
    """replay of the closest-point traversal -> (dict distance / geometry_ids / primitive_ids, inner nodes, leaf triangles)"""
    b = np.ascontiguousarray(bvh_bytes, dtype=np.uint8)
    q = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    n = len(q)
    out = {"distance": np.empty(n, np.float32), "geometry_ids": np.empty(n, np.uint32), "primitive_ids": np.empty(n, np.uint32)}
    counts = np.zeros(2, np.int64)
    lib().ref_mesh_traverse_closest(_ptr(b), _ptr(q), n, _ptr(out["distance"]), _ptr(out["geometry_ids"]), _ptr(out["primitive_ids"]), _ptr(counts))
    return out, int(counts[0]), int(counts[1])


def traverse_count(bvh_bytes, rays, tnear=0.0, tfar=np.inf, any_hit=False):
    """replay of the count (any_hit: occlusion) traversal -> (int32 counts, inner nodes, leaf triangles)"""
    b = np.ascontiguousarray(bvh_bytes, dtype=np.uint8)
    r = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 6)
    out = np.empty(len(r), np.int32)
    counts = np.zeros(2, np.int64)
    lib().ref_mesh_traverse_count(_ptr(b), _ptr(r), len(r), float(tnear), float(tfar), int(bool(any_hit)), _ptr(out), _ptr(counts))
    return out, int(counts[0]), int(counts[1])
