"""Mesh ray casting on the GPU: Open3D's `t.geometry.RaycastingScene` (the reference's synthetic depth generator,
N/3DM/synthetic_depth_generator.py:74-97: `create_rays_pinhole` + `cast_rays(...)["t_hit"]` as a depth map).

The scene's BVH is built on the device (csrc/bslam_mesh_raycast.cu) and every query runs there; the results equal the
brute-force CPU reference tests/mesh_raycast_ref.c bit for bit (parity with Open3D / Embree is unpinned, DESIGN.md
section 7).  There is no CPU path.
"""
from __future__ import annotations

import numpy as np

from . import _lib, ops
from .geometry import to_numpy

INVALID_ID = 0xFFFFFFFF
_INDEX_DTYPES = ("int32", "int64", "uint32")
_KEYS = ("t_hit", "geometry_ids", "primitive_ids", "primitive_uvs", "primitive_normals")   # C ABI output order


def _mesh_arrays(mesh):
    """(vertices, triangles) of ours (`.vertices` / `.triangles`, torch CUDA tensors stay on the device), a legacy
    Open3D mesh (same names) or a tensor Open3D mesh (`.vertex.positions` / `.triangle.indices`)"""
    if hasattr(mesh, "vertex") and hasattr(mesh, "triangle"):
        return mesh.vertex.positions.numpy(), mesh.triangle.indices.numpy()
    return mesh.vertices, mesh.triangles


def _indices(t, dev):
    """[T,3] int32 CUDA tensor of int32 / int64 / uint32 indices; values beyond int32 become -1 or INT32_MAX, which the
    build rejects as out of range like any other bad index"""
    torch = _lib.require_cuda()
    name = ops._dtype_name(t)
    if name not in _INDEX_DTYPES:
        raise RuntimeError(f"RaycastingScene.add_triangles: triangle indices must be int32, int64 or uint32 (got {name})")
    if not hasattr(t, "is_cuda"):
        t = torch.from_numpy(np.ascontiguousarray(to_numpy(t)).astype(np.int64 if name != "int32" else np.int32))
    t = t.to(dev)
    if t.dtype != torch.int32:
        t = t.to(torch.int64).clamp_(-1, 2 ** 31 - 1).to(torch.int32)
    return t.reshape(-1, 3).contiguous()


class RaycastingScene:
    """Open3D `t.geometry.RaycastingScene`: add triangle meshes, then cast rays against all of them.

    Geometry g is the index of the add_triangles call that added it, primitive p the triangle's row within it.  The
    BVH is (re)built on the first cast after an add_triangles (Open3D commits its scene the same way); the build checks
    the triangle indices on the device and synchronises once for it."""

    def __init__(self, device=None):
        self.torch = _lib.require_cuda()
        self.device = ops._device(device)
        self._geoms = []           # (vertices [V,3] f32, triangles [T,3] i32) CUDA tensors
        self._bvh = None

    def add_triangles(self, vertices, triangles=None) -> int:
        """add_triangles(mesh) or add_triangles(vertices [V,3], triangles [T,3]) -> geometry id.  Vertices are float
        (stored as float32), indices int32 / int64 / uint32; numpy, torch (CPU or CUDA) or Open3D arrays."""
        if triangles is None:
            vertices, triangles = _mesh_arrays(vertices)
        v = ops.as_cuda(vertices, self.torch.float32, self.device).reshape(-1, 3)
        t = _indices(triangles, self.device)
        self._geoms.append((v, t))
        self._bvh = None
        return len(self._geoms) - 1

    def _commit(self):
        if self._bvh is not None:
            return self._bvh
        torch, L = self.torch, _lib.load()
        verts = torch.cat([v for v, _ in self._geoms]) if self._geoms else torch.zeros((0, 3), dtype=torch.float32, device=self.device)
        tris = torch.cat([t for _, t in self._geoms]) if self._geoms else torch.zeros((0, 3), dtype=torch.int32, device=self.device)
        geom = np.zeros((len(self._geoms) + 1, 2), np.int64)
        geom[1:, 0] = np.cumsum([len(t) for _, t in self._geoms])
        geom[1:, 1] = np.cumsum([len(v) for v, _ in self._geoms])
        n_tris = int(geom[-1, 0])
        if n_tris >= 2 ** 31 - 1:
            raise RuntimeError(f"RaycastingScene: too many triangles ({n_tris})")
        bvh = torch.empty(L.bslam_mesh_bvh_bytes(n_tris), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            ws_bytes = L.bslam_mesh_build_workspace_bytes(n_tris, len(self._geoms)) if n_tris else 0
            if n_tris and ws_bytes == 0:
                raise RuntimeError("RaycastingScene: the BVH build's sort cannot be sized on this device")
            ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=self.device)
            _lib.check(L.bslam_mesh_build(_lib.ptr(verts), len(verts), _lib.ptr(tris), n_tris, _lib.ptr(geom), len(self._geoms), _lib.ptr(bvh),
                                          _lib.ptr(ws), _lib.stream_ptr(self.device)))
        self._bvh = bvh
        return bvh

    def _outputs(self, lead, uvs, normals):
        torch = self.torch
        out = {"t_hit": torch.empty(lead, dtype=torch.float32, device=self.device),
               "geometry_ids": torch.empty(lead, dtype=torch.uint32, device=self.device),
               "primitive_ids": torch.empty(lead, dtype=torch.uint32, device=self.device)}
        if uvs:
            out["primitive_uvs"] = torch.empty(lead + (2,), dtype=torch.float32, device=self.device)
        if normals:
            out["primitive_normals"] = torch.empty(lead + (3,), dtype=torch.float32, device=self.device)
        return out

    def cast_rays(self, rays, uvs: bool = True, normals: bool = True) -> dict:
        """rays [..., 6] float32 {origin, direction} (direction not normalised; hits at o + t d, t >= 0) -> dict of CUDA
        tensors with the rays' leading shape: t_hit (+inf on a miss), geometry_ids / primitive_ids uint32 (INVALID_ID
        on a miss), primitive_uvs [..., 2] and primitive_normals [..., 3] (0 on a miss; left out when not asked for)."""
        torch, L = self.torch, _lib.load()
        if ops._dtype_name(rays) != "float32" or len(rays.shape) < 1 or rays.shape[-1] != 6:
            raise RuntimeError(f"RaycastingScene.cast_rays: rays must be float32 [..., 6] (got {ops._dtype_name(rays)} {tuple(rays.shape)})")
        r = ops.as_cuda(rays, torch.float32, self.device)
        lead = tuple(r.shape[:-1])
        bvh = self._commit()
        out = self._outputs(lead, uvs, normals)
        with torch.cuda.device(self.device):
            _lib.check(L.bslam_mesh_cast_rays(_lib.ptr(bvh), _lib.ptr(r), r.numel() // 6, *(_lib.ptr(out.get(k)) for k in _KEYS),
                                              _lib.stream_ptr(self.device)))
        return out

    @staticmethod
    def create_rays_pinhole(intrinsic_matrix, extrinsic_matrix, width_px: int, height_px: int, device=None):
        """[height_px, width_px, 6] float32 CUDA rays of a pinhole camera (K 3x3, extrinsic 4x4 world -> camera): origin
        the camera centre, direction R^T K^-1 (x + 0.5, y + 0.5, 1), so that t_hit is the camera-frame depth."""
        torch = _lib.require_cuda()
        dev = ops._device(device)
        K = np.ascontiguousarray(to_numpy(intrinsic_matrix), dtype=np.float64).reshape(3, 3)
        E = np.ascontiguousarray(to_numpy(extrinsic_matrix), dtype=np.float64).reshape(4, 4)
        W, H = int(width_px), int(height_px)
        out = torch.empty((H, W, 6), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.load().bslam_mesh_rays_pinhole(1, H, W, _lib.ptr(K), _lib.ptr(E), _lib.ptr(out), _lib.stream_ptr(dev)))
        return out

    def cast_pinhole(self, intrinsic, extrinsics, width_px: int | None = None, height_px: int | None = None, uvs: bool = True,
                     normals: bool = True) -> dict:
        """Batched `cast_rays(create_rays_pinhole(K, E, W, H))` without storing the rays: intrinsic is a 3x3 K (then
        width_px / height_px are required) or a PinholeCameraIntrinsic; extrinsics [F,4,4] or one 4x4 world -> camera.
        -> the dict of cast_rays with a leading F ([F, H, W, ...]), pixel for pixel equal to it."""
        torch, L = self.torch, _lib.load()
        if hasattr(intrinsic, "intrinsic_matrix"):
            K = intrinsic.intrinsic_matrix
            width_px = intrinsic.width if width_px is None else width_px
            height_px = intrinsic.height if height_px is None else height_px
        else:
            K = intrinsic
        if width_px is None or height_px is None:
            raise RuntimeError("RaycastingScene.cast_pinhole: width_px and height_px are required with a 3x3 intrinsic matrix")
        K = np.ascontiguousarray(to_numpy(K), dtype=np.float64).reshape(3, 3)
        E = np.ascontiguousarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 4, 4)
        F, W, H = len(E), int(width_px), int(height_px)
        bvh = self._commit()
        out = self._outputs((F, H, W), uvs, normals)
        with torch.cuda.device(self.device):
            _lib.check(L.bslam_mesh_cast_pinhole(_lib.ptr(bvh), F, H, W, _lib.ptr(K), _lib.ptr(E), *(_lib.ptr(out.get(k)) for k in _KEYS),
                                                 _lib.stream_ptr(self.device)))
        return out
