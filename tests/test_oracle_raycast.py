"""Ray cast: closed forms of both flavours on the CPU reference (tests/raycast_ref.c, `ref_raycast`), and the C ABI's
argument checks, which need no device."""
import ctypes

import numpy as np
import pytest

import oracle
import raycast_ref
from bodyslam_b200 import _lib

W, H = 160, 120
K = (150.0, 150.0, 80.0, 60.0)
VL = 0.004
ORIGIN = (-0.128, -0.128, 0.0)      # on the 16-voxel block grid (block = 0.064 m)


def plane_depth(D):
    return np.full((H, W), D, np.float32)


def sphere_depth(centre, R):
    """z-depth of the first intersection of each pixel ray (x - cx) / fx, (y - cy) / fy, 1 with the sphere; 0 = miss"""
    ys, xs = np.mgrid[0:H, 0:W].astype(np.float64)
    d = np.stack([(xs - K[2]) / K[0], (ys - K[3]) / K[1], np.ones_like(xs)], -1)
    c = np.asarray(centre, np.float64)
    a = (d * d).sum(-1)
    b = -2 * (d @ c)
    disc = b * b - 4 * a * (c @ c - R * R)
    t = np.where(disc >= 0, (-b - np.sqrt(np.maximum(disc, 0))) / (2 * a), 0.0)
    return t.astype(np.float32)


def legacy_volume(depth, frames=1):
    V = oracle.o3d.Volume(64, VL, 4 * VL, ORIGIN, with_color=True)
    rgb = np.full((H, W, 3), (200, 100, 50), np.uint8)
    for _ in range(frames):
        V.integrate(depth, K, np.eye(4), rgb=rgb)
    return V


class TensorVolume:
    """oracle volume integrated by integrate_vbg + the blocks any frame / the last frame activated"""

    def __init__(self, depth_m, frames):
        self.V = oracle.o3d.Volume(64, VL, 4 * VL, ORIGIN, with_color=True)
        u16 = np.rint(depth_m * 1000.0).astype(np.uint16)
        rgb = np.full((H, W, 3), (200, 100, 50), np.uint8)
        self.allocated = np.zeros((4, 4, 4), bool)
        for _ in range(frames):
            _, touched = self.V.integrate_vbg(u16, K, np.eye(4), rgb=rgb, depth_scale=1000.0, depth_max=3.0, trunc_voxel_multiplier=4.0,
                                              return_touched=True)
            self.touched = touched.astype(bool)
            self.allocated |= self.touched


def tensor_volume(depth_m, frames=1):
    return TensorVolume(depth_m, frames)


def cast(V, flavour, pose=np.eye(4), **kw):
    if flavour == "legacy":
        return raycast_ref.raycast(V, K, np.linalg.inv(pose), W, H, **kw)
    kw.setdefault("weight_threshold", 3.0)
    kw.setdefault("allocated", V.allocated)
    kw.setdefault("range_blocks", V.touched)
    return raycast_ref.raycast_vbg(V.V, K, pose, W, H, depth_scale=1.0, trunc_voxel_multiplier=4.0, **kw)


@pytest.mark.parametrize("flavour", ["legacy", "tensor"])
def test_plane_closed_form(flavour):
    D = 0.12
    V = legacy_volume(plane_depth(D)) if flavour == "legacy" else tensor_volume(plane_depth(D), frames=3)
    r = cast(V, flavour)
    hit = r["depth"][0] > 0
    assert hit.mean() >= 0.95, hit.mean()
    assert np.abs(r["depth"][0][hit] - D).max() <= VL
    assert np.abs(r["vertex"][0][hit][:, 2] - r["depth"][0][hit]).max() <= 1e-6
    # normals: away from the frustum's edge, where never-observed voxels of observed bricks (tsdf 0) bend the gradient
    inner = np.zeros_like(hit)
    inner[8:-8, 8:-8] = True
    n = r["normal"][0][hit & inner]
    assert len(n) >= 0.9 * inner.sum()
    # the legacy sdf is scaled by the pixel's ray length, which tilts its gradient a little off the plane's normal
    assert np.abs(n - np.array([0, 0, -1], np.float32)).max() <= (1e-2 if flavour == "legacy" else 1e-3)
    assert np.abs(r["color"][0][hit] - np.array([200, 100, 50], np.float32) / 255).max() <= 1e-5
    assert r["samples"] > hit.sum()


@pytest.mark.parametrize("flavour", ["legacy", "tensor"])
def test_sphere_closed_form(flavour):
    centre, R = (0.0, 0.0, 0.14), 0.05
    ref = sphere_depth(centre, R)
    ref_mm = np.rint(ref * 1000.0) / 1000.0
    V = legacy_volume(ref) if flavour == "legacy" else tensor_volume(ref, frames=3)
    r = cast(V, flavour)
    d = r["depth"][0]
    hit = d > 0
    assert hit[sphere_depth(centre, 0.9 * R) > 0].all()
    # away from the grazing rim: the march samples the nearest voxel, not the ray's own point, so on a slope its depth
    # is off by the slope times up to a voxel; the tensor flavour's projective sdf (no ray-length factor) doubles that
    inner = sphere_depth(centre, (0.8 if flavour == "legacy" else 0.7) * R) > 0
    truth = ref if flavour == "legacy" else ref_mm
    assert np.abs(d[inner] - truth[inner]).max() <= (1 if flavour == "legacy" else 2) * VL
    assert np.abs(d[hit & (truth > 0)] - truth[hit & (truth > 0)]).max() <= 4 * VL


@pytest.mark.parametrize("flavour", ["legacy", "tensor"])
def test_rays_that_leave_the_box_or_start_beyond_depth_max_miss(flavour):
    D = 0.12
    V = legacy_volume(plane_depth(D)) if flavour == "legacy" else tensor_volume(plane_depth(D), frames=3)
    away = np.diag([1.0, -1.0, -1.0, 1.0])                  # looking down -z, out of the box
    assert not cast(V, flavour, pose=away)["depth"].any()
    if flavour == "legacy":      # the tensor flavour's range comes from the blocks (see test_tensor_flavour_needs_allocated_blocks)
        assert not cast(V, flavour, depth_min=0.5, depth_max=3.0)["depth"].any()
        assert not cast(V, flavour, depth_min=0.0, depth_max=0.1)["depth"].any()
        assert not cast(V, flavour, depth_min=3.0, depth_max=2.0)["depth"].any()
    full = cast(V, flavour)
    assert full["depth"].any()
    for k in ("vertex", "normal", "color"):
        assert not full[k][0][full["depth"][0] == 0].any(), k


def test_tensor_flavour_needs_allocated_blocks():
    V = tensor_volume(plane_depth(0.12), frames=3)
    assert cast(V, "tensor")["depth"].any()
    none = np.zeros_like(V.allocated)
    assert not cast(V, "tensor", allocated=none)["depth"].any()
    assert not cast(V, "tensor", range_blocks=none)["depth"].any()


def test_c_abi_argument_errors_do_not_need_a_device():
    L = _lib.load()
    K4 = np.array(K, np.float64)
    E = np.eye(4).reshape(-1)
    out = ctypes.c_void_p(16)          # never dereferenced: the arguments are rejected first
    assert L.bslam_tsdf_raycast(None, 1, H, W, _lib.ptr(K4), _lib.ptr(E), 1.0, 0.0, 3.0, 0.0, out, None, None, None, None) == _lib.E_ARG
    assert b"NULL" in L.bslam_last_error()
    for F, h, w in ((-1, H, W), (1, 0, W), (1, H, -3)):
        assert L.bslam_tsdf_raycast(None, F, h, w, _lib.ptr(K4), _lib.ptr(E), 1.0, 0.0, 3.0, 0.0, out, None, None, None, None) == _lib.E_ARG
        assert b"Unsupported image format" in L.bslam_last_error()
    assert L.bslam_tsdf_raycast(None, 1, H, W, _lib.ptr(K4), _lib.ptr(E), 0.0, 0.0, 3.0, 0.0, out, None, None, None, None) == _lib.E_ARG
    assert L.bslam_tsdf_raycast(None, 1, H, W, _lib.ptr(K4), _lib.ptr(E), 1.0, 0.0, 3.0, -1.0, out, None, None, None, None) == _lib.E_ARG
    assert L.bslam_vbg_raycast(None, out, 4, W, _lib.ptr(K4), _lib.ptr(E), 1.0, 0.1, 3.0, 3.0, 8.0, out, None, None, None, out, None) == _lib.E_ARG
    assert b"Unsupported image format" in L.bslam_last_error()
    assert L.bslam_vbg_raycast(None, out, H, W, _lib.ptr(K4), _lib.ptr(E), 1.0, 0.1, 3.0, 3.0, 8.0, out, None, None, None, out, None) == _lib.E_ARG
    assert L.bslam_vbg_raycast_workspace_bytes(H, W) == (H // 8) * (W // 8) * 8
    assert L.bslam_vbg_raycast_workspace_bytes(4, W) == 0
