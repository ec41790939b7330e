"""Free (brick, frame) pairs -- `-m gpu`.

The cull marks a pair free when every voxel of the brick whose pixel holds a valid depth lies at
least 2 * sdf_trunc in front of that depth; the integrate kernel then updates those voxels with
t == 1 without classifying them.  The volumes must stay bit-identical to the CPU oracle: compared
by sha256 of tsdf and weight, plus the per-frame update counts."""
import hashlib

import numpy as np
import pytest
import torch

import oracle
from bodyslam_b200.geometry import PinholeCameraIntrinsic
from bodyslam_b200.tsdf import DenseTSDFVolume
from util import small_scene

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def assert_same_volume(vol, V, color=False):
    out = vol.export_dense(with_color=color)
    t, w = out[0].cpu().numpy(), out[1].cpu().numpy()
    assert sha(w) == sha(V.grid("weight")), "weights differ"
    assert sha(t) == sha(V.grid("tsdf")), f"tsdf differs (max {np.abs(t - V.grid('tsdf')).max()})"
    if color:
        assert np.abs(out[2].cpu().numpy() - V.color.reshape(out[2].shape)).max() <= 1e-3


def integrate_both(depth_f32, K, E, res, vl, trunc, origin, rgb=None, unit=False):
    """GPU batch integration and the oracle over the same f32 frames -> (vol, V, gpu counts, oracle counts)."""
    F, H, W = depth_f32.shape
    vol = DenseTSDFVolume(vl, trunc, res, origin, color=rgb is not None, device=torch.device("cuda", 0), unit_activation=unit)
    counts = torch.zeros(F, dtype=torch.int64, device="cuda")
    col = None if rgb is None else torch.from_numpy(rgb).cuda()
    vol.integrate_batch(torch.from_numpy(depth_f32).cuda(), col, PinholeCameraIntrinsic(W, H, *K), E, update_counts=counts)
    V = oracle.o3d.Volume(res, vl, trunc, origin, with_color=rgb is not None)
    oc = []
    for i in range(F):
        c = None if rgb is None else rgb[i]
        oc.append(V.integrate_scalable(depth_f32[i], K, E[i], rgb=c) if unit else V.integrate(depth_f32[i], K, E[i], rgb=c))
    return vol, V, counts.cpu().numpy(), np.array(oc)


def free_share(vol, depth_f32, K, E):
    """dry_stats of one dry run over the frames: (free pairs, all pairs)"""
    F, H, W = depth_f32.shape
    vol.dry_stats(True)
    vol.count_updates(torch.from_numpy(depth_f32).cuda(), PinholeCameraIntrinsic(W, H, *K), E)
    s = vol.dry_stats(True)
    return s["free_pairs"], s["warp_frame_pairs"]


@pytest.mark.parametrize("res", [128, 256])
def test_laparoscopy_sweep_matches_oracle_with_free_pairs(cuda, res):
    sc = small_scene("laparoscopy512", res=res, frames=6)
    d = oracle.o3d.depth_from_u16(sc["depth_u16"])
    vol, V, gc, oc = integrate_both(d, sc["K"], sc["E"], res, sc["voxel_length"], sc["sdf_trunc"], sc["origin"])
    assert oc.sum() > 1000
    assert np.array_equal(gc, oc), f"per-frame update counts differ: {gc} vs {oc}"
    assert_same_volume(vol, V)
    n_free, n_pairs = free_share(vol, d, sc["K"], sc["E"])
    assert 0 < n_free < n_pairs


# a wall facing the camera (world = camera frame); 64^3 voxels of 2 mm, sdf_trunc = 4 voxels, the box on the
# 32-voxel unit grid from z = 64 mm.  Brick layer bz ends at voxel centre z0 + (8 bz + 7.5) vl.
W_, H_ = 160, 120
K_ = (100.0, 100.0, 79.5, 59.5)
VL, TRUNC, RES = 0.002, 0.008, 64
ORIGIN = np.array([-0.064, -0.064, 0.064])


def wall(D, F=1, invalid_every=0):
    d = np.full((F, H_, W_), D, np.float32)
    if invalid_every:
        d.reshape(F, -1)[:, ::invalid_every] = 0.0
    return d


def eye(F):
    return np.repeat(np.eye(4)[None], F, axis=0)


@pytest.mark.parametrize("gap", [-1, 0, 1])
def test_wall_at_the_free_margin(cuda, gap):
    """the last voxel layer of brick layer 2 lies 2*trunc + gap voxels in front of the wall"""
    D = ORIGIN[2] + (8 * 2 + 7.5) * VL + (2 * TRUNC / VL + gap) * VL
    d = wall(D, F=2, invalid_every=7)
    vol, V, gc, oc = integrate_both(d, K_, eye(2), RES, VL, TRUNC, ORIGIN)
    assert oc.sum() > 0
    assert np.array_equal(gc, oc)
    assert_same_volume(vol, V)
    n_free, n_pairs = free_share(vol, d, K_, eye(2))
    assert 0 < n_free < n_pairs


def test_large_invalid_regions_and_depth_beyond_truncation(cuda):
    sc = small_scene("laparoscopy512", res=128, frames=4)
    u = sc["depth_u16"].copy()
    u[0, :, : u.shape[2] // 2] = 0           # half the image without depth
    u[1, : u.shape[1] // 3] = 4000           # beyond depth_trunc = 3 m: dropped by the conversion
    u[2, u.shape[1] // 2 :, u.shape[2] // 2 :] = 2500   # valid but far behind the volume
    u[3, ::3] = 0                            # every third row invalid
    d = oracle.o3d.depth_from_u16(u)
    vol, V, gc, oc = integrate_both(d, sc["K"], sc["E"], 128, sc["voxel_length"], sc["sdf_trunc"], sc["origin"])
    assert np.array_equal(gc, oc)
    assert_same_volume(vol, V)
    # the fused uint16 path (conversion in the depth statistics pass) gives the same volume
    vol2 = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 128, sc["origin"], color=False, device=cuda)
    counts = torch.zeros(4, dtype=torch.int64, device=cuda)
    vol2.integrate_u16_batch(torch.from_numpy(u).cuda(), None, sc["intrinsic"], sc["E"], 1000.0, 3.0, update_counts=counts)
    assert np.array_equal(counts.cpu().numpy(), oc)
    assert_same_volume(vol2, V)


def band_then_free_frames():
    """frame 0 puts the wall inside brick layer 3 (tsdf != 1 there and in front of it); frames 1.. move it back
    so far that those bricks become free pairs: their updates take the (tsdf*w + 1)/(w + 1) division"""
    d0 = wall(ORIGIN[2] + 30 * VL, invalid_every=5)
    d1 = wall(ORIGIN[2] + 60 * VL, F=3, invalid_every=11)
    return np.concatenate([d0, d1]), eye(4)


def test_band_voxels_later_updated_by_free_pairs(cuda):
    d, E = band_then_free_frames()
    vol, V, gc, oc = integrate_both(d, K_, E, RES, VL, TRUNC, ORIGIN)
    assert np.array_equal(gc, oc)
    assert_same_volume(vol, V)
    t, w = V.grid("tsdf"), V.grid("weight")
    assert ((w > 1) & (t != 1.0) & (t > 0)).any(), "no voxel went through the division"
    n_free, _ = free_share(vol, d[1:], K_, E[1:])
    assert n_free > 0


@pytest.mark.parametrize("unit", [False, True])
def test_color_and_unit_volumes(cuda, unit):
    d, E = band_then_free_frames()
    rng = np.random.default_rng(3)
    rgb = rng.integers(0, 256, size=d.shape + (3,), dtype=np.uint8)
    vol, V, gc, oc = integrate_both(d, K_, E, RES, VL, TRUNC, ORIGIN, rgb=rgb, unit=unit)
    assert oc.sum() > 0
    assert np.array_equal(gc, oc)
    assert_same_volume(vol, V, color=True)
    n_free, _ = free_share(vol, d, K_, E)
    assert n_free > 0
