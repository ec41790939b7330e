"""Ray casting on the GPU (csrc/bslam_raycast.cu) against its CPU reference (tests/raycast_ref.c; parity with Open3D
unpinned): `DenseTSDFVolume.raycast` (legacy flavour) and `MAP.synthesize_model_frame` (tensor flavour) -- `-m gpu`."""
import numpy as np
import pytest
import torch

import oracle
import raycast_ref
from bodyslam_b200 import _lib
from bodyslam_b200.tsdf import MAP, DenseTSDFVolume
from test_gpu_map import FakeRGBD, k3x3
from util import small_scene

pytestmark = pytest.mark.gpu

KEYS = ("depth", "vertex", "normal", "color")


def unit_origin(origin, vl):
    ul = vl * 32
    return np.floor(np.asarray(origin, dtype=np.float64) / ul + 0.5) * ul


def between(Ea, Eb):
    """world -> camera pose halfway between two extrinsics: Ea's rotation, the mean camera centre"""
    Pa, Pb = np.linalg.inv(Ea), np.linalg.inv(Eb)
    P = Pa.copy()
    P[:3, 3] = 0.5 * (Pa[:3, 3] + Pb[:3, 3])
    return np.linalg.inv(P)


def oracle_of(vol):
    """oracle volume holding the GPU volume's exported grids"""
    t, w, c = (x.cpu().numpy() for x in vol.export_dense(with_color=True))
    V = oracle.o3d.Volume((vol.nx, vol.ny, vol.nz), vol.voxel_length, vol.sdf_trunc, vol.origin, with_color=True)
    V.tsdf[:], V.weight[:], V.color[:] = t.reshape(-1), w.reshape(-1), c.reshape(-1)
    return V


def assert_same(gpu, ref):
    hit = gpu["depth"].cpu().numpy() > 0
    assert np.array_equal(hit, ref["depth"] > 0), f"hit masks differ in {(hit != (ref['depth'] > 0)).sum()} pixels"
    for k in KEYS:
        if k in ref:
            g = gpu[k].cpu().numpy()
            assert np.array_equal(g, ref[k]), f"{k} differs by {np.abs(g - ref[k]).max()}"
    return hit


@pytest.fixture(scope="module", params=["dense", "unit_activation"])
def legacy(request):
    sc = small_scene("laparoscopy512", res=128, frames=6)
    vl = sc["voxel_length"]
    vol = DenseTSDFVolume(vl, sc["sdf_trunc"], 128, unit_origin(sc["origin"], vl), color=True, device="cuda:0",
                          unit_activation=request.param == "unit_activation")
    dev = torch.device("cuda", 0)
    from bodyslam_b200 import ops

    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, dev)
    vol.integrate_batch(depth, torch.as_tensor(sc["color"], device=dev), sc["intrinsic"], sc["E"])
    return sc, vol


def test_legacy_raycast_matches_oracle(legacy):
    sc, vol = legacy
    V = oracle_of(vol)
    poses = list(sc["E"]) + [between(sc["E"][0], sc["E"][1]), between(sc["E"][2], sc["E"][3])]
    before = [x.clone() for x in vol.export_dense(with_color=True)]
    gpu = vol.raycast(sc["intrinsic"], np.stack(poses))
    for x, y in zip(before, vol.export_dense(with_color=True)):
        assert torch.equal(x, y), "the ray cast changed the volume"
    ref = raycast_ref.raycast(V, sc["K"], np.stack(poses), sc["W"], sc["H"])
    hit = assert_same(gpu, ref)
    assert hit[:len(sc["E"])].mean(axis=(1, 2)).min() > 0.5, hit.mean(axis=(1, 2))
    # F poses in one call == F single calls; depth only == the same depth
    for i in (0, len(poses) - 1):
        one = vol.raycast(sc["intrinsic"], poses[i])
        for k in KEYS:
            assert torch.equal(one[k][0], gpu[k][i]), k
    bare = vol.raycast(sc["intrinsic"], poses[0], normals=False, colors=False)
    assert set(bare) == {"depth", "vertex"} and torch.equal(bare["depth"][0], gpu["depth"][0])
    # another threshold and range
    g2 = vol.raycast(sc["intrinsic"], poses[1], depth_min=0.05, depth_max=0.2, depth_scale=1000.0, weight_threshold=2.0)
    assert_same(g2, raycast_ref.raycast(V, sc["K"], poses[1], sc["W"], sc["H"], depth_min=0.05, depth_max=0.2, depth_scale=1000.0,
                                        weight_threshold=2.0))


def test_brick_flag_bit0_iff_some_weight(legacy):
    _, vol = legacy
    w = vol.export_dense()[1].cpu().numpy()
    nb = [n // 8 for n in (vol.nx, vol.ny, vol.nz)]
    any_w = (w.reshape(nb[0], 8, nb[1], 8, nb[2], 8) != 0).any(axis=(1, 3, 5))          # [bx, by, bz]
    flags = vol.storage_layers()["flags"].cpu().numpy().reshape(nb[2], nb[1], nb[0])       # (bz * nby + by) * nbx + bx
    assert np.array_equal((flags & 1).astype(bool).transpose(2, 1, 0), any_w)
    assert any_w.any() and not any_w.all()


def test_map_synthesize_model_frame_matches_oracle(cuda):
    sc = small_scene("laparoscopy512", res=64, frame_ids=np.arange(0, 10, 2))
    vs, res = 0.0058, 96
    bs = vs * 16
    centre = sc["origin"] + 0.5 * 64 * sc["voxel_length"]
    origin = np.floor((centre - 0.5 * res * vs) / bs + 0.5) * bs
    m = MAP(640, 480, k3x3(sc["K"]), "CUDA:0", 1000.0, voxel_size=vs, trunc_voxel_multiplier=4.0, resolution=res, origin=origin)
    with pytest.raises(RuntimeError, match="nothing integrated"):
        m.synthesize_model_frame()
    V = oracle.o3d.Volume(res, vs, vs * 4.0, origin, with_color=True)
    poses = [np.linalg.inv(E) for E in sc["E"]]
    allocated = np.zeros((res // 16,) * 3, bool)
    for i in range(5):
        fr = FakeRGBD(sc["depth_u16"][i], sc["color"][i], 1000.0)
        m.integrate(fr, i, poses[i])
        _, touched = V.integrate_vbg(sc["depth_u16"][i], sc["K"], poses[i], rgb=sc["color"][i], depth_scale=1000.0, depth_max=fr.depth_max,
                                     trunc_voxel_multiplier=4.0, return_touched=True)
        touched = touched.astype(bool)
        allocated |= touched
        assert np.array_equal(m.allocated_blocks().cpu().numpy(), allocated)
        assert np.array_equal(m.allocated_blocks(last_frame=True).cpu().numpy(), touched)
        gpu = m.synthesize_model_frame()
        ref = raycast_ref.raycast_vbg(V, sc["K"], poses[i], 640, 480, allocated, touched, depth_scale=1000.0, weight_threshold=min(i, 3),
                                      trunc_voxel_multiplier=4.0)
        hit = assert_same(gpu, ref)
        if i >= 3:
            assert hit.mean() > 0.5, (i, hit.mean())
    g2 = m.synthesize_model_frame(depth_min=0.05, depth_max=0.3, enable_color=False, weight_threshold=1.0)
    assert "color" not in g2
    assert_same(g2, raycast_ref.raycast_vbg(V, sc["K"], poses[4], 640, 480, allocated, touched, depth_scale=1000.0, depth_min=0.05,
                                            depth_max=0.3, weight_threshold=1.0, trunc_voxel_multiplier=4.0, colors=False))


def test_raycast_rejections(cuda):
    sc = small_scene("laparoscopy512", res=32, frames=1)
    vl = sc["voxel_length"]
    plain = DenseTSDFVolume(vl, sc["sdf_trunc"], 64, sc["origin"], color=False, device="cuda:0")
    with pytest.raises(RuntimeError, match="colour"):
        plain.raycast(sc["intrinsic"], sc["E"][0], colors=True)
    with pytest.raises(RuntimeError, match="Unsupported image format"):
        plain.raycast((0, 480) + tuple(sc["K"]), sc["E"][0])
    with pytest.raises(RuntimeError, match="single-box"):
        DenseTSDFVolume(vl, sc["sdf_trunc"], (64, 64, 32), sc["origin"], color=False, device="cuda:0", gz0=32, z_total=64).raycast(
            sc["intrinsic"], sc["E"][0])
    with pytest.raises(RuntimeError, match="single-box"):
        DenseTSDFVolume(vl, sc["sdf_trunc"], (64, 64, 32), sc["origin"], color=False, device="cuda:0", z_total=64, z_interleave=2).raycast(
            sc["intrinsic"], sc["E"][0])
    with pytest.raises(RuntimeError, match="whole 8"):
        DenseTSDFVolume(vl, sc["sdf_trunc"], 60, sc["origin"], color=False, device="cuda:0").raycast(sc["intrinsic"], sc["E"][0])
    small = MAP(4, 4, k3x3(sc["K"]), "CUDA:0", 1000.0, resolution=64, color=False)
    small.integrate_batch(np.zeros((1, 4, 4), np.uint16), None, np.eye(4)[None], 1.0)
    with pytest.raises(RuntimeError, match="Unsupported image format"):
        small.synthesize_model_frame()
    L = _lib.load()
    m = MAP(640, 480, k3x3(sc["K"]), "CUDA:0", 1000.0, resolution=64, color=False)
    out = torch.empty(640 * 480 * 3, device=cuda)
    ws = torch.empty(L.bslam_vbg_raycast_workspace_bytes(480, 640), dtype=torch.uint8, device=cuda)
    K = np.asarray(sc["K"], np.float64)
    P = np.eye(4).reshape(-1)
    rc = L.bslam_vbg_raycast(m.model._h, _lib.ptr(m._ws), 480, 640, _lib.ptr(K), _lib.ptr(P), 1000.0, 0.1, 3.0, 0.0, 8.0, _lib.ptr(out), None, None,
                             _lib.ptr(out), _lib.ptr(ws), _lib.stream_ptr(cuda))
    assert rc == _lib.E_ARG and b"colour" in L.bslam_last_error()
