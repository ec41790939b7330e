"""Ray casting of z-sharded legacy volumes (`ShardedTSDF.raycast`, bslam_tsdf_raycast_segment / _shade) -- `-m gpu`.

Single GPU: a volume is built as one box and its brick layers are copied into N slab volumes on the same device; a
test-local driver runs the rounds through the C entry points, with the all-reduce of the ray states and the composite
done as int32 sums of torch tensors.  Every map must equal `DenseTSDFVolume.raycast` of the box as int32 bit patterns.
Multi-GPU (`ShardedTSDF.raycast` over NCCL) runs when at least 2 GPUs are visible."""
import os
import socket

import numpy as np
import pytest
import torch

from bodyslam_b200 import _lib
from bodyslam_b200.sharding import slab_bounds
from bodyslam_b200.tsdf import DenseTSDFVolume
from test_gpu_raycast_edges import Analytic, ext_of, intr, look_at
from util import small_scene

pytestmark = pytest.mark.gpu


def slabs_of(box, bounds):
    """the box cut into contiguous slab volumes: every brick layer (voxels, colour, flags) copied as the re-shard does"""
    out = []
    src = box.storage_layers()
    for z0, z1 in bounds:
        s = DenseTSDFVolume(box.voxel_length, box.sdf_trunc, (box.nx, box.ny, z1 - z0), box.origin, color=box.color, device=box.device,
                            gz0=z0, z_total=box.nz)
        for k, dst in s.storage_layers().items():
            dst.copy_(src[k][z0 // 8:z1 // 8])
        out.append(s)
    return out


def cast_slabs(slabs, bounds, K6, E, depth_min=0.0, depth_max=3.0, depth_scale=1.0, weight_threshold=0.0, normals=True, colors=None):
    """ShardedTSDF.raycast's protocol on one device; -> (maps, rounds)"""
    N, dev = len(slabs), slabs[0].device
    E = np.asarray(E, np.float64).reshape(-1, 4, 4)
    W, H = K6[0], K6[1]
    F, n = E.shape[0], E.shape[0] * K6[0] * K6[1]
    colors = slabs[0].color if colors is None else colors
    z = np.asarray([b[0] for b in bounds] + [bounds[-1][1]], np.int32)
    state = torch.zeros(4 * n + 1, dtype=torch.int32, device=dev)
    rounds = 0
    while F and rounds < N:
        parts = []
        for s in slabs:
            st = state.clone()
            s.raycast_segment(st, z, rounds == 0, K6, E, depth_min, depth_max, weight_threshold)
            parts.append(st)
        state = torch.stack(parts).sum(0, dtype=torch.int32)
        rounds += 1
        if int(state[-1]) == 0:
            break
    assert F == 0 or int(state[-1]) == 0, "rays still marching after N rounds"
    keys = ["depth", "vertex"] + (["normal"] if normals else []) + (["color"] if colors else [])
    total = {k: torch.zeros(n * (1 if k == "depth" else 3), dtype=torch.int32, device=dev) for k in keys}
    for i, s in enumerate(slabs):
        lo = slabs[i - 1].raycast_halo(True) if i > 0 else None
        hi = slabs[i + 1].raycast_halo(False) if i + 1 < N else None
        out = {k: torch.full((n * (1 if k == "depth" else 3),), float("nan"), device=dev) for k in keys}
        s.raycast_shade(state, z, lo, hi, K6, E, out, depth_scale)
        for k in keys:
            assert not torch.isnan(out[k]).any(), f"{k}: pixels never written"
            total[k] += out[k].view(torch.int32)
    return {k: v.view(torch.float32).view((F, H, W) + (() if k == "depth" else (3,))) for k, v in total.items()}, rounds


def assert_bits(a, b):
    assert set(a) == set(b), (set(a), set(b))
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, k
        d = (a[k].contiguous().view(torch.int32) != b[k].contiguous().view(torch.int32))
        assert not d.any(), f"{k}: {int(d.sum())} elements differ"


def check(box, N, K6, E, **kw):
    bounds = slab_bounds(box.nz, N)
    maps, rounds = cast_slabs(slabs_of(box, bounds), bounds, K6, E, **kw)
    ref = box.raycast(K6, E, **kw)
    assert_bits(maps, ref)
    assert rounds <= N
    return ref


def poses(sc):
    """camera -> world: the analytic scene's own poses, then above and below the box looking along -z / +z, a camera
    on a slab boundary plane, rays with d_z == 0, grazing a boundary plane"""
    c, o, vl = sc.centre, sc.origin, sc.vl
    ext = np.array(sc.res) * vl
    P = list(sc.poses())
    P.append(look_at(c + np.array([0.01, 0.02, 2.0 * ext[2]]), c))                     # above, along -z
    P.append(look_at(c - np.array([0.02, -0.01, 2.0 * ext[2]]), c))                    # below, along +z
    zb = o[2] + 16 * vl                                                                 # a slab boundary plane
    P.append(look_at(np.array([c[0], c[1], zb]), c + np.array([0.0, 0.0, 0.3 * ext[2]])))
    flat = np.eye(4)                                                                    # optical axis along x: the centre row has d_z == 0
    flat[:3, :3] = np.array([[0.0, 0.0, 1.0], [0.0, 1.0, 0.0], [-1.0, 0.0, 0.0]])
    flat[:3, 3] = [o[0] - 0.05, c[1], o[2] + 24 * vl]
    P.append(flat)
    P.append(look_at(np.array([o[0] - 0.05, c[1], zb + 1e-4]), np.array([o[0] + ext[0], c[1] + 0.01, zb + 3e-4])))   # grazing
    return np.stack(P)


@pytest.fixture(scope="module")
def scene(cuda):
    sc = Analytic((64, 40, 96), holes=True, seed=11)
    return sc, sc.volume(cuda)


@pytest.mark.parametrize("N", [1, 2, 3, 8, 12])
def test_slabs_equal_the_box(scene, N):
    sc, box = scene
    ref = check(box, N, intr(33, 17), ext_of(poses(sc)))
    assert (ref["depth"] > 0).any(axis=(1, 2)).sum() >= 6


@pytest.mark.parametrize("N", [2, 5])
def test_camera_1km_away(scene, N):
    sc, box = scene
    P = look_at(sc.centre - 1000.0 * np.array([0.0, 0.6, 0.8]), sc.centre)
    ref = check(box, N, (33, 17, 1.5e5, 1.5e5, 16.3, 8.2), ext_of(P), depth_min=999.0, depth_max=1001.0, depth_scale=1000.0)
    assert (ref["depth"] > 0).any()


def test_plane_across_a_boundary(cuda):
    """a plane surface just above a slab boundary: hits whose sample and trilinear base lie in different slabs, and
    normals / colours whose corners straddle the boundary"""
    sc = Analytic((32, 32, 64), seed=4)
    z = np.arange(64)
    for zp in (16.0 - 0.5, 16.0 - 0.45, 16.0 + 0.3, 32.0 + 0.5):
        sc.tsdf[:] = np.clip((zp - (z + 0.5)) * sc.vl / sc.trunc, -1, 1).astype(np.float32)[None, None, :]
        box = sc.volume(cuda)
        P = [look_at(sc.origin + np.array([0.1, 0.1, -0.05]) + np.array([0.01 * i, 0.0, 0.0]), sc.origin + np.array([0.1 + 0.02 * i, 0.1, 0.1]))
             for i in range(4)]
        for N in (2, 4, 8):
            ref = check(box, N, intr(31, 9), ext_of(np.stack(P)))
            assert (ref["depth"] > 0).any(axis=(1, 2)).all()


def test_output_combinations_colour_and_thresholds(cuda):
    sc = Analytic((64, 40, 96), holes=True, seed=5)
    E = ext_of(poses(sc))
    for color in (True, False):
        box = sc.volume(cuda, color)
        for normals in (True, False):
            for colors in ((True, False) if color else (False,)):
                check(box, 3, intr(31, 9), E, normals=normals, colors=colors)
        for thr in (1.0, 2.0, 3.0):
            check(box, 4, intr(31, 9), E, weight_threshold=thr)


def test_depth_windows(scene):
    sc, box = scene
    E = ext_of(sc.front())
    z_c = float((E[:3, :3] @ sc.centre + E[:3, 3])[2])
    for lo, hi in ((z_c, z_c), (0.5, 0.1), (z_c - 0.9 * sc.R, z_c - 0.2 * sc.R), (z_c - 0.5 * sc.R, 3.0)):
        check(box, 4, intr(33, 17), E, depth_min=lo, depth_max=hi)


@pytest.mark.parametrize("F,W,H", [(0, 9, 17), (1, 1, 1), (65, 9, 17), (130, 9, 17), (2, 641, 479)])
def test_frames_and_image_sizes(cuda, F, W, H):
    sc = Analytic((16, 48, 24), holes=True, seed=3)
    box = sc.volume(cuda)
    a = np.linspace(0, 2 * np.pi, max(F, 1), endpoint=False)
    P = [look_at(sc.centre + (3.0 * sc.R + 0.05) * np.array([np.sin(t), 0.3 * np.cos(3 * t), -np.cos(t)]), sc.centre) for t in a[:F]]
    E = ext_of(np.stack(P)) if F else np.zeros((0, 4, 4))
    for N in (2, 3):
        ref = check(box, N, intr(W, H), E)
        assert ref["depth"].shape == (F, H, W)


def test_laparoscopy_scene(cuda):
    sc = small_scene("laparoscopy512", res=128, frames=6)
    from bodyslam_b200 import ops
    box = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 128, sc["origin"], color=True, device=cuda)
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    box.integrate_batch(depth, torch.as_tensor(sc["color"], device=cuda), sc["intrinsic"], sc["E"])
    for N in (2, 4, 8):
        ref = check(box, N, intr(160, 120), sc["E"], depth_min=0.01, depth_max=3.0)
        assert (ref["depth"] > 0).any()


def test_guard_bands_of_state_and_outputs(cuda):
    sc = Analytic((16, 48, 24), holes=True, seed=1)
    box = sc.volume(cuda)
    bounds = slab_bounds(24, 3)
    slabs = slabs_of(box, bounds)
    z = np.asarray([0, 8, 16, 24], np.int32)
    F, W, H = 3, 37, 23
    E = np.ascontiguousarray(ext_of(np.stack([look_at(sc.centre + np.array([0.01 * i, 0.0, -0.3]), sc.centre) for i in range(F)])).reshape(-1))
    K = np.array(intr(W, H)[2:], np.float64)
    n, pad = F * H * W, 4 * H * W + 256
    state = torch.full((4 * n + 1 + pad,), -7, dtype=torch.int32, device=cuda)
    L = _lib.load()
    rc = L.bslam_tsdf_raycast_segment(slabs[1]._h, 3, _lib.ptr(z), 1, F, H, W, _lib.ptr(K), _lib.ptr(E), 0.0, 3.0, 0.0, _lib.ptr(state), _lib.stream_ptr(cuda))
    assert rc == _lib.OK, L.bslam_last_error()
    assert (state[4 * n + 1:] == -7).all() and not (state[:4 * n] == -7).any()
    outs = {k: torch.full((c * (n + pad),), float("nan"), device=cuda) for k, c in (("depth", 1), ("vertex", 3), ("normal", 3), ("color", 3))}
    lo, hi = slabs[0].raycast_halo(True), slabs[2].raycast_halo(False)
    assert lo.numel() == L.bslam_tsdf_raycast_halo_bytes(slabs[0]._h, 1) and hi.numel() == L.bslam_tsdf_raycast_halo_bytes(slabs[2]._h, 2)
    rc = L.bslam_tsdf_raycast_shade(slabs[1]._h, 3, _lib.ptr(z), _lib.ptr(lo), _lib.ptr(hi), F, H, W, _lib.ptr(K), _lib.ptr(E), 1.0, _lib.ptr(state[:4 * n + 1]),
                                    *(_lib.ptr(outs[k]) for k in ("depth", "vertex", "normal", "color")), _lib.stream_ptr(cuda))
    assert rc == _lib.OK, L.bslam_last_error()
    for k, c in (("depth", 1), ("vertex", 3), ("normal", 3), ("color", 3)):
        assert not torch.isnan(outs[k][:c * n]).any() and torch.isnan(outs[k][c * n:]).all(), k


def test_rejections(cuda):
    sc = Analytic((16, 48, 24), seed=2)
    box = sc.volume(cuda)
    slabs = slabs_of(box, slab_bounds(24, 3))
    L = _lib.load()
    K = np.array(intr(9, 7)[2:], np.float64)
    E = np.ascontiguousarray(ext_of(sc.front()).reshape(-1))
    st = torch.zeros(4 * 63 + 1, dtype=torch.int32, device=cuda)
    out = torch.zeros(63, device=cuda)

    def seg(vol, z, F=1, state=st):
        z = np.asarray(z, np.int32)
        return L.bslam_tsdf_raycast_segment(vol._h, len(z) - 1, _lib.ptr(z), 1, F, 7, 9, _lib.ptr(K), _lib.ptr(E), 0.0, 3.0, 0.0, _lib.ptr(state),
                                            _lib.stream_ptr(cuda))

    def shade(vol, z, lo, hi, F=1):
        z = np.asarray(z, np.int32)
        return L.bslam_tsdf_raycast_shade(vol._h, len(z) - 1, _lib.ptr(z), _lib.ptr(lo), _lib.ptr(hi), F, 7, 9, _lib.ptr(K), _lib.ptr(E), 1.0,
                                          _lib.ptr(st), _lib.ptr(out), None, None, None, _lib.stream_ptr(cuda))

    assert seg(slabs[1], [0, 8, 16, 24]) == _lib.OK
    assert seg(slabs[1], [0, 8, 24]) == _lib.E_ARG                       # the slab is not one of the bounds
    assert seg(slabs[1], [0, 8, 12, 24]) == _lib.E_ARG                   # not whole bricks
    assert seg(slabs[1], [8, 16, 24]) == _lib.E_ARG                      # does not start at 0
    assert seg(slabs[1], [0, 16, 8, 24]) == _lib.E_ARG                   # not increasing
    inter = DenseTSDFVolume(sc.vl, sc.trunc, (16, 48, 8), sc.origin, color=True, device=cuda, gz0=8, z_total=24, z_interleave=3)
    assert seg(inter, [0, 8, 16, 24]) == _lib.E_ARG                      # interleaved box
    assert seg(slabs[1], [0, 8, 16, 24], F=0, state=None) == _lib.OK     # F = 0: NULL buffers, nothing launched
    lo, hi = slabs[0].raycast_halo(True), slabs[2].raycast_halo(False)
    assert shade(slabs[1], [0, 8, 16, 24], lo, hi) == _lib.OK
    assert shade(slabs[1], [0, 8, 16, 24], None, hi) == _lib.E_ARG      # missing halo below
    assert shade(slabs[1], [0, 8, 16, 24], lo, None) == _lib.E_ARG      # missing halo above
    assert shade(slabs[0], [0, 8, 16, 24], lo, slabs[1].raycast_halo(False)) == _lib.E_ARG   # a halo below the bottom slab
    assert shade(slabs[2], [0, 8, 16, 24], slabs[1].raycast_halo(True), None) == _lib.OK


# ------------------------------------------------------------------ multi-GPU: ShardedTSDF.raycast over NCCL
def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import sys
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from bodyslam_b200 import ops
        from bodyslam_b200.geometry import RGBDImage
        from bodyslam_b200.odometry import Method, rgbd_odometry_multi_scale
        from bodyslam_b200.sharding import ShardedTSDF
        from util import small_scene as scene_of
        sc = scene_of("laparoscopy512", res=128, frames=20)
        K6 = sc["intrinsic"]
        depth_all = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, dev)
        color_all = torch.as_tensor(sc["color"], device=dev)
        ok = True
        for layout in ("interleaved", "contiguous"):
            for color in (True, False):
                sh = ShardedTSDF(sc["voxel_length"], sc["sdf_trunc"], 128, sc["origin"], color=color, device=dev, rank=rank, world_size=world, layout=layout)
                sh.integrate_batch(depth_all[:6].clone(), color_all[:6].clone() if color else None, K6, sc["E"][:6])
                got = sh.raycast(K6, sc["E"][:6], depth_min=0.01, broadcast_from=0 if color else None)
                if rank == 0:
                    ref = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 128, sc["origin"], color=color, device=dev,
                                          unit_activation=sh.unit_activation)
                    ref.integrate_batch(depth_all[:6], color_all[:6] if color else None, K6, sc["E"][:6])
                    want = ref.raycast(K6, sc["E"][:6], depth_min=0.01)
                    ok = ok and set(got) == set(want) and all(torch.equal(got[k].view(torch.int32), want[k].view(torch.int32)) for k in want)
                else:
                    ok = ok and got is None

        # the dense SLAM loop on the sharded map: integrate, ray cast, track on rank 0 against the ray-cast map (world ->
        # camera extrinsics; the ray cast's vertex map is in the camera frame of the previous pose), integrate the new pose
        K3 = np.array([[K6[2], 0.0, K6[4]], [0.0, K6[3], K6[5]], [0.0, 0.0, 1.0]])

        def loop(cast, integrate):
            T = [np.asarray(sc["E"][0], np.float64)]
            maps = []
            integrate(0, T[0])
            for i in range(1, 20):
                m = cast(T[-1])
                Ti = None
                if m is not None:
                    maps.append({k: v.clone() for k, v in m.items()})
                    res = rgbd_odometry_multi_scale(RGBDImage(None, depth_all[i]), RGBDImage(None, m["depth"][0]), K3, depth_scale=1.0,
                                                    method=Method.PointToPlane)
                    Ti = np.linalg.inv(res.transformation) @ T[-1]      # frame i -> previous camera is M: E_i = M^-1 E_prev
                T.append(Ti)
                integrate(i, Ti)
            return T, maps

        sh = ShardedTSDF(sc["voxel_length"], sc["sdf_trunc"], 128, sc["origin"], color=True, device=dev, rank=rank, world_size=world)
        d = torch.empty_like(depth_all[0:1])
        c = torch.empty_like(color_all[0:1])

        def integ_sh(i, E):
            if rank == 0:
                d.copy_(depth_all[i:i + 1]); c.copy_(color_all[i:i + 1])
            sh.integrate_batch(d, c, K6, E if rank == 0 else np.zeros((1, 4, 4)), broadcast_from=0)

        T_sh, maps_sh = loop(lambda E: sh.raycast(K6, E if rank == 0 else None, depth_min=0.01, broadcast_from=0), integ_sh)
        if rank == 0:
            ref = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 128, sc["origin"], color=True, device=dev, unit_activation=sh.unit_activation)
            T_1, maps_1 = loop(lambda E: ref.raycast(K6, E, depth_min=0.01),
                               lambda i, E: ref.integrate_batch(depth_all[i:i + 1], color_all[i:i + 1], K6, np.asarray(E).reshape(1, 4, 4)))
            ok = ok and all(np.array_equal(a, b) for a, b in zip(T_sh, T_1)) and len(maps_sh) == len(maps_1) == 19
            ok = ok and all(torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)) for a, b in zip(maps_sh, maps_1) for k in b)
            ret.put(("ok" if ok else "sharded ray cast differs from the single-GPU ray cast", 0))
    except Exception as e:
        ret.put((f"rank {rank}: {type(e).__name__}: {e}", 0))
        raise
    finally:
        dist.destroy_process_group()


def test_sharded_raycast_multi_gpu():
    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
    msg, _ = ret.get(timeout=5)
    assert msg == "ok", msg
