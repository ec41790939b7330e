"""Mesh ray casting on the GPU (csrc/bslam_mesh_raycast.cu, `RaycastingScene`) against its brute-force CPU reference
(tests/mesh_raycast_ref.c): every output equal as int32 bit patterns -- `-m gpu`."""
import numpy as np
import pytest
import torch

import mesh_raycast_ref as R
from bodyslam_b200 import _lib
from bodyslam_b200 import synthetic as S
from bodyslam_b200.geometry import PinholeCameraIntrinsic, TriangleMesh
from bodyslam_b200.raycasting import RaycastingScene
from bodyslam_b200.tsdf import DenseTSDFVolume
from meshes import cube, icosphere, random_rays, soup, watertight_rays

pytestmark = pytest.mark.gpu

KEYS = ("t_hit", "geometry_ids", "primitive_ids", "primitive_uvs", "primitive_normals")
K640 = np.array([[525.0, 0, 319.5], [0, 525.0, 239.5], [0, 0, 1]])


def bits(x):
    if hasattr(x, "is_cuda"):
        x = x.contiguous().view(torch.int32).cpu().numpy()
    return np.ascontiguousarray(x).view(np.int32)


def assert_same(gpu, ref, keys=KEYS):
    for k in keys:
        g, r = bits(gpu[k]), bits(ref[k])
        assert g.shape == r.shape, (k, g.shape, r.shape)
        bad = g != r
        assert not bad.any(), f"{k}: {bad.sum()} of {bad.size} values differ"


def scene_of(geoms, cuda):
    sc = RaycastingScene(cuda)
    for v, t in geoms:
        sc.add_triangles(v, t)
    return sc


def check(geoms, rays, cuda):
    sc = scene_of(geoms, cuda)
    out = sc.cast_rays(torch.as_tensor(rays, device=cuda))
    ref = R.cast_rays(geoms, rays)
    assert_same(out, ref)
    return ref


def look_at(eye, target, up=(0.0, 0.0, 1.0)):
    """world -> camera extrinsic of a camera at eye looking at target (camera y down)"""
    eye, target = np.asarray(eye, float), np.asarray(target, float)
    z = target - eye
    z /= np.linalg.norm(z)
    x = np.cross(z, up)
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    E = np.eye(4)
    E[:3, :3] = np.stack([x, y, z])
    E[:3, 3] = -E[:3, :3] @ eye
    return E


def special_rays(v, t, seed=0):
    """axis-aligned, in a box face / triangle plane, from inside boxes and on triangles, at vertices and edges, NaN / 0"""
    rng = np.random.default_rng(seed)
    fin = v[np.isfinite(v).all(1)]
    lo, hi = fin.min(0), fin.max(0)
    c = 0.5 * (lo + hi)
    out = []
    for ax in range(3):
        for s in (1.0, -1.0):
            d = np.zeros(3, np.float32)
            d[ax] = s
            o = c.copy()
            o[ax] = lo[ax] - 1 if s > 0 else hi[ax] + 1
            pts = rng.uniform(lo, hi, size=(64, 3)).astype(np.float32)
            pts[:, ax] = o[ax]
            pts[:8] = v[rng.choice(len(v), 8)]                # through vertices along the axis
            pts[:8, ax] = o[ax]
            out.append(np.concatenate([pts, np.broadcast_to(d, pts.shape)], 1))
            face = pts.copy()
            face[:, (ax + 1) % 3] = lo[(ax + 1) % 3]          # lying in a face plane of the scene box
            out.append(np.concatenate([face, np.broadcast_to(d, pts.shape)], 1))
    tri = v[t[rng.choice(len(t), min(len(t), 64))]]
    tri = np.where(np.isfinite(tri), tri, 0.0)
    on = tri.mean(1)                                          # start on a triangle
    out.append(np.concatenate([on, rng.normal(size=on.shape)], 1))
    inplane = tri[:, 1] - tri[:, 0]                           # along a triangle's plane through its vertex
    out.append(np.concatenate([tri[:, 0] - inplane, inplane], 1))
    e = 0.5 * (tri[:, 0] + tri[:, 1])                         # at shared edges and vertices from outside
    src = c + 2.0 * (hi - lo + 1) * rng.normal(size=e.shape)
    out.append(np.concatenate([src, e - src], 1))
    out.append(np.concatenate([src, tri[:, 2] - src], 1))
    out.append(np.concatenate([rng.uniform(lo, hi, size=(64, 3)), rng.normal(size=(64, 3))], 1))   # inside boxes
    out.append(np.array([[np.nan, 0, 0, 0, 0, 1], [0, 0, 0, 0, 0, 0], [0, 0, 0, np.nan, 1, 0], [0, 0, 0, np.inf, 0, 0]]))
    return np.ascontiguousarray(np.concatenate(out), dtype=np.float32)


# ------------------------------------------------------------------ meshes


@pytest.mark.parametrize("n", [0, 1, 2, 3, 16, 17, 1024, 1025])
def test_small_soups(cuda, n):
    v, t = soup(max(n, 1), seed=n)
    v, t = v[:3 * n], t[:n]
    rays = np.concatenate([random_rays(3000, seed=n), special_rays(v, t, n) if n else random_rays(10, seed=1)])
    check([(v, t)], rays, cuda)


@pytest.mark.parametrize("name", ["cube", "icosphere"])
def test_closed_meshes(cuda, name):
    v, t = cube() if name == "cube" else icosphere(3)
    origin = [0.5, 0.4, 0.6] if name == "cube" else [0.1, -0.2, 0.05]
    rays = np.concatenate([watertight_rays(v, t, origin, 4000), special_rays(v, t)])
    ref = check([(v, t)], rays, cuda)
    assert np.isfinite(ref["t_hit"][:len(v)]).all()


def test_marching_cubes_sphere(cuda):
    n, vl = 64, 0.01
    origin = np.array([-0.32, -0.32, -0.32])
    g = (np.arange(n) + 0.5) * vl
    X, Y, Z = np.meshgrid(g + origin[0], g + origin[1], g + origin[2], indexing="ij")
    trunc = 4 * vl
    tsdf = np.clip((np.sqrt(X ** 2 + Y ** 2 + Z ** 2) - 0.2) / trunc, -1, 1).astype(np.float32)
    vol = DenseTSDFVolume(vl, trunc, n, origin, color=False, device=cuda)
    vol.import_dense(tsdf, np.ones_like(tsdf))
    mesh = vol.extract_triangle_mesh()
    assert mesh.triangles.shape[0] > 1000
    sc = RaycastingScene(cuda)
    assert sc.add_triangles(mesh) == 0                        # CUDA tensors, no host round trip
    v, t = mesh.vertices.cpu().numpy(), mesh.triangles.cpu().numpy()
    rays = np.concatenate([watertight_rays(v, t, [0.01, -0.02, 0.03], 4000), special_rays(v, t)])
    assert_same(sc.cast_rays(torch.as_tensor(rays, device=cuda)), R.cast_rays([(v, t)], rays))
    E = np.stack([look_at([0.6 * np.cos(a), 0.6 * np.sin(a), 0.2], [0, 0, 0]) for a in np.linspace(0, 6, 4)])
    out = sc.cast_pinhole(K640 * [[0.25], [0.25], [1]], E, 160, 120)
    ref = [R.cast_rays([(v, t)], R.rays_pinhole(K640 * [[0.25], [0.25], [1]], e, 160, 120)) for e in E]
    assert_same(out, {k: np.stack([r[k] for r in ref]) for k in KEYS})
    assert np.isfinite(ref[0]["t_hit"]).mean() > 0.2


def test_soup_100k(cuda):
    v, t = soup(100_000, seed=7)
    rays = np.concatenate([random_rays(6000, seed=7), special_rays(v[np.isfinite(v).all(1)], t[:1000], 7)])
    check([(v, t)], rays, cuda)


def test_equal_centroids_deepest_tree(cuda):
    rng = np.random.default_rng(5)
    n = 4000
    a = rng.integers(-100, 100, size=(n, 3)).astype(np.float32)
    b = rng.integers(-100, 100, size=(n, 3)).astype(np.float32)
    v = np.stack([a, b, -(a + b)], 1).reshape(-1, 3)           # integers: every centroid is exactly 0
    t = np.arange(3 * n, dtype=np.int32).reshape(n, 3)
    check([(v, t)], np.concatenate([random_rays(3000, seed=5, scale=150.0), special_rays(v, t, 5)]), cuda)


def test_several_geometries(cuda):
    c, ct = cube()
    s, st = icosphere(2)
    sv, stt = soup(500, seed=3)
    geoms = [(c, ct), (s[:0], st[:0]), (s * 0.4 + 0.5, st), (sv, stt), (c, ct)]   # an empty one and a duplicate
    rays = np.concatenate([random_rays(4000, seed=3), special_rays(c, ct, 3), watertight_rays(c, ct, [0.5, 0.5, 0.5], 500)])
    ref = check(geoms, rays, cuda)
    assert set(np.unique(ref["geometry_ids"])) >= {0, 2, 3}
    assert 4 not in set(ref["geometry_ids"].tolist())          # the duplicate of geometry 0 never wins


def test_input_kinds(cuda):
    v, t = icosphere(1)
    rays = watertight_rays(v, t, [0, 0, 0], 200)
    ref = R.cast_rays([(v, t)], rays)
    for tv, tt in ((v, t.astype(np.int64)), (v.astype(np.float64), t.astype(np.uint32)),
                   (torch.as_tensor(v), torch.as_tensor(t.astype(np.int64))), (torch.as_tensor(v, device=cuda), torch.as_tensor(t, device=cuda))):
        sc = RaycastingScene(cuda)
        sc.add_triangles(TriangleMesh(tv, tt))
        assert_same(sc.cast_rays(rays), ref)
    out = scene_of([(v, t)], cuda).cast_rays(torch.as_tensor(rays, device=cuda).reshape(2, -1, 6)[:, :7])
    assert out["t_hit"].shape == (2, 7) and out["primitive_normals"].shape == (2, 7, 3)


# ------------------------------------------------------------------ pinhole


@pytest.mark.parametrize("WH", [(1, 1), (2, 3), (31, 9), (33, 17), (160, 120), (641, 479)])
def test_pinhole_grids(cuda, WH):
    W, H = WH
    v, t = icosphere(2)
    K = np.array([[0.8 * W + 1, 0, W / 2], [0, 0.8 * W + 1, H / 2], [0, 0, 1]])
    E = look_at([2.5, 0.3, 0.4], [0, 0, 0])
    rays = RaycastingScene.create_rays_pinhole(K, E, W, H, device=cuda)
    ref_rays = R.rays_pinhole(K, E, W, H)
    assert np.array_equal(bits(rays), bits(ref_rays))
    sc = scene_of([(v, t)], cuda)
    ref = R.cast_rays([(v, t)], ref_rays)
    assert_same(sc.cast_rays(rays), ref)
    assert_same(sc.cast_pinhole(K, E, W, H), {k: x[None] for k, x in ref.items()})


@pytest.mark.parametrize("F", [0, 1, 65, 130])
def test_cast_pinhole_equals_cast_rays(cuda, F):
    v, t = icosphere(2)
    W, H = 40, 30
    K = np.array([[40.0, 0, 20], [0, 40.0, 15], [0, 0, 1]])
    a = np.linspace(0, 2 * np.pi, max(F, 1), endpoint=False)
    E = np.stack([look_at([2 * np.cos(x), 2 * np.sin(x), 0.3 * np.sin(3 * x)], [0.1, 0, 0]) for x in a])[:F].reshape(F, 4, 4)
    sc = scene_of([(v, t)], cuda)
    out = sc.cast_pinhole(PinholeCameraIntrinsic(W, H, 40.0, 40.0, 20, 15), E)
    assert out["t_hit"].shape == (F, H, W)
    if F == 0:
        return
    rays = torch.stack([RaycastingScene.create_rays_pinhole(K, e, W, H, device=cuda) for e in E])
    assert_same(out, sc.cast_rays(rays))
    depth_only = sc.cast_pinhole(K, E, W, H, uvs=False, normals=False)
    assert set(depth_only) == {"t_hit", "geometry_ids", "primitive_ids"}
    assert_same(depth_only, out, ("t_hit", "geometry_ids", "primitive_ids"))


# ------------------------------------------------------------------ C ABI


def test_guard_bands_and_rejections(cuda):
    L = _lib.load()
    v, t = icosphere(1)
    sc = scene_of([(v, t)], cuda)
    bvh = sc._commit()
    rays = torch.as_tensor(watertight_rays(v, t, [0, 0, 0], 100), device=cuda)
    n, G = rays.shape[0], 64
    ref = R.cast_rays([(v, t)], rays.cpu().numpy())
    bufs = {k: torch.full((G + n * w + G,), -7, dtype=torch.int32, device=cuda) for k, w in zip(KEYS, (1, 1, 1, 2, 3))}
    views = [bufs[k][G:G + n * w] for k, w in zip(KEYS, (1, 1, 1, 2, 3))]
    st = _lib.stream_ptr(cuda)
    _lib.check(L.bslam_mesh_cast_rays(_lib.ptr(bvh), _lib.ptr(rays), n, *(_lib.ptr(x) for x in views), st))
    for k, x in zip(KEYS, views):
        assert np.array_equal(x.cpu().numpy(), bits(ref[k]).reshape(-1)), k
    for k in KEYS:
        b = bufs[k].cpu().numpy()
        assert (b[:G] == -7).all() and (b[-G:] == -7).all(), f"{k} wrote outside its buffer"
    # n = 0 / F = 0 accept NULL; NULL with n > 0 is an argument error
    assert L.bslam_mesh_cast_rays(None, None, 0, None, None, None, None, None, st) == _lib.OK
    assert L.bslam_mesh_cast_pinhole(None, 0, 4, 4, None, None, None, None, None, None, None, st) == _lib.OK
    assert L.bslam_mesh_cast_rays(_lib.ptr(bvh), None, n, *(_lib.ptr(x) for x in views), st) == _lib.E_ARG
    assert L.bslam_mesh_cast_rays(_lib.ptr(bvh), _lib.ptr(rays), n, None, _lib.ptr(views[1]), _lib.ptr(views[2]), None, None, st) == _lib.E_ARG
    assert L.bslam_mesh_rays_pinhole(1, 4, 4, None, None, None, st) == _lib.E_ARG
    # an index out of range is found on the device and named
    bad = RaycastingScene(cuda)
    bad.add_triangles(v, t)
    bad.add_triangles(v, np.array([[0, 1, 2], [0, 1, len(v)]], np.int32))
    with pytest.raises(RuntimeError, match="triangle 1 of geometry 1"):
        bad.cast_rays(rays)
    neg = RaycastingScene(cuda)
    neg.add_triangles(v, np.array([[0, -1, 2]], np.int64))
    with pytest.raises(RuntimeError, match="out of range"):
        neg.cast_rays(rays)
    big = RaycastingScene(cuda)
    big.add_triangles(v, np.array([[0, 1, 2 ** 33]], np.int64))
    with pytest.raises(RuntimeError, match="out of range"):
        big.cast_rays(rays)
    for wrong in (rays.double(), rays[:, :5].contiguous(), rays.reshape(-1)):
        with pytest.raises(RuntimeError):
            sc.cast_rays(wrong)
    with pytest.raises(RuntimeError):
        sc.add_triangles(v, t.astype(np.float32))


def test_lazy_rebuild(cuda):
    v, t = cube()
    sc = RaycastingScene(cuda)
    rays = watertight_rays(v, t, [0.5, 0.5, 0.5], 100)
    a = sc.cast_rays(rays)
    assert torch.isinf(a["t_hit"]).all()                       # empty scene
    sc.add_triangles(v, t)
    assert torch.isfinite(sc.cast_rays(rays)["t_hit"]).all()
    assert sc.add_triangles(v * 0.5 + 0.25, t) == 1
    assert_same(sc.cast_rays(rays), R.cast_rays([(v, t), (v * 0.5 + 0.25, t)], rays))


# ------------------------------------------------------------------ full size


@pytest.mark.slow
def test_laparoscopy_mesh_full_size(cuda):
    """BASELINE configs[3] (laparoscopy512, 1000 frames) integrated in full, its ~1 M-triangle marching-cubes mesh cast at
    640 x 480: a seeded subset of 20 000 pixels equals the brute force; depth loosely agrees with the TSDF ray cast of
    the same volume (the mesh rays pass through pixel centres x + 0.5, the TSDF rays through x: a sub-pixel shift)"""
    cfg = S.config("laparoscopy512")
    F, W, H, Kt = cfg["frames"], cfg["W"], cfg["H"], cfg["K"]
    E = cfg["extrinsics"](F)
    intr = PinholeCameraIntrinsic(W, H, *Kt)
    depth_u16 = torch.empty((F, H, W), dtype=torch.uint16, device=cuda)
    for lo in range(0, F, 100):
        depth_u16[lo:lo + 100] = S.render(cfg["surface"], E[lo:lo + 100], K=Kt, W=W, H=H, device=cuda, with_color=False, first_frame=lo)[0]
    vol = DenseTSDFVolume(cfg["voxel_length"], cfg["sdf_trunc"], cfg["resolution"], cfg["origin"], color=False, device=cuda)
    vol.integrate_u16_chunks(depth_u16, None, intr, E, vol.stream_chunks(F), 1000.0, 3.0)
    del depth_u16
    mesh = vol.extract_triangle_mesh()
    assert mesh.triangles.shape[0] > 500_000
    sc = RaycastingScene(cuda)
    sc.add_triangles(mesh)
    pose = E[F // 2]
    out = sc.cast_pinhole(intr, pose)
    idx = np.random.default_rng(0).choice(W * H, 20_000, replace=False)
    rays = R.rays_pinhole(intr.intrinsic_matrix, pose, W, H).reshape(-1, 6)[idx]
    ref = R.cast_rays([(mesh.vertices.cpu().numpy(), mesh.triangles.cpu().numpy())], rays)
    # the subset is taken from the bit patterns on the host: torch has no CUDA indexing of uint32 tensors
    assert_same({k: bits(x).reshape((W * H,) + x.shape[3:])[idx] for k, x in out.items()}, ref)
    t = out["t_hit"][0].cpu().numpy()
    d = vol.raycast(intr, pose, normals=False, colors=False)["depth"][0].cpu().numpy()
    both = np.isfinite(t) & (d > 0)
    assert both.mean() > 0.5
    assert np.median(np.abs(t[both] - d[both])) < cfg["voxel_length"]
