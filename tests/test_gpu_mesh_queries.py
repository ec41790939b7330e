"""Point and ray queries of `RaycastingScene` on the GPU (closest points, distances, occupancy, signed distances,
intersection counts, occlusion; csrc/bslam_mesh_raycast.cu) against the brute-force CPU reference
(tests/mesh_query_ref.c): every output equal as int32 bit patterns -- `-m gpu`."""
import numpy as np
import pytest
import torch

import mesh_query_ref as Q
import mesh_raycast_ref as R
from bodyslam_b200 import _lib
from bodyslam_b200 import synthetic as S
from bodyslam_b200.geometry import PinholeCameraIntrinsic
from bodyslam_b200.raycasting import RaycastingScene
from bodyslam_b200.tsdf import DenseTSDFVolume
from meshes import cube, icosphere, random_rays, soup
from test_gpu_mesh_raycast import special_rays

pytestmark = pytest.mark.gpu

CP_KEYS = ("points", "geometry_ids", "primitive_ids", "primitive_uvs", "primitive_normals")


def bits(x):
    if hasattr(x, "is_cuda"):
        x = x.contiguous()
        x = (x.to(torch.int32) if x.dtype == torch.bool else x.view(torch.int32)).cpu().numpy()
    x = np.ascontiguousarray(x)
    return x.astype(np.int32) if x.dtype == np.bool_ else x.view(np.int32)


def assert_bits(gpu, ref, what):
    g, r = bits(gpu), bits(ref)
    assert g.shape == r.shape, (what, g.shape, r.shape)
    bad = g != r
    assert not bad.any(), f"{what}: {bad.sum()} of {bad.size} values differ"


def scene_of(geoms, cuda):
    sc = RaycastingScene(cuda)
    for v, t in geoms:
        sc.add_triangles(v, t)
    return sc


def special_points(v, t, seed=0, closed=False):
    """on vertices, shared edges (midpoints), faces (random barycentric) and centroids, near and inside the scene box,
    far away (1e3, 1e30), equidistant from two triangles, NaN / inf"""
    rng = np.random.default_rng(seed)
    fin = np.isfinite(v).all(1)
    w = v[fin] if fin.any() else np.zeros((1, 3), np.float32)
    lo, hi = w.min(0), w.max(0)
    c, ext = 0.5 * (lo + hi), (hi - lo).max() + 1e-3
    out = [w[rng.choice(len(w), min(len(w), 128))]]                           # vertices
    if len(t):
        tri = v[t[rng.choice(len(t), min(len(t), 128))]]
        ok = np.isfinite(tri).all((1, 2))
        tri = tri[ok] if ok.any() else np.zeros((1, 3, 3), np.float32)
        out.append(0.5 * (tri[:, 0] + tri[:, 1]))                             # edges (shared in closed meshes)
        out.append(tri.mean(1))                                               # centroids
        b = rng.dirichlet([1, 1, 1], size=len(tri))
        out.append(np.einsum("nk,nkd->nd", b, tri.astype(np.float64)))        # on faces
        nrm = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
        nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-30)
        out.append(tri.mean(1) + 0.01 * ext * nrm)                           # just off faces
        if len(tri) > 1:
            out.append(0.5 * (tri[:-1].mean(1) + tri[1:].mean(1)))           # between two centroids
    out.append(rng.uniform(lo - 0.2 * ext, hi + 0.2 * ext, size=(512, 3)))   # near and inside the box
    if closed:
        out.append(c + 0.3 * ext * rng.uniform(-1, 1, size=(256, 3)))         # deep inside
    out.append(c + 1e3 * rng.normal(size=(32, 3)))
    out.append(1e30 * rng.normal(size=(8, 3)))
    out.append(np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [np.nan] * 3]))
    return np.ascontiguousarray(np.concatenate(out), dtype=np.float32)


def check_points(sc, geoms, pts, cuda, nsamples=(1, 3)):
    q = torch.as_tensor(pts, device=cuda)
    ref = Q.closest_points(geoms, pts)
    out = sc.compute_closest_points(q)
    assert set(out) == set(CP_KEYS)
    for k in CP_KEYS:
        assert_bits(out[k], ref[k], k)
    assert_bits(sc.compute_distance(q), ref["distance"], "distance")
    for ns in nsamples:
        occ, sd = Q.occupancy(geoms, pts, ns)
        assert_bits(sc.compute_occupancy(q, nsamples=ns), occ, f"occupancy nsamples={ns}")
        assert_bits(sc.compute_signed_distance(q, 0, ns), sd, f"signed distance nsamples={ns}")
    return ref


def check_rays(sc, geoms, rays, cuda):
    r = torch.as_tensor(rays, device=cuda)
    assert_bits(sc.count_intersections(r), Q.count_intersections(geoms, rays), "counts")
    assert_bits(sc.test_occlusions(r), Q.test_occlusions(geoms, rays), "occlusion [0, inf]")
    sub = rays[::max(1, len(rays) // 1000)]                                 # bounds exactly at hit values of these rays
    rs = torch.as_tensor(sub, device=cuda)
    t = R.cast_rays(geoms, sub)["t_hit"]
    hits = np.unique(t[np.isfinite(t)])
    picks = hits[np.linspace(0, len(hits) - 1, min(len(hits), 4)).astype(int)] if len(hits) else np.array([1.0], np.float32)
    for th in picks:
        th = float(th)
        for tnear, tfar in ((th, np.inf), (0.0, th), (th, th), (th, 0.5 * th), (float(np.nextafter(np.float32(th), np.float32(np.inf))), np.inf)):
            assert_bits(sc.test_occlusions(rs, tnear, tfar), Q.test_occlusions(geoms, sub, tnear, tfar), f"occlusion [{tnear}, {tfar}]")


def check(geoms, pts, rays, cuda, nsamples=(1, 3)):
    sc = scene_of(geoms, cuda)
    check_points(sc, geoms, pts, cuda, nsamples)
    check_rays(sc, geoms, rays, cuda)
    return sc


# ------------------------------------------------------------------ meshes


@pytest.mark.parametrize("n", [0, 1, 2, 3, 16, 17, 1024, 1025])
def test_small_soups(cuda, n):
    v, t = soup(max(n, 1), seed=n)
    v, t = v[:3 * n], t[:n]
    rays = np.concatenate([random_rays(2000, seed=n), special_rays(v, t, n) if n else random_rays(10, seed=1)])
    check([(v, t)], special_points(v, t, n), rays, cuda, nsamples=(1, 3, Q.MAX_SAMPLES))


@pytest.mark.parametrize("name", ["cube", "icosphere"])
def test_closed_meshes(cuda, name):
    v, t = cube() if name == "cube" else icosphere(3)
    pts = special_points(v, t, 1, closed=True)
    rays = np.concatenate([special_rays(v, t), random_rays(2000, seed=2)])
    check([(v, t)], pts, rays, cuda, nsamples=(1, 3, Q.MAX_SAMPLES))
    occ, _ = Q.occupancy([(v, t)], pts, 3)
    assert 0.1 < occ.mean() < 0.9


def test_marching_cubes_sphere(cuda):
    n, vl = 64, 0.01
    origin = np.array([-0.32, -0.32, -0.32])
    g = (np.arange(n) + 0.5) * vl
    X, Y, Z = np.meshgrid(g + origin[0], g + origin[1], g + origin[2], indexing="ij")
    tsdf = np.clip((np.sqrt(X ** 2 + Y ** 2 + Z ** 2) - 0.2) / (4 * vl), -1, 1).astype(np.float32)
    vol = DenseTSDFVolume(vl, 4 * vl, n, origin, color=False, device=cuda)
    vol.import_dense(tsdf, np.ones_like(tsdf))
    mesh = vol.extract_triangle_mesh()
    sc = RaycastingScene(cuda)
    sc.add_triangles(mesh)                                                    # CUDA tensors
    v, t = mesh.vertices.cpu().numpy(), mesh.triangles.cpu().numpy()
    geoms = [(v, t)]
    pts = special_points(v, t, 3, closed=True)
    check_points(sc, geoms, pts, cuda, nsamples=(1, 3))
    check_rays(sc, geoms, np.concatenate([special_rays(v, t, 3), random_rays(2000, seed=3, scale=0.3)]), cuda)
    occ, sd = Q.occupancy(geoms, pts, 3)
    r = np.linalg.norm(pts.astype(np.float64), axis=1)
    away = np.isfinite(r) & (np.abs(r - 0.2) > 2 * vl)
    assert np.array_equal(occ[away] == 1, r[away] < 0.2)


def test_soup_100k(cuda):
    v, t = soup(100_000, seed=7)
    pts = special_points(v, t, 7)
    rays = np.concatenate([random_rays(3000, seed=7), special_rays(v[np.isfinite(v).all(1)], t[:1000], 7)])
    sc = check([(v, t)], pts, rays, cuda, nsamples=(1,))
    sub = pts[::8]
    for ns in (3, Q.MAX_SAMPLES):
        occ, sd = Q.occupancy([(v, t)], sub, ns)
        assert_bits(sc.compute_signed_distance(torch.as_tensor(sub, device=cuda), nsamples=ns), sd, f"signed distance nsamples={ns}")


def test_equal_centroids_deepest_tree(cuda):
    rng = np.random.default_rng(5)
    n = 4000
    a = rng.integers(-100, 100, size=(n, 3)).astype(np.float32)
    b = rng.integers(-100, 100, size=(n, 3)).astype(np.float32)
    v = np.stack([a, b, -(a + b)], 1).reshape(-1, 3)                           # every centroid is exactly 0
    t = np.arange(3 * n, dtype=np.int32).reshape(n, 3)
    pts = np.concatenate([special_points(v, t, 5), np.zeros((4, 3), np.float32), rng.integers(-3, 3, size=(64, 3)).astype(np.float32)])
    check([(v, t)], pts, np.concatenate([random_rays(2000, seed=5, scale=150.0), special_rays(v, t, 5)]), cuda)


def test_several_geometries(cuda):
    c, ct = cube()
    s, st = icosphere(2)
    sv, stt = soup(500, seed=3)
    geoms = [(c, ct), (s[:0], st[:0]), (s * 0.4 + 0.5, st), (sv, stt), (c, ct)]     # an empty one and a duplicate
    pts = np.concatenate([special_points(c, ct, 3, closed=True), special_points(sv, stt, 4)])
    check(geoms, pts, np.concatenate([random_rays(2000, seed=3), special_rays(c, ct, 3)]), cuda, nsamples=(1, 3, Q.MAX_SAMPLES))
    ids = Q.closest_points(geoms, pts)["geometry_ids"]
    assert 4 not in set(ids.tolist()) and {0, 2, 3} <= set(ids.tolist())       # the duplicate of geometry 0 never wins


def test_equidistant_triangles(cuda):
    """mirror planes and duplicated triangles in both orders: ties of the key resolved to the smaller (g, p) whatever
    the traversal visits first"""
    v = np.array([[-1, -1, 0], [1, -1, 0], [1, 1, 0], [-1, 1, 0]], np.float32)
    t = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    geoms = [(v, np.concatenate([t[::-1]] * 3)), (v * [1, 1, -1] + [0, 0, 2], t), (v, t)]
    rng = np.random.default_rng(9)
    pts = np.concatenate([np.concatenate([rng.uniform(-1.5, 1.5, size=(500, 2)), np.full((500, 1), 1.0)], 1),
                          np.concatenate([rng.uniform(-1.5, 1.5, size=(500, 2)), rng.uniform(-1, 3, size=(500, 1))], 1),
                          v, 0.5 * (v + np.roll(v, 1, 0)), [[0, 0, 1], [0.5, 0.5, 1], [0, 0, 0]]]).astype(np.float32)
    check(geoms, pts, np.concatenate([random_rays(1000, seed=9), special_rays(v, t, 9)]), cuda)


def test_input_kinds_and_shapes(cuda):
    v, t = icosphere(1)
    sc = scene_of([(v, t)], cuda)
    pts = special_points(v, t, 11, closed=True)[:120]
    ref = Q.closest_points([(v, t)], pts)
    for q in (pts, torch.as_tensor(pts), torch.as_tensor(pts, device=cuda)):
        assert_bits(sc.compute_distance(q), ref["distance"], type(q).__name__)
    out = sc.compute_closest_points(torch.as_tensor(pts, device=cuda).reshape(2, 3, 20, 3))
    assert out["points"].shape == (2, 3, 20, 3) and out["primitive_ids"].shape == (2, 3, 20) and out["primitive_uvs"].shape == (2, 3, 20, 2)
    assert sc.compute_occupancy(pts.reshape(4, 30, 3), 0, 3).shape == (4, 30)
    rays = random_rays(60, seed=11).reshape(3, 20, 6)
    cnt, occl = sc.count_intersections(rays), sc.test_occlusions(rays, 0.0, 2.0, 0)
    assert cnt.shape == (3, 20) and cnt.dtype == torch.int32 and occl.dtype == torch.bool
    assert_bits(cnt, Q.count_intersections([(v, t)], rays), "counts")
    assert_bits(occl, Q.test_occlusions([(v, t)], rays, 0.0, 2.0), "occlusion")
    assert sc.compute_distance(np.zeros((0, 3), np.float32)).shape == (0,)               # zero queries
    assert sc.count_intersections(np.zeros((0, 6), np.float32)).shape == (0,)
    for wrong in (pts.astype(np.float64), pts[:, :2], pts.reshape(-1)):
        with pytest.raises(RuntimeError):
            sc.compute_distance(wrong)
    for ns in (0, 2, Q.MAX_SAMPLES + 1, 1.5):
        with pytest.raises(RuntimeError, match="nsamples"):
            sc.compute_occupancy(pts, nsamples=ns)
        with pytest.raises(RuntimeError, match="nsamples"):
            sc.compute_signed_distance(pts, nsamples=ns)
    for tnear, tfar in ((-1.0, 1.0), (float("nan"), 1.0), (0.0, float("nan"))):
        with pytest.raises(RuntimeError, match="bounds"):
            sc.test_occlusions(rays, tnear, tfar)


def test_lazy_commit_and_empty_scene(cuda):
    v, t = cube()
    sc = RaycastingScene(cuda)
    pts = np.array([[0.5, 0.5, 0.5], [2, 2, 2]], np.float32)
    assert torch.isinf(sc.compute_distance(pts)).all()
    assert (sc.compute_occupancy(pts) == 0).all() and (sc.count_intersections(random_rays(8)) == 0).all()
    assert (sc.compute_closest_points(pts)["geometry_ids"].view(torch.int32) == -1).all()
    sc.add_triangles(v, t)
    assert sc.compute_occupancy(pts).cpu().tolist() == [1.0, 0.0]
    sc.add_triangles(v * 0.5 + 0.25, t)
    geoms = [(v, t), (v * 0.5 + 0.25, t)]
    check_points(sc, geoms, special_points(v, t, 12, closed=True), cuda)


# ------------------------------------------------------------------ C ABI


def test_guard_bands_and_rejections(cuda):
    L = _lib.load()
    v, t = icosphere(1)
    sc = scene_of([(v, t)], cuda)
    bvh = sc._commit()
    pts = torch.as_tensor(special_points(v, t, 13, closed=True)[:100], device=cuda)
    rays = torch.as_tensor(random_rays(100, seed=13), device=cuda)
    n, G = 100, 64
    st = _lib.stream_ptr(cuda)
    ref = Q.closest_points([(v, t)], pts.cpu().numpy())
    occ, sd = Q.occupancy([(v, t)], pts.cpu().numpy(), 3)
    cnt = Q.count_intersections([(v, t)], rays.cpu().numpy())
    widths = {"points": 3, "geometry_ids": 1, "primitive_ids": 1, "primitive_uvs": 2, "primitive_normals": 3, "distance": 1, "occupancy": 1,
              "signed": 1, "counts": 1}
    bufs = {k: torch.full((G + n * w + G,), -7, dtype=torch.int32, device=cuda) for k, w in widths.items()}
    view = {k: bufs[k][G:G + n * w] for k, w in widths.items()}
    occl = torch.full((G + n + G,), 0xA5, dtype=torch.uint8, device=cuda)
    P = _lib.ptr
    _lib.check(L.bslam_mesh_closest_points(P(bvh), P(pts), n, *(P(view[k]) for k in CP_KEYS), st))
    _lib.check(L.bslam_mesh_distance(P(bvh), P(pts), n, P(view["distance"]), st))
    _lib.check(L.bslam_mesh_occupancy(P(bvh), P(pts), n, 3, P(view["occupancy"]), P(view["signed"]), st))
    _lib.check(L.bslam_mesh_count_intersections(P(bvh), P(rays), n, P(view["counts"]), st))
    _lib.check(L.bslam_mesh_test_occlusions(P(bvh), P(rays), n, 0.0, float("inf"), P(occl[G:G + n]), st))
    want = {**{k: ref[k] for k in CP_KEYS}, "distance": ref["distance"], "occupancy": occ, "signed": sd, "counts": cnt}
    for k in widths:
        assert np.array_equal(view[k].cpu().numpy(), bits(want[k]).reshape(-1)), k
        b = bufs[k].cpu().numpy()
        assert (b[:G] == -7).all() and (b[-G:] == -7).all(), f"{k} wrote outside its buffer"
    o = occl.cpu().numpy()
    assert np.array_equal(o[G:G + n], (cnt > 0).astype(np.uint8)) and (o[:G] == 0xA5).all() and (o[-G:] == 0xA5).all()
    # occupancy without the signed distance, and the directions
    only = torch.empty(n, dtype=torch.float32, device=cuda)
    _lib.check(L.bslam_mesh_occupancy(P(bvh), P(pts), n, 3, P(only), None, st))
    assert_bits(only, occ, "occupancy alone")
    d = np.empty((Q.MAX_SAMPLES, 3), np.float32)
    _lib.check(L.bslam_mesh_occupancy_directions(Q.MAX_SAMPLES, P(d)))
    assert np.array_equal(bits(d), bits(Q.directions()))
    # n = 0 accepts NULL; NULL required outputs, bad nsamples and bad bounds are argument errors
    for call in (lambda: L.bslam_mesh_closest_points(None, None, 0, None, None, None, None, None, st),
                 lambda: L.bslam_mesh_distance(None, None, 0, None, st),
                 lambda: L.bslam_mesh_occupancy(None, None, 0, 1, None, None, st),
                 lambda: L.bslam_mesh_count_intersections(None, None, 0, None, st),
                 lambda: L.bslam_mesh_test_occlusions(None, None, 0, 0.0, 1.0, None, st)):
        assert call() == _lib.OK
    E = _lib.E_ARG
    assert L.bslam_mesh_closest_points(P(bvh), P(pts), n, P(view["points"]), P(view["geometry_ids"]), P(view["primitive_ids"]), None,
                                       P(view["primitive_normals"]), st) == E
    assert L.bslam_mesh_distance(P(bvh), P(pts), n, None, st) == E
    assert L.bslam_mesh_distance(P(bvh), P(pts), -1, P(view["distance"]), st) == E
    assert L.bslam_mesh_occupancy(P(bvh), P(pts), n, 3, None, None, st) == E
    for ns in (0, 2, 32, 33, -1):
        assert L.bslam_mesh_occupancy(P(bvh), P(pts), n, ns, P(only), None, st) == E
    assert L.bslam_mesh_count_intersections(P(bvh), None, n, P(view["counts"]), st) == E
    for tnear, tfar in ((-1.0, 1.0), (float("nan"), 1.0), (0.0, float("nan"))):
        assert L.bslam_mesh_test_occlusions(P(bvh), P(rays), n, tnear, tfar, P(occl[G:G + n]), st) == E
    assert L.bslam_mesh_occupancy_directions(32, P(d)) == E
    torch.cuda.synchronize()
    assert bufs["counts"][:G].eq(-7).all()


# ------------------------------------------------------------------ full size


@pytest.mark.slow
def test_laparoscopy_mesh_full_size(cuda):
    """BASELINE configs[3] (laparoscopy512, 1000 frames) integrated in full, its ~1 M-triangle marching-cubes mesh:
    20 000 seeded points (near the surface and throughout the box) and 20 000 rays of a pose equal the brute force"""
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
    del vol
    v, t = mesh.vertices.cpu().numpy(), mesh.triangles.cpu().numpy()
    geoms = [(v, t)]
    sc = RaycastingScene(cuda)
    sc.add_triangles(mesh)
    rng = np.random.default_rng(0)
    lo = np.asarray(cfg["origin"], np.float64)
    hi = lo + cfg["resolution"] * cfg["voxel_length"]
    pts = np.concatenate([v[rng.choice(len(v), 10_000)] + rng.normal(scale=2 * cfg["voxel_length"], size=(10_000, 3)),
                          rng.uniform(lo, hi, size=(10_000, 3))]).astype(np.float32)
    q = torch.as_tensor(pts, device=cuda)
    ref = Q.closest_points(geoms, pts)                   # about 2e10 point-triangle pairs: one brute-force pass
    out = sc.compute_closest_points(q)
    for k in CP_KEYS:
        assert_bits(out[k], ref[k], k)
    assert_bits(sc.compute_distance(q), ref["distance"], "distance")
    sub = pts[::10]                                      # occupancy and signed distance on a 2 000-point subset
    occ, sd = Q.occupancy(geoms, sub, 1)
    assert_bits(sc.compute_signed_distance(torch.as_tensor(sub, device=cuda)), sd, "signed distance")
    assert_bits(sc.compute_occupancy(sub), occ, "occupancy")
    rays = R.rays_pinhole(intr.intrinsic_matrix, E[F // 2], W, H).reshape(-1, 6)[rng.choice(W * H, 20_000, replace=False)]
    r = torch.as_tensor(rays, device=cuda)
    assert_bits(sc.count_intersections(r), Q.count_intersections(geoms, rays), "counts")
    th = float(np.median(R.cast_rays(geoms, rays[:200])["t_hit"]))
    assert_bits(sc.test_occlusions(r[::10], 0.0, th), Q.test_occlusions(geoms, rays[::10], 0.0, th), "occlusion")
