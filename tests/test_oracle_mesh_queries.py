"""The mesh queries' brute-force CPU reference (tests/mesh_query_ref.c: closest points, distances, occupancy, signed
distances, intersection counts, occlusion) against closed forms -- no GPU needed."""
import numpy as np
import pytest

import mesh_query_ref as Q
import mesh_raycast_ref as R
from meshes import cube, icosphere, rays_through

INVALID = 0xFFFFFFFF
TRI = (np.array([[0, 0, 0], [2, 0, 0], [0, 2, 0]], np.float32), np.array([[0, 1, 2]], np.int32))


def square(z=2.0, s=1.0):
    v = np.array([[-s, -s, z], [s, -s, z], [s, s, z], [-s, s, z]], np.float32)
    return v, np.array([[0, 1, 2], [0, 2, 3]], np.int32)


def test_the_seven_voronoi_regions_of_a_triangle():
    # (query, closest point, uv = weights of v1, v2); every query sits 0.5 above or off the plane z = 0
    cases = [([-1, -1, 0.5], [0, 0, 0], [0, 0]),          # vertex v0
             ([3, -1, 0], [2, 0, 0], [1, 0]),             # vertex v1
             ([-1, 3, 0], [0, 2, 0], [0, 1]),             # vertex v2
             ([1, -1, 0], [1, 0, 0], [0.5, 0]),           # edge v0 v1
             ([-1, 1, 0], [0, 1, 0], [0, 0.5]),           # edge v0 v2
             ([2, 2, 0], [1, 1, 0], [0.5, 0.5]),          # edge v1 v2
             ([0.5, 0.5, 0.5], [0.5, 0.5, 0], [0.25, 0.25])]   # face
    q = np.array([c[0] for c in cases], np.float32)
    out = Q.closest_points([TRI], q)
    np.testing.assert_array_equal(out["points"], np.array([c[1] for c in cases], np.float32))
    np.testing.assert_array_equal(out["primitive_uvs"], np.array([c[2] for c in cases], np.float32))
    np.testing.assert_array_equal(out["distance"], np.linalg.norm(q - out["points"], axis=1).astype(np.float32))
    assert np.all(out["geometry_ids"] == 0) and np.all(out["primitive_ids"] == 0)
    np.testing.assert_array_equal(out["primitive_normals"], np.tile([0, 0, 1], (len(q), 1)).astype(np.float32))


def test_plane_at_known_distance():
    rng = np.random.default_rng(2)
    q = np.concatenate([rng.uniform(-0.9, 0.9, size=(300, 2)), rng.choice([-3.0, 0.5, 7.0], size=(300, 1))], 1).astype(np.float32)
    out = Q.closest_points([square(2.0)], q)
    np.testing.assert_allclose(out["distance"], np.abs(q[:, 2] - 2.0), rtol=1e-6)
    np.testing.assert_allclose(out["points"][:, :2], q[:, :2], atol=1e-6)
    assert np.all(out["points"][:, 2] == 2.0)
    np.testing.assert_array_equal(Q.count_intersections([square(2.0)], np.concatenate([q, np.tile([0, 0, 1], (300, 1))], 1)),
                                  (q[:, 2] <= 2.0).astype(np.int32))


@pytest.mark.parametrize("name", ["cube", "icosphere"])
def test_occupancy_and_sign_of_closed_meshes(name):
    rng = np.random.default_rng(4)
    if name == "cube":
        v, t = cube()
        p = rng.uniform(-0.5, 1.5, size=(3000, 3)).astype(np.float32)
        inside = np.all((p > 0) & (p < 1), axis=1)
        far = np.min(np.abs(np.concatenate([p, p - 1], 1)), axis=1) > 1e-3
    else:
        v, t = icosphere(3)
        p = rng.uniform(-1.5, 1.5, size=(3000, 3)).astype(np.float32)
        r = np.linalg.norm(p.astype(np.float64), axis=1)
        inside, far = r < 1, np.abs(r - 1) > 0.02             # the chords of icosphere(3) sag by < 0.005
    for ns in (1, 3, Q.MAX_SAMPLES):
        occ, sd = Q.occupancy([(v, t)], p, ns)
        np.testing.assert_array_equal(occ[far], inside[far].astype(np.float32))
        assert np.array_equal(np.signbit(sd[far]), inside[far])
    dist = Q.closest_points([(v, t)], p)["distance"]
    np.testing.assert_array_equal(np.abs(sd), dist)


def test_ray_through_a_closed_mesh_counts_two():
    for v, t in (cube(), icosphere(2)):
        c = v.mean(0)
        rays = rays_through(c + [5.0, 0.3, -0.2], [c + [0.01, -0.02, 0.03], c + [-0.1, 0.1, 0.05]])
        np.testing.assert_array_equal(Q.count_intersections([(v, t)], rays), [2, 2])
        back = rays.copy()
        back[:, 3:] *= -1                                      # pointing away: nothing at t >= 0
        np.testing.assert_array_equal(Q.count_intersections([(v, t)], back), [0, 0])
        inner = np.concatenate([np.tile(c, (2, 1)), rays[:, 3:]], 1)
        np.testing.assert_array_equal(Q.count_intersections([(v, t)], inner), [1, 1])


def test_shared_edge_counts_both_triangles():
    ray = np.array([[0.25, 0.25, 0, 0, 0, 1]], np.float32)    # through the diagonal of the square's two triangles
    assert Q.count_intersections([square()], ray)[0] == 2


def test_occlusion_bounds_are_inclusive():
    ray = np.array([[0.25, -0.5, -3.0, 0, 0, 0.5]], np.float32)     # hits z = 2 at t = 10 exactly
    assert R.cast_rays([square()], ray)["t_hit"][0] == 10.0
    sc = [square()]
    for tnear, tfar, want in ((0.0, np.inf, True), (10.0, 10.0, True), (0.0, 10.0, True), (10.0, np.inf, True),
                              (np.nextafter(np.float32(10), np.float32(20)), np.inf, False), (0.0, np.nextafter(np.float32(10), np.float32(0)), False),
                              (11.0, 9.0, False), (np.inf, np.inf, False)):
        assert Q.test_occlusions(sc, ray, tnear, tfar)[0] == want, (tnear, tfar)
    for tnear, tfar in ((-1.0, 1.0), (np.nan, 1.0), (0.0, np.nan)):
        with pytest.raises(ValueError):
            Q.test_occlusions(sc, ray, tnear, tfar)


def test_equidistant_triangles_resolve_to_the_smaller_id():
    v, t = square(0.0)
    out = Q.closest_points([(v, t)], np.array([[0.0, 0.0, 1.0], [0.5, 0.5, 0.0], [-1, -1, 3]], np.float32))
    assert out["primitive_ids"].tolist() == [0, 0, 0]
    dup = [(v, np.concatenate([t[::-1], t[::-1]])), (v, t)]
    out = Q.closest_points(dup, np.array([[0.5, -0.5, 1.0], [-0.5, 0.5, 1.0]], np.float32))
    assert out["geometry_ids"].tolist() == [0, 0] and out["primitive_ids"].tolist() == [1, 0]
    mirror = [(v, t), (v * [1, 1, -1] + [0, 0, 2], t)]           # planes z = 0 and z = 2, query at z = 1
    out = Q.closest_points(mirror, np.array([[0.3, -0.2, 1.0]], np.float32))
    assert out["geometry_ids"].tolist() == [0] and out["distance"][0] == 1.0


def test_non_finite_queries_and_the_empty_scene():
    q = np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [0.1, 0.2, 0.3]], np.float32)
    for geoms, n_bad in (([TRI], 3), ([], 4), ([(TRI[0][:0], TRI[1][:0])], 4)):
        out = Q.closest_points(geoms, q)
        assert np.all(np.isinf(out["distance"][:n_bad])) and np.all(out["distance"][:n_bad] > 0)
        assert np.all(out["geometry_ids"][:n_bad] == INVALID) and np.all(out["primitive_ids"][:n_bad] == INVALID)
        for k in ("points", "primitive_uvs", "primitive_normals"):
            assert np.all(out[k][:n_bad] == 0), k
        occ, sd = Q.occupancy(geoms, q, 3)
        assert np.all(occ[:n_bad] == 0) and np.all(sd[:n_bad] == np.inf)
    far = Q.closest_points([TRI], np.array([[3e38, 0, 0], [-3e38, -3e38, 0]], np.float32))
    assert np.all(far["distance"] == np.inf) and np.all(far["primitive_ids"] == 0)       # d^2 overflows: still the triangle
    assert np.all(np.isfinite(far["points"]))


def test_nsamples_must_be_odd_and_at_most_the_set():
    v, t = cube()
    q = np.array([[0.5, 0.5, 0.5]], np.float32)
    for ns in (0, 2, 4, Q.MAX_SAMPLES + 1, Q.MAX_SAMPLES + 2, -1):
        with pytest.raises(ValueError):
            Q.occupancy([(v, t)], q, ns)
    assert Q.occupancy([(v, t)], q, Q.MAX_SAMPLES)[0][0] == 1.0


def test_direction_set():
    d = Q.directions()
    assert d.shape == (Q.MAX_SAMPLES, 3) and d.dtype == np.float32
    np.testing.assert_allclose(np.linalg.norm(d.astype(np.float64), axis=1), 1.0, atol=1e-6)
    assert np.abs(d).min() >= 0.024 and np.abs(d).max() < 0.99        # off the coordinate planes and axes
    np.testing.assert_array_equal(Q.directions(5), d[:5])              # a prefix of one fixed sequence
    assert len(np.unique(d, axis=0)) == Q.MAX_SAMPLES
