"""The mesh ray cast's brute-force CPU reference (tests/mesh_raycast_ref.c) against closed forms -- no GPU needed."""
import numpy as np

import mesh_raycast_ref as R
from meshes import cube, icosphere, rays_through, watertight_rays

INVALID = 0xFFFFFFFF


def square(z=2.0, s=1.0):
    v = np.array([[-s, -s, z], [s, -s, z], [s, s, z], [-s, s, z]], np.float32)
    return v, np.array([[0, 1, 2], [0, 2, 3]], np.int32)


def test_plane_at_known_distance():
    rng = np.random.default_rng(1)
    xy = rng.uniform(-0.9, 0.9, size=(500, 2)).astype(np.float32)
    targets = np.concatenate([xy, np.full((500, 1), 2.0, np.float32)], 1)
    rays = rays_through([0, 0, 0], targets)
    out = R.cast_rays([square()], rays)
    assert np.all(out["geometry_ids"] == 0)
    np.testing.assert_allclose(out["t_hit"], 1.0, rtol=2e-6)                   # direction ends on the plane
    axis = R.cast_rays([square()], np.array([[0.25, 0.5, -3, 0, 0, 0.5]], np.float32))
    assert axis["t_hit"][0] == 10.0 and axis["geometry_ids"][0] == 0
    np.testing.assert_array_equal(np.abs(out["primitive_normals"][:, 2]), 1.0)


def test_closed_meshes_are_watertight():
    for (v, t), origins in ((cube(), [[0.5, 0.5, 0.5], [0.25, 0.5, 0.75], [0.1, 0.9, 0.3]]),
                            (icosphere(2), [[0, 0, 0], [0.3, -0.2, 0.1], [-0.5, 0.25, 0.4]])):
        for o in origins:
            rays = watertight_rays(v, t, o)
            out = R.cast_rays([(v, t)], rays)
            assert np.all(np.isfinite(out["t_hit"])), f"{np.sum(~np.isfinite(out['t_hit']))} rays escaped from {o}"
            assert np.all(out["primitive_ids"] < len(t))


def test_uv_reconstructs_the_hit_point():
    v, t = icosphere(1)
    rays = watertight_rays(v, t, [0.1, 0.2, -0.1], n_random=500)
    out = R.cast_rays([(v, t)], rays)
    tri = v[t[out["primitive_ids"].astype(np.int64)]].astype(np.float64)
    u, w = out["primitive_uvs"][:, 0:1].astype(np.float64), out["primitive_uvs"][:, 1:2].astype(np.float64)
    p_uv = (1 - u - w) * tri[:, 0] + u * tri[:, 1] + w * tri[:, 2]
    p_t = rays[:, :3].astype(np.float64) + out["t_hit"][:, None].astype(np.float64) * rays[:, 3:].astype(np.float64)
    assert np.abs(p_uv - p_t).max() < 1e-5
    n = out["primitive_normals"]
    np.testing.assert_allclose(np.linalg.norm(n, axis=1), 1.0, atol=1e-6)


def test_duplicates_resolve_to_the_smaller_id():
    v, t = square()
    dup = (v, np.concatenate([t, t]))
    rays = rays_through([0, 0, 0], [[0.3, -0.4, 2.0], [-0.5, 0.6, 2.0]])
    out = R.cast_rays([dup], rays)
    assert out["primitive_ids"].tolist() == [0, 1]
    out = R.cast_rays([(v[:0], t[:0]), dup, dup], rays)
    assert out["geometry_ids"].tolist() == [1, 1] and out["primitive_ids"].tolist() == [0, 1]
    # a shared edge: both triangles accept the ray, the smaller primitive wins
    out = R.cast_rays([square()], rays_through([0, 0, 0], [[0.5, 0.5, 2.0]]))
    assert out["primitive_ids"].tolist() == [0]


def test_degenerate_collinear_and_non_finite_triangles_never_hit():
    v = np.array([[0, 0, 2], [1, 0, 2], [1, 0, 2],           # two equal vertices
                  [0, 0, 2], [1, 1, 2], [2, 2, 2],           # collinear
                  [0, 0, 2], [0, 0, 2], [0, 0, 2],           # a point
                  [-1, -1, 2], [1, -1, 2], [np.nan, 1, 2],   # NaN
                  [-1, -1, 2], [np.inf, -1, 2], [0, 1, 2]],  # inf
                 np.float32)
    t = np.arange(15, dtype=np.int32).reshape(5, 3)
    targets = np.concatenate([v, [[0.5, 0, 2], [1, 1, 2], [0, -0.5, 2], [0.2, 0.1, 2]]]).astype(np.float32)
    out = R.cast_rays([(v, t)], rays_through([0.1, 0.05, 0], np.where(np.isfinite(targets), targets, 0)))
    assert np.all(np.isinf(out["t_hit"])) and np.all(out["geometry_ids"] == INVALID) and np.all(out["primitive_ids"] == INVALID)
    assert np.all(out["primitive_uvs"] == 0) and np.all(out["primitive_normals"] == 0)


def test_nan_zero_and_infinite_rays_miss():
    rays = np.array([[0, 0, 0, 0, 0, 1], [np.nan, 0, 0, 0, 0, 1], [0, 0, 0, 0, np.nan, 1], [0, 0, 0, 0, 0, 0],
                     [0, 0, 0, 0, 0, np.inf], [0, 0, -np.inf, 0, 0, 1]], np.float32)
    out = R.cast_rays([square()], rays)
    assert out["t_hit"][0] == 2.0
    assert np.all(np.isinf(out["t_hit"][1:])) and np.all(out["primitive_ids"][1:] == INVALID)


def test_ray_starting_on_a_triangle_hits_at_zero():
    rays = np.array([[0.25, -0.5, 2.0, 0.1, 0.2, 1.0], [0.25, -0.5, 2.0, 0.1, 0.2, -1.0], [0.25, -0.5, 2.0, 1.0, 0.0, 0.0]], np.float32)
    out = R.cast_rays([square()], rays)
    assert np.all(out["t_hit"][:2] == 0.0) and np.all(out["geometry_ids"][:2] == 0)
    assert np.isinf(out["t_hit"][2])                   # a ray lying in the triangle's plane: det = 0, no hit
    behind = R.cast_rays([square()], np.array([[0, 0, 2.5, 0, 0, 1]], np.float32))      # the plane lies behind: t < 0
    assert np.isinf(behind["t_hit"][0])


def test_pinhole_directions_have_unit_camera_z():
    K = np.array([[525.0, 0, 319.5], [0, 530.0, 241.25], [0, 0, 1]])
    rng = np.random.default_rng(3)
    for _ in range(3):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        w, x, y, z = q
        Rm = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                       [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                       [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
        E = np.eye(4)
        E[:3, :3], E[:3, 3] = Rm, rng.normal(size=3)
        rays = R.rays_pinhole(K, E, 64, 48)
        cam = rays[..., 3:].astype(np.float64) @ Rm.T
        np.testing.assert_allclose(cam[..., 2], 1.0, atol=1e-5)
        np.testing.assert_allclose(cam[..., 0], np.broadcast_to((np.arange(64) + 0.5 - 319.5) / 525.0, (48, 64)), atol=1e-5)
        np.testing.assert_allclose(rays[0, 0, :3], -Rm.T @ E[:3, 3], atol=1e-5)
    # t_hit of a fronto-parallel plane is its camera depth
    Kp = np.array([[100.0, 0, 16], [0, 100.0, 12], [0, 0, 1]])
    out = R.cast_rays([square(2.0, 5.0)], R.rays_pinhole(Kp, np.eye(4), 32, 24))
    np.testing.assert_allclose(out["t_hit"], 2.0, rtol=1e-6)
