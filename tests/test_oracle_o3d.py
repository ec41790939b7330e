"""The C oracle against closed-form expectations of the Open3D semantics it restates (CPU only)."""
import numpy as np
import pytest

import oracle
from bodyslam_b200 import synthetic as S

K = S.K_640


def plane_depth(z, H=480, W=640):
    return np.full((H, W), z, np.float32)


def test_depth_from_u16_scale_and_trunc():
    u = np.array([0, 1, 999, 1000, 2999, 3000, 3001, 65535], np.uint16)
    d = oracle.o3d.depth_from_u16(u, 1000.0, 3.0)
    assert d.dtype == np.float32
    assert np.array_equal(d, np.array([0, np.float32(1) / np.float32(1000), np.float32(999) / np.float32(1000), 1.0,
                                       np.float32(2999) / np.float32(1000), 0, 0, 0], np.float32))


def test_backproject_order_formula_and_inverse_extrinsic():
    d = np.zeros((4, 5), np.float32)
    d[1, 2], d[0, 4], d[3, 0] = 2.0, 1.0, 0.5
    fx, fy, cx, cy = 100.0, 110.0, 2.5, 1.5
    E = np.eye(4)
    E[:3, 3] = [0.1, -0.2, 0.3]
    th = 0.3
    E[:3, :3] = [[np.cos(th), -np.sin(th), 0], [np.sin(th), np.cos(th), 0], [0, 0, 1]]
    xyz, _ = oracle.o3d.backproject(d, (fx, fy, cx, cy), E)
    assert xyz.shape == (3, 3)                                   # row-major order of valid pixels
    want = []
    for (v, u) in ((0, 4), (1, 2), (3, 0)):
        z = float(d[v, u])
        p = np.array([(u - cx) * z / fx, (v - cy) * z / fy, z, 1.0])
        want.append((np.linalg.inv(E) @ p)[:3])
    assert np.allclose(xyz, np.array(want), atol=1e-15)
    full, _ = oracle.o3d.backproject(d, (fx, fy, cx, cy), E, valid_only=False)
    assert full.shape == (20, 3) and np.isnan(full).all(axis=1).sum() == 17
    s2, _ = oracle.o3d.backproject(d, (fx, fy, cx, cy), E, stride=2)
    assert len(s2) == 1                                          # only (0,4) lies on the stride-2 lattice


def test_integrate_plane_gives_analytic_tsdf_and_unit_weights():
    n, vl, trunc = 64, 0.004, 0.02
    V = oracle.o3d.Volume(n, vl, trunc, origin=(-0.128, -0.128, 0.0))
    upd = V.integrate(plane_depth(0.15), K, np.eye(4))
    w, t = V.grid("weight"), V.grid("tsdf")
    assert upd == int((w == 1).sum()) == V.occupied() and set(np.unique(w)) == {0.0, 1.0}
    # voxel on the optical axis column: sdf = (d - z) * ray multiplier, truncated to [-1, 1]
    fx, fy, cx, cy = K
    ix = iy = 32
    for iz in range(n):
        z = (iz + 0.5) * vl
        x, y = (ix + 0.5) * vl - 0.128, (iy + 0.5) * vl - 0.128
        uf, vf = x * fx / z + cx + 0.5, y * fy / z + cy + 0.5
        if not (0.0001 <= uf < 640 - 0.0001 and 0.0001 <= vf < 480 - 0.0001):
            assert w[ix, iy, iz] == 0                            # projects outside the image
            continue
        u, v = int(uf), int(vf)
        mult = np.sqrt(((u - cx) / fx) ** 2 + ((v - cy) / fy) ** 2 + 1)
        sdf = (0.15 - z) * mult
        if sdf > -trunc:
            assert w[ix, iy, iz] == 1 and abs(t[ix, iy, iz] - min(1.0, sdf / trunc)) < 1e-5
        else:
            assert w[ix, iy, iz] == 0
    # second identical frame: weights 2, tsdf unchanged (running mean of equal values)
    t0 = t.copy()
    V.integrate(plane_depth(0.15), K, np.eye(4))
    assert set(np.unique(V.grid("weight"))) == {0.0, 2.0} and np.abs(V.grid("tsdf") - t0).max() < 1e-6


def test_z_restart_modes_and_slab_mode_are_consistent():
    cfg = S.config("laparoscopy512")
    E = cfg["extrinsics"](1000)[[10, 500]]
    depth, _ = S.render(cfg["surface"], E, device="cpu", with_color=False)
    d = oracle.o3d.depth_from_u16(depth.numpy())
    args = dict(voxel_length=cfg["voxel_length"] * 8, sdf_trunc=cfg["sdf_trunc"] * 8, origin=cfg["origin"])
    lit = oracle.o3d.Volume(64, **args)
    brk = oracle.o3d.Volume(64, **args)
    for i in range(2):
        a = lit.integrate(d[i], cfg["K"], E[i], z_restart=0)
        b = brk.integrate(d[i], cfg["K"], E[i], z_restart=8)
        assert abs(a - b) <= 0.001 * a
    same = lit.weight == brk.weight
    assert same.mean() > 0.9995 and np.abs(lit.tsdf - brk.tsdf)[same].mean() < 1e-5
    # slab [32, 64) integrated on its own equals the slice of the full volume, in both modes
    for zr, full in ((8, brk), (0, lit)):
        slab = oracle.o3d.Volume((64, 64, 32), gz0=32, **args)
        for i in range(2):
            slab.integrate(d[i], cfg["K"], E[i], z_restart=zr)
        assert np.array_equal(slab.grid("weight"), full.grid("weight")[:, :, 32:])
        assert np.array_equal(slab.grid("tsdf"), full.grid("tsdf")[:, :, 32:])


def test_color_running_mean():
    V = oracle.o3d.Volume(32, 0.008, 0.04, origin=(-0.128, -0.128, 0.0), with_color=True)
    rgb = np.zeros((480, 640, 3), np.uint8)
    rgb[..., 0], rgb[..., 1] = 200, 100
    V.integrate(plane_depth(0.15), K, np.eye(4), rgb=rgb)
    rgb[..., 0] = 100
    V.integrate(plane_depth(0.15), K, np.eye(4), rgb=rgb)
    c = V.color.reshape(-1, 3)[V.weight == 2]
    assert np.allclose(c, [150, 100, 0])
    m = V.extract_mesh()
    assert np.allclose(m["colors"], np.array([150, 100, 0]) / 255.0)


def test_mesh_and_points_of_a_plane():
    n, vl = 48, 0.004
    V = oracle.o3d.Volume(n, vl, 0.02, origin=(-0.096, -0.096, 0.05))
    V.integrate(plane_depth(0.15), K, np.eye(4))
    m = V.extract_mesh()
    assert len(m["triangles"]) > 500
    assert np.abs(m["vertices"][:, 2] - 0.15).max() < 2e-4      # ray-distance sdf bends the plane slightly off-axis
    assert m["triangles"].min() == 0 and m["triangles"].max() == len(m["vertices"]) - 1
    p = V.extract_points()
    assert len(p["points"]) > 200 and np.abs(p["points"][:, 2] - 0.15).max() < 2e-4
    assert np.all(p["normals"][:, 2] < -0.99)                   # towards the camera
    assert np.all(p["keys"][:, 3] == 2)                         # crossings only along z


def test_weight_zero_corner_suppresses_cubes():
    n = 8
    V = oracle.o3d.Volume(n, 1.0, 1.0)
    z = (np.arange(n) + 0.5)[None, None, :] * np.ones((n, n, 1))
    V.tsdf[:] = np.clip((z - 4.0) / 2, -1, 1).astype(np.float32).reshape(-1)
    V.weight[:] = 1
    full = V.extract_mesh()
    assert len(full["triangles"]) == 2 * (n - 1) ** 2
    w = V.grid("weight")
    w[3, 3, 3] = 0                                               # kills the 4 cubes touching it in the crossing layer
    holed = V.extract_mesh()
    assert len(holed["triangles"]) == 2 * ((n - 1) ** 2 - 4)


def test_scalable_units_follow_the_sampled_points_closed_form():
    """orc_scalable_integrate (ScalableTSDFVolume, A.3 step 7): a fronto-parallel plane at depth d seen with
    identity pose activates exactly the units hit by floor((p -+ trunc) / unit_len) of the stride-8 points,
    leaves every other voxel at weight 0, and inside activated units equals the dense rule up to the
    per-unit evaluation of the voxel centres."""
    n, vl, trunc, d = 128, 0.002, 0.01, 0.15           # unit_len = 0.064, box = [-0.128, 0.128]^2 x [0, 0.256]
    org = (-0.128, -0.128, 0.0)
    V = oracle.o3d.Volume(n, vl, trunc, origin=org)
    D = oracle.o3d.Volume(n, vl, trunc, origin=org)
    upd, touched = V.integrate_scalable(plane_depth(d), K, np.eye(4), return_touched=True)
    D.integrate(plane_depth(d), K, np.eye(4))
    fx, fy, cx, cy = K
    ul = vl * 32
    want = np.zeros((4, 4, 4), bool)
    for i in range(0, 480, 8):
        for j in range(0, 640, 8):
            p = np.array([(j - cx) * d / fx, (i - cy) * d / fy, d])
            lo = np.floor((p - trunc) / ul).astype(int) - np.rint(np.array(org) / ul).astype(int)
            hi = np.floor((p + trunc) / ul).astype(int) - np.rint(np.array(org) / ul).astype(int)
            lo, hi = np.maximum(lo, 0), np.minimum(hi, 3)
            if np.all(lo <= hi):
                want[lo[0]:hi[0] + 1, lo[1]:hi[1] + 1, lo[2]:hi[2] + 1] = True
    assert np.array_equal(touched.astype(bool), want)
    assert want.sum() < want.size                      # the free space in front of the plane stays closed
    w = V.grid("weight")
    unit_of = lambda a: np.repeat(np.repeat(np.repeat(a, 32, 0), 32, 1), 32, 2)
    assert not w[~unit_of(want)].any()                 # un-activated units are never written
    assert upd == int((w > 0).sum())
    # inside the activated units: same voxels as the dense rule (the plane is far from any pixel border here)
    same_set = (w > 0) == ((D.grid("weight") > 0) & unit_of(want))
    assert same_set.mean() > 0.9999
    both = (w > 0) & (D.grid("weight") > 0)
    assert np.abs(V.grid("tsdf")[both] - D.grid("tsdf")[both]).max() < 2e-3


@pytest.mark.parametrize("pose", ["identity", "x90", "oblique"])
def test_scalable_activation_of_non_finite_huge_and_boundary_points(pose):
    """orc_scalable_integrate's activated units equal the NumPy restatement (tests/unit_activation_ref.py) for +-inf, NaN,
    -0, negative, subnormal, 1e30 and FLT_MAX depths (+inf also on the principal point) and for points whose w -+ trunc
    lands exactly on a unit face or one float32 step beside it; a non-finite world coordinate activates nothing"""
    import unit_activation_ref as ref
    rng = np.random.default_rng(len(pose))
    vl, ur, trunc = 1.0 / 64, 8, 1.0 / 16                 # unit 1/8 m: every face below is exact in f64
    dims, origin = (64, 64, 64), (-0.5, -0.5, -0.5)       # units -4 .. 3: global unit 0 inside the box
    if pose == "identity":
        R = np.eye(3)
    elif pose == "x90":
        R = np.array([[1.0, 0, 0], [0, 0, -1], [0, 1, 0]])
    else:
        q = rng.normal(size=4)
        a, b, c, d = q / np.linalg.norm(q)
        R = np.array([[a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c)],
                      [2 * (b * c + a * d), a * a - b * b + c * c - d * d, 2 * (c * d - a * b)],
                      [2 * (b * d - a * c), 2 * (c * d + a * b), a * a - b * b - c * c + d * d]])
    E = np.eye(4)
    E[:3, :3] = R.T
    E[:3, 3] = -R.T @ (-0.75 * R[:, 2])                    # 0.75 m behind the box centre, looking at it
    H = W = 16
    Kc = (12.0, 12.0, 8.0, 8.0)                            # the principal point is a sampled pixel (stride 2)
    vals = [np.nan, np.inf, -np.inf, -0.0, -0.25, 2.0 ** -149, 1e30, float(np.finfo(np.float32).max)]
    frames = []
    for k in range(3):
        d = np.zeros((H, W), np.float32)
        d[::2, ::2] = rng.choice(np.array(vals, np.float32), (H // 2, W // 2))
        d[8, 8] = np.inf
        frames.append(d)
    # on the optical axis w = -0.75 + depth along the view direction: w -+ trunc on the faces -1/8, 0, 1/8
    edges = sorted({np.float32(0.75 + f + s * trunc) for f in (-0.125, 0.0, 0.125) for s in (-1, 1)})
    d = np.zeros((H, W), np.float32)
    for n, z in enumerate(edges):
        d[0, 2 * n:2 * n + 2] = np.inf
        d[8, 8] = z
        for v in (np.nextafter(z, np.float32(0)), z, np.nextafter(z, np.float32(9))):
            e = d.copy()
            e[8, 8] = v
            frames.append(e)
    non_finite = 0
    for d in frames:
        V = oracle.o3d.Volume(dims, vl, trunc, origin)
        _, touched = V.integrate_scalable(d, Kc, E, unit_res=ur, stride=2, return_touched=True)
        want = ref.unit_activation(d, Kc, E, dims, vl, trunc, origin, ur, 2)
        assert np.array_equal(touched.astype(bool), want["touched"])
        w, finite = ref.sampled_world_points(d, Kc, E, 2)
        non_finite += int((~finite).sum())
        if finite.sum() == 0:
            assert not touched.any()
    assert non_finite > 30
    if pose != "oblique":
        # +inf on the principal point gives NaN on every axis under a pose of exact zeros
        w, finite = ref.sampled_world_points(frames[0], Kc, E, 2)
        assert np.isnan(w).all(axis=1).any()


def test_scalable_needs_whole_units_on_the_world_grid():
    V = oracle.o3d.Volume(72, 0.004, 0.02, origin=(-0.144,) * 3)
    with pytest.raises(ValueError):
        V.integrate_scalable(plane_depth(0.1), K, np.eye(4))
    V = oracle.o3d.Volume(64, 0.004, 0.02, origin=(-0.1,) * 3)
    with pytest.raises(ValueError):
        V.integrate_scalable(plane_depth(0.1), K, np.eye(4))


def test_cofactor_inverse_matches_lapack():
    import ctypes as C
    rng = np.random.default_rng(3)
    for _ in range(20):
        q, _r = np.linalg.qr(rng.normal(size=(3, 3)))
        E = np.eye(4)
        E[:3, :3] = q * np.sign(np.linalg.det(q))
        E[:3, 3] = rng.normal(size=3)
        out = np.zeros(16)
        oracle.o3d.lib().orc_invert4x4(E.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
        assert np.abs(out.reshape(4, 4) - np.linalg.inv(E)).max() < 1e-14


def test_scalable_all_units_is_the_dense_rule_with_per_unit_arithmetic():
    """`all_units=True` (the oracle of the product's unit_arithmetic mode): every unit is swept; it updates a superset of
    what the activation rule updates, with identical values wherever both updated a voxel equally often; and it differs
    from the brick-restart dense sweep only by float32 rounding of the voxel centres / the z recurrence"""
    from util import small_scene
    sc = small_scene("laparoscopy512", res=64, frames=3, with_color=False)
    ul = sc["voxel_length"] * 32
    origin = np.floor(sc["origin"] / ul + 0.5) * ul
    A = oracle.o3d.Volume(64, sc["voxel_length"], sc["sdf_trunc"], origin)
    S = oracle.o3d.Volume(64, sc["voxel_length"], sc["sdf_trunc"], origin)
    D = oracle.o3d.Volume(64, sc["voxel_length"], sc["sdf_trunc"], origin)
    for i in range(3):
        d = oracle.o3d.depth_from_u16(sc["depth_u16"][i])
        na = A.integrate_scalable(d, sc["K"], sc["E"][i], all_units=True)
        ns = S.integrate_scalable(d, sc["K"], sc["E"][i])
        nd = D.integrate(d, sc["K"], sc["E"][i], z_restart=8)
        assert na >= ns > 0 and abs(na - nd) <= 0.01 * nd
    assert np.all(A.weight >= S.weight)
    same = A.weight == S.weight
    assert np.array_equal(A.tsdf[same], S.tsdf[same])
    agree = A.weight == D.weight
    assert agree.mean() > 0.999 and np.abs(A.tsdf[agree] - D.tsdf[agree]).max() < 1e-3


def test_vbg_oracle_on_a_fronto_parallel_plane():
    """tensor-pipeline oracle (row f4): a plane at depth d seen from the identity pose -- voxels in front of it within
    the truncation get the projective sdf (d - z) / trunc, voxels more than trunc behind it are untouched, only blocks
    around the plane (and along the rays' [d - trunc, d + trunc] span) are activated"""
    vs, res = 0.01, 64
    origin = (-0.32, -0.32, 0.0)                   # blocks of 0.16 m: origin on the block grid
    V = oracle.o3d.Volume(res, vs, 0.04, origin)
    K = (300.0, 300.0, 159.5, 119.5)
    depth = np.full((240, 320), 400, np.uint16)    # 0.4 m
    n, touched = V.integrate_vbg(depth, K, np.eye(4), depth_scale=1000.0, depth_max=3.0, trunc_voxel_multiplier=4.0, return_touched=True)
    assert n > 1000
    zs = np.nonzero(touched.any(axis=(0, 1)))[0]
    assert zs.min() == 2 and zs.max() <= 2 + 1     # 0.36 .. 0.44 m lies in block z = 2 (0.32 .. 0.48 m)
    w, t = V.grid("weight"), V.grid("tsdf")
    x = y = res // 2                                # near the optical axis; voxel z index k sits at z = k * vs (corner convention)
    for k in range(32, 48):
        z = np.float32(k) * np.float32(vs)
        sdf = np.float32(0.4) - z
        if sdf < -0.04 - 1e-6:
            assert w[x, y, k] == 0
        elif abs(sdf) < 0.04 - 1e-6:
            assert w[x, y, k] == 1 and abs(t[x, y, k] - sdf / 0.04) < 1e-5
    assert w[x, y, 10] == 0                         # free space far in front: its block was never activated
    # depth_max cuts the frame off entirely
    V2 = oracle.o3d.Volume(res, vs, 0.04, origin)
    assert V2.integrate_vbg(depth, K, np.eye(4), depth_scale=1000.0, depth_max=0.3) == 0
    # the extraction flavour of the tensor pipeline (weight >= 3) drops once-seen surface, the legacy rule keeps it
    legacy = V.extract_mesh()
    oracle.o3d.set_extract_flavour(3.0, 0.0)
    try:
        thr = V.extract_mesh()
    finally:
        oracle.o3d.set_extract_flavour(0.0, 0.5)
    assert len(legacy["triangles"]) > 0 and len(thr["triangles"]) == 0
