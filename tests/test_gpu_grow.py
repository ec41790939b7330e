"""Box growth (`TSDF(grow=True)`, `DenseTSDFVolume.set_auto_grow` / `grow_to` / `unit_bounds`, bslam_tsdf_grow_box and the
relocating bslam_tsdf_copy).  "Equal" is always bit for bit (uint32 patterns); the reference each time is a fresh volume
created with the grown volume's final origin and resolution, given the same frames."""
import copy
import ctypes as C
import warnings

import numpy as np
import pytest
import torch

import oracle
from bodyslam_b200 import _lib, ops
from bodyslam_b200 import synthetic as S
from bodyslam_b200.geometry import PinholeCameraIntrinsic
from bodyslam_b200.tsdf import TSDF, DenseTSDFVolume

VL, TRUNC = 0.002, 0.01                 # 2 mm voxels, 64 mm units
START_RES, START_ORIGIN = 128, (-0.128,) * 3
N_FRAMES = 300


# ---------------------------------------------------------------- policy (host only)
def grow_box(u0, nu, lo, hi):
    L = _lib.load()
    u0, nu = np.array(u0, np.int64), np.array(nu, np.int64)
    b = np.ascontiguousarray(np.concatenate([lo, hi]).astype(np.int64))
    n0, n1, st = np.zeros(3, np.int64), np.zeros(3, np.int64), C.c_int()
    _lib.check(L.bslam_tsdf_grow_box(_lib.ptr(u0), _lib.ptr(nu), _lib.ptr(b), _lib.ptr(n0), _lib.ptr(n1), C.byref(st)))
    return st.value, n0.tolist(), n1.tolist()


def test_grow_box_policy_union_plus_a_quarter_per_moved_side():
    # already inside, or nothing requested: unchanged
    assert grow_box([-2] * 3, [4] * 3, [-2, -1, 0], [1, 1, 1]) == (_lib.GROW_OK, [-2] * 3, [4] * 3)
    assert grow_box([-2] * 3, [4] * 3, [5] * 3, [-5] * 3) == (_lib.GROW_OK, [-2] * 3, [4] * 3)
    # one unit beyond -x: union [-3, 1], slack max(1, 4 // 4) = 1 on that side only
    assert grow_box([-2] * 3, [4] * 3, [-3, 0, 0], [0, 0, 0]) == (_lib.GROW_GROWN, [-4, -2, -2], [6, 4, 4])
    # +z far away and -y: each moved side gets a quarter of the old extent on its axis
    assert grow_box([0, 0, 0], [16, 8, 16], [0, -1, 3], [3, 2, 40]) == (_lib.GROW_GROWN, [0, -3, 0], [16, 11, 45])
    # both sides of one axis
    assert grow_box([0, 0, 0], [8, 8, 8], [-1, 0, 0], [8, 0, 0]) == (_lib.GROW_GROWN, [-3, 0, 0], [14, 8, 8])


def test_grow_box_caps_drop_slack_then_refuse():
    # 65 536 units: the union reaching the cap exactly is granted without slack, one unit more is refused
    assert grow_box([0, 0, 0], [1, 1, 65530], [0, 0, 0], [0, 0, 65535]) == (_lib.GROW_GROWN, [0, 0, 0], [1, 1, 65536])
    assert grow_box([0, 0, 0], [1, 1, 65530], [0, 0, 0], [0, 0, 65536])[0] == _lib.GROW_CAP_UNITS
    # shared-memory rows nux * nuy * ceil(nuz / 32) <= 4096
    assert grow_box([0, 0, 0], [64, 63, 8], [0, 0, 0], [0, 63, 0]) == (_lib.GROW_GROWN, [0, 0, 0], [64, 64, 8])
    assert grow_box([0, 0, 0], [64, 63, 8], [0, 0, 0], [0, 64, 0])[0] == _lib.GROW_CAP_ROW_WORDS
    # the slack of a side that would break a cap is dropped, another side keeps its own
    assert grow_box([0, 0, 0], [64, 60, 8], [0, 0, 0], [0, 63, 8]) == (_lib.GROW_GROWN, [0, 0, 0], [64, 64, 11])
    # indices from a huge finite depth (clamped to +-2^40) are beyond every cap
    assert grow_box([0, 0, 0], [4, 4, 4], [0, 0, -(1 << 40)], [0, 0, 0])[0] == _lib.GROW_CAP_UNITS
    assert grow_box([0, 0, 0], [4, 4, 4], [0, 0, 0], [0, 0, 1 << 40])[0] == _lib.GROW_CAP_UNITS


def test_grow_box_rejects_a_box_that_already_breaks_a_cap():
    L = _lib.load()
    u0, nu, b = np.zeros(3, np.int64), np.array([1, 1, 65537], np.int64), np.zeros(6, np.int64)
    out, st = np.zeros(3, np.int64), C.c_int()
    assert L.bslam_tsdf_grow_box(_lib.ptr(u0), _lib.ptr(nu), _lib.ptr(b), _lib.ptr(out), _lib.ptr(out), C.byref(st)) == _lib.E_ARG


# ---------------------------------------------------------------- scenes
def _rot_y90():
    """world rotation p' = (z, y, -x): the lumen (which advances along +z and bends to +x) advances along +x' and bends to -z'"""
    R = np.eye(4)
    R[:3, :3] = [[0, 0, 1], [0, 1, 0], [-1, 0, 0]]
    return R


@pytest.fixture(scope="module")
def lumen(cuda):
    lum = S.Lumen()
    E_render = S.lumen_trajectory(lum, N_FRAMES, step=0.001)
    depth_u16, color = S.render(lum, E_render, device=cuda, seed=3)
    E = np.ascontiguousarray(E_render @ np.linalg.inv(_rot_y90()))     # world -> camera in the rotated world
    depth = ops.depth_from_u16(depth_u16, 1000.0, 3.0, cuda)
    return dict(E=E, depth_u16=depth_u16, color=color, depth=depth, intrinsic=PinholeCameraIntrinsic(640, 480, *S.K_640))


def _fresh(res, origin, cuda, color=True):
    return DenseTSDFVolume(VL, TRUNC, res, origin, color=color, device=cuda, unit_activation=True)


def _bits(t):
    return t.contiguous().view(torch.int32).cpu().numpy()


def assert_volumes_equal(a, b):
    assert (a.nx, a.ny, a.nz) == (b.nx, b.ny, b.nz) and np.array_equal(a.origin, b.origin)
    for x, y in zip(a.export_dense(True), b.export_dense(True)):
        assert np.array_equal(_bits(x), _bits(y))


def assert_points_equal(p, q):
    for f in ("points", "colors", "normals"):
        x, y = getattr(p, f), getattr(q, f)
        assert (x is None) == (y is None)
        if x is not None:
            assert np.array_equal(_bits(x), _bits(y)), f


def _box(vol):
    return tuple(vol.origin.tolist()), (vol.nx, vol.ny, vol.nz)


_REF = {}


def reference(sc, box, cuda, n=N_FRAMES):
    """pre-sized volume of box (origin, resolution) given frames [0, n) in one batch -> (volume, update counts)"""
    key = (box, n)
    if key not in _REF:
        v = _fresh(box[1], box[0], cuda)
        counts = torch.zeros(n, dtype=torch.int64, device=cuda)
        v.integrate_batch(sc["depth"][:n], sc["color"][:n], sc["intrinsic"], sc["E"][:n], update_counts=counts)
        _REF[key] = (v, counts.cpu().numpy())
    return _REF[key]


# ---------------------------------------------------------------- 1. trajectory
@pytest.mark.gpu
def test_lumen_trajectory_per_frame_equals_the_presized_box(lumen, cuda):
    from bodyslam_b200.geometry import RGBDImage
    t = TSDF(voxel_length=VL, sdf_trunc=TRUNC, resolution=START_RES, origin=START_ORIGIN, device=cuda, grow=True)
    history, snaps = [_box(t.tsdf)], {}
    for i in range(N_FRAMES):
        t.build_3D_map(RGBDImage(lumen["color"][i], lumen["depth"][i]), lumen["intrinsic"], lumen["E"][i])
        pcd = t.extract_pcd()
        if _box(t.tsdf) != history[-1]:
            history.append(_box(t.tsdf))
        if i in (40, 150):
            snaps[i] = (_box(t.tsdf), [x.clone() for x in t.tsdf.export_dense(True)], pcd)
    assert t.tsdf.frames_integrated == N_FRAMES and t.tsdf.growth_events == len(history) - 1
    # growth happened more than once, along more than one axis, toward negative unit indices too
    assert len(history) >= 3, history
    lo = np.array([h[0] for h in history])
    hi = lo + np.array([h[1] for h in history]) * VL
    d_lo, d_hi = np.diff(lo, axis=0), np.diff(hi, axis=0)
    assert (d_lo < 0).any() and ((d_lo < 0).any(axis=0) | (d_hi > 0).any(axis=0)).sum() >= 2, history
    # final state and every snapshot against pre-sized boxes
    ref, _ = reference(lumen, history[-1], cuda)
    assert_volumes_equal(t.tsdf, ref)
    assert_points_equal(t.extract_pcd(), ref.extract_point_cloud())
    for i, (box, dense, pcd) in snaps.items():
        r = _fresh(box[1], box[0], cuda)
        r.integrate_batch(lumen["depth"][:i + 1], lumen["color"][:i + 1], lumen["intrinsic"], lumen["E"][:i + 1])
        for x, y in zip(dense, r.export_dense(True)):
            assert np.array_equal(_bits(x), _bits(y)), i
        assert_points_equal(pcd, r.extract_point_cloud())
    # everything after growth: mesh, ray cast, deepcopy
    dims = (ref.nx, ref.ny, ref.nz)
    assert t.extract_mesh().canonical_digest(dims) == ref.extract_triangle_mesh().canonical_digest(dims)
    Ec = lumen["E"][::60]
    a, b = t.tsdf.raycast(lumen["intrinsic"], Ec), ref.raycast(lumen["intrinsic"], Ec)
    assert a.keys() == b.keys() and all(np.array_equal(_bits(a[k]), _bits(b[k])) for k in a)
    assert_volumes_equal(copy.deepcopy(t.tsdf), ref)


def _auto(cuda):
    v = _fresh(START_RES, START_ORIGIN, cuda)
    v.set_auto_grow(True)
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [64, 65, 257])
def test_lumen_integrate_batch_equals_the_presized_box(lumen, cuda, batch):
    v = _auto(cuda)
    counts = torch.zeros(N_FRAMES, dtype=torch.int64, device=cuda)
    for f0 in range(0, N_FRAMES, batch):
        f1 = min(f0 + batch, N_FRAMES)
        v.integrate_batch(lumen["depth"][f0:f1], lumen["color"][f0:f1], lumen["intrinsic"], lumen["E"][f0:f1], update_counts=counts[f0:f1])
    assert v.growth_events >= 1
    ref, ref_counts = reference(lumen, _box(v), cuda)
    assert_volumes_equal(v, ref)
    assert np.array_equal(counts.cpu().numpy(), ref_counts)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["u16_batch", "host", "u16_chunks"])
def test_lumen_u16_paths_equal_the_presized_box(lumen, cuda, path):
    v = _auto(cuda)
    counts = torch.zeros(N_FRAMES, dtype=torch.int64, device=cuda)
    d, c, K, E = lumen["depth_u16"], lumen["color"], lumen["intrinsic"], lumen["E"]
    if path == "u16_batch":
        for f0 in range(0, N_FRAMES, 100):
            v.integrate_u16_batch(d[f0:f0 + 100], c[f0:f0 + 100], K, E[f0:f0 + 100], update_counts=counts[f0:f0 + 100])
    elif path == "host":
        v.integrate_host(d.cpu().pin_memory(), c.cpu().pin_memory(), K, E, update_counts=counts)
        assert v.growth_events == 1         # all poses known up front: one bounds pass, one growth
    else:
        v.integrate_u16_chunks(d, c, K, E, v.stream_chunks(N_FRAMES), update_counts=counts)
    torch.cuda.synchronize()
    ref, ref_counts = reference(lumen, _box(v), cuda)
    assert_volumes_equal(v, ref)
    assert np.array_equal(counts.cpu().numpy(), ref_counts)


@pytest.mark.gpu
def test_unit_bounds_agree_across_depth_forms(lumen, cuda):
    v = _fresh(START_RES, START_ORIGIN, cuda)
    K, E = lumen["intrinsic"], lumen["E"][:70]
    b = v.unit_bounds(lumen["depth"][:70], K, E)
    assert b is not None and np.array_equal(b, v.unit_bounds(lumen["depth_u16"][:70], K, E))
    assert np.array_equal(b, v.unit_bounds(lumen["depth_u16"][:70, ::8, ::8].contiguous(), K, E, sampled=True))
    assert np.array_equal(b, v.unit_bounds(lumen["depth"][:70, ::8, ::8].contiguous(), K, E, sampled=True))


# ---------------------------------------------------------------- 2. oracle
@pytest.mark.gpu
def test_short_grown_sequence_equals_the_oracle(lumen, cuda):
    v = _auto(cuda)
    ids = list(range(0, 160, 10))          # 16 frames
    for i in ids:
        v.integrate_batch(lumen["depth"][i:i + 1], lumen["color"][i:i + 1], lumen["intrinsic"], lumen["E"][i:i + 1])
    assert v.growth_events >= 1
    V = oracle.o3d.Volume((v.nx, v.ny, v.nz), VL, TRUNC, v.origin, with_color=True)
    K = S.K_640
    for i in ids:
        V.integrate_scalable(lumen["depth"][i].cpu().numpy(), K, lumen["E"][i], rgb=lumen["color"][i].cpu().numpy())
    t, w, c = v.export_dense(True)
    assert np.array_equal(_bits(t).reshape(-1), V.tsdf.view(np.int32))
    assert np.array_equal(_bits(w).reshape(-1), V.weight.view(np.int32))
    assert np.array_equal(_bits(c).reshape(-1), V.color.view(np.int32))


# ---------------------------------------------------------------- 3. boundaries
UL = 0.5                 # voxel 2^-6 m, unit 0.5 m, trunc 2^-4 m: every boundary below is exact in f64
BVL, BTRUNC = 1.0 / 64, 1.0 / 16
BK = PinholeCameraIntrinsic(8, 8, 100.0, 100.0, 0.0, 0.0)     # stride 8: only pixel (0, 0) is sampled, at x = y = 0


def _face_pose(axis, sign):
    """world -> camera pose whose optical axis is sign * e_axis (camera at the world origin)"""
    R = np.zeros((3, 3))
    R[:, 2] = 0
    R[axis, 2] = sign
    others = [a for a in range(3) if a != axis]
    R[others[0], 0] = 1
    R[others[1], 1] = 1
    if np.linalg.det(R) < 0:
        R[others[0], 0] = -1
    c2w = np.eye(4)
    c2w[:3, :3] = R
    return np.linalg.inv(c2w)


def _small_box(cuda):
    v = DenseTSDFVolume(BVL, BTRUNC, 64, (-UL,) * 3, color=False, device=cuda, unit_activation=True)     # units -1, 0
    v.set_auto_grow(True)
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("sign", [1, -1])
def test_planes_on_unit_boundaries_grow_exactly_when_a_unit_outside_is_activated(cuda, axis, sign):
    # w = sign * z.  +face: w + trunc = 0.5 activates unit 1 (outside), one f32 step less does not.
    # -face: w - trunc = -0.5 stays in unit -1 (inside), one f32 step more reaches unit -2 (outside).
    z_edge = np.float32(UL - BTRUNC)
    cases = [(z_edge, sign > 0), (np.nextafter(z_edge, np.float32(0)), False), (np.nextafter(z_edge, np.float32(1)), True)]
    for z, grows in cases:
        v = _small_box(cuda)
        d = torch.zeros((1, 8, 8), dtype=torch.float32, device=cuda)
        d[0, 0, 0] = float(z)
        E = _face_pose(axis, sign)[None]
        b = v.unit_bounds(d, BK, E)
        w = sign * float(z)
        expect_lo, expect_hi = np.floor((w - BTRUNC) / UL), np.floor((w + BTRUNC) / UL)
        assert b[0, axis] == expect_lo and b[1, axis] == expect_hi
        v.integrate_batch(d, None, BK, E)
        if grows:
            # the policy: the side that moved gains its unit plus max(1, 2 // 4) = 1 unit of slack
            assert v.growth_events == 1
            n = [2, 2, 2]
            n[axis] = 4
            assert (v.nx, v.ny, v.nz) == tuple(32 * k for k in n)
            assert v.origin[axis] == (-UL if sign > 0 else -3 * UL)
        else:
            assert v.growth_events == 0 and (v.nx, v.ny, v.nz) == (64, 64, 64)


@pytest.mark.gpu
def test_invalid_and_non_finite_depths_cause_no_growth(cuda):
    E = _face_pose(2, 1)[None]
    for val in [0.0, float("nan"), -0.0, -5.0, float("inf"), float("-inf")]:
        v = _small_box(cuda)
        d = torch.full((1, 8, 8), val, dtype=torch.float32, device=cuda)
        assert v.unit_bounds(d, BK, E) is None
        v.integrate_batch(d, None, BK, E)
        assert v.growth_events == 0 and v.grow_capped is None
    # 1e30 m: far beyond the caps, clamped instead of wrapped; the box stays and the point is counted as clipped
    v = _small_box(cuda)
    d = torch.full((1, 8, 8), 1e30, dtype=torch.float32, device=cuda)
    b = v.unit_bounds(d, BK, E)
    assert b[0, 2] == 1 << 40 and b[1, 2] == 1 << 40
    v.integrate_batch(d, None, BK, E)
    assert v.growth_events == 0 and v.grow_capped is not None and v.clip_stats()["outside"] == 1


# ---------------------------------------------------------------- 4. caps
@pytest.mark.gpu
def test_largest_policy_boxes_are_accepted_by_unit_activation_and_one_more_unit_is_not(cuda):
    # 65 536 units (nuz through z_total, so that the box itself stays small)
    st, _, nu = grow_box([0, 0, 0], [1, 1, 65535], [0, 0, 0], [0, 0, 65535])
    assert st == _lib.GROW_GROWN and nu == [1, 1, 65536]
    for nuz, ok in [(65536, True), (65537, False)]:
        v = DenseTSDFVolume(0.001, 0.004, 32, (0.0, 0.0, 0.0), color=False, device=cuda, z_total=32 * nuz)
        if ok:
            v.set_unit_activation(32, 8)
        else:
            with pytest.raises(RuntimeError, match="too many units"):
                v.set_unit_activation(32, 8)
    # nux * nuy * ceil(nuz / 32) = 4096
    st, _, nu = grow_box([0, 0, 0], [64, 63, 1], [0, 0, 0], [0, 63, 0])
    assert st == _lib.GROW_GROWN and nu == [64, 64, 1]
    for nx, ok in [(2048, True), (2080, False)]:
        v = DenseTSDFVolume(0.001, 0.004, (nx, 2048, 8), (0.0, 0.0, 0.0), color=False, device=cuda, z_total=32)
        if ok:
            v.set_unit_activation(32, 8)
        else:
            with pytest.raises(RuntimeError, match="too many units"):
                v.set_unit_activation(32, 8)
        del v


@pytest.mark.gpu
def test_request_beyond_the_caps_keeps_the_box_counts_and_warns(lumen, cuda):
    d = lumen["depth"][:4].clone()
    d[:, 100:400, :] = 1e30          # most sampled points far beyond the caps
    t = TSDF(voxel_length=VL, sdf_trunc=TRUNC, resolution=START_RES, origin=START_ORIGIN, device=cuda, grow=True)
    from bodyslam_b200.geometry import RGBDImage
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        for i in range(4):
            t.build_3D_map(RGBDImage(lumen["color"][i], d[i]), lumen["intrinsic"], lumen["E"][i])
            t.extract_pcd()
    assert t.tsdf.growth_events == 0 and t.tsdf.grow_capped is not None and t.clipped_fraction() > 0.5
    assert any("could not grow" in str(w.message) and "65 536" in str(w.message) for w in rec)
    ref = _fresh(START_RES, START_ORIGIN, cuda)
    ref.integrate_batch(d, lumen["color"][:4], lumen["intrinsic"], lumen["E"][:4])
    assert_volumes_equal(t.tsdf, ref)


# ---------------------------------------------------------------- 5. relocation
def _random_state(res, color, seed):
    g = np.random.default_rng(seed)
    n = int(np.prod(res))
    t = g.uniform(-1, 1, n).astype(np.float32)
    w = np.where(g.random(n) < 0.3, 0.0, g.integers(1, 200, n)).astype(np.float32)
    c = g.uniform(0, 255, (n, 3)).astype(np.float32) if color else None
    return t, w, c


@pytest.mark.gpu
@pytest.mark.parametrize("color", [False, True])
@pytest.mark.parametrize("src_res,dst_res,off", [
    ((32, 32, 32), (64, 64, 64), (0, 0, 0)),
    ((32, 32, 32), (64, 64, 64), (4, 0, 4)),
    ((24, 40, 16), (56, 48, 40), (1, 1, 3)),
    ((16, 16, 16), (16, 320, 320), (0, 17, 38)),        # 1600 brick rows: more than the kernel's grid
    ((8, 8, 8), (1032, 16, 8), (128, 1, 0)),            # one row of 129 bricks: longer than a 256-thread chunk
])
def test_relocation_pads_with_reset_values(cuda, color, src_res, dst_res, off):
    L = _lib.load()
    vl = 0.01
    o_src = np.array([0.08, -0.16, 0.24])
    o_dst = o_src - np.array(off) * 8 * vl
    src = DenseTSDFVolume(vl, 0.04, src_res, o_src, color=color, device=cuda)
    dst = DenseTSDFVolume(vl, 0.04, dst_res, o_dst, color=color, device=cuda)
    t, w, c = _random_state(src_res, color, sum(src_res) + sum(off))
    src.import_dense(t, w, c)
    _lib.check(L.bslam_tsdf_copy(src._h, dst._h, _lib.stream_ptr(cuda)))
    sl = tuple(slice(8 * o, 8 * o + n) for o, n in zip(off, src_res))
    exp_t, exp_w = np.zeros(dst_res, np.float32), np.zeros(dst_res, np.float32)
    exp_t[sl], exp_w[sl] = t.reshape(src_res), w.reshape(src_res)
    out = dst.export_dense(True)
    assert np.array_equal(_bits(out[0]), exp_t.view(np.int32)) and np.array_equal(_bits(out[1]), exp_w.view(np.int32))
    if color:
        exp_c = np.zeros(dst_res + (3,), np.float32)
        exp_c[sl] = c.reshape(src_res + (3,))
        assert np.array_equal(_bits(out[2]), exp_c.view(np.int32))
    # brick flags, seen through the storage layers ([bz, by * nbx + bx])
    fs = src.storage_layers()["flags"].cpu().numpy()
    sb = [n // 8 for n in src_res]
    db = [n // 8 for n in dst_res]
    exp_f = np.zeros((db[2], db[1], db[0]), np.uint8)
    exp_f[off[2]:off[2] + sb[2], off[1]:off[1] + sb[1], off[0]:off[0] + sb[0]] = fs.reshape(sb[2], sb[1], sb[0])
    assert np.array_equal(dst.storage_layers()["flags"].cpu().numpy().reshape(db[2], db[1], db[0]), exp_f)
    # equal geometry: the plain copy, unchanged
    same = copy.deepcopy(src)
    for x, y in zip(same.export_dense(True), src.export_dense(True)):
        assert np.array_equal(_bits(x), _bits(y))


@pytest.mark.gpu
def test_relocation_into_a_box_that_does_not_contain_the_source_is_an_argument_error(cuda):
    L = _lib.load()
    src = DenseTSDFVolume(0.01, 0.04, 32, (0.0, 0.0, 0.0), color=False, device=cuda)
    for res, origin in [((64, 64, 64), (0.01, 0.0, 0.0)),        # not a whole brick apart
                        ((64, 64, 64), (0.08, 0.0, 0.0)),        # source starts before the destination
                        ((64, 64, 40), (0.0, 0.0, -0.16)),       # source sticks out at the top
                        ((16, 64, 64), (0.0, 0.0, 0.0))]:        # smaller along x
        dst = DenseTSDFVolume(0.01, 0.04, res, origin, color=False, device=cuda)
        assert L.bslam_tsdf_copy(src._h, dst._h, _lib.stream_ptr(cuda)) == _lib.E_ARG
        assert b"geometry mismatch" in L.bslam_last_error()
    dst = DenseTSDFVolume(0.01, 0.04, 64, (0.0, 0.0, 0.0), color=True, device=cuda)   # colour differs
    assert L.bslam_tsdf_copy(src._h, dst._h, _lib.stream_ptr(cuda)) == _lib.E_ARG


# ---------------------------------------------------------------- 6. the replay
@pytest.mark.gpu
def test_update_map_after_pg_with_growth_equals_the_replay_into_the_final_box(lumen, cuda, tmp_path):
    import cv2
    from bodyslam_b200.slam_utils import update_map_after_pg
    ids = list(range(0, 300, 15))
    rgb_paths, depth_paths = [], []
    for i in ids:
        rp, dp = str(tmp_path / f"rgb_{i}.png"), str(tmp_path / f"depth_{i}.png")
        cv2.imwrite(rp, lumen["color"][i].cpu().numpy()[:, :, ::-1])
        cv2.imwrite(dp, lumen["depth_u16"][i].cpu().numpy())
        rgb_paths.append(rp); depth_paths.append(dp)
    E = [lumen["E"][i] for i in ids]
    kw = dict(voxel_length=VL, sdf_trunc=TRUNC, resolution=START_RES, origin=START_ORIGIN)
    t = update_map_after_pg(E, rgb_paths, depth_paths, 1000, "CUDA:0", lumen["intrinsic"], grow=True, **kw)
    assert t.tsdf.growth_events == 1
    kw.update(resolution=(t.tsdf.nx, t.tsdf.ny, t.tsdf.nz), origin=tuple(t.tsdf.origin))
    r = update_map_after_pg(E, rgb_paths, depth_paths, 1000, "CUDA:0", lumen["intrinsic"], **kw)
    assert_volumes_equal(t.tsdf, r.tsdf)


# ---------------------------------------------------------------- 7. refusals
@pytest.mark.gpu
def test_auto_grow_refusals(cuda):
    dense = DenseTSDFVolume(VL, TRUNC, 128, START_ORIGIN, color=False, device=cuda)
    arith = DenseTSDFVolume(VL, TRUNC, 128, START_ORIGIN, color=False, device=cuda, unit_arithmetic=True)
    shard = DenseTSDFVolume(VL, TRUNC, (128, 128, 64), START_ORIGIN, color=False, device=cuda, gz0=64, z_total=128, unit_activation=True)
    inter = DenseTSDFVolume(VL, TRUNC, (128, 128, 64), START_ORIGIN, color=False, device=cuda, z_total=128, z_interleave=2)
    for v in (dense, arith, shard, inter):
        with pytest.raises(RuntimeError, match="set_auto_grow"):
            v.set_auto_grow(True)
    with pytest.raises(RuntimeError, match="unit activation"):
        TSDF(voxel_length=VL, sdf_trunc=TRUNC, resolution=128, origin=(0.001, 0.0, 0.0), device=cuda, grow=True)
    v = _auto(cuda)
    K = PinholeCameraIntrinsic(64, 48, 50.0, 50.0, 32.0, 24.0)
    d16 = torch.zeros((1, 48, 64), dtype=torch.uint16, device=cuda)
    scratch = torch.empty((1, 48, 64), dtype=torch.float32, device=cuda)
    with pytest.raises(RuntimeError, match="prepare_u16"):
        v.prepare_u16(d16, K, np.eye(4)[None], scratch)
    with pytest.raises(RuntimeError, match="integrate_prepared"):
        v.integrate_prepared(None)
    with pytest.raises(RuntimeError, match="integrate_streamed"):
        v.integrate_streamed([(0, 1)], K, np.eye(4)[None], lambda k, stage, free: (d16, None, None))
