"""Unit activation (ScalableTSDFVolume semantics: `unit_mark_kernel<kMarkUnits>`, the unit masks of both culls, the per-unit
voxel centres and z restart) at the edges its parity tests skip -- `-m gpu`.

The parity tests integrate rendered u16 frames with 32^3 units and stride 8 on 640 x 480 images into boxes of at most 32
units along z.  Here every case integrates the same frames on the GPU and with the oracle's `integrate_scalable(unit_res=,
stride=)` and asserts, bit for bit: tsdf, weight (and colour) as uint32 patterns, the per-frame update counts and the dry
run's counts; the units that hold weight must lie in the oracle's activated set.  The frames are NumPy geometry chosen so
that each case controls which edge it reaches:
  * unit sizes 8 .. 64 with strides 1 .. 16 on ragged images, the last sampled row and column carrying their own units;
  * ranges whose w -+ trunc lands exactly on a unit face (and one float32 depth step either side), on every axis, both
    directions, at negative unit indices;
  * two mask words per (ux, uy) row (nuz = 64): ranges across uz = 31 | 32, a whole word, more than 32 units;
  * the largest box both unit caps accept (65 536 units, 4 096 shared words);
  * launches of 31 .. 257 frames whose neighbours activate different units;
  * z-slabs and interleaved z-shards with 8^3 and 16^3 units;
  * NaN / inf / -0 / negative / subnormal / huge f32 depths (a point whose world coordinate is not finite activates nothing);
  * u16 depth at exactly depth_trunc; `clip_stats()` against `unit_activation_ref`; growth at 16^3 units and stride 3.
The CPU tests at the bottom check that the generators reach the edges they are built for."""
import numpy as np
import pytest
import torch

import oracle
import unit_activation_ref as ref
from bodyslam_b200.geometry import PinholeCameraIntrinsic

F32_MAX = float(np.finfo(np.float32).max)
SUBNORMAL = float(np.array([1], np.uint32).view(np.float32)[0])

# ---------------------------------------------------------------- geometry


def extrinsic(R, c):
    """world -> camera 4x4 (f64) of a camera with rotation R (camera -> world columns) at centre c"""
    R = np.asarray(R, dtype=np.float64)
    E = np.eye(4)
    E[:3, :3] = R.T
    E[:3, 3] = -R.T @ np.asarray(c, dtype=np.float64)
    return E


def rot(axis, quarter_turns):
    """exact rotation by a multiple of 90 degrees (entries 0 / +-1)"""
    c, s = [(1, 0), (0, 1), (-1, 0), (0, -1)][quarter_turns % 4]
    i, j = [(1, 2), (2, 0), (0, 1)][axis]
    R = np.eye(3)
    R[i, i], R[i, j], R[j, i], R[j, j] = c, -s, s, c
    return R


def small_rotation(rng, angle):
    """a rotation by at most `angle` radians about a random axis"""
    a = rng.normal(size=3)
    a /= np.linalg.norm(a)
    th = rng.uniform(-angle, angle)
    Kx = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx


def plane_depth(H, W, K, d0, slope=(0.0, 0.0)):
    """depth of a plane seen along the optical axis: d0 + slope . (x/z, y/z), f32"""
    fx, fy, cx, cy = K
    u = (np.arange(W) - cx) / fx
    v = (np.arange(H) - cy) / fy
    return (d0 + slope[0] * u[None, :] + slope[1] * v[:, None]).astype(np.float32)


def face_pose(axis, sign, centre):
    """world -> camera pose at `centre` whose optical axis is sign * e_axis"""
    R = np.zeros((3, 3))
    R[axis, 2] = sign
    others = [a for a in range(3) if a != axis]
    R[others[0], 0] = 1
    R[others[1], 1] = 1
    if np.linalg.det(R) < 0:
        R[others[0], 0] = -1
    return extrinsic(R, centre)


# ---------------------------------------------------------------- the GPU / oracle comparison


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def make_volume(dims, vl, trunc, origin, unit_res, stride, color=False, gz0=0, z_total=None, z_interleave=1, zpw=0, batch=0):
    from bodyslam_b200.tsdf import DenseTSDFVolume
    vol = DenseTSDFVolume(vl, trunc, dims, origin, color=color, device=torch.device("cuda", 0), gz0=gz0, z_total=z_total,
                          z_interleave=z_interleave, unit_activation=True, unit_resolution=unit_res, depth_sampling_stride=stride)
    vol.set_z_split(zpw)
    vol.set_batch(batch)
    return vol


def gpu_integrate(vol, depth, K, E, rgb=None):
    F, H, W = depth.shape
    counts = torch.zeros(F, dtype=torch.int64, device="cuda")
    col = None if rgb is None else torch.from_numpy(np.ascontiguousarray(rgb)).cuda()
    vol.integrate_batch(torch.from_numpy(np.ascontiguousarray(depth)).cuda(), col, PinholeCameraIntrinsic(W, H, *K), E,
                        update_counts=counts)
    return counts.cpu().numpy()


def oracle_integrate(V, depth, K, E, unit_res, stride, rgb=None):
    """-> (per-frame counts, per-frame activated units [F, nux, nuy, nuz])"""
    counts, touched = [], []
    for i in range(len(depth)):
        n, t = V.integrate_scalable(depth[i], K, E[i], rgb=None if rgb is None else rgb[i], unit_res=unit_res, stride=stride,
                                    return_touched=True)
        counts.append(n)
        touched.append(t.astype(bool))
    return np.array(counts, np.int64), np.stack(touched)


def assert_grids(got, V, color=False, what="", sl=None):
    """got: export_dense(...) of a GPU volume; sl: the oracle's slice of the grid it holds"""
    sl = sl if sl is not None else (slice(None),) * 3
    names = ("tsdf", "weight")
    for k, name in enumerate(names):
        g, r = got[k].cpu().numpy(), V.grid(name)[sl]
        bad = bits(g) != bits(r)
        assert not bad.any(), f"{what}: {int(bad.sum())} {name} values differ, e.g. {g[bad][:4]} vs {r[bad][:4]}"
    if color:
        c = got[2].cpu().numpy()
        r = V.color.reshape((V.nx, V.ny, V.nz, 3))[sl]
        bad = bits(c) != bits(r)
        assert not bad.any(), f"{what}: {int(bad.sum())} colour values differ"


def weighted_units(w, unit_res):
    nx, ny, nz = w.shape
    return (w.reshape(nx // unit_res, unit_res, ny // unit_res, unit_res, nz // unit_res, unit_res) != 0).any(axis=(1, 3, 5))


def check_case(depth, K, E, dims, vl, trunc, origin, unit_res, stride, rgb=None, zpw=0, batch=0, what=""):
    """integrate on the GPU and in the oracle; assert tsdf / weight / colour / per-frame counts / dry-run counts bit for bit,
    the units that hold weight inside the activated ones, and the restatement's activated set equal to the oracle's.
    -> (vol, V, counts, touched [F, nux, nuy, nuz])"""
    E = np.asarray(E, dtype=np.float64).reshape(-1, 4, 4)
    color = rgb is not None
    V = oracle.o3d.Volume(dims, vl, trunc, origin, with_color=color)
    oc, touched = oracle_integrate(V, depth, K, E, unit_res, stride, rgb)
    vol = make_volume(dims, vl, trunc, origin, unit_res, stride, color=color, zpw=zpw, batch=batch)
    gc = gpu_integrate(vol, depth, K, E, rgb)
    assert np.array_equal(gc, oc), f"{what}: per-frame update counts differ: {gc} vs {oc}"
    out = vol.export_dense(with_color=color)
    assert_grids(out, V, color, what)
    assert not (weighted_units(V.grid("weight"), unit_res) & ~touched.any(axis=0)).any(), f"{what}: weight outside the activated units"
    for f in range(len(depth)):
        want = ref.unit_activation(depth[f], K, E[f], dims, vl, trunc, origin, unit_res, stride)["touched"]
        assert np.array_equal(want, touched[f]), f"{what}: frame {f}: the restatement's activated units differ from the oracle's"
    F, H, W = depth.shape
    dc = vol.count_updates(torch.from_numpy(np.ascontiguousarray(depth)).cuda(), PinholeCameraIntrinsic(W, H, *K), E).cpu().numpy()
    assert np.array_equal(dc, oc), f"{what}: dry-run counts differ: {dc} vs {oc}"
    return vol, V, oc, touched


def assert_activation_matters(V, touched, unit_res):
    """units that hold weight next to activated units and to units that do not: the comparison can see a wrong unit"""
    wu = weighted_units(V.grid("weight"), unit_res)
    assert wu.any() and not wu.all(), "every unit or no unit holds weight"


# ================================================================ 1. unit sizes x strides on ragged images


def stride_frames(W, H, K, F, stride, rng, near, far):
    """tilted planes seen from cameras that drift across the box; the pixels from the last sampled column to the image edge
    see a nearer surface than the rest (and those from the last sampled row one between the two), so the points of that
    column activate units no other point does"""
    fx, fy, cx, cy = K
    D, E = [], []
    j_last, i_last = ((W - 1) // stride) * stride, ((H - 1) // stride) * stride
    for f in range(F):
        d = plane_depth(H, W, K, rng.uniform(*far), rng.uniform(-0.05, 0.05, 2))
        d[rng.random(d.shape) < 0.05] = 0.0
        d[i_last:, :] = 0.5 * (near[1] + far[0])
        d[:, j_last:] = rng.uniform(*near)
        D.append(d)
        c = np.array([rng.uniform(-0.03, 0.03), rng.uniform(-0.03, 0.03), -0.2])
        E.append(extrinsic(small_rotation(rng, 0.1), c))
    return np.stack(D), np.stack(E)


STRIDE_IMAGES = [(17, 9), (33, 31), (641, 479)]


@pytest.mark.gpu
@pytest.mark.parametrize("stride", [1, 2, 3, 8, 16])
@pytest.mark.parametrize("unit_res", [8, 16, 32, 64])
def test_unit_sizes_and_strides_on_ragged_images(cuda, unit_res, stride):
    """box 0.25 m wide of 2 - 4 units per axis; images whose width and height are not multiples of the stride (and one
    narrower than the stride); 3 frames (the per-brick cull) and 11 frames (the warp cull)"""
    rng = np.random.default_rng(unit_res * 100 + stride)
    nu = 2 if unit_res == 64 else 4
    n = nu * unit_res
    vl = 0.25 / n
    dims, origin, trunc = (n, n, n + unit_res), (-0.125, -0.125, 0.0), 0.012      # the top unit layer lies beyond every surface
    sizes = [s for s in STRIDE_IMAGES if s[0] * s[1] < 300_000 or stride >= 3] + ([(stride - 3, 5)] if stride > 3 else [])
    for k, (W, H) in enumerate(sizes):
        K = (2.0 * W, 2.0 * W, (W - 1) / 2 + 0.25, (H - 1) / 2 - 0.25)
        F = 11 if k % 2 else 3
        D, E = stride_frames(W, H, K, F, stride, rng, near=(0.25, 0.3), far=(0.33, 0.42))
        vol, V, oc, touched = check_case(D, K, E, dims, vl, trunc, origin, unit_res, stride, what=f"{W}x{H}, F = {F}")
        assert oc.sum() > 0
        assert_activation_matters(V, touched, unit_res)
        if W % stride and W > stride:
            # the last sampled column activates units the rest of its frame does not
            nolast = D.copy()
            nolast[:, :, ((W - 1) // stride) * stride] = 0.0
            assert any(not np.array_equal(ref.unit_activation(nolast[f], K, E[f], dims, vl, trunc, origin, unit_res, stride)["touched"],
                                          touched[f]) for f in range(F)), f"{W}x{H}: the last sampled column adds no unit"


# ================================================================ 2. exact unit faces (kMarkUnits)

BVL, BTRUNC = 1.0 / 64, 1.0 / 16        # every face below is exact in f64


def face_frames(unit_res, axis, sign):
    """pixel (0, 0), the only one sampled at stride 8 of an 8 x 8 image with cx = cy = 0, lies on the optical axis; the
    camera sits 4 units behind the box centre.  Its depth puts w - trunc or w + trunc on the unit faces -1, 0, +1 (w = the
    world coordinate along `axis`), or one float32 step before or after.  Every other pixel sees far beyond the box, so an
    activated unit in view collects free-space updates."""
    ul = BVL * unit_res
    zs = sorted({f * ul + s * BTRUNC + 4 * ul for f in (-1, 0, 1) for s in (-1, 1)})
    D = []
    for z in zs:
        z = np.float32(z)
        for v in (np.nextafter(z, np.float32(0)), z, np.nextafter(z, np.float32(10))):
            d = np.full((8, 8), 20 * ul, np.float32)
            d[0, 0] = v
            D.append(d)
    c = np.zeros(3)
    c[axis] = -sign * 4 * ul
    E = np.stack([face_pose(axis, sign, c)] * len(D))
    return np.stack(D), E


@pytest.mark.gpu
@pytest.mark.parametrize("unit_res", [8, 16])
@pytest.mark.parametrize("axis", [0, 1, 2])
@pytest.mark.parametrize("sign", [1, -1])
def test_ranges_ending_exactly_on_unit_faces(cuda, unit_res, axis, sign):
    """box of units -2 .. 1 per axis: w -+ trunc on the faces between units -2 | -1, -1 | 0 and 0 | 1, and one float32
    step of depth either side; in launches of 6 frames (the per-brick cull) and of all 12 (the warp cull)"""
    ul = BVL * unit_res
    n = 4 * unit_res
    D, E = face_frames(unit_res, axis, sign)
    K = (10.0, 10.0, 0.0, 0.0)
    for batch in (6, 0):
        vol, V, oc, touched = check_case(D, K, E, (n, n, n), BVL, BTRUNC, (-2 * ul,) * 3, unit_res, 8, batch=batch,
                                         what=f"axis {axis} sign {sign} batch {batch}")
    # each exact face and its neighbours activate different units, and the per-frame counts see the difference
    ranges = [set(np.flatnonzero(touched[f].any(axis=tuple(a for a in range(3) if a != axis)))) for f in range(len(D))]
    for g in range(0, len(D), 3):
        assert ranges[g] != ranges[g + 1] or ranges[g + 1] != ranges[g + 2], (g, ranges[g:g + 3])
        assert len({int(oc[g]), int(oc[g + 1]), int(oc[g + 2])}) > 1, oc[g:g + 3]
    assert 0 in set().union(*ranges) and 3 in set().union(*ranges)        # global units -2 and 1 reached


# ================================================================ 3. two mask words per row

WVL = 1.0 / 256                          # 8^3 units of 1/32 m; 256 x 256 x 512 voxels: 32 x 32 x 64 units


def word_frames(targets):
    """a camera at (0.5, 0.5, -0.25) looks along +z; the four sampled pixels (stride 8 of 16 x 16) put points at world
    z = target (in units), every other pixel sees beyond the box"""
    ul = WVL * 8
    K = (16.0, 16.0, 8.0, 8.0)
    D = []
    for t in targets:
        d = np.full((16, 16), 3.0, np.float32)
        d[::8, ::8] = np.float32(t * ul + 0.25)
        D.append(d)
    E = np.stack([extrinsic(np.eye(3), (0.5, 0.5, -0.25))] * len(targets))
    return np.stack(D), E, K


@pytest.mark.gpu
@pytest.mark.parametrize("trunc_units,targets", [
    (15.5, [32.0, 47.5, 16.0, 24.0, 60.0, 2.0, 31.75]),      # across 31 | 32 from mid-word, words 1 and 0 exactly, cut ranges
    (20.0, [32.0, 40.5, 20.0]),                               # 41 units: longer than a word
])
def test_ranges_across_the_mask_words_of_a_row(cuda, trunc_units, targets):
    ul = WVL * 8
    D, E, K = word_frames(targets)
    trunc = trunc_units * ul
    vol, V, oc, touched = check_case(D, K, E, (256, 256, 512), WVL, trunc, (0.0, 0.0, 0.0), 8, 8, what=f"trunc {trunc_units} units")
    z_ranges = []
    for f in range(len(D)):
        uz = np.flatnonzero(touched[f].any(axis=(0, 1)))
        z_ranges.append((int(uz.min()), int(uz.max())))
    assert any(lo < 32 <= hi and lo % 32 for lo, hi in z_ranges), z_ranges            # crosses 31 | 32, starts mid-word
    if trunc_units == 15.5:
        assert (32, 63) in z_ranges and (0, 31) in z_ranges, z_ranges                # exactly one whole word
    else:
        assert max(hi - lo + 1 for lo, hi in z_ranges) > 32, z_ranges
    assert_activation_matters(V, touched, 8)


# ================================================================ 4. the caps


@pytest.mark.gpu
def test_largest_box_both_unit_caps_accept(cuda):
    """512 x 512 x 128 voxels of 8^3 units: 64 * 64 * 16 = 65 536 units and 64 * 64 * 1 = 4 096 shared words.  Cameras look
    at the (+x, +y) corner, so the last row of units (ux = uy = 63), the last word, activates"""
    rng = np.random.default_rng(4096)
    vl = 1.0 / 256
    W, H = 48, 40
    K = (40.0, 40.0, 23.5, 19.5)
    D, E = [], []
    for f in range(3):
        D.append(plane_depth(H, W, K, rng.uniform(0.45, 0.6), rng.uniform(-0.05, 0.05, 2)))
        E.append(extrinsic(small_rotation(rng, 0.05), (1.95 + rng.uniform(-0.02, 0.02), 1.95 + rng.uniform(-0.02, 0.02), -0.3)))
    vol, V, oc, touched = check_case(np.stack(D), K, np.stack(E), (512, 512, 128), vl, 0.02, (0.0, 0.0, 0.0), 8, 4, what="caps")
    assert touched.shape[1:] == (64, 64, 16)
    assert touched[:, 63, 63].any() and weighted_units(V.grid("weight"), 8)[63, 63].any()
    assert_activation_matters(V, touched, 8)


# ================================================================ 5. launches of many frames


def batch_frames(F, rng):
    """a camera that sweeps across a 64^3 box of 8^3 units: neighbouring frames activate different units"""
    W, H = 20, 16
    K = (18.0, 18.0, 9.5, 7.5)
    D, E = [], []
    for f in range(F):
        s = f / max(F - 1, 1)
        c = np.array([-0.2 + 0.4 * s + rng.uniform(-0.01, 0.01), 0.15 * np.sin(7 * s), -0.15])
        E.append(extrinsic(small_rotation(rng, 0.1), c))
        d = plane_depth(H, W, K, rng.uniform(0.2, 0.35), rng.uniform(-0.05, 0.05, 2))
        d[rng.random(d.shape) < 0.05] = 0.0
        D.append(d)
    return np.stack(D), np.stack(E), K


@pytest.mark.gpu
@pytest.mark.parametrize("F", [31, 32, 33, 64, 65, 256, 257])
def test_launches_of_many_frames(cuda, F):
    """one call of F frames in launches of min(F, 256) (set_batch): frame f's units go to mask word f >> 5, and the masks
    are cleared between the launches of 257 frames"""
    rng = np.random.default_rng(F)
    D, E, K = batch_frames(F, rng)
    vol, V, oc, touched = check_case(D, K, E, (64, 64, 64), 1.0 / 128, 0.01, (-0.25, -0.25, 0.0), 8, 2, batch=min(F, 256),
                                     what=f"F = {F}")
    # frames 32 apart activate different units (what a wrong mask word would mix up)
    assert sum(not np.array_equal(touched[f], touched[f - 32]) for f in range(32, F)) >= (F - 32) // 2
    assert_activation_matters(V, touched, 8)


# ================================================================ 6. z-shards with small units


@pytest.mark.gpu
@pytest.mark.parametrize("unit_res", [8, 16])
@pytest.mark.parametrize("layout", ["slab", "interleave2", "interleave4"])
def test_z_shards_with_small_units_equal_the_whole_grid_oracle(cuda, unit_res, layout):
    """the whole 64 x 64 x 128 grid in z-slabs of 32 planes (gz0 = 0, 32, 64, 96) or in 2 / 4 interleaved shards (rank r
    holds brick layers r, r + k, ...; a 16^3 unit's two layers live on different ranks), each for z splits 2 / 4 / 8: every
    shard equals its part of the whole-grid oracle"""
    rng = np.random.default_rng(unit_res + len(layout))
    vl, trunc, stride = 1.0 / 256, 0.01, 4
    origin = (-0.125, -0.125, 0.0)
    W, H = 40, 30
    K = (30.0, 30.0, 19.5, 14.5)
    D, E = [], []
    for f in range(5):
        D.append(plane_depth(H, W, K, rng.uniform(0.27, 0.55), rng.uniform(-0.2, 0.2, 2)))
        E.append(extrinsic(small_rotation(rng, 0.15), (rng.uniform(-0.02, 0.02), rng.uniform(-0.02, 0.02), -0.25)))
    D, E = np.stack(D), np.stack(E)
    V = oracle.o3d.Volume((64, 64, 128), vl, trunc, origin)
    oc, touched = oracle_integrate(V, D, K, E, unit_res, stride)
    assert_activation_matters(V, touched, unit_res)
    k = 1 if layout == "slab" else int(layout[-1])
    for zpw in (2, 4, 8):
        union = np.zeros((64, 64, 128), bool)
        for r in range(4 if k == 1 else k):
            if k == 1:
                vol = make_volume((64, 64, 32), vl, trunc, origin, unit_res, stride, gz0=32 * r, z_total=128, zpw=zpw)
                planes = np.arange(32 * r, 32 * r + 32)
            else:
                vol = make_volume((64, 64, 128 // k), vl, trunc, origin, unit_res, stride, gz0=8 * r, z_total=128, z_interleave=k, zpw=zpw)
                planes = np.concatenate([np.arange(8 * (l * k + r), 8 * (l * k + r) + 8) for l in range(128 // (8 * k))])
            gpu_integrate(vol, D, K, E)
            assert_grids(vol.export_dense(), V, what=f"{layout} rank {r} zpw {zpw}", sl=(slice(None), slice(None), planes))
            union[:, :, planes] = True
        assert union.all()


# ================================================================ 7. special f32 depths


def special_frames(R, rng):
    """a far wall (3 m: beyond the box and its trunc band, so no real point activates a unit of the box) with NaN, +-inf,
    -0, negative, subnormal, 1e30 and FLT_MAX pixels on sampled positions, +inf also on (cx, cy), on cx alone and on cy
    alone.  Frame 0 holds only +inf pixels; the last frame adds a plane through the box"""
    W, H, stride = 33, 25, 4
    K = (30.0, 30.0, 16.0, 12.0)            # the principal point is a sampled pixel
    vals = [np.nan, np.inf, -np.inf, -0.0, -0.5, SUBNORMAL, 1e30, F32_MAX]
    sampled = [(i, j) for i in range(0, H, stride) for j in range(0, W, stride)]
    D = []
    for f in range(4):
        d = np.full((H, W), 3.0, np.float32)
        pick = rng.choice(len(sampled), 12, replace=False)
        for n, p in enumerate(pick):
            d[sampled[p]] = np.inf if f == 0 else vals[n % len(vals)]
        d[12, 16] = np.inf
        d[0, 16] = np.inf if f != 1 else F32_MAX
        d[12, 0] = np.inf if f != 2 else np.nan
        D.append(d)
    band = plane_depth(H, W, K, 0.62, (0.05, -0.03))
    band[::stride, ::stride][rng.random(band[::stride, ::stride].shape) < 0.2] = np.inf
    D.append(band)
    c = -0.6 * R[:, 2] + np.array([0.01, -0.02, 0.015])
    E = np.stack([extrinsic(R, c)] * len(D))
    return np.stack(D), E, K, stride


SPECIAL_POSES = {"identity": np.eye(3), "x90": rot(0, 1), "y270": rot(1, 3), "z180": rot(2, 2)}


@pytest.mark.gpu
@pytest.mark.parametrize("pose", list(SPECIAL_POSES) + ["oblique0", "oblique1"])
def test_special_depths_activate_no_unit(cuda, pose):
    """box of 8^3 units -4 .. 3 per axis, world unit 0 in view: with exact zeros in the pose every +inf pixel gives a NaN
    world coordinate, which must activate no unit; huge finite depths land far outside the box"""
    rng = np.random.default_rng(len(pose) * 7 + ord(pose[-1]))
    R = SPECIAL_POSES.get(pose)
    if R is None:
        R = small_rotation(rng, 0.6)
    D, E, K, stride = special_frames(R, rng)
    vl, ur = 1.0 / 128, 8
    dims, origin = (64, 64, 64), (-0.25, -0.25, -0.25)
    vol, V, oc, touched = check_case(D, K, E, dims, vl, 0.02, origin, ur, stride, what=pose)
    assert not touched[0].any() and oc[0] == 0       # frame 0: only +inf and a far wall
    assert touched[-1].any() and oc[-1] > 0          # the plane through the box still activates its units
    # world unit 0 (local 4, 4, 4) is in view: activated by the all-units rule, it would collect updates in frame 0
    A = oracle.o3d.Volume(dims, vl, 0.02, origin)
    A.integrate_scalable(D[0], K, E[0], unit_res=ur, stride=stride, all_units=True)
    assert weighted_units(A.grid("weight"), ur)[4, 4, 4]
    st = vol.clip_stats()
    want = [ref.unit_activation(D[f], K, E[f], dims, vl, 0.02, origin, ur, stride) for f in range(len(D))]
    assert st == {k: sum(w[k] for w in want) for k in ("points", "outside", "partly_outside")}, st


# ================================================================ 8. u16 depth at the threshold


@pytest.mark.gpu
def test_u16_depth_at_exactly_depth_trunc_activates_its_units(cuda):
    """u = 3300 at scale 1000 with depth_trunc 3.3 is kept (Open3D compares in double); 3301 is dropped"""
    W, H = 24, 16
    K = (20.0, 20.0, 11.5, 7.5)
    u16 = np.full((3, H, W), 3300, np.uint16)
    u16[1, ::4, :] = 3301
    u16[2, :, ::3] = 0
    E = np.stack([extrinsic(np.eye(3), (0.01 * f, -0.01 * f, -3.2)) for f in range(3)])
    dims, vl, trunc, origin, ur, stride = (64, 64, 64), 1.0 / 128, 0.02, (-0.25, -0.25, 0.0), 16, 2
    d = oracle.o3d.depth_from_u16(u16, 1000.0, 3.3)
    assert float(d[0, 0, 0]) == np.float32(3300) / np.float32(1000)
    V = oracle.o3d.Volume(dims, vl, trunc, origin)
    oc, touched = oracle_integrate(V, d, K, E, ur, stride)
    assert oc.min() > 0 and touched.any(axis=(1, 2, 3)).all()
    vol = make_volume(dims, vl, trunc, origin, ur, stride)
    counts = torch.zeros(3, dtype=torch.int64, device="cuda")
    vol.integrate_u16_batch(torch.from_numpy(u16).cuda(), None, PinholeCameraIntrinsic(W, H, *K), E, 1000.0, 3.3, update_counts=counts)
    assert np.array_equal(counts.cpu().numpy(), oc)
    assert_grids(vol.export_dense(), V, what="u16 at depth_trunc")


# ================================================================ 9. clip_stats()


def clip_frames(rng, stride):
    """depth uniform over a range that starts in front of the box and ends behind it, seen from six sides (every face gets
    points inside, straddling it within trunc, and outside), plus the special values on sampled pixels"""
    W, H = 37, 29
    K = (22.0, 22.0, 18.0, 14.0)
    D, E = [], []
    for axis in range(3):
        for sign in (1, -1):
            c = np.zeros(3)
            c[axis] = -sign * 0.4
            c += rng.uniform(-0.02, 0.02, 3)
            E.append(face_pose(axis, sign, c))
            d = rng.uniform(0.05, 0.75, (H, W)).astype(np.float32)
            d[rng.random(d.shape) < 0.05] = 0.0
            for n, v in enumerate([np.nan, np.inf, -np.inf, -0.0, -1.0, SUBNORMAL, 1e30, F32_MAX]):
                d[stride * rng.integers(0, (H - 1) // stride + 1), stride * rng.integers(0, (W - 1) // stride + 1)] = v
            d[14, 18] = np.inf                    # on the principal point
            D.append(d)
    return np.stack(D), np.stack(E), K


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["unit", "dense", "dense_shard"])
def test_clip_stats_count_exactly(cuda, mode):
    """points / outside / partly_outside of `clip_stats()` equal the restatement in unit mode (stride 3, 8^3 units) and in
    dense mode with the clip check (stride 2), also on a z-slab of the grid (the count is over the whole grid's z extent)"""
    from bodyslam_b200.tsdf import DenseTSDFVolume
    rng = np.random.default_rng(len(mode))
    vl, trunc = 1.0 / 128, 0.03
    dims, origin = (64, 64, 64), (-0.25, -0.25, -0.25)
    stride = 3 if mode == "unit" else 2
    D, E, K = clip_frames(rng, stride)
    if mode == "unit":
        vol = make_volume(dims, vl, trunc, origin, 8, stride)
        want = [ref.unit_activation(D[f], K, E[f], dims, vl, trunc, origin, 8, stride) for f in range(len(D))]
    else:
        shard = mode == "dense_shard"
        vol = DenseTSDFVolume(vl, trunc, (64, 64, 32) if shard else dims, origin, color=False, device=cuda,
                              gz0=32 if shard else 0, z_total=64)
        vol.set_clip_check(stride)
        want = [ref.dense_clip(D[f], K, E[f], dims, vl, trunc, origin, stride) for f in range(len(D))]
    gpu_integrate(vol, D, K, E)
    total = {k: sum(w[k] for w in want) for k in ("points", "outside", "partly_outside")}
    assert vol.clip_stats() == total
    # the frames reach every class: inside, straddling a face, outside
    assert 0 < total["partly_outside"] and 0 < total["outside"] < total["points"] - total["partly_outside"], total
    assert vol.clip_stats(reset=True) == total and vol.clip_stats() == {"points": 0, "outside": 0, "partly_outside": 0}


# ================================================================ 10. growth with 16^3 units and stride 3


@pytest.mark.gpu
def test_growth_with_small_units_through_the_sampled_gather(cuda):
    """`integrate_host` with auto-growth bounds the frames from their stride-3 pixels gathered on the host; the grown box
    equals a box of its final size given the same frames, and the oracle"""
    rng = np.random.default_rng(16)
    vl, trunc, ur, stride = 1.0 / 128, 0.02, 16, 3
    W, H = 41, 31
    K = (30.0, 30.0, 20.0, 15.0)
    F = 12
    u16 = np.empty((F, H, W), np.uint16)
    E = []
    for f in range(F):
        u16[f] = np.clip(plane_depth(H, W, K, rng.uniform(0.3, 0.4), rng.uniform(-0.05, 0.05, 2)) * 1000, 0, 65535).astype(np.uint16)
        u16[f][rng.random((H, W)) < 0.05] = 0
        E.append(extrinsic(small_rotation(rng, 0.1), (0.08 * f, -0.03 * f, -0.2)))
    E = np.stack(E)
    intr = PinholeCameraIntrinsic(W, H, *K)
    vol = make_volume(64, vl, trunc, (-0.25, -0.25, 0.0), ur, stride)
    vol.set_auto_grow(True)
    counts = torch.zeros(F, dtype=torch.int64, device="cuda")
    vol.integrate_host(torch.from_numpy(u16).pin_memory(), None, intr, E, update_counts=counts)
    torch.cuda.synchronize()
    assert vol.growth_events == 1 and vol.nx > 64
    pre = make_volume((vol.nx, vol.ny, vol.nz), vl, trunc, vol.origin, ur, stride)
    pc = torch.zeros(F, dtype=torch.int64, device="cuda")
    pre.integrate_u16_batch(torch.from_numpy(u16).cuda(), None, intr, E, update_counts=pc)
    assert torch.equal(counts, pc)
    for a, b in zip(vol.export_dense(), pre.export_dense()):
        assert np.array_equal(bits(a.cpu().numpy()), bits(b.cpu().numpy()))
    V = oracle.o3d.Volume((vol.nx, vol.ny, vol.nz), vl, trunc, vol.origin)
    oc, touched = oracle_integrate(V, oracle.o3d.depth_from_u16(u16), K, E, ur, stride)
    assert np.array_equal(counts.cpu().numpy(), oc)
    assert_grids(vol.export_dense(), V, what="grown")


# ================================================================ CPU checks of the generators (oracle only)


def test_face_frames_put_the_range_ends_on_unit_faces():
    """for every face frame the exact depth lands w -+ trunc on a face and its neighbours one float32 step either side"""
    for ur in (8, 16):
        ul = BVL * ur
        for axis in range(3):
            for sign in (1, -1):
                D, E = face_frames(ur, axis, sign)
                ends = set()
                for f in range(len(D)):
                    w, finite = ref.sampled_world_points(D[f], (10.0, 10.0, 0.0, 0.0), E[f], 8)
                    assert finite.all() and len(w) == 1 and w[0, axis - 1] == 0.0
                    lo_hi = ((w[0, axis] - BTRUNC) / ul, (w[0, axis] + BTRUNC) / ul)
                    if f % 3 == 1:
                        assert any(float(x).is_integer() for x in lo_hi), lo_hi
                    ends |= {int(np.floor(x)) for x in lo_hi}
                assert {-2, -1, 0, 1} <= ends, ends


def test_special_frames_give_non_finite_world_points():
    """with exact zeros in the pose +inf pixels give NaN world coordinates; huge depths stay finite"""
    rng = np.random.default_rng(0)
    D, E, K, stride = special_frames(np.eye(3), rng)
    w, finite = ref.sampled_world_points(D[0], K, E[0], stride)
    assert np.isnan(w).all(axis=1).sum() >= 12
    w, finite = ref.sampled_world_points(D[1], K, E[1], stride)
    assert np.isfinite(w).all(axis=1).sum() > 0 and (np.abs(w[finite]) > 1e29).any()
