"""Edges of the depth-image kernels that their parity tests (test_gpu_mdem.py, test_gpu_edge.py) skip:
K1 (`bslam_colorize`, `bslam_scale_u16`, `bslam_median_u16`, `bslam_minmax_u8`), K1f (`bslam_colorize_f32`),
a4 (`bslam_depth_from_u16` and its fused forms) and K2 (`bslam_backproject`).

Everything is compared as bit patterns (+0 and -0 differ, NaN masks must match) with a plain reference:
colour and percentiles with oracle.mdem and NumPy itself, a4 and back-projection order with oracle.o3d, and
back-projected coordinates with a float64 evaluation and the error bound derived beside `bp_bound`.
The tests without the gpu mark check, on the CPU, that the constructed inputs hit the case they are built for
and that the rules the GPU tests rely on hold."""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from bodyslam_b200 import _lib, mdem, ops
from bodyslam_b200 import synthetic as S
from bodyslam_b200.geometry import PinholeCameraIntrinsic, RGBDImage, inverse4x4
from bodyslam_b200.tsdf import DenseTSDFVolume

gpu = pytest.mark.gpu
f32 = np.float32
EPS = 2.0 ** -24
LUT = mdem.get_cmap_lut("viridis")


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view({1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


def assert_bits(got, want, what=""):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype, want.dtype)
    bad = bits(got) != bits(want)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} differ, first at {np.argwhere(bad)[:3].tolist()}"


def assert_same_f64(got, want, what=""):
    """one float64 value: equal bit patterns, or both NaN (np.percentile's NaN has no pinned payload)"""
    g, w = np.float64(got), np.float64(want)
    assert (np.isnan(g) and np.isnan(w)) or bits(np.array([g])) == bits(np.array([w])), (what, g, w)


# ====================================================================================== K1: uint16 and fused metres
def k1_reference(img, invalid_val, p_lo, p_hi):
    """(vmin, vmax, rgba) of the reference: np.percentile of the valid pixels, then oracle.mdem.colorize with them"""
    valid = img[img != invalid_val] if invalid_val is not None else img.ravel()
    if valid.size:
        vmin, vmax = np.percentile(valid, p_lo), np.percentile(valid, p_hi)
    else:
        vmin = vmax = 0.0
    inv = -99 if invalid_val is None else invalid_val
    return vmin, vmax, oracle.mdem.colorize(img, LUT, vmin=vmin, vmax=vmax, invalid_val=inv)


def check_k1_u16(u16, invalid_val=0, p_lo=2.0, p_hi=85.0):
    rgba, _, stats = ops.colorize_u16(LUT, depth_u16=u16, invalid_val=invalid_val, p_lo=p_lo, p_hi=p_hi, return_stats=True)
    rgba, stats = rgba.cpu().numpy(), stats.cpu().numpy()
    for b in range(u16.shape[0]):
        vmin, vmax, ref = k1_reference(u16[b], invalid_val, p_lo, p_hi)
        assert_same_f64(stats[b, 0], vmin, f"vmin of image {b}")
        assert_same_f64(stats[b, 1], vmax, f"vmax of image {b}")
        assert_bits(rgba[b], ref.reshape(rgba[b].shape), f"rgba of image {b}")


def depth_batch(rng, B, H, W, invalid_frac=0.1):
    """a different smooth field + noise per image (own offset and range), so statistics leaking between images show"""
    yy, xx = np.mgrid[0:H, 0:W]
    out = np.empty((B, H, W), np.uint16)
    for b in range(B):
        lo = rng.integers(1, 40000)
        span = rng.integers(1, 20000)
        f = 0.5 + 0.5 * np.sin(xx / rng.uniform(3, 40) + rng.uniform(0, 6)) * np.cos(yy / rng.uniform(3, 40))
        d = lo + span * f + rng.normal(0, rng.uniform(0, 30), (H, W))
        d = np.clip(d, 1, 65535).astype(np.uint16)
        d[rng.uniform(size=(H, W)) < invalid_frac] = 0
        out[b] = d
    return out


# B and image sizes: H*W = 0, 1, 2 and 3 (mod 4), single pixels, single rows / columns across a 4096-pixel block
K1_BATCHES = [(1, 1, 1), (2, 1, 4097), (5, 4097, 1), (64, 37, 23), (65, 45, 101), (300, 3, 2), (5, 64, 64), (3, 70, 70),
              (2, 90, 91), (1, 2049, 3)]


@gpu
@pytest.mark.parametrize("B,H,W", K1_BATCHES)
def test_k1_batches_of_every_size_residue(cuda, B, H, W):
    check_k1_u16(depth_batch(np.random.default_rng(B * 7919 + H * 31 + W), B, H, W))


@gpu
@pytest.mark.parametrize("B,H,W", [(5, 37, 23), (3, 1, 4097), (64, 64, 64)])
def test_k1_fused_from_metres_batches(cuda, B, H, W):
    """float32 metres -> (m * 256).astype(uint16) fused with the histogram; u16 and RGBA per image"""
    rng = np.random.default_rng(B + H + W)
    m = (rng.uniform(0.05, 8.0, (B, H, W)) * rng.uniform(0.2, 1.0, (B, 1, 1))).astype(f32)
    m[rng.uniform(size=m.shape) < 0.05] = 0.0
    rgba, u16, stats = ops.colorize_u16(LUT, depth_m=m, invalid_val=0, return_stats=True)
    want = (m * f32(256)).astype(np.uint16)
    assert_bits(u16.cpu().numpy(), want, "u16")
    rgba, stats = rgba.cpu().numpy(), stats.cpu().numpy()
    for b in range(B):
        vmin, vmax, ref = k1_reference(want[b], 0, 2.0, 85.0)
        assert_same_f64(stats[b, 0], vmin)
        assert_same_f64(stats[b, 1], vmax)
        assert_bits(rgba[b], ref.reshape(rgba[b].shape), f"rgba of image {b}")


# ---------------------------------------------------------------- shared-histogram window edges
WINDOW = 4096          # bins of the shared window of scale_hist_kernel, anchored at the block minimum
BLOCK_PX = 4096        # pixels per block (256 threads x 16)


def window_edge_image(rng):
    """rows of 4096 pixels = one histogram block each:
    row 0: min m, values m + 4095 (last shared bin) and m + 4096 (first global bin), uniform 4-pixel groups of one value
           (merged across the warp by match.any) beside mixed ones;
    row 1: a dense window (every bin of the first 512 occupied) -> word-interleaved flush;
    row 2: a sparse window (a handful of values) -> 16-byte flush, plus the same uniform / mixed mix;
    row 3: no valid pixel;
    row 4: values all >= the window (min + 4096 and beyond) except the minimum itself."""
    H = 5
    img = np.zeros((H, BLOCK_PX), np.uint16)
    m = 20000
    r0 = np.full(BLOCK_PX, m + 100, np.uint16)
    r0[0] = m
    r0[4:8] = m + 4095          # a uniform group at the last shared bin
    r0[8:12] = m + 4096         # a uniform group at the first global bin
    r0[12:16] = [m + 4095, m + 4096, m + 4095, m + 4096]   # a mixed group straddling the edge
    g = r0[16:2048].reshape(-1, 4)   # 4-pixel groups of the first half; the 32 lanes of a warp read 32 consecutive groups
    g[0::2] = m + 7             # every other group uniform, all of one value: match.any merges 16 per warp ...
    g[1::2] = [m + 7, m + 8, m + 7, m + 8]   # ... beside mixed groups that add pixel by pixel
    r0[2048:] = np.tile(np.array([m + 100, m + 101], np.uint16), 1024)      # the second half: mixed groups only
    r0[2000:2004] = [m + 4095, m + 4095, m + 4095, m + 4094]
    img[0] = r0
    img[1] = 30000 + (np.arange(BLOCK_PX) % 512)
    r2 = np.full(BLOCK_PX, 5000, np.uint16)
    r2[rng.choice(BLOCK_PX, 40, replace=False)] = 5000 + rng.choice([1, 2, 130, 700, 1500, 3001, 4095], 40)
    r2[1024:1032] = 5003
    r2[1025] = 5002
    img[2] = r2
    img[3] = 0
    r4 = np.full(BLOCK_PX, 60000, np.uint16)
    r4[77] = 60000 - 4097
    r4[1::3] = 64000
    img[4] = r4
    return img


def flush_modes(block_vals):
    """per 128-bin warp segment of the shared window: 'dense' (> 8 of its 32 16-byte words occupied) or 'sparse'"""
    valid = block_vals[block_vals != 0].astype(np.int64)
    base = valid.min()
    rel = valid - base
    hist = np.bincount(rel[rel < WINDOW], minlength=WINDOW)
    words = hist.reshape(-1, 4).any(1).reshape(-1, 32).sum(1)
    return {"dense" if w > 8 else "sparse" for w in words if w}


def test_window_edge_blocks_hit_their_cases():
    img = window_edge_image(np.random.default_rng(0))
    r0 = img[0]
    m = int(r0.min())
    assert m + 4095 in r0 and m + 4096 in r0
    g = r0.reshape(-1, 32, 4)              # [warp load][lane][pixel of the lane's group]
    uni = (g == g[..., :1]).all(2)
    assert uni.any() and (~uni).any()
    # some warp load holds two or more uniform groups of the same value (the match.any merge), next to mixed groups
    merged = [np.unique(g[w][uni[w], 0], return_counts=True)[1].max() for w in range(g.shape[0]) if uni[w].any() and (~uni[w]).any()]
    assert merged and max(merged) >= 2
    # percentiles 30 / 40 of row 0 fall on both sides of the end of its m + 7 run: a merge that counted one group per
    # value instead of all of them would move both
    def without_merge(row):
        out = []
        for w in row.reshape(-1, 32, 4):
            u = (w == w[:, :1]).all(1)
            out.extend(w[~u].ravel())
            for val in np.unique(w[u, 0]):
                out.extend([val] * 4)
        return np.array(out)
    assert np.percentile(r0, 30) == m + 7 and np.percentile(r0, 40) == m + 8
    assert np.percentile(without_merge(r0), 30) != m + 7
    assert "dense" in flush_modes(img[1]) and flush_modes(img[2]) == {"sparse"}
    assert not (img[3] != 0).any()
    assert int(img[4].max()) - int(img[4].min()) >= WINDOW


@gpu
@pytest.mark.parametrize("offset", [0, 1, 3])
def test_k1_window_edge_blocks(cuda, offset):
    """the blocks above as one image, and shifted by 1 / 3 pixels so that they straddle blocks and lose alignment"""
    img = window_edge_image(np.random.default_rng(1)).ravel()
    img = np.concatenate([np.full(offset, 7, np.uint16), img])
    n = img.size
    u16 = np.stack([img, np.roll(img, 4096), img[::-1].copy()]).reshape(3, 1, n)
    check_k1_u16(u16, invalid_val=0)
    check_k1_u16(u16, invalid_val=None, p_lo=0.0, p_hi=100.0)
    row0 = np.concatenate([np.full(offset, 20100, np.uint16), window_edge_image(np.random.default_rng(1))[0]])
    check_k1_u16(row0.reshape(1, 1, -1), invalid_val=0, p_lo=30.0, p_hi=40.0)


# ---------------------------------------------------------------- invalid_val and percentiles
PERCENTILES = [(2.0, 85.0), (0.0, 100.0), (50.0, 50.0), (2.5, 99.99), (85.0, 2.0), (100.0, 0.0)]


@gpu
@pytest.mark.parametrize("invalid_val", [0, 65535, 30000, 12345, None])
@pytest.mark.parametrize("p", PERCENTILES)
def test_k1_invalid_values_and_percentiles(cuda, invalid_val, p):
    rng = np.random.default_rng(5)
    u16 = depth_batch(rng, 3, 37, 23, invalid_frac=0.0)
    u16 = np.where(u16 == 12345, 12346, u16).astype(np.uint16)      # 12345: a value no pixel holds
    marks = rng.uniform(size=u16.shape) < 0.15
    u16[0][marks[0]] = 0
    u16[1][marks[1]] = 65535
    u16[2][marks[2]] = 30000
    u16[2, 0, :5] = 65535
    check_k1_u16(u16, invalid_val=invalid_val, p_lo=p[0], p_hi=p[1])


@gpu
@pytest.mark.parametrize("vals", [[4242], [63, 64], [127, 128], [64 * 517 - 1, 64 * 517], [65534, 65535], [0, 1], [9, 9]])
@pytest.mark.parametrize("p", PERCENTILES + [(33.3, 66.7)])
def test_k1_one_and_two_valid_pixels(cuda, vals, p):
    """n = 1 and 2, with neighbours on both sides of a 64-bin group of the statistics kernel"""
    img = np.full((1, 9, 13), 1000, np.uint16)
    flat = img.reshape(-1)
    flat[5:5 + len(vals)] = vals
    inv = 1000
    check_k1_u16(img, invalid_val=inv, p_lo=p[0], p_hi=p[1])


@gpu
def test_k1_ranks_straddling_64_bin_groups(cuda):
    """many pixels, wanted ranks whose two neighbours sit in adjacent 64-bin groups of different threads"""
    n = 1001
    v = np.full(n, 64 * 300 - 1, np.uint16)
    v[n // 2 + 1:] = 64 * 300
    v[:20] = 64 * 10 - 1
    v[20:21] = 64 * 10
    rng = np.random.default_rng(2)
    img = rng.permutation(v).reshape(1, 7, 143)
    for p in [(0.1, 50.0), (1.9, 2.0), (2.0, 50.05), (49.95, 85.0)]:
        check_k1_u16(img, invalid_val=None, p_lo=p[0], p_hi=p[1])


# ---------------------------------------------------------------- metres -> u16 (a1) at the truncation edges
def metre_edges():
    k = np.arange(0, 65536, 37, dtype=np.int64)
    at = (k / 256.0).astype(f32)
    below = np.nextafter(at, f32(-np.inf)).astype(f32)
    return np.concatenate([at, below[1:], f32([0.0, -0.0, 255.99998, np.nextafter(f32(256), f32(0))])])


SATURATING = {-1.5: 0, -0.001: 0, -np.inf: 0, np.nan: 0, -np.nan: 0, np.inf: 65535, 256.0: 65535, 300.0: 65535,
              1e30: 65535, -1e30: 0}


def test_metre_edges_are_in_range_and_distinct_from_their_neighbours():
    m = metre_edges()
    assert m.min() >= 0 and m.max() < 256
    q = (m * f32(256)).astype(np.uint16)
    at = (np.arange(1, 65536, 37) / 256.0).astype(f32)
    assert np.array_equal((at * f32(256)).astype(np.uint16), np.arange(1, 65536, 37))
    assert np.array_equal((np.nextafter(at, f32(0)) * f32(256)).astype(np.uint16), np.arange(1, 65536, 37) - 1)
    assert q.max() == 65535


@gpu
def test_metres_to_u16_at_every_edge_and_saturation(cuda):
    m = metre_edges()
    n = m.size
    pad = (-n) % 4 + 1                     # H*W = 1 (mod 4): the tail takes the scalar path
    sat_in = np.array(list(SATURATING.keys()), np.float64).astype(f32)
    sat_in[4] = -sat_in[3]                 # a NaN with the sign bit set
    sat_want = np.array(list(SATURATING.values()), np.uint16)
    x = np.concatenate([m, np.full(pad, 1.0, f32), sat_in])
    want = np.concatenate([(m * f32(256)).astype(np.uint16), np.full(pad, 256, np.uint16), sat_want])
    assert_bits(ops.scale_to_u16(x).cpu().numpy(), want, "scale_to_u16")
    _, u16 = ops.colorize_u16(LUT, depth_m=x.reshape(1, 1, -1), invalid_val=0)
    assert_bits(u16.cpu().numpy().ravel(), want, "colorize_u16's u16")


# ---------------------------------------------------------------- median and min-max
@gpu
@pytest.mark.parametrize("B,n", [(1, 1), (1, 2), (3, 7), (4, 8), (5, 4097), (2, 4099), (65, 37 * 23)])
@pytest.mark.parametrize("invalid_val", [None, 0, 500])
def test_median_u16(cuda, B, n, invalid_val):
    rng = np.random.default_rng(B * 100 + n)
    x = rng.integers(0, 1000, (B, n)).astype(np.uint16)
    if invalid_val is not None:
        x[:, -1] = np.uint16(invalid_val + 1)      # at least one valid pixel per image
    got = ops.median_u16(x, invalid_val=invalid_val).cpu().numpy()
    for b in range(B):
        v = x[b] if invalid_val is None else x[b][x[b] != invalid_val]
        assert_same_f64(got[b], np.median(v), f"median of image {b}")


@gpu
@pytest.mark.parametrize("B,H,W", [(1, 1, 1), (3, 37, 23), (65, 5, 7), (2, 64, 64)])
def test_minmax_colormap_batches_and_constant_images(cuda, B, H, W):
    rng = np.random.default_rng(H * W)
    d = rng.integers(0, 65536, (B, H, W)).astype(np.uint16)
    d[0] = 777                                # max == min: 0/0, which NumPy casts to 0 on this platform and the kernel pins
    lut = mdem.get_cmap_lut("jet")[:, :3].copy()
    gray, bgr = ops.minmax_colormap(d, lut_bgr=lut)
    gray, bgr = gray.cpu().numpy(), bgr.cpu().numpy()
    for b in range(B):
        mn, mx = float(d[b].min()), float(d[b].max())
        if mn == mx:
            want = np.zeros(d[b].shape, np.uint8)
        else:
            want = oracle.mdem.minmax_u8(d[b])
        assert_bits(gray[b], want, f"gray of image {b}")
        assert_bits(bgr[b], lut[want], f"colour of image {b}")


# ====================================================================================== K1f: float32 images
def check_k1f(value, invalid_val=None, vmin=None, vmax=None, p_lo=2.0, p_hi=85.0):
    """GPU vs np.percentile (vmin / vmax) and oracle.mdem.colorize (RGBA), image by image"""
    value = np.ascontiguousarray(value, dtype=f32)
    rgba, stats = ops.colorize_f32(LUT, value, invalid_val=invalid_val, vmin=vmin, vmax=vmax, p_lo=p_lo, p_hi=p_hi, return_stats=True)
    rgba, stats = rgba.cpu().numpy(), stats.cpu().numpy()
    with np.errstate(all="ignore"):
        for b in range(value.shape[0]):
            img = value[b]
            inv = np.nan if invalid_val is None else f32(invalid_val)
            valid = img[~(img == inv)]
            lo = np.percentile(valid, p_lo) if vmin is None else f32(vmin)
            hi = np.percentile(valid, p_hi) if vmax is None else f32(vmax)
            assert_same_f64(stats[b, 0], lo, f"vmin of image {b}")
            assert_same_f64(stats[b, 1], hi, f"vmax of image {b}")
            # the percentile side as np.percentile returns it (np.float32), an explicit side as the caller's Python float
            ref = oracle.mdem.colorize(img.copy(), LUT, vmin=lo if vmin is None else vmin, vmax=hi if vmax is None else vmax,
                                       invalid_val=inv).reshape(rgba[b].shape)
            if (p_lo, p_hi) == (2.0, 85.0) and vmin is None and vmax is None:
                assert_bits(oracle.mdem.colorize(img.copy(), LUT, invalid_val=inv).reshape(ref.shape), ref, "reference's own percentiles")
            assert_bits(rgba[b], ref, f"rgba of image {b}")
    return rgba, stats


FMAX = np.finfo(f32).max
NEG_NAN = np.array([0xFFC00001], np.uint32).view(f32)[0]
POS_NAN = np.array([0x7FC00123], np.uint32).view(f32)[0]


def special_image(rng, case):
    v = rng.uniform(0.2, 4.0, (1, 37, 23)).astype(f32)
    flat = v.reshape(-1)
    if case == "one_nan":
        flat[100] = np.nan
    elif case == "one_negative_nan":
        flat[7] = NEG_NAN
    elif case == "many_nan":
        flat[::3] = POS_NAN
        flat[1::7] = NEG_NAN
    elif case == "infinities":
        flat[::11] = np.inf
        flat[5::13] = -np.inf
    elif case == "plus_inf_only":
        flat[:40] = np.inf
    elif case == "signed_zeros":
        flat[::2] = -0.0
        flat[1::4] = 0.0
    elif case == "subnormals":
        flat[:] = (rng.integers(1, 1 << 23, flat.size).astype(np.uint32)).view(f32)
        flat[::5] = -flat[::5]
    elif case == "flt_max":
        flat[::4] = FMAX
        flat[1::4] = -FMAX
    elif case == "all_invalid_but_one":
        flat[:] = 0.0
        flat[333] = 1.25
    return v


SPECIAL_CASES = ["one_nan", "one_negative_nan", "many_nan", "infinities", "plus_inf_only", "signed_zeros", "subnormals",
                 "flt_max", "all_invalid_but_one"]


@gpu
@pytest.mark.parametrize("case", SPECIAL_CASES)
@pytest.mark.parametrize("invalid_val", [0.0, None, float("nan"), -0.0])
def test_k1f_special_values(cuda, case, invalid_val):
    v = special_image(np.random.default_rng(3), case)
    if case == "all_invalid_but_one" and invalid_val is None:
        pytest.skip("needs an invalid marker")
    check_k1f(v, invalid_val=invalid_val)


@gpu
def test_k1f_nan_paints_every_valid_pixel_bad(cuda):
    """np.percentile of data holding a NaN is NaN, so the reference paints every valid pixel (0, 0, 0, 0)"""
    v = special_image(np.random.default_rng(4), "one_nan")
    v.reshape(-1)[:50] = 0.0
    rgba, stats = check_k1f(v, invalid_val=0.0)
    assert np.isnan(stats).all()
    valid = v[0] != 0
    assert not rgba[0][valid].any() and (rgba[0][~valid] == [128, 128, 128, 255]).all()
    # an explicit side stays as given; the percentile side is still NaN
    _, st = check_k1f(v, invalid_val=0.0, vmin=0.5)
    assert st[0, 0] == 0.5 and np.isnan(st[0, 1])
    _, st = check_k1f(v, invalid_val=0.0, vmin=0.5, vmax=3.0)
    assert st[0].tolist() == [0.5, 3.0]


@gpu
@pytest.mark.parametrize("lo,hi", [(0.1, None), (None, 3.3), (0.1, 3.3), (1e-46, 1e39), (2.0000001, 2.0000002), (2.00000001, 2.00000002),
                                   (3.3, 0.1), (None, 2.00000001)])
def test_k1f_explicit_bounds_not_representable_in_float32(cuda, lo, hi):
    v = np.random.default_rng(6).uniform(0.0, 4.0, (2, 29, 31)).astype(f32)
    v[1] *= f32(0.5)
    check_k1f(v, invalid_val=0.0, vmin=lo, vmax=hi)


def lerp_branch_pair():
    """float32 a < b for which NumPy's two _lerp branches at t = 0.5 round differently (NumPy takes b - diff * 0.5)"""
    rng = np.random.default_rng(7)
    while True:
        a = f32(rng.uniform(0.5, 4.0))
        b = f32(a * f32(rng.uniform(1.0, 3.0)))
        d = f32(b - a)
        if f32(a + d * f32(0.5)) != f32(b - d * f32(0.5)):
            return a, b


def test_lerp_branch_pair_takes_numpys_second_branch():
    a, b = lerp_branch_pair()
    d = f32(b - a)
    first, second = f32(a + d * f32(0.5)), f32(b - d * f32(0.5))
    assert first != second
    x = np.array([a - 1, a, b, b + 1], f32)            # n = 4, p = 50: virtual index 1.5, gamma exactly 0.5
    assert np.percentile(x, 50) == second


@gpu
def test_k1f_median_of_even_n_takes_the_second_lerp_branch(cuda):
    a, b = lerp_branch_pair()
    rng = np.random.default_rng(8)
    half = 500
    lo = rng.uniform(0.1, float(a), half - 1).astype(f32)
    hi = rng.uniform(float(b), float(b) + 3, half - 1).astype(f32)
    v = rng.permutation(np.concatenate([lo, [a, b], hi]).astype(f32)).reshape(1, 20, 50)
    _, stats = check_k1f(v, p_lo=50.0, p_hi=50.0)
    d = f32(b - a)
    assert stats[0, 0] == float(f32(b - d * f32(0.5)))


def big_n_values(n, p_lo, p_hi):
    """n distinct float32 values with a wide gap right after each wanted rank, so that a different gamma shows"""
    idx = []
    for p in (p_lo, p_hi):
        virt = f32(n - 1) * (f32(p) / f32(100))
        idx.append(int(np.floor(virt)))
    keys = np.arange(n, dtype=np.uint32) + np.uint32(0x3F800000)      # consecutive floats from 1.0
    v = keys.view(f32).copy()
    v[idx[0] + 1:] += f32(1000.0)
    v[idx[1] + 1:] += f32(100000.0)
    return v


def np_lerp32(a, b, t):
    d = f32(b - a)
    return f32(b - d * (f32(1) - t)) if t >= 0.5 else f32(a + d * t)


def test_big_n_virtual_index_rounds_in_float32():
    """above 2^24 the float32 virtual index differs from the one computed in double and rounded once, and the
    constructed values make that difference change the percentile"""
    for extra in (2, 4):
        n = (1 << 24) + extra
        v = big_n_values(n, 2.0, 85.0)
        assert np.all(np.diff(v) >= 0)          # sorted (the percentiles below index it directly)
        for p in (2.0, 85.0):
            q = f32(p) / f32(100)
            v32, v64 = f32(n - 1) * q, f32(np.float64(n - 1) * np.float64(q))
            i32, i64 = int(np.floor(v32)), int(np.floor(v64))
            want = np_lerp32(v[i32], v[min(i32 + 1, n - 1)], f32(v32 - f32(i32)))
            other = np_lerp32(v[i64], v[min(i64 + 1, n - 1)], f32(v64 - f32(i64)))
            assert np.percentile(v, p) == want
            if p == 2.0:            # (at 85 % the index is above 2^23: both round to the same float32)
                assert v32 != v64 and want != other


@gpu
@pytest.mark.parametrize("extra", [2, 3, 4, 101])
def test_k1f_more_than_2_24_valid_pixels(cuda, extra):
    n = (1 << 24) + extra
    v = big_n_values(n, 2.0, 85.0)
    v = np.random.default_rng(extra).permutation(v).reshape(1, 1, n)
    check_k1f(v)


@gpu
def test_k1f_batches_with_own_distributions(cuda):
    """per image: all wanted ranks in one high-half bin, in two, in four distinct bins; and a shifted copy"""
    rng = np.random.default_rng(9)
    H, W = 33, 35
    n = H * W
    one_bin = (np.uint32(0x3FC00000) + rng.integers(0, 65536, n).astype(np.uint32)).view(f32)
    two = np.where(rng.uniform(size=n) < 0.5, one_bin, (np.uint32(0x40400000) + rng.integers(0, 65536, n).astype(np.uint32)).view(f32))
    wide = rng.uniform(-50, 50, n).astype(f32)
    expo = np.exp(rng.normal(0, 4, n)).astype(f32)
    v = np.stack([one_bin, two, wide, expo, wide + f32(1000)]).reshape(5, H, W).astype(f32)
    for p in [(2.0, 85.0), (0.0, 100.0), (50.0, 50.0), (49.9, 50.1)]:
        check_k1f(v, p_lo=p[0], p_hi=p[1])


# ====================================================================================== a4: uint16 -> metres
A4_SCALES = [1000.0, 5000.0, 256.0, 1.0, 0.1, 3.7]


def a4_depth(scale):
    return np.arange(65536, dtype=np.uint16).astype(f32) / f32(scale)


def a4_thresholds(scale):
    exact = float(a4_depth(scale)[3333])                 # a threshold exactly equal to some f32(u) / scale
    return [3.0, 3.3, 0.7, 2.9, 0.1, exact, float(np.nextafter(exact, np.inf)), 0.0, None, float("inf")]


def a4_threshold_f32(t):
    """the float32 threshold the host hands the kernels: the smallest float >= t (0 = no truncation)"""
    if t is None or not t > 0:
        return f32(0)
    x = f32(t)
    return np.nextafter(x, f32(np.inf)) if float(x) < t else x


def a4_oracle(u16, scale, t):
    """oracle.o3d.depth_from_u16; 0 and None mean "no truncation" here (the oracle itself would zero everything)"""
    return oracle.o3d.depth_from_u16(u16, scale, float("inf") if t is None or t <= 0 else t)


def test_a4_float_threshold_equals_the_double_comparison():
    for scale in A4_SCALES:
        p = a4_depth(scale)
        for t in a4_thresholds(scale):
            tf = a4_threshold_f32(t)
            kept_gpu = ~((tf > 0) & (p >= tf))
            kept_ref = np.ones(p.shape, bool) if t is None or t <= 0 else ~(p.astype(np.float64) >= t)
            assert np.array_equal(kept_gpu, kept_ref), (scale, t)
    # rounding the threshold to nearest instead drops depths the reference keeps
    for scale, t, u in [(1000.0, 3.3, 3300), (5000.0, 0.7, 3500)]:
        p = a4_depth(scale)[u]
        assert p >= f32(t) and not float(p) >= t


@gpu
@pytest.mark.parametrize("scale", A4_SCALES)
def test_a4_all_inputs_every_threshold(cuda, scale):
    u = np.arange(65536, dtype=np.uint16).reshape(256, 256)
    color = np.zeros((256, 256, 3), np.uint8)
    for t in a4_thresholds(scale):
        want = a4_oracle(u, scale, t)
        assert_bits(ops.depth_from_u16(u, scale, t).cpu().numpy(), want, f"depth_from_u16 scale {scale} trunc {t}")
        rgbd = RGBDImage.create_from_color_and_depth(color, u, depth_scale=scale, depth_trunc=t)
        assert_bits(rgbd.depth.cpu().numpy(), want, f"create_from_color_and_depth scale {scale} trunc {t}")
        odd = u.reshape(-1)[:65535].reshape(5, 13107)       # H*W odd: the scalar tail
        assert_bits(ops.depth_from_u16(odd, scale, t).cpu().numpy(), want.reshape(-1)[:65535].reshape(5, 13107))


def wall_frames():
    """a 32x24 view of a wall at exactly 3.3 m (u = 3300 at scale 1000), then one with 3299 / 3300 / 3301 mixed"""
    f0 = np.full((24, 32), 3300, np.uint16)
    f1 = np.array([3299, 3300, 3301], np.uint16)[np.random.default_rng(10).integers(0, 3, (24, 32))]
    return np.stack([f0, f1])


@gpu
def test_a4_fused_integration_keeps_the_wall_at_the_threshold(cuda):
    K = (400.0, 400.0, 16.0, 12.0)
    E = np.stack([np.eye(4), np.eye(4)])
    vl, trunc = 0.004, 0.02
    origin = np.array([-0.064, -0.064, 3.3 - 0.064])
    u16 = wall_frames()
    vol = DenseTSDFVolume(vl, trunc, 32, origin, color=False, device=cuda)
    vol.integrate_u16_batch(torch.from_numpy(u16).to(cuda), None, PinholeCameraIntrinsic(32, 24, *K), E, 1000.0, 3.3)
    V = oracle.o3d.Volume(32, vl, trunc, origin)
    for i in range(2):
        V.integrate(oracle.o3d.depth_from_u16(u16[i], 1000.0, 3.3), K, E[i])
    t, w = (x.cpu().numpy() for x in vol.export_dense())
    assert V.grid("weight").max() == 2.0, "the oracle integrates the wall"
    assert_bits(w, V.grid("weight"), "weight")
    assert_bits(t, V.grid("tsdf"), "tsdf")


@gpu
def test_a4_unit_bounds_of_uint16_frames_at_the_threshold(cuda):
    K = (400.0, 400.0, 16.0, 12.0)
    E = np.stack([np.eye(4), np.eye(4)])
    vl = 0.004
    ul = 32 * vl
    v = DenseTSDFVolume(vl, 0.02, 64, (-ul, -ul, 25 * ul), color=False, device=cuda, unit_activation=True)
    intr = PinholeCameraIntrinsic(32, 24, *K)
    u16 = wall_frames()
    for frames in (u16, u16[:1]):           # frame 0 alone: every pixel is 3300, so rounding 3.3 down leaves no point
        Ef = E[:len(frames)]
        for scale, t in [(1000.0, 3.3), (1000.0, 3.0), (1000.0, None)]:
            ref = torch.from_numpy(a4_oracle(frames, scale, t)).to(cuda)
            got = v.unit_bounds(torch.from_numpy(np.ascontiguousarray(frames)).to(cuda), intr, Ef, scale, t)
            want = v.unit_bounds(ref, intr, Ef)
            assert (got is None) == (want is None) and (got is None or np.array_equal(got, want)), (t, got, want)
            assert (got is None) == (t == 3.0), (t, got)


@gpu
def test_a4_prepared_launch_keeps_the_wall_at_the_threshold(cuda):
    """the two-stream halves (bslam_tsdf_prepare_u16 + bslam_tsdf_integrate_prepared) at trunc 3.3: the scratch holds
    the a4 conversion of the oracle and the volume equals the oracle's"""
    K = (400.0, 400.0, 16.0, 12.0)
    E = np.stack([np.eye(4), np.eye(4)])
    vl, trunc = 0.004, 0.02
    origin = np.array([-0.064, -0.064, 3.3 - 0.064])
    u16 = wall_frames()
    vol = DenseTSDFVolume(vl, trunc, 32, origin, color=False, device=cuda)
    scratch = torch.empty(u16.shape, dtype=torch.float32, device=cuda)
    vol.prepare_u16(torch.from_numpy(u16).to(cuda), PinholeCameraIntrinsic(32, 24, *K), E, scratch, 1000.0, 3.3)
    vol.integrate_prepared()
    torch.cuda.synchronize()
    want = np.stack([oracle.o3d.depth_from_u16(u16[i], 1000.0, 3.3) for i in range(2)])
    assert_bits(scratch.cpu().numpy(), want, "prepared a4 scratch")
    V = oracle.o3d.Volume(32, vl, trunc, origin)
    for i in range(2):
        V.integrate(want[i], K, E[i])
    t, w = (x.cpu().numpy() for x in vol.export_dense())
    assert V.grid("weight").max() == 2.0
    assert_bits(w, V.grid("weight"), "weight")
    assert_bits(t, V.grid("tsdf"), "tsdf")


# ====================================================================================== K2: back-projection
# Error bound of the kernel's coordinates against the exact value of the reference's formula
#   p_r = M_r0 x + M_r1 y + M_r2 d + M_r3,   x = (u - cx) d / fx,   y = (v - cy) d / fy      (float64 M, K)
# The kernel evaluates, with e = 2^-24 the float32 unit roundoff:
#   K cast to float32:   cx' = cx (1 + d1), fx' = fx (1 + d2)                                |di| <= e
#   inv_fx = f32(1 / fx'):                                                                   one rounding
#   x' = f32(f32(f32(u - cx') * d) * inv_fx):                                                three roundings
#   so |x' - x| <= 5e |x| + e |cx| d / fx   (first order; the same for y)
#   the pose cast to float32: M'_rc = M_rc (1 + d),                                           |d| <= e
#   p'_r = fmaf(M'_r0, x', fmaf(M'_r1, y', fmaf(M'_r2, d, M'_r3))): each fmaf rounds once, so the innermost
#   error reaches (|M_r2 d| + |M_r3|) three times, |M_r1 y| twice and |M_r0 x| once.
# Summing: |p'_r - p_r| <= e (7 |M_r0 x| + 8 |M_r1 y| + 4 |M_r2 d| + 4 |M_r3| + |M_r0| d |cx| / fx + |M_r1| d |cy| / fy).
# bp_bound takes 8 for every term (second-order terms and the float64 reference's own ~2^-52 are far below that slack)
# plus 2^-146 absolute for subnormal intermediates.
def bp_pixels(depth, stride):
    H, W = depth.shape
    v, u = np.mgrid[0:H:stride, 0:W:stride]
    d = depth[::stride, ::stride]
    return u.ravel().astype(np.float64), v.ravel().astype(np.float64), d.ravel().astype(np.float64)


def bp_bound(u, v, d, K, M):
    fx, fy, cx, cy = (float(k) for k in K)
    x, y = (u - cx) * d / fx, (v - cy) * d / fy
    A = np.abs(M)
    s = A[:, 0][None] * np.abs(x)[:, None] + A[:, 1][None] * np.abs(y)[:, None] + A[:, 2][None] * np.abs(d)[:, None] + A[:, 3][None]
    k = A[:, 0][None] * (d * abs(cx) / fx)[:, None] + A[:, 1][None] * (d * abs(cy) / fy)[:, None]
    return EPS * (8.0 * s + k) + 2.0 ** -146, s


def bp_exact(u, v, d, K, M):
    """the reference's formula in float64 (like orc_backproject, any evaluation order: its error is ~2^-52)"""
    fx, fy, cx, cy = (float(k) for k in K)
    x, y = (u - cx) * d / fx, (v - cy) * d / fy
    return ((M[:, 0][None] * x[:, None] + M[:, 1][None] * y[:, None]) + M[:, 2][None] * d[:, None]) + M[:, 3][None]


def bp_emulate(depth, K, M, stride=1):
    """the kernel's float32 operation order on the CPU (fmaf as a float64 fma rounded once more: off by at most
    a double rounding, far inside the bound)"""
    u, v, d = bp_pixels(depth, stride)
    ok = d > 0
    u, v = u[ok].astype(f32), v[ok].astype(f32)
    d = d[ok].astype(f32)
    fx, fy, cx, cy = (f32(k) for k in K)
    ifx, ify = f32(1.0 / float(fx)), f32(1.0 / float(fy))
    x = ((u - cx) * d) * ifx
    y = ((v - cy) * d) * ify
    Mf = M.astype(f32)

    def fma(a, b, c):
        return (np.float64(a) * b.astype(np.float64) + np.asarray(c, np.float64)).astype(f32)

    return np.stack([fma(Mf[r, 0], x, fma(Mf[r, 1], y, fma(Mf[r, 2], d, np.full(d.shape, Mf[r, 3])))) for r in range(3)], 1)


def bp_pose(rng, big_t=False):
    a = rng.normal(size=3)
    a *= rng.uniform(0.1, 2.5) / np.linalg.norm(a)
    th = np.linalg.norm(a)
    k = a / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    R = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx
    E = np.eye(4)
    E[:3, :3] = R
    E[:3, 3] = rng.uniform(-3, 3, 3) if big_t else rng.uniform(-0.2, 0.2, 3)
    return E


MEAN_MIN_POINTS, MEAN_LIMIT = 800, 0.15


def bp_check(xyz, counts, depth, K, E, stride=1, valid_only=True, rgb_out=None, rgb_in=None, mean_check=False):
    """count and order exact against orc_backproject, coordinates within bp_bound, colour bit-exact.  mean_check: also
    the per-image mean error against the formula on the kernel's own inputs.  Rounding leaves that mean near zero only
    for some geometries: random depths in the frames of the chunk and scan tests stay below 0.06 (the CPU emulation over
    hundreds of poses), while the bench's k / 1000 m depths or a small fx with a small translation reach about 0.1
    without any error in the inputs, so the check runs where it has a margin."""
    off = 0
    for i in range(depth.shape[0]):
        ref, refc = oracle.o3d.backproject(depth[i], K, E[i], rgb=None if rgb_in is None else rgb_in[i], stride=stride, valid_only=valid_only)
        n = int(counts[i])
        assert n == len(ref), (i, n, len(ref))
        got = xyz[off:off + n].astype(np.float64)
        u, v, d = bp_pixels(depth[i], stride)
        keep = (d > 0) if valid_only else np.ones(d.shape, bool)
        u, v, d = u[keep], v[keep], d[keep]
        M = inverse4x4(E[i])[:3, :]
        with np.errstate(all="ignore"):
            bound, _ = bp_bound(u, v, d, K, M)
            fin = np.isfinite(ref)
            assert np.array_equal(np.isnan(got), np.isnan(ref)), f"NaN mask of image {i}"
            assert np.array_equal(got[~fin & ~np.isnan(ref)], ref[~fin & ~np.isnan(ref)]), f"infinities of image {i}"
            err = np.abs(got - ref)
            assert (err[fin] <= bound[fin]).all(), f"image {i}: worst error / bound {np.max(err[fin] / bound[fin])}"
            # no systematic error against the formula on the kernel's own float32 inputs (a pose entry one float32 ulp
            # off stays inside the bound but moves this mean; over 1 000 points its spread is about 0.02)
            pts = fin.all(1) & (d > 0)
            if mean_check and pts.sum() >= MEAN_MIN_POINTS:
                _, s = bp_bound(u[pts], v[pts], d[pts], K, M)
                m = np.mean((got[pts] - bp_exact_kernel_inputs(u[pts], v[pts], d[pts], K, M)) / (EPS * s), 0)
                assert (np.abs(m) < MEAN_LIMIT).all(), f"image {i}: mean error {m} of the bound's scale"
        if rgb_out is not None:
            gc, rc = rgb_out[off:off + n], refc.astype(f32)
            assert np.array_equal(np.isnan(gc), np.isnan(rc)), f"colour NaN mask of image {i}"
            assert_bits(np.nan_to_num(gc), np.nan_to_num(rc), f"colour of image {i}")
        off += n
    assert off == xyz.shape[0]


def test_colour_quotient_is_the_float32_quotient():
    c = np.arange(256)
    assert_bits((c / 255.0).astype(f32), c.astype(f32) / f32(255))


def test_bp_bound_holds_for_the_kernel_order_and_is_tight():
    rng = np.random.default_rng(11)
    H, W = 240, 320
    K = (957.3, 951.1, 161.7, 118.2)
    depth = rng.uniform(0.05, 3.0, (H, W)).astype(f32)
    depth[rng.uniform(size=(H, W)) < 0.05] = 0
    depth[:, 161:163] = 0.4                      # columns at u ~ cx
    depth[0, :8] = [1e-40, 1e-30, 1e30, 3e4, 7e-3, 0.4, 0.40000001, 65.535]
    E = bp_pose(rng)
    M = inverse4x4(E)[:3, :]
    u, v, d = bp_pixels(depth, 1)
    ok = d > 0
    u, v, d = u[ok], v[ok], d[ok]
    ref, _ = oracle.o3d.backproject(depth, K, E)
    bound, s = bp_bound(u, v, d, K, M)
    emu = bp_emulate(depth, K, M).astype(np.float64)
    assert (np.abs(emu - ref) <= bound).all()
    # cx shifted by 1/256 px breaks the bound
    Ks = (K[0], K[1], K[2] + 1 / 256, K[3])
    assert (np.abs(bp_emulate(depth, Ks, M).astype(np.float64) - ref) > bound).any()
    # a pose row perturbed by one float32 ulp: inside the per-point bound, but a systematic error that the mean of
    # the normalised error against the formula evaluated exactly on the kernel's own inputs shows
    exact = bp_exact_kernel_inputs(u, v, d, K, M)
    mean_ok = np.mean((emu - exact) / (EPS * s), 0)
    assert (np.abs(mean_ok) < MEAN_LIMIT).all(), mean_ok
    Mf = M.astype(f32)
    terms = np.array([np.mean((u - K[2]) * d / K[0]), np.mean((v - K[3]) * d / K[1]), np.mean(d), 1.0])
    r = int(np.argmax(np.abs(Mf * terms).sum(1) / s.mean(0)))
    Mp = Mf.copy()
    Mp[r] = np.nextafter(Mf[r], (np.sign(Mf[r]) * np.sign(terms) * np.inf).astype(f32))
    emu_p = bp_emulate(depth, K, Mp.astype(np.float64)).astype(np.float64)
    assert (np.abs(emu_p - ref) <= bound).all()
    assert abs(np.mean((emu_p - exact) / (EPS * s), 0)[r]) > 0.5


def test_mean_error_check_per_image_catches_one_ulp_poses():
    """bp_check's per-image mean, on 40 x 30 frames like the chunk tests: below MEAN_LIMIT for the kernel's order of
    operations, above it for most poses with a row one float32 ulp off"""
    rng = np.random.default_rng(15)
    K = (37.5, 36.0, 19.3, 15.1)
    clean, moved = [], []
    for i in range(120):
        d = random_frames(rng, 1, 30, 40)[0]
        M = inverse4x4(bp_pose(rng, big_t=True))[:3, :]
        u, v, dd = bp_pixels(d, 1)
        ok = dd > 0
        u, v, dd = u[ok], v[ok], dd[ok]
        assert ok.sum() >= MEAN_MIN_POINTS
        _, s = bp_bound(u, v, dd, K, M)
        exact = bp_exact_kernel_inputs(u, v, dd, K, M)
        clean.append(np.abs(np.mean((bp_emulate(d, K, M) - exact) / (EPS * s), 0)).max())
        Mf = M.astype(f32)
        r = i % 3
        Mf[r] = np.nextafter(Mf[r], (np.sign(Mf[r]) * np.inf).astype(f32))
        moved.append(abs(np.mean((bp_emulate(d, K, Mf.astype(np.float64)) - exact) / (EPS * s), 0)[r]))
    assert max(clean) < MEAN_LIMIT / 2
    assert np.mean(np.array(moved) > MEAN_LIMIT) > 0.8


def bp_exact_kernel_inputs(u, v, d, K, M):
    """the formula in float64 on what the kernel is handed: K and the pose rounded to float32, fx and fy replaced by
    1 / f32(1 / f32(fx)) (the kernel multiplies by that reciprocal).  The kernel's error against this is rounding
    alone, with no systematic part."""
    Kf = [float(f32(k)) for k in K]
    fx_eff, fy_eff = 1.0 / float(f32(1.0 / Kf[0])), 1.0 / float(f32(1.0 / Kf[1]))
    return bp_exact(u, v, d, (fx_eff, fy_eff, Kf[2], Kf[3]), M.astype(f32).astype(np.float64))


def run_bp(depth, K, E, stride=1, valid_only=True, color=None):
    out = ops.backproject(depth, K, E, color=color, stride=stride, valid_only=valid_only, return_counts=True)
    xyz, rgb, counts = (None if t is None else t.cpu().numpy() for t in out)
    return xyz, rgb, counts


def random_frames(rng, B, H, W, lo=0.05, hi=3.0, invalid=0.1):
    d = rng.uniform(lo, hi, (B, H, W)).astype(f32)
    d[rng.uniform(size=d.shape) < invalid] = 0
    return d


@gpu
@pytest.mark.parametrize("B", [1, 63, 64, 65, 129, 130])
def test_k2_pose_chunks(cuda, B):
    """emit launches carry at most 64 poses: every frame has its own pose, so a pose from the wrong chunk shows"""
    rng = np.random.default_rng(B)
    H, W = 30, 40
    depth = random_frames(rng, B, H, W)
    E = np.stack([bp_pose(rng, big_t=True) for _ in range(B)])
    K = (37.5, 36.0, 19.3, 15.1)
    rgb_in = rng.integers(0, 256, (B, H, W, 3)).astype(np.uint8)
    xyz, rgb, counts = run_bp(depth, K, E, color=rgb_in)
    bp_check(xyz, counts, depth, K, E, rgb_out=rgb, rgb_in=rgb_in, mean_check=True)


@gpu
@pytest.mark.parametrize("B,H,W", [(1100, 8, 8), (130, 480, 640)])
def test_k2_scan_over_more_than_1024_ctas(cuda, B, H, W):
    rng = np.random.default_rng(B)
    depth = random_frames(rng, B, H, W, invalid=0.3)
    E = np.stack([bp_pose(rng) for _ in range(B)])
    K = (W * 1.5, W * 1.5, W / 2 - 0.5, H / 2 + 0.25)
    xyz, _, counts = run_bp(depth, K, E)
    bp_check(xyz, counts, depth, K, E, mean_check=True)


@gpu
@pytest.mark.parametrize("stride", [1, 2, 3, 8, 16])
@pytest.mark.parametrize("B,H,W", [(1, 1, 1), (2, 1, 301), (3, 301, 1), (3, 37, 23), (2, 65535, 2), (1, 2, 65535), (2, 257, 129)])
def test_k2_strides_and_shapes(cuda, stride, B, H, W):
    rng = np.random.default_rng(stride * 1000 + H + W)
    depth = random_frames(rng, B, H, W, invalid=0.2)
    E = np.stack([bp_pose(rng) for _ in range(B)])
    K = (max(W, 2) * 0.9, max(H, 2) * 0.9, W / 2, H / 3)
    xyz, _, counts = run_bp(depth, K, E, stride=stride)
    bp_check(xyz, counts, depth, K, E, stride=stride)
    xyz, _, counts = run_bp(depth, K, E, stride=stride, valid_only=False)
    bp_check(xyz, counts, depth, K, E, stride=stride, valid_only=False)


@gpu
@pytest.mark.parametrize("valid_only", [True, False])
@pytest.mark.parametrize("with_color", [True, False])
def test_k2_special_depths(cuda, valid_only, with_color):
    rng = np.random.default_rng(12)
    B, H, W = 3, 17, 33                                  # H*W odd: images 1 and 2 are not 16-byte aligned
    depth = random_frames(rng, B, H, W, invalid=0.0)
    specials = np.array([np.nan, NEG_NAN, np.inf, -np.inf, -0.0, 0.0, -1.0, 1e-40, -1e-40, 1e-45, 1e30, 1e34, FMAX / 1e6], f32)
    for b in range(B):
        flat = depth[b].reshape(-1)
        flat[rng.choice(flat.size, 3 * specials.size, replace=False)] = np.tile(specials, 3)
    depth[0, 5, 16] = np.inf                             # u == cx: 0 * inf
    E = np.stack([bp_pose(rng) for _ in range(B)])
    K = (30.0, 30.0, 16.0, 8.0)
    rgb_in = rng.integers(0, 256, (B, H, W, 3)).astype(np.uint8) if with_color else None
    xyz, rgb, counts = run_bp(depth, K, E, valid_only=valid_only, color=rgb_in)
    bp_check(xyz, counts, depth, K, E, valid_only=valid_only, rgb_out=rgb, rgb_in=rgb_in)
    if with_color and not valid_only:
        refc = np.concatenate([oracle.o3d.backproject(depth[i], K, E[i], rgb=rgb_in[i], valid_only=False)[1] for i in range(B)])
        assert np.array_equal(np.isnan(rgb), np.isnan(refc))


@gpu
def test_k2_bound_is_tight_on_the_gpu(cuda):
    """the GPU against the float64 formula: inside bp_bound everywhere and no systematic error
    (a pose row one float32 ulp off shows here; see test_bp_bound_holds_for_the_kernel_order_and_is_tight)"""
    rng = np.random.default_rng(13)
    H, W = 480, 640
    depth = random_frames(rng, 1, H, W, invalid=0.05)
    K = (957.3, 951.1, 321.7, 238.2)
    E = bp_pose(rng)
    xyz, _, counts = run_bp(depth, K, E[None])
    bp_check(xyz, counts, depth, K, E[None])
    M = inverse4x4(E)[:3, :]
    u, v, d = bp_pixels(depth[0], 1)
    ok = d > 0
    _, s = bp_bound(u[ok], v[ok], d[ok], K, M)
    exact = bp_exact_kernel_inputs(u[ok], v[ok], d[ok], K, M)
    m = np.mean((xyz.astype(np.float64) - exact) / (EPS * s), 0)
    assert (np.abs(m) < MEAN_LIMIT).all(), m


# ---------------------------------------------------------------- the C ABI: capacity, guard bands, argument errors
SENT = 0x7FBADBAD


def sentinel(n, dtype=torch.float32):
    return torch.full((n,), SENT, dtype=torch.int32, device="cuda").view(dtype)


@gpu
@pytest.mark.parametrize("with_color", [True, False])
def test_k2_capacity_and_guard_bands(cuda, with_color):
    rng = np.random.default_rng(14)
    B, H, W = 3, 37, 23
    depth = torch.from_numpy(random_frames(rng, B, H, W, invalid=0.3)).to(cuda)
    rgb_in = torch.from_numpy(rng.integers(0, 256, (B, H, W, 3)).astype(np.uint8)).to(cuda) if with_color else None
    E = np.stack([bp_pose(rng) for _ in range(B)])
    K = (30.0, 31.0, 11.0, 18.0)
    full_xyz, full_rgb, full_counts = run_bp(depth, K, E, color=rgb_in)
    total = int(full_counts.sum())
    L = _lib.load()
    Mp = np.ascontiguousarray(inverse4x4(E)[:, :3, :].reshape(B, 12), dtype=f32)
    Kf = np.ascontiguousarray(K, dtype=f32)
    G = 64
    for capacity in [0, 1, 255, 256, 257, total - 1, total]:
        xyz = sentinel(3 * (capacity + 2 * G))
        rgb = sentinel(3 * (capacity + 2 * G)) if with_color else None
        counts = torch.full((B + 1 + 2 * G,), -7, dtype=torch.int64, device=cuda)
        ws = torch.empty(L.bslam_backproject_workspace_bytes(B, H, W, 1), dtype=torch.uint8, device=cuda)
        rc = L.bslam_backproject(_lib.ptr(depth), _lib.ptr(rgb_in), B, H, W, 1, _lib.ptr(Kf), _lib.ptr(Mp), 1,
                                 ctypes.c_void_p(xyz.data_ptr() + 12 * G),
                                 None if rgb is None else ctypes.c_void_p(rgb.data_ptr() + 12 * G), capacity,
                                 ctypes.c_void_p(counts.data_ptr() + 8 * G), _lib.ptr(ws), _lib.stream_ptr(cuda))
        assert rc == 0
        torch.cuda.synchronize()
        c = counts.cpu().numpy()
        assert (c[:G] == -7).all() and (c[G + B + 1:] == -7).all()
        assert c[G:G + B].tolist() == full_counts.tolist() and c[G + B] == total
        for buf, full in ((xyz, full_xyz), (rgb, full_rgb)):
            if buf is None:
                continue
            a = buf.cpu().numpy().view(np.uint32).reshape(-1, 3)
            assert (a[:G] == SENT).all() and (a[G + capacity:] == SENT).all(), capacity
            assert_bits(a[G:G + capacity].view(f32), full[:capacity], f"first {capacity} rows")


@gpu
def test_k2_argument_errors(cuda):
    L = _lib.load()
    d = torch.zeros(16, dtype=torch.float32, device=cuda)
    out = torch.zeros(48, dtype=torch.float32, device=cuda)
    cnt = torch.zeros(4, dtype=torch.int64, device=cuda)
    ws = torch.zeros(4096, dtype=torch.uint8, device=cuda)
    K = np.array([1, 1, 0, 0], f32)
    M = np.zeros(12, f32)
    s = _lib.stream_ptr(cuda)

    def call(H, W, rgb=None, rgb8=None):
        return L.bslam_backproject(_lib.ptr(d), _lib.ptr(rgb8), 1, H, W, 1, _lib.ptr(K), _lib.ptr(M), 1, _lib.ptr(out), _lib.ptr(rgb), 1,
                                   _lib.ptr(cnt), _lib.ptr(ws), s)

    assert call(65536, 1) == -1 and call(1, 65536) == -1
    assert call(65535, 32769) == -1                      # H * W >= 2^31
    assert call(4, 4, rgb=out) == -1                     # colour output without the RGB8 image
    assert call(4, 4) == 0


# ====================================================================================== full size (BASELINE configs[2])
def bench_frames(B, dev):
    cfg = S.config("laparoscopy512")
    E = cfg["extrinsics"](cfg["frames"])
    Eb = E[np.linspace(0, len(E) - 1, 64).astype(int)]
    if B == 65:
        Eb = np.concatenate([Eb, E[7:8]])
    K = tuple(k * 3.0 for k in cfg["K"])
    d, _ = S.render(cfg["surface"], Eb, K=K, W=1920, H=1080, device=dev, with_color=False)
    return (d.to(torch.float32) / 1000.0).contiguous(), K, Eb


@gpu
@pytest.mark.slow
def test_k1_bench_shape_64x1080p(cuda):
    metres, _, _ = bench_frames(64, cuda)
    rgba, u16 = ops.colorize_u16(LUT, depth_m=metres, invalid_val=0)
    m = metres.cpu().numpy()
    want = (m * f32(256)).astype(np.uint16)
    assert_bits(u16.cpu().numpy(), want, "u16")
    rgba = rgba.cpu().numpy()
    for b in range(64):
        assert_bits(rgba[b], oracle.mdem.colorize(want[b], LUT, invalid_val=0), f"rgba of image {b}")


@gpu
@pytest.mark.slow
@pytest.mark.parametrize("B", [64, 65])
def test_k2_bench_shape_1080p(cuda, B):
    metres, K, Eb = bench_frames(B, cuda)
    xyz, _, counts = run_bp(metres, K, Eb)
    bp_check(xyz, counts, metres.cpu().numpy(), K, Eb)
