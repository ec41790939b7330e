"""Brick integration (`brick_integrate_kernel` and its cull) at the edges of its variants and shortcuts -- `-m gpu`.

The suite's other parity tests integrate smooth renders from realistic trajectories into boxes of at most
256^3, so they exercise one kernel instantiation (4 z layers per warp with the long-chain phase) and reach
the cull's boundaries only by chance.  Here every case integrates the same f32 frames (or the same u16
frames through the fused path) on the GPU and in the CPU oracle and asserts, bit for bit:
  * tsdf and weight of the exported grids (compared as uint32 bit patterns, so +0 / -0 count),
  * colour, when present,
  * the per-frame update counts, and the dry run's (`count_updates`) counts.
The frames are NumPy geometry (planes, steps, spikes, noise, holes) chosen so that each case controls which
boundary it hits:
  A. the production instantiations (8 z layers per warp without the long-chain phase: the 512^3 bench),
     and the long-chain phase with chains that actually reach it;
  B. the cull's classes -- near (IEEE projection), inner (no bounds test), free (t = 1), dropped -- at
     camera placements, rotations, principal points and depth content that sit on their boundaries;
  C. the update arithmetic at its preconditions: weights around 2^24, tiny / signed-zero / subnormal tsdf,
     t == 0 updates (exact-depth frames) that take the out-of-line division;
  D. the launch structure: batch sizes around the cull and mask-word boundaries, the frame chunking, the
     tile-pyramid batch limit, the image-size limits.
The CPU tests at the bottom check the generators themselves against the oracle alone."""
import numpy as np
import pytest
import torch

import oracle
from bodyslam_b200.geometry import PinholeCameraIntrinsic

TWO24 = float(2 ** 24)

# ---------------------------------------------------------------- float32 geometry as the kernels form it


def voxel_centres(n, origin, vl, start=0):
    """float((double)(half + vl * (float)i) + origin) for i = start .. start + n - 1 (Open3D's voxel centre, f32)"""
    vlf = np.float32(vl)
    half = np.float32(vlf * np.float32(0.5))
    i = np.arange(start, start + n, dtype=np.float32)
    return ((half + vlf * i).astype(np.float64) + float(origin)).astype(np.float32)


def camera_z(E, dims, vl, origin, gz0=0):
    """float32 camera-space z of every voxel [nx, ny, nz] under the brick-restart recurrence (oracle z_restart = 8):
    E * p evaluated at each brick base, + E[2, 2] * vl per layer in between, no FMA"""
    nx, ny, nz = dims
    Ef = np.asarray(E, dtype=np.float64).reshape(4, 4).astype(np.float32)
    px = voxel_centres(nx, origin[0], vl)[:, None, None]
    py = voxel_centres(ny, origin[1], vl)[None, :, None]
    pz = voxel_centres(nz, origin[2], vl, start=gz0)[None, None, :]
    direct = ((Ef[2, 0] * px + Ef[2, 1] * py) + Ef[2, 2] * pz) + Ef[2, 3]
    direct = np.broadcast_to(direct, (nx, ny, nz))
    dzz = np.float32(Ef[2, 2] * np.float32(vl))
    z = np.empty((nx, ny, nz), np.float32)
    for k in range(nz):
        z[:, :, k] = direct[:, :, k] if (gz0 + k) % 8 == 0 else z[:, :, k - 1] + dzz
    return z


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


def oblique(rng):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    a, b, c, d = q
    return np.array([[a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c)],
                     [2 * (b * c + a * d), a * a - b * b + c * c - d * d, 2 * (c * d - a * b)],
                     [2 * (b * d - a * c), 2 * (c * d + a * b), a * a - b * b - c * c + d * d]])


def rotations(rng, n_oblique=3):
    """identity, every 90-degree multiple about each axis (exact zeros in E), a few oblique ones"""
    out = [np.eye(3)] + [rot(a, q) for a in range(3) for q in (1, 2, 3)]
    return out + [oblique(rng) for _ in range(n_oblique)]


# ---------------------------------------------------------------- depth content


def plane_depth(H, W, K, d0, slope=(0.0, 0.0)):
    """depth of a plane seen along the optical axis: d0 + slope . (x/z, y/z), f32"""
    fx, fy, cx, cy = K
    u = (np.arange(W) - cx) / fx
    v = (np.arange(H) - cy) / fy
    return (d0 + slope[0] * u[None, :] + slope[1] * v[:, None]).astype(np.float32)


def dirty(d, rng, noise=0.0, holes=0.0, specials=True):
    """noise, holes and, in f32 frames, the values the oracle skips or saturates: NaN, +inf, -0.0, negative"""
    d = d.copy()
    if noise:
        d += rng.normal(0.0, noise, d.shape).astype(np.float32)
    if holes:
        d[rng.random(d.shape) < holes] = 0.0
    if specials and d.size >= 8:
        idx = rng.choice(d.size, size=min(d.size, 8), replace=False)
        d.reshape(-1)[idx] = np.array([np.nan, np.inf, -0.0, -0.01, np.nan, np.inf, -0.0, -1.0], np.float32)[:len(idx)]
    return d


# ---------------------------------------------------------------- the GPU / oracle comparison


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def seed_oracle(V, state):
    if state is not None:
        t, w = state[:2]
        V.tsdf[:] = np.asarray(t, np.float32).reshape(-1)
        V.weight[:] = np.asarray(w, np.float32).reshape(-1)
        if V.color is not None and len(state) > 2:
            V.color[:] = np.asarray(state[2], np.float32).reshape(-1)


def make_volume(dims, vl, trunc, origin, color=False, gz0=0, z_total=None, unit=False, state=None, zpw=0, batch=0):
    from bodyslam_b200.tsdf import DenseTSDFVolume
    vol = DenseTSDFVolume(vl, trunc, dims, origin, color=color, device=torch.device("cuda", 0), gz0=gz0, z_total=z_total,
                          unit_activation=unit)
    if state is not None:
        t, w = (torch.from_numpy(np.ascontiguousarray(x, np.float32).reshape(-1)) for x in state[:2])
        c = torch.from_numpy(np.ascontiguousarray(state[2], np.float32).reshape(-1)) if (color and len(state) > 2) else None
        vol.import_dense(t, w, c)
    vol.set_z_split(zpw)
    vol.set_batch(batch)
    return vol


def gpu_integrate(vol, depth, K, E, rgb=None, u16=None):
    """one integrate call over all frames -> per-frame update counts"""
    F, H, W = depth.shape
    intr = PinholeCameraIntrinsic(W, H, *K)
    counts = torch.zeros(F, dtype=torch.int64, device="cuda")
    col = None if rgb is None else torch.from_numpy(np.ascontiguousarray(rgb)).cuda()
    if u16 is not None:
        vol.integrate_u16_batch(torch.from_numpy(u16).cuda(), col, intr, E, 1000.0, 3.0, update_counts=counts)
    else:
        vol.integrate_batch(torch.from_numpy(np.ascontiguousarray(depth)).cuda(), col, intr, E, update_counts=counts)
    return counts.cpu().numpy()


def oracle_integrate(V, depth, K, E, rgb=None, unit=False):
    return np.array([V.integrate_scalable(depth[i], K, E[i], rgb=None if rgb is None else rgb[i]) if unit
                     else V.integrate(depth[i], K, E[i], rgb=None if rgb is None else rgb[i]) for i in range(len(depth))], np.int64)


def assert_same(vol, V, color=False, what=""):
    out = vol.export_dense(with_color=color)
    t, w = out[0].cpu().numpy(), out[1].cpu().numpy()
    bad_w = int((bits(w) != bits(V.grid("weight"))).sum())
    assert bad_w == 0, f"{what}: {bad_w} weights differ"
    bad_t = bits(t) != bits(V.grid("tsdf"))
    assert not bad_t.any(), f"{what}: {int(bad_t.sum())} tsdf values differ, e.g. {t[bad_t][:4]} vs {V.grid('tsdf')[bad_t][:4]}"
    if color:
        c = out[2].cpu().numpy()
        ref = V.color.reshape(c.shape)
        bad_c = bits(c) != bits(ref)
        assert not bad_c.any(), f"{what}: {int(bad_c.sum())} colour values differ, e.g. {c[bad_c][:4]} vs {ref[bad_c][:4]}"


def check_case(depth, K, E, dims, vl, trunc, origin, rgb=None, gz0=0, z_total=None, unit=False, state=None, zpw=0, batch=0,
               u16=None, what="", stats=None):
    """integrate on the GPU and in the oracle from the same frames (and the same imported state); assert
    tsdf / weight / colour / per-frame counts / dry-run counts bit for bit.  -> (vol, V, counts)"""
    E = np.asarray(E, dtype=np.float64).reshape(-1, 4, 4)
    color = rgb is not None
    V = oracle.o3d.Volume(dims, vl, trunc, origin, gz0=gz0, with_color=color)
    seed_oracle(V, state)
    oc = oracle_integrate(V, depth, K, E, rgb, unit)
    vol = make_volume(dims, vl, trunc, origin, color, gz0, z_total, unit, state, zpw, batch)
    gc = gpu_integrate(vol, depth, K, E, rgb, u16)
    assert np.array_equal(gc, oc), f"{what}: per-frame update counts differ: {gc} vs {oc}"
    assert_same(vol, V, color, what)
    F, H, W = depth.shape
    vol.dry_stats(True)
    dc = vol.count_updates(torch.from_numpy(np.ascontiguousarray(depth)).cuda(), PinholeCameraIntrinsic(W, H, *K), E).cpu().numpy()
    assert np.array_equal(dc, oc), f"{what}: dry-run counts differ: {dc} vs {oc}"
    if stats is not None:
        for k, v in vol.dry_stats(True).items():
            stats[k] = stats.get(k, 0) + v
    return vol, V, oc


def assert_sweep_reached_every_class(stats):
    """the sweep produced free pairs, pairs in the image and (warp, frame) pairs that updated nothing"""
    assert stats["free_pairs"] > 0, stats
    assert stats["pairs_in_image"] > 0, stats
    assert stats["warp_frame_pairs"] > stats["pairs_updating"] > 0, stats


# ---------------------------------------------------------------- B / C / D scene: a small box, 2 mm voxels

VL, TRUNC = 0.002, 0.008
DIMS = (40, 40, 40)                      # 125 bricks, ragged-free; 80 mm edge
ORIGIN = np.array([-0.040, -0.040, 0.0])
CENTRE = ORIGIN + 0.5 * np.array(DIMS) * VL


def centre_on_voxel(i, j, k, dz=0.0):
    """world position of voxel (i, j, k)'s float32 centre (+ dz along z)"""
    return np.array([voxel_centres(1, ORIGIN[0], VL, i)[0], voxel_centres(1, ORIGIN[1], VL, j)[0],
                     float(voxel_centres(1, ORIGIN[2], VL, k)[0]) + dz], dtype=np.float64)


def brick_corner(i, j, k):
    return ORIGIN + np.array([i, j, k], dtype=np.float64) * 8 * VL


def placements():
    """camera centres: inside the box, on a voxel centre of a brick base layer (voxels at z == 0), 5e-5 off it
    (|z| < 1e-4), on a brick face, on a brick corner and on the voxel centre at a brick corner (voxels at z == 0
    under every 90-degree rotation), behind and beside the box"""
    return {
        "inside": CENTRE + np.array([0.0013, -0.0021, 0.0007]),
        "voxel_centre": centre_on_voxel(20, 20, 16),
        "voxel_centre_mid_brick": centre_on_voxel(13, 21, 19),
        "near_plus": centre_on_voxel(20, 20, 16, 5e-5),
        "near_minus": centre_on_voxel(20, 20, 16, -5e-5),
        "brick_face": np.array([CENTRE[0] + 0.0011, CENTRE[1] - 0.0017, brick_corner(0, 0, 2)[2]]),
        "brick_corner": brick_corner(2, 3, 2),
        "brick_corner_voxel": centre_on_voxel(16, 24, 16),
        "behind": np.array([CENTRE[0], CENTRE[1], ORIGIN[2] - 0.05]),
        "beside": np.array([ORIGIN[0] - 0.03, CENTRE[1], CENTRE[2]]),
    }


def scene_frames(K, W, H, R_list, c, rng, F_per=1, d_range=(0.01, 0.09), rgb=False):
    """frames of noisy, holed, tilted planes (NaN / inf / -0 / negative pixels included) for every rotation"""
    E, D = [], []
    for R in R_list:
        for _ in range(F_per):
            E.append(extrinsic(R, c))
            d0 = rng.uniform(*d_range)
            D.append(dirty(plane_depth(H, W, K, d0, rng.uniform(-0.02, 0.02, 2)), rng, noise=0.001, holes=0.05))
    D = np.stack(D)
    col = rng.integers(0, 256, size=D.shape + (3,), dtype=np.uint8) if rgb else None
    return D, np.stack(E), col


# ================================================================ A. production variants


def lap_scene(frames, frame_ids=None):
    """the bench's laparoscopy scene (512^3 @ 1 mm, 640 x 480): rendered u16 frames and colour"""
    from util import small_scene
    return small_scene("laparoscopy512", res=512, frames=frames, frame_ids=frame_ids)


SLAB_DIMS, SLAB_GZ0 = (512, 512, 144), 368      # 73 728 bricks: 8 z layers per warp, no long-chain phase


@pytest.fixture(scope="module")
def slab():
    """8 laparoscopy frames into the z-slab around the cavity's far wall, oracle with colour"""
    sc = lap_scene(8)
    d = oracle.o3d.depth_from_u16(sc["depth_u16"])
    V = oracle.o3d.Volume(SLAB_DIMS, sc["voxel_length"], sc["sdf_trunc"], sc["origin"], gz0=SLAB_GZ0, with_color=True)
    oc = oracle_integrate(V, d, sc["K"], sc["E"], sc["color"])
    assert oc.min() > 1000 and oc.sum() > 5_000_000, oc
    return sc, d, V, oc


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["plain", "color", "u16", "zpw4"])
def test_slab_production_variant_matches_oracle(cuda, slab, mode):
    """73 728 bricks select ZPW = 8 without the long-chain phase (the 512^3 bench's instantiations, the plain one
    with its load-first path); colour (640 x 480 RGB frames are whole 4-byte words, so this case reads every frame in
    place -- the padded copy of a ragged batch's last frame is exercised by test_image_sizes); `set_z_split(4)` gives
    the same bits"""
    sc, d, V, oc = slab
    color = mode == "color"
    vol = make_volume(SLAB_DIMS, sc["voxel_length"], sc["sdf_trunc"], sc["origin"], color=color, gz0=SLAB_GZ0, z_total=512,
                      zpw=4 if mode == "zpw4" else 0)
    gc = gpu_integrate(vol, d, sc["K"], sc["E"], sc["color"] if color else None, u16=sc["depth_u16"] if mode == "u16" else None)
    assert np.array_equal(gc, oc), (gc, oc)
    assert_same(vol, V, color, mode)
    if mode == "plain":
        # the dry-run instantiation of the same selection
        vol.dry_stats(True)
        dc = vol.count_updates(torch.from_numpy(d).cuda(), sc["intrinsic"], sc["E"]).cpu().numpy()
        assert np.array_equal(dc, oc)
        st = vol.dry_stats(True)
        assert st["free_pairs"] > 0 and st["warp_frame_pairs"] > st["pairs_updating"] > 0, st


@pytest.mark.gpu
def test_slab_unit_activation_matches_scalable_oracle(cuda):
    """unit activation at ZPW = 8 without the long-chain phase: 512 x 512 x 160 on the 32^3 unit grid (81 920 bricks)"""
    sc = lap_scene(6)
    d = oracle.o3d.depth_from_u16(sc["depth_u16"])
    origin = np.array(sc["origin"], dtype=np.float64)
    origin[2] += 352 * sc["voxel_length"]           # z = 96 mm: three 32 mm units
    dims = (512, 512, 160)
    vol, V, oc = check_case(d, sc["K"], sc["E"], dims, sc["voxel_length"], sc["sdf_trunc"], origin, rgb=sc["color"], unit=True,
                            what="unit slab")
    assert oc.min() > 10_000, oc


@pytest.mark.gpu
@pytest.mark.slow
def test_full_laparoscopy_volume_fresh_and_on_a_preintegrated_state(cuda):
    """the bench's configuration: 512^3, 640 x 480, 8 frames into a fresh volume, then 8 more on top"""
    sc = lap_scene(16)
    d = oracle.o3d.depth_from_u16(sc["depth_u16"])
    V = oracle.o3d.Volume(512, sc["voxel_length"], sc["sdf_trunc"], sc["origin"])
    vol = make_volume(512, sc["voxel_length"], sc["sdf_trunc"], sc["origin"])
    for lo, hi in ((0, 8), (8, 16)):
        oc = oracle_integrate(V, d[lo:hi], sc["K"], sc["E"][lo:hi])
        gc = gpu_integrate(vol, d[lo:hi], sc["K"], sc["E"][lo:hi])
        assert np.array_equal(gc, oc), (lo, gc, oc)
        assert_same(vol, V, what=f"frames {lo}..{hi}")
    assert float(V.weight.max()) >= 2


@pytest.mark.gpu
def test_long_chain_phase_claims_bricks_and_matches_batches_of_8(cuda):
    """a 40^3 box (125 bricks) that all 256 frames of one launch see: most bricks carry chains of 249..256 frames,
    which the whole-CTA phase takes; the same frames in launches of 8 and the oracle give the same bits"""
    rng = np.random.default_rng(7)
    W, H, K = 48, 40, (40.0, 41.0, 23.5, 19.5)
    E, D = [], []
    for i in range(256):
        c = CENTRE + np.array([rng.uniform(-0.01, 0.01), rng.uniform(-0.01, 0.01), -0.17])
        E.append(extrinsic(oblique_small(rng, 0.03), c))
        D.append(dirty(plane_depth(H, W, K, 0.215 + rng.uniform(-0.005, 0.01), rng.uniform(-0.02, 0.02, 2)), rng, 0.001, 0.03))
    D, E = np.stack(D), np.stack(E)
    vol, V, oc = check_case(D, K, E, DIMS, VL, TRUNC, ORIGIN, what="256-frame launch")
    hist = vol.chain_histogram()          # of the last launch: count_updates over the same 256 frames
    assert hist[31] > 0.5 * sum(hist), hist
    b8 = make_volume(DIMS, VL, TRUNC, ORIGIN, batch=8)
    assert np.array_equal(gpu_integrate(b8, D, K, E), oc)
    assert_same(b8, V, what="batches of 8")


def oblique_small(rng, angle):
    """a rotation by at most `angle` radians about a random axis"""
    a = rng.normal(size=3)
    a /= np.linalg.norm(a)
    th = rng.uniform(-angle, angle)
    Kx = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx


# ================================================================ B. cull boundaries


@pytest.mark.gpu
@pytest.mark.parametrize("place", list(placements()))
def test_camera_placements_and_rotations(cuda, place):
    """each placement seen under the identity, every 90-degree rotation about each axis and oblique rotations;
    colour included (the camera-plane voxels take the IEEE projection, every other class occurs as well)"""
    rng = np.random.default_rng(sum(map(ord, place)))
    W, H, K = 40, 32, (30.0, 34.0, 19.5, 15.5)
    D, E, rgb = scene_frames(K, W, H, rotations(rng), placements()[place], rng, rgb=True)
    stats = {}
    check_case(D, K, E, DIMS, VL, TRUNC, ORIGIN, rgb=rgb, what=place, stats=stats)
    if place not in ("behind", "beside"):
        assert_sweep_reached_every_class(stats)


@pytest.mark.gpu
def test_principal_point_steps_brick_edges_across_the_image_border(cuda):
    """identity pose, brick edges x = 16k mm at z = 100..180 mm: cx steps by 1/16 px so the projected edges (and the
    inner margin of 1.5 / 2.5 px) cross u = 0 and u = W; the same in y with cy"""
    rng = np.random.default_rng(11)
    W, H = 32, 24
    c = np.array([brick_corner(2, 2, 0)[0], brick_corner(2, 2, 0)[1], -0.1])
    stats = {}
    for k in range(32):
        frac = k / 16.0
        for K in ((50.0, 52.0, 0.0 + frac, 11.5), (50.0, 52.0, 15.5, 0.0 + frac), (50.0, 52.0, W - frac, H - frac)):
            d = np.stack([dirty(plane_depth(H, W, K, 0.1 + rng.uniform(0.01, 0.09)), rng, 0.001, 0.02) for _ in range(2)])
            check_case(d, K, np.stack([extrinsic(np.eye(3), c)] * 2), DIMS, VL, TRUNC, ORIGIN, what=f"cx/cy {K}", stats=stats)
    assert_sweep_reached_every_class(stats)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [(30.0, 45.0, 19.5, 15.5), (45.0, 30.0, 19.5, 15.5), (30.0, 30.0, -7.25, 15.5), (30.0, 30.0, 19.5, 40.75),
                               (30.0, 30.0, 55.0, -12.0), (30.0, 30.0, 0.0, 0.0), (30.0, 30.0, 40.0, 32.0)])
def test_intrinsics_off_centre_and_outside_the_image(cuda, K):
    """fx != fy, principal points off-centre, on the image corner and outside the image"""
    rng = np.random.default_rng(int(K[2] * 7 + K[3] * 3 + K[0]) & 0xffff)
    W, H = 40, 32
    D, E, _ = scene_frames(K, W, H, rotations(rng, 2), placements()["behind"] + np.array([0.0, 0.0, 0.02]), rng,
                           d_range=(0.05, 0.14))
    stats = {}
    check_case(D, K, E, DIMS, VL, TRUNC, ORIGIN, what=f"K {K}", stats=stats)
    assert stats["pairs_in_image"] > 0


def tile_content_frames(W, H, K, rng, kind):
    """depth whose tile extremes decide the cull: a camera at z = -30 mm looks at the box (z in [0, 80] mm);
    'spikes': near background (in front of the box: every brick dropped by the tile max) with single far
    pixels in odd tiles; 'near_pixel': far background (every brick free) with single near pixels in odd tiles;
    'single': one valid pixel per tile, everything else a hole"""
    F = 4
    D = np.empty((F, H, W), np.float32)
    for f in range(F):
        if kind == "spikes":
            d = np.full((H, W), 0.015, np.float32)
            val = lambda: rng.uniform(0.04, 0.12)
        elif kind == "near_pixel":
            d = np.full((H, W), 0.30, np.float32)
            val = lambda: rng.uniform(0.035, 0.11)
        else:
            d = np.zeros((H, W), np.float32)
            val = lambda: rng.uniform(0.035, 0.12)
        for ty in range((H + 15) // 16):
            for tx in range((W + 15) // 16):
                if kind == "spikes" and tx % 2 == 0 and ty % 2 == 0:
                    continue
                if kind == "near_pixel" and not (tx % 4 == 1 and ty % 2 == 1):     # sparse: far tiles stay free
                    continue
                y = min(H - 1, 16 * ty + rng.integers(0, 16))
                x = min(W - 1, 16 * tx + rng.integers(0, 16))
                d[y, x] = val()
        D[f] = d
    c = np.array([CENTRE[0] + 0.0007, CENTRE[1] - 0.0013, -0.03])
    E = np.stack([extrinsic(oblique_small(rng, 0.05), c) for _ in range(F)])
    return D, E


@pytest.mark.gpu
@pytest.mark.parametrize("trunc_vox", [4, 12])
def test_walls_swept_across_the_free_margin(cuda, trunc_vox):
    """a wall facing the camera, stepped in 0.7 mm increments over two brick layers: brick layers pass from the
    band into free space, some of them at exactly the free margin.  With sdf_trunc = 12 voxels a brick whose far side
    lies less than 2 * sdf_trunc in front of the wall still has voxels with t < 1"""
    rng = np.random.default_rng(trunc_vox)
    trunc = trunc_vox * VL
    W, H, K = 48, 40, (60.0, 61.0, 23.5, 19.5)
    c = np.array([CENTRE[0] + 0.0009, CENTRE[1] - 0.0011, -0.06])
    D, E = [], []
    for k in range(46):
        d0 = 0.06 + brick_corner(0, 0, 1)[2] + 2 * trunc + 0.0007 * k - 0.016
        D.append(dirty(plane_depth(H, W, K, d0), rng, 0.0, 0.02, specials=k % 5 == 0))
        E.append(extrinsic(np.eye(3) if k % 2 else oblique_small(rng, 0.02), c))
    stats = {}
    check_case(np.stack(D), K, np.stack(E), DIMS, VL, trunc, ORIGIN, what=f"walls, trunc {trunc_vox} vl", stats=stats)
    assert_sweep_reached_every_class(stats)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["spikes", "near_pixel", "single"])
def test_single_pixels_decide_the_tile_extremes(cuda, kind):
    """single pixels set a tile's max (spikes), its valid minimum (one near pixel among far ones: decides free) or
    are the tile's only valid pixel; odd tile columns / rows included, so the coarse pyramid levels must carry them"""
    rng = np.random.default_rng(len(kind))
    W, H, K = 160, 128, (100.0, 100.0, 79.5, 63.5)
    D, E = tile_content_frames(W, H, K, rng, kind)
    stats = {}
    vol, V, oc = check_case(D, K, E, DIMS, VL, TRUNC, ORIGIN, what=kind, stats=stats)
    assert oc.sum() > 0
    if kind == "near_pixel":
        assert stats["free_pairs"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(1, 1), (15, 17), (16, 16), (17, 16), (33, 9), (8192, 8)])
def test_image_sizes(cuda, W, H):
    """tiny images, tile-ragged sizes and the widest accepted image (512 tiles of 16 px); colour too, 3 frames from
    inside the box, so that the RGB batch of most sizes is not a whole number of 4-byte words (the launch's last frame
    is then read from a padded copy, see set_rgb_last)"""
    rng = np.random.default_rng(W * 100 + H)
    K = (0.9 * W, 1.0 * H, (W - 1) / 2, (H - 1) / 2)     # about 60 x 53 degrees whatever the size, fx != fy
    D, E, rgb = scene_frames(K, W, H, rotations(rng, 1)[:3], placements()["inside"], rng, d_range=(0.01, 0.05), rgb=True)
    stats = {}
    vol, V, oc = check_case(D, K, E, DIMS, VL, TRUNC, ORIGIN, rgb=rgb, what=f"{W}x{H}", stats=stats)
    assert oc.sum() > 0 and oc[-1] > 0, oc          # the last frame (the padded copy for most sizes) updates voxels
    assert stats["pairs_in_image"] > 0, stats


@pytest.mark.gpu
def test_image_size_limits_are_argument_errors(cuda):
    """8193 px wide exceeds the tile rows; 32 768 px tall would make the packed pixel (v << 16) | u negative"""
    vol = make_volume(DIMS, VL, TRUNC, ORIGIN)
    E = extrinsic(np.eye(3), placements()["behind"])[None]
    for W, H in ((8193, 8), (16, 32768)):
        d = torch.full((1, H, W), 0.1, dtype=torch.float32, device="cuda")
        with pytest.raises(RuntimeError, match="image too large"):
            vol.integrate_batch(d, None, PinholeCameraIntrinsic(W, H, 20.0, 20.0, W / 2, H / 2), E)
        with pytest.raises(RuntimeError, match="image too large"):
            vol.integrate_u16_batch(torch.full((1, H, W), 100, dtype=torch.uint16, device="cuda"), None,
                                    PinholeCameraIntrinsic(W, H, 20.0, 20.0, W / 2, H / 2), E)
    assert float(vol.export_dense()[1].max().item()) == 0.0
    # the tallest accepted image integrates like the oracle
    W, H, K = 16, 32767, (20.0, 20.0, 7.5, 32760.0)
    rng = np.random.default_rng(5)
    d = dirty(np.full((1, H, W), 0.1, np.float32), rng, 0.002, 0.01)
    check_case(d, K, E, DIMS, VL, TRUNC, ORIGIN, rgb=rng.integers(0, 256, (1, H, W, 3), dtype=np.uint8), what="H = 32767")


# ================================================================ C. arithmetic at its preconditions

C_DIMS = (32, 32, 32)
C_ORIGIN = np.array([-0.032, -0.032, 0.02])
C_K = (40.0, 40.0, 31.5, 31.5)
C_W = C_H = 64


def tiny_positive_floats():
    sub = np.array([1], np.uint32).view(np.float32)[0]                  # smallest subnormal
    return np.array([1e-29, 1e-31, 1e-35, 1e-38, 5e-39, sub, np.float32(7e-42)], np.float32)


def imported_states(seed=0):
    """tsdf / weight / colour per voxel, drawn from the boundary values: weights 0, 1, 2^24 - 2, 2^24 - 1, 2^24, 2^25
    (and small random ones), tsdf +-1, 1 - ulp, +-0, 1e-29, 1e-31, subnormal (and log-uniform tiny ones), colour 0 / 255"""
    rng = np.random.default_rng(seed)
    n = int(np.prod(C_DIMS))
    one_m = np.nextafter(np.float32(1), np.float32(0))
    t_vals = np.concatenate([np.array([1.0, -1.0, one_m, 0.0, -0.0, 0.5, -0.25], np.float32), tiny_positive_floats(),
                             -tiny_positive_floats()])
    w_vals = np.array([0.0, 1.0, TWO24 - 2, TWO24 - 1, TWO24, 2 * TWO24], np.float32)
    t = t_vals[rng.integers(0, len(t_vals), n)]
    w = w_vals[rng.integers(0, len(w_vals), n)]
    # a third of the voxels: log-uniform tiny tsdf with small random weights -- numerators below 1e-30 in t == 0 updates
    k = rng.random(n) < 0.33
    t[k] = (np.exp(rng.uniform(np.log(1e-44), np.log(1e-29), k.sum())) * rng.choice([-1, 1], k.sum())).astype(np.float32)
    w[k] = rng.integers(1, 5000, k.sum()).astype(np.float32)
    c = rng.choice(np.array([0.0, 255.0], np.float32), n * 3)
    m = rng.random(n * 3) < 0.3
    c[m] = rng.uniform(0.0, 255.0, int(m.sum())).astype(np.float32)
    return t.reshape(C_DIMS), w.reshape(C_DIMS), c.reshape(C_DIMS + (3,))


def exact_z_frames(n_frames=5):
    """identity pose: every voxel of a layer has the same float32 camera z, so a pixel whose depth IS that z gives
    the layer's voxels that project there t == 0 (the numerator of the blend is then the stored tsdf * w).  Frame f
    puts pixel (u, v) on layer (u + 2 v) % 4 + 5 f: that layer lay more than sdf_trunc behind the earlier frames'
    surfaces, so it still holds its imported tsdf when its t == 0 update comes"""
    z = camera_z(np.eye(4), C_DIMS, VL, C_ORIGIN)[0, 0]
    base = (np.arange(C_W)[None, :] + 2 * np.arange(C_H)[:, None]) % 4
    return np.stack([z[base + 5 * f].astype(np.float32) for f in range(n_frames)])


def arithmetic_frames(seed=0):
    """identity-pose frames over the imported states: far wall (free pairs, t == 1), walls through the box
    (the band), exact-depth frames (t == 0) first, while the tiny imported tsdf values are still there; the far wall
    twice, so the 2^24 - 2 weights cross 2^24"""
    rng = np.random.default_rng(seed)
    far = plane_depth(C_H, C_W, C_K, 0.25)
    mid = plane_depth(C_H, C_W, C_K, 0.05, (0.01, -0.01))
    near = dirty(plane_depth(C_H, C_W, C_K, 0.07), rng, 0.002, 0.05)
    D = np.concatenate([exact_z_frames(), far[None], mid[None], near[None], far[None]])
    E = np.stack([np.eye(4)] * len(D))
    rgb = rng.integers(0, 256, size=D.shape + (3,), dtype=np.uint8)
    return D, E, rgb


@pytest.mark.gpu
@pytest.mark.parametrize("color", [False, True])
def test_blend_at_weight_and_tsdf_extremes(cuda, color):
    """imported states at the blend's preconditions, then free / band / exact-depth (t == 0) frames"""
    D, E, rgb = arithmetic_frames()
    state = imported_states()
    stats = {}
    vol, V, oc = check_case(D, C_K, E, C_DIMS, VL, TRUNC, C_ORIGIN, rgb=rgb if color else None, state=state, what="states",
                            stats=stats)
    assert stats["free_pairs"] > 0
    assert float(V.weight.max()) >= TWO24


@pytest.mark.gpu
def test_blend_with_the_fused_u16_path(cuda):
    """the same imported states through the fused u16 conversion (frames in whole millimetres)"""
    rng = np.random.default_rng(3)
    u16 = np.stack([np.full((C_H, C_W), 250, np.uint16), rng.integers(40, 120, (C_H, C_W)).astype(np.uint16),
                    np.full((C_H, C_W), 60, np.uint16)])
    u16[1][rng.random((C_H, C_W)) < 0.1] = 0
    d = oracle.o3d.depth_from_u16(u16)
    check_case(d, C_K, np.stack([np.eye(4)] * 3), C_DIMS, VL, TRUNC, C_ORIGIN, state=imported_states(1), u16=u16, what="u16")


SUB = 2.0 ** -149      # smallest subnormal


def subnormal_midpoint_states(seed=0):
    """weight 5 and tsdf = +-3 (2m + 1) * 2^-149: a t == 0 update divides tsdf * 5 by 6 and the exact quotient lies
    halfway between two subnormals, so only a correctly rounded division (ties to even) gets it right"""
    rng = np.random.default_rng(seed)
    n = int(np.prod(C_DIMS))
    k = 3 * (2 * rng.integers(0, 4000, n) + 1)
    t = (k * SUB * rng.choice([-1.0, 1.0], n)).astype(np.float32)
    return t.reshape(C_DIMS), np.full(C_DIMS, 5.0, np.float32)


def colour_midpoint_states(byte, seed=0):
    """colour blends whose exact quotient lies within ~2^-48 (relative) of a rounding midpoint: weight w = b - 1 for an
    odd b in [2^23, 2^24) and a colour c with fl(fl(c * w) + byte) == a, where a / b is that close to a midpoint M of
    [128, 256) (b (2k + 1) = +-1 mod 2^25).  A reciprocal a few ulp off rounds some of them the wrong way.
    -> (tsdf, weight, colour [.., 3]), voxels without such a construction keep weight 0"""
    rng = np.random.default_rng(seed)
    n = int(np.prod(C_DIMS))
    w = np.zeros(n, np.float32)
    c = np.zeros(n, np.float32)
    for i in range(n):
        b = int(rng.integers(2 ** 22, 2 ** 23)) * 2 + 1
        inv = pow(b, -1, 2 ** 25)
        odd, s = (inv, 1) if inv >= 2 ** 24 else (2 ** 25 - inv, -1)
        if odd >= 250 * 2 ** 17:
            continue
        a = (b * odd - s) // 2 ** 25 * 256                     # a / b = odd / 2^17 (a midpoint) -+ 2^-17 / b
        ww = np.float32(b - 1)
        c0 = np.float32((a - byte) / float(b - 1))
        for cand in (c0, np.nextafter(c0, np.float32(0)), np.nextafter(c0, np.float32(1e9))):
            if float(np.float32(np.float32(cand * ww) + np.float32(byte))) == float(a):
                w[i], c[i] = ww, cand
                break
    col = np.repeat(c[:, None], 3, axis=1)
    return np.full(C_DIMS, 0.5, np.float32), w.reshape(C_DIMS), col.reshape(C_DIMS + (3,))


@pytest.mark.gpu
def test_subnormal_numerators_halfway_between_two_quotients(cuda):
    """t == 0 updates of subnormal tsdf * w: the out-of-line IEEE division rounds the exact midpoints to even"""
    D = exact_z_frames()
    check_case(D, C_K, np.stack([np.eye(4)] * len(D)), C_DIMS, VL, TRUNC, C_ORIGIN, state=subnormal_midpoint_states(),
               what="subnormal midpoints")


@pytest.mark.gpu
def test_colour_quotients_next_to_a_rounding_midpoint(cuda):
    """colour blends at weights near 2^23 whose quotients sit next to a midpoint: correct rounding needs the Newton
    step of the shared reciprocal"""
    byte = 17
    far = plane_depth(C_H, C_W, C_K, 0.25)
    D = np.stack([far, far])
    rgb = np.full(D.shape + (3,), byte, np.uint8)
    check_case(D, C_K, np.stack([np.eye(4)] * 2), C_DIMS, VL, TRUNC, C_ORIGIN, rgb=rgb, state=colour_midpoint_states(byte),
               what="colour midpoints")


# ================================================================ D. launch structure


def launch_frames(F, W, H, K, seed):
    rng = np.random.default_rng(seed)
    E, D = [], []
    for i in range(F):
        c = CENTRE + np.array([rng.uniform(-0.02, 0.02), rng.uniform(-0.02, 0.02), -0.12 - rng.uniform(0, 0.03)])
        E.append(extrinsic(oblique_small(rng, 0.2), c))
        D.append(dirty(plane_depth(H, W, K, 0.12 + rng.uniform(-0.02, 0.06), rng.uniform(-0.03, 0.03, 2)), rng, 0.001, 0.03,
                       specials=i % 3 == 0))
    return np.stack(D), np.stack(E)


@pytest.mark.gpu
@pytest.mark.parametrize("F", [8, 9, 32, 33, 64, 65, 256, 257])
def test_batch_sizes_match_oracle_and_single_frame_calls(cuda, F):
    """the small cull (F <= 8) against the warp cull, every 32-frame mask-word boundary, chunking above 256"""
    W, H, K = 40, 30, (36.0, 35.0, 20.25, 14.75)
    D, E = launch_frames(F, W, H, K, F)
    rgb = np.random.default_rng(F).integers(0, 256, size=D.shape + (3,), dtype=np.uint8)
    vol, V, oc = check_case(D, K, E, DIMS, VL, TRUNC, ORIGIN, rgb=rgb, what=f"F = {F}")
    one = make_volume(DIMS, VL, TRUNC, ORIGIN, color=True)
    for i in range(F):
        assert gpu_integrate(one, D[i:i + 1], K, E[i:i + 1], rgb[i:i + 1])[0] == oc[i]
    assert_same(one, V, True, "one frame per call")


@pytest.mark.gpu
def test_large_frames_halve_the_launch_batch(cuda):
    """130 frames of 2048 x 1536: the tile pyramid of 256 such frames outgrows its reservation, so launches carry
    128 frames (128 + 2 here); equal to the oracle and to one frame per call"""
    W, H, K = 2048, 1536, (1400.0, 1420.0, 1023.5, 767.5)
    F = 130
    rng = np.random.default_rng(130)
    E = np.stack([extrinsic(oblique_small(rng, 0.1), CENTRE + np.array([rng.uniform(-0.01, 0.01), rng.uniform(-0.01, 0.01), -0.12]))
                  for _ in range(F)])
    D = np.empty((F, H, W), np.float32)
    base = plane_depth(H, W, K, 0.12)
    for i in range(F):
        D[i] = base + np.float32(rng.uniform(-0.02, 0.06))
        D[i, rng.integers(0, H, 2000), rng.integers(0, W, 2000)] = 0.0
    vol, V, oc = check_case(D, K, E, DIMS, VL, TRUNC, ORIGIN, what="2048 x 1536")
    # the same call in launches of 128 + 2 frames: two timed integrate launches
    timed = make_volume(DIMS, VL, TRUNC, ORIGIN)
    timed.profile(True)
    gpu_integrate(timed, D, K, E)
    assert timed.profile_read()[1] == 2
    assert_same(timed, V, what="profiled")
    one = make_volume(DIMS, VL, TRUNC, ORIGIN)
    for i in range(F):
        gpu_integrate(one, D[i:i + 1], K, E[i:i + 1])
    assert_same(one, V, what="one frame per call")


# ================================================================ CPU checks of the generators (oracle only)


def test_exact_z_frames_give_t_zero_updates_in_the_oracle():
    """on a fresh volume one frame's tsdf IS its t: the exact-depth frames must produce t == 0 on many voxels"""
    D = exact_z_frames()
    V = oracle.o3d.Volume(C_DIMS, VL, TRUNC, C_ORIGIN)
    n = V.integrate(D[0], C_K, np.eye(4))
    t, w = V.grid("tsdf"), V.grid("weight")
    zero = (w == 1) & (t == 0)
    assert n > 0 and zero.sum() > 200, zero.sum()
    # and the numpy recurrence is the oracle's: the t == 0 voxels sit exactly at their pixel's depth
    z = camera_z(np.eye(4), C_DIMS, VL, C_ORIGIN)
    assert np.all(np.isin(z[zero], D[0]))


def test_imported_states_reach_weights_of_2_24_and_tiny_numerators():
    D, E, rgb = arithmetic_frames()
    t, w, c = imported_states()
    assert {0.0, 1.0, TWO24 - 2, TWO24 - 1, TWO24, 2 * TWO24} <= set(np.unique(w).tolist())
    assert (np.signbit(t) & (t == 0)).any() and ((t != 0) & (np.abs(t) < np.finfo(np.float32).tiny)).any()
    V = oracle.o3d.Volume(C_DIMS, VL, TRUNC, C_ORIGIN, with_color=True)
    seed_oracle(V, (t, w, c))
    w0 = V.grid("weight").copy()
    n_exact = len(exact_z_frames())
    for i in range(n_exact):
        V.integrate(D[i], C_K, E[i], rgb=rgb[i])
    # t == 0 updates of voxels with a tiny stored tsdf (numerator tsdf * w below 1e-30): the result stays tiny
    t1 = V.grid("tsdf")
    tiny = (w0 > 0) & (np.abs(t) * np.maximum(w0, 1) < 1e-30) & (t != 0) & (V.grid("weight") > w0) & (np.abs(t1) < 1e-30)
    assert tiny.sum() > 300, tiny.sum()
    for i in range(n_exact, len(D)):
        V.integrate(D[i], C_K, E[i], rgb=rgb[i])
    w1 = V.grid("weight")
    assert ((w0 == TWO24 - 2) & (w1 == TWO24)).any(), "no weight crossed 2^24 - 1 -> 2^24"
    assert ((w0 == TWO24) & (w1 == TWO24)).any()
    assert ((w0 == 2 * TWO24) & (w1 == 2 * TWO24)).any()


def test_placements_put_voxels_on_and_next_to_the_camera_plane():
    """the boundary placements give voxels at float32 z == 0 and at 0 < |z| < 1e-4, also under the exact rotations"""
    P = placements()
    for R in [np.eye(3)] + [rot(a, q) for a in range(3) for q in (1, 2, 3)]:
        z = camera_z(extrinsic(R, P["brick_corner_voxel"]), DIMS, VL, ORIGIN)
        assert (z == 0).sum() >= 40 * 40, R
    z = camera_z(extrinsic(np.eye(3), P["voxel_centre"]), DIMS, VL, ORIGIN)
    assert (z == 0).sum() == 40 * 40
    for name in ("near_plus", "near_minus"):
        for R in [np.eye(3), rot(0, 2), rot(1, 2), rot(2, 1), rot(2, 3)]:
            z = camera_z(extrinsic(R, P[name]), DIMS, VL, ORIGIN)
            n0, nt = int((z == 0).sum()), int(((z != 0) & (np.abs(z) < 1e-4)).sum())
            assert nt == 40 * 40 and n0 == 0, (name, R, n0, nt)
    # the camera on a brick face: the voxel layers around it lie half a voxel in front and behind
    z = camera_z(extrinsic(np.eye(3), P["brick_face"]), DIMS, VL, ORIGIN)
    assert (np.abs(z) <= 0.5 * VL + 1e-7).any() and (z < 0).any() and (z > 0).any()


def test_rotations_are_exact_and_orthonormal():
    rng = np.random.default_rng(0)
    for R in rotations(rng):
        assert np.allclose(R @ R.T, np.eye(3), atol=1e-12) and np.isclose(np.linalg.det(R), 1.0)
    for a in range(3):
        for q in range(4):
            assert set(np.unique(rot(a, q)).tolist()) <= {-1.0, 0.0, 1.0}


def test_midpoint_states_sit_where_they_should():
    """the subnormal states divide to exact midpoints in the oracle's t == 0 updates; the colour states' quotients lie
    within 2^-22 ulp of a midpoint and the oracle rounds them correctly"""
    from fractions import Fraction
    t, w = subnormal_midpoint_states()
    D = exact_z_frames()
    V = oracle.o3d.Volume(C_DIMS, VL, TRUNC, C_ORIGIN)
    seed_oracle(V, (t, w))
    V.integrate(D[0], C_K, np.eye(4))
    t1, w1 = V.grid("tsdf"), V.grid("weight")
    hit = (w1 == 6) & (t1 == (t * np.float32(5)) / np.float32(6))
    assert hit.sum() > 200, hit.sum()
    q = Fraction(float(t[hit][0])) * 5 / 6
    assert (q / Fraction(SUB)).denominator == 2            # exactly halfway between two subnormals
    byte = 17
    t, w, c = colour_midpoint_states(byte)
    ok = w > 0
    assert ok.mean() > 0.5, ok.mean()
    V = oracle.o3d.Volume(C_DIMS, VL, TRUNC, C_ORIGIN, with_color=True)
    seed_oracle(V, (t, w, c))
    far = plane_depth(C_H, C_W, C_K, 0.25)
    V.integrate(far, C_K, np.eye(4), rgb=np.full((C_H, C_W, 3), byte, np.uint8))
    updated = ok & (V.grid("weight") == w + 1)
    assert updated.sum() > 500, updated.sum()
    out = V.color.reshape(C_DIMS + (3,))[..., 0]
    for i in np.flatnonzero(updated.reshape(-1))[:200]:
        ww, cc = w.reshape(-1)[i], c[..., 0].reshape(-1)[i]
        a = Fraction(float(np.float32(np.float32(cc * ww) + np.float32(byte))))
        exact = a / (Fraction(float(ww)) + 1)
        ulp = Fraction(2) ** -16
        frac = (exact / ulp) - int(exact / ulp)
        assert abs(frac - Fraction(1, 2)) < Fraction(2) ** -22, float(frac)    # within 2^-22 ulp of a midpoint
        assert Fraction(float(out.reshape(-1)[i])) == round(exact / ulp) * ulp      # the oracle rounds it correctly
