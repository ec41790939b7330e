"""Edges of the ray cast (csrc/bslam_raycast.cu) and of the `MAP` integrator (csrc/bslam_vbg.cu) -- `-m gpu`.

Bit-for-bit comparisons with the CPU references (tests/raycast_ref.c, the oracle's orc_vbg_integrate) at what the parity
tests of test_gpu_raycast.py / test_gpu_map.py leave out: image sizes that are not multiples of the 32 x 8 ray tile, the
8-pixel range cell or the 4-pixel touch stride; batches across the 64-frame chunks of both entry points; non-cubic boxes
and negative block indices; every output combination, depth window, weight threshold and awkward pose.  The legacy volumes
are analytic (a sphere and a plane, imported with `import_dense`), so their geometry is known exactly.  Closed-form checks
in float64 on the GPU's own output catch mistakes the kernel and the reference could share, and guard bands around
C ABI output buffers catch pixels that are never written and writes into the wrong frame.  The full-size 512^3
comparison is `-m "gpu and slow"`."""
import copy

import numpy as np
import pytest
import torch

import oracle
import raycast_ref
from bodyslam_b200 import _lib, ops
from bodyslam_b200 import synthetic as S
from bodyslam_b200.geometry import PinholeCameraIntrinsic
from bodyslam_b200.tsdf import MAP, DenseTSDFVolume
from test_gpu_map import FakeRGBD, k3x3
from test_gpu_raycast import KEYS, assert_same
from util import small_scene

pytestmark = pytest.mark.gpu

BOXES = [(8, 8, 8), (16, 48, 24), (64, 40, 96)]
SIZES = [(1, 1), (7, 5), (31, 9), (33, 17), (8, 700), (641, 479)]
SPHERE_RGB = np.array([200.0, 100.0, 50.0], np.float32)


# ------------------------------------------------------------------ analytic legacy volumes
class Analytic:
    """A sphere in front of a plane (z = zp, the camera side is z < zp) in a box of `res` voxels; tsdf = clamp(signed
    distance / sdf_trunc, -1, 1) at voxel centres; weights 1..3.  holes: ~1/5 of the bricks at weight 0 (never the
    sphere's) and ~1/20 of the voxels with tsdf < 0 at weight 0 inside the others."""

    def __init__(self, res, holes=False, seed=0):
        self.res = tuple(res)
        n = np.array(res)
        self.vl = 0.2 / max(res)
        self.trunc = 4 * self.vl
        ext = n * self.vl
        self.origin = np.array([-0.0913, 0.0371, 0.1523]) - 0.5 * ext + np.array([0.0, 0.0, 0.05])
        self.centre = self.origin + ext * np.array([0.47, 0.52, 0.42])
        self.R = 0.22 * ext.min()
        self.zp = self.origin[2] + 0.8 * ext[2]
        p = self.origin + (np.indices(res).transpose(1, 2, 3, 0) + 0.5) * self.vl          # voxel centres [nx,ny,nz,3]
        ds = np.linalg.norm(p - self.centre, axis=-1) - self.R
        dp = self.zp - p[..., 2]
        self.tsdf = np.clip(np.minimum(ds, dp) / self.trunc, -1.0, 1.0).astype(np.float32)
        rng = np.random.default_rng(seed)
        self.weight = rng.integers(1, 4, size=res).astype(np.float32)
        col = np.empty(tuple(res) + (3,), np.float32)
        col[...] = SPHERE_RGB
        rel = (p - self.origin) / ext
        plane = dp < ds
        col[plane] = np.stack([255.0 * rel[..., 0], np.full(res, 128.0), 255.0 * rel[..., 1]], -1)[plane].astype(np.float32)
        self.color = col
        if holes:
            nb = n // 8
            brick = rng.random(tuple(nb)) < 0.2
            near_sphere = (np.abs(ds) < 2 * self.trunc).reshape(nb[0], 8, nb[1], 8, nb[2], 8).any(axis=(1, 3, 5))
            brick &= ~near_sphere
            self.weight[np.repeat(np.repeat(np.repeat(brick, 8, 0), 8, 1), 8, 2)] = 0.0
            self.weight[(self.tsdf < 0) & (rng.random(res) < 0.05)] = 0.0

    def volume(self, dev, color=True):
        vol = DenseTSDFVolume(self.vl, self.trunc, self.res, self.origin, color=color, device=dev)
        vol.import_dense(self.tsdf, self.weight, self.color if color else None)
        return vol

    def oracle(self, color=True):
        V = oracle.o3d.Volume(self.res, self.vl, self.trunc, self.origin, with_color=color)
        V.tsdf[:], V.weight[:] = self.tsdf.reshape(-1), self.weight.reshape(-1)
        if color:
            V.color[:] = self.color.reshape(-1)
        return V

    def front(self):
        """in front of the box (z below it), looking at the sphere"""
        return look_at(self.centre - np.array([0.1, -0.05, 1.0]) * (self.centre[2] - self.origin[2] + 3 * self.R), self.centre)

    def poses(self):
        """camera -> world: front, inside the box, inside the sphere (the march starts at tsdf < 0), looking away,
        identity rotation, grazing along the plane"""
        c, R, o = self.centre, self.R, self.origin
        ext = np.array(self.res) * self.vl
        inside_box = np.array([c[0] + 0.3 * R, c[1] - 0.2 * R, 0.5 * (o[2] + c[2] - R)])
        ident = np.eye(4)
        ident[:3, 3] = c - np.array([0.0, 0.0, 2.5 * R])
        grazing = np.array([o[0] + 0.05 * ext[0], c[1] + 0.1 * R, self.zp - 0.5 * self.vl])
        return np.stack([self.front(), look_at(inside_box, c + np.array([0.1, 0.0, 0.0]) * R),
                         look_at(c + 0.1 * R, c + np.array([0.3, 0.2, 1.0])),
                         look_at(self.front()[:3, 3], self.front()[:3, 3] - np.array([0.0, 0.1, 1.0])), ident,
                         look_at(grazing, grazing + np.array([1.0, 0.05, 0.01]))])


def look_at(eye, target, down=(0.0, 1.0, 0.0)):
    """camera -> world 4x4: z from eye towards target, y as close to `down` as it can be"""
    eye, target = np.asarray(eye, np.float64), np.asarray(target, np.float64)
    z = (target - eye) / np.linalg.norm(target - eye)
    x = np.cross(np.asarray(down, np.float64), z)
    if np.linalg.norm(x) < 1e-6:
        x = np.cross((1.0, 0.0, 0.0), z)
    x /= np.linalg.norm(x)
    P = np.eye(4)
    P[:3, 0], P[:3, 1], P[:3, 2], P[:3, 3] = x, np.cross(z, x), z, eye
    return P


def ext_of(P):
    """rigid inverse in float64: camera -> world <-> world -> camera"""
    P = np.asarray(P, np.float64)
    if P.ndim == 3:
        return np.stack([ext_of(p) for p in P])
    E = np.eye(4)
    E[:3, :3] = P[:3, :3].T
    E[:3, 3] = -P[:3, :3].T @ P[:3, 3]
    return E


def intr(W, H, integer_centre=False):
    f = 0.9 * max(W, H) + 1.0
    if integer_centre:
        return (W, H, f, f, float(W // 2), float(H // 2))
    return (W, H, f, 1.03 * f, (W - 1) / 2 + 0.37, (H - 1) / 2 - 0.21)


def cast_both(vol, V, K6, E, **kw):
    gpu = vol.raycast(K6, E, **kw)
    ref = raycast_ref.raycast(V, K6[2:], E, K6[0], K6[1], **kw)
    return gpu, ref, assert_same(gpu, ref)


@pytest.fixture(scope="module", params=BOXES, ids=lambda r: "x".join(map(str, r)))
def box(request, cuda):
    sc = Analytic(request.param, holes=True, seed=sum(request.param))
    return sc, sc.volume(cuda), sc.oracle()


@pytest.fixture(scope="module")
def clean(cuda):
    sc = Analytic((64, 40, 96))
    return sc, sc.volume(cuda), sc.oracle()


# ------------------------------------------------------------------ 1. legacy flavour on analytic volumes
@pytest.mark.parametrize("W,H", SIZES)
def test_legacy_image_sizes_and_poses(box, W, H):
    sc, vol, V = box
    E = ext_of(sc.poses())
    hits = 0
    for integer_centre in (False, True):
        _, _, hit = cast_both(vol, V, intr(W, H, integer_centre), E)
        hits += hit[0].sum()
    if W * H > 1:
        assert hits > 0, "the front view hits nothing"


def test_legacy_camera_1km_away(box):
    sc, vol, V = box
    P = look_at(sc.centre - 1000.0 * np.array([0.0, 0.6, 0.8]), sc.centre)
    K6 = (33, 17, 1.5e5, 1.5e5, 16.3, 8.2)
    _, ref, hit = cast_both(vol, V, K6, ext_of(P), depth_min=999.0, depth_max=1001.0, depth_scale=1000.0)
    assert hit.any()


@pytest.mark.parametrize("F", [0, 1, 63, 64, 65, 130])
def test_legacy_batches_across_chunks(cuda, F):
    """the 64-pose chunks of bslam_tsdf_raycast: every frame equals the reference and its own single-pose call"""
    sc = Analytic((16, 48, 24), holes=True, seed=3)
    vol, V = sc.volume(cuda), sc.oracle()
    K6 = intr(33, 17)
    a = np.linspace(0, 2 * np.pi, max(F, 1), endpoint=False)
    dist = 3.0 * sc.R + 0.5 * sc.vl * np.array(sc.res).max()
    P = [look_at(sc.centre + dist * np.array([np.sin(t), 0.3 * np.cos(3 * t), -np.cos(t)]), sc.centre) for t in a[:F]]
    E = ext_of(np.stack(P)) if F else np.zeros((0, 4, 4))
    gpu = vol.raycast(K6, E)
    assert all(gpu[k].shape[:3] == (F, 17, 33) for k in KEYS)
    if F == 0:
        return
    ref = raycast_ref.raycast(V, K6[2:], E, 33, 17)
    hit = assert_same(gpu, ref)
    assert hit.any(axis=(1, 2)).all(), "some view sees nothing"
    for i in range(F):
        one = vol.raycast(K6, E[i])
        for k in KEYS:
            assert torch.equal(one[k][0], gpu[k][i]), (i, k)


def test_legacy_output_combinations(cuda):
    sc = Analytic((64, 40, 96), holes=True, seed=5)
    K6 = intr(31, 9)
    E = ext_of(sc.poses())
    for color in (True, False):
        vol, V = sc.volume(cuda, color), sc.oracle(color)
        full = None
        for normals in (True, False):
            for colors in ((True, False) if color else (False,)):
                gpu, _, _ = cast_both(vol, V, K6, E, normals=normals, colors=colors)
                assert set(gpu) == {"depth", "vertex"} | ({"normal"} if normals else set()) | ({"color"} if colors else set())
                full = full or gpu
                for k in gpu:
                    assert torch.equal(gpu[k], full[k]), k


def test_legacy_depth_windows(cuda):
    sc = Analytic((16, 48, 24), seed=7)
    vol, V = sc.volume(cuda), sc.oracle()
    K6 = intr(33, 17)
    P = sc.front()
    E = ext_of(P)
    z_c = float((E[:3, :3] @ sc.centre + E[:3, 3])[2])          # camera z of the sphere's centre
    g, _, hit = cast_both(vol, V, K6, E, depth_min=z_c - 0.5 * sc.R, depth_max=3.0)     # starts inside the sphere
    assert hit.any()
    for lo, hi in ((z_c, z_c), (z_c, z_c - sc.R), (0.5, 0.1)):
        g, _, hit = cast_both(vol, V, K6, E, depth_min=lo, depth_max=hi)
        assert not hit.any() and all(not g[k].any() for k in g)
    g, _, hit = cast_both(vol, V, K6, E, depth_min=z_c - 0.9 * sc.R, depth_max=z_c - 0.2 * sc.R)      # cuts the sphere
    assert hit.any()


@pytest.mark.parametrize("thr", [0.0, 1.0, 2.0, 2.5, 3.0, 100.0])
def test_legacy_weight_thresholds(box, thr):
    sc, vol, V = box
    _, _, hit = cast_both(vol, V, intr(33, 17), ext_of(sc.poses()), weight_threshold=thr)
    if thr == 100.0:
        assert not hit.any()


def test_threshold_equal_to_the_stored_weight_is_valid(cuda):
    sc = Analytic((16, 48, 24))
    sc.weight[:] = 2.0
    vol, V = sc.volume(cuda), sc.oracle()
    E = ext_of(sc.front())
    assert cast_both(vol, V, intr(33, 17), E, weight_threshold=2.0)[2].any()
    assert not cast_both(vol, V, intr(33, 17), E, weight_threshold=np.nextafter(np.float32(2.0), np.float32(3.0)))[2].any()


# ------------------------------------------------------------------ 2. guard bands through the C ABI
TILE = 32 * 8


def guarded(n, dev):
    return torch.full((n,), float("nan"), dtype=torch.float32, device=dev)


def check_guard(bufs, n_pix):
    for name, (buf, ch) in bufs.items():
        b = buf.cpu().numpy()
        assert not np.isnan(b[:ch * n_pix]).any(), f"{name}: {np.isnan(b[:ch * n_pix]).sum()} elements never written"
        assert np.isnan(b[ch * n_pix:]).all(), f"{name}: written past the end"


@pytest.mark.parametrize("F,W,H", [(1, 7, 5), (65, 31, 9), (130, 33, 17), (2, 641, 479)])
def test_tsdf_raycast_guard_bands(cuda, F, W, H):
    sc = Analytic((16, 48, 24), holes=True, seed=1)
    vol = sc.volume(cuda)
    P = [look_at(sc.centre + (3 * sc.R + 0.05) * np.array([np.sin(t), 0.2, -np.cos(t)]), sc.centre) for t in np.linspace(0, 6, F)]
    E = np.ascontiguousarray(ext_of(np.stack(P)).reshape(-1))
    K = np.array(intr(W, H)[2:], np.float64)
    n = F * H * W
    pad = H * W + TILE
    bufs = {k: (guarded(ch * (n + pad), cuda), ch) for k, ch in (("depth", 1), ("vertex", 3), ("normal", 3), ("color", 3))}
    L = _lib.load()
    rc = L.bslam_tsdf_raycast(vol._h, F, H, W, _lib.ptr(K), _lib.ptr(E), 1.0, 0.0, 3.0, 0.0, *(_lib.ptr(bufs[k][0]) for k in KEYS),
                              _lib.stream_ptr(cuda))
    assert rc == _lib.OK, L.bslam_last_error()
    check_guard(bufs, n)
    api = vol.raycast(intr(W, H), E.reshape(F, 4, 4))
    for k in KEYS:
        assert torch.equal(bufs[k][0][:bufs[k][1] * n], api[k].reshape(-1)), k


@pytest.mark.parametrize("W,H", [(9, 17), (37, 23), (100, 75)])
def test_vbg_raycast_guard_bands(cuda, W, H):
    sc = small_scene("laparoscopy512", res=64, frame_ids=np.arange(0, 8, 2), W=W, H=H)
    m = map_for(sc, 64, 4.0)
    poses = ext_of(sc["E"])
    m.integrate_batch(sc["depth_u16"], sc["color"], poses, 3.0)
    L = _lib.load()
    n = H * W
    pad = n + TILE
    bufs = {k: (guarded(ch * (n + pad), cuda), ch) for k, ch in (("depth", 1), ("vertex", 3), ("normal", 3), ("color", 3))}
    ws = torch.empty(max(L.bslam_vbg_raycast_workspace_bytes(H, W), 1), dtype=torch.uint8, device=cuda)
    K = np.asarray(m._K, np.float64)
    P = np.ascontiguousarray(poses[-1].reshape(-1))
    rc = L.bslam_vbg_raycast(m.model._h, _lib.ptr(m._ws), H, W, _lib.ptr(K), _lib.ptr(P), 1000.0, 0.1, 3.0, 3.0, 4.0,
                             *(_lib.ptr(bufs[k][0]) for k in KEYS), _lib.ptr(ws), _lib.stream_ptr(cuda))
    assert rc == _lib.OK, L.bslam_last_error()
    check_guard(bufs, n)
    api = m.synthesize_model_frame()
    for k in KEYS:
        assert torch.equal(bufs[k][0][:bufs[k][1] * n], api[k].reshape(-1)), k


# ------------------------------------------------------------------ 3. closed forms in float64 on the GPU's output
def rays(P, K6):
    """float64 camera centre and per-pixel world directions (camera z component 1) [H,W,3]"""
    W, H, fx, fy, cx, cy = K6
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    dc = np.stack([(x - cx) / fx, (y - cy) / fy, np.ones_like(x)], -1)
    return P[:3, 3], dc @ P[:3, :3].T


def sphere_t(o, d, c, R):
    """ray parameter of the first intersection with the sphere (nan: none)"""
    oc = o - c
    a = (d * d).sum(-1)
    b = (d * oc).sum(-1)
    disc = b * b - a * ((oc * oc).sum() - R * R)
    with np.errstate(invalid="ignore"):
        return np.where(disc >= 0, (-b - np.sqrt(disc)) / a, np.nan)


@pytest.mark.parametrize("pose", ["front", "inside_box", "identity", "oblique"])
def test_legacy_closed_forms(clean, pose):
    sc, vol, _ = clean
    names = ["front", "inside_box", "inside_sphere", "away", "identity", "grazing"]
    P = sc.poses()[names.index(pose)] if pose in names else look_at(sc.centre + np.array([0.4, -0.3, -0.6]) * 4 * sc.R, sc.centre)
    K6 = intr(64, 48, integer_centre=pose == "identity")
    W, H, fx, fy, cx, cy = K6
    scale = 1000.0
    g = {k: v[0].cpu().numpy().astype(np.float64) for k, v in vol.raycast(K6, ext_of(P), depth_scale=scale).items()}
    hit = g["depth"] > 0
    miss = ~hit
    for k in KEYS:
        assert not g[k][miss].any(), f"{k} of a miss is not 0"
    assert hit.sum() > 100
    v, depth = g["vertex"], g["depth"] / scale
    y, x = np.mgrid[0:H, 0:W]
    assert np.abs(fx * v[..., 0] / v[..., 2] + cx - x)[hit].max() <= 1e-3
    assert np.abs(fy * v[..., 1] / v[..., 2] + cy - y)[hit].max() <= 1e-3
    ulp = np.finfo(np.float32).eps * (np.linalg.norm(P[:3, 3]) + depth)
    assert (np.abs(v[..., 2] - depth) <= 8 * ulp)[hit].all()
    nlen = np.linalg.norm(g["normal"], axis=-1)
    assert ((np.abs(nlen - 1.0) <= 1e-5) | (nlen == 0))[hit].all()      # 0: every gradient component dropped
    # the sphere
    o, d = rays(P, K6)
    t = sphere_t(o, d, sc.centre, sc.R)
    core = ~np.isnan(sphere_t(o, d, sc.centre, 0.9 * sc.R))
    # away from the rim: the march samples the voxel holding the point, so on a slope its depth is off by up to about
    # half a voxel over the cosine of the incidence (0.7 R: cos >= 0.71)
    inner = ~np.isnan(sphere_t(o, d, sc.centre, 0.7 * sc.R))
    assert core.sum() > 50 and hit[core].all(), f"{(~hit[core]).sum()} rays through the sphere's core miss"
    assert np.abs(depth - t)[inner].max() <= sc.vl
    assert (np.abs(nlen - 1.0) <= 1e-5)[core].all()
    assert ((g["normal"] * v).sum(-1)[core] < 0).all(), "sphere normals face away from the camera"
    c = g["color"]
    on_sphere = inner & (sc.zp - (o + t[..., None] * d)[..., 2] > 6 * sc.vl)
    assert np.abs(c[on_sphere] - SPHERE_RGB / 255.0).max() <= 1e-6


# ------------------------------------------------------------------ 4. tensor flavour (MAP)
def map_origin(res, vs, centre=(0.0, 0.0, 0.0)):
    bs = vs * 16
    return np.floor((np.asarray(centre) - 0.5 * np.asarray(res) * vs) / bs + 0.5) * bs


def map_for(sc, res, mult, vs=0.0058, color=True):
    res3 = (res,) * 3 if np.isscalar(res) else tuple(res)
    return MAP(sc["W"], sc["H"], k3x3(sc["K"]), "CUDA:0", 1000.0, voxel_size=vs, trunc_voxel_multiplier=mult, resolution=res3,
               origin=map_origin(res3, vs), color=color)


def oracle_for(m, color=True):
    return oracle.o3d.Volume((m.model.nx, m.model.ny, m.model.nz), m.voxel_size, m.voxel_size * m.trunc_voxel_multiplier, m.model.origin,
                             with_color=color)


def same_grids(m, V):
    out = m.model.export_dense(with_color=V.color is not None)
    assert np.array_equal(out[1].cpu().numpy(), V.grid("weight")), "weights differ"
    assert np.array_equal(out[0].cpu().numpy(), V.grid("tsdf")), "tsdf differs"
    if V.color is not None:
        assert np.array_equal(out[2].cpu().numpy().reshape(-1), V.color), "colour differs"


def same_cast(m, V, pose, allocated, touched, thr, **kw):
    assert np.array_equal(m.allocated_blocks().cpu().numpy(), allocated)
    assert np.array_equal(m.allocated_blocks(last_frame=True).cpu().numpy(), touched)
    gpu = m.synthesize_model_frame(**kw)
    ref = raycast_ref.raycast_vbg(V, m._K, pose, m.width, m.height, allocated, touched, depth_scale=m.depth_scale, weight_threshold=thr,
                                  trunc_voxel_multiplier=m.trunc_voxel_multiplier, colors=kw.get("enable_color", True) and V.color is not None,
                                  depth_min=kw.get("depth_min", 0.1), depth_max=kw.get("depth_max", 3.0))
    return assert_same(gpu, ref)


def run_frame_by_frame(m, V, sc, ids, mult, color=True):
    """MAP.integrate and the oracle frame by frame; grids, blocks and the synthesized frame after every frame"""
    poses = ext_of(sc["E"])
    allocated = np.zeros([n // 16 for n in (V.nx, V.ny, V.nz)], bool)
    hits = []
    for j, i in enumerate(ids):
        fr = FakeRGBD(sc["depth_u16"][j], sc["color"][j] if color else None, 1000.0)
        m.integrate(fr, i, poses[j])
        _, touched = V.integrate_vbg(sc["depth_u16"][j], sc["K"], poses[j], rgb=sc["color"][j] if color else None, depth_scale=1000.0,
                                     depth_max=fr.depth_max, trunc_voxel_multiplier=mult, return_touched=True)
        touched = touched.astype(bool)
        allocated |= touched
        same_grids(m, V)
        hits.append(same_cast(m, V, poses[j], allocated, touched, min(i, 3)))
    return hits


@pytest.mark.parametrize("W,H", [(100, 75), (9, 17), (8, 8), (642, 483)])
def test_map_image_sizes(cuda, W, H):
    """W, H not multiples of the range cell (8) or the touch stride (4).  Below 16 pixels in W or H the range map is
    always empty, in both: a block's projected box spans at most one cell column (or row), and such boxes are dropped,
    so every ray misses."""
    sc = small_scene("laparoscopy512", res=64, frame_ids=np.arange(0, 10, 2), W=W, H=H)
    m = map_for(sc, 96, 4.0)
    hits = run_frame_by_frame(m, oracle_for(m), sc, range(5), 4.0)
    if W < 16 or H < 16:
        assert not any(h.any() for h in hits)
    else:
        assert hits[-1].mean() > 0.3


def test_map_130_frames_in_one_batch(cuda):
    """bslam_vbg_integrate's 64-frame chunks (64 + 64 + 2): per-frame counts, grids, the last frame's blocks and the
    synthesized frame against the oracle run frame by frame; split calls (1 + 63 + 66) give the same map"""
    F = 130
    ids = np.linspace(0, 999, F).astype(int)
    ids[[65, -1]] = ids[[-1, 65]]         # the last frame looks elsewhere than the frames before it
    sc = small_scene("laparoscopy512", res=64, frame_ids=ids, W=160, H=120)
    poses = ext_of(sc["E"])
    dmax = [float((d.astype(np.float32) / 1000.0).max()) for d in sc["depth_u16"]]
    m = map_for(sc, 64, 4.0)
    counts = torch.zeros(F, dtype=torch.int64, device=cuda)
    m.integrate_batch(sc["depth_u16"], sc["color"], poses, dmax, update_counts=counts)
    V = oracle_for(m)
    allocated = np.zeros((4, 4, 4), bool)
    co, touched = [], []
    for i in range(F):
        n, t = V.integrate_vbg(sc["depth_u16"][i], sc["K"], poses[i], rgb=sc["color"][i], depth_scale=1000.0, depth_max=dmax[i],
                               trunc_voxel_multiplier=4.0, return_touched=True)
        co.append(n)
        touched.append(t.astype(bool))
        allocated |= touched[-1]
    assert counts.cpu().tolist() == co
    assert min(co[64:]) > 0, "a frame of the later chunks updates nothing"
    assert not np.array_equal(touched[-1], touched[-2]) and not np.array_equal(touched[-1], touched[128]), "the last frame is not distinct"
    same_grids(m, V)
    assert same_cast(m, V, poses[-1], allocated, touched[-1], 3.0).mean() > 0.3
    m2 = map_for(sc, 64, 4.0)
    c2 = torch.zeros(F, dtype=torch.int64, device=cuda)
    for lo, hi in ((0, 1), (1, 64), (64, F)):
        m2.integrate_batch(sc["depth_u16"][lo:hi], sc["color"][lo:hi], poses[lo:hi], dmax[lo:hi], update_counts=c2[lo:hi])
    assert torch.equal(c2, counts)
    for x, y in zip(m2.model.export_dense(True), m.model.export_dense(True)):
        assert torch.equal(x, y)
    assert torch.equal(m2.allocated_blocks(last_frame=True), m.allocated_blocks(last_frame=True))


def test_map_last_frame_all_zero_depth(cuda):
    sc = small_scene("laparoscopy512", res=64, frame_ids=[0, 2, 4], W=100, H=75)
    m = map_for(sc, 64, 4.0)
    depth = sc["depth_u16"].copy()
    depth[-1] = 0
    m.integrate_batch(depth, sc["color"], ext_of(sc["E"]), 3.0)
    assert m.allocated_blocks().any() and not m.allocated_blocks(last_frame=True).any()
    out = m.synthesize_model_frame()
    assert all(not v.any() for v in out.values())


def test_map_non_cubic_box_below_zero(cuda):
    sc = small_scene("laparoscopy512", res=64, frame_ids=np.arange(0, 10, 2), W=160, H=120)
    res = (48, 96, 64)
    m = map_for(sc, res, 4.0)
    b0 = np.rint(m.model.origin / (m.voxel_size * 16))
    assert (b0 < 0).all(), b0
    hits = run_frame_by_frame(m, oracle_for(m), sc, range(5), 4.0)
    assert hits[-1].mean() > 0.2


def test_map_reference_defaults(cuda):
    """trunc_voxel_multiplier 8, no colour, the default weight threshold min(frame_id, 3)"""
    ids = [0, 1, 2, 3, 7]
    sc = small_scene("laparoscopy512", res=64, frame_ids=np.array(ids) * 2, W=100, H=75, with_color=False)
    m = MAP(100, 75, k3x3(sc["K"]), "CUDA:0", 1000.0, resolution=64, origin=map_origin((64,) * 3, 0.0058), color=False)
    V = oracle_for(m, color=False)
    hits = run_frame_by_frame(m, V, sc, ids, 8.0, color=False)
    assert hits[-1].any()
    # the legacy cast of the block-integrated box
    V.sdf_trunc = m.model.sdf_trunc
    K6 = (100, 75) + tuple(sc["K"])
    gpu = m.model.raycast(K6, sc["E"], weight_threshold=1.0)
    assert assert_same(gpu, raycast_ref.raycast(V, sc["K"], sc["E"], 100, 75, weight_threshold=1.0)).any()


def corner_u(pose, K, keys, bl):
    """EstimateRange's u / 8 and v / 8 of the 8 corners of blocks `keys` [n,3] (world block grid), in the kernel's
    float32 operation order; corners with z <= 0 are nan"""
    E = ext_of(pose)[:3].astype(np.float32)
    f32 = np.float32
    out = []
    for i in range(8):
        corner = keys + np.array([i & 1, (i >> 1) & 1, (i >> 2) & 1])
        w = corner.astype(f32) * f32(bl)
        c = [((E[r, 0] * w[:, 0] + E[r, 1] * w[:, 1]) + E[r, 2] * w[:, 2]) + E[r, 3] for r in range(3)]
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            inv = f32(1.0) / c[2]
            u = (f32(K[0]) * c[0] * inv + f32(K[2])) / f32(8.0)
            v = (f32(K[1]) * c[1] * inv + f32(K[3])) / f32(8.0)
        out.append(np.where(c[2] > 0, u, np.nan))
        out.append(np.where(c[2] > 0, v, np.nan))
    return np.stack(out, -1)


def test_map_range_estimate_of_a_corner_on_the_camera_plane(cuda):
    """A surface closer than the truncation activates the block holding the camera.  A corner of that block 1e-10 m in
    front of the camera plane projects to |u| / 8 far beyond 2^31, where the float -> int conversion saturates on the
    GPU and is undefined in C (x86: INT_MIN).  That block's box differs between the two, but the activated blocks
    around it share the corner and cover the same cells with the same depths, so the range maps and casts agree."""
    W, H, vs, mult = 64, 48, 0.0058, 8.0
    K = np.array([40.0, 40.0, 32.0, 24.0])
    th = np.arctan(0.5)
    R = np.array([[np.cos(th), 0, np.sin(th)], [0, 1, 0], [-np.sin(th), 0, np.cos(th)]])      # yaw: camera -> world
    pose = np.eye(4)
    pose[:3, :3] = R
    pose[:3, 3] = -0.02 * R[:, 0] - 1e-10 * R[:, 2]          # world corner (0, 0, 0) at camera (0.02, 0, 1e-10)
    m = MAP(W, H, k3x3(K), "CUDA:0", 1000.0, voxel_size=vs, trunc_voxel_multiplier=mult, resolution=64, origin=(-2 * 16 * vs,) * 3)
    V = oracle.o3d.Volume(64, vs, vs * mult, m.model.origin, with_color=True)
    depth = np.full((H, W), 20, np.uint16)            # 2 cm: closer than the 4.64 cm truncation
    rgb = np.full((H, W, 3), 90, np.uint8)
    m.integrate_batch(depth, rgb, pose[None], 3.0)
    _, touched = V.integrate_vbg(depth, K, pose, rgb=rgb, depth_scale=1000.0, depth_max=3.0, trunc_voxel_multiplier=mult, return_touched=True)
    touched = touched.astype(bool)
    bl = np.float32(vs) * np.float32(16)
    keys = np.argwhere(touched) - 2
    assert (keys == np.floor(pose[:3, 3] / bl)).all(axis=1).any(), "the camera's block is not activated"
    uv = corner_u(pose, K, keys, bl)
    assert np.nanmax(np.abs(uv)) > 2.0 ** 31, np.nanmax(np.abs(uv))
    same_grids(m, V)
    same_cast(m, V, pose, touched, touched, 0.0)
    same_cast(m, V, pose, touched, touched, 0.0, depth_min=0.0)


# ------------------------------------------------------------------ 5. volume lifecycle
def test_reset_copy_and_reimport(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=3, W=160, H=120)
    vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 64, sc["origin"], color=True, device=cuda)
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    vol.integrate_batch(depth, torch.as_tensor(sc["color"], device=cuda), sc["intrinsic"], sc["E"])
    base = vol.raycast(sc["intrinsic"], sc["E"])
    assert (base["depth"] > 0).float().mean() > 0.3
    twin = copy.deepcopy(vol)
    fresh = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 64, sc["origin"], color=True, device=cuda)
    fresh.import_dense(*vol.export_dense(with_color=True))
    for other in (twin, fresh):
        out = other.raycast(sc["intrinsic"], sc["E"])
        for k in KEYS:
            assert torch.equal(out[k], base[k]), k
    vol.reset()
    assert all(not v.any() for v in vol.raycast(sc["intrinsic"], sc["E"]).values())
    out = twin.raycast(sc["intrinsic"], sc["E"])          # the copy is its own storage
    assert torch.equal(out["depth"], base["depth"])


# ------------------------------------------------------------------ 6. full size
@pytest.mark.slow
def test_full_size_parity(cuda):
    """BASELINE configs[3] (laparoscopy512, 1000 frames) integrated in full, ray cast from 8 trajectory poses; and MAP at
    the reference's defaults (256^3, 5.8 mm, multiplier 8, no colour) on the same frames: bit-equal with the reference"""
    cfg = S.config("laparoscopy512")
    F, W, H, K = cfg["frames"], cfg["W"], cfg["H"], cfg["K"]
    E = cfg["extrinsics"](F)
    intrinsic = PinholeCameraIntrinsic(W, H, *K)
    depth_u16 = torch.empty((F, H, W), dtype=torch.uint16, device=cuda)
    for lo in range(0, F, 100):
        depth_u16[lo:lo + 100] = S.render(cfg["surface"], E[lo:lo + 100], K=K, W=W, H=H, device=cuda, with_color=False, first_frame=lo)[0]
    vol = DenseTSDFVolume(cfg["voxel_length"], cfg["sdf_trunc"], cfg["resolution"], cfg["origin"], color=False, device=cuda)
    vol.integrate_u16_chunks(depth_u16, None, intrinsic, E, vol.stream_chunks(F), 1000.0, 3.0)
    poses = E[np.linspace(0, F - 1, 8).astype(int)]
    gpu = vol.raycast(intrinsic, poses, colors=False)
    V = oracle.o3d.Volume(cfg["resolution"], cfg["voxel_length"], cfg["sdf_trunc"], cfg["origin"])
    t, w = (x.cpu().numpy() for x in vol.export_dense())
    V.tsdf, V.weight = t.reshape(-1), w.reshape(-1)
    del t, w
    hit = assert_same(gpu, raycast_ref.raycast(V, K, poses, W, H, colors=False))
    assert hit.mean() > 0.5
    del V, vol, gpu
    vs, res = 0.0058, 256
    centre = np.asarray(cfg["origin"]) + 0.5 * cfg["resolution"] * cfg["voxel_length"]
    m = MAP(W, H, k3x3(K), "CUDA:0", 1000.0, resolution=res, origin=map_origin((res,) * 3, vs, centre), color=False)
    P_all = ext_of(E)
    for lo in range(0, F, 200):
        m.integrate_batch(depth_u16[lo:lo + 200], None, P_all[lo:lo + 200], 3.0)
    V = oracle.o3d.Volume(res, vs, vs * 8.0, m.model.origin)
    t, w = (x.cpu().numpy() for x in m.model.export_dense())
    V.tsdf, V.weight = t.reshape(-1), w.reshape(-1)
    hit = same_cast(m, V, P_all[-1], m.allocated_blocks().cpu().numpy(), m.allocated_blocks(last_frame=True).cpu().numpy(), 3.0)
    assert hit.mean() > 0.3
