"""K4 surface extraction (csrc/bslam_extract.cu) at the shapes, values and sizes its parity tests skip -- `-m gpu`
(the 264^3 box and the 50 000-brick cache case are `-m "gpu and slow"`).

Bar, against the CPU oracle (`oracle.o3d.Volume.extract_mesh` / `extract_points`): counts, vertex-key sets, canonical
triangles and point keys EXACT; vertex positions, mesh colours, point positions, normals and point colours BIT FOR BIT
equal to the oracle's float64 rounded once to float32 (GPU and oracle evaluate the same float64 expressions in the same
order, nvcc -fmad=false / gcc -ffp-contract=off).

Covered: multi-CTA prefix sums (8192, 8193 and 16 400 bricks; 35 937 bricks at 264^3) with the surface everywhere, only
in the first CTA's bricks and only in the last CTA's; boxes with dims 1..9 and 15..17 per axis and off-grid origins;
tsdf exactly on 0, -0.0, +-0.98, +-1 and the next floats on either side; weight-0 voxels; the `MAP` flavour with integer
weights 1..5 and thresholds 0, 1, 2.5, 3, 4; slab seams (ragged top slab, single-brick-layer slab, empty middle slab,
negative corners only on the neighbour's boundary plane) through the Python merge and through `bslam_mesh_merge`, with
colour; emit capacities below the counts; the incremental point cache (128 / 129-point bricks, the slot pool running
out, a one-brick change, normals off, colour-less volumes, every integration path as a writer).

Not covered: `scan_totals_kernel` above 1024 CTAs and the "too many bricks" rejection above 2048 CTAs -- they need more
than 8.4 M bricks (>= 34 GB of volume) and an oracle pass over more than 4 * 10^9 voxels.

Threshold 0 of the `MAP` flavour: the GPU keeps a voxel when weight > 0, the oracle (Open3D's legacy rule) when
weight != 0.  They differ only for negative or NaN weights, which no integrator writes;
`test_map_flavour_threshold_zero_ignores_negative_weights` pins the difference.
"""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
from bodyslam_b200 import _lib
from bodyslam_b200.sharding import merge_slab_meshes
from bodyslam_b200.tsdf import MAP, DenseTSDFVolume
from test_gpu_extract import analytic_field, gpu_volume
from util import canon_mesh, small_scene

pytestmark = pytest.mark.gpu

VL = 0.01
ORIGIN = (0.1234, -0.2071, 0.3333)         # off the voxel grid of the volume's own corner


# ---------------------------------------------------------------------------------------------- fields and references
def wave_field(dims, seed=0, region=None):
    """smooth periodic tsdf with a surface in every 8^3 brick; region: bool [nx,ny,nz] mask of valid voxels (weight 1,
    elsewhere weight 0 and tsdf 1)"""
    rng = np.random.default_rng(seed)
    x, y, z = np.meshgrid(*(np.arange(n, dtype=np.float64) for n in dims), indexing="ij")
    p = rng.uniform(0, 6.28, size=3)
    t = 0.45 * np.sin(1.3 * x + 0.45 * z + p[0]) + 0.4 * np.sin(1.7 * y + 0.31 * z + p[1]) + 0.25 * np.sin(0.77 * z + p[2])
    t = np.clip(t * 1.6, -1, 1).astype(np.float32)
    w = np.ones(dims, np.float32)
    if region is not None:
        t[~region] = 1.0
        w[~region] = 0.0
    return t, w


def rand_color(dims, seed=1):
    return np.random.default_rng(seed).uniform(0, 255, size=tuple(dims) + (3,)).astype(np.float32)


def ref_volume(t, w, color=None, origin=ORIGIN, gz0=0, vl=VL):
    V = oracle.o3d.Volume(t.shape, vl, 0.04, origin, gz0=gz0, with_color=color is not None)
    V.tsdf[:] = t.reshape(-1)
    V.weight[:] = w.reshape(-1)
    if color is not None:
        V.color[:] = color.reshape(-1)
    return V


def dev_volume(cuda, t, w, color=None, origin=ORIGIN, **kw):
    return gpu_volume(cuda, t, w, vl=VL, origin=origin, color=color, **kw)


def key_code(keys, dims):
    k = np.asarray(keys).astype(np.int64)
    return ((k[:, 0] * (dims[1] + 1) + k[:, 1]) * (dims[2] + 1) + k[:, 2]) * 4 + k[:, 3]


def f32(a):
    return np.asarray(a, dtype=np.float64).astype(np.float32)


def assert_bits(got, want, what):
    got, want = np.asarray(got, np.float32), f32(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not np.array_equal(got.view(np.int32), want.view(np.int32)):
        bad = np.nonzero(got.view(np.int32) != want.view(np.int32))
        d = np.abs(got.astype(np.float64) - want.astype(np.float64)).max()
        raise AssertionError(f"{what}: {len(bad[0])} values differ from float32(oracle), max |diff| {d:.3g}")


def check_mesh(mesh, ref, dims, color=False):
    """exact counts, keys and canonical triangles; vertices (and colours) bit for bit"""
    V, K, T = (x.cpu().numpy() for x in (mesh.vertices, mesh.vertex_keys, mesh.triangles))
    assert len(V) == len(ref["vertices"]) and len(T) == len(ref["triangles"]), (len(V), len(ref["vertices"]), len(T), len(ref["triangles"]))
    kc, vc, tc = canon_mesh(V, K, T, dims)
    ko, vo, to = canon_mesh(ref["vertices"], ref["keys"], ref["triangles"], dims)
    assert np.array_equal(kc, ko), "vertex edge keys differ"
    assert np.array_equal(tc, to), "triangles differ after canonical ordering"
    assert_bits(vc, vo, "vertices")
    if color:
        og, oo = np.argsort(key_code(K, dims)), np.argsort(key_code(ref["keys"], dims))
        assert_bits(mesh.vertex_colors.cpu().numpy()[og], ref["colors"][oo], "vertex colours")


def check_points(pcd, ref, dims, color=False, normals=True):
    kg = pcd.point_keys.cpu().numpy()
    assert len(kg) == len(ref["keys"]), (len(kg), len(ref["keys"]))
    cg, co = key_code(kg, dims), key_code(ref["keys"], dims)
    og, oo = np.argsort(cg), np.argsort(co)
    assert np.array_equal(cg[og], co[oo]), "point keys differ"
    assert_bits(pcd.points.cpu().numpy()[og], ref["points"][oo], "points")
    if normals:
        assert_bits(pcd.normals.cpu().numpy()[og], ref["normals"][oo], "normals")
    if color:
        assert_bits(pcd.colors.cpu().numpy()[og], ref["colors"][oo], "point colours")


def check_both(cuda, t, w, color=None, origin=ORIGIN, min_tris=0):
    V = ref_volume(t, w, color, origin)
    vol = dev_volume(cuda, t, w, color, origin)
    ref = V.extract_mesh()
    assert len(ref["triangles"]) >= min_tris
    check_mesh(vol.extract_triangle_mesh(), ref, t.shape, color is not None)
    check_points(vol.extract_point_cloud(), V.extract_points(), t.shape, color is not None)
    return vol, ref


# ---------------------------------------------------------------------------------------------- 1. multi-CTA scans
def bricks_with(keys, dims):
    k = np.asarray(keys).astype(np.int64) // 8
    nbx, nby = (dims[0] + 7) // 8, (dims[1] + 7) // 8
    return np.unique((k[:, 2] * nby + k[:, 1]) * nbx + k[:, 0])


@pytest.mark.parametrize("dims", [(8, 8, 8 * 8192), (8, 8, 8 * 8193), (16, 16, 8 * 4100)], ids=["8192", "8193", "16400"])
def test_multi_cta_scans_surface_in_every_brick(cuda, dims):
    t, w = wave_field(dims, seed=sum(dims))
    vol, ref = check_both(cuda, t, w, origin=ORIGIN)
    nb = np.prod([(n + 7) // 8 for n in dims])
    assert len(bricks_with(ref["keys"], dims)) == nb          # every brick emits: every CTA of every scan is non-empty


@pytest.mark.parametrize("where", ["first_cta", "last_cta"])
def test_multi_cta_scans_surface_in_one_cta(cuda, where):
    dims = (16, 16, 8 * 4100)                                  # 16 400 bricks: CTAs of 8192, 8192 and 16 bricks
    z = np.arange(dims[2])
    zmask = z < 8 * 2048 if where == "first_cta" else z >= 8 * 4096
    region = np.broadcast_to(zmask[None, None, :], dims)
    t, w = wave_field(dims, seed=7, region=region)
    col = rand_color(dims, seed=3)
    vol, ref = check_both(cuda, t, w, color=col, min_tris=1000)
    b = bricks_with(ref["keys"], dims)
    assert (b.max() < 8192) if where == "first_cta" else (b.min() >= 16384 - 4)


@pytest.mark.slow
def test_multi_cta_scans_264_cube(cuda):
    dims = (264,) * 3                                          # 35 937 bricks: 5 scan CTAs
    t, w = analytic_field(264, "noise", seed=11)
    w[np.random.default_rng(2).uniform(size=dims) < 0.02] = 0
    col = rand_color(dims, seed=4)
    check_both(cuda, t, w, color=col, min_tris=10**5)


# ---------------------------------------------------------------------------------------------- 2. shapes
SHAPES = [(1, 9, 17), (9, 1, 8), (2, 2, 2), (8, 8, 8), (17, 15, 9), (3, 16, 5), (15, 17, 16), (9, 9, 9), (4, 7, 2), (16, 3, 15),
          (1, 1, 1), (6, 17, 3)]


@pytest.mark.parametrize("dims", SHAPES, ids=["x".join(map(str, d)) for d in SHAPES])
@pytest.mark.parametrize("with_color", [False, True])
def test_small_and_ragged_boxes(cuda, dims, with_color):
    t, w = wave_field(dims, seed=int(np.prod(dims)))
    w[np.random.default_rng(5).uniform(size=dims) < 0.05] = 0
    col = rand_color(dims) if with_color else None
    vol, ref = check_both(cuda, t, w, color=col, origin=(-0.377, 0.0412, 1.9999))
    if min(dims) < 2:
        assert len(ref["vertices"]) == 0                       # no cube at all: empty, not an error
    pcd = vol.extract_point_cloud()
    if min(dims) < 3:
        assert pcd.points.shape[0] == 0                        # no interior voxel


# ---------------------------------------------------------------------------------------------- 3. values at the thresholds
def special_values():
    vals = [0.0, -0.0, 0.98, -0.98, 1.0, -1.0]
    out = []
    for v in vals:
        f = np.float32(v)
        out += [f, np.nextafter(f, np.float32(2)), np.nextafter(f, np.float32(-2))]
    return np.array(out + [0.3, -0.3, 0.5, -0.7], np.float32)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_tsdf_at_the_thresholds(cuda, seed):
    dims = (23, 18, 20)
    rng = np.random.default_rng(seed)
    t = rng.choice(special_values(), size=dims).astype(np.float32)
    w = rng.integers(1, 4, size=dims).astype(np.float32)
    w[rng.uniform(size=dims) < 0.1] = 0                        # weight-0 voxels next to valid ones
    col = rand_color(dims, seed)
    assert np.signbit(t[t == 0]).any() and (t == np.float32(-0.98)).any()
    check_both(cuda, t, w, color=col, min_tris=100)


def set_flavour(vol, thr, pos_half):
    _lib.check(vol._L.bslam_tsdf_set_extract_flavour(vol._h, float(thr), float(pos_half)))


@pytest.mark.parametrize("thr", [0.0, 1.0, 2.5, 3.0, 4.0])
def test_map_flavour_integer_weights(cuda, thr):
    dims = (32, 24, 17)
    t, _ = wave_field(dims, seed=9)
    x, y, z = np.meshgrid(*(np.arange(n) for n in dims), indexing="ij")
    w = (1 + (x // 3 + 2 * (y // 3) + 3 * (z // 3) + int(thr)) % 5).astype(np.float32)   # stored weights 1..5 in 3^3 blocks
    col = rand_color(dims, seed=8)
    origin = (0.32, -0.48, 0.16)
    V = ref_volume(t, w, col, origin)
    vol = dev_volume(cuda, t, w, col, origin)
    set_flavour(vol, thr, 0.0)
    oracle.o3d.set_extract_flavour(thr, 0.0)
    try:
        ref, refp = V.extract_mesh(), V.extract_points()
    finally:
        oracle.o3d.set_extract_flavour(0.0, 0.5)
    assert len(ref["triangles"]) > 50 and len(refp["points"]) > 50
    check_mesh(vol.extract_triangle_mesh(), ref, dims, color=True)
    check_points(vol.extract_point_cloud(), refp, dims, color=True)


def test_map_flavour_extraction_of_a_map(cuda):
    """`MAP.extract_pcd` / `extract_mesh` after integration: positions, normals and colours, not only counts"""
    sc = small_scene("laparoscopy512", res=64, frame_ids=np.arange(0, 10, 2))
    vs, res = 0.0058, 96
    bs = vs * 16
    centre = sc["origin"] + 0.5 * 64 * sc["voxel_length"]
    origin = np.floor((centre - 0.5 * res * vs) / bs + 0.5) * bs
    K = np.array([[sc["K"][0], 0, sc["K"][2]], [0, sc["K"][1], sc["K"][3]], [0, 0, 1]])
    m = MAP(640, 480, K, "CUDA:0", 1000.0, voxel_size=vs, trunc_voxel_multiplier=4.0, resolution=res, origin=origin)
    poses = np.stack([np.linalg.inv(E) for E in sc["E"]])
    dmax = [float((d.astype(np.float32) / 1000.0).max()) for d in sc["depth_u16"]]
    m.integrate_batch(sc["depth_u16"], sc["color"], poses, dmax)
    t, w, c = (x.cpu().numpy() for x in m.model.export_dense(with_color=True))
    V = ref_volume(t, w, c, origin, vl=vs)
    oracle.o3d.set_extract_flavour(3.0, 0.0)
    try:
        ref, refp = V.extract_mesh(), V.extract_points()
    finally:
        oracle.o3d.set_extract_flavour(0.0, 0.5)
    assert len(refp["points"]) > 1000 and (w == 3).any()
    check_mesh(m.extract_mesh(), ref, (res,) * 3, color=True)
    check_points(m.extract_pcd(), refp, (res,) * 3, color=True)


def test_map_flavour_threshold_zero_ignores_negative_weights(cuda):
    """threshold 0: the GPU rule is weight > 0, the oracle's weight != 0 -- equal for every weight an integrator writes
    (>= 0); a negative weight is invalid on the GPU and valid in the oracle"""
    dims = (16, 16, 16)
    t, w = wave_field(dims, seed=3)
    w[5:9, 5:9, 5:9] = -1.0
    vol = dev_volume(cuda, t, w, origin=(0.0, 0.0, 0.0))
    set_flavour(vol, 0.0, 0.0)
    oracle.o3d.set_extract_flavour(0.0, 0.0)
    try:
        ref_neg = ref_volume(t, w, origin=(0.0, 0.0, 0.0)).extract_mesh()
        w0 = w.copy()
        w0[w0 < 0] = 0
        ref_zero = ref_volume(t, w0, origin=(0.0, 0.0, 0.0)).extract_mesh()
    finally:
        oracle.o3d.set_extract_flavour(0.0, 0.5)
    mesh = vol.extract_triangle_mesh()
    check_mesh(mesh, ref_zero, dims)                           # negative weight == weight 0 on the GPU
    assert len(ref_neg["triangles"]) > len(ref_zero["triangles"])


# ---------------------------------------------------------------------------------------------- 4. slab seams
def slab_volumes(cuda, t, w, col, bounds):
    nz = t.shape[2]
    return [dev_volume(cuda, t[:, :, a:b].copy(), w[:, :, a:b].copy(), None if col is None else col[:, :, a:b].copy(), gz0=a, z_total=nz)
            for a, b in bounds]


def slab_meshes(vols, color):
    out = []
    for i, v in enumerate(vols):
        lo = vols[i - 1].export_plane(vols[i - 1].nz - 1) if i > 0 else None
        hi = vols[i + 1].export_plane(0) if i + 1 < len(vols) else None
        hc = vols[i + 1].export_plane_color(0) if (color and i + 1 < len(vols)) else None
        out.append(v.extract_triangle_mesh(halo_lo=lo, halo_hi=hi, halo_hi_color=hc))
    return out


def merge_on_gpu(parts, bounds, nx, ny):
    """bslam_mesh_merge on the slab rows concatenated in one buffer (what the gather side of ShardedTSDF does)"""
    L = _lib.load()
    n = len(parts)
    nv = np.array([p.vertices.shape[0] for p in parts], np.int64)
    nt = np.array([p.triangles.shape[0] for p in parts], np.int64)
    keys = torch.cat([p.vertex_keys for p in parts]).contiguous()
    tris = torch.cat([p.triangles for p in parts]).contiguous()
    ws = torch.empty(L.bslam_mesh_merge_workspace_bytes(n, nx, ny), dtype=torch.uint8, device=keys.device)
    zoff = np.array([a for a, _ in bounds], np.int32)
    unres = np.full(1, -1, np.int64)
    _lib.check(L.bslam_mesh_merge(n, _lib.ptr(nv), _lib.ptr(nt), _lib.ptr(zoff), nx, ny, _lib.ptr(keys), _lib.ptr(tris), _lib.ptr(ws),
                                  _lib.ptr(unres), _lib.stream_ptr(keys.device)))
    cols = torch.cat([p.vertex_colors for p in parts]) if parts[0].vertex_colors is not None else None
    from bodyslam_b200.geometry import TriangleMesh
    return TriangleMesh(torch.cat([p.vertices for p in parts]), tris, cols, keys), int(unres[0])


def seam_field(case):
    if case == "ragged_top":
        t, w = analytic_field(48, "noise", seed=5)
        return t[:, :40, :45].copy(), w[:, :40, :45].copy(), [(0, 16), (16, 32), (32, 45)]
    if case == "two_slabs":
        t, w = analytic_field(40, "holes", seed=2)
        return t, w, [(0, 24), (24, 40)]
    if case == "one_layer_middle":
        t, w = analytic_field(40, "noise", seed=6)
        return t, w, [(0, 16), (16, 24), (24, 40)]
    if case == "empty_middle":
        t, w = wave_field((32, 24, 48), seed=4)
        t[:, :, 15:33] = 0.7                                   # nothing changes sign from plane 15 to plane 32
        return t, w, [(0, 16), (16, 32), (32, 48)]
    if case == "negative_only_on_boundary":
        t = np.full((24, 24, 32), 0.6, np.float32)
        w = np.ones_like(t)
        rng = np.random.default_rng(1)
        m = rng.uniform(size=(24, 24)) < 0.3
        t[:, :, 16][m] = -0.4                                  # the only negative voxels: plane 0 of the upper slab
        return t, w, [(0, 16), (16, 32)]
    raise ValueError(case)


SEAMS = ["ragged_top", "two_slabs", "one_layer_middle", "empty_middle", "negative_only_on_boundary"]


@pytest.mark.parametrize("case", SEAMS)
@pytest.mark.parametrize("merge", ["python", "bslam_mesh_merge"])
def test_slab_seams_give_the_full_mesh_with_colour(cuda, case, merge):
    t, w, bounds = seam_field(case)
    dims = t.shape
    col = rand_color(dims, seed=len(case))
    ref = ref_volume(t, w, col).extract_mesh()
    assert len(ref["triangles"]) > 20
    vols = slab_volumes(cuda, t, w, col, bounds)
    parts = slab_meshes(vols, color=True)
    if case == "empty_middle":
        assert parts[1].vertices.shape[0] == 0 and parts[1].triangles.shape[0] == 0
    if case == "negative_only_on_boundary":
        assert (parts[0].triangles < 0).any() and parts[0].vertices.shape[0] > 0
    if merge == "python":
        mesh = merge_slab_meshes(parts, [a for a, _ in bounds], ny=dims[1])
    else:
        mesh, unres = merge_on_gpu(parts, bounds, dims[0], dims[1])
        assert unres == 0
    check_mesh(mesh, ref, dims, color=True)


def test_slab_mesh_without_colour_plane_is_an_argument_error(cuda):
    t, w, bounds = seam_field("two_slabs")
    col = rand_color(t.shape)
    lo, hi = slab_volumes(cuda, t, w, col, bounds)
    with pytest.raises(RuntimeError, match="colour plane"):
        lo.extract_triangle_mesh(halo_hi=hi.export_plane(0))
    # colour-less volumes need no colour plane, and export_plane_color refuses them
    a, b = slab_volumes(cuda, t, w, None, bounds)
    m = a.extract_triangle_mesh(halo_hi=b.export_plane(0))
    assert m.vertex_colors is None and m.vertices.shape[0] > 0
    with pytest.raises(RuntimeError, match="no colour"):
        b.export_plane_color(0)


def test_mesh_merge_rejections_and_unresolved_references(cuda):
    L = _lib.load()
    t, w, bounds = seam_field("ragged_top")
    dims = t.shape
    ref = ref_volume(t, w).extract_mesh()
    parts = slab_meshes(slab_volumes(cuda, t, w, None, bounds), color=False)
    # a fabricated reference to an edge the next slab does not have: counted as unresolved
    bad = [copy.copy(p) for p in parts]
    tr = parts[0].triangles.clone()
    neg = torch.nonzero(tr < 0)
    assert len(neg) > 0
    tr[neg[0, 0], neg[0, 1]] = -(1 + 3)                      # edge code 3 = axis 3 of voxel (0, 0): never a vertex
    bad[0].triangles = tr
    _, unres = merge_on_gpu(bad, bounds, dims[0], dims[1])
    assert unres == 1
    # a reference from the top slab has no next slab: unresolved too
    bad = [copy.copy(p) for p in parts]
    tr = parts[-1].triangles.clone()
    tr[0, 0] = -1
    bad[-1].triangles = tr
    _, unres = merge_on_gpu(bad, bounds, dims[0], dims[1])
    assert unres == 1
    # the real slabs resolve
    mesh, unres = merge_on_gpu(parts, bounds, dims[0], dims[1])
    assert unres == 0
    check_mesh(mesh, ref, dims)

    dev = cuda
    ws = torch.zeros(L.bslam_mesh_merge_workspace_bytes(65, 8, 8), dtype=torch.uint8, device=dev)
    keys = torch.zeros((4, 4), dtype=torch.int32, device=dev)
    tris = torch.zeros((1, 3), dtype=torch.int32, device=dev)
    st = _lib.stream_ptr(dev)

    def call(n, kptr):
        nv = np.zeros(n, np.int64)
        nt = np.zeros(n, np.int64)
        z = np.arange(n, dtype=np.int32) * 8
        return L.bslam_mesh_merge(n, _lib.ptr(nv), _lib.ptr(nt), _lib.ptr(z), 8, 8, kptr, _lib.ptr(tris), _lib.ptr(ws), None, st)

    assert call(64, _lib.ptr(keys)) == _lib.OK                # the 64-slab limit itself is accepted
    assert call(65, _lib.ptr(keys)) == _lib.E_ARG
    assert call(0, _lib.ptr(keys)) == _lib.E_ARG
    assert call(2, C.c_void_p(keys.data_ptr() + 4)) == _lib.E_ARG
    assert "16-byte aligned" in L.bslam_last_error().decode()


def test_mesh_merge_64_slabs(cuda):
    """the most slabs bslam_mesh_merge takes, one brick layer each, with colour"""
    dims = (16, 16, 8 * 64)
    t, w = wave_field(dims, seed=12)
    col = rand_color(dims, seed=6)
    bounds = [(8 * i, 8 * i + 8) for i in range(64)]
    ref = ref_volume(t, w, col).extract_mesh()
    parts = slab_meshes(slab_volumes(cuda, t, w, col, bounds), color=True)
    mesh, unres = merge_on_gpu(parts, bounds, dims[0], dims[1])
    assert unres == 0
    check_mesh(mesh, ref, dims, color=True)


# ---------------------------------------------------------------------------------------------- 5. capacity and coverage
GUARD = 64


def guarded(rows, width, dtype):
    """NaN / sentinel filled buffer with GUARD rows more than the full output: a write past a capacity below the count
    stays inside the allocation and shows"""
    if dtype == torch.float32:
        return torch.full((rows + GUARD, width), float("nan"), dtype=dtype, device="cuda")
    return torch.full((rows + GUARD, width), -123456789, dtype=dtype, device="cuda")


def untouched(t, start):
    tail = t[start:]
    return bool(torch.isnan(tail).all()) if t.dtype == torch.float32 else bool((tail == -123456789).all())


def mc_emit_raw(vol, cap_v, cap_t, colors=True):
    L = vol._L
    V, T = vol.mc_count()
    v, k, c, tr = guarded(V, 3, torch.float32), guarded(V, 4, torch.int32), guarded(V, 3, torch.float32), guarded(T, 3, torch.int32)
    _lib.check(L.bslam_mc_emit(vol._h, None, None, None, _lib.ptr(v), _lib.ptr(k), _lib.ptr(c) if colors else None, cap_v, _lib.ptr(tr), cap_t,
                               _lib.stream_ptr(vol.device)))
    torch.cuda.synchronize()
    return v, k, c, tr


def test_mc_emit_capacity_below_the_counts(cuda):
    t, w = analytic_field(40, "noise", seed=1)
    col = rand_color(t.shape)
    vol = dev_volume(cuda, t, w, col)
    V, T = vol.mc_count()
    assert V > 1000 and T > 1000
    full = mc_emit_raw(vol, V, T)
    for x in full:                                              # full capacity: every row written, nothing past the end
        assert not torch.isnan(x[:x.shape[0] - GUARD]).any() if x.dtype == torch.float32 else not (x[:x.shape[0] - GUARD] == -123456789).any()
        assert untouched(x, x.shape[0] - GUARD)
    for cap_v, cap_t in ((V // 3, T // 2), (0, T - 1), (V - 1, 0), (1, 1)):
        part = mc_emit_raw(vol, cap_v, cap_t)
        for x, y, cap in zip(part, full, (cap_v, cap_v, cap_v, cap_t)):
            assert torch.equal(x[:cap], y[:cap]), cap
            assert untouched(x, cap), cap
    ref = ref_volume(t, w, col).extract_mesh()
    from bodyslam_b200.geometry import TriangleMesh
    v, k, c, tr = full
    check_mesh(TriangleMesh(v[:V], tr[:T], c[:V], k[:V]), ref, t.shape, color=True)


def test_points_emit_capacity_below_the_count(cuda):
    t, w = analytic_field(40, "holes", seed=4)
    col = rand_color(t.shape)
    vol = dev_volume(cuda, t, w, col)
    L = vol._L
    cnt = np.zeros(1, np.int64)

    def emit(cap):
        _lib.check(L.bslam_points_count(vol._h, _lib.ptr(cnt), _lib.stream_ptr(cuda)))
        n = max(int(cnt[0]), cap)
        out = [guarded(n, 3, torch.float32), guarded(n, 3, torch.float32), guarded(n, 3, torch.float32), guarded(n, 4, torch.int32)]
        _lib.check(L.bslam_points_emit(vol._h, *(_lib.ptr(x) for x in out), cap, _lib.stream_ptr(cuda)))
        torch.cuda.synchronize()
        return out

    _lib.check(L.bslam_points_count(vol._h, _lib.ptr(cnt), _lib.stream_ptr(cuda)))
    P = int(cnt[0])
    full = emit(P)
    assert P > 1000
    for x in full:
        assert untouched(x, P)
        assert not (torch.isnan(x[:P]).any() if x.dtype == torch.float32 else (x[:P] == -123456789).any())
    for cap in (P // 2, P - 1, 1, 0):
        part = emit(cap)
        for x, y in zip(part, full):
            assert torch.equal(x[:cap], y[:cap]) and untouched(x, cap), cap
    from bodyslam_b200.geometry import PointCloud
    check_points(PointCloud(full[0][:P], full[2][:P], full[1][:P], full[3][:P]), ref_volume(t, w, col).extract_points(), t.shape, color=True)


# ---------------------------------------------------------------------------------------------- 6. incremental point cache
def brick_flags(vol):
    nbx, nby, nbz = (vol.nx + 7) // 8, (vol.ny + 7) // 8, (vol.nz + 7) // 8
    return vol.storage_layers()["flags"].cpu().numpy().reshape(nbz, nby, nbx)


def candidates(flags):
    """bricks b with flag bit 1 on any of b + {0,1}^3 (mc_mark_kernel)"""
    f = (flags & 2) != 0
    c = np.zeros_like(f)
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                c[:f.shape[0] - dz, :f.shape[1] - dy, :f.shape[2] - dx] |= f[dz:, dy:, dx:]
    return c


def dilate(m):
    out = np.zeros_like(m)
    p = np.pad(m, 1)
    for dz in range(3):
        for dy in range(3):
            for dx in range(3):
                out |= p[dz:dz + m.shape[0], dy:dy + m.shape[1], dx:dx + m.shape[2]]
    return out


def points_per_brick(pcd, vol):
    nbx, nby, nbz = (vol.nx + 7) // 8, (vol.ny + 7) // 8, (vol.nz + 7) // 8
    k = pcd.point_keys.cpu().numpy().astype(np.int64) // 8
    return np.bincount((k[:, 2] * nby + k[:, 1]) * nbx + k[:, 0], minlength=nbx * nby * nbz).reshape(nbz, nby, nbx)


def assert_same_cloud(inc, vol, normals=True):
    ref = copy.deepcopy(vol)
    ref.set_incremental_points(False)
    full = ref.extract_point_cloud(normals=normals)
    for a, b in ((inc.points, full.points), (inc.normals, full.normals), (inc.colors, full.colors), (inc.point_keys, full.point_keys)):
        assert (a is None) == (b is None)
        if a is not None:
            assert torch.equal(a, b)
    return full


def slab_pattern(dims, seed=None):
    """tsdf < 0 on x = 2, 3, 4 of every brick, > 0 elsewhere: every interior brick holds 2 x 64 = 128 points (seed:
    random magnitudes in [0.1, 0.9], else 0.5)"""
    t = np.full(dims, 0.5, np.float32)
    if seed is not None:
        t = np.random.default_rng(seed).uniform(0.1, 0.9, size=dims).astype(np.float32)
    xl = np.arange(dims[0]) % 8
    t[(xl >= 2) & (xl <= 4)] *= -1
    return t, np.ones(dims, np.float32)


def test_cache_bricks_of_128_and_129_points(cuda):
    dims = (24, 24, 40)
    t, w = slab_pattern(dims)
    t[14, 11, 32] = -0.5       # a z-crossing owned by voxel (14, 11, 31): brick (1, 1, 3) holds 129 points
    col = rand_color(dims)
    vol = dev_volume(cuda, t, w, col)
    vol.set_incremental_points(True, normals=True)
    first = vol.extract_point_cloud()
    check_points(first, ref_volume(t, w, col).extract_points(), dims, color=True)
    ppb = points_per_brick(first, vol)
    assert ppb[1, 1, 1] == 128 and ppb[3, 1, 1] == 129
    big = int((ppb > 128).sum())
    for _ in range(2):                                         # nothing changed: only bricks over 128 points are recomputed
        again = vol.extract_point_cloud()
        cand, rec = vol.points_last_stats()
        assert rec == big and cand == int(candidates(brick_flags(vol)).sum())
        assert_same_cloud(again, vol)


def one_pixel_frame(vol, target, depth_m):
    """a 1x1 depth frame whose camera sits 2 voxels in front (-x) of world point `target` looking along +x: it updates the
    voxels of a short cone around the target"""
    R = np.array([[0, 1, 0], [0, 0, 1], [1, 0, 0]], np.float64)        # camera z = world x
    c = np.asarray(target, np.float64) - np.array([2 * vol.voxel_length, 0, 0])
    E = np.eye(4)
    E[:3, :3] = R
    E[:3, 3] = -R @ c
    from bodyslam_b200.geometry import PinholeCameraIntrinsic
    intr = PinholeCameraIntrinsic(1, 1, 1.0, 1.0, 0.5, 0.5)            # one pixel, a wide cone
    depth = torch.full((1, 1, 1), float(depth_m), dtype=torch.float32, device=vol.device)
    color = torch.full((1, 1, 1, 3), 200, dtype=torch.uint8, device=vol.device)
    return depth, color, intr, E[None]


def expected_recomputed(vol, ppb_before):
    """bricks the incremental count pass recomputes: candidates whose 3x3x3 neighbourhood changed, or that hold more
    than 128 points"""
    f = brick_flags(vol)
    return int((candidates(f) & (dilate((f & 4) != 0) | (ppb_before > 128))).sum())


def test_cache_one_brick_change_recomputes_its_neighbourhood(cuda):
    dims = (40, 40, 40)
    t, w = slab_pattern(dims, seed=21)                          # <= 128 points per brick: clean bricks come from the cache
    vol = DenseTSDFVolume(VL, 1.2 * VL, dims, (0.0, 0.0, 0.0), color=True, device=cuda)    # short band: the frame stays in one brick
    vol.import_dense(t, w, rand_color(dims))
    vol.set_incremental_points(True, normals=True)
    first = vol.extract_point_cloud()
    ppb = points_per_brick(first, vol)
    target = (np.array([20, 20, 20]) + 0.5) * VL                   # centre of brick (2, 2, 2)
    vol.integrate_batch(*one_pixel_frame(vol, target, 2.2 * VL))
    dirty = (brick_flags(vol) & 4) != 0
    assert 1 <= dirty.sum() <= 2, np.argwhere(dirty)
    want = expected_recomputed(vol, ppb)
    inc = vol.extract_point_cloud()
    cand, rec = vol.points_last_stats()
    assert rec == want and 1 < rec < cand and (points_per_brick(first, vol) <= 128).all()
    assert_same_cloud(inc, vol)
    assert not torch.equal(inc.points, first.points) or not torch.equal(inc.normals, first.normals)


@pytest.mark.parametrize("with_color,normals", [(True, False), (False, True), (False, False)])
def test_cache_ragged_box_border_bricks(cuda, with_color, normals):
    dims = (37, 22, 29)                                         # ragged: every border brick is partial
    t, w = slab_pattern(dims, seed=2)
    col = rand_color(dims) if with_color else None
    vol = dev_volume(cuda, t, w, col, origin=(0.0, 0.0, 0.0))
    vol.set_incremental_points(True, normals=normals)
    first = vol.extract_point_cloud(normals=normals)
    refp = ref_volume(t, w, col, origin=(0.0, 0.0, 0.0)).extract_points(normals=normals)
    check_points(first, refp, dims, color=with_color, normals=normals)
    ppb = points_per_brick(first, vol)
    # change a corner brick and a brick on the +x face
    for target in ((np.array([2, 2, 2]) + 0.5) * VL, (np.array([34, 12, 13]) + 0.5) * VL):
        d, c, intr, E = one_pixel_frame(vol, target, 1.8 * VL)
        vol.integrate_batch(d, c if with_color else None, intr, E)
    want = expected_recomputed(vol, ppb)
    inc = vol.extract_point_cloud(normals=normals)
    cand, rec = vol.points_last_stats()
    assert rec == want and rec < cand
    assert_same_cloud(inc, vol, normals=normals)


@pytest.mark.slow
def test_cache_slot_pool_runs_out(cuda):
    dims = (8, 8, 8 * 50000)                                    # 50 000 candidate bricks > 49 152 cache slots
    t, w = slab_pattern(dims)                                   # <= 96 points per brick: every brick asks for a slot
    col = rand_color(dims)
    vol = dev_volume(cuda, t, w, col, origin=(0.0, 0.0, 0.0))
    vol.set_incremental_points(True, normals=True)
    first = vol.extract_point_cloud()
    check_points(first, ref_volume(t, w, col, origin=(0.0, 0.0, 0.0)).extract_points(), dims, color=True)
    ppb = points_per_brick(first, vol)
    small = int(((ppb > 0) & (ppb <= 128)).sum())
    assert small > 49152
    again = vol.extract_point_cloud()
    cand, rec = vol.points_last_stats()
    assert cand == 50000 and rec == cand - int((ppb == 0).sum()) - 49152
    assert_same_cloud(again, vol)
    # one frame that touches part of the box
    vol.integrate_batch(*one_pixel_frame(vol, (np.array([4, 4, 8 * 30000 + 4]) + 0.5) * VL, 2.2 * VL))
    inc = vol.extract_point_cloud()
    assert vol.points_last_stats()[1] >= rec
    assert_same_cloud(inc, vol)


def scene_volume(cuda, res=64, unit=False, color=True):
    sc = small_scene("laparoscopy512", res=res, frame_ids=np.arange(0, 40, 10), with_color=color)
    vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], res, sc["origin"], color=color, device=cuda, unit_activation=unit)
    vol.set_incremental_points(True, normals=True)
    return sc, vol


@pytest.mark.parametrize("writer", ["integrate_batch", "integrate_u16_batch", "integrate_host", "unit_activation", "colourless"])
def test_cache_every_writer_marks_changed_bricks(cuda, writer):
    from bodyslam_b200 import ops
    unit = writer == "unit_activation"
    sc, vol = scene_volume(cuda, res=128 if unit else 64, unit=unit, color=writer != "colourless")
    col = None if sc["color"] is None else torch.from_numpy(sc["color"]).to(cuda)

    def write(i):
        sl = slice(i, i + 1)
        c = None if col is None else col[sl]
        if writer == "integrate_u16_batch":
            vol.integrate_u16_batch(torch.from_numpy(sc["depth_u16"][sl]).to(cuda), c, sc["intrinsic"], sc["E"][sl])
        elif writer == "integrate_host":
            vol.integrate_host(sc["depth_u16"][sl], None if sc["color"] is None else sc["color"][sl], sc["intrinsic"], sc["E"][sl])
        else:
            vol.integrate_batch(ops.depth_from_u16(sc["depth_u16"][sl], 1000.0, 3.0, cuda), c, sc["intrinsic"], sc["E"][sl])

    write(0)
    first = vol.extract_point_cloud()
    assert first.points.shape[0] > 100
    for i in range(1, len(sc["E"])):
        write(i)
        inc = vol.extract_point_cloud()
        cand, rec = vol.points_last_stats()
        assert 0 < rec <= cand
        assert_same_cloud(inc, vol)


def test_cache_map_integrate_batch_marks_changed_bricks(cuda):
    sc = small_scene("laparoscopy512", res=64, frame_ids=np.arange(0, 10, 2))
    vs, res = 0.0058, 64
    bs = vs * 16
    centre = sc["origin"] + 0.5 * 64 * sc["voxel_length"]
    origin = np.floor((centre - 0.5 * res * vs) / bs + 0.5) * bs
    K = np.array([[sc["K"][0], 0, sc["K"][2]], [0, sc["K"][1], sc["K"][3]], [0, 0, 1]])
    m = MAP(640, 480, K, "CUDA:0", 1000.0, voxel_size=vs, trunc_voxel_multiplier=4.0, resolution=res, origin=origin)
    m.model.set_incremental_points(True, normals=True)
    poses = np.stack([np.linalg.inv(E) for E in sc["E"]])
    dmax = [float((d.astype(np.float32) / 1000.0).max()) for d in sc["depth_u16"]]
    seen = 0
    for i in range(len(poses)):
        m.integrate_batch(sc["depth_u16"][i:i + 1], sc["color"][i:i + 1], poses[i:i + 1], dmax[i:i + 1])
        inc = m.extract_pcd()
        ref = copy.deepcopy(m.model)
        set_flavour(ref, 3.0, 0.0)
        full = ref.extract_point_cloud()
        seen = max(seen, int(full.points.shape[0]))
        for a, b in ((inc.points, full.points), (inc.normals, full.normals), (inc.colors, full.colors), (inc.point_keys, full.point_keys)):
            assert torch.equal(a, b)
    assert seen > 100
