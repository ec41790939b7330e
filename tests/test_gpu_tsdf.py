"""K3 parity: CUDA TSDF integration (through the C ABI) vs the CPU oracle -- `-m gpu`.

Bar (BASELINE.json north_star): bit-exact updated-voxel sets / weights / per-frame update
counts; tsdf within 1e-4 * sdf_trunc (asserted exactly equal here, since kernel and oracle
share the float32 operation order)."""
import copy

import numpy as np
import pytest
import torch

import oracle
from bodyslam_b200 import _lib
from bodyslam_b200.geometry import RGBDImage
from bodyslam_b200.tsdf import TSDF, DenseTSDFVolume
from util import small_scene

pytestmark = pytest.mark.gpu


def run_oracle(sc, frames=None, z_restart=8, color=False, dims=None, gz0=0, z_total=None):
    dims = dims or (sc["resolution"],) * 3
    V = oracle.o3d.Volume(dims, sc["voxel_length"], sc["sdf_trunc"], sc["origin"], gz0=gz0, with_color=color)
    counts = []
    for i in (range(len(sc["E"])) if frames is None else frames):
        d = oracle.o3d.depth_from_u16(sc["depth_u16"][i])
        counts.append(V.integrate(d, sc["K"], sc["E"][i], rgb=sc["color"][i] if color else None, z_restart=z_restart))
    return V, np.array(counts)


def run_gpu(sc, cuda, zmarch=_lib.ZMARCH_BRICK, color=False, dims=None, gz0=0, z_total=None, batch=True):
    dims = dims or (sc["resolution"],) * 3
    vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], dims, sc["origin"], color=color, device=cuda, gz0=gz0, z_total=z_total)
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    col = torch.from_numpy(sc["color"]).to(cuda) if color else None
    counts = torch.zeros(len(sc["E"]), dtype=torch.int64, device=cuda)
    if batch:
        vol.integrate_batch(depth, col, sc["intrinsic"], sc["E"], zmarch=zmarch, update_counts=counts)
    else:
        for i in range(len(sc["E"])):
            vol.integrate(RGBDImage(None if col is None else col[i], depth[i]), sc["intrinsic"], sc["E"][i], zmarch=zmarch)
    return vol, counts.cpu().numpy()


def assert_volume_equal(vol, V, trunc, color=False):
    out = vol.export_dense(with_color=color)
    t, w = out[0].cpu().numpy(), out[1].cpu().numpy()
    assert np.array_equal(w, V.grid("weight")), "weights / occupancy differ"
    assert np.array_equal(w != 0, V.grid("weight") != 0)
    dt = np.abs(t - V.grid("tsdf")).max()
    assert dt <= 1e-4 * trunc, f"tsdf differs by {dt}"
    assert np.array_equal(t, V.grid("tsdf")), f"tsdf not bit-exact (max diff {dt})"
    if color:
        c = out[2].cpu().numpy()
        ref = V.color.reshape(c.shape)
        assert np.array_equal(c, ref), f"colour not bit-exact (max diff {np.abs(c - ref).max()})"


@pytest.mark.parametrize("scene,res", [("laparoscopy512", 128), ("colonoscopy256", 64)])
def test_integrate_batch_matches_oracle(cuda, scene, res):
    sc = small_scene(scene, res=res, frames=6)
    V, oc = run_oracle(sc)
    vol, gc = run_gpu(sc, cuda)
    assert oc.sum() > 1000
    assert np.array_equal(gc, oc), f"per-frame update counts differ: {gc} vs {oc}"
    assert_volume_equal(vol, V, sc["sdf_trunc"])
    assert V.occupied() == int((vol.export_dense()[1] != 0).sum().item())


def test_reference_literal_truncation_ratio(cuda):
    """the reference's literal parameters ratio: sdf_trunc = 100 voxels (tsdf.py:6)"""
    sc = small_scene("colonoscopy256", res=64, frames=4)
    sc["sdf_trunc"] = 100 * sc["voxel_length"]
    V, oc = run_oracle(sc)
    vol, gc = run_gpu(sc, cuda)
    assert np.array_equal(gc, oc)
    assert_volume_equal(vol, V, sc["sdf_trunc"])


def test_single_frame_calls_equal_batch(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=5)
    a, _ = run_gpu(sc, cuda, batch=True)
    b, _ = run_gpu(sc, cuda, batch=False)
    for x, y in zip(a.export_dense(), b.export_dense()):
        assert torch.equal(x, y)


def test_literal_zmarch_matches_open3d_literal_oracle(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=4)
    V, oc = run_oracle(sc, z_restart=0)
    vol, gc = run_gpu(sc, cuda, zmarch=_lib.ZMARCH_LITERAL)
    assert np.array_equal(gc, oc)
    assert_volume_equal(vol, V, sc["sdf_trunc"])


def test_brick_restart_deviation_from_literal_is_small(cuda):
    """the fast path restarts the float32 z recurrence every 8 voxels; quantify what that changes"""
    sc = small_scene("laparoscopy512", res=128, frames=6)
    lit, _ = run_gpu(sc, cuda, zmarch=_lib.ZMARCH_LITERAL)
    brk, _ = run_gpu(sc, cuda, zmarch=_lib.ZMARCH_BRICK)
    (tl, wl), (tb, wb) = lit.export_dense(), brk.export_dense()
    flips = int((wl != wb).sum().item())
    occupied = int((wl != 0).sum().item())
    same = wl == wb
    dt = (tl - tb)[same].abs()
    moved = int((dt > 1e-4).sum().item())
    print(f"literal vs brick-restart: {flips} weight flips, {moved} tsdf moves > 1e-4 of {occupied} occupied voxels, "
          f"max |dtsdf| {float(dt.max().item()):.4f}")
    # a few ulp of difference in the projected pixel only matters where (int)u_f flips at a pixel
    # border; those voxels see a neighbouring depth sample
    assert flips <= max(10, 2e-4 * occupied), f"{flips} of {occupied} voxels changed weight"
    assert moved <= max(10, 1e-3 * occupied), f"{moved} of {occupied} voxels changed tsdf"
    assert float(dt.mean().item()) <= 1e-5


def test_ragged_resolution_and_color(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=4)
    dims = (60, 52, 44)
    V, oc = run_oracle(sc, color=True, dims=dims)
    vol, gc = run_gpu(sc, cuda, color=True, dims=dims)
    assert np.array_equal(gc, oc)
    assert_volume_equal(vol, V, sc["sdf_trunc"], color=True)


def test_z_slab_equals_slice_of_full_volume(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=4)
    full, _ = run_gpu(sc, cuda)
    tf, wf = full.export_dense()
    for gz0 in (0, 32):
        slab, _ = run_gpu(sc, cuda, dims=(64, 64, 32), gz0=gz0, z_total=64)
        ts, ws = slab.export_dense()
        assert torch.equal(ws, wf[:, :, gz0:gz0 + 32])
        assert torch.equal(ts, tf[:, :, gz0:gz0 + 32])
    # and against the oracle's slab mode
    V, _ = run_oracle(sc, dims=(64, 64, 32), gz0=32)
    assert np.array_equal(ws.cpu().numpy(), V.grid("weight"))


def test_long_batch_chunking(cuda):
    """F > BSLAM_MAX_BATCH: 300 small frames in one call == frame-by-frame oracle"""
    sc = small_scene("colonoscopy256", res=32, frames=300, W=160, H=120, with_color=False)
    V, oc = run_oracle(sc)
    vol, gc = run_gpu(sc, cuda)
    assert np.array_equal(gc, oc)
    assert_volume_equal(vol, V, sc["sdf_trunc"])
    assert float(vol.export_dense()[1].max().item()) > 50


def test_dry_run_counts_leave_volume_untouched(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=3)
    vol, gc = run_gpu(sc, cuda)
    before = [x.clone() for x in vol.export_dense()]
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    c = vol.count_updates(depth, sc["intrinsic"], sc["E"]).cpu().numpy()
    assert np.array_equal(c, gc)
    for x, y in zip(before, vol.export_dense()):
        assert torch.equal(x, y)


def test_tsdf_dropin_api_and_errors(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=2)
    tsdf = TSDF(voxel_length=sc["voxel_length"], sdf_trunc=sc["sdf_trunc"], resolution=64, origin=sc["origin"], device=cuda,
                unit_activation=False)
    rgbd = RGBDImage.create_from_color_and_depth(sc["color"][0], sc["depth_u16"][0], depth_scale=1000, depth_trunc=3.0,
                                                 convert_rgb_to_intensity=False)
    tsdf.build_3D_map(rgbd, sc["intrinsic"], sc["E"][0])
    w0 = tsdf.tsdf.export_dense()[1].clone()
    cp = tsdf.build_copy_3D_map(rgbd, sc["intrinsic"], sc["E"][0])
    assert torch.equal(tsdf.tsdf.export_dense()[1], w0), "build_copy_3D_map must not touch the original"
    assert float(cp.export_dense()[1].max().item()) == 2.0
    V = oracle.o3d.Volume(64, sc["voxel_length"], sc["sdf_trunc"], sc["origin"], with_color=True)
    V.integrate(oracle.o3d.depth_from_u16(sc["depth_u16"][0]), sc["K"], sc["E"][0], rgb=sc["color"][0])
    assert np.array_equal(w0.cpu().numpy(), V.grid("weight"))
    # Open3D raises RuntimeError on size / dtype mismatch
    bad = RGBDImage(sc["color"][0][:100], rgbd.depth[:100])
    with pytest.raises(RuntimeError, match="Unsupported image format"):
        tsdf.build_3D_map(bad, sc["intrinsic"], sc["E"][0])
    with pytest.raises(RuntimeError, match="Unsupported image format"):
        tsdf.build_3D_map(RGBDImage(sc["color"][0], sc["depth_u16"][0]), sc["intrinsic"], sc["E"][0])
    # empty frame (all invalid) is a no-op
    z = RGBDImage(sc["color"][0], np.zeros((sc["H"], sc["W"]), np.float32))
    tsdf.build_3D_map(z, sc["intrinsic"], sc["E"][0])
    assert torch.equal(tsdf.tsdf.export_dense()[1], w0)


def test_device_arithmetic_selftest(cuda):
    """the kernels' shared-reciprocal division and magic-number floor equal IEEE `/` and (int) casts"""
    import ctypes
    from bodyslam_b200 import _lib as L
    bad = ctypes.c_ulonglong(123)
    with torch.cuda.device(cuda):
        L.check(L.load().bslam_selftest(200_000_000, 1234, ctypes.byref(bad), L.stream_ptr(cuda)))
    assert bad.value == 0, f"{bad.value} mismatches against IEEE division / integer conversion"


def test_batch_size_does_not_change_results(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=12)
    ref, rc = run_gpu(sc, cuda)
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    for batch in (1, 5):
        vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 64, sc["origin"], color=False, device=cuda)
        vol.set_batch(batch)
        vol.integrate_batch(depth, None, sc["intrinsic"], sc["E"])
        for x, y in zip(ref.export_dense(), vol.export_dense()):
            assert torch.equal(x, y)


def test_rgbd_loader_and_update_map_after_pg_from_png_files(cuda, tmp_path):
    """a4 + a11 through the reference's file-based entry points (slam_utils.py:124-135,172-264)"""
    import cv2
    from bodyslam_b200.slam_utils import RGBD, update_map_after_pg
    sc = small_scene("laparoscopy512", res=64, frames=5)
    rgb_paths, depth_paths = [], []
    for i in range(5):
        rp, dp = str(tmp_path / f"rgb_{i}.png"), str(tmp_path / f"depth_{i}.png")
        cv2.imwrite(rp, sc["color"][i][:, :, ::-1])
        cv2.imwrite(dp, sc["depth_u16"][i])
        rgb_paths.append(rp); depth_paths.append(dp)
    fr = RGBD(rgb_paths[0], depth_paths[0], device="CUDA:0", depth_scale=1000, depth_trunc=3.0)
    ref_d = oracle.o3d.depth_from_u16(sc["depth_u16"][0])
    assert (fr.height, fr.width) == (sc["H"], sc["W"])
    assert np.array_equal(fr.rgbd_tsdf.depth.cpu().numpy(), ref_d)
    assert np.array_equal(fr.rgbd_tsdf.color.cpu().numpy(), sc["color"][0])
    cvd = sc["depth_u16"][0].astype(np.float32) / 1000
    assert np.array_equal(fr.cv2_depth.cpu().numpy(), cvd) and fr.depth_min == float(cvd.min()) and fr.depth_max == float(cvd.max())
    jet = cv2.applyColorMap(oracle.mdem.minmax_u8(sc["depth_u16"][0]), cv2.COLORMAP_JET)
    assert np.array_equal(fr.colored_depth.cpu().numpy(), jet)
    tsdf = update_map_after_pg(list(sc["E"]), rgb_paths, depth_paths, 1000, "CUDA:0", sc["intrinsic"],
                               voxel_length=sc["voxel_length"], sdf_trunc=sc["sdf_trunc"], resolution=64, origin=sc["origin"],
                               unit_activation=False)
    V, _ = run_oracle(sc, color=True)
    assert_volume_equal(tsdf.tsdf, V, sc["sdf_trunc"], color=True)
    # frame-by-frame through the drop-in classes gives the same map
    t2 = TSDF(voxel_length=sc["voxel_length"], sdf_trunc=sc["sdf_trunc"], resolution=64, origin=sc["origin"], device=cuda,
              unit_activation=False)
    for i in range(5):
        t2.build_3D_map(RGBD(rgb_paths[i], depth_paths[i], "CUDA:0").rgbd_tsdf, sc["intrinsic"], sc["E"][i])
    for x, y in zip(tsdf.tsdf.export_dense(True), t2.tsdf.export_dense(True)):
        assert torch.equal(x, y)
    pcd = t2.extract_pcd()
    mesh = t2.extract_mesh()
    assert pcd.points.shape[0] > 100 and mesh.triangles.shape[0] > 100 and mesh.vertex_colors is not None
    t2.save_mesh(str(tmp_path / "m.ply")); t2.save_pcd(str(tmp_path / "p.ply"))
    from bodyslam_b200.io import read_ply
    v, f = read_ply(str(tmp_path / "m.ply"))
    assert len(v) == mesh.vertices.shape[0] and len(f) == mesh.triangles.shape[0]


def test_fused_u16_integrate_equals_a4_then_integrate(cuda):
    """bslam_tsdf_integrate_u16 (a4 fused into the first pass) == bslam_depth_from_u16 + bslam_tsdf_integrate,
    bit for bit, and its scratch holds exactly the a4 output; also against the oracle."""
    from bodyslam_b200 import ops
    sc = small_scene("laparoscopy512", res=96, frames=5, with_color=False)
    a, ca = run_gpu(sc, cuda)
    b = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 96, sc["origin"], color=False, device=cuda)
    cb = torch.zeros(5, dtype=torch.int64, device=cuda)
    scratch = b.integrate_u16_batch(torch.from_numpy(sc["depth_u16"]).to(cuda), None, sc["intrinsic"], sc["E"], 1000.0, 3.0, update_counts=cb)
    assert torch.equal(scratch, ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda))
    ta, wa = a.export_dense()
    tb, wb = b.export_dense()
    assert torch.equal(ta, tb) and torch.equal(wa, wb)
    assert np.array_equal(ca, cb.cpu().numpy())
    V, co = run_oracle(sc)
    assert np.array_equal(co, cb.cpu().numpy())
    assert_volume_equal(b, V, sc["sdf_trunc"])


@pytest.mark.parametrize("W,H", [(600, 480), (333, 201)])
def test_fused_u16_integrate_odd_image_sizes(cuda, W, H):
    """widths that are not a multiple of 4 / 16 take the scalar path of the fused conversion"""
    sc = small_scene("laparoscopy512", res=64, frames=3, W=W, H=H, with_color=False)
    vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 64, sc["origin"], color=False, device=cuda)
    counts = torch.zeros(3, dtype=torch.int64, device=cuda)
    vol.integrate_u16_batch(torch.from_numpy(sc["depth_u16"]).to(cuda), None, sc["intrinsic"], sc["E"], update_counts=counts)
    V, co = run_oracle(sc)
    assert np.array_equal(co, counts.cpu().numpy())
    assert_volume_equal(vol, V, sc["sdf_trunc"])


def test_integrate_host_ramped_chunks_equal_one_batch(cuda):
    """streamed host frames (ramp of small chunks first) == one resident batch; counts per frame too"""
    sc = small_scene("laparoscopy512", res=64, frames=40, with_color=False, frame_ids=np.arange(0, 1000, 25))
    a, ca = run_gpu(sc, cuda)
    b = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 64, sc["origin"], color=False, device=cuda)
    cb = torch.zeros(40, dtype=torch.int64, device=cuda)
    host = torch.from_numpy(sc["depth_u16"]).pin_memory()
    b.integrate_host(host, None, sc["intrinsic"], sc["E"], chunk=8, update_counts=cb)   # chunks: ramp disabled above chunk, 5 x 8
    c = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 64, sc["origin"], color=False, device=cuda)
    for f0, f1 in [(0, 3), (3, 10), (10, 40)]:
        c.integrate_u16_batch(torch.from_numpy(sc["depth_u16"][f0:f1]).to(cuda), None, sc["intrinsic"], sc["E"][f0:f1])
    for v in (b, c):
        assert torch.equal(a.export_dense()[0], v.export_dense()[0]) and torch.equal(a.export_dense()[1], v.export_dense()[1])
    assert np.array_equal(ca, cb.cpu().numpy())


@pytest.mark.parametrize("zpw", [8, 4, 2])
def test_z_split_variants_are_bit_identical(cuda, zpw):
    """a brick's 8 layers shared by 2, 4 or 8 warps (bslam_tsdf_set_z_split): same volume, same counts,
    ragged box (nz not a multiple of 8) and colour included"""
    sc = small_scene("laparoscopy512", res=72, frames=5)
    dims = (72, 70, 68)
    vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], dims, sc["origin"], color=True, device=cuda)
    vol.set_z_split(zpw)
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    counts = torch.zeros(5, dtype=torch.int64, device=cuda)
    vol.integrate_batch(depth, torch.from_numpy(sc["color"]).to(cuda), sc["intrinsic"], sc["E"], update_counts=counts)
    V, co = run_oracle(sc, color=True, dims=dims)
    assert np.array_equal(co, counts.cpu().numpy())
    assert_volume_equal(vol, V, sc["sdf_trunc"], color=True)
    assert np.array_equal(vol.count_updates(depth, sc["intrinsic"], sc["E"]).cpu().numpy(), co)


@pytest.mark.parametrize("scene,res,trunc_mul", [("laparoscopy512", 128, 1.0), ("laparoscopy512", 128, 8.0), ("colonoscopy256", 64, 1.0)])
def test_unit_activation_matches_scalable_oracle(cuda, scene, res, trunc_mul):
    """ScalableTSDFVolume semantics (what the reference's TSDF() builds, N/3DM/tsdf.py:7-12): per frame only
    the 32^3 units activated by the stride-8 back-projected points +- sdf_trunc are integrated, voxel
    centres evaluated per unit.  Bit-exact against the oracle's restatement (A.3 step 7): activated-voxel
    sets, weights, per-frame counts, tsdf, colour; and different from the dense rule."""
    sc = small_scene(scene, res=res, frames=5)
    trunc = sc["sdf_trunc"] * trunc_mul
    ul = sc["voxel_length"] * 32
    sc["origin"] = np.floor(sc["origin"] / ul + 0.5) * ul        # the box must sit on the world unit grid
    vol = DenseTSDFVolume(sc["voxel_length"], trunc, res, sc["origin"], color=True, device=cuda, unit_activation=True)
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    counts = torch.zeros(5, dtype=torch.int64, device=cuda)
    vol.integrate_batch(depth, torch.from_numpy(sc["color"]).to(cuda), sc["intrinsic"], sc["E"], update_counts=counts)
    V = oracle.o3d.Volume(res, sc["voxel_length"], trunc, sc["origin"], with_color=True)
    D = oracle.o3d.Volume(res, sc["voxel_length"], trunc, sc["origin"])
    co = []
    for i in range(5):
        d = oracle.o3d.depth_from_u16(sc["depth_u16"][i])
        co.append(V.integrate_scalable(d, sc["K"], sc["E"][i], rgb=sc["color"][i]))
        D.integrate(d, sc["K"], sc["E"][i])
    assert counts.cpu().tolist() == co
    assert_volume_equal(vol, V, trunc, color=True)
    assert V.occupied() <= D.occupied() and (scene != "laparoscopy512" or V.occupied() < D.occupied()), \
        "unit activation must leave un-activated space untouched"
    # frame by frame (the SLAM loop) gives the same map as the batch; deepcopy keeps the mode
    t = TSDF(voxel_length=sc["voxel_length"], sdf_trunc=trunc, resolution=res, origin=sc["origin"], device=cuda)
    assert t.tsdf.unit_activation
    for i in range(5):
        t.tsdf = t.build_copy_3D_map(RGBDImage(sc["color"][i], depth[i]), sc["intrinsic"], sc["E"][i])
    for x, y in zip(vol.export_dense(True), t.tsdf.export_dense(True)):
        assert torch.equal(x, y)
    # extraction on the sparse-activated volume equals the oracle's
    mesh, ref = vol.extract_triangle_mesh(), V.extract_mesh()
    from util import canon_mesh
    a = canon_mesh(mesh.vertices.cpu().numpy(), mesh.vertex_keys.cpu().numpy(), mesh.triangles.cpu().numpy(), (res,) * 3)
    b = canon_mesh(ref["vertices"], ref["keys"], ref["triangles"], (res,) * 3)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2])


def test_unit_activation_needs_an_aligned_box(cuda):
    with pytest.raises(RuntimeError, match="whole 32\\^3 units|multiple of the unit length"):
        DenseTSDFVolume(0.004, 0.02, 72, (-0.144,) * 3, color=False, device=cuda, unit_activation=True)
    with pytest.raises(RuntimeError, match="multiple of the unit length"):
        DenseTSDFVolume(0.004, 0.02, 64, (-0.1,) * 3, color=False, device=cuda, unit_activation=True)
    # the drop-in falls back to the dense rule when the box cannot hold whole units
    assert not TSDF(voxel_length=0.004, sdf_trunc=0.02, resolution=72, device=cuda, color=False).tsdf.unit_activation
    assert TSDF(voxel_length=0.004, sdf_trunc=0.02, resolution=64, device=cuda, color=False).tsdf.unit_activation


@pytest.mark.parametrize("scale,trunc", [(1000.0, 3.0), (256.0, 0.0), (999.5, 0.2), (5000.0, 3.0), (3.0, 1000.0)])
def test_fused_depth_conversion_is_ieee_exact_for_any_scale(cuda, scale, trunc):
    """the fused a4 pass divides through a precomputed reciprocal + residual correction only after the
    device has checked all 65 536 quotients for that divisor against IEEE division"""
    from bodyslam_b200 import ops
    g = torch.Generator().manual_seed(int(scale))
    u16 = torch.randint(0, 65536, (2, 48, 64), generator=g, dtype=torch.int32).to(torch.uint16)
    u16[0, 0, :8] = torch.tensor([0, 1, 2, 999, 1000, 65535, 32768, 3000], dtype=torch.int32).to(torch.uint16)
    intr = small_scene("laparoscopy512", res=32, frames=1, W=64, H=48, with_color=False)
    vol = DenseTSDFVolume(intr["voxel_length"], intr["sdf_trunc"], 32, intr["origin"], color=False, device=cuda)
    scratch = vol.integrate_u16_batch(u16.to(cuda), None, intr["intrinsic"], np.stack([intr["E"][0]] * 2), depth_scale=scale, depth_trunc=trunc)
    ref = oracle.o3d.depth_from_u16(u16.numpy(), scale, trunc if trunc > 0 else 1e30)
    assert np.array_equal(scratch.cpu().numpy(), ref)
    assert torch.equal(scratch, ops.depth_from_u16(u16, scale, trunc, cuda))


def test_unit_mode_is_literal_open3d_per_unit_recurrence_on_interleaved_shards(cuda):
    """unit-activation mode restarts the float32 z recurrence at every UNIT base (Open3D's per-unit
    UniformTSDFVolume starts it there): oracle z_restart = 0, zero deviation -- also when the volume is an
    interleaved z-shard (brick layers of one unit live on different ranks) and for every z split"""
    sc = small_scene("laparoscopy512", res=128, frames=5, with_color=False)
    ul = sc["voxel_length"] * 32
    origin = np.floor(sc["origin"] / ul + 0.5) * ul
    V = oracle.o3d.Volume(128, sc["voxel_length"], sc["sdf_trunc"], origin)
    V8 = oracle.o3d.Volume(128, sc["voxel_length"], sc["sdf_trunc"], origin)
    co = []
    for i in range(5):
        d = oracle.o3d.depth_from_u16(sc["depth_u16"][i])
        co.append(V.integrate_scalable(d, sc["K"], sc["E"][i], z_restart=0))
        V8.integrate_scalable(d, sc["K"], sc["E"][i], z_restart=8)
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    for zpw in (8, 4, 2):
        vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 128, origin, color=False, device=cuda, unit_activation=True)
        vol.set_z_split(zpw)
        counts = torch.zeros(5, dtype=torch.int64, device=cuda)
        vol.integrate_batch(depth, None, sc["intrinsic"], sc["E"], update_counts=counts)
        assert counts.cpu().tolist() == co
        assert_volume_equal(vol, V, sc["sdf_trunc"])
    # 4 interleaved shards (rank r owns brick layers r, r + 4, ...): their union equals the literal oracle
    tf, wf = (x.cpu().numpy() for x in vol.export_dense())
    for r in range(4):
        sh = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], (128, 128, 32), origin, color=False, device=cuda, gz0=8 * r, z_total=128,
                             z_interleave=4, unit_activation=True)
        sh.integrate_batch(depth, None, sc["intrinsic"], sc["E"])
        ts, ws = (x.cpu().numpy() for x in sh.export_dense())
        for l in range(4):
            g = (l * 4 + r) * 8
            assert np.array_equal(ws[:, :, l * 8:l * 8 + 8], V.grid("weight")[:, :, g:g + 8])
            assert np.array_equal(ts[:, :, l * 8:l * 8 + 8], V.grid("tsdf")[:, :, g:g + 8])
    assert np.array_equal(wf, V.grid("weight")) and np.array_equal(tf, V.grid("tsdf"))


def test_clip_statistics_and_warning_when_the_scene_leaves_the_box(cuda):
    """the reference's ScalableTSDFVolume is unbounded, the box is not: dropped depth points are counted
    (unit mode and dense mode) and the drop-in warns on extraction"""
    sc = small_scene("laparoscopy512", res=64, frames=3, with_color=False)
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    n_pts = sum(int((oracle.o3d.depth_from_u16(sc["depth_u16"][i])[::8, ::8] > 0).sum()) for i in range(3))
    for unit in (False, True):
        # a 0.256 m cube around the origin: the cavity wall (> 0.2 m away) lies outside
        t = TSDF(voxel_length=0.004, sdf_trunc=0.02, resolution=64, origin=(-0.128,) * 3, device=cuda, color=False, unit_activation=unit)
        assert t.tsdf.unit_activation == unit
        for i in range(3):
            t.build_3D_map(RGBDImage(None, depth[i]), sc["intrinsic"], sc["E"][i])
        st = t.tsdf.clip_stats()
        assert st["points"] == n_pts and st["outside"] > 0.9 * n_pts, st
        with pytest.warns(UserWarning, match="outside the volume box"):
            t.extract_mesh()
        # a box that covers the scene drops nothing and stays silent
        ul = sc["voxel_length"] * 32
        t = TSDF(voxel_length=sc["voxel_length"], sdf_trunc=sc["sdf_trunc"], resolution=64, origin=np.floor(sc["origin"] / ul + 0.5) * ul,
                 device=cuda, color=False, unit_activation=unit)
        for i in range(3):
            t.build_3D_map(RGBDImage(None, depth[i]), sc["intrinsic"], sc["E"][i])
        st = t.tsdf.clip_stats()
        assert st["points"] == n_pts and st["outside"] == 0
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            assert t.extract_mesh().triangles.shape[0] > 0


def test_sharded_front_end_on_one_gpu_equals_the_drop_in(cuda):
    """ShardedTSDF(world_size=1) takes numpy / host / device u16 frames and has TSDF()'s unit-activation default"""
    from bodyslam_b200.sharding import ShardedTSDF
    sc = small_scene("laparoscopy512", res=64, frames=4, with_color=False)
    ul = sc["voxel_length"] * 32
    origin = np.floor(sc["origin"] / ul + 0.5) * ul
    ref = TSDF(voxel_length=sc["voxel_length"], sdf_trunc=sc["sdf_trunc"], resolution=64, origin=origin, device=cuda, color=False)
    assert ref.tsdf.unit_activation
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    for i in range(4):
        ref.build_3D_map(RGBDImage(None, depth[i]), sc["intrinsic"], sc["E"][i])
    for src in (sc["depth_u16"], torch.from_numpy(sc["depth_u16"]), torch.from_numpy(sc["depth_u16"]).to(cuda)):
        sh = ShardedTSDF(sc["voxel_length"], sc["sdf_trunc"], 64, origin, color=False, device=cuda, rank=0, world_size=1)
        assert sh.unit_activation and sh.tsdf.unit_activation
        sh.integrate_stream(src, sc["intrinsic"], sc["E"])
        for x, y in zip(sh.tsdf.export_dense(), ref.tsdf.export_dense()):
            assert torch.equal(x, y)


def test_stage_profile_reports_every_stage(cuda):
    sc = small_scene("laparoscopy512", res=64, frames=4, with_color=False)
    vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 64, sc["origin"], color=False, device=cuda)
    vol.profile(True)
    vol.integrate_u16_batch(torch.from_numpy(sc["depth_u16"]).to(cuda), None, sc["intrinsic"], sc["E"])
    stages, n = vol.profile_read_stages()
    ms, n2 = vol.profile_read()
    assert n == n2 == 1 and set(stages) == {"depth_stats_a4", "marks_culls_order", "brick_integrate"}
    assert all(v > 0 for v in stages.values()) and abs(ms - stages["brick_integrate"]) < 1e-9


@pytest.mark.slow
def test_config1_colonoscopy_256_full_size_values(cuda):
    """BASELINE configs[1] at FULL size: 300 frames, 640x480 -> 256^3 @ 2 mm; tsdf / weight VALUES (not counts)
    bit-exact against the oracle (dense rule, z_restart 8) and against the literal per-unit oracle in
    unit-activation mode; mesh vertex / triangle counts equal"""
    from bodyslam_b200 import synthetic as S
    from bodyslam_b200.geometry import PinholeCameraIntrinsic
    cfg = S.config("colonoscopy256")
    E = cfg["extrinsics"](300)
    depth_u16, _ = S.render(cfg["surface"], E, K=cfg["K"], W=640, H=480, device=cuda, with_color=False)
    intr = PinholeCameraIntrinsic(640, 480, *cfg["K"])
    d_np = depth_u16.cpu().numpy()
    ul = cfg["voxel_length"] * 32
    org_u = np.floor(np.asarray(cfg["origin"]) / ul + 0.5) * ul
    for unit, origin in ((False, np.asarray(cfg["origin"], dtype=np.float64)), (True, org_u)):
        vol = DenseTSDFVolume(cfg["voxel_length"], cfg["sdf_trunc"], 256, origin, color=False, device=cuda, unit_activation=unit)
        counts = torch.zeros(300, dtype=torch.int64, device=cuda)
        vol.integrate_u16_batch(depth_u16, None, intr, E, update_counts=counts)
        V = oracle.o3d.Volume(256, cfg["voxel_length"], cfg["sdf_trunc"], origin)
        co = []
        for i in range(300):
            d = oracle.o3d.depth_from_u16(d_np[i])
            co.append(V.integrate_scalable(d, cfg["K"], E[i]) if unit else V.integrate(d, cfg["K"], E[i]))
        assert counts.cpu().tolist() == co
        assert_volume_equal(vol, V, cfg["sdf_trunc"])
        mesh, ref = vol.extract_triangle_mesh(), V.extract_mesh()
        assert int(mesh.vertices.shape[0]) == len(ref["vertices"]) and int(mesh.triangles.shape[0]) == len(ref["triangles"])
        assert len(ref["triangles"]) > 10000


def test_dense_rule_with_the_references_per_unit_arithmetic(cuda):
    """`unit_arithmetic=True`: every voxel of the box is integrated (north_star's dense volume) but with the voxel centres
    and the float32 z recurrence of ScalableTSDFVolume's 32^3 units -- literal Open3D arithmetic, oracle z_restart = 0 with
    every unit touched; on the units the reference would have activated the values ARE the reference's"""
    sc = small_scene("laparoscopy512", res=128, frames=5)
    ul = sc["voxel_length"] * 32
    origin = np.floor(sc["origin"] / ul + 0.5) * ul
    vol = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], 128, origin, color=True, device=cuda, unit_arithmetic=True)
    from bodyslam_b200 import ops
    depth = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, cuda)
    counts = torch.zeros(5, dtype=torch.int64, device=cuda)
    vol.integrate_batch(depth, torch.from_numpy(sc["color"]).to(cuda), sc["intrinsic"], sc["E"], update_counts=counts)
    A = oracle.o3d.Volume(128, sc["voxel_length"], sc["sdf_trunc"], origin, with_color=True)      # every unit, per-unit arithmetic
    S = oracle.o3d.Volume(128, sc["voxel_length"], sc["sdf_trunc"], origin, with_color=True)      # the reference: activated units only
    co, act = [], np.zeros((4, 4, 4), bool)
    for i in range(5):
        d = oracle.o3d.depth_from_u16(sc["depth_u16"][i])
        co.append(A.integrate_scalable(d, sc["K"], sc["E"][i], rgb=sc["color"][i], all_units=True))
        _, touched = S.integrate_scalable(d, sc["K"], sc["E"][i], rgb=sc["color"][i], return_touched=True)
        act |= touched.astype(bool)
    assert counts.cpu().tolist() == co
    assert_volume_equal(vol, A, sc["sdf_trunc"], color=True)
    # a voxel of a unit that EVERY frame that could update it also activated holds the reference's value; check the
    # units activated by all 5 frames' union where the scalable oracle and the all-units oracle agree on the weights
    t, w = (x.cpu().numpy() for x in vol.export_dense())
    same_w = w == S.grid("weight")
    assert same_w.mean() > 0.5 and np.array_equal(t[same_w], S.grid("tsdf")[same_w])
    # deepcopy keeps the mode
    c2 = copy.deepcopy(vol)
    assert c2.unit_arithmetic and not c2.unit_activation
