"""Multi-scale RGB-D odometry on the GPU (csrc/bslam_odometry.cu) against its CPU reference (tests/odometry_ref.c;
parity with Open3D unpinned): prepared maps bit for bit, the linearisation's sums, full multi-scale runs, the batched
sequence and the `MAP` frame-to-model tracking loop -- `-m gpu`."""
import inspect

import numpy as np
import pytest
import torch

import odometry_ref as R
from bodyslam_b200 import _lib
from bodyslam_b200 import odometry as od
from bodyslam_b200 import synthetic as S
from bodyslam_b200.geometry import RGBDImage
from bodyslam_b200.tsdf import MAP
from test_gpu_map import FakeRGBD, k3x3

pytestmark = pytest.mark.gpu

REF_CRIT = ((10, 1e-6, 1e-6), (5, 1e-6, 1e-6), (3, 1e-6, 1e-6))
METHODS = [od.Method.PointToPlane, od.Method.Intensity, od.Method.Hybrid]


def same_bits(a, b, what=""):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    assert np.array_equal(na, nb), f"{what}: NaN masks differ in {(na != nb).sum()} values"
    diff = a.view(np.uint32)[~na] != b.view(np.uint32)[~nb]
    assert not diff.any(), f"{what}: {diff.sum()} values differ, by up to {np.abs(a[~na] - b[~nb]).max()}"


@pytest.fixture(scope="module")
def scenes():
    """4 consecutive frames of the laparoscopy sweep (cavity) and of the colonoscopy lumen at 640 x 480"""
    lum = S.Lumen()
    out = {}
    for name, surf, E in (("cavity", S.Cavity(), S.cavity_sweep(1000)[:4]), ("lumen", lum, S.lumen_trajectory(lum, 300)[100:112:3])):
        d, c = S.render(surf, E, K=S.K_640)
        out[name] = (d.numpy(), c.numpy(), E)
    return out


def gpu_prepare(depth, color, K, levels, depth_scale=1000.0, depth_max=3.0, trunc=0.07):
    L = _lib.load()
    d = torch.as_tensor(np.ascontiguousarray(depth)).cuda()
    c = None if color is None else torch.as_tensor(np.ascontiguousarray(color)).cuda()
    F, H, W = d.shape
    fb = L.bslam_odom_frame_bytes(H, W, levels)
    buf = torch.empty(max(F * fb // 4, 1), dtype=torch.float32, device="cuda")
    K4 = np.asarray(K, np.float64)
    _lib.check(L.bslam_odom_prepare(_lib.ptr(d), int(d.dtype == torch.float32), _lib.ptr(c), int(c is not None and c.dtype == torch.float32), F, H, W,
                                    levels, _lib.ptr(K4), depth_scale, depth_max, trunc, _lib.ptr(buf), _lib.stream_ptr()))
    return buf[:F * fb // 4].view(F, -1)


def gpu_linearize(buf, pairs, H, W, levels, level, K, method, Ts, params=(0.07, 0.05, 0.1)):
    L = _lib.load()
    P = len(pairs)
    ws = torch.empty(L.bslam_odom_workspace_bytes(P, H, W, levels), dtype=torch.uint8, device="cuda")
    sums = torch.empty((P, 29), dtype=torch.float64, device="cuda")
    hp = np.ascontiguousarray(pairs, np.int32)
    hT = np.ascontiguousarray(Ts, np.float64).reshape(P, 16)
    _lib.check(L.bslam_odom_linearize(_lib.ptr(buf), buf.shape[0], _lib.ptr(hp), P, H, W, levels, level, _lib.ptr(np.asarray(K, np.float64)), int(method),
                                      *params, _lib.ptr(hT), _lib.ptr(sums), _lib.ptr(ws), _lib.stream_ptr()))
    return sums.cpu().numpy()


def ref_frames(depth, color, K, levels, **kw):
    return R.Frames(depth, color, K, levels, **kw)


def check_track(res, ref, what=""):
    assert ref["status"] == 0, what
    assert np.abs(res.transformation - ref["T"]).max() <= 1e-9, (what, np.abs(res.transformation - ref["T"]).max())
    assert abs(res.inlier_rmse - ref["rmse"]) <= 1e-9 * ref["rmse"], what
    assert abs(res.fitness - ref["fitness"]) <= 1e-9 * ref["fitness"], what


# ------------------------------------------------------------------------------------------------ prepared maps
@pytest.mark.parametrize("dtypes", ["u16_u8", "f32_f32"])
def test_prepared_maps_bit_for_bit(scenes, dtypes):
    d, c, _ = scenes["cavity"]
    if dtypes == "f32_f32":        # the ray cast's units: z * depth_scale and colour in [0, 1]
        d = (d.astype(np.float32) * np.float32(1.0003)).astype(np.float32)
        c = c.astype(np.float32) / np.float32(255)
    ref = ref_frames(d, c, S.K_640, 4)
    gpu = gpu_prepare(d, c, S.K_640, 4).cpu().numpy()
    for f in range(d.shape[0]):
        for l in range(4):
            g = R.Frames.__new__(R.Frames)
            g.__dict__.update(ref.__dict__, data=gpu)
            for k, v in ref.planes(f, l).items():
                same_bits(g.planes(f, l)[k], v, f"frame {f} level {l} {k}")


@pytest.mark.parametrize("HW,levels", [((479, 641), 3), ((17, 9), 3), ((8, 8), 3), ((8, 8), 4), ((1, 1), 1)])
def test_prepared_maps_odd_sizes(HW, levels):
    h, w = HW
    rng = np.random.default_rng(h * 1000 + w)
    d = rng.integers(150, 400, size=(2, h, w)).astype(np.uint16)
    d[rng.random(d.shape) < 0.1] = 0
    c = rng.integers(0, 256, size=(2, h, w, 3)).astype(np.uint8)
    K = (0.8 * w, 0.8 * w, w / 2, h / 2)
    same_bits(gpu_prepare(d, c, K, levels, trunc=0.03).cpu().numpy(), ref_frames(d, c, K, levels, depth_outlier_trunc=0.03).data, f"{HW}")
    same_bits(gpu_prepare(d, None, K, levels).cpu().numpy(), ref_frames(d, None, K, levels).data, f"{HW} no colour")


# ------------------------------------------------------------------------------------------------ linearisation
def test_linearize_sums(scenes):
    d, c, E = scenes["cavity"]
    ref = ref_frames(d, c, S.K_640, 3)
    buf = gpu_prepare(d, c, S.K_640, 3)
    pairs = [(0, 1), (1, 2), (2, 3), (3, 0), (1, 1)]
    Ts = [E[b] @ np.linalg.inv(E[a]) for a, b in pairs]
    Ts[0] = np.eye(4)
    for method in METHODS:
        for level in range(3):
            g = gpu_linearize(buf, pairs, 480, 640, 3, level, S.K_640, method, Ts)
            for p, (a, b) in enumerate(pairs):
                r = ref.linearize(a, b, level, Ts[p], int(method))
                assert g[p, 28] == r[28] and r[28] > 1000, (method, level, p)
                assert np.all(np.abs(g[p, :28] - r[:28]) <= 1e-10 * np.abs(r[:28]).max()), (method, level, p)
            again = gpu_linearize(buf, pairs, 480, 640, 3, level, S.K_640, method, Ts)
            assert np.array_equal(g.view(np.uint64), again.view(np.uint64))
            # a pair's sums do not depend on the other pairs of the launch
            alone = gpu_linearize(buf, pairs[2:3], 480, 640, 3, level, S.K_640, method, Ts[2:3])
            assert np.array_equal(alone[0].view(np.uint64), g[2].view(np.uint64))


# ------------------------------------------------------------------------------------------------ full runs
@pytest.mark.parametrize("name", ["cavity", "lumen"])
@pytest.mark.parametrize("method", METHODS)
def test_multi_scale_matches_reference(scenes, name, method):
    d, c, E = scenes[name]
    ref = ref_frames(d, c, S.K_640, 3)
    K3 = k3x3(S.K_640)
    for a, b in ((0, 1), (1, 2), (2, 3)):
        r = ref.track(a, b, int(method), REF_CRIT)
        if r["status"]:                       # point-to-plane on the lumen (see test_oracle_odometry)
            with pytest.raises(RuntimeError, match="Singular 6x6 linear system detected, tracking failed."):
                od.rgbd_odometry_multi_scale(RGBDImage(c[a], d[a]), RGBDImage(c[b], d[b]), K3, method=method)
            continue
        res = od.rgbd_odometry_multi_scale(RGBDImage(c[a], d[a]), RGBDImage(torch.as_tensor(c[b]).cuda(), torch.as_tensor(d[b]).cuda()), K3,
                                           method=method)
        check_track(res, r, f"{name} {method.name} {a}->{b}")
        seq = od.rgbd_odometry_sequence(d[a:b + 1], c[a:b + 1], K3, method=method)
        assert seq.iterations.cpu().numpy().tolist() == [list(r["iters"])]


def test_edge_shapes_and_criteria(scenes):
    d, c, E = scenes["cavity"]
    K3 = k3x3(S.K_640)
    ref = ref_frames(d, c, S.K_640, 4)
    crit4 = ((4, 1e-6, 1e-6), (3, 1e-6, 1e-6), (0, 1e-6, 1e-6), (2, 1e-6, 1e-6))
    for method in METHODS:
        r = ref.track(0, 1, int(method), crit4)
        res = od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), K3, method=method,
                                           criteria_list=[od.OdometryConvergenceCriteria(m, rr, rf) for m, rr, rf in crit4])
        check_track(res, r, f"4 levels {method.name}")
        one = ref_frames(d, c, S.K_640, 1).track(0, 1, int(method), ((7, 1e-6, 1e-6),))
        check_track(od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), K3, method=method,
                                                 criteria_list=[od.OdometryConvergenceCriteria(7)]), one, f"1 level {method.name}")
    # every max_iteration 0: the init comes back
    init = E[1] @ np.linalg.inv(E[0])
    res = od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), K3, init, criteria_list=[od.OdometryConvergenceCriteria(0)] * 2)
    assert np.array_equal(res.transformation, init) and res.fitness == 0.0
    # float32 depth and colour: the ray cast's units
    df, cf = d.astype(np.float32), c.astype(np.float32) / np.float32(255)
    r = ref_frames(df, cf, S.K_640, 3).track(0, 1, int(od.Method.Hybrid), REF_CRIT)
    check_track(od.rgbd_odometry_multi_scale(RGBDImage(cf[0], df[0]), RGBDImage(cf[1], df[1]), K3), r, "float32 inputs")
    # all-invalid source and depth_max cutting everything: singular
    with pytest.raises(RuntimeError, match="Singular 6x6"):
        od.rgbd_odometry_multi_scale(RGBDImage(c[0], np.zeros_like(d[0])), RGBDImage(c[1], d[1]), K3)
    with pytest.raises(RuntimeError, match="Singular 6x6"):
        od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), K3, depth_max=0.01)
    with pytest.raises(RuntimeError, match="needs the colour"):
        od.rgbd_odometry_multi_scale(RGBDImage(None, d[0]), RGBDImage(None, d[1]), K3)


@pytest.mark.parametrize("HW", [(479, 641), (17, 9), (8, 8)])
def test_odd_sizes_match_reference(HW):
    h, w = HW
    lum = S.Lumen()
    E = S.lumen_trajectory(lum, 300)[[50, 51]]
    K = (S.K_640[0] * w / 640, S.K_640[1] * h / 480, S.K_640[2] * w / 640, S.K_640[3] * h / 480)
    d, c = (x.numpy() for x in S.render(lum, E, K=K, W=w, H=h, invalid_frac=0.0))
    ref = ref_frames(d, c, K, 3)
    for method in METHODS:
        crit = ((3, 1e-6, 1e-6), (2, 1e-6, 1e-6), (2, 1e-6, 1e-6))
        r = ref.track(0, 1, int(method), crit)
        kw = dict(method=method, criteria_list=[od.OdometryConvergenceCriteria(m) for m, _, _ in crit])
        if r["status"]:
            with pytest.raises(RuntimeError, match="Singular"):
                od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), k3x3(K), **kw)
        else:
            check_track(od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), k3x3(K), **kw), r, f"{HW} {method.name}")
    if HW == (8, 8):
        with pytest.raises(RuntimeError, match="Unsupported image format"):
            od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), k3x3(K), criteria_list=[od.OdometryConvergenceCriteria(1)] * 5)


# ------------------------------------------------------------------------------------------------ sequences
@pytest.mark.parametrize("F", [0, 1, 2, 130])
def test_sequence_equals_single_calls(F):
    w, h = 80, 60
    K = (S.K_640[0] / 8, S.K_640[1] / 8, S.K_640[2] / 8, S.K_640[3] / 8)
    E = S.cavity_sweep(1000)[:max(F, 1)][:F]
    d, c = S.render(S.Cavity(), E, K=K, W=w, H=h) if F else (torch.zeros((0, h, w), dtype=torch.uint16), torch.zeros((0, h, w, 3), dtype=torch.uint8))
    crit = [od.OdometryConvergenceCriteria(4), od.OdometryConvergenceCriteria(3)]
    seq = od.rgbd_odometry_sequence(d, c, k3x3(K), criteria_list=crit)
    assert seq.transformations.shape == (max(F - 1, 0), 4, 4) and seq.iterations.shape == (max(F - 1, 0), 2)
    T = seq.transformations.cpu().numpy()
    rmse, fit = seq.inlier_rmse.cpu().numpy(), seq.fitness.cpu().numpy()
    assert not seq.status.any()
    for i in range(F - 1):
        one = od.rgbd_odometry_multi_scale(RGBDImage(c[i], d[i]), RGBDImage(c[i + 1], d[i + 1]), k3x3(K), criteria_list=crit)
        assert np.array_equal(one.transformation, T[i]) and one.inlier_rmse == rmse[i] and one.fitness == fit[i], i
    if F == 130:           # and the reference, on a few pairs across the chunk seams
        ref = ref_frames(d.numpy(), c.numpy(), K, 2)
        for i in (0, 62, 63, 64, 126, 128):
            r = ref.track(i, i + 1, int(od.Method.Hybrid), ((4, 1e-6, 1e-6), (3, 1e-6, 1e-6)))
            assert np.abs(T[i] - r["T"]).max() <= 1e-9 and list(seq.iterations[i].cpu().numpy()) == list(r["iters"])


@pytest.mark.parametrize("method", METHODS)
def test_converged_and_running_pairs_share_launches(method):
    """loose criteria: some pairs stop early at the coarse level and then run the next one, some stop early at the fine
    level, some run every iteration -- all in one bslam_odom_track call, each equal to the reference"""
    w, h = 80, 60
    K = (S.K_640[0] / 8, S.K_640[1] / 8, S.K_640[2] / 8, S.K_640[3] / 8)
    d, c = (x.numpy() for x in S.render(S.Cavity(), S.cavity_sweep(1000)[:40], K=K, W=w, H=h))
    crit = ((6, 1e-2, 1e-2), (6, 1e-2, 1e-2))
    seq = od.rgbd_odometry_sequence(d, c, k3x3(K), method=method, criteria_list=[od.OdometryConvergenceCriteria(*x) for x in crit])
    ref = ref_frames(d, c, K, 2)
    refs = [ref.track(i, i + 1, int(method), crit) for i in range(39)]
    its = np.array([r["iters"] for r in refs])
    assert (its == 6).all(axis=1).any()
    assert ((its[:, 0] == 6) & (its[:, 1] < 6)).any()
    assert ((its[:, 0] < 6) & (its[:, 1] > 0)).any()
    assert np.array_equal(seq.iterations.cpu().numpy(), its)
    assert not seq.status.any()
    T, rmse, fit = seq.transformations.cpu().numpy(), seq.inlier_rmse.cpu().numpy(), seq.fitness.cpu().numpy()
    for i, r in enumerate(refs):
        check_track(od.OdometryResult(T[i], float(rmse[i]), float(fit[i])), r, f"pair {i}")
    # criteria every change meets: a level stops after its second iteration, since its first has no previous fitness
    # (a previous fitness carried over from the coarser level would stop the finer one after one)
    loose = ((6, 1e3, 1e3), (6, 1e3, 1e3))
    seq = od.rgbd_odometry_sequence(d, c, k3x3(K), method=method, criteria_list=[od.OdometryConvergenceCriteria(*x) for x in loose])
    its = np.array([ref.track(i, i + 1, int(method), loose)["iters"] for i in range(39)])
    assert (its == 2).all() and np.array_equal(seq.iterations.cpu().numpy(), its)


def test_c_abi_outputs_inside_guard_bands(scenes):
    d, c, E = scenes["cavity"]
    L = _lib.load()
    buf = gpu_prepare(d, c, S.K_640, 3)
    P, G = 3, 64
    pairs = np.array([[0, 1], [1, 2], [2, 3]], np.int32)
    init = np.tile(np.eye(4).reshape(1, 16), (P, 1))
    mi = np.array([3, 2, 1], np.int32)
    rel = np.full(3, 1e-6)
    bands = {k: torch.full((n + 2 * G,), float("nan"), dtype=torch.float64, device="cuda") for k, n in (("T", P * 16), ("rf", P * 2))}
    ints = {k: torch.full((n + 2 * G,), -7, dtype=torch.int32, device="cuda") for k, n in (("it", P * 3), ("st", P))}
    ws = torch.empty(L.bslam_odom_workspace_bytes(P, 480, 640, 3), dtype=torch.uint8, device="cuda")
    _lib.check(L.bslam_odom_track(_lib.ptr(buf), 4, _lib.ptr(pairs), P, 480, 640, 3, _lib.ptr(np.asarray(S.K_640, np.float64)), 2, _lib.ptr(mi),
                                  _lib.ptr(rel), _lib.ptr(rel), 0.07, 0.05, 0.1, _lib.ptr(init), _lib.ptr(bands["T"][G:]), _lib.ptr(bands["rf"][G:]),
                                  _lib.ptr(ints["it"][G:]), _lib.ptr(ints["st"][G:]), _lib.ptr(ws), _lib.stream_ptr()))
    for k, t in bands.items():
        t = t.cpu().numpy()
        assert np.isnan(t[:G]).all() and np.isnan(t[-G:]).all() and not np.isnan(t[G:-G]).any(), k
    for k, t in ints.items():
        t = t.cpu().numpy()
        assert (t[:G] == -7).all() and (t[-G:] == -7).all() and (t[G:-G] >= 0).all(), k
    # F = 0 / P = 0: nothing launched, NULL outputs accepted
    _lib.check(L.bslam_odom_track(None, 0, None, 0, 480, 640, 3, _lib.ptr(np.asarray(S.K_640, np.float64)), 2, _lib.ptr(mi), _lib.ptr(rel), _lib.ptr(rel),
                                  0.07, 0.05, 0.1, None, None, None, None, None, None, _lib.stream_ptr()))
    sums = torch.full((2 * G + 29,), float("nan"), dtype=torch.float64, device="cuda")
    _lib.check(L.bslam_odom_linearize(_lib.ptr(buf), 4, _lib.ptr(pairs[:1]), 1, 480, 640, 3, 0, _lib.ptr(np.asarray(S.K_640, np.float64)), 0, 0.07, 0.05,
                                      0.1, _lib.ptr(init[:1]), _lib.ptr(sums[G:]), _lib.ptr(ws), _lib.stream_ptr()))
    s = sums.cpu().numpy()
    assert np.isnan(s[:G]).all() and np.isnan(s[-G:]).all() and not np.isnan(s[G:-G]).any()


# ------------------------------------------------------------------------------------------------ MAP tracking loop
# drift of the tracked camera centre from the ground truth at the last of the 60 frames: 0.0885 m measured on a B200.
# The target (the ray cast) is smooth; the input frame's millimetre steps bias the residuals, and seen from inside the
# near-spherical cavity the rotations are weakly constrained (test_oracle_odometry::test_point_to_plane_error_source).
DRIFT_BAR_M = 0.1


def test_map_tracking_loop_matches_reference():
    K = S.K_640
    E = S.cavity_sweep(1000)[:60]
    d, c = (x.numpy() for x in S.render(S.Cavity(), E, K=K))
    m = MAP(640, 480, k3x3(K), "CUDA:0", 1000.0, voxel_size=0.002, resolution=256)
    T = np.linalg.inv(E[0])
    for i in range(60):
        fr = FakeRGBD(d[i], c[i], 1000.0)
        if i > 0:
            mf = m.synthesize_model_frame()
            res = m.track_frame_to_model(fr, mf)
            src = ref_frames(d[i], None, K, 3)
            tgt = ref_frames(mf["depth"][0].cpu().numpy(), None, K, 3)
            src.data = np.concatenate([src.data, tgt.data])
            r = src.track(0, 1, int(od.Method.PointToPlane), ((6, 1e-6, 1e-6), (3, 1e-6, 1e-6), (1, 1e-6, 1e-6)))
            check_track(res, r, f"step {i}")
            T = T @ res.transformation
        m.integrate(fr, i, T)
    drift = np.linalg.norm(T[:3, 3] - np.linalg.inv(E[-1])[:3, 3])
    print(f"MAP tracking drift after 60 frames: {drift:.6f} m")
    assert drift <= DRIFT_BAR_M, drift


def test_signatures():
    sig = inspect.signature(od.rgbd_odometry_multi_scale)
    assert list(sig.parameters) == ["source", "target", "intrinsics", "init_source_to_target", "depth_scale", "depth_max", "criteria_list", "method",
                                    "params"]
    assert sig.parameters["depth_scale"].default == 1000.0 and sig.parameters["depth_max"].default == 3.0
    assert np.array_equal(sig.parameters["init_source_to_target"].default, np.eye(4))
    assert [c.max_iteration for c in sig.parameters["criteria_list"].default] == [10, 5, 3]
    assert sig.parameters["method"].default == od.Method.Hybrid
    assert od.OdometryLossParams() == od.OdometryLossParams(0.07, 0.05, 0.1)
    assert od.OdometryConvergenceCriteria(3) == od.OdometryConvergenceCriteria(3, 1e-6, 1e-6)
    t = inspect.signature(MAP.track_frame_to_model)
    assert list(t.parameters)[1:] == ["input_rgbd", "model_frame", "depth_scale", "depth_max", "depth_diff", "method", "criteria"]
    assert t.parameters["method"].default == od.Method.PointToPlane and t.parameters["criteria"].default == (6, 3, 1)
    assert t.parameters["depth_diff"].default == 0.07 and t.parameters["depth_max"].default == 3.0
    s = inspect.signature(od.rgbd_odometry_sequence)
    assert list(s.parameters)[:4] == ["depth", "color", "intrinsics", "inits"]
