"""The RGB-D odometry (csrc/bslam_odometry.cu) at the edges its parity tests (test_gpu_odometry.py) skip: both branches of
the Huber terms, the projection rules at exact borders, pair batches across the 128-pair init launches up to the
65 535-pair limit, singular pairs inside shared launches, per-pair sequence inits across the 64-frame chunks, unusual
preparation inputs, reduce tiles at 1024-pixel seams and a 1080p frame, `MAP.track_frame_to_model` with colour, and a
second device -- `-m gpu`.  The reference is the CPU mirror tests/odometry_ref.c, and for the linearisation also its
independent float64 restatement `odometry_ref.linearize_f64`."""
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
from test_gpu_odometry import METHODS, REF_CRIT, check_track, gpu_linearize, gpu_prepare, same_bits

pytestmark = pytest.mark.gpu

# (depth_outlier_trunc, depth_huber_delta, intensity_huber_delta): the defaults, a set that puts many inliers in both
# branches, an all-linear and an all-quadratic one (test_oracle_odometry.HUBER_SETS lists the branch coverage of each)
HUBER_SETS = [(0.07, 0.05, 0.1), (0.07, 0.002, 0.01), (0.07, 0.0, 0.0), (0.07, 1e3, 1e3)]
K_80 = tuple(k / 8 for k in S.K_640)                      # 80 x 60


def small_K(w):
    return tuple(k * w / 640 for k in S.K_640)


def check_sums(g, r, what=""):
    """bslam_odom_linearize against ref_odom_linearize: the inlier count exactly, the other sums up to their order"""
    assert g[28] == r[28], (what, g[28], r[28])
    assert np.all(np.abs(g[:28] - r[:28]) <= 1e-10 * max(np.abs(r[:28]).max(), 1e-300)), (what, np.abs(g - r).max())


def gpu_track(buf, F, pairs, H, W, levels, K, method, crit, inits, params=(0.07, 0.05, 0.1), guard=0):
    """bslam_odom_track directly -> dict(T [P,4,4], rf [P,2], iters [P,L], status [P]); guard > 0 puts guard bands of that
    many NaN / -7 values around every output and checks them"""
    L = _lib.load()
    P = len(pairs)
    hp = np.ascontiguousarray(pairs, np.int32).reshape(P, 2)
    hT = np.ascontiguousarray(inits, np.float64).reshape(P, 16)
    mi = np.array([c[0] for c in crit], np.int32)
    rr = np.array([c[1] for c in crit], np.float64)
    rfit = np.array([c[2] for c in crit], np.float64)
    G = guard
    outs = {"T": torch.full((P * 16 + 2 * G,), float("nan"), dtype=torch.float64, device="cuda"),
            "rf": torch.full((P * 2 + 2 * G,), float("nan"), dtype=torch.float64, device="cuda"),
            "iters": torch.full((P * levels + 2 * G,), -7, dtype=torch.int32, device="cuda"),
            "status": torch.full((P + 2 * G,), -7, dtype=torch.int32, device="cuda")}
    # a zeroed workspace: pair state a launch failed to initialise reads as frame 0 under a zero pose (no inlier)
    ws = torch.zeros(L.bslam_odom_workspace_bytes(P, H, W, levels), dtype=torch.uint8, device="cuda")
    _lib.check(L.bslam_odom_track(_lib.ptr(buf), F, _lib.ptr(hp), P, H, W, levels, _lib.ptr(np.asarray(K, np.float64)), int(method), _lib.ptr(mi),
                                  _lib.ptr(rfit), _lib.ptr(rr), *params, _lib.ptr(hT), _lib.ptr(outs["T"][G:]), _lib.ptr(outs["rf"][G:]),
                                  _lib.ptr(outs["iters"][G:]), _lib.ptr(outs["status"][G:]), _lib.ptr(ws), _lib.stream_ptr()))
    res = {k: v.cpu().numpy() for k, v in outs.items()}
    if G:
        for k in ("T", "rf"):
            assert np.isnan(res[k][:G]).all() and np.isnan(res[k][-G:]).all() and not np.isnan(res[k][G:-G]).any(), k
        for k in ("iters", "status"):
            assert (res[k][:G] == -7).all() and (res[k][-G:] == -7).all() and (res[k][G:-G] >= 0).all(), k
        res = {k: v[G:-G] for k, v in res.items()}
    return dict(T=res["T"].reshape(P, 4, 4), rf=res["rf"].reshape(P, 2), iters=res["iters"].reshape(P, levels), status=res["status"])


def gpu_linearize_batch(buf, pairs, H, W, levels, level, K, method, Ts, params=(0.07, 0.05, 0.1)):
    """bslam_odom_linearize with a zeroed workspace (as gpu_track), for batches of more than one init launch"""
    L = _lib.load()
    P = len(pairs)
    ws = torch.zeros(L.bslam_odom_workspace_bytes(P, H, W, levels), dtype=torch.uint8, device="cuda")
    sums = torch.full((P, 29), float("nan"), dtype=torch.float64, device="cuda")
    hp = np.ascontiguousarray(pairs, np.int32)
    hT = np.ascontiguousarray(Ts, np.float64).reshape(P, 16)
    _lib.check(L.bslam_odom_linearize(_lib.ptr(buf), buf.shape[0], _lib.ptr(hp), P, H, W, levels, level, _lib.ptr(np.asarray(K, np.float64)), int(method),
                                      *params, _lib.ptr(hT), _lib.ptr(sums), _lib.ptr(ws), _lib.stream_ptr()))
    return sums.cpu().numpy()


def rot(axis, angle):
    c, s = np.cos(angle), np.sin(angle)
    i, j = [(1, 2), (2, 0), (0, 1)][axis]
    M = np.eye(4)
    M[i, i] = M[j, j] = c
    M[i, j], M[j, i] = -s, s
    return M


def trans(x=0.0, y=0.0, z=0.0):
    M = np.eye(4)
    M[:3, 3] = (x, y, z)
    return M


@pytest.fixture(scope="module")
def cavity640():
    E = S.cavity_sweep(1000)[:3]
    d, c = (x.numpy() for x in S.render(S.Cavity(), E, K=S.K_640))
    return d, c, E, R.Frames(d, c, S.K_640, 3), gpu_prepare(d, c, S.K_640, 3)


@pytest.fixture(scope="module")
def cavity80():
    E = S.cavity_sweep(1000)[:130]
    d, c = (x.numpy() for x in S.render(S.Cavity(), E, K=K_80, W=80, H=60))
    return d, c, E


# ------------------------------------------------------------------------------------------------ B. Huber branches
@pytest.mark.parametrize("params", HUBER_SETS, ids=lambda p: "-".join(map(str, p)))
@pytest.mark.parametrize("method", METHODS, ids=lambda m: m.name)
def test_huber_branches_linearize(cavity640, method, params):
    d, c, E, ref, buf = cavity640
    pairs = [(0, 1), (1, 2)]
    Ts = [np.eye(4), E[2] @ np.linalg.inv(E[1])]
    for level in range(3):
        g = gpu_linearize(buf, pairs, 480, 640, 3, level, S.K_640, method, Ts, params)
        for p, (a, b) in enumerate(pairs):
            r = ref.linearize(a, b, level, Ts[p], int(method), params)
            check_sums(g[p], r, (level, p))
            f = R.linearize_f64(ref, a, b, level, Ts[p], int(method), params)
            # the GPU differs from the mirror by its summation order (<= 1e-10), the mirror from linearize_f64 by `tol`
            assert abs(g[p, 28] - f["sums"][28]) <= f["ambiguous"], (level, p)
            assert np.all(np.abs(g[p, :28] - f["sums"][:28]) <= f["tol"][:28] + 1e-10 * np.abs(r[:28]).max()), (level, p)
            if params[1] == 0.0:           # deltas 0: huber' = +-0 and huber = 0
                assert np.all(g[p, 21:28] == 0), (level, p)


@pytest.mark.parametrize("params", HUBER_SETS, ids=lambda p: "-".join(map(str, p)))
@pytest.mark.parametrize("method", METHODS, ids=lambda m: m.name)
def test_huber_branches_track(cavity80, method, params):
    d, c, E = cavity80
    ref = R.Frames(d[:2], c[:2], K_80, 2)
    crit = ((5, 1e-6, 1e-6), (4, 1e-6, 1e-6))
    init = rot(0, 0.01) @ rot(1, -0.02) @ trans(0.003, -0.002, 0.001) @ (E[1] @ np.linalg.inv(E[0]))
    r = ref.track(0, 1, int(method), crit, init=init, params=params)
    kw = dict(method=method, criteria_list=[od.OdometryConvergenceCriteria(*x) for x in crit], params=od.OdometryLossParams(*params))
    res = od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), k3x3(K_80), init, **kw)
    check_track(res, r, f"{method.name} {params}")
    seq = od.rgbd_odometry_sequence(d[:2], c[:2], k3x3(K_80), inits=init[None], **kw)
    assert seq.iterations.cpu().numpy().tolist() == [list(r["iters"])]
    if params[1] == 0.0:
        # zero gradient: x = 0 every iteration, so the pose comes back bit for bit; rmse 0 makes the relative-rmse test
        # 0 / 0, so no level converges and each runs all its iterations
        assert np.array_equal(res.transformation.view(np.uint64), init.view(np.uint64))
        assert np.array_equal(r["T"], init) and res.inlier_rmse == 0.0
        assert list(r["iters"]) == [5, 4]


# ------------------------------------------------------------------------------------------------ C. projection borders
PH, PW = 6, 15           # odd width: roundf and rintf also differ at the last column


def plane_scene():
    """both frames: a fronto-parallel plane at depth 1 (float32, depth_scale 1), fx = fy = 1 and half-integer cx, cy,
    so a source pixel x under a translation (tx, 0, 0) projects to uf = x + tx exactly; the intensity is a ramp in u,
    so the sums show which column was gathered"""
    depth = np.ones((2, PH, PW), np.float32)
    ramp = (np.float32(0.05) + np.float32(0.06) * np.arange(PW, dtype=np.float32)).astype(np.float32)
    color = np.repeat(np.broadcast_to(ramp, (2, PH, PW))[..., None], 3, -1).astype(np.float32).copy()
    K = (1.0, 1.0, 7.5, 2.5)
    return depth, color, K


def round_half_away(x):
    return int(np.sign(x) * np.floor(abs(x) + 0.5))


@pytest.mark.parametrize("tx", [-0.5, 0.5, -0.75, -0.25, PW - 1.25, PW - 0.75, PW - 0.5])
def test_projection_borders(tx):
    depth, color, K = plane_scene()
    ref = R.Frames(depth, color, K, 1, depth_scale=1.0)
    buf = gpu_prepare(depth, color, K, 1, depth_scale=1.0)
    T = trans(tx)
    # closed form: the pre-test uf in (-1, W), then roundf (half away from zero) inside [0, W)
    cols = [x for x in range(PW) if -1 < x + tx < PW and 0 <= round_half_away(x + tx) < PW]
    for method in METHODS:
        g = gpu_linearize(buf, [(0, 1)], PH, PW, 1, 0, K, method, [T])[0]
        r = ref.linearize(0, 1, 0, T, int(method))
        if method == od.Method.PointToPlane:      # the last row and column have no normal
            n = (PH - 1) * sum(round_half_away(x + tx) < PW - 1 for x in cols)
        else:
            n = PH * len(cols)
        assert g[28] == n, (method.name, tx, g[28], n)
        check_sums(g, r, (method.name, tx))
        if method == od.Method.Intensity and tx % 1 != 0.5:
            # r = I(u) - I(x) = 0.06 (u - x) per pixel.  (At half-integer uf linearize_f64 cannot tell which way float32
            # rounds it and counts every pixel as ambiguous, so only the other shifts are compared with it.)
            f = R.linearize_f64(ref, 0, 1, 0, T, int(method))
            assert f["ambiguous"] == 0 and f["sums"][28] == n
            assert np.all(np.abs(g[:28] - f["sums"][:28]) <= f["tol"][:28] + 1e-10 * np.abs(r[:28]).max())


@pytest.mark.parametrize("name,T", [("behind z-2", trans(z=-2.0)), ("rot180 y", rot(1, np.pi)), ("vz=0", trans(z=-1.0)),
                                    ("grazing", trans(z=-1.0 + 2.0 ** -20)), ("grazing rot", rot(1, np.arctan(1 / 6.5)))])
def test_points_behind_and_grazing_the_camera(name, T):
    """every point behind the camera: count 0, and a track ends singular at its first evaluation.  vz = 0 exactly
    (z - 1) is also rejected by the uf pre-test, so it cannot tell <= 0 from < 0; the grazing inits put vz a few ulps
    above 0 (all points, or the column x = 14 under a rotation about y)"""
    depth, color, K = plane_scene()
    ref = R.Frames(depth, color, K, 2, depth_scale=1.0)
    buf = gpu_prepare(depth, color, K, 2, depth_scale=1.0)
    for method in METHODS:
        g = gpu_linearize(buf, [(0, 1)], PH, PW, 2, 0, K, method, [T])[0]
        check_sums(g, ref.linearize(0, 1, 0, T, int(method)), (name, method.name))
        if name in ("behind z-2", "rot180 y", "vz=0", "grazing"):
            assert g[28] == 0
        r = ref.track(0, 1, int(method), ((3, 1e-6, 1e-6), (3, 1e-6, 1e-6)), init=T)
        out = gpu_track(buf, 2, [(0, 1)], PH, PW, 2, K, method, ((3, 1e-6, 1e-6), (3, 1e-6, 1e-6)), [T])
        assert out["status"][0] == r["status"] and out["iters"][0].tolist() == list(r["iters"]), (name, method.name)
        if g[28] == 0:
            assert r["status"] == 1 and list(r["iters"]) == [1, 0]
            assert np.array_equal(out["T"][0], T) and np.array_equal(r["T"], T)
        else:
            assert np.abs(out["T"][0] - r["T"]).max() <= 1e-9


# ------------------------------------------------------------------------------------------------ D. pair batches
@pytest.fixture(scope="module")
def batch80(cavity80):
    d, c, E = cavity80
    d, c, E = d[:4], c[:4], E[:4]
    return d, c, E, R.Frames(d, c, K_80, 2), gpu_prepare(d, c, K_80, 2)


def batch_pairs(P, E):
    """pair p: (p % 3) -> (p % 3 + 1) from the ground truth times a small rotation that depends on p"""
    pairs = [(p % 3, p % 3 + 1) for p in range(P)]
    inits = [rot(p % 3, 1e-3 * ((p * 37) % 11 - 5)) @ (E[b] @ np.linalg.inv(E[a])) for p, (a, b) in enumerate(pairs)]
    return pairs, inits


@pytest.mark.parametrize("P", [127, 128, 129, 256, 257, 1000])
def test_pair_batches_across_init_launches(batch80, P):
    d, c, E, ref, buf = batch80
    crit = ((4, 1e-6, 1e-6), (3, 1e-6, 1e-6))
    pairs, inits = batch_pairs(P, E)
    out = gpu_track(buf, 4, pairs, 60, 80, 2, K_80, od.Method.Hybrid, crit, inits, guard=64)
    refs = {}                          # the (pair, init) combinations repeat every 33 pairs
    for p in range(P):
        key = (p % 3, (p * 37) % 11)
        if key not in refs:
            refs[key] = ref.track(*pairs[p], int(od.Method.Hybrid), crit, init=inits[p])
        r = refs[key]
        assert out["status"][p] == r["status"] == 0, p
        assert np.abs(out["T"][p] - r["T"]).max() <= 1e-9 and out["iters"][p].tolist() == list(r["iters"]), p
        assert abs(out["rf"][p, 0] - r["rmse"]) <= 1e-9 * r["rmse"] and abs(out["rf"][p, 1] - r["fitness"]) <= 1e-9 * r["fitness"], p
    # linearize splits its init launches the same way
    Ts = inits[:P]
    g = gpu_linearize_batch(buf, pairs, 60, 80, 2, 0, K_80, od.Method.Hybrid, Ts)
    for p in sorted({0, 126, 127, 128, 129, P - 2, P - 1} & set(range(P))):
        check_sums(g[p], ref.linearize(*pairs[p], 0, Ts[p], int(od.Method.Hybrid)), p)


def test_pair_batch_at_the_grid_limit(cavity80):
    """65 535 pairs, the most one call takes (they run in gridDim.y), at 16 x 16 with one level and two iterations"""
    d, c, E = cavity80
    K16 = small_K(16)
    d16, c16 = (x.numpy() for x in S.render(S.Cavity(), E[:2], K=K16, W=16, H=16, invalid_frac=0.0))
    ref = R.Frames(d16, c16, K16, 1)
    buf = gpu_prepare(d16, c16, K16, 1)
    P = 65535
    base = E[1] @ np.linalg.inv(E[0])
    poses = [rot(k % 3, 2e-3 * (k - 4)) @ base for k in range(8)]
    inits = np.stack([poses[p % 8] for p in range(P)])
    crit = ((2, 1e-6, 1e-6),)
    out = gpu_track(buf, 2, [(0, 1)] * P, 16, 16, 1, K16, od.Method.Hybrid, crit, inits, guard=64)
    for k in range(8):
        r = ref.track(0, 1, int(od.Method.Hybrid), crit, init=poses[k])
        idx = np.arange(k, P, 8)
        assert (out["status"][idx] == r["status"]).all() and (out["iters"][idx] == r["iters"]).all(), k
        T = out["T"][idx]
        assert (T.view(np.uint64) == T[0].view(np.uint64)).all() and (out["rf"][idx].view(np.uint64) == out["rf"][k].view(np.uint64)).all(), k
        assert np.abs(T[0] - r["T"]).max() <= 1e-9, k


# ------------------------------------------------------------------------------------------------ E. singular pairs
@pytest.mark.parametrize("method", [od.Method.PointToPlane, od.Method.Hybrid], ids=lambda m: m.name)
def test_singular_pairs_inside_a_sequence(cavity80, method):
    """frames 30 and 63 (at the chunk seam: pair 63 is the first of the second chunk) have no valid depth, so the four
    pairs touching them are singular at their first evaluation.  Frame 45 has valid depth on even rows and columns
    only: its level-0 normals and depth gradients are all NaN, while level 1 (whose pixels are its even pixels' means)
    is complete, so pair 44 -> 45 succeeds at the coarse level and turns singular at the fine one (built, not found)."""
    d, c, E = cavity80
    d, c = d[:70].copy(), c[:70]
    for k in (30, 63):
        d[k] = 0
    sparse = np.zeros_like(d[45])
    sparse[::2, ::2] = d[45][::2, ::2]
    d[45] = sparse
    crit = ((4, 1e-6, 1e-6), (3, 1e-6, 1e-6))
    kw = dict(method=method, criteria_list=[od.OdometryConvergenceCriteria(4), od.OdometryConvergenceCriteria(3)])
    seq = od.rgbd_odometry_sequence(d, c, k3x3(K_80), **kw)
    T, rmse, fit = seq.transformations.cpu().numpy(), seq.inlier_rmse.cpu().numpy(), seq.fitness.cpu().numpy()
    its, status = seq.iterations.cpu().numpy(), seq.status.cpu().numpy()
    ref = R.Frames(d, c, K_80, 2)
    singular = {29, 30, 62, 63, 44}
    for i in range(69):
        if i not in singular:
            assert status[i] == 0, i
            one = od.rgbd_odometry_multi_scale(RGBDImage(c[i], d[i]), RGBDImage(c[i + 1], d[i + 1]), k3x3(K_80), **kw)
            assert np.array_equal(one.transformation.view(np.uint64), T[i].view(np.uint64)), i
            assert one.inlier_rmse == rmse[i] and one.fitness == fit[i], i
            continue
        r = ref.track(i, i + 1, int(method), crit)
        assert status[i] == 1 and r["status"] == 1, i
        assert its[i].tolist() == list(r["iters"]), (i, its[i], r["iters"])
        assert abs(rmse[i] - r["rmse"]) <= 1e-9 * r["rmse"] and abs(fit[i] - r["fitness"]) <= 1e-9 * r["fitness"], i
        if i == 44:                  # the pose before the failed solve: the coarse level's result
            assert its[i][0] >= 1 and its[i][1] == 1 and np.abs(T[i] - r["T"]).max() <= 1e-9 and not np.array_equal(T[i], np.eye(4))
        else:
            assert its[i].tolist() == [1, 0] and np.array_equal(T[i], np.eye(4)) and fit[i] == 0.0, i
        with pytest.raises(RuntimeError, match="Singular 6x6"):
            od.rgbd_odometry_multi_scale(RGBDImage(c[i], d[i]), RGBDImage(c[i + 1], d[i + 1]), k3x3(K_80), **kw)


# ------------------------------------------------------------------------------------------------ F. sequence inits
@pytest.mark.parametrize("F", [64, 65, 130])
def test_sequence_inits_across_chunks(cavity80, F):
    d, c, E = cavity80
    d, c, E = d[:F], c[:F], E[:F]
    rng = np.random.default_rng(F)
    inits = np.stack([rot(0, rng.normal(0, 2e-3)) @ rot(1, rng.normal(0, 2e-3)) @ trans(*rng.normal(0, 1e-3, 3)) @ (E[i + 1] @ np.linalg.inv(E[i]))
                      for i in range(F - 1)])
    kw = dict(method=od.Method.Hybrid, criteria_list=[od.OdometryConvergenceCriteria(4), od.OdometryConvergenceCriteria(3)])
    seq = od.rgbd_odometry_sequence(d, c, k3x3(K_80), inits=torch.as_tensor(inits), **kw)
    T, its = seq.transformations.cpu().numpy(), seq.iterations.cpu().numpy()
    assert not seq.status.any()
    for i in range(F - 1):
        one = od.rgbd_odometry_multi_scale(RGBDImage(c[i], d[i]), RGBDImage(c[i + 1], d[i + 1]), k3x3(K_80), inits[i], **kw)
        assert np.array_equal(one.transformation.view(np.uint64), T[i].view(np.uint64)), i
    ref = R.Frames(d, c, K_80, 2)
    for i in sorted({0, 62, 63, 64, 126, 127} & set(range(F - 1))):
        r = ref.track(i, i + 1, int(od.Method.Hybrid), ((4, 1e-6, 1e-6), (3, 1e-6, 1e-6)), init=inits[i])
        assert np.abs(T[i] - r["T"]).max() <= 1e-9 and its[i].tolist() == list(r["iters"]), i
    # the identity inits give a different answer, so the inits were used
    plain = od.rgbd_odometry_sequence(d, c, k3x3(K_80), **kw).transformations.cpu().numpy()
    assert not np.array_equal(plain, T)
    for n in (F - 2, F):
        with pytest.raises(RuntimeError, match="inits"):
            od.rgbd_odometry_sequence(d, c, k3x3(K_80), inits=np.tile(np.eye(4), (n, 1, 1)), **kw)


# ------------------------------------------------------------------------------------------------ G. preparation inputs
def odd_inputs(depth_max, depth_scale):
    """2 frames of 23 x 37 float32 depth and float colour with every awkward value"""
    h, w = 23, 37
    rng = np.random.default_rng(7)
    d = (rng.uniform(0.15, 0.4, (2, h, w)) * depth_scale).astype(np.float32)
    top = np.float32(np.float32(depth_max) * np.float32(depth_scale))
    special = np.array([np.nan, np.inf, -np.inf, -1.0, -0.0, 0.0, 1e-45, 1e-40, np.finfo(np.float32).tiny, top, np.nextafter(top, np.float32(0)),
                        np.nextafter(top, np.float32(np.inf)), np.float32(depth_max), 3e38], np.float32)
    flat = d.reshape(-1)
    pos = rng.choice(flat.size, size=(special.size, 12), replace=False)
    for v, p in zip(special, pos):
        flat[p] = v
    c = rng.uniform(0, 1, (2, h, w, 3)).astype(np.float32)
    cf = c.reshape(-1)
    for v, p in zip(np.array([np.nan, -0.5, 1.5, -0.0, 1e-40, np.inf], np.float32), rng.choice(cf.size, size=(6, 20), replace=False)):
        cf[p] = v
    return d, c, (0.8 * w, 0.8 * w, w / 2 - 0.3, h / 2 + 0.2)


@pytest.mark.parametrize("depth_scale,trunc", [(1.0, 0.07), (1000.0, 0.07), (999.7, 0.07), (5000.3, 0.03), (1.0, 0.0), (999.7, 1e30)])
def test_preparation_of_unusual_inputs(depth_scale, trunc):
    d, c, K = odd_inputs(3.0, depth_scale)
    ref = R.Frames(d, c, K, 3, depth_scale=depth_scale, depth_max=3.0, depth_outlier_trunc=trunc)
    gpu = gpu_prepare(d, c, K, 3, depth_scale=depth_scale, depth_max=3.0, trunc=trunc).cpu().numpy()
    for f in range(2):
        for l in range(3):
            g = R.Frames.__new__(R.Frames)
            g.__dict__.update(ref.__dict__, data=gpu)
            for k, v in ref.planes(f, l).items():
                same_bits(g.planes(f, l)[k], v, f"frame {f} level {l} {k}")
    if trunc == 0.0:                  # PyrDownDepth keeps no neighbour: every coarse depth is NaN
        assert all(np.isnan(ref.planes(f, l)["depth"]).all() for f in range(2) for l in (1, 2))
    same_bits(gpu_prepare(d, None, K, 3, depth_scale=depth_scale, trunc=trunc).cpu().numpy(),
              R.Frames(d, None, K, 3, depth_scale=depth_scale, depth_outlier_trunc=trunc).data, "no colour")


@pytest.mark.parametrize("trunc", [0.0, 1e30])
def test_track_at_extreme_outlier_truncation(cavity80, trunc):
    d, c, E = cavity80
    df, cf = d[:2].astype(np.float32) * np.float32(0.9997), c[:2].astype(np.float32) / np.float32(255)
    crit = ((4, 1e-6, 1e-6), (3, 1e-6, 1e-6), (2, 1e-6, 1e-6))
    params = (trunc, 0.05, 0.1)
    ref = R.Frames(df, cf, K_80, 3, depth_scale=999.7, depth_outlier_trunc=trunc)
    kw = dict(depth_scale=999.7, criteria_list=[od.OdometryConvergenceCriteria(m) for m, _, _ in crit], params=od.OdometryLossParams(*params))
    for method in METHODS:
        r = ref.track(0, 1, int(method), crit, params=params)
        if trunc == 0.0:                  # the coarsest level is all NaN: singular at its first evaluation
            assert r["status"] == 1 and list(r["iters"]) == [1, 0, 0]
            with pytest.raises(RuntimeError, match="Singular 6x6"):
                od.rgbd_odometry_multi_scale(RGBDImage(cf[0], df[0]), RGBDImage(cf[1], df[1]), k3x3(K_80), method=method, **kw)
            seq = od.rgbd_odometry_sequence(df, cf, k3x3(K_80), method=method, **kw)
            assert seq.status.cpu().tolist() == [1] and seq.iterations.cpu().tolist() == [[1, 0, 0]]
        else:
            check_track(od.rgbd_odometry_multi_scale(RGBDImage(cf[0], df[0]), RGBDImage(cf[1], df[1]), k3x3(K_80), method=method, **kw), r,
                        method.name)


# ------------------------------------------------------------------------------------------------ H. tile seams, 1080p
@pytest.mark.parametrize("HW,levels", [((32, 32), 2), ((25, 41), 2), ((64, 64), 2), ((50, 82), 2), ((48, 64), 2)])
def test_reduce_tile_seams(HW, levels):
    """level sizes of 1024 k and 1024 k + 1 pixels (the reduce's tile), at level 0 and at level 1"""
    h, w = HW
    E = S.cavity_sweep(1000)[:2]
    K = (S.K_640[0] * w / 640, S.K_640[1] * h / 480, S.K_640[2] * w / 640, S.K_640[3] * h / 480)
    d, c = (x.numpy() for x in S.render(S.Cavity(), E, K=K, W=w, H=h, invalid_frac=0.0))
    ref = R.Frames(d, c, K, levels)
    buf = gpu_prepare(d, c, K, levels)
    T = E[1] @ np.linalg.inv(E[0])
    for method in METHODS:
        for level in range(levels):
            for Tp in (np.eye(4), T):
                check_sums(gpu_linearize(buf, [(0, 1)], h, w, levels, level, K, method, [Tp])[0], ref.linearize(0, 1, level, Tp, int(method)),
                           (HW, method.name, level))
        crit = ((4, 1e-6, 1e-6), (3, 1e-6, 1e-6))
        r = ref.track(0, 1, int(method), crit)
        out = gpu_track(buf, 2, [(0, 1)], h, w, levels, K, method, crit, [np.eye(4)])
        assert out["status"][0] == r["status"] and out["iters"][0].tolist() == list(r["iters"]), (HW, method.name)
        assert np.abs(out["T"][0] - r["T"]).max() <= 1e-9, (HW, method.name)


def test_1080p_pair():
    """1920 x 1080: 2025 tiles at level 0, about 8 partials per solve thread (the reference takes well under 20 s)"""
    K = tuple(k * 3 for k in S.K_640)
    E = S.cavity_sweep(1000)[:2]
    d, c = (x.numpy() for x in S.render(S.Cavity(), E, K=K, W=1920, H=1080))
    ref = R.Frames(d, c, K, 3)
    buf = gpu_prepare(d, c, K, 3)
    T = E[1] @ np.linalg.inv(E[0])
    for level in range(3):
        check_sums(gpu_linearize(buf, [(0, 1)], 1080, 1920, 3, level, K, od.Method.Hybrid, [T])[0], ref.linearize(0, 1, level, T, int(od.Method.Hybrid)),
                   level)
    r = ref.track(0, 1, int(od.Method.Hybrid), REF_CRIT)
    check_track(od.rgbd_odometry_multi_scale(RGBDImage(c[0], d[0]), RGBDImage(c[1], d[1]), k3x3(K)), r, "1080p")


# ------------------------------------------------------------------------------------------------ I. MAP with colour
@pytest.mark.parametrize("method", [od.Method.Intensity, od.Method.Hybrid], ids=lambda m: m.name)
def test_map_tracking_with_colour(method):
    """frame-to-model tracking with the photometric methods: the target colour is the ray cast's float32 in [0, 1], the
    source uint8; depth_diff 0.05 and an explicit depth_scale of 1250 (the frames are in millimetres, so both frames
    shrink by 0.8 and the result differs from the map's own scale).  The map integrates at the ground-truth poses."""
    K = S.K_640
    E = S.cavity_sweep(1000)[:12]
    d, c = (x.numpy() for x in S.render(S.Cavity(), E, K=K))
    m = MAP(640, 480, k3x3(K), "CUDA:0", 1000.0, voxel_size=0.002, resolution=256)
    ds, crit = 1250.0, ((6, 1e-6, 1e-6), (3, 1e-6, 1e-6), (1, 1e-6, 1e-6))
    for i in range(12):
        fr = FakeRGBD(d[i], c[i], 1000.0)
        if i > 0:
            mf = m.synthesize_model_frame()
            assert "color" in mf
            res = m.track_frame_to_model(fr, mf, depth_scale=ds, depth_diff=0.05, method=method)
            mc = mf["color"][0].cpu().numpy()
            assert mc.dtype == np.float32 and np.nanmax(mc) <= 1.0
            src = R.Frames(d[i], c[i], K, 3, depth_scale=ds, depth_outlier_trunc=0.05)
            tgt = R.Frames(mf["depth"][0].cpu().numpy(), mc, K, 3, depth_scale=ds, depth_outlier_trunc=0.05)
            src.data = np.concatenate([src.data, tgt.data])
            r = src.track(0, 1, int(method), crit, params=(0.05, 0.05, 0.1))
            check_track(res, r, f"step {i}")
            default = m.track_frame_to_model(fr, mf, depth_diff=0.05, method=method)
            assert not np.array_equal(default.transformation, res.transformation)
        m.integrate(fr, i, np.linalg.inv(E[i]))


# ------------------------------------------------------------------------------------------------ J. another device
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_second_device_matches_first(cavity80):
    d, c, E = cavity80
    d, c = d[:6], c[:6]
    kw = dict(criteria_list=[od.OdometryConvergenceCriteria(4), od.OdometryConvergenceCriteria(3)])
    torch.cuda.set_device(0)
    out = {}
    for dev in ("cuda:0", "cuda:1"):
        dt, ct = torch.as_tensor(d, device=dev), torch.as_tensor(c, device=dev)
        one = od.rgbd_odometry_multi_scale(RGBDImage(ct[0], dt[0]), RGBDImage(ct[1], dt[1]), k3x3(K_80), **kw)
        seq = od.rgbd_odometry_sequence(dt, ct, k3x3(K_80), **kw)
        assert seq.transformations.device == torch.device(dev)
        out[dev] = (one.transformation, seq.transformations.cpu().numpy(), seq.iterations.cpu().numpy())
        assert torch.cuda.current_device() == 0
    for a, b in zip(out["cuda:0"], out["cuda:1"]):
        assert np.array_equal(a, b)
