"""Multi-scale RGB-D odometry: the CPU reference (tests/odometry_ref.c; parity with Open3D unpinned) against closed
forms, and the C ABI's argument checks, which need no device."""
import ctypes

import numpy as np
import pytest

import odometry_ref as R
from bodyslam_b200 import _lib
from bodyslam_b200 import synthetic as S

SQRT_LAMBDA_DEPTH, SQRT_LAMBDA_INTENSITY = 0.98386991, 0.17888544
W, H = 96, 72
K = (80.0, 82.0, 47.5, 35.5)


def delta_T(x):
    """DeltaT of the update: [Rz(gamma) Ry(beta) Rx(alpha) | t], x = (alpha, beta, gamma, tx, ty, tz)"""
    a, b, g = x[:3]
    Rz = np.array([[np.cos(g), -np.sin(g), 0], [np.sin(g), np.cos(g), 0], [0, 0, 1]])
    Ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
    Rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
    M = np.eye(4)
    M[:3, :3] = Rz @ Ry @ Rx
    M[:3, 3] = x[3:]
    return M


# target: depth and intensity linear in the pixel coordinates, so 0.125 x Sobel is their exact gradient
DEPTH_RAMP = (0.30, 4e-4, -3e-4)          # z = a + b u + c v
INT_RAMP = (0.45, 2e-3, 1.5e-3)           # I = a + b u + c v


def ramp(c, u, v):
    return c[0] + c[1] * u + c[2] * v


def ramp_frames(T_src_to_tgt, levels=1):
    """frame 0 = source (the target's surface and colour seen from T^-1), frame 1 = target; float32 depth (metres) and
    colour (grey = the intensity)"""
    v, u = np.mgrid[0:H, 0:W].astype(np.float64)
    zt = ramp(DEPTH_RAMP, u, v)
    It = ramp(INT_RAMP, u, v)
    # source pixels: march each source ray to the target's surface z(u, v) by fixed-point iteration in float64
    Ti = np.linalg.inv(T_src_to_tgt)
    xn, yn = (u - K[2]) / K[0], (v - K[3]) / K[1]
    zs = np.full_like(u, 0.3)
    for _ in range(60):
        p = np.stack([xn * zs, yn * zs, zs], -1) @ T_src_to_tgt[:3, :3].T + T_src_to_tgt[:3, 3]
        ut, vt = K[0] * p[..., 0] / p[..., 2] + K[2], K[1] * p[..., 1] / p[..., 2] + K[3]
        zs = zs + (ramp(DEPTH_RAMP, ut, vt) - p[..., 2]) * 0.9
    Is = ramp(INT_RAMP, ut, vt)
    assert Ti.shape == (4, 4)
    depth = np.stack([zs, zt]).astype(np.float32)
    color = np.repeat(np.stack([Is, It])[..., None], 3, -1).astype(np.float32)
    return R.Frames(depth, color, K, levels, depth_scale=1.0, depth_max=3.0)


def continuous_residual(fr, method, T, x, y, rounded=False):
    """float64 photometric (and depth) residual(s) of source pixel (x, y) with the target's depth / intensity read
    continuously, or at the rounded pixel as the reference reads them"""
    s = fr.planes(0, 0)
    V = np.array([s["vx"][y, x], s["vy"][y, x], s["vz"][y, x]], np.float64)
    p = T[:3, :3] @ V + T[:3, 3]
    u, v = K[0] * p[0] / p[2] + K[2], K[1] * p[1] / p[2] + K[3]
    if rounded:
        u, v = np.round(u), np.round(v)
    rI = ramp(INT_RAMP, u, v) - float(s["intensity"][y, x])
    if method == R.INTENSITY:
        return np.array([rI])
    return np.array([SQRT_LAMBDA_INTENSITY * rI, SQRT_LAMBDA_DEPTH * (ramp(DEPTH_RAMP, u, v) - p[2])])


@pytest.mark.parametrize("method", [R.POINT_TO_PLANE, R.INTENSITY, R.HYBRID])
def test_jacobians_are_the_derivatives_of_the_residuals(method):
    T_true = delta_T(np.array([0.004, -0.006, 0.003, 0.002, -0.001, 0.003]))
    fr = ramp_frames(T_true)
    T = delta_T(np.array([0.001, 0.0, -0.001, 0.0005, 0.0, -0.0005])) @ T_true     # off the solution: residuals != 0
    checked = 0
    for (x, y) in ((20, 15), (48, 36), (70, 50), (30, 60)):
        n, J, r = fr.pixel(0, 1, 0, T, method, x, y, trunc=0.07)
        assert n == (2 if method == R.HYBRID else 1)
        if method == R.POINT_TO_PLANE:
            s, t = fr.planes(0, 0), fr.planes(1, 0)
            V = np.array([s["vx"][y, x], s["vy"][y, x], s["vz"][y, x]], np.float64)
            Tf = T.astype(np.float32).astype(np.float64)
            p = Tf[:3, :3] @ V + Tf[:3, 3]
            u, v = int(np.round(K[0] * p[0] / p[2] + K[2])), int(np.round(K[1] * p[1] / p[2] + K[3]))
            Vt = np.array([t["vx"][v, u], t["vy"][v, u], t["vz"][v, u]], np.float64)
            nt = np.array([t["nx"][v, u], t["ny"][v, u], t["nz"][v, u]], np.float64)

            def res(e):
                q = delta_T(e) @ Tf
                return np.array([(q[:3, :3] @ V + q[:3, 3] - Vt) @ nt])
            assert abs(res(np.zeros(6))[0] - r[0]) <= 1e-6
        else:
            def res(e):
                return continuous_residual(fr, method, delta_T(e) @ T, x, y)
            rr = continuous_residual(fr, method, T.astype(np.float32).astype(np.float64), x, y, rounded=True)
            assert np.abs(rr - r).max() <= 2e-6, (rr, r)
        h = 1e-6
        num = np.stack([(res(h * np.eye(6)[k]) - res(-h * np.eye(6)[k])) / (2 * h) for k in range(6)], -1)
        scale = np.abs(num).max()
        assert np.abs(num - J).max() <= 2e-3 * scale, (num, J)
        checked += 1
    assert checked == 4


@pytest.fixture(scope="module")
def scenes():
    """two frames, 3 frames apart, of the laparoscopy sweep (cavity) and of the colonoscopy lumen at 640 x 480"""
    cav = S.config("laparoscopy512")["extrinsics"](1000)[[0, 1]]
    lum = S.Lumen()
    El = S.lumen_trajectory(lum, 300)[[100, 103]]
    out = {}
    for name, surf, E in (("cavity", S.Cavity(), cav), ("lumen", lum, El)):
        d, c = S.render(surf, E, K=S.K_640)
        out[name] = (R.Frames(d.numpy(), c.numpy(), S.K_640, 3), E[1] @ np.linalg.inv(E[0]))
    return out


# measured on this reference: the photometric methods land within ~1e-4 rad / 3e-4 m.  Point-to-plane on raw
# millimetre depth: the 1 mm steps at ~0.2 mm pixel spacing make most level-0 normals (0, 0, 1); on the cavity it ends
# 0.07 / 0.012 m off, and on the lumen (a tube: sliding along it is unconstrained) it ends singular.
BARS = {("cavity", R.INTENSITY): (2e-4, 1e-4), ("cavity", R.HYBRID): (1e-4, 5e-5),
        ("lumen", R.INTENSITY): (5e-4, 5e-4), ("lumen", R.HYBRID): (3e-4, 2e-4)}


@pytest.mark.parametrize("name", ["cavity", "lumen"])
@pytest.mark.parametrize("method", [R.INTENSITY, R.HYBRID])
def test_recovers_known_motion(scenes, name, method):
    fr, truth = scenes[name]
    r = fr.track(0, 1, method)
    assert r["status"] == 0 and list(r["iters"]) == [10, 5, 3]
    rot, trans = np.abs(r["T"][:3, :3] - truth[:3, :3]).max(), np.abs(r["T"][:3, 3] - truth[:3, 3]).max()
    assert rot <= BARS[name, method][0] and trans <= BARS[name, method][1], (rot, trans)
    assert 0.6 < r["fitness"] < 1.0 and 0 < r["rmse"] < 0.01


def test_point_to_plane_on_millimetre_depth(scenes):
    """the documented weakness above, pinned so that a change of it is noticed"""
    fr, truth = scenes["cavity"]
    r = fr.track(0, 1, R.POINT_TO_PLANE)
    assert r["status"] == 0 and np.abs(r["T"] - truth).max() < 0.1
    assert fr.track(0, 1, R.POINT_TO_PLANE, criteria=((10, 1e-6, 1e-6), (5, 1e-6, 1e-6), (0, 1e-6, 1e-6)))["status"] == 0
    fr, _ = scenes["lumen"]
    assert fr.track(0, 1, R.POINT_TO_PLANE)["status"] == 1


def test_point_to_plane_error_source():
    """where point-to-plane's error on the cavity comes from: exact (unquantised) depth in both frames recovers the
    motion; a millimetre-quantised source against an exact target -- what MAP.track_frame_to_model sees, the target
    being the ray cast -- does not, because the rotations are weakly constrained (A^T A's three smallest eigenvalues,
    the rotation directions, lie four orders of magnitude below the translations')"""
    E = S.cavity_sweep(1000)[[0, 1]]
    exact = []
    for e in E:
        o, d = S._rays(S.K_640, 640, 480, np.linalg.inv(e), "cpu")
        exact.append((S.Cavity().depth(o, d).numpy() * 1000.0).astype(np.float32))
    truth = E[1] @ np.linalg.inv(E[0])
    crit = ((6, 1e-6, 1e-6), (3, 1e-6, 1e-6), (1, 1e-6, 1e-6))
    fr = R.Frames(np.stack(exact), None, S.K_640, 3)
    r = fr.track(0, 1, R.POINT_TO_PLANE, crit)
    assert np.abs(r["T"] - truth).max() <= 5e-4         # measured 1.2e-4
    S28 = fr.linearize(0, 1, 0, truth, R.POINT_TO_PLANE)
    A = np.zeros((6, 6))
    A[np.triu_indices(6)] = S28[:21]
    A = A + np.triu(A, 1).T
    w, V = np.linalg.eigh(A)
    assert w[2] < 1e-3 * w[3] and np.all(np.linalg.norm(V[:3, :3], axis=0) > 0.98)      # mostly rotation
    src = R.Frames(np.floor(exact[0] + 0.5).astype(np.uint16), None, S.K_640, 3)
    src.data = np.concatenate([src.data, fr.data[1:]])
    r = src.track(0, 1, R.POINT_TO_PLANE, crit)
    assert np.abs(r["T"] - truth).max() >= 5e-3         # measured 1.5e-2


def test_convergence_stops_levels_early():
    w, h = 80, 60
    K = (S.K_640[0] / 8, S.K_640[1] / 8, S.K_640[2] / 8, S.K_640[3] / 8)
    d, c = S.render(S.Cavity(), S.cavity_sweep(1000)[:40], K=K, W=w, H=h)
    fr = R.Frames(d.numpy(), c.numpy(), K, 2)
    its = np.array([fr.track(i, i + 1, R.POINT_TO_PLANE, ((6, 1e-2, 1e-2),) * 2)["iters"] for i in range(39)])
    assert (its == 6).all(axis=1).any() and ((its[:, 0] == 6) & (its[:, 1] < 6)).any() and ((its[:, 0] < 6) & (its[:, 1] > 0)).any()
    # a pair that stops early at a level ran at least two iterations there: the first has no previous fitness
    assert its.min() >= 2
    never = np.array([fr.track(i, i + 1, R.POINT_TO_PLANE, ((6, 0.0, 0.0),) * 2)["iters"] for i in range(39)])
    assert (never == 6).all()


@pytest.mark.parametrize("method", [R.POINT_TO_PLANE, R.INTENSITY, R.HYBRID])
def test_identity(scenes, method):
    fr, _ = scenes["cavity"]
    r = fr.track(0, 0, method)
    assert r["status"] == 0
    assert np.abs(r["T"] - np.eye(4)).max() <= 1e-12
    p = fr.planes(0, 0)
    valid = ~np.isnan(p["depth"])
    if method == R.POINT_TO_PLANE:        # inliers need their own normal
        valid &= ~np.isnan(p["nx"])
    else:
        valid &= ~np.isnan(p["dix"]) & ~np.isnan(p["diy"])
        if method == R.HYBRID:
            valid &= ~np.isnan(p["ddx"]) & ~np.isnan(p["ddy"])
    assert r["fitness"] == valid.mean()
    assert r["rmse"] == 0.0


@pytest.mark.parametrize("HW", [(480, 640), (479, 641), (17, 9), (8, 8), (1, 1), (5, 300)])
def test_pyramid_sizes(HW):
    h, w = HW
    levels = 1 + min(int(np.log2(h)), int(np.log2(w)))
    d = np.full((h, w), 200, np.uint16)
    fr = R.Frames(d, None, (100.0, 100.0, w / 2, h / 2), levels)
    assert [fr.planes(0, l)["depth"].shape for l in range(levels)] == [(h >> l, w >> l) for l in range(levels)]
    assert fr.data.shape[1] == 12 * sum((h >> l) * (w >> l) for l in range(levels))
    assert np.all(fr.planes(0, levels - 1)["depth"] == np.float32(0.2))
    L = _lib.load()
    assert L.bslam_odom_frame_bytes(h, w, levels) == 4 * fr.data.shape[1]
    assert L.bslam_odom_frame_bytes(h, w, levels + 1) == 0        # a level below 1 x 1


def test_prepared_maps_closed_forms():
    fr = ramp_frames(np.eye(4))
    t = fr.planes(1, 0)
    inner = (slice(1, H - 1), slice(1, W - 1))
    assert np.abs(0.125 * t["dix"][inner] - INT_RAMP[1]).max() <= 1e-6
    assert np.abs(0.125 * t["diy"][inner] - INT_RAMP[2]).max() <= 1e-6
    assert np.abs(0.125 * t["ddx"][inner] - DEPTH_RAMP[1]).max() <= 1e-6
    v, u = np.mgrid[0:H, 0:W]
    assert np.abs(t["vx"] - (u - K[2]) * t["depth"] / K[0]).max() <= 1e-6
    n = np.stack([t["nx"], t["ny"], t["nz"]], -1)
    assert np.isnan(n[-1]).all() and np.isnan(n[:, -1]).all() and not np.isnan(n[:-1, :-1]).any()
    assert np.abs(np.linalg.norm(n[:-1, :-1], axis=-1) - 1).max() <= 1e-6
    # invalid depth: <= 0, >= depth_max, NaN
    d = np.array([[0, 1, 2999, 3000, 65535]], np.uint16)
    p = R.Frames(d, None, K, 1).planes(0, 0)["depth"]
    assert np.isnan(p[0, [0, 3, 4]]).all() and p[0, 1] == np.float32(0.001) and p[0, 2] == np.float32(2.999)
    rgb = np.array([[[255, 0, 0], [0, 255, 0], [0, 0, 255], [10, 20, 30], [255, 255, 255]]], np.uint8)
    I = R.Frames(d, rgb, K, 1).planes(0, 0)["intensity"]
    assert I[0, 4] == np.float32((np.float32(0.299) * 255 + np.float32(0.587) * 255 + np.float32(0.114) * 255) / np.float32(255))
    assert np.abs(I[0] - (rgb @ np.array([0.299, 0.587, 0.114])) / 255).max() <= 1e-6


def test_pyrdown_depth_skips_outliers_and_invalid_centres():
    d = np.full((8, 8), 0.5, np.float32)
    d[2, 3] = 0.9            # farther than 2 x depth_outlier_trunc from the centre (2, 2): left out of its mean
    d[4, 4] = np.nan         # centre of level-1 pixel (2, 2)
    p = R.Frames(d, None, K, 2, depth_scale=1.0).planes(0, 1)["depth"]
    assert p[1, 1] == np.float32(0.5) and np.isnan(p[2, 2])


def test_singular_system():
    d = np.zeros((2, 48, 64), np.uint16)           # no valid source pixel
    d[1] = 300
    fr = R.Frames(d, np.zeros(d.shape + (3,), np.uint8), (50.0, 50.0, 32.0, 24.0), 2)
    for method in (R.POINT_TO_PLANE, R.INTENSITY, R.HYBRID):
        r = fr.track(0, 1, method, criteria=((4, 1e-6, 1e-6), (4, 1e-6, 1e-6)))
        assert r["status"] == 1 and list(r["iters"]) == [1, 0] and r["fitness"] == 0.0
        assert np.array_equal(r["T"], np.eye(4))
    # a plane seen head-on: point-to-plane cannot fix the in-plane motion
    flat = np.full((2, 48, 64), 300, np.uint16)
    assert R.Frames(flat, None, (50.0, 50.0, 32.0, 24.0), 1).track(0, 1, R.POINT_TO_PLANE, criteria=((3, 1e-6, 1e-6),))["status"] == 1


def test_c_abi_argument_errors_do_not_need_a_device():
    L = _lib.load()
    K4 = np.array(K, np.float64)
    out = ctypes.c_void_p(16)          # never dereferenced: the arguments are rejected first
    pairs = np.array([[0, 1]], np.int32)
    mi = np.array([3, 2], np.int32)
    rel = np.full(2, 1e-6)
    init = np.eye(4).reshape(-1)

    def track(F=2, P=1, h=H, w=W, levels=2, method=0, pairs=pairs, frames=out, K=K4, mi=mi):
        return L.bslam_odom_track(frames, F, _lib.ptr(pairs), P, h, w, levels, _lib.ptr(K), method, _lib.ptr(mi), _lib.ptr(rel), _lib.ptr(rel),
                                  0.07, 0.05, 0.1, _lib.ptr(init), out, out, out, out, out, None)

    assert track(frames=None) == _lib.E_ARG and b"NULL" in L.bslam_last_error()
    assert track(K=None) == _lib.E_ARG and b"NULL" in L.bslam_last_error()
    for h, w, levels in ((0, W, 1), (H, -1, 1), (8, 8, 5), (17, 9, 5), (H, W, 0), (H, W, 17)):
        assert track(h=h, w=w, levels=levels) == _lib.E_ARG and b"Unsupported image format" in L.bslam_last_error()
    assert track(method=3) == _lib.E_ARG and b"method" in L.bslam_last_error()
    assert track(pairs=np.array([[0, 2]], np.int32)) == _lib.E_ARG and b"out of range" in L.bslam_last_error()
    assert track(pairs=np.array([[-1, 0]], np.int32)) == _lib.E_ARG
    assert track(F=0) == _lib.E_ARG
    assert track(mi=np.array([3, -1], np.int32)) == _lib.E_ARG
    assert L.bslam_odom_track(None, 0, None, 0, H, W, 2, _lib.ptr(K4), 0, _lib.ptr(mi), _lib.ptr(rel), _lib.ptr(rel), 0.07, 0.05, 0.1, None,
                              None, None, None, None, None, None) == _lib.OK          # P = 0: nothing to do
    assert L.bslam_odom_prepare(None, 0, None, 0, 1, H, W, 2, _lib.ptr(K4), 1000.0, 3.0, 0.07, out, None) == _lib.E_ARG
    assert b"NULL" in L.bslam_last_error()
    assert L.bslam_odom_prepare(out, 2, None, 0, 1, H, W, 2, _lib.ptr(K4), 1000.0, 3.0, 0.07, out, None) == _lib.E_ARG
    assert L.bslam_odom_prepare(out, 0, None, 0, 1, 8, 8, 5, _lib.ptr(K4), 1000.0, 3.0, 0.07, out, None) == _lib.E_ARG
    assert L.bslam_odom_prepare(out, 0, None, 0, 1, H, W, 2, _lib.ptr(K4), 0.0, 3.0, 0.07, out, None) == _lib.E_ARG
    assert L.bslam_odom_prepare(None, 0, None, 0, 0, H, W, 2, _lib.ptr(K4), 1000.0, 3.0, 0.07, None, None) == _lib.OK
    assert L.bslam_odom_linearize(out, 2, _lib.ptr(pairs), 1, H, W, 2, 2, _lib.ptr(K4), 0, 0.07, 0.05, 0.1, _lib.ptr(init), out, out,
                                  None) == _lib.E_ARG and b"level" in L.bslam_last_error()
    # gridDim.y limits: frames per prepare call, pairs per track / linearize call
    assert L.bslam_odom_prepare(out, 0, None, 0, 65536, H, W, 2, _lib.ptr(K4), 1000.0, 3.0, 0.07, out, None) == _lib.E_ARG
    assert track(P=65536) == _lib.E_ARG and b"65535" in L.bslam_last_error()
    assert L.bslam_odom_workspace_bytes(0, H, W, 2) == 0 and L.bslam_odom_workspace_bytes(3, 8, 8, 5) == 0
    assert L.bslam_odom_workspace_bytes(3, 480, 640, 3) >= 3 * 300 * 29 * 8


# Huber parameter sets (depth_outlier_trunc, depth_huber_delta, intensity_huber_delta) and the branches each puts at
# least 30 % of the inliers in, for the residual of each method: on the cavity pair below at the identity pose the
# point-to-plane residuals stay under 0.05 and 90 % of the photometric ones under 0.1, so the defaults exercise the
# quadratic branch only; (0.07, 0.002, 0.01) splits both residuals of the hybrid and the point-to-plane residual, and
# sends 89 % of the intensity residuals to the linear branch; deltas of 0 put every non-zero residual in the linear
# branch, 1e3 every residual in the quadratic one.
HUBER_SETS = {(0.07, 0.05, 0.1): {R.POINT_TO_PLANE: {"depth": "q"}, R.INTENSITY: {"intensity": "q"}, R.HYBRID: {"intensity": "q", "depth": "q"}},
              (0.07, 0.002, 0.01): {R.POINT_TO_PLANE: {"depth": "ql"}, R.INTENSITY: {"intensity": "l"}, R.HYBRID: {"intensity": "ql", "depth": "ql"}},
              (0.07, 0.0, 0.0): {R.POINT_TO_PLANE: {"depth": "l"}, R.INTENSITY: {"intensity": "l"}, R.HYBRID: {"intensity": "l", "depth": "l"}},
              (0.07, 1e3, 1e3): {R.POINT_TO_PLANE: {"depth": "q"}, R.INTENSITY: {"intensity": "q"}, R.HYBRID: {"intensity": "q", "depth": "q"}}}


@pytest.fixture(scope="module")
def cavity_pair():
    E = S.cavity_sweep(1000)[:2]
    d, c = S.render(S.Cavity(), E, K=S.K_640)
    return R.Frames(d.numpy(), c.numpy(), S.K_640, 2), E[1] @ np.linalg.inv(E[0])


@pytest.mark.parametrize("params", list(HUBER_SETS), ids=lambda p: "-".join(map(str, p)))
@pytest.mark.parametrize("method", [R.POINT_TO_PLANE, R.INTENSITY, R.HYBRID])
def test_linearize_matches_float64_restatement(cavity_pair, method, params):
    """the mirror's 29 sums against odometry_ref.linearize_f64, an independent float64 evaluation of the same
    linearisation.  Tolerance: linearize_f64's `tol`, derived there from the float32 rounding of J, r and the Huber terms
    (running error analysis, <= 24 roundings of u = 2^-24 each relative to the operands' magnitudes) plus the whole terms
    of the pixels whose projection or rejection decision lies within that bound of its threshold.  Measured over these
    cases: the differences reach at most 4.5 % of the bound, the bound at most 0.35 % of the largest entry of AᵀA, and
    at most 0.19 % of the inliers are ambiguous."""
    fr, truth = cavity_pair
    for level, T in ((0, np.eye(4)), (1, truth)):
        ref = fr.linearize(0, 1, level, T, method, params)
        f = R.linearize_f64(fr, 0, 1, level, T, method, params)
        assert f["inliers"] > 50000 >> (2 * level), level
        assert abs(ref[28] - f["sums"][28]) <= f["ambiguous"], (level, ref[28], f["sums"][28], f["ambiguous"])
        assert np.all(np.abs(ref[:28] - f["sums"][:28]) <= f["tol"][:28]), (level, np.abs(ref - f["sums"]) / f["tol"])
        # the bound stays far below a wrong branch's effect: 1 % of the largest entry of AᵀA (measured 0.35 %)
        assert np.all(f["tol"][:21] <= 1e-2 * np.abs(f["sums"][:21]).max()), level
        if level == 0:                    # the branch coverage this set claims (identity pose, as in HUBER_SETS)
            n = f["inliers"]
            for name, claim in HUBER_SETS[params][method].items():
                quad, lin = f["branches"][name]
                assert quad + lin == n
                if "q" in claim:
                    assert quad >= 0.3 * n, (name, quad, n)
                if "l" in claim:
                    assert lin >= 0.3 * n, (name, lin, n)
            if params[1] == 0.0:          # all-linear with delta 0: no gradient, no loss
                assert np.all(ref[21:28] == 0) and np.all(f["sums"][21:28] == 0)
