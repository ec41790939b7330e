"""Multi-scale RGB-D odometry on the GPU: Open3D's tensor `t.pipelines.odometry.rgbd_odometry_multi_scale`
(point-to-plane, intensity and hybrid), which the reference's `_compute_vo_o3d` (N/3DM/visual_odometry.py:97-120)
calls for every frame pair, and the batched `rgbd_odometry_sequence` for offline VO over a recorded sequence.

Same names, signature and defaults as Open3D, so a call site can switch imports.  The kernels are in
csrc/bslam_odometry.cu; their semantics are written down in the CPU reference tests/odometry_ref.c.  Parity with
Open3D itself is unpinned (restated from knowledge of its source; DESIGN.md section 7 lists the recalled details).
Frames are duck-typed like the rest of the package: `.depth` [H,W] uint16 (raw, divided by depth_scale) or float32,
`.color` [H,W,3] uint8 or float32 in [0, 1] (only read by the intensity methods); NumPy or torch, CPU or CUDA.
"""
from __future__ import annotations

import enum
from dataclasses import dataclass

import numpy as np

from . import _lib, ops
from .geometry import to_numpy


class Method(enum.IntEnum):
    PointToPlane = 0
    Intensity = 1
    Hybrid = 2


@dataclass
class OdometryConvergenceCriteria:
    max_iteration: int
    relative_rmse: float = 1e-6
    relative_fitness: float = 1e-6


@dataclass
class OdometryLossParams:
    depth_outlier_trunc: float = 0.07
    depth_huber_delta: float = 0.05
    intensity_huber_delta: float = 0.1


@dataclass
class OdometryResult:
    transformation: np.ndarray      # 4x4 float64, source -> target
    inlier_rmse: float
    fitness: float


@dataclass
class OdometrySequenceResult:
    """pair i tracks frame i -> frame i + 1; CUDA tensors"""
    transformations: object         # [F-1,4,4] float64
    inlier_rmse: object             # [F-1] float64
    fitness: object                 # [F-1] float64
    iterations: object              # [F-1,L] int32, evaluations per criteria entry (coarsest level first)
    status: object                  # [F-1] int32: 0 = ok, 1 = singular system (the pose is the one before it)


_EYE = np.eye(4)
_EYE.setflags(write=False)
_DEFAULT_CRITERIA = (OdometryConvergenceCriteria(10), OdometryConvergenceCriteria(5), OdometryConvergenceCriteria(3))
_SEQUENCE_CHUNK = 64                # frames prepared at a time by rgbd_odometry_sequence (consecutive chunks share one)


def _intrinsics(intrinsics):
    K = intrinsics.intrinsic_matrix if hasattr(intrinsics, "intrinsic_matrix") else intrinsics
    K = np.asarray(to_numpy(K.numpy() if hasattr(K, "numpy") and not hasattr(K, "detach") else K), dtype=np.float64)
    if K.shape != (3, 3):
        raise RuntimeError("rgbd_odometry: intrinsics must be a 3x3 matrix")
    return np.array([K[0, 0], K[1, 1], K[0, 2], K[1, 2]], dtype=np.float64)


def _criteria(criteria_list):
    crit = [c if isinstance(c, OdometryConvergenceCriteria) else OdometryConvergenceCriteria(int(c)) for c in criteria_list]
    if not crit:
        raise RuntimeError("rgbd_odometry: criteria_list must not be empty")
    return (np.array([c.max_iteration for c in crit], np.int32), np.array([c.relative_fitness for c in crit], np.float64),
            np.array([c.relative_rmse for c in crit], np.float64))


def _as_images(x, kind, dev, lead):
    """-> (contiguous CUDA tensor, dtype code) of a depth ([..,H,W], uint16 / float32) or colour ([..,H,W,3], uint8 /
    float32) image stack; `lead` = number of leading frame dims"""
    torch = _lib.require_cuda()
    name = ops._dtype_name(x)
    table = {"depth": {"uint16": (torch.uint16, 0), "float32": (torch.float32, 1)},
             "color": {"uint8": (torch.uint8, 0), "float32": (torch.float32, 1)}}[kind]
    if name not in table:
        raise RuntimeError(f"rgbd_odometry: unsupported {kind} dtype {name} (depth: uint16 / float32, color: uint8 / float32)")
    dtype, code = table[name]
    t = ops.as_cuda(x, dtype, dev)
    if kind == "depth" and t.dim() == lead + 3 and t.shape[-1] == 1:
        t = t[..., 0]
    if t.dim() != lead + (2 if kind == "depth" else 3) or (kind == "color" and t.shape[-1] != 3):
        raise RuntimeError(f"rgbd_odometry: {kind} has shape {tuple(t.shape)}")
    return t.contiguous(), code


def _device_of(*xs):
    for x in xs:
        if getattr(x, "is_cuda", False):
            return x.device
    return None


class _Tracker:
    """prepared-frame buffer and workspace for one image size / level count / method"""

    def __init__(self, H, W, K, depth_scale, depth_max, criteria_list, method, params, dev):
        self.torch = _lib.require_cuda()
        self.L = _lib.load()
        self.H, self.W, self.K, self.dev = int(H), int(W), K, ops._device(dev)
        self.max_iter, self.rel_fit, self.rel_rmse = _criteria(criteria_list)
        self.levels = len(self.max_iter)
        self.method = int(Method(method))
        self.params = params
        self.depth_scale, self.depth_max = float(depth_scale), float(depth_max)
        self.frame_bytes = self.L.bslam_odom_frame_bytes(self.H, self.W, self.levels)
        if self.frame_bytes == 0:
            raise RuntimeError(f"[rgbd_odometry] Unsupported image format. ({self.H} x {self.W} has no {self.levels} levels of at least 1 x 1)")
        self.frames = None

    def prepare(self, depth, color, F):
        """(re)fill the buffer with F frames (CUDA tensors from _as_images; frame k of the stack is frame k)"""
        torch = self.torch
        n = F * self.frame_bytes // 4
        if self.frames is None or self.frames.numel() < n:
            self.frames = torch.empty(max(n, 1), dtype=torch.float32, device=self.dev)
        self.prepare_at(0, depth, color, F)

    def prepare_at(self, f0, depth, color, F):
        (d, dcode), (c, ccode) = depth, color if color is not None else (None, 0)
        p = self.params
        out = self.torch.narrow(self.frames, 0, f0 * self.frame_bytes // 4, F * self.frame_bytes // 4) if F else None
        with self.torch.cuda.device(self.dev):
            _lib.check(self.L.bslam_odom_prepare(_lib.ptr(d), dcode, _lib.ptr(c), ccode, F, self.H, self.W, self.levels, _lib.ptr(self.K),
                                                 self.depth_scale, self.depth_max, float(p.depth_outlier_trunc), _lib.ptr(out),
                                                 _lib.stream_ptr(self.dev)))

    def track(self, F, pairs, inits, T, rf, iters, status):
        torch = self.torch
        P = len(pairs)
        p = self.params
        ws = torch.empty(max(self.L.bslam_odom_workspace_bytes(P, self.H, self.W, self.levels), 1), dtype=torch.uint8, device=self.dev)
        h_pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        h_init = np.ascontiguousarray(inits, dtype=np.float64).reshape(-1, 16)
        with torch.cuda.device(self.dev):
            _lib.check(self.L.bslam_odom_track(_lib.ptr(self.frames), F, _lib.ptr(h_pairs), P, self.H, self.W, self.levels, _lib.ptr(self.K),
                                               self.method, _lib.ptr(self.max_iter), _lib.ptr(self.rel_fit), _lib.ptr(self.rel_rmse),
                                               float(p.depth_outlier_trunc), float(p.depth_huber_delta), float(p.intensity_huber_delta),
                                               _lib.ptr(h_init), _lib.ptr(T), _lib.ptr(rf), _lib.ptr(iters), _lib.ptr(status), _lib.ptr(ws),
                                               _lib.stream_ptr(self.dev)))


def _needs_color(method):
    return Method(method) != Method.PointToPlane


def rgbd_odometry_multi_scale(source, target, intrinsics, init_source_to_target=_EYE, depth_scale: float = 1000.0, depth_max: float = 3.0,
                              criteria_list=_DEFAULT_CRITERIA, method=Method.Hybrid, params: OdometryLossParams = OdometryLossParams()):
    """Open3D `t.pipelines.odometry.rgbd_odometry_multi_scale`: the transform taking `source` points into `target`'s
    camera frame, by Gauss-Newton over len(criteria_list) pyramid levels (criteria_list[0] = the coarsest).  Raises
    RuntimeError("Singular 6x6 linear system detected, tracking failed.") like Open3D.  Synchronises once."""
    torch = _lib.require_cuda()
    dev = _device_of(source.depth, target.depth)
    ds, dt = _as_images(source.depth, "depth", dev, 0), _as_images(target.depth, "depth", dev, 0)
    if ds[0].shape != dt[0].shape:
        raise RuntimeError(f"[rgbd_odometry] Unsupported image format. (source {tuple(ds[0].shape)}, target {tuple(dt[0].shape)})")
    H, W = ds[0].shape
    cs = ct = None
    if _needs_color(method):
        if source.color is None or target.color is None:
            raise RuntimeError(f"rgbd_odometry: {Method(method).name} needs the colour of both frames")
        cs, ct = _as_images(source.color, "color", dev, 0), _as_images(target.color, "color", dev, 0)
        if cs[0].shape[:2] != (H, W) or ct[0].shape[:2] != (H, W):
            raise RuntimeError("[rgbd_odometry] Unsupported image format. (colour and depth sizes differ)")
    tr = _Tracker(H, W, _intrinsics(intrinsics), depth_scale, depth_max, criteria_list, method, params, dev)
    tr.frames = torch.empty(2 * tr.frame_bytes // 4, dtype=torch.float32, device=tr.dev)
    tr.prepare_at(0, ds, cs, 1)
    tr.prepare_at(1, dt, ct, 1)
    T = torch.empty((1, 4, 4), dtype=torch.float64, device=tr.dev)
    rf = torch.empty((1, 2), dtype=torch.float64, device=tr.dev)
    iters = torch.empty((1, tr.levels), dtype=torch.int32, device=tr.dev)
    status = torch.empty(1, dtype=torch.int32, device=tr.dev)
    init = np.asarray(to_numpy(init_source_to_target.numpy() if hasattr(init_source_to_target, "numpy") and not hasattr(init_source_to_target, "detach")
                               else init_source_to_target), dtype=np.float64).reshape(4, 4)
    tr.track(2, [(0, 1)], init[None], T, rf, iters, status)
    host = torch.cat([T.reshape(-1), rf.reshape(-1), status.to(torch.float64)]).cpu().numpy()
    if host[18] != 0:
        raise RuntimeError("Singular 6x6 linear system detected, tracking failed.")
    return OdometryResult(host[:16].reshape(4, 4).copy(), float(host[16]), float(host[17]))


def rgbd_odometry_sequence(depth, color, intrinsics, inits=None, depth_scale: float = 1000.0, depth_max: float = 3.0,
                           criteria_list=_DEFAULT_CRITERIA, method=Method.Hybrid, params: OdometryLossParams = OdometryLossParams()):
    """Tracks every consecutive pair i -> i + 1 of depth [F,H,W] (color [F,H,W,3] | None) from inits [F-1,4,4] (None =
    identity), with the semantics of rgbd_odometry_multi_scale: pair i's result has the bits of the single call.  Frames
    are prepared 64 at a time, consecutive chunks sharing one frame, so device memory does not grow with F.  Singular
    pairs are reported in `status` instead of raised.  -> OdometrySequenceResult of CUDA tensors (no synchronisation)."""
    torch = _lib.require_cuda()
    dev = ops._device(_device_of(depth))
    dname = ops._dtype_name(depth)
    shape = tuple(depth.shape)
    if len(shape) != 3:
        raise RuntimeError(f"rgbd_odometry_sequence: depth must be [F,H,W], got {shape}")
    F, H, W = shape
    if _needs_color(method) and color is None and F > 1:
        raise RuntimeError(f"rgbd_odometry_sequence: {Method(method).name} needs colour")
    tr = _Tracker(H, W, _intrinsics(intrinsics), depth_scale, depth_max, criteria_list, method, params, dev)
    P = max(F - 1, 0)
    I = np.broadcast_to(_EYE, (P, 4, 4)) if inits is None else np.asarray(to_numpy(inits), dtype=np.float64).reshape(-1, 4, 4)
    if I.shape[0] != P:
        raise RuntimeError(f"rgbd_odometry_sequence: {F} frames need {P} inits, got {I.shape[0]}")
    T = torch.empty((P, 4, 4), dtype=torch.float64, device=tr.dev)
    rf = torch.empty((P, 2), dtype=torch.float64, device=tr.dev)
    iters = torch.empty((P, tr.levels), dtype=torch.int32, device=tr.dev)
    status = torch.empty(P, dtype=torch.int32, device=tr.dev)
    for s in range(0, P, _SEQUENCE_CHUNK - 1):
        e = min(s + _SEQUENCE_CHUNK, F)
        n = e - s
        d = _as_images(depth[s:e], "depth", tr.dev, 1)
        if d[1] != {"uint16": 0, "float32": 1}[dname] or tuple(d[0].shape[1:]) != (H, W):
            raise RuntimeError("rgbd_odometry_sequence: inconsistent depth")
        c = _as_images(color[s:e], "color", tr.dev, 1) if (color is not None and _needs_color(method)) else None
        tr.prepare(d, c, n)
        tr.track(n, [(i, i + 1) for i in range(n - 1)], I[s:s + n - 1], T[s:s + n - 1], rf[s:s + n - 1], iters[s:s + n - 1], status[s:s + n - 1])
    return OdometrySequenceResult(T, rf[:, 0], rf[:, 1], iters, status)
