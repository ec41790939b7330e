"""3DM reconstruction entry points -- drop-in for the reference's `N/3DM/tsdf.py`.

`TSDF` keeps the reference signatures (tsdf.py:5-52): `TSDF(voxel_length, sdf_trunc)`, `.tsdf`,
`build_3D_map`, `build_copy_3D_map`, `extract_pcd`, `extract_mesh`, `save_pcd`, `save_mesh`.
Where the reference wraps Open3D's CPU `ScalableTSDFVolume`, `.tsdf` here is a
`DenseTSDFVolume`: the dense N^3 equivalent (Open3D UniformTSDFVolume semantics) living
brick-ordered in B200 HBM and driven by the hand-written kernels in csrc/.  Extra, non-breaking
keyword arguments choose the box (`resolution`, `origin`), colour integration and the device.
Both volumes can be ray cast: `DenseTSDFVolume.raycast` and `MAP.synthesize_model_frame` render depth, vertex,
normal and colour maps of the map from a pose (csrc/bslam_raycast.cu).
"""
from __future__ import annotations

import copy as _copy
import ctypes as C

import numpy as np

from . import _lib, ops
from .geometry import PointCloud, TriangleMesh, intrinsic_params, to_numpy
from .odometry import Method


class DenseTSDFVolume:
    """Dense TSDF box on one GPU.  Method names follow Open3D's volume (`integrate`,
    `extract_triangle_mesh`, `extract_point_cloud`, `reset`) so reference code that reaches through
    `TSDF.tsdf` keeps working.

    resolution : int or (nx, ny, nz) voxels;  origin : world position of the grid corner
    (default: the cube is centred on the world origin);  gz0 : global z index of local plane 0
    (z-slab sharding, multiple of 8);  color : integrate RGB8 like the reference's
    `TSDFVolumeColorType.RGB8` (tsdf.py:10).
    """

    def __init__(self, voxel_length: float, sdf_trunc: float, resolution=512, origin=None, color: bool = True,
                 device=None, gz0: int = 0, z_total: int | None = None, z_interleave: int = 1,
                 unit_activation: bool = False, unit_resolution: int = 32, depth_sampling_stride: int = 8, unit_arithmetic: bool = False):
        torch = _lib.require_cuda()
        self._L = _lib.load()
        self.device = ops._device(device)
        if np.isscalar(resolution):
            resolution = (int(resolution),) * 3
        self.nx, self.ny, self.nz = (int(r) for r in resolution)
        self.voxel_length = float(voxel_length)
        self.sdf_trunc = float(sdf_trunc)
        self.gz0 = int(gz0)
        self.z_total = int(z_total) if z_total is not None else self.nz
        if origin is None:
            origin = (-0.5 * self.nx * self.voxel_length, -0.5 * self.ny * self.voxel_length, -0.5 * self.z_total * self.voxel_length)
        self.origin = np.ascontiguousarray(origin, dtype=np.float64)
        self.color = bool(color)
        nbytes = self._L.bslam_tsdf_storage_bytes(self.nx, self.ny, self.nz, int(self.color))
        self._storage = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_create(C.byref(self._h), self.nx, self.ny, self.nz, self.gz0, self.voxel_length,
                                                 self.sdf_trunc, _lib.ptr(self.origin), int(self.color), self.device.index,
                                                 _lib.ptr(self._storage), _lib.stream_ptr(self.device)))
        self.z_interleave = int(z_interleave)
        if self.z_interleave != 1:
            _lib.check(self._L.bslam_tsdf_set_z_interleave(self._h, self.z_interleave))
        self.unit_activation = bool(unit_activation)
        self.unit_arithmetic = bool(unit_arithmetic) and not self.unit_activation
        if self.unit_activation:
            self.set_unit_activation(unit_resolution, depth_sampling_stride)
        elif self.unit_arithmetic:
            # dense rule (every voxel of the box) with the reference's per-unit arithmetic: voxel centres and the float32 z
            # recurrence evaluated per 32^3 unit like ScalableTSDFVolume's units -- on the voxels of the units the reference
            # would have activated the result is the reference's, bit for bit (oracle: integrate_scalable(all_units=True))
            _lib.check(self._L.bslam_tsdf_set_unit_activation(self._h, int(unit_resolution), -1, int(self.z_total)))
            self.unit_resolution, self.depth_sampling_stride = int(unit_resolution), -1
        self.frames_integrated = 0

    def set_unit_activation(self, unit_resolution: int = 32, depth_sampling_stride: int = 8):
        """ScalableTSDFVolume semantics (what the reference's `TSDF()` builds, tsdf.py:7-12): a frame
        integrates only the unit_resolution^3 units its stride-sampled depth points (+- sdf_trunc)
        activate; 0 switches back to the dense UniformTSDFVolume rule.  Raises RuntimeError when the
        box does not consist of whole units on the world unit grid."""
        _lib.check(self._L.bslam_tsdf_set_unit_activation(self._h, int(unit_resolution), int(depth_sampling_stride), int(self.z_total)))
        self.unit_activation = unit_resolution > 0
        self.unit_resolution, self.depth_sampling_stride = int(unit_resolution), int(depth_sampling_stride)

    @staticmethod
    def unit_aligned(resolution, voxel_length, origin, unit_resolution: int = 32) -> bool:
        """can a box with this geometry run in unit-activation mode?"""
        res = (int(resolution),) * 3 if np.isscalar(resolution) else tuple(int(r) for r in resolution)
        ul = float(voxel_length) * unit_resolution
        o = np.asarray(origin, dtype=np.float64)
        return all(r % unit_resolution == 0 for r in res) and bool(np.all(np.abs(np.rint(o / ul) * ul - o) <= 1e-9 * np.maximum(1.0, np.abs(o))))

    def storage_layers(self):
        """views of the storage as brick layers: dict(vox [nbz, bytes], flags [nbz, nbx*nby][, color [nbz, bytes]]).
        A brick layer (all bricks with one bz) is contiguous in each region -- the unit z-re-sharding moves."""
        off = (C.c_size_t * 4)()
        _lib.check(self._L.bslam_tsdf_layout(self._h, off))
        nbx, nby, nbz = (self.nx + 7) // 8, (self.ny + 7) // 8, (self.nz + 7) // 8
        nb = nbx * nby * nbz
        out = {"vox": self._storage[off[0]:off[0] + nb * 4096].view(nbz, nbx * nby * 4096),
               "flags": self._storage[off[2]:off[2] + nb].view(nbz, nbx * nby)}
        if self.color:
            out["color"] = self._storage[off[1]:off[1] + nb * 6144].view(nbz, nbx * nby * 6144)
        return out

    # ------------------------------------------------------------------ lifetime
    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._L.bslam_tsdf_destroy(h)
            except Exception:
                pass
            self._h = C.c_void_p()

    def __deepcopy__(self, memo):
        """`deepcopy(self.tsdf)` of tsdf.py:24 -> device-to-device clone."""
        torch = _lib.require_cuda()
        other = DenseTSDFVolume(self.voxel_length, self.sdf_trunc, (self.nx, self.ny, self.nz), self.origin, self.color,
                                self.device, self.gz0, self.z_total, self.z_interleave, self.unit_activation,
                                getattr(self, "unit_resolution", 32), max(getattr(self, "depth_sampling_stride", 8), 1),
                                unit_arithmetic=self.unit_arithmetic)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_copy(self._h, other._h, _lib.stream_ptr(self.device)))
        other.frames_integrated = self.frames_integrated
        return other

    def reset(self):
        torch = _lib.require_cuda()
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_reset(self._h, _lib.stream_ptr(self.device)))
        self.frames_integrated = 0

    # ------------------------------------------------------------------ integration
    def _check_frame(self, depth, color, intrinsic):
        W, H, fx, fy, cx, cy = intrinsic_params(intrinsic)
        if depth.dim() == 2:
            depth = depth.unsqueeze(0)
        if depth.dim() != 3 or depth.shape[1] != H or depth.shape[2] != W:
            raise RuntimeError("[DenseTSDFVolume::Integrate] Unsupported image format.")
        if self.color:
            if color is None or color.numel() != depth.shape[0] * H * W * 3:
                raise RuntimeError("[DenseTSDFVolume::Integrate] Unsupported image format.")
        return depth, (W, H, fx, fy, cx, cy)

    def integrate(self, rgbd, intrinsic, extrinsic, zmarch: int = _lib.ZMARCH_BRICK):
        """Open3D `volume.integrate(rgbd, intrinsic, extrinsic)` -- one frame (tsdf.py:22).

        rgbd: object with `.depth` (H,W f32 metres) and `.color` (H,W,3 u8); numpy, torch CPU/CUDA
        or Open3D images.  extrinsic: 4x4 world->camera (f64).
        """
        torch = _lib.require_cuda()
        name = ops._dtype_name(rgbd.depth)
        if name != "float32":
            raise RuntimeError("[DenseTSDFVolume::Integrate] Unsupported image format.")
        depth = ops.as_cuda(rgbd.depth, torch.float32, self.device)
        color = None
        if self.color:
            c = getattr(rgbd, "color", None)
            if c is None or ops._dtype_name(c) != "uint8":
                raise RuntimeError("[DenseTSDFVolume::Integrate] Unsupported image format.")
            color = ops.as_cuda(c, torch.uint8, self.device)
        self.integrate_batch(depth, color, intrinsic, np.asarray(to_numpy(extrinsic), dtype=np.float64).reshape(1, 4, 4), zmarch=zmarch)

    def integrate_batch(self, depth, color, intrinsic, extrinsics, zmarch: int = _lib.ZMARCH_BRICK, update_counts=None, dry_run=False):
        """F frames in order (the `update_map_after_pg` replay shape, slam_utils.py:124-135).

        depth [F,H,W] f32 CUDA (or anything `as_cuda` takes), color [F,H,W,3] u8 or None,
        extrinsics [F,4,4] f64 world->camera.  update_counts: optional u64-as-i64 CUDA tensor [F]
        accumulating the number of voxels updated per frame.
        """
        torch = _lib.require_cuda()
        depth = ops.as_cuda(depth, torch.float32, self.device)
        if color is not None:
            color = ops.as_cuda(color, torch.uint8, self.device)
        depth, (W, H, fx, fy, cx, cy) = self._check_frame(depth, color if self.color else None, intrinsic)
        F = depth.shape[0]
        E = np.ascontiguousarray(np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 16))
        if E.shape[0] != F:
            raise RuntimeError(f"integrate_batch: {F} frames but {E.shape[0]} extrinsics")
        K = np.array([fx, fy, cx, cy], dtype=np.float64)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_integrate(self._h, _lib.ptr(depth), _lib.ptr(color) if self.color else None, F, H, W,
                                                    _lib.ptr(K), _lib.ptr(E), int(zmarch), _lib.ptr(update_counts), int(bool(dry_run)),
                                                    _lib.stream_ptr(self.device)))
        if not dry_run:
            self.frames_integrated += F

    def integrate_u16_batch(self, depth_u16, color, intrinsic, extrinsics, depth_scale: float = 1000.0, depth_trunc: float = 3.0,
                            scratch=None, update_counts=None):
        """F uint16 frames in order with the 3DM depth conversion (slam_utils.py:212-220) fused into
        the integration's first pass.  depth_u16 [F,H,W] uint16 CUDA; scratch: optional f32 CUDA
        tensor with >= F*H*W elements that receives the converted frames (returned)."""
        torch = _lib.require_cuda()
        if ops._dtype_name(depth_u16) != "uint16":
            raise RuntimeError("[DenseTSDFVolume::Integrate] Unsupported image format.")
        depth_u16 = ops.as_cuda(depth_u16, torch.uint16, self.device)
        if color is not None:
            color = ops.as_cuda(color, torch.uint8, self.device)
        depth_u16, (W, H, fx, fy, cx, cy) = self._check_frame(depth_u16, color if self.color else None, intrinsic)
        F = depth_u16.shape[0]
        E = np.ascontiguousarray(np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 16))
        if E.shape[0] != F:
            raise RuntimeError(f"integrate_u16_batch: {F} frames but {E.shape[0]} extrinsics")
        if scratch is None or scratch.numel() < F * H * W:
            scratch = torch.empty((F, H, W), dtype=torch.float32, device=self.device)
        K = np.array([fx, fy, cx, cy], dtype=np.float64)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_integrate_u16(self._h, _lib.ptr(depth_u16), float(depth_scale), float(depth_trunc or 0.0),
                                                        _lib.ptr(scratch), _lib.ptr(color) if self.color else None, F, H, W,
                                                        _lib.ptr(K), _lib.ptr(E), _lib.ptr(update_counts), _lib.stream_ptr(self.device)))
        self.frames_integrated += F
        return scratch

    # ------------------------------------------------------------------ two-stream launch pipeline
    def prep_stream(self):
        """side stream for the part of a launch that does not touch the volume (conversion, statistics, culling)"""
        torch = _lib.require_cuda()
        if getattr(self, "_prep_stream", None) is None:
            self._prep_stream = torch.cuda.Stream(self.device)
        return self._prep_stream

    def copy_stream(self):
        """side stream on which the streamed entry points bring frames to the device (host copies, NCCL transfers)"""
        torch = _lib.require_cuda()
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(self.device)
        return self._copy_stream

    def prepare_u16(self, depth_u16, intrinsic, extrinsics, scratch, depth_scale: float = 1000.0, depth_trunc: float = 3.0, wait=None):
        """enqueue the preparation of one launch (<= 256 frames; see bslam_tsdf_prepare_u16) on the side stream.
        `wait`: optional callable run with the side stream current (e.g. `work.wait` of an NCCL transfer or
        `lambda: stream.wait_event(ev)`) -- what the frames' arrival is ordered by.  Up to two launches ahead."""
        torch = _lib.require_cuda()
        W, H, fx, fy, cx, cy = intrinsic_params(intrinsic)
        if depth_u16.dim() == 2:
            depth_u16 = depth_u16.unsqueeze(0)
        if (not depth_u16.is_cuda or depth_u16.dtype != torch.uint16 or depth_u16.dim() != 3 or depth_u16.shape[1] != H or depth_u16.shape[2] != W
                or not depth_u16.is_contiguous()):
            raise RuntimeError("[DenseTSDFVolume::Integrate] Unsupported image format.")
        F = depth_u16.shape[0]
        E = np.ascontiguousarray(np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 16))
        if E.shape[0] != F:
            raise RuntimeError(f"prepare_u16: {F} frames but {E.shape[0]} extrinsics")
        if scratch is None or scratch.numel() < F * H * W:
            raise RuntimeError("prepare_u16: the f32 scratch must hold the launch's frames")
        K = np.array([fx, fy, cx, cy], dtype=np.float64)
        ps = self.prep_stream()
        with torch.cuda.device(self.device), torch.cuda.stream(ps):
            if wait is not None:
                wait()
            _lib.check(self._L.bslam_tsdf_prepare_u16(self._h, _lib.ptr(depth_u16), float(depth_scale), float(depth_trunc or 0.0), _lib.ptr(scratch),
                                                      F, H, W, _lib.ptr(K), _lib.ptr(E), C.c_void_p(ps.cuda_stream)))
        self._prepared = getattr(self, "_prepared", [])
        self._prepared.append((F, depth_u16, scratch))      # keep the buffers alive until the launch is integrated

    def integrate_prepared(self, color=None, update_counts=None):
        """enqueue the integration of the oldest prepared launch on the current stream"""
        torch = _lib.require_cuda()
        F, _, _ = self._prepared.pop(0)
        if self.color and color is None:
            raise RuntimeError("[DenseTSDFVolume::Integrate] Unsupported image format.")
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_integrate_prepared(self._h, _lib.ptr(color) if self.color else None, _lib.ptr(update_counts),
                                                             _lib.stream_ptr(self.device)))
        self.frames_integrated += F

    def integrate_streamed(self, chunks, intrinsic, extrinsics, arrive, depth_scale: float = 1000.0, depth_trunc: float = 3.0,
                           update_counts=None, color_staging: bool = False):
        """The two-stream launch pipeline that every streamed entry point runs, chunk k of `chunks` [(f0, f1)] after
        chunk k-1: the arrival of chunk k+2 is enqueued, then the preparation of chunk k+1 on the side stream, then the
        integration of chunk k on the current stream.  The caller says how frames arrive:
            arrive(k, stage, free) -> (depth_u16, color, wait)
        enqueues the arrival of chunk k.  `stage` = (uint16 [n,H,W], f32 [n,H,W], uint8 [n,H,W,3] | None) are the
        staging buffers chunk k may use (the f32 one always receives its converted frames), `free` is the event after
        which the current stream no longer reads them.  It returns the chunk's uint16 frames on the device, its colour
        (or None) and the callable the side stream runs before the preparation (or None)."""
        torch = _lib.require_cuda()
        if not chunks:
            return
        W, H = intrinsic_params(intrinsic)[:2]
        E = np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 4, 4)
        with torch.cuda.device(self.device):
            main = torch.cuda.current_stream(self.device)
            stage = self._staging(max(f1 - f0 for f0, f1 in chunks), H, W, color_staging)
            free = self._stage_free
            self.prep_stream().wait_stream(main)         # the frames (and earlier launches) are ordered by the current stream
            arrived = {}

            def prep(k):
                f0, f1 = chunks[k]
                self.prepare_u16(arrived[k][0], intrinsic, E[f0:f1], stage[k % 3][1], depth_scale, depth_trunc, wait=arrived[k][2])

            for k in range(min(2, len(chunks))):
                arrived[k] = arrive(k, stage[k % 3], free[k % 3])
            prep(0)
            for k, (f0, f1) in enumerate(chunks):
                if k + 2 < len(chunks):
                    arrived[k + 2] = arrive(k + 2, stage[(k + 2) % 3], free[(k + 2) % 3])
                if k + 1 < len(chunks):
                    prep(k + 1)
                self.integrate_prepared(arrived.pop(k)[1], None if update_counts is None else update_counts[f0:f1])
                free[k % 3] = torch.cuda.Event()
                free[k % 3].record(main)

    def integrate_u16_chunks(self, depth_u16, color, intrinsic, extrinsics, chunks, depth_scale: float = 1000.0, depth_trunc: float = 3.0,
                             update_counts=None):
        """device-resident uint16 frames, launch after launch through the two-stream pipeline: chunk k+1 is converted and
        culled on the side stream while chunk k integrates (`chunks`: [(f0, f1)], each <= 256 frames)."""

        def arrive(k, stage, free):      # already on the device and ordered by the current stream
            f0, f1 = chunks[k]
            return depth_u16[f0:f1], None if color is None else color[f0:f1], None

        self.integrate_streamed(chunks, intrinsic, extrinsics, arrive, depth_scale, depth_trunc, update_counts)

    @staticmethod
    def stream_chunks(F: int, chunk: int = 256, ramp=(32, 64, 128), multiple_of: int = 1):
        """[(f0, f1)] for streamed integration: a short ramp first, so that the compute stream starts
        after a 32-frame copy instead of a full chunk, then near-equal chunks of at most `chunk`.
        multiple_of: chunk sizes (except the last) are multiples of it (even split over N ranks)."""
        out, f = [], 0
        q = max(1, int(multiple_of))
        for r in ramp:
            r = -(-r // q) * q
            if F - f <= chunk or r >= chunk:
                break
            out.append((f, f + r))
            f += r
        rest = F - f
        if rest > 0:
            n = -(-rest // chunk)
            units = -(-rest // q)                      # units of q frames, spread over n chunks
            base, extra = divmod(units, n)
            for i in range(n):
                m = min((base + (1 if i < extra else 0)) * q, F - f)
                if m > 0:
                    out.append((f, f + m))
                    f += m
        return out

    def _staging(self, n, H, W, use_color, count=3):
        torch = _lib.require_cuda()
        key = (n, H, W, use_color, count)
        if getattr(self, "_stage_key", None) != key:
            dev = self.device
            self._stage = [(torch.empty((n, H, W), dtype=torch.uint16, device=dev),
                            torch.empty((n, H, W), dtype=torch.float32, device=dev),
                            torch.empty((n, H, W, 3), dtype=torch.uint8, device=dev) if use_color else None)
                           for _ in range(count)]
            self._stage_key = key
            # event per staging buffer: the compute stream is done with it.  Kept across calls, so the
            # first copies of the next replay overlap the tail of this one instead of waiting for it.
            # Fresh buffers start with an event recorded on the allocating (current) stream: the caching
            # allocator may hand out a block whose previous user's kernels are still queued there, and
            # the first side-stream copy / NCCL receive into it must wait for them.
            self._stage_free = []
            for _ in range(count):
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(dev))
                self._stage_free.append(ev)
        return self._stage

    def integrate_host(self, depth_u16, color, intrinsic, extrinsics, depth_scale: float = 1000.0, depth_trunc: float = 3.0,
                       chunk: int = 256, update_counts=None):
        """Frames that live in HOST memory (ideally pinned): uint16 depth [F,H,W] (+ uint8 colour
        [F,H,W,3]) are streamed to the device in chunks on a side stream, double-buffered, while
        the previous chunk is converted (a4, fused) and integrated (K3) on the current stream -- the
        shape of `update_map_after_pg` once the PNGs are decoded.  Frame order is preserved.
        """
        torch = _lib.require_cuda()
        if ops._dtype_name(depth_u16) != "uint16":
            raise RuntimeError("[DenseTSDFVolume::IntegrateHost] Unsupported image format.")
        if not hasattr(depth_u16, "is_cuda"):
            depth_u16 = torch.from_numpy(np.ascontiguousarray(to_numpy(depth_u16)))
        if color is not None and not hasattr(color, "is_cuda"):
            color = torch.from_numpy(np.ascontiguousarray(to_numpy(color)))
        use_color = self.color and color is not None
        if self.color and color is None:
            raise RuntimeError("[DenseTSDFVolume::IntegrateHost] Unsupported image format.")
        chunks = self.stream_chunks(depth_u16.shape[0], chunk)
        cs = self.copy_stream()

        def arrive(k, stage, free):      # H2D of chunk k on the copy stream, once the current stream is done with its buffers
            f0, f1 = chunks[k]
            u16, _, col = stage
            with torch.cuda.stream(cs):
                cs.wait_event(free)
                u16[:f1 - f0].copy_(depth_u16[f0:f1], non_blocking=True)
                if use_color:
                    col[:f1 - f0].copy_(color[f0:f1], non_blocking=True)
                copied = torch.cuda.Event()
                copied.record(cs)
            return u16[:f1 - f0], col[:f1 - f0] if use_color else None, copied.wait

        self.integrate_streamed(chunks, intrinsic, extrinsics, arrive, depth_scale, depth_trunc, update_counts, use_color)

    def count_updates(self, depth, intrinsic, extrinsics, zmarch: int = _lib.ZMARCH_BRICK):
        """U_f of SURVEY.md 8(d): voxels each frame WOULD update (volume untouched) -> i64 [F]."""
        torch = _lib.require_cuda()
        depth = ops.as_cuda(depth, torch.float32, self.device)
        F = 1 if depth.dim() == 2 else depth.shape[0]
        counts = torch.zeros(F, dtype=torch.int64, device=self.device)
        col, self.color = self.color, False
        try:
            self.integrate_batch(depth, None, intrinsic, extrinsics, zmarch=zmarch, update_counts=counts, dry_run=True)
        finally:
            self.color = col
        return counts

    def dry_stats(self, reset: bool = True):
        """culling statistics of the dry runs since the last reset (see bslam_tsdf_dry_stats) -> dict"""
        out = (C.c_ulonglong * 5)()
        _lib.check(self._L.bslam_tsdf_dry_stats(self._h, out, int(bool(reset)), _lib.stream_ptr(self.device)))
        return {"warp_frame_pairs": int(out[0]), "pairs_in_image": int(out[1]), "pairs_updating": int(out[2]), "voxels_tested": int(out[3]),
                "free_pairs": int(out[4])}

    def chain_histogram(self):
        """active bricks of the last integrate launch by number of active frames (32 buckets of 8 frames)"""
        out = (C.c_uint * 32)()
        _lib.check(self._L.bslam_tsdf_chain_histogram(self._h, out, _lib.stream_ptr(self.device)))
        return list(out)

    def set_z_split(self, z_layers_per_warp: int):
        """z layers per integrate warp: 8, 4, 2 or 0 = automatic (see bslam_tsdf_set_z_split)"""
        _lib.check(self._L.bslam_tsdf_set_z_split(self._h, int(z_layers_per_warp)))

    def set_batch(self, frames_per_launch: int):
        """frames per integrate launch (0 = library default, max 256)"""
        _lib.check(self._L.bslam_tsdf_set_batch(self._h, int(frames_per_launch)))

    def profile(self, enable: bool = True):
        """bracket the dominant integrate kernel with CUDA events (bench.py roofline)"""
        _lib.check(self._L.bslam_tsdf_profile(self._h, int(bool(enable))))

    def profile_read(self):
        """-> (accumulated kernel ms, launches) since profile(True); synchronises"""
        ms, n = C.c_double(), C.c_longlong()
        _lib.check(self._L.bslam_tsdf_profile_read(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def profile_read_stages(self):
        """-> ({stage: accumulated ms}, launches) since profile(True): the timeline of the integrate launches"""
        ms, n = (C.c_double * 3)(), C.c_longlong()
        _lib.check(self._L.bslam_tsdf_profile_read_stages(self._h, ms, C.byref(n)))
        return {"depth_stats_a4": ms[0], "marks_culls_order": ms[1], "brick_integrate": ms[2]}, n.value

    def set_clip_check(self, sampling_stride: int = 8):
        """dense mode: count the stride-sampled depth points of every integrated frame that fall outside the
        box (unit-activation mode always does); 0 = off.  See `clip_stats`."""
        _lib.check(self._L.bslam_tsdf_set_clip_check(self._h, int(sampling_stride), int(self.z_total)))

    def clip_stats(self, reset: bool = False):
        """The reference's volume is unbounded, this box is not: -> dict(points, outside, partly_outside) over the
        sampled depth points of the frames integrated so far (synchronises)."""
        out = (C.c_ulonglong * 3)()
        _lib.check(self._L.bslam_tsdf_clip_stats(self._h, out, int(bool(reset)), _lib.stream_ptr(self.device)))
        return {"points": int(out[0]), "outside": int(out[1]), "partly_outside": int(out[2])}

    # ------------------------------------------------------------------ dense views (parity / interchange)
    def export_dense(self, with_color: bool = False):
        """(tsdf, weight[, color]) as [nx,ny,nz] f32 CUDA tensors in Open3D order x*ny*nz + y*nz + z."""
        torch = _lib.require_cuda()
        n = self.nx * self.ny * self.nz
        t = torch.empty(n, dtype=torch.float32, device=self.device)
        w = torch.empty(n, dtype=torch.float32, device=self.device)
        c = torch.empty(n * 3, dtype=torch.float32, device=self.device) if (with_color and self.color) else None
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_export(self._h, _lib.ptr(t), _lib.ptr(w), _lib.ptr(c), _lib.stream_ptr(self.device)))
        shp = (self.nx, self.ny, self.nz)
        out = (t.view(shp), w.view(shp))
        return out + (c.view(shp + (3,)),) if c is not None else out

    def import_dense(self, tsdf, weight, color=None):
        torch = _lib.require_cuda()
        t = ops.as_cuda(tsdf, torch.float32, self.device)
        w = ops.as_cuda(weight, torch.float32, self.device)
        c = ops.as_cuda(color, torch.float32, self.device) if (color is not None and self.color) else None
        if t.numel() != self.nx * self.ny * self.nz or w.numel() != t.numel():
            raise RuntimeError("import_dense: shape mismatch")
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_import(self._h, _lib.ptr(t), _lib.ptr(w), _lib.ptr(c), _lib.stream_ptr(self.device)))

    def export_plane(self, z: int):
        """{tsdf, weight} of local plane z as a [nx, ny, 2] f32 CUDA tensor (slab halo)."""
        torch = _lib.require_cuda()
        p = torch.empty((self.nx, self.ny, 2), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_export_plane(self._h, int(z), _lib.ptr(p), _lib.stream_ptr(self.device)))
        return p

    def export_plane_color(self, z: int):
        """colour of local plane z as a [nx, ny, 3] f32 CUDA tensor in [0, 255] (colour halo of the slab below)."""
        torch = _lib.require_cuda()
        p = torch.empty((self.nx, self.ny, 3), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_export_plane_color(self._h, int(z), _lib.ptr(p), _lib.stream_ptr(self.device)))
        return p

    # ------------------------------------------------------------------ ray casting
    def _raycast_outputs(self, F, H, W, normals, colors):
        torch = _lib.require_cuda()
        dev = self.device
        out = {"depth": torch.empty((F, H, W), dtype=torch.float32, device=dev),
               "vertex": torch.empty((F, H, W, 3), dtype=torch.float32, device=dev)}
        if normals:
            out["normal"] = torch.empty((F, H, W, 3), dtype=torch.float32, device=dev)
        if colors:
            out["color"] = torch.empty((F, H, W, 3), dtype=torch.float32, device=dev)
        return out

    def raycast(self, intrinsic, extrinsics, depth_min: float = 0.0, depth_max: float = 3.0, depth_scale: float = 1.0,
                weight_threshold: float = 0.0, normals: bool = True, colors=None):
        """Render the volume from F poses: one ray per pixel marches the TSDF to its first zero crossing of valid voxels
        (weight >= weight_threshold; != 0 when it is 0) between depth_min and depth_max (metres along the camera z).
        extrinsics: [F,4,4] or one 4x4 world -> camera (f64).  colors: None = when the volume has colour.
        -> dict of CUDA f32 tensors: depth [F,H,W] (z * depth_scale), vertex [F,H,W,3] (camera frame), normal
        [F,H,W,3] (camera frame, unit) when `normals`, color [F,H,W,3] in [0, 1] when colours are asked for; pixels
        whose ray hits nothing are 0.  The volume is not changed (single-box volumes, dims multiples of 8)."""
        torch = _lib.require_cuda()
        W, H, fx, fy, cx, cy = intrinsic_params(intrinsic)
        E = np.ascontiguousarray(np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 16))
        colors = self.color if colors is None else bool(colors)
        out = self._raycast_outputs(E.shape[0], H, W, normals, colors)
        K = np.array([fx, fy, cx, cy], dtype=np.float64)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_raycast(self._h, E.shape[0], H, W, _lib.ptr(K), _lib.ptr(E), float(depth_scale), float(depth_min),
                                                  float(depth_max), float(weight_threshold), _lib.ptr(out["depth"]), _lib.ptr(out["vertex"]),
                                                  _lib.ptr(out.get("normal")), _lib.ptr(out.get("color")), _lib.stream_ptr(self.device)))
        return out

    # ------------------------------------------------------------------ ray casting of z-slabs (ShardedTSDF.raycast)
    def raycast_halo(self, up: bool):
        """what this slab gives a neighbour for `raycast_shade`, packed as bslam_tsdf_raycast_halo_bytes bytes (uint8 CUDA
        tensor): up=True -> its top plane for the slab above, up=False -> its two bottom planes for the slab below; each
        with the colour planes of colour volumes and the brick flags of the layer holding them."""
        torch = _lib.require_cuda()
        zs = [self.nz - 1] if up else [0, 1]
        parts = [self.export_plane(z).view(torch.uint8).reshape(-1) for z in zs]
        if self.color:
            parts += [self.export_plane_color(z).view(torch.uint8).reshape(-1) for z in zs]
        parts.append(self.storage_layers()["flags"][-1 if up else 0])
        return torch.cat(parts)

    def raycast_segment(self, state, slab_z, first: bool, intrinsic, extrinsics, depth_min: float = 0.0, depth_max: float = 3.0,
                        weight_threshold: float = 0.0):
        """one round of the segment march on this slab of the grid cut at planes `slab_z` (bslam_tsdf_raycast_segment);
        state: int32 CUDA tensor of 4 * F * H * W + 1 words, overwritten with this slab's share of the next state."""
        torch = _lib.require_cuda()
        W, H, fx, fy, cx, cy = intrinsic_params(intrinsic)
        E = np.ascontiguousarray(np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 16))
        z = np.ascontiguousarray(slab_z, dtype=np.int32)
        K = np.array([fx, fy, cx, cy], dtype=np.float64)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_raycast_segment(self._h, len(z) - 1, _lib.ptr(z), int(bool(first)), E.shape[0], H, W, _lib.ptr(K), _lib.ptr(E),
                                                          float(depth_min), float(depth_max), float(weight_threshold), _lib.ptr(state),
                                                          _lib.stream_ptr(self.device)))

    def raycast_shade(self, state, slab_z, halo_lo, halo_hi, intrinsic, extrinsics, out, depth_scale: float = 1.0):
        """this slab's share of the maps of the finished rays in `state` (bslam_tsdf_raycast_shade) into the tensors of
        `out` (keys as `raycast`); halo_lo / halo_hi: `raycast_halo` of the slabs below (up=True) / above (up=False)."""
        torch = _lib.require_cuda()
        W, H, fx, fy, cx, cy = intrinsic_params(intrinsic)
        E = np.ascontiguousarray(np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 16))
        z = np.ascontiguousarray(slab_z, dtype=np.int32)
        K = np.array([fx, fy, cx, cy], dtype=np.float64)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_tsdf_raycast_shade(self._h, len(z) - 1, _lib.ptr(z), _lib.ptr(halo_lo), _lib.ptr(halo_hi), E.shape[0], H, W,
                                                        _lib.ptr(K), _lib.ptr(E), float(depth_scale), _lib.ptr(state), _lib.ptr(out["depth"]),
                                                        _lib.ptr(out.get("vertex")), _lib.ptr(out.get("normal")), _lib.ptr(out.get("color")),
                                                        _lib.stream_ptr(self.device)))

    # ------------------------------------------------------------------ extraction
    def mc_count(self, halo_lo=None, halo_hi=None):
        """first phase of the marching cubes: (vertices, triangles) this box will emit (synchronises)"""
        torch = _lib.require_cuda()
        cnt = np.zeros(2, np.int64)
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_mc_count(self._h, _lib.ptr(halo_lo), _lib.ptr(halo_hi), _lib.ptr(cnt), _lib.stream_ptr(self.device)))
        return int(cnt[0]), int(cnt[1])

    def mc_emit(self, verts, keys, cols, tris, halo_lo=None, halo_hi=None, halo_hi_color=None):
        """second phase: write this box's mesh into caller tensors (slices of a gathered mesh, for example):
        verts [V,3] f32, keys [V,4] i32, cols [V,3] f32 | None, tris [T,3] i32 -- all contiguous CUDA tensors.
        halo_hi_color: `export_plane_color(0)` of the slab above; needed for colours together with halo_hi."""
        torch = _lib.require_cuda()
        V, T = int(verts.shape[0]), int(tris.shape[0])
        if not (V or T):
            return
        for t in (verts, keys, cols, tris):
            if t is not None and not t.is_contiguous():
                raise RuntimeError("mc_emit: output tensors must be contiguous")
        with torch.cuda.device(self.device):
            _lib.check(self._L.bslam_mc_emit(self._h, _lib.ptr(halo_lo), _lib.ptr(halo_hi), _lib.ptr(halo_hi_color), _lib.ptr(verts),
                                             _lib.ptr(keys), _lib.ptr(cols) if self.color else None, V, _lib.ptr(tris), T,
                                             _lib.stream_ptr(self.device)))

    def extract_triangle_mesh(self, halo_lo=None, halo_hi=None, halo_hi_color=None) -> TriangleMesh:
        """Open3D `extract_triangle_mesh()` (tsdf.py:43) -- compacted marching cubes on the GPU.  Slab of a z-sharded
        volume: halo_lo / halo_hi are the neighbours' planes (`export_plane`), halo_hi_color the upper one's colour."""
        torch = _lib.require_cuda()
        V, T = self.mc_count(halo_lo, halo_hi)
        verts = torch.empty((V, 3), dtype=torch.float32, device=self.device)
        keys = torch.empty((V, 4), dtype=torch.int32, device=self.device)
        cols = torch.empty((V, 3), dtype=torch.float32, device=self.device) if self.color else None
        tris = torch.empty((T, 3), dtype=torch.int32, device=self.device)
        self.mc_emit(verts, keys, cols, tris, halo_lo, halo_hi, halo_hi_color)
        return TriangleMesh(verts, tris, cols, keys)

    def set_incremental_points(self, enable: bool = True, normals: bool = True):
        """incremental `extract_point_cloud` for the per-frame cadence (N/3DM/slam.py:126,195): only the bricks whose
        neighbourhood an integration changed since the last extraction are re-extracted, the others come from a per-brick
        cache; identical output.  `normals` fixes whether normals are produced in this mode."""
        _lib.check(self._L.bslam_points_set_incremental(self._h, int(bool(enable)), int(bool(normals))))
        self._pts_incremental = bool(enable)
        self._pts_inc_normals = bool(normals)

    def points_last_stats(self):
        """(surface-candidate bricks, bricks recomputed) of the last extract_point_cloud"""
        out = (C.c_longlong * 2)()
        _lib.check(self._L.bslam_points_last_stats(self._h, out))
        return int(out[0]), int(out[1])

    def extract_point_cloud(self, normals: bool = True) -> PointCloud:
        """Open3D `extract_point_cloud()` (tsdf.py:40)."""
        torch = _lib.require_cuda()
        if getattr(self, "_pts_incremental", False) and bool(normals) != self._pts_inc_normals:
            # a one-off request with the other normals setting: full extraction, the cache starts over afterwards
            inc_n = self._pts_inc_normals
            self.set_incremental_points(False)
            try:
                return self.extract_point_cloud(normals)
            finally:
                self.set_incremental_points(True, inc_n)
        cnt = np.zeros(1, np.int64)
        with torch.cuda.device(self.device):
            st = _lib.stream_ptr(self.device)
            _lib.check(self._L.bslam_points_count(self._h, _lib.ptr(cnt), st))
            P = int(cnt[0])
            pts = torch.empty((P, 3), dtype=torch.float32, device=self.device)
            nrm = torch.empty((P, 3), dtype=torch.float32, device=self.device) if normals else None
            cols = torch.empty((P, 3), dtype=torch.float32, device=self.device) if self.color else None
            keys = torch.empty((P, 4), dtype=torch.int32, device=self.device)
            if P:
                _lib.check(self._L.bslam_points_emit(self._h, _lib.ptr(pts), _lib.ptr(nrm), _lib.ptr(cols), _lib.ptr(keys), P, st))
        return PointCloud(pts, cols, nrm, keys)


class TSDF:
    """Drop-in for the reference's `TSDF` (N/3DM/tsdf.py:5-52)."""

    def __init__(self, voxel_length: float = 0.001, sdf_trunc: float = 0.1, resolution=512, origin=None,
                 color: bool = True, device=None, unit_activation=None):
        """unit_activation: True = ScalableTSDFVolume semantics (volume_unit_resolution 32, depth_sampling_stride
        8, tsdf.py:11-12): a frame only integrates the 32^3 units its sampled depth points activate, exactly
        what the reference object does; False = every voxel of the box follows the UniformTSDFVolume rule
        (the dense form BASELINE.json's north_star asks for).  None (default): True when the box consists
        of whole units on the world unit grid (the default 512^3 box does), else False.

        origin: world position of the box corner.  None (default): the box starts centred on the world origin and
        is RE-CENTRED ON THE FIRST FRAME's back-projected depth points (snapped to the 32-voxel unit grid) when that
        frame would otherwise mostly fall outside it -- the reference's hashed volume is unbounded, and its SLAM
        loop starts at the identity pose looking down +z (N/3DM/slam.py), i.e. at a surface that lies in front of,
        not around, the origin."""
        res = (int(resolution),) * 3 if np.isscalar(resolution) else tuple(int(r) for r in resolution)
        org = origin if origin is not None else tuple(-0.5 * r * voxel_length for r in res)
        self._auto_origin = origin is None
        self._unit_request = unit_activation
        self._make = lambda o, ua: DenseTSDFVolume(voxel_length=voxel_length, sdf_trunc=sdf_trunc, resolution=resolution, origin=o,
                                                   color=color, device=device, unit_activation=ua)
        if unit_activation is None:
            unit_activation = DenseTSDFVolume.unit_aligned(res, voxel_length, org)
        self.tsdf = self._make(origin, bool(unit_activation))
        if not unit_activation:
            self.tsdf.set_clip_check(8)
        self.tsdf.set_incremental_points(True, normals=True)      # extract_pcd() runs after every frame in the reference's loop
        self._clip_warned = 0.0
        self._next_clip_check = 1      # frames_integrated at which the next (synchronising) clip check is due

    def auto_centre(self, depth, intrinsic, extrinsic) -> bool:
        """Called with the first frame (f32 metres, H x W) when no origin was given: if fewer than half of its
        stride-8 back-projected points fall inside the (still empty) box, rebuild the box centred on their median,
        snapped to the 32-voxel unit grid.  Returns True when the box moved."""
        import warnings

        if not self._auto_origin or self.tsdf.frames_integrated:
            return False
        self._auto_origin = False
        torch = _lib.require_cuda()
        v = self.tsdf
        W, H, fx, fy, cx, cy = intrinsic_params(intrinsic)
        d = ops.as_cuda(depth, torch.float32, v.device).reshape(1, H, W)
        xyz, _ = ops.backproject(d, (fx, fy, cx, cy), np.asarray(to_numpy(extrinsic), dtype=np.float64).reshape(1, 4, 4), stride=8, device=v.device)
        if xyz.shape[0] == 0:
            return False
        ext = np.array([v.nx, v.ny, v.nz]) * v.voxel_length
        lo = torch.as_tensor(v.origin, dtype=torch.float32, device=v.device)
        hi = torch.as_tensor(v.origin + ext, dtype=torch.float32, device=v.device)
        inside = float(((xyz >= lo) & (xyz < hi)).all(dim=1).float().mean().item())
        if inside >= 0.5:
            return False
        centre = xyz.median(dim=0).values.cpu().numpy().astype(np.float64)
        ul = v.voxel_length * 32
        new_origin = np.floor((centre - 0.5 * ext) / ul + 0.5) * ul
        ua = self._unit_request
        if ua is None:
            ua = DenseTSDFVolume.unit_aligned((v.nx, v.ny, v.nz), v.voxel_length, new_origin)
        self.tsdf = self._make(tuple(new_origin), bool(ua))
        if not ua:
            self.tsdf.set_clip_check(8)
        self.tsdf.set_incremental_points(True, normals=True)
        warnings.warn(f"TSDF: only {100 * inside:.0f} % of the first frame's depth points fell inside the default box around the world "
                      f"origin; the box was re-centred on them: origin = ({new_origin[0]:.3f}, {new_origin[1]:.3f}, {new_origin[2]:.3f}) m, "
                      f"edge {ext[0]:.3f} m (pass origin= / resolution= to TSDF() to choose the box yourself)")
        return True

    def clipped_fraction(self) -> float:
        """share of the sampled depth points integrated so far that fell OUTSIDE the bounded box (the
        reference's ScalableTSDFVolume is unbounded and would have kept them)"""
        st = self.tsdf.clip_stats()
        return st["outside"] / st["points"] if st["points"] else 0.0

    def _warn_if_clipped(self):
        import warnings

        # the counters live on the device: read them at frames 1, 4, 16, ... so the per-frame cadence
        # (extract_pcd after every build_3D_map, N/3DM/slam.py:195) does not pay a device round trip per call
        if self.tsdf.frames_integrated < self._next_clip_check:
            return
        while self._next_clip_check <= self.tsdf.frames_integrated:
            self._next_clip_check *= 4
        frac = self.clipped_fraction()
        if frac > 0.01 and frac > 1.5 * self._clip_warned:
            self._clip_warned = frac
            lo = self.tsdf.origin
            hi = lo + np.array([self.tsdf.nx, self.tsdf.ny, self.tsdf.z_total]) * self.tsdf.voxel_length
            warnings.warn(f"TSDF: {100 * frac:.1f} % of the depth points integrated so far lie outside the volume box "
                          f"[{lo[0]:.3f}, {hi[0]:.3f}] x [{lo[1]:.3f}, {hi[1]:.3f}] x [{lo[2]:.3f}, {hi[2]:.3f}] m and were dropped "
                          f"(the reference's ScalableTSDFVolume is unbounded); pass resolution= / origin= to TSDF() to cover the scene")

    def build_3D_map(self, rgbd, intrinsic, extrinsic):
        '''
        This function reconstruct the 3D model from the pseudo-rgbd using TSDF
        :param rgbd: pseudo-rgbd
        :param intrinsic: intrinsic parameter of the camera
        :param extrinsic: the global position of the camera
        :return:
        '''
        if self._auto_origin and ops._dtype_name(rgbd.depth) == "float32":
            self.auto_centre(rgbd.depth, intrinsic, extrinsic)
        self.tsdf.integrate(rgbd, intrinsic, extrinsic)

    def build_copy_3D_map(self, rgbd, intrinsic, extrinsic):
        if self._auto_origin and ops._dtype_name(rgbd.depth) == "float32":
            self.auto_centre(rgbd.depth, intrinsic, extrinsic)
        tsdf_copy = _copy.deepcopy(self.tsdf)
        tsdf_copy.integrate(rgbd, intrinsic, extrinsic)
        return tsdf_copy

    def save_pcd(self, saving_path: str):
        from .io import write_point_cloud

        pcd = self.extract_pcd()
        write_point_cloud(saving_path, pcd)

    def extract_pcd(self):
        self._warn_if_clipped()
        return self.tsdf.extract_point_cloud()

    def extract_mesh(self) -> TriangleMesh:
        self._warn_if_clipped()
        return self.tsdf.extract_triangle_mesh()

    def save_mesh(self, saving_path: str):
        from .io import write_triangle_mesh

        mesh = self.extract_mesh()
        write_triangle_mesh(saving_path, mesh)


class MAP:
    """Drop-in for the reference's `MAP` (N/3DM/tsdf.py:56-108): the tensor-pipeline reconstruction
    (`o3d.t.pipelines.slam.Model`: VoxelBlockGrid of 16^3 blocks, projective TSDF, `depth_max` cut,
    `trunc_voxel_multiplier`).  Same constructor and methods; the blocks live in a bounded dense box
    (extra kwargs `resolution`, `origin`, `color`) instead of Open3D's hash map of `block_count` blocks
    (`block_count` is accepted and ignored; ray points that leave the box are counted, see `clip_stats`).
    Extraction follows the tensor pipeline's defaults: weight threshold 3, vertices on voxel corners.
    `synthesize_model_frame` ray casts the map from the pose of the last integrated frame (Open3D's
    `Model.synthesize_model_frame`); `integrate` does not call it (the reference discards its result).
    """

    BLOCK = 16

    def __init__(self, width, height, intrinsic, device, depth_scale, voxel_size=0.0058, block_count=40000, trunc_voxel_multiplier=8.0,
                 resolution=512, origin=None, color: bool = True, weight_threshold: float = 3.0):
        torch = _lib.require_cuda()
        self.width, self.height = int(width), int(height)
        K = np.asarray(to_numpy(intrinsic), dtype=np.float64) if not hasattr(intrinsic, "intrinsic_matrix") else np.asarray(intrinsic.intrinsic_matrix, dtype=np.float64)
        if K.shape != (3, 3):
            raise RuntimeError("[MAP] intrinsic must be a 3x3 matrix (the tensor pipeline takes o3d.core.Tensor(K))")
        self._K = np.array([K[0, 0], K[1, 1], K[0, 2], K[1, 2]], dtype=np.float64)
        self.depth_scale = float(depth_scale)
        self.voxel_size = float(voxel_size)
        self.block_count = int(block_count)
        self.trunc_voxel_multiplier = float(trunc_voxel_multiplier)
        dev = str(device).lower() if device is not None else None
        dev = ops._device(dev if (dev is not None and "cuda" in dev) else None)
        res = (int(resolution),) * 3 if np.isscalar(resolution) else tuple(int(r) for r in resolution)
        if any(r % self.BLOCK for r in res):
            raise RuntimeError(f"[MAP] the box must consist of whole {self.BLOCK}^3 blocks")
        if origin is None:
            bs = self.voxel_size * self.BLOCK
            origin = tuple(-(r // (2 * self.BLOCK)) * bs for r in res)
        # sdf_trunc of the underlying box is only used by the legacy integrator; keep it consistent anyway
        self.model = DenseTSDFVolume(self.voxel_size, self.voxel_size * self.trunc_voxel_multiplier, res, origin, color=color, device=dev)
        _lib.check(self.model._L.bslam_tsdf_set_extract_flavour(self.model._h, float(weight_threshold), 0.0))
        self._ws = torch.zeros(self.model._L.bslam_vbg_workspace_bytes(*res), dtype=torch.uint8, device=dev)
        self.poses = {}
        self._last_pose, self._frame_id = None, -1
        self._range_ws = None

    def integrate_batch(self, depth_u16, color, poses, depth_max, update_counts=None):
        """F frames in order: depth_u16 [F,H,W] uint16 (raw, divided by depth_scale in the kernel), color
        [F,H,W,3] uint8 | None, poses [F,4,4] camera->world, depth_max scalar or [F]."""
        torch = _lib.require_cuda()
        vol = self.model
        if ops._dtype_name(depth_u16) != "uint16":
            raise RuntimeError("[MAP::Integrate] Unsupported image format.")
        d = ops.as_cuda(depth_u16, torch.uint16, vol.device)
        if d.dim() == 2:
            d = d.unsqueeze(0)
        F = d.shape[0]
        if d.shape[1] != self.height or d.shape[2] != self.width:
            raise RuntimeError("[MAP::Integrate] Unsupported image format.")
        c = None
        if vol.color:
            if color is None or ops._dtype_name(color) != "uint8":
                raise RuntimeError("[MAP::Integrate] Unsupported image format.")
            c = ops.as_cuda(color, torch.uint8, vol.device)
            if c.numel() != F * self.height * self.width * 3:
                raise RuntimeError("[MAP::Integrate] Unsupported image format.")
        P = np.ascontiguousarray(np.asarray(to_numpy(poses), dtype=np.float64).reshape(-1, 16))
        if P.shape[0] != F:
            raise RuntimeError(f"MAP.integrate_batch: {F} frames but {P.shape[0]} poses")
        dm = np.ascontiguousarray(np.broadcast_to(np.asarray(depth_max, dtype=np.float64), (F,)))
        with torch.cuda.device(vol.device):
            _lib.check(vol._L.bslam_vbg_integrate(vol._h, _lib.ptr(d), _lib.ptr(c), F, self.height, self.width, _lib.ptr(self._K), _lib.ptr(P),
                                                  _lib.ptr(dm), self.depth_scale, self.trunc_voxel_multiplier, _lib.ptr(self._ws),
                                                  _lib.ptr(update_counts), _lib.stream_ptr(vol.device)))
        vol.frames_integrated += F
        if F:
            self._last_pose, self._frame_id = P[-1].copy(), vol.frames_integrated - 1

    def integrate(self, curr_rgbd, i, curr_global_pose):
        """reference signature (tsdf.py:71): `curr_rgbd` is an `RGBD` (uses `.o3d_t_depth`, `.o3d_t_color`,
        `.depth_max`), `curr_global_pose` the 4x4 camera->world pose of frame i (`update_frame_pose`)."""
        pose = np.asarray(to_numpy(curr_global_pose), dtype=np.float64).reshape(4, 4)
        self.poses[int(i)] = pose
        self.integrate_batch(curr_rgbd.o3d_t_depth, curr_rgbd.o3d_t_color if self.model.color else None, pose[None], curr_rgbd.depth_max)
        self._frame_id = int(i)

    def synthesize_model_frame(self, depth_min: float = 0.1, depth_max: float = 3.0, enable_color: bool = True, weight_threshold: float = -1.0):
        """Open3D `Model.synthesize_model_frame`: ray cast the map at width x height from the pose of the last integrated
        frame, over the ray ranges of the blocks that frame activated.  weight_threshold < 0: min(frame_id, 3), frame_id =
        the last `i` given to `integrate` (as recalled from Open3D's SynthesizeModelFrame).  -> dict of CUDA f32 tensors
        depth [1,H,W] (raw units: z * depth_scale), vertex / normal [1,H,W,3] (camera frame), color [1,H,W,3] in [0, 1]
        (colour maps and enable_color only); pixels whose ray hits nothing are 0."""
        torch = _lib.require_cuda()
        if self._last_pose is None:
            raise RuntimeError("[MAP::SynthesizeModelFrame] nothing integrated yet")
        vol = self.model
        if weight_threshold < 0:
            weight_threshold = min(float(self._frame_id), 3.0)
        H, W = self.height, self.width
        out = vol._raycast_outputs(1, H, W, True, enable_color and vol.color)
        nbytes = vol._L.bslam_vbg_raycast_workspace_bytes(H, W)
        if self._range_ws is None or self._range_ws.numel() < nbytes:
            self._range_ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=vol.device)
        P = np.ascontiguousarray(self._last_pose.reshape(16))
        with torch.cuda.device(vol.device):
            _lib.check(vol._L.bslam_vbg_raycast(vol._h, _lib.ptr(self._ws), H, W, _lib.ptr(self._K), _lib.ptr(P), self.depth_scale, float(depth_min),
                                                float(depth_max), float(weight_threshold), self.trunc_voxel_multiplier, _lib.ptr(out["depth"]),
                                                _lib.ptr(out["vertex"]), _lib.ptr(out["normal"]), _lib.ptr(out.get("color")), _lib.ptr(self._range_ws),
                                                _lib.stream_ptr(vol.device)))
        return out

    def track_frame_to_model(self, input_rgbd, model_frame, depth_scale=None, depth_max: float = 3.0, depth_diff: float = 0.07, method=Method.PointToPlane,
                             criteria=(6, 3, 1)):
        """Open3D `Model.track_frame_to_model`: `odometry.rgbd_odometry_multi_scale` from the input frame (`.o3d_t_depth`,
        `.o3d_t_color`, as `integrate` reads them) to `model_frame`, the dict `synthesize_model_frame` returns, from the
        identity, with OdometryLossParams(depth_diff) and criteria = max iterations per level, coarsest first.
        depth_scale None = the map's.  -> OdometryResult; compose
        `T_frame_to_model = T_frame_to_model @ result.transformation`."""
        from . import odometry as od
        from .geometry import RGBDImage

        method = Method(method)
        needs_color = method != Method.PointToPlane
        src = RGBDImage(input_rgbd.o3d_t_color if needs_color else None, input_rgbd.o3d_t_depth)
        depth = model_frame["depth"]
        color = model_frame.get("color") if needs_color else None
        tgt = RGBDImage(None if color is None else color.reshape(color.shape[-3:]), depth.reshape(depth.shape[-2:]))
        K = np.array([[self._K[0], 0.0, self._K[2]], [0.0, self._K[1], self._K[3]], [0.0, 0.0, 1.0]])
        return od.rgbd_odometry_multi_scale(src, tgt, K, depth_scale=self.depth_scale if depth_scale is None else float(depth_scale),
                                            depth_max=depth_max, criteria_list=[od.OdometryConvergenceCriteria(int(c)) for c in criteria],
                                            method=method, params=od.OdometryLossParams(depth_diff))

    def allocated_blocks(self, last_frame: bool = False):
        """bool CUDA tensor [nbx, nby, nbz] of the 16^3 blocks of the box: activated by any frame integrated so far (the
        VoxelBlockGrid's allocated blocks), or with `last_frame` by the last integrated frame only (synchronises)."""
        torch = _lib.require_cuda()
        vol = self.model
        nb = [n // self.BLOCK for n in (vol.nx, vol.ny, vol.nz)]
        n = nb[0] * nb[1] * nb[2]
        bit = torch.arange(32, dtype=torch.int32, device=vol.device)
        if last_frame:
            f = int(self._ws[16:20].view(torch.int32).item())
            masks = self._ws[256:256 + n * 8].view(torch.int32).view(n, 2)[:, f >> 5]
            return ((masks >> (f & 31)) & 1).bool().view(nb)
        off = 256 + n * 8
        words = self._ws[off:off + (n + 31) // 32 * 4].view(torch.int32)
        return ((words[:, None] >> bit) & 1).bool().reshape(-1)[:n].view(nb)

    def clip_stats(self):
        """ray points of the block activation seen / outside the bounded box (the reference's hash map is unbounded)"""
        out = (C.c_ulonglong * 2)()
        _lib.check(self.model._L.bslam_vbg_stats(_lib.ptr(self._ws), out, _lib.stream_ptr(self.model.device)))
        return {"points": int(out[0]), "outside": int(out[1])}

    def extract_pcd(self):
        return self.model.extract_point_cloud()

    def extract_mesh(self) -> TriangleMesh:
        return self.model.extract_triangle_mesh()

    def save_pcd(self, saving_path: str):
        from .io import write_point_cloud

        write_point_cloud(saving_path, self.extract_pcd())

    def save_mesh(self, saving_path: str):
        from .io import write_triangle_mesh

        write_triangle_mesh(saving_path, self.extract_mesh())
