#!/usr/bin/env python
"""bench.py -- fused frames/s of the depth->TSDF hot path on B200 (BASELINE.json metric).

Default workload (`config.workload`): BASELINE configs[3], the 1000-frame synthetic laparoscopy sweep,
640x480 u16 depth -> 512^3 TSDF @ 1 mm (sdf_trunc 5 mm).  `--workload colonoscopy256` = configs[1],
`--workload gastroscopy1024` = configs[4]; configs[2] (64 x 1080p scale + colorize + back-project)
and configs[0] (one frame) are timed as `extras` of every N = 1 run.

One STEP = one pass of the hot path over the whole trajectory: a4 depth scaling (u16 -> metres, trunc,
fused into the first pass) + K3 TSDF integration of all frames in order into the resident volume.
  value : frames/s with the u16 depth already in HBM (integration only -- the BASELINE metric);
  e2e   : the same pass through the public API from pinned HOST buffers (H2D inside the timed region)
          FOLLOWED BY one marching-cubes extraction and the D2H copy of the mesh and of the per-frame
          update counts (configs[3]: "integrate ... + marching cubes").
N > 1 (torchrun, one rank per GPU): the volume is cut into z-shards (strong scaling: same total work),
frames reach the ranks over NCCL inside the timed region, the mesh is gathered on rank 0.

The JSON line also carries `parity` (tsdf / weight sha256 and mesh sizes of the GPU volume against the
CPU oracle on the frames the CPU leg integrates, dense rule and ScalableTSDFVolume rule), `roofline`,
`cpu_baseline`, `reference_literal` (the object the reference's `TSDF()` literally builds: RGB8 + 32^3 unit
activation) and `slam_cadence` (one `build_3D_map` + one `extract_pcd` per frame, N/3DM/slam.py:179,195).

`--impl reference` times the reference's CPU path (the Open3D-equivalent oracle, all host threads) on
bounded samples of the same workload.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "frames/s"
WORKLOADS = {
    "laparoscopy512": ("configs[3]", "synthetic laparoscopy sweep"),
    "colonoscopy256": ("configs[1]", "synthetic colonoscopy trajectory"),
    "gastroscopy1024": ("configs[4]", "long synthetic gastroscopy trajectory"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="laparoscopy512", choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=0, help="frames per step (default: the config's; debug only)")
    ap.add_argument("--resolution", type=int, default=0, help="override the grid (debug only; invalidates the metric)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg (and with it the parity block)")
    ap.add_argument("--no-mc", action="store_true", help="leave the mesh extraction out of e2e (debug only)")
    ap.add_argument("--no-extras", action="store_true", help="skip configs[0]/[2], reference-literal and cadence legs")
    ap.add_argument("--batch", type=int, default=0, help="frames per integrate launch (0 = library default)")
    ap.add_argument("--settle", type=float, default=1.5, help="seconds of untimed steps before the warm-up (device clocks / memory settle)")
    ap.add_argument("--cpu-budget", type=float, default=6.0, help="seconds of CPU oracle work per timed CPU leg")
    ap.add_argument("--deviation", action="store_true", help="also quantify brick-restart vs literal z recurrence over all frames (slow validation kernel)")
    ap.add_argument("--zpw", type=int, default=0, help="z layers per integrate warp (0 = library default; tuning aid)")
    ap.add_argument("--const-depth", type=int, default=0, help="EXPERIMENT: replace every frame by this constant uint16 depth (limit studies with BSLAM_EXPERIMENT; not a bench value)")
    ap.add_argument("--resident-layout", default="rank0", choices=["rank0", "sharded"],
                    help="N > 1, where the resident u16 frames live before the timed region: all on rank 0 (NCCL broadcast per chunk) or 1/N of every "
                         "chunk in each rank's HBM (NCCL all-gather per chunk)")
    ap.add_argument("--emulate-shard", default="", help="R/N: time rank R's shard of an N-GPU run on ONE GPU (no NCCL; development aid)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last timed steps computed as DIR/<name>.npy (float32 / float64; arrays over "
                         "the size cap as a fixed seeded sample), to compare two builds output for output (single GPU only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.emulate_shard):
        ap.error("--dump-outputs needs the GPU arm without --emulate-shard")
    return args


def metric_name(res):
    return f"fused frames/s (640x480 depth -> {res}^3 TSDF)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(args, world, res, F):
    """DRAM bytes per brick_integrate_kernel launch from the committed `ncu --set full` capture
    (profiles/traffic.json); only quoted when this run has the captured run's shape."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))["brick_integrate_kernel"]
    except Exception:
        return None, None
    if world != t.get("n_gpus", 1) or res != t.get("resolution") or (args.batch or 256) != t.get("frames_per_launch") or F != t.get("frames"):
        return None, "profiles/traffic.json holds a different configuration"
    return t["dram_bytes_per_launch"], t["source"]


class ClockSampler:
    """nvidia-smi polled every 25 ms for the whole run; only samples whose timestamp falls inside a
    timed window (resident / e2e loops) are reported, so the clocks are the ones under load."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        self.windows = []
        self.path = f"/tmp/bslam_clocks_{os.getpid()}.csv"
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25", "-i", str(index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        import datetime

        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.06)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.close()
        rows = []
        for line in open(self.path):
            t = [x.strip() for x in line.split(",")]
            if len(t) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(t[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(t[1]), float(t[2]), [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                                                                 "sw_power_cap"), t[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        try:
            os.remove(self.path)
        except OSError:
            pass
        inside = [r for r in rows if any(a - 0.005 <= r[0] <= b + 0.005 for a, b in self.windows)]
        where = "inside the timed regions"
        if not inside and rows and self.windows:   # timed regions shorter than the poll period: nearest sample to each window
            inside = [min(rows, key=lambda r: abs(r[0] - 0.5 * (a + b))) for a, b in self.windows]
            where = "nearest to the timed regions (regions shorter than the 25 ms poll period)"
        if inside:
            out.update(sm_mhz=float(np.median([r[1] for r in inside])), sm_max_mhz=float(max(r[2] for r in inside)),
                       reasons=sorted({n for r in inside for n in r[3]}), samples=len(inside), sampled=where)
        return out


def workload(args):
    from bodyslam_b200 import synthetic as S

    cfg = S.config(args.workload)
    F = args.frames or cfg["frames"]
    E = cfg["extrinsics"](cfg["frames"])
    if F != cfg["frames"]:
        E = E[np.linspace(0, cfg["frames"] - 1, F).astype(int)]
    res = args.resolution or cfg["resolution"]
    scale = cfg["resolution"] / res
    return cfg, F, E, res, cfg["voxel_length"] * scale, cfg["sdf_trunc"] * scale


def config_dict(args, F, W, H, res, vl, trunc):
    """identical in both arms (the driver compares them)"""
    tag, desc = WORKLOADS[args.workload]
    return {"workload": f"{args.workload}: {F}-frame {desc}, {W}x{H} u16 depth -> {res}^3 TSDF @ {vl * 1e3:g} mm, "
                        f"sdf_trunc {trunc * 1e3:g} mm (BASELINE {tag})",
            "frames_per_step": F, "resolution": res, "voxel_length_m": vl, "sdf_trunc_m": trunc, "image": f"{W}x{H} uint16 (3DM units, depth_scale 1000, depth_trunc 3.0)",
            "volume_rule": "dense: every voxel of the box follows Open3D's UniformTSDFVolume::Integrate rule (north_star); the ScalableTSDFVolume "
                           "rule the reference's TSDF() applies (32^3 unit activation, RGB8) is measured beside it as reference_literal",
            "l2": f"inputs larger than L2 ({F * W * H * 2 / 1e9:.2f} GB u16 depth + {res ** 3 * 8 / 1e9:.2f} GB volume per step vs 126 MB)"}


# --dump-outputs: at most 2 x 8 MiB of voxels + 12 + 24 + 8 MiB of rows = 60 MiB in all
DUMP_VOXELS = 1 << 21
DUMP_ROWS = 1 << 20


def dump_sample(n, cap):
    """indices of a fixed seeded sample of `cap` out of n items (sorted), or None when all n fit"""
    if n <= cap:
        return None
    return np.sort(np.random.default_rng(0).choice(n, cap, replace=False))


def dump_rows(a, cap=DUMP_ROWS):
    sel = dump_sample(len(a), cap)
    return a if sel is None else a[sel]


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def unit_origin(origin, vl):
    """nearest origin on the world unit grid (ScalableTSDFVolume semantics need whole 32^3 units)"""
    ul = vl * 32
    return np.floor(np.asarray(origin, dtype=np.float64) / ul + 0.5) * ul


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_timed(fn, frame_ids, budget_s, max_frames):
    """run fn(k, frame id) over the sample until the time budget is used -> (frames/s, n, results)"""
    out, t_used, n = [], 0.0, 0
    for k, fi in enumerate(frame_ids[:max_frames]):
        t0 = time.perf_counter()
        out.append(fn(k, fi))
        t_used += time.perf_counter() - t0
        n += 1
        if t_used > budget_s:
            break
    return n / t_used, n, out


def cpu_legs(cfg, E, sample_u16, sample_rgb, ids, res, vl, trunc, budget_s):
    """The oracle (Open3D-equivalent CPU path, all host threads) on sample frames:
    dense sweep (UniformTSDFVolume rule, z_restart 8 like the GPU fast path), and the ScalableTSDFVolume rule
    with RGB8 (what the reference's TSDF() does) under two thread schedules.  Returns timings + the volumes."""
    import oracle

    oracle.o3d.set_num_threads(host_threads())
    K = cfg["K"]
    org_u = unit_origin(cfg["origin"], vl)
    out = {"cores": oracle.o3d.num_threads()}
    V = oracle.o3d.Volume(res, vl, trunc, cfg["origin"])
    V.integrate(oracle.o3d.depth_from_u16(sample_u16[0]), K, E[ids[0]])      # warm-up: page faults of the volume
    V.tsdf[:] = 0
    V.weight[:] = 0
    fps, n, counts = cpu_timed(lambda k, fi: V.integrate(oracle.o3d.depth_from_u16(sample_u16[k]), K, E[fi]), ids, budget_s, 400)
    out.update(dense_fps=fps, dense_frames=n, dense_counts=counts, dense_volume=V)
    if res % 32 == 0:
        S = oracle.o3d.Volume(res, vl, trunc, org_u, with_color=True)
        S.integrate_scalable(oracle.o3d.depth_from_u16(sample_u16[0]), K, E[ids[0]], rgb=sample_rgb[0])
        S.tsdf[:] = 0
        S.weight[:] = 0
        S.color[:] = 0
        fps, n, counts = cpu_timed(lambda k, fi: S.integrate_scalable(oracle.o3d.depth_from_u16(sample_u16[k]), K, E[fi], rgb=sample_rgb[k]),
                                   ids, budget_s, len(ids))
        out.update(scalable_fps=fps, scalable_frames=n, scalable_counts=counts, scalable_volume=S)
        # Open3D's own threading: touched units one after the other, OpenMP over x inside each 32^3 unit
        oracle.o3d.set_scalable_schedule(True)
        T = oracle.o3d.Volume(res, vl, trunc, org_u, with_color=True)
        fps, n, _ = cpu_timed(lambda k, fi: T.integrate_scalable(oracle.o3d.depth_from_u16(sample_u16[k]), K, E[fi], rgb=sample_rgb[k]),
                              ids, 0.5 * budget_s, len(ids))
        oracle.o3d.set_scalable_schedule(False)
        out.update(scalable_open3d_schedule_fps=fps, scalable_open3d_schedule_frames=n)
        del T
    return out


def run_reference(args):
    """--impl reference: the reference's CPU path on bounded samples (rank 0 only; all host threads --
    torchrun exports OMP_NUM_THREADS=1, which is overridden here)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle

    from bodyslam_b200 import synthetic as S

    cfg, F, E, res, vl, trunc = workload(args)
    oracle.o3d.set_num_threads(host_threads())
    cores = oracle.o3d.num_threads()
    per_step = 4 if res <= 512 else 1
    n_total = per_step * (args.steps + args.warmup)
    ids = np.linspace(0, len(E) - 1, n_total).astype(int)
    depth, color = S.render(cfg["surface"], E[ids], K=cfg["K"], W=cfg["W"], H=cfg["H"], device="cpu", with_color=True)
    depth, color = depth.numpy(), color.numpy()
    V = oracle.o3d.Volume(res, vl, trunc, cfg["origin"])
    k = 0
    t_steps = []
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        for _ in range(per_step):
            V.integrate(oracle.o3d.depth_from_u16(depth[k]), cfg["K"], E[ids[k]])
            k += 1
        if s >= args.warmup:
            t_steps.append(time.perf_counter() - t0)
    total = sum(t_steps)
    fps = per_step * args.steps / total
    del V
    extra = {}
    if res % 32 == 0:
        org_u = unit_origin(cfg["origin"], vl)
        for name, o3d_like in (("scalable_fps", False), ("scalable_open3d_schedule_fps", True)):
            oracle.o3d.set_scalable_schedule(o3d_like)
            Sv = oracle.o3d.Volume(res, vl, trunc, org_u, with_color=True)
            Sv.integrate_scalable(oracle.o3d.depth_from_u16(depth[0]), cfg["K"], E[ids[0]], rgb=color[0])
            f, n, _ = cpu_timed(lambda kk, fi: Sv.integrate_scalable(oracle.o3d.depth_from_u16(depth[kk]), cfg["K"], E[fi], rgb=color[kk]),
                                ids, args.cpu_budget, len(ids))
            extra[name] = f
            extra[name.replace("_fps", "_frames")] = n
            del Sv
        oracle.o3d.set_scalable_schedule(False)
    sample = (f"{per_step} frames per step sampled evenly from the {len(E)}-frame trajectory, {res}^3 dense sweep per frame "
              f"(oracle/o3d_oracle.c: Open3D UniformTSDFVolume::Integrate restated, OpenMP over x like Open3D)")
    line = {"impl": "reference", "metric": metric_name(res), "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, len(E), cfg["W"], cfg["H"], res, vl, trunc),
            "reference_arm": "CPU restatement of the Open3D calls the reference makes (Open3D itself is not installable offline): value = the dense "
                             "UniformTSDFVolume sweep, like for like with the GPU arm's dense rule; reference_literal = ScalableTSDFVolume rule "
                             "(32^3 units, stride-8 activation, RGB8) -- units spread over the threads, and with Open3D's own schedule",
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "dense_fps": fps, **extra},
            "reference_literal": {"value": extra.get("scalable_fps"), "unit": UNIT, "open3d_schedule_value": extra.get("scalable_open3d_schedule_fps")},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist

    from bodyslam_b200 import _lib, ops
    from bodyslam_b200 import synthetic as S
    from bodyslam_b200.geometry import PinholeCameraIntrinsic, RGBDImage
    from bodyslam_b200.sharding import ShardedTSDF
    from bodyslam_b200.tsdf import TSDF, DenseTSDFVolume

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single-GPU run")
    _lib.require_cuda()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    emu = None
    if args.emulate_shard:
        emu = tuple(int(x) for x in args.emulate_shard.split("/"))
        assert world == 1 and 0 <= emu[0] < emu[1]

    cfg, F, E, res, vl, trunc = workload(args)
    W, H = cfg["W"], cfg["H"]
    intr = PinholeCameraIntrinsic(W, H, *cfg["K"])
    t_start = time.time()

    def log(msg):
        if rank == 0:
            print(f"[bench +{time.time() - t_start:5.1f}s] {msg}", file=sys.stderr, flush=True)

    # ---- inputs: every rank renders its share of the trajectory on its GPU (u16 depth in 3DM units, mm), all-gathered
    per = -(-F // world)
    lo, hi = min(rank * per, F), min((rank + 1) * per, F)
    depth_u16 = torch.zeros((per * world, H, W), dtype=torch.uint16, device=dev)
    if hi > lo:
        depth_u16[lo:hi] = S.render(cfg["surface"], E[lo:hi], K=cfg["K"], W=W, H=H, device=dev, with_color=False, first_frame=lo)[0]
    if world > 1:
        dist.all_gather_into_tensor(depth_u16.view(torch.uint8), depth_u16[rank * per:(rank + 1) * per].view(torch.uint8).clone())
    depth_u16 = depth_u16[:F]
    if args.const_depth:
        depth_u16 = torch.full_like(depth_u16.view(torch.int16), args.const_depth).view(torch.uint16)
    log(f"rendered {F} frames")

    # N > 1: round-robin brick layers (rank r owns every N-th 8-voxel layer) -> balanced whatever the view
    if emu:
        n_emu = emu[1]
        vol = DenseTSDFVolume(vl, trunc, (res, res, res // n_emu), cfg["origin"], color=False, device=dev, gz0=8 * emu[0], z_total=res, z_interleave=n_emu)
        sh = None
        interleaved = True
    else:
        sh = ShardedTSDF(vl, trunc, res, cfg["origin"], color=False, device=dev, rank=rank, world_size=world, unit_activation=False)
        vol = sh.tsdf
        interleaved = sh.layout == "interleaved"
    if args.batch:
        vol.set_batch(args.batch)
    if args.zpw:
        vol.set_z_split(args.zpw)
    chunk = args.batch or 256
    chunks = vol.stream_chunks(F, chunk, ramp=ShardedTSDF.stream_ramp(world, True))   # integrate launches of a resident step

    dev_share = None
    if world > 1 and args.resident_layout == "sharded":
        # every rank keeps the frames ingest_share() assigns to it (1/N of every chunk) in ITS HBM
        sel_share = torch.as_tensor(ShardedTSDF.ingest_share(F, rank, world, chunk), device=dev)
        dev_share = depth_u16.view(torch.int16)[sel_share].view(torch.uint16).contiguous()

    def step(src_u16, counts=None):
        """one pass of the hot path over the whole trajectory through the public API.  a4 is fused into the
        integration's first pass.  N > 1: the frames reach every rank over NCCL chunk by chunk inside the timed
        region -- all-gathered from the ranks' resident shares (default) or broadcast from rank 0 -- the transfer
        of chunk k+1 (and the H2D of chunk k+2 when the source is host memory) overlapping the integration of chunk k."""
        if dev_share is not None and src_u16 is depth_u16:
            sh.integrate_stream_sharded(dev_share, intr, E, depth_scale=1000.0, depth_trunc=3.0, chunk=chunk, update_counts=counts)
            return
        if emu:
            vol.integrate_u16_chunks(src_u16, None, intr, E, chunks, 1000.0, 3.0, counts)
            return
        sh.integrate_stream(src_u16, intr, E, src=0, depth_scale=1000.0, depth_trunc=3.0, chunk=chunk, update_counts=counts)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- algorithmic bytes: U_f = voxels each frame updates (dry run, untimed), summed over shards
    depth_f = ops.depth_from_u16(depth_u16, 1000.0, 3.0, dev)
    vol.dry_stats(True)
    uf_local = vol.count_updates(depth_f, intr, E)
    cull = vol.dry_stats(True)
    uf = uf_local.clone()
    if world > 1:
        dist.all_reduce(uf)
    uf_total = int(uf.sum().item())
    bytes_algo_local = 16 * int(uf_local.sum().item()) + 4 * W * H * F   # SURVEY.md 8(d): 16 B x updated voxels + 4*W*H per frame
    if res > 512 or args.no_extras:
        del depth_f

    # ---- device-resident timing
    sampler = ClockSampler(local) if rank == 0 else None
    # a fresh box runs its first ~second of kernels a few % slow (measured: 3.77 ms per integrate launch in
    # the first process, 3.66 ms in the third, same code): let the device settle before the W warm-up steps
    t_settle = time.time()
    step(depth_u16)
    torch.cuda.synchronize()
    n_settle = torch.tensor([int(args.settle / max(time.time() - t_settle, 1e-3))], device=dev)
    if world > 1:
        dist.broadcast(n_settle, 0)          # every rank must run the same number of (collective) steps
    for _ in range(int(n_settle.item())):
        step(depth_u16)
    # the number of settle steps follows the clock: start the warm-up from an empty volume so that what the timed
    # steps leave in it depends on --warmup and --steps alone (the work of a step does not depend on the volume)
    vol.reset()
    for _ in range(args.warmup):
        step(depth_u16)
    vol.profile(True)
    barrier()
    tw0 = time.time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step(depth_u16)
    ev1.record()
    barrier()
    if sampler:
        sampler.window(tw0, time.time())
    ms_local = ev0.elapsed_time(ev1)
    ms_total = max_over_ranks(ms_local)
    stage_ms, k_launches = vol.profile_read_stages()
    k_ms = stage_ms["brick_integrate"]
    vol.profile(False)
    dumps = {}
    if args.dump_outputs:
        # the resident volume after the last timed step, at the same seeded voxel sample in both grids
        t, w = vol.export_dense()
        sel = dump_sample(t.numel(), DUMP_VOXELS)
        sel = slice(None) if sel is None else torch.from_numpy(sel).to(dev)
        dumps["tsdf"], dumps["weight"] = t.view(-1)[sel].cpu().numpy(), w.view(-1)[sel].cpu().numpy()
        del t, w, sel
    fps = args.steps * F / (ms_total / 1e3)
    # per-rank timeline of one step (CUDA events inside the library), gathered on rank 0
    steps_prof = max(1, min(args.steps, k_launches // max(len(chunks), 1)))
    mine = {k: v / steps_prof for k, v in stage_ms.items()}
    mine["step_total"] = ms_local / args.steps
    # the preparation of launch k+1 (first two stages, side stream) overlaps the integration of launch k: the stage times
    # are each stage's own busy time, their sum may exceed the step
    mine["step_minus_integrate"] = mine["step_total"] - stage_ms["brick_integrate"] / steps_prof
    timeline = [mine]
    if world > 1:
        g = [None] * world
        dist.all_gather_object(g, mine)
        timeline = g
    log(f"resident: {fps:.1f} frames/s, {ms_total / args.steps:.2f} ms/step, integrate kernel {k_ms / max(k_launches, 1):.3f} ms x "
        f"{k_launches} launches, U_f mean {uf_total / F:.0f} voxels/frame; stages ms/step {json.dumps({k: round(v, 3) for k, v in mine.items()})}")

    # ---- end to end: pinned host u16 -> H2D -> a4 -> K3 -> marching cubes -> D2H of the mesh + per-frame update counts
    # N = 1: the whole trajectory in one pinned host buffer.  N > 1: sharded ingest -- every rank holds 1/N of
    # each chunk in ITS pinned host memory (as N decoder processes would), copies it over its own PCIe link
    # and the pieces are all-gathered over NVLink; a single host buffer on rank 0 would cap the job at one
    # link's 53 GB/s (86 k frames/s).  h2d_bytes_per_step counts all ranks.  The mesh is gathered on rank 0.
    e2e = None
    mesh_info = {}
    if not emu:
        share = ShardedTSDF.ingest_share(F, rank, world, chunk)
        host_u16 = torch.empty((len(share), H, W), dtype=torch.uint16).pin_memory()
        host_counts = torch.empty(F, dtype=torch.int64).pin_memory()
        host_u16.copy_(depth_u16.view(torch.int16)[torch.as_tensor(share, device=dev)].view(torch.uint16))
        counts = torch.zeros(F, dtype=torch.int64, device=dev)
        host_mesh = {}

        def e2e_step():
            # public API: pinned host frames in; mesh (vertices, triangles) and per-frame update counts out in host memory
            counts.zero_()
            if world == 1:
                step(host_u16, counts)
            else:
                sh.integrate_stream_sharded(host_u16, intr, E, depth_scale=1000.0, depth_trunc=3.0, chunk=chunk, update_counts=counts)
            host_counts.copy_(counts, non_blocking=True)
            if args.no_mc:
                return None
            mesh = sh.extract_mesh()             # N > 1: re-shard to slabs, halo exchange, per-slab cubes, gather + merge on rank 0
            if mesh is not None:
                nv, nt = int(mesh.vertices.shape[0]), int(mesh.triangles.shape[0])
                if "v" not in host_mesh or host_mesh["v"].shape[0] < nv or host_mesh["t"].shape[0] < nt:
                    host_mesh["v"] = torch.empty((max(nv, 1) * 5 // 4, 3), dtype=torch.float32).pin_memory()
                    host_mesh["t"] = torch.empty((max(nt, 1) * 5 // 4, 3), dtype=torch.int32).pin_memory()
                host_mesh["v"][:nv].copy_(mesh.vertices, non_blocking=True)
                host_mesh["t"][:nt].copy_(mesh.triangles, non_blocking=True)
            return mesh

        e2e_step()
        e2e_step()
        barrier()
        tw0 = time.time()
        ev0.record()
        for _ in range(args.steps):
            mesh = e2e_step()
        ev1.record()
        barrier()
        if sampler:
            sampler.window(tw0, time.time())
        ms_e2e = max_over_ranks(ev0.elapsed_time(ev1))
        fps_e2e = args.steps * F / (ms_e2e / 1e3)
        nv = nt = 0
        if mesh is not None:
            nv, nt = int(mesh.vertices.shape[0]), int(mesh.triangles.shape[0])
        mesh_info = {"mc_vertices": nv, "mc_triangles": nt}
        if args.dump_outputs:
            # what the last e2e step handed back in host memory
            dumps["update_counts"] = dump_rows(host_counts.numpy().astype(np.float64))
            if mesh is not None:
                dumps["mesh_vertices"] = dump_rows(host_mesh["v"][:nv].numpy())
                dumps["mesh_triangles"] = dump_rows(host_mesh["t"][:nt].numpy().astype(np.float64))
        e2e = {"value": fps_e2e, "unit": UNIT, "h2d_bytes_per_step": F * H * W * 2 + F * 128, "d2h_bytes_per_step": F * 8 * world + nv * 12 + nt * 12,
               "ms_per_step": ms_e2e / args.steps,
               "includes": "H2D of the u16 frames, a4 + K3 over all frames, " + ("no mesh (--no-mc)" if args.no_mc else
                           "one marching-cubes extraction (count + emit" + (", slab re-shard + halo exchange + gather on rank 0" if world > 1 else "") +
                           "), D2H of vertices + triangles") + " and of the per-frame update counts",
               "ingest": "one pinned host buffer" if world == 1 else f"sharded: each of the {world} ranks feeds 1/{world} of every chunk from its own pinned host memory, pieces all-gathered over NVLink"}
        log(f"e2e: {fps_e2e:.1f} frames/s, {ms_e2e / args.steps:.2f} ms/step, mesh {nv} vertices / {nt} triangles")
        del mesh
        if world > 1 and not args.no_mc:
            prof = []
            for _ in range(3):
                barrier()
                sh.extract_mesh(profile=True)
                prof.append(sh.last_extract_profile)
            mine_x = {k: float(np.median([p[k] for p in prof])) for k in prof[0]}
            allx = [None] * world
            dist.all_gather_object(allx, mine_x)
            mesh_info["extract_mesh_phase_ms_max_over_ranks"] = {k: max(x[k] for x in allx) for k in mine_x}
            log(f"multi-GPU extraction phases (ms, max over ranks, synchronised between phases): {json.dumps({k: round(v, 2) for k, v in mesh_info['extract_mesh_phase_ms_max_over_ranks'].items()})}")
    clocks = sampler.stop() if sampler else None   # samples inside both timed regions (resident + e2e)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumps.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
        log(f"outputs written to {args.dump_outputs}: " + ", ".join(f"{k} {a.dtype}{list(a.shape)}" for k, a in dumps.items()))

    # ---- N > 1: the gathered mesh of one clean pass must equal the single-GPU mesh
    parity = {}
    if world > 1 and not args.no_mc:
        sh.tsdf.reset()
        step(depth_u16)
        m = sh.extract_mesh()
        if rank == 0:
            ref = DenseTSDFVolume(vl, trunc, res, cfg["origin"], color=False, device=dev)
            for f0, f1 in DenseTSDFVolume.stream_chunks(F, 256, ramp=()):
                ref.integrate_u16_batch(depth_u16[f0:f1], None, intr, E[f0:f1], 1000.0, 3.0)
            rm = ref.extract_triangle_mesh()
            a, b = m.canonical_digest((res,) * 3), rm.canonical_digest((res,) * 3)
            parity["mesh_identical_to_1gpu"] = a == b
            parity["mesh_vertices"], parity["mesh_triangles"] = int(m.vertices.shape[0]), int(m.triangles.shape[0])
            parity["mesh_1gpu_vertices"], parity["mesh_1gpu_triangles"] = int(rm.vertices.shape[0]), int(rm.triangles.shape[0])
            log(f"{world}-GPU mesh identical to the 1-GPU mesh: {a == b} ({parity['mesh_vertices']} vertices, {parity['mesh_triangles']} triangles)")
            del ref, rm
        del m

    extras = {}
    ref_lit = None
    cadence = None
    deviation = None
    single = world == 1 and not emu
    if args.deviation and single:
        # brick-restart (fast path, oracle z_restart = 8) vs Open3D's literal march from z = 0, over ALL frames of the workload
        lit = DenseTSDFVolume(vl, trunc, res, cfg["origin"], color=False, device=dev)
        brk = DenseTSDFVolume(vl, trunc, res, cfg["origin"], color=False, device=dev)
        dd = depth_f if res <= 512 and not args.no_extras else ops.depth_from_u16(depth_u16, 1000.0, 3.0, dev)
        for f0, f1 in DenseTSDFVolume.stream_chunks(F, 256, ramp=()):
            lit.integrate_batch(dd[f0:f1], None, intr, E[f0:f1], zmarch=_lib.ZMARCH_LITERAL)
            brk.integrate_batch(dd[f0:f1], None, intr, E[f0:f1])
        (tl, wl), (tb, wb) = lit.export_dense(), brk.export_dense()
        occ = int((wl != 0).sum().item())
        flips = int((wl != wb).sum().item())
        same = wl == wb
        dt = (tl - tb).abs()
        deviation = {"frames": F, "occupied_voxels": occ, "voxels_with_different_weight": flips, "share": flips / max(occ, 1),
                     "max_weight_difference": float((wl - wb).abs().max().item()),
                     "voxels_with_tsdf_moved_over_1e-4_trunc_units": int(((dt > 1e-4) & same).sum().item()),
                     "mean_abs_dtsdf_where_weights_agree": float(dt[same].mean().item()), "max_abs_dtsdf": float(dt.max().item()),
                     "mesh_counts_literal": None, "mesh_counts_brick": None}
        ml, mb = lit.extract_triangle_mesh(), brk.extract_triangle_mesh()
        deviation["mesh_counts_literal"] = [int(ml.vertices.shape[0]), int(ml.triangles.shape[0])]
        deviation["mesh_counts_brick"] = [int(mb.vertices.shape[0]), int(mb.triangles.shape[0])]
        log(f"z-recurrence deviation (brick restart vs literal, {F} frames): {json.dumps(deviation)}")
        del lit, brk, tl, wl, tb, wb, dt, same, ml, mb

    # The legs below decorate the headline line; none of them may take it down: an exception is recorded in the JSON
    # (details.extras_error / cpu_error) and printed to stderr, the line is still emitted.
    def run_extras():
        nonlocal ref_lit, cadence
        def timed(fn, n=5, warm=2):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(n):
                fn()
            ev1.record()
            torch.cuda.synchronize()
            return ev0.elapsed_time(ev1) / n

        # ---- the object the reference's TSDF() literally builds: RGB8 + 32^3 unit activation (tsdf.py:7-12)
        if res % 32 == 0:
            _, col = S.render(cfg["surface"], E, K=cfg["K"], W=W, H=H, device=dev, with_color=True)
            org_u = unit_origin(cfg["origin"], vl)
            lvol = DenseTSDFVolume(vl, trunc, res, org_u, color=True, device=dev, unit_activation=True)
            lchunks = DenseTSDFVolume.stream_chunks(F, chunk, ramp=())

            def lit_step():
                lvol.integrate_u16_chunks(depth_u16, col, intr, E, lchunks, 1000.0, 3.0)

            ms = timed(lit_step, n=max(3, args.steps // 4))
            host_col = torch.empty((F, H, W, 3), dtype=torch.uint8).pin_memory()
            host_col.copy_(col)
            host_d = torch.empty((F, H, W), dtype=torch.uint16).pin_memory()
            host_d.copy_(depth_u16)
            hv, ht = {}, {}

            def lit_e2e():
                lvol.integrate_host(host_d, host_col, intr, E, 1000.0, 3.0, chunk)
                m = lvol.extract_triangle_mesh()
                hv["v"], ht["t"] = m.vertices.cpu(), m.triangles.cpu()
                hv["c"] = m.vertex_colors.cpu()

            ms2 = timed(lit_e2e, n=max(3, args.steps // 4), warm=1)
            uf_lit = None
            ref_lit = {"value": F / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "e2e_value": F / (ms2 / 1e3), "e2e_ms_per_step": ms2,
                       "what": "RGB8 colour integration + ScalableTSDFVolume unit activation (volume_unit_resolution 32, depth_sampling_stride 8), "
                               "float32 z recurrence restarted at every unit base = Open3D's literal per-unit arithmetic; e2e adds H2D of u16 depth + "
                               "RGB8 colour, one coloured mesh extraction and its D2H",
                       "h2d_bytes_per_step": F * H * W * 5 + F * 128, "mesh_vertices": int(hv["v"].shape[0]), "mesh_triangles": int(ht["t"].shape[0]),
                       "clip": lvol.clip_stats()}
            log(f"reference-literal (RGB8 + unit activation): {ref_lit['value']:.1f} frames/s resident, {ref_lit['e2e_value']:.1f} e2e")
            del lvol, host_col, host_d

            # ---- SLAM cadence (N/3DM/slam.py:179,195): one build_3D_map + one extract_pcd per frame, through the drop-in
            tsdf = TSDF(voxel_length=vl, sdf_trunc=trunc, resolution=res, origin=org_u, device=dev)
            n_cad = min(F, 200)
            frames = [RGBDImage(col[i], depth_f[i]) for i in range(n_cad)]
            pts = []

            rec_frac = []

            def cadence_run():
                tsdf.tsdf.reset()
                pts.clear()
                rec_frac.clear()
                for i in range(n_cad):
                    tsdf.build_3D_map(frames[i], intr, E[i])
                    pts.append(int(tsdf.extract_pcd().points.shape[0]))
                    cand, rec = tsdf.tsdf.points_last_stats()
                    rec_frac.append(rec / max(cand, 1))

            cadence_run()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            cadence_run()
            torch.cuda.synchronize()
            dt_cad = time.perf_counter() - t0
            # where a frame's time goes: integration stages by CUDA events, the rest is extract_pcd + Python
            tsdf.tsdf.reset()
            tsdf.tsdf.profile(True)
            t1 = time.perf_counter()
            for i in range(n_cad):
                tsdf.build_3D_map(frames[i], intr, E[i])
            torch.cuda.synchronize()
            dt_int = time.perf_counter() - t1
            st_cad, n_l = tsdf.tsdf.profile_read_stages()
            tsdf.tsdf.profile(False)
            cadence = {"value": n_cad / dt_cad, "unit": UNIT, "frames": n_cad, "ms_per_frame": 1e3 * dt_cad / n_cad,
                       "what": "TSDF.build_3D_map(rgbd) + TSDF.extract_pcd() per frame (RGB8, unit activation), wall clock incl. Python",
                       "points_last_frame": pts[-1], "point_counts": list(pts),
                       "incremental_extraction": "bricks whose 3x3x3 neighbourhood the frame changed are re-extracted, the rest is copied from a per-brick cache",
                       "bricks_recomputed_share_mean": float(np.mean(rec_frac)), "bricks_recomputed_share_last": float(rec_frac[-1]),
                       "integrate_only_ms_per_frame": 1e3 * dt_int / n_cad,
                       "integrate_stage_ms_per_frame": {k: v / max(n_l, 1) for k, v in st_cad.items()}}
            log(f"SLAM cadence: {cadence['value']:.1f} frames/s ({cadence['ms_per_frame']:.2f} ms per integrate + extract_pcd)")
            del tsdf, frames

        # ---- dense rule with the reference's per-unit arithmetic (literal Open3D voxel centres + z recurrence per 32^3 unit)
        if res % 32 == 0:
            uvol = DenseTSDFVolume(vl, trunc, res, unit_origin(cfg["origin"], vl), color=False, device=dev, unit_arithmetic=True)
            uchunks = DenseTSDFVolume.stream_chunks(F, chunk, ramp=())
            ms = timed(lambda: uvol.integrate_u16_chunks(depth_u16, None, intr, E, uchunks, 1000.0, 3.0), n=max(3, args.steps // 4))
            extras["dense_unit_arithmetic"] = {"value": F / (ms / 1e3), "unit": UNIT, "ms_per_step": ms,
                                               "what": "every voxel of the box integrated (dense rule) with ScalableTSDFVolume's per-unit voxel centres and float32 z "
                                                       "recurrence: the oracle runs Open3D's literal arithmetic (z_restart 0), nothing bent to the kernel"}
            del uvol

        # ---- row f4: the tensor-pipeline integrator behind `MAP` (N/3DM/tsdf.py:56-108), reference defaults
        # (voxel_size 5.8 mm, 16^3 blocks, trunc_voxel_multiplier 8) on a 256^3 box around the scene
        try:
            from bodyslam_b200.tsdf import MAP

            Kmat = np.array([[cfg["K"][0], 0, cfg["K"][2]], [0, cfg["K"][1], cfg["K"][3]], [0, 0, 1.0]])
            mp = MAP(W, H, Kmat, "CUDA:0" if dev.index == 0 else f"CUDA:{dev.index}", 1000.0, resolution=256, color=False)
            n_map = min(F, 256)
            poses = np.stack([np.linalg.inv(E[i]) for i in range(n_map)])
            ms = timed(lambda: mp.integrate_batch(depth_u16[:n_map], None, poses, 3.0), n=3, warm=1)
            extras["map_tensor_pipeline"] = {"frames_per_s": n_map / (ms / 1e3), "frames": n_map, "voxel_size_m": 0.0058, "resolution": 256,
                                             "mesh_triangles": int(mp.extract_mesh().triangles.shape[0]), "clip": mp.clip_stats()}
            del mp
        except Exception as e:      # the extra leg must never take the headline down
            extras["map_tensor_pipeline"] = {"error": f"{type(e).__name__}: {e}"}

        # ---- BASELINE configs[2]: 64-frame batched 1080p depth scale + colorize + back-project
        from bodyslam_b200 import mdem

        # input: 64 views of the same synthetic scene rendered at 1080p (intrinsics scaled x3), 2 % invalid pixels,
        # as float32 METRES (what ZoeDepth hands to the MDEM post-processing)
        B, Hh, Ww = 64, 1080, 1920
        K1080 = tuple(k * 3.0 for k in cfg["K"])
        Eb = E[np.linspace(0, len(E) - 1, B).astype(int)]
        d1080, _ = S.render(cfg["surface"], Eb, K=K1080, W=Ww, H=Hh, device=dev, with_color=False)
        metres = (d1080.to(torch.float32) / 1000.0).contiguous()
        del d1080
        lut = mdem.get_cmap_lut("viridis")
        ms = timed(lambda: ops.colorize_u16(lut, depth_m=metres, invalid_val=0))
        px = B * Hh * Ww
        peak = load_peaks()[0]
        extras["configs2_k1_scale_colorize_1080p_x64"] = {"ms": ms, "frames_per_s": B / (ms / 1e3), "algorithmic_GBps": 10 * px / 1e9 / (ms / 1e3),
                                                          "frac_of_hbm_peak": 10 * px / 1e9 / (ms / 1e3) / peak, "algorithmic_bytes": "10 B/px (4 r + 2 w + 4 w)",
                                                          "input": "64 rendered 1080p views of the workload's scene, f32 metres, 2 % invalid"}
        res_bp = {}

        def bp():
            res_bp["xyz"], _ = ops.backproject(metres, K1080, Eb)

        ms = timed(bp, 3)
        nvalid = int(res_bp["xyz"].shape[0])
        by = 4 * px + 12 * nvalid
        extras["configs2_k2_backproject_1080p_x64"] = {"ms": ms, "points": nvalid, "frames_per_s": B / (ms / 1e3), "algorithmic_GBps": by / 1e9 / (ms / 1e3),
                                                       "frac_of_hbm_peak": by / 1e9 / (ms / 1e3) / peak, "algorithmic_bytes": "4 B/px + 12 B/valid point"}
        del metres, res_bp
        # ---- BASELINE configs[0]: one 640x480 frame: scale + colorize + 3DM depth scaling + back-projection (latency)
        one = (depth_u16[0].to(torch.float32) / 1000.0).contiguous()

        def single_frame():
            rgba, u16 = ops.colorize_u16(lut, depth_m=one, invalid_val=0)
            d = ops.depth_from_u16(u16, 1000.0, 3.0, dev)
            return ops.backproject(d, cfg["K"], E[0])

        t0 = time.perf_counter()
        for _ in range(20):
            single_frame()
        torch.cuda.synchronize()
        ms = timed(single_frame, 20)
        extras["configs0_single_frame_scale_colorize_backproject"] = {"ms": ms, "frames_per_s": 1e3 / ms, "note": "latency of four API calls incl. one D2H of the point count"}
        ms = timed(lambda: ops.depth_from_u16(depth_u16, 1000.0, 3.0), 3)
        extras["a4_depth_from_u16_GBps"] = 6 * F * H * W / 1e9 / (ms / 1e3)
        t0 = time.perf_counter()
        pcd = vol.extract_point_cloud()
        torch.cuda.synchronize()
        extras["points_ms"], extras["points"] = 1e3 * (time.perf_counter() - t0), int(pcd.points.shape[0])
        del pcd

    if single and not args.no_extras and res <= 512:
        try:
            run_extras()
        except Exception as e:
            import traceback
            traceback.print_exc(file=sys.stderr)
            extras["extras_error"] = f"{type(e).__name__}: {e}"

    # ---- CPU baseline + parity (rank 0, N = 1): the oracle on a bounded sample of the same frames, then the
    # SAME frames in the SAME order into fresh GPU volumes: tsdf / weight grids must be bit-identical
    cpu = None
    cpu_error = None

    def run_cpu_legs():
        nonlocal cpu
        import oracle

        ids = np.unique(np.linspace(0, F - 1, min(F, 400)).astype(int))
        ids = ids[np.random.default_rng(0).permutation(len(ids))]   # any prefix of the sample is spread over the trajectory
        sel = torch.as_tensor(ids, device=dev)
        sample_u16 = depth_u16.view(torch.int16)[sel].view(torch.uint16)
        _, sample_rgb = S.render(cfg["surface"], E[ids], K=cfg["K"], W=W, H=H, device=dev, with_color=True)
        su16_np = sample_u16.cpu().numpy()
        legs = cpu_legs(cfg, E, su16_np, sample_rgb.cpu().numpy(), ids, res, vl, trunc, args.cpu_budget)
        log(f"CPU oracle: dense {legs['dense_fps']:.1f} frames/s ({legs['dense_frames']} frames), scalable {legs.get('scalable_fps', 0):.1f}, "
            f"scalable with Open3D's schedule {legs.get('scalable_open3d_schedule_fps', 0):.1f}, {legs['cores']} threads")
        # dense rule
        n = legs["dense_frames"]
        V = legs.pop("dense_volume")
        g = DenseTSDFVolume(vl, trunc, res, cfg["origin"], color=False, device=dev)
        gc = torch.zeros(n, dtype=torch.int64, device=dev)
        g.integrate_u16_batch(sample_u16[:n], None, intr, E[ids[:n]], 1000.0, 3.0, update_counts=gc)
        t, w = g.export_dense()
        gm = g.extract_triangle_mesh()
        om = V.extract_mesh()
        parity["dense"] = {"frames": n, "resolution": res, "tsdf_equal": digest(t.cpu().numpy()) == digest(V.tsdf), "weight_equal": digest(w.cpu().numpy()) == digest(V.weight),
                           "update_counts_equal": gc.cpu().tolist() == [int(c) for c in legs["dense_counts"]],
                           "mesh_counts_equal": [int(gm.vertices.shape[0]), int(gm.triangles.shape[0])] == [len(om["vertices"]), len(om["triangles"])],
                           "mesh_vertices": int(gm.vertices.shape[0]), "mesh_triangles": int(gm.triangles.shape[0]),
                           "occupied_voxels": int(V.occupied()), "oracle": "oracle/o3d_oracle.c orc_tsdf_integrate (z_restart 8) + orc_extract_mesh"}
        ca = gm.canonical((res,) * 3)
        from bodyslam_b200.geometry import TriangleMesh
        cb = TriangleMesh(om["vertices"], om["triangles"], None, om["keys"]).canonical((res,) * 3)
        parity["dense"]["mesh_topology_equal"] = bool(np.array_equal(ca[0], cb[0]) and np.array_equal(ca[2], cb[2]))
        parity["dense"]["mesh_max_vertex_error_m"] = float(np.abs(ca[1] - cb[1]).max()) if len(ca[1]) == len(cb[1]) and len(ca[1]) else None
        del V, g, t, w, gm, om, ca, cb
        if "scalable_volume" in legs:
            n = legs["scalable_frames"]
            Sv = legs.pop("scalable_volume")
            g = DenseTSDFVolume(vl, trunc, res, unit_origin(cfg["origin"], vl), color=True, device=dev, unit_activation=True)
            gc = torch.zeros(n, dtype=torch.int64, device=dev)
            g.integrate_u16_batch(sample_u16[:n], sample_rgb[:n], intr, E[ids[:n]], 1000.0, 3.0, update_counts=gc)
            t, w, c = g.export_dense(with_color=True)
            gm = g.extract_triangle_mesh()
            om = Sv.extract_mesh()
            parity["scalable_rgb8"] = {"frames": n, "resolution": res, "tsdf_equal": digest(t.cpu().numpy()) == digest(Sv.tsdf), "weight_equal": digest(w.cpu().numpy()) == digest(Sv.weight),
                                       "update_counts_equal": gc.cpu().tolist() == [int(x) for x in legs["scalable_counts"]],
                                       "color_max_abs_error_0_255": float(np.abs(c.cpu().numpy().reshape(-1) - Sv.color).max()),
                                       "mesh_counts_equal": [int(gm.vertices.shape[0]), int(gm.triangles.shape[0])] == [len(om["vertices"]), len(om["triangles"])],
                                       "mesh_vertices": int(gm.vertices.shape[0]), "mesh_triangles": int(gm.triangles.shape[0]), "occupied_voxels": int(Sv.occupied()),
                                       "oracle": "oracle/o3d_oracle.c orc_scalable_integrate (z_restart 0 = Open3D's literal per-unit recurrence) + orc_extract_mesh"}
            del Sv, g, t, w, c, gm, om
        if res % 32 == 0:
            n = min(legs["dense_frames"], 48)
            org_u = unit_origin(cfg["origin"], vl)
            Av = oracle.o3d.Volume(res, vl, trunc, org_u)
            ac = [int(Av.integrate_scalable(oracle.o3d.depth_from_u16(su16_np[k]), cfg["K"], E[ids[k]], all_units=True)) for k in range(n)]
            g = DenseTSDFVolume(vl, trunc, res, org_u, color=False, device=dev, unit_arithmetic=True)
            gc = torch.zeros(n, dtype=torch.int64, device=dev)
            g.integrate_u16_batch(sample_u16[:n], None, intr, E[ids[:n]], 1000.0, 3.0, update_counts=gc)
            t, w = g.export_dense()
            parity["dense_unit_arithmetic"] = {"frames": n, "resolution": res, "tsdf_equal": digest(t.cpu().numpy()) == digest(Av.tsdf),
                                               "weight_equal": digest(w.cpu().numpy()) == digest(Av.weight), "update_counts_equal": gc.cpu().tolist() == ac,
                                               "oracle": "oracle/o3d_oracle.c orc_scalable_integrate, every unit touched, z_restart 0 (Open3D's literal per-unit arithmetic)"}
            del Av, g, t, w
        if cadence is not None:
            # the same cadence on the CPU oracle (ScalableTSDFVolume rule + extract_point_cloud), first frames of the trajectory
            n_c = 3
            d3, c3 = depth_u16[:n_c].cpu().numpy(), S.render(cfg["surface"], E[:n_c], K=cfg["K"], W=W, H=H, device=dev, with_color=True)[1].cpu().numpy()
            Cv = oracle.o3d.Volume(res, vl, trunc, unit_origin(cfg["origin"], vl), with_color=True)
            cp, t0 = [], time.perf_counter()
            for i in range(n_c):
                Cv.integrate_scalable(oracle.o3d.depth_from_u16(d3[i]), cfg["K"], E[i], rgb=c3[i])
                cp.append(int(len(Cv.extract_points()["points"])))
            dt_c = time.perf_counter() - t0
            cadence["cpu_oracle"] = {"value": n_c / dt_c, "unit": UNIT, "frames": n_c, "point_counts": cp,
                                     "point_counts_equal_gpu": cp == cadence["point_counts"][:n_c], "cores": legs["cores"]}
            cadence["point_counts"] = cadence["point_counts"][:8] + ["..."] + cadence["point_counts"][-2:]
            parity["slam_cadence_point_counts_equal"] = cadence["cpu_oracle"]["point_counts_equal_gpu"]
            del Cv
        log(f"parity: {json.dumps(parity)}")
        cpu = {"value": legs["dense_fps"], "unit": UNIT, "cores": legs["cores"], "kind": "port",
               "sample": f"{legs['dense_frames']} frames drawn evenly (seeded shuffle, {args.cpu_budget:g} s budget) from the {F}-frame trajectory, {res}^3 dense sweep per "
                         f"frame (oracle/o3d_oracle.c, OpenMP over x like Open3D); the GPU integrates the same frames in the same order for `parity`",
               "dense_fps": legs["dense_fps"], "scalable_fps": legs.get("scalable_fps"), "scalable_frames": legs.get("scalable_frames"),
               "scalable_open3d_schedule_fps": legs.get("scalable_open3d_schedule_fps"),
               "scalable_note": "ScalableTSDFVolume rule + RGB8 (what the reference's TSDF() runs): only the 32^3 units activated by the stride-8 sampled points are swept; "
                                "scalable_fps spreads the units over the threads, scalable_open3d_schedule_fps keeps Open3D's own schedule (units serial, OpenMP over x inside a unit)"}

    if rank == 0 and single and not args.no_cpu_baseline:
        try:
            run_cpu_legs()
        except Exception as e:
            import traceback
            traceback.print_exc(file=sys.stderr)
            cpu_error = f"{type(e).__name__}: {e}"

    if rank == 0:
        peak, peak_src = load_peaks()
        # per <=256-frame chunk: 2 memsets + depth_stats (+ fused a4), tmax_mip, frame_soa, super_cull, brick_cull, order, brick_integrate
        launches_per_step = 7 * len(chunks)
        steps_timed = k_launches // len(chunks)
        ach = (bytes_algo_local * steps_timed / 1e9) / (k_ms * (steps_timed * len(chunks) / k_launches) / 1e3) if k_ms > 0 and steps_timed else None
        traffic, traffic_src = load_traffic(args, world, res, F)
        line = {
            "metric": metric_name(res), "value": fps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, F, W, H, res, vl, trunc),
            "details": {"step": "a4 depth scaling (fused into the first pass) + K3 integrate of all frames, volume resident",
                        "culling": {"voxels_tested_per_frame": cull["voxels_tested"] / F, "updated_over_tested": (int(uf_local.sum().item()) / cull["voxels_tested"]) if cull["voxels_tested"] else None},
                        "resident_frames": (None if world == 1 else ("1/N of every chunk resident in each rank's HBM, all-gathered over NVLink per chunk" if dev_share is not None
                                                                     else "all frames resident on rank 0, broadcast over NVLink per chunk")),
                        "parallelism": (f"round-robin brick-layer z-shards x{world}" if interleaved else f"z-slab x{world}") if world > 1 else
                                       (f"EMULATED shard {emu[0]} of {emu[1]} on one GPU (development aid, not a bench value)" if emu else "single GPU"),
                        "voxels_updated_per_frame": uf_total / F, "timeline_ms_per_step_by_rank": timeline, **mesh_info, **extras},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "hbm", "kernel": "brick_integrate_kernel", "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": (ach / peak) if ach else None, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": bytes_algo_local, "kernel_ms_per_step": k_ms / k_launches * len(chunks) if k_launches else None,
                         "kernel_launches": k_launches,
                         "dram_frac_of_peak": (traffic / (k_ms / k_launches / 1e3) / 1e9 / peak) if traffic and k_launches else None,
                         "note": "achieved = ALGORITHMIC bytes (16 B x voxels updated per frame, oracle-equal count, + 4*W*H per frame; SURVEY 8d) over the CUDA-event time of "
                                 "the kernel. The kernel keeps a voxel in registers across the <=256 frames of a launch, so the DRAM bytes actually moved (`traffic`, "
                                 "`dram_frac_of_peak`) are far below this figure: the kernel is issue-bound, not HBM-bound"},
            "cpu_baseline": cpu,
            "cpu_error": cpu_error,
            "parity": parity or None,
            "reference_literal": ref_lit,
            "slam_cadence": cadence,
            "zmarch_deviation": deviation,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
