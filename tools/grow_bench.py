"""Box growth measurement: one JSON line.

relocate     bslam_tsdf_copy into a larger box (the growth step), with colour: 256^3 -> 512^3 and 512^3 -> 1024x512x512.
             CUDA events over repeated copies after a warm-up; GB/s = (source storage read + destination storage written)
             over kernel time, against the measured HBM peak.
idle_cost    what auto-grow costs when nothing grows: the laparoscopy sweep (BASELINE configs[3] geometry, 512^3 box that
             holds it) at the SLAM cadence, build_3D_map + extract_pcd per frame, TSDF(grow=True) against TSDF(), the two
             alternated three times in one process (frames/s, median).
lumen        the colonoscopy lumen (Lumen(), 2 mm voxels) over 300 frames from a 128^3 box around the first camera with
             grow=True, against a box pre-sized to the grown one's final box: frames/s end to end at the SLAM cadence,
             growth events, final box, peak device memory allocated through torch (the volume storage; the library's own
             scratch buffers are not included).
Run from the repository root: python tools/grow_bench.py
"""
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bodyslam_b200 import _lib, ops  # noqa: E402
from bodyslam_b200 import synthetic as S  # noqa: E402
from bodyslam_b200.geometry import PinholeCameraIntrinsic, RGBDImage  # noqa: E402
from bodyslam_b200.tsdf import TSDF, DenseTSDFVolume  # noqa: E402

HBM_PEAK_GBS = 6534.8      # measured HBM copy bandwidth of a B200 (README), the peak of every roofline here


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.splitlines()[0].split(",")))) if r.returncode == 0 and r.stdout else {}


def relocate(dev, src_res, dst_res, reps=10):
    L = _lib.load()
    vl = 0.001
    src = DenseTSDFVolume(vl, 0.005, src_res, (0.0, 0.0, 0.0), color=True, device=dev)
    off = [(d - s) // 2 // 8 * 8 for s, d in zip(src_res, dst_res)]
    dst = DenseTSDFVolume(vl, 0.005, dst_res, tuple(-o * vl for o in off), color=True, device=dev)
    st = _lib.stream_ptr(dev)
    for _ in range(2):
        _lib.check(L.bslam_tsdf_copy(src._h, dst._h, st))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        _lib.check(L.bslam_tsdf_copy(src._h, dst._h, st))
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b) / reps       # includes the 24-byte counter copy that follows each kernel
    nbytes = L.bslam_tsdf_storage_bytes(*src_res, 1) + L.bslam_tsdf_storage_bytes(*dst_res, 1)
    gbs = nbytes / ms / 1e6
    return {"src": list(src_res), "dst": list(dst_res), "ms": round(ms, 3), "bytes": int(nbytes), "GB_s": round(gbs, 1),
            "share_of_hbm_peak": round(gbs / HBM_PEAK_GBS, 3)}


def slam_cadence(t, depth, color, E, intr):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(depth.shape[0]):
        t.build_3D_map(RGBDImage(color[i], depth[i]), intr, E[i])
        t.extract_pcd()
    torch.cuda.synchronize()
    return depth.shape[0] / (time.perf_counter() - t0)


def main():
    dev = torch.device("cuda", 0)
    out = {"gpu": gpu_info()}
    out["relocate"] = [relocate(dev, (256,) * 3, (512,) * 3), relocate(dev, (512,) * 3, (1024, 512, 512))]
    torch.cuda.empty_cache()

    cfg = S.config("laparoscopy512")
    F = 300
    E = cfg["extrinsics"](cfg["frames"])[:: cfg["frames"] // F][:F]
    d16, col = S.render(cfg["surface"], E, K=cfg["K"], W=cfg["W"], H=cfg["H"], device=dev)
    depth = ops.depth_from_u16(d16, 1000.0, 3.0, dev)
    intr = PinholeCameraIntrinsic(cfg["W"], cfg["H"], *cfg["K"])
    kw = dict(voxel_length=cfg["voxel_length"], sdf_trunc=cfg["sdf_trunc"], resolution=cfg["resolution"], origin=cfg["origin"], device=dev)
    rates = {False: [], True: []}
    grown = 0
    slam_cadence(TSDF(**kw), depth[:20], col[:20], E[:20], intr)      # warm-up
    for _ in range(3):
        for g in (False, True):
            t = TSDF(grow=g, **kw)
            rates[g].append(slam_cadence(t, depth, col, E, intr))
            grown += t.tsdf.growth_events
            del t
    out["idle_cost"] = {"frames": F, "resolution": cfg["resolution"], "fps_grow_off": [round(r, 1) for r in rates[False]],
                        "fps_grow_on": [round(r, 1) for r in rates[True]], "median_off": round(statistics.median(rates[False]), 1),
                        "median_on": round(statistics.median(rates[True]), 1), "growth_events": grown}
    del depth, col, d16
    torch.cuda.empty_cache()

    lum = S.Lumen()
    E = S.lumen_trajectory(lum, 300, step=0.001)
    d16, col = S.render(lum, E, device=dev, seed=3)
    depth = ops.depth_from_u16(d16, 1000.0, 3.0, dev)
    intr = PinholeCameraIntrinsic(640, 480, *S.K_640)
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    t = TSDF(voxel_length=0.002, sdf_trunc=0.01, resolution=128, origin=(-0.128,) * 3, device=dev, grow=True)
    fps_grow = slam_cadence(t, depth, col, E, intr)
    peak_grow = torch.cuda.max_memory_allocated(dev) - base
    origin = tuple(t.tsdf.origin.tolist())
    box = dict(origin=[round(x, 6) for x in origin], resolution=[t.tsdf.nx, t.tsdf.ny, t.tsdf.nz])
    events = t.tsdf.growth_events
    final_bytes = t.tsdf._storage.numel()
    del t
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    p = TSDF(voxel_length=0.002, sdf_trunc=0.01, resolution=tuple(box["resolution"]), origin=origin, device=dev)
    fps_pre = slam_cadence(p, depth, col, E, intr)
    peak_pre = torch.cuda.max_memory_allocated(dev) - base
    out["lumen"] = {"frames": 300, "start": [128] * 3, "final_box": box, "growth_events": events, "fps_grow": round(fps_grow, 1),
                    "fps_presized": round(fps_pre, 1), "peak_torch_bytes_grow": int(peak_grow), "peak_torch_bytes_presized": int(peak_pre),
                    "final_storage_bytes": int(final_bytes)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
