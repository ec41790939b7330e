"""Multi-scale RGB-D odometry measurement: one JSON line.

single_pair   rgbd_odometry_multi_scale on consecutive frames of the laparoscopy sweep (BASELINE configs[3], 640x480 u16
              depth + u8 colour), one pair per call with a synchronise (the VO cadence): Hybrid (10, 5, 3) and
              PointToPlane (6, 3, 1), median / p90 ms over 200 pairs.
sequence      rgbd_odometry_sequence over the 1000-frame sweep, Hybrid (10, 5, 3): pairs/s.
map_loop      MAP at 256^3 (2 mm voxels, colour): integrate + synthesize_model_frame + track_frame_to_model per frame.
cpu_baseline  the CPU reference (tests/odometry_ref.c, all host threads): prepare + Hybrid track of 8 pairs.
parity        max |T_gpu - T_ref| over those 8 pairs, and whether their iteration counts agree.
reduce        bslam_odom_linearize (reduce + sum kernels) at level 0 for 64 pairs, Hybrid, CUDA events: us per pair
              iteration, and its algorithmic bytes (per source pixel: vertex + intensity read, 16 B; per inlier: the
              target's depth, intensity and 4 gradients, 24 B) over that time.  A pair's 8.8 MB of maps stays in L2.
trace         torch.profiler over 20 single Hybrid pairs: kernel time per pair and launches per pair, beside the wall time.
Run from the repository root: python tools/odometry_bench.py
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import odometry_ref as R  # noqa: E402
from bodyslam_b200 import _lib  # noqa: E402
from bodyslam_b200 import odometry as od  # noqa: E402
from bodyslam_b200 import synthetic as S  # noqa: E402
from bodyslam_b200.geometry import RGBDImage  # noqa: E402
from bodyslam_b200.tsdf import MAP  # noqa: E402

HBM_PEAK_GBS = 6534.8      # measured HBM copy bandwidth of a B200 (SURVEY.md)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.splitlines()[0].split(",")))) if r.returncode == 0 and r.stdout else {}


class Frame:
    def __init__(self, d, c):
        self.o3d_t_depth, self.o3d_t_color, self.depth_max = d, c, 3.0


def main():
    dev = torch.device("cuda", 0)
    cfg = S.config("laparoscopy512")
    F, W, H, K = cfg["frames"], cfg["W"], cfg["H"], cfg["K"]
    K3 = np.array([[K[0], 0, K[2]], [0, K[1], K[3]], [0, 0, 1]])
    E = cfg["extrinsics"](F)
    depth = torch.empty((F, H, W), dtype=torch.uint16, device=dev)
    color = torch.empty((F, H, W, 3), dtype=torch.uint8, device=dev)
    for lo in range(0, F, 100):
        depth[lo:lo + 100], color[lo:lo + 100] = S.render(cfg["surface"], E[lo:lo + 100], K=K, W=W, H=H, device=dev, first_frame=lo)
    out = {"metric": "rgbd_odometry", "gpu": gpu_info(), "image": f"{W}x{H}", "frames": F}

    # ---- single pair per call
    runs = {"hybrid_10_5_3": dict(method=od.Method.Hybrid), "point_to_plane_6_3_1": dict(
        method=od.Method.PointToPlane, criteria_list=[od.OdometryConvergenceCriteria(n) for n in (6, 3, 1)])}
    out["single_pair"] = {}
    for name, kw in runs.items():
        pair = lambda i: od.rgbd_odometry_multi_scale(RGBDImage(color[i], depth[i]), RGBDImage(color[i + 1], depth[i + 1]), K3, **kw)  # noqa: E731
        for i in range(10):
            pair(i)
        ms = []
        for i in range(200):
            t0 = time.perf_counter()
            try:
                pair(i)
            except RuntimeError:
                pass
            ms.append((time.perf_counter() - t0) * 1e3)
        out["single_pair"][name] = {"pairs": 200, "median_ms": float(np.median(ms)), "p90_ms": float(np.percentile(ms, 90))}

    # ---- sequence
    od.rgbd_odometry_sequence(depth[:70], color[:70], K3)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    seq = od.rgbd_odometry_sequence(depth, color, K3)
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    out["sequence"] = {"pairs": F - 1, "s": s, "pairs_per_s": (F - 1) / s, "singular": int(seq.status.sum().item())}

    # ---- MAP loop
    m = MAP(W, H, K3, "CUDA:0", 1000.0, voxel_size=0.002, resolution=256)
    T = np.linalg.inv(E[0])
    n_map = 200
    t0 = None
    for i in range(n_map):
        if i == 10:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
        fr = Frame(depth[i], color[i])
        if i:
            try:
                T = T @ m.track_frame_to_model(fr, m.synthesize_model_frame()).transformation
            except RuntimeError:      # singular: keep the previous pose
                pass
        m.integrate(fr, i, T)
    torch.cuda.synchronize()
    ms_map = (time.perf_counter() - t0) * 1e3 / (n_map - 10)
    out["map_loop"] = {"box": "256^3 @ 2 mm, colour", "frames": n_map - 10, "ms_per_frame": ms_map, "frames_per_s": 1e3 / ms_map,
                       "drift_m": float(np.linalg.norm(T[:3, 3] - np.linalg.inv(E[n_map - 1])[:3, 3]))}

    # ---- cpu baseline + parity
    ids = np.linspace(0, F - 2, 8).astype(int)
    dn, cn = depth.cpu().numpy(), color.cpu().numpy()
    t0 = time.perf_counter()
    refs = []
    for i in ids:
        fr = R.Frames(dn[i:i + 2], cn[i:i + 2], K, 3)
        refs.append(fr.track(0, 1, R.HYBRID))
    cpu_s = (time.perf_counter() - t0) / len(ids)
    Tg = seq.transformations.cpu().numpy()
    it = seq.iterations.cpu().numpy()
    out["cpu_baseline"] = {"pairs": len(ids), "threads": os.cpu_count(), "s_per_pair": cpu_s, "pairs_per_s": 1 / cpu_s}
    out["parity"] = {"max_abs_T_dev": float(max(np.abs(Tg[i] - r["T"]).max() for i, r in zip(ids, refs))),
                     "iterations_equal": bool(all(list(it[i]) == list(r["iters"]) for i, r in zip(ids, refs)))}

    # ---- reduce kernel
    L = _lib.load()
    P = 64
    buf = torch.empty(65 * L.bslam_odom_frame_bytes(H, W, 3) // 4, dtype=torch.float32, device=dev)
    K4 = np.asarray(K, np.float64)
    _lib.check(L.bslam_odom_prepare(_lib.ptr(depth[:65]), 0, _lib.ptr(color[:65]), 0, 65, H, W, 3, _lib.ptr(K4), 1000.0, 3.0, 0.07, _lib.ptr(buf),
                                    _lib.stream_ptr()))
    pairs = np.array([[i, i + 1] for i in range(P)], np.int32)
    Ts = np.tile(np.eye(4).reshape(1, 16), (P, 1))
    ws = torch.empty(L.bslam_odom_workspace_bytes(P, H, W, 3), dtype=torch.uint8, device=dev)
    sums = torch.empty((P, 29), dtype=torch.float64, device=dev)

    def lin():
        _lib.check(L.bslam_odom_linearize(_lib.ptr(buf), 65, _lib.ptr(pairs), P, H, W, 3, 0, _lib.ptr(K4), 2, 0.07, 0.05, 0.1, _lib.ptr(Ts), _lib.ptr(sums),
                                          _lib.ptr(ws), _lib.stream_ptr()))
    for _ in range(5):
        lin()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(50):
        lin()
    b.record()
    b.synchronize()
    us = a.elapsed_time(b) * 1e3 / 50 / P
    inliers = float(sums[:, 28].mean().item())
    nbytes = 16.0 * W * H + 24.0 * inliers
    out["reduce"] = {"pairs_per_launch": P, "us_per_pair_iteration": us, "inliers_per_pair": inliers, "algorithmic_bytes_per_pair": nbytes,
                     "achieved_gb_per_s": nbytes / (us * 1e3), "hbm_peak_gb_per_s": HBM_PEAK_GBS, "share_of_hbm_peak": nbytes / (us * 1e3) / HBM_PEAK_GBS}

    # ---- trace of single pairs
    try:
        out["trace"] = trace(color, depth, K3)
    except Exception as e:       # the profiler's event API differs between torch versions
        out["trace"] = {"error": repr(e)}
    print(json.dumps(out))


def trace(color, depth, K3):
    from torch.profiler import ProfilerActivity, profile

    pair = lambda i: od.rgbd_odometry_multi_scale(RGBDImage(color[i], depth[i]), RGBDImage(color[i + 1], depth[i + 1]), K3)  # noqa: E731
    t0 = time.perf_counter()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i in range(20):
            pair(i)
    wall = (time.perf_counter() - t0) * 1e3 / 20
    kern = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" and e.name.startswith(("_ZN5bslam", "bslam", "void bslam")):
            k = e.name.split("(")[0]
            kern.setdefault(k, [0, 0.0])
            kern[k][0] += 1
            kern[k][1] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    ktot = sum(v[1] for v in kern.values()) / 20 / 1e3
    return {"pairs": 20, "wall_ms_per_pair_profiled": wall, "kernel_ms_per_pair": ktot,
                    "launches_per_pair": sum(v[0] for v in kern.values()) / 20,
            "kernels": {k.replace("void ", ""): {"calls": v[0], "us": v[1]} for k, v in kern.items()}}


if __name__ == "__main__":
    main()
