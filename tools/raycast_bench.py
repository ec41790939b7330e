"""Ray-cast measurement: one JSON line.

tsdf512       BASELINE configs[3] (laparoscopy512, 1000 frames) integrated in full, then ray cast at 640x480 (depth,
              vertex, normal) from 256 trajectory poses: 64 poses per call (frames/s, Mrays/s) and one pose per call
              with a synchronise, the SLAM cadence (median ms per frame).
map_defaults  MAP at the reference defaults (5.8 mm voxels, 256^3 box, trunc_voxel_multiplier 8, no colour) on the same
              frames: integrate + synthesize_model_frame per frame (frames/s).
cpu_baseline  the ray cast's CPU reference (tests/raycast_ref.c, all host threads) on 8 of the poses.
parity        the CPU reference ray casts the GPU's own exported grids (and MAP's allocated blocks) for those 8 poses (MAP:
              from its last pose); hit masks and depth must be equal.
roofline      algorithmic bytes (8 B per voxel sample the reference's march read + output bytes) over the batched call
              time, against the measured HBM peak.  The march is a chain of dependent gathers per ray, so a low share
              of peak is expected: the kernel is bound by latency, not bandwidth.
Times are CUDA events after a warm-up.  Run from the repository root: python tools/raycast_bench.py
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

import oracle  # noqa: E402
import raycast_ref  # noqa: E402
from bodyslam_b200 import synthetic as S  # noqa: E402
from bodyslam_b200.geometry import PinholeCameraIntrinsic  # noqa: E402
from bodyslam_b200.tsdf import MAP, DenseTSDFVolume  # noqa: E402

HBM_PEAK_GBS = 6534.8      # measured HBM copy bandwidth of a B200 (SURVEY.md), the peak of every roofline here


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.splitlines()[0].split(",")))) if r.returncode == 0 and r.stdout else {}


def events_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def main():
    dev = torch.device("cuda", 0)
    gpu = gpu_info()
    cfg = S.config("laparoscopy512")
    F, W, H, K = cfg["frames"], cfg["W"], cfg["H"], cfg["K"]
    E = cfg["extrinsics"](F)
    intr = PinholeCameraIntrinsic(W, H, *K)
    depth_u16 = torch.empty((F, H, W), dtype=torch.uint16, device=dev)
    for lo in range(0, F, 100):
        depth_u16[lo:lo + 100] = S.render(cfg["surface"], E[lo:lo + 100], K=K, W=W, H=H, device=dev, with_color=False, first_frame=lo)[0]
    out = {"metric": "raycast", "gpu": gpu, "image": f"{W}x{H}", "outputs": "depth + vertex + normal (f32)"}

    # ---- tsdf512
    vol = DenseTSDFVolume(cfg["voxel_length"], cfg["sdf_trunc"], cfg["resolution"], cfg["origin"], color=False, device=dev)
    vol.integrate_u16_chunks(depth_u16, None, intr, E, vol.stream_chunks(F), 1000.0, 3.0)
    poses = E[np.linspace(0, F - 1, 256).astype(int)]
    cast = lambda P: vol.raycast(intr, P, depth_min=0.0, depth_max=3.0, colors=False)      # noqa: E731
    for i in range(0, 256, 64):
        cast(poses[i:i + 64])
    torch.cuda.synchronize()
    ms_batch = events_ms(lambda: [cast(poses[i:i + 64]) for i in range(0, 256, 64)], 5) / 4
    single = []
    for i in range(256):
        t0 = time.perf_counter()
        cast(poses[i])
        torch.cuda.synchronize()
        single.append((time.perf_counter() - t0) * 1e3)
    fps = 64 / (ms_batch / 1e3)
    out["tsdf512"] = {"volume": f"{cfg['resolution']}^3 @ {cfg['voxel_length'] * 1e3:g} mm, {F} frames integrated", "poses": 256,
                      "batched_64": {"ms_per_call": ms_batch, "frames_per_s": fps, "mrays_per_s": fps * W * H / 1e6},
                      "per_frame_sync": {"median_ms": float(np.median(single[8:])), "p90_ms": float(np.percentile(single[8:], 90))}}

    # ---- map_defaults
    vs, res = 0.0058, 256
    bs = vs * 16
    centre = np.asarray(cfg["origin"]) + 0.5 * cfg["resolution"] * cfg["voxel_length"]
    m = MAP(W, H, np.array([[K[0], 0, K[2]], [0, K[1], K[3]], [0, 0, 1]]), "CUDA:0", 1000.0, resolution=res,
            origin=np.floor((centre - 0.5 * res * vs) / bs + 0.5) * bs, color=False)
    P_all = np.linalg.inv(E)
    for i in range(8):
        m.integrate_batch(depth_u16[i], None, P_all[i][None], 3.0)
        m.synthesize_model_frame()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(8, F):
        m.integrate_batch(depth_u16[i], None, P_all[i][None], 3.0)
        m.synthesize_model_frame()
    torch.cuda.synchronize()
    out["map_defaults"] = {"box": f"{res}^3 @ 5.8 mm", "frames": F - 8, "frames_per_s": (F - 8) / (time.perf_counter() - t0)}

    # ---- cpu_baseline + parity (the GPU's own grids)
    ids = np.linspace(0, 255, 8).astype(int)
    t, w = (x.cpu().numpy() for x in vol.export_dense())
    V = oracle.o3d.Volume(cfg["resolution"], cfg["voxel_length"], cfg["sdf_trunc"], cfg["origin"])
    V.tsdf, V.weight = t.reshape(-1), w.reshape(-1)
    del t, w
    t0 = time.perf_counter()
    ref = raycast_ref.raycast(V, K, poses[ids], W, H, colors=False)
    cpu_s = time.perf_counter() - t0
    g = {k: v.cpu().numpy() for k, v in cast(poses[ids]).items()}
    out["cpu_baseline"] = {"poses": len(ids), "threads": oracle.o3d.num_threads(), "s": cpu_s, "frames_per_s": len(ids) / cpu_s}
    par = {"hit_equal": bool(np.array_equal(g["depth"] > 0, ref["depth"] > 0)), "depth_equal": bool(np.array_equal(g["depth"], ref["depth"])),
           "hit_fraction": float((ref["depth"] > 0).mean())}
    for k in ("vertex", "normal"):
        par[f"{k}_max_dev"] = float(np.abs(g[k] - ref[k]).max())
    del V
    mt, mw = (x.cpu().numpy() for x in m.model.export_dense())
    MV = oracle.o3d.Volume(res, vs, vs * 8.0, m.model.origin)
    MV.tsdf, MV.weight = mt.reshape(-1), mw.reshape(-1)
    mg = {k: v.cpu().numpy() for k, v in m.synthesize_model_frame().items()}
    mref = raycast_ref.raycast_vbg(MV, K, P_all[F - 1], W, H, m.allocated_blocks().cpu().numpy(), m.allocated_blocks(last_frame=True).cpu().numpy(),
                                   depth_scale=1000.0, weight_threshold=3.0, trunc_voxel_multiplier=8.0, colors=False)
    par["map_hit_equal"] = bool(np.array_equal(mg["depth"] > 0, mref["depth"] > 0))
    par["map_depth_equal"] = bool(np.array_equal(mg["depth"], mref["depth"]))
    par["map_hit_fraction"] = float((mref["depth"] > 0).mean())
    for k in ("vertex", "normal"):
        par[f"map_{k}_max_dev"] = float(np.abs(mg[k] - mref[k]).max())
    out["parity"] = par

    # ---- roofline (batched call)
    bytes_per_frame = 8.0 * ref["samples"] / len(ids) + 28.0 * W * H
    gbs = bytes_per_frame * fps / 1e9
    out["roofline"] = {"samples_per_ray": ref["samples"] / (len(ids) * W * H), "algorithmic_bytes_per_frame": bytes_per_frame,
                       "achieved_gb_per_s": gbs, "hbm_peak_gb_per_s": HBM_PEAK_GBS, "share_of_peak": gbs / HBM_PEAK_GBS,
                       "bound": "latency of the dependent gathers of the march, not bandwidth"}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
