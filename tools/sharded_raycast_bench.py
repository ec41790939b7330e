"""Sharded ray-cast measurement (`ShardedTSDF.raycast`): one JSON line from rank 0.

Run under torchrun from the repository root, one process per GPU:
    torchrun --nproc_per_node N tools/sharded_raycast_bench.py [--frames 200] [--res 512] [--scene laparoscopy512]
The scene's frames are integrated into the sharded volume (interleaved layout), then 640x480 depth + vertex + normal
maps are ray cast at 1 and at 64 poses per call.  Reported per pose: the median wall-clock of a whole call (with a
synchronise), and from a separate profiled call the split into re-shard, halo exchange, rounds (with their count) and
shade + composite.  Rank 0 also ray casts a single-GPU `DenseTSDFVolume` of the same grid (N = 1 reference; at 512^3).
The per-frame loop (integrate one frame, ray cast, track with rgbd_odometry_multi_scale on rank 0) is timed over 20
frames.  The card name and power limit are read in the same run.  Nothing is written to the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bodyslam_b200 import ops  # noqa: E402
from bodyslam_b200 import synthetic as S  # noqa: E402
from bodyslam_b200.geometry import PinholeCameraIntrinsic, RGBDImage  # noqa: E402
from bodyslam_b200.odometry import Method, rgbd_odometry_multi_scale  # noqa: E402
from bodyslam_b200.sharding import ShardedTSDF  # noqa: E402
from bodyslam_b200.tsdf import DenseTSDFVolume  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def median_ms(fn, reps, dev):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(dev)
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scene", default="laparoscopy512")
    ap.add_argument("--res", type=int, default=512)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    cfg = S.config(a.scene)
    scale = cfg["resolution"] / a.res
    E_all = cfg["extrinsics"](cfg["frames"])
    ids = np.linspace(0, cfg["frames"] - 1, a.frames).astype(int)
    E = E_all[ids]
    K = cfg["K"]
    W, H = cfg["W"], cfg["H"]
    intr = PinholeCameraIntrinsic(W, H, *K)
    depth_u16, _ = S.render(cfg["surface"], E, K=K, W=W, H=H, device=dev, seed=0, with_color=False)
    depth = ops.depth_from_u16(depth_u16, 1000.0, 3.0, dev)
    vl, trunc, origin = cfg["voxel_length"] * scale, cfg["sdf_trunc"] * scale, np.asarray(cfg["origin"], np.float64)
    sh = ShardedTSDF(vl, trunc, a.res, origin, color=False, device=dev, rank=rank, world_size=world)
    for f0 in range(0, a.frames, 64):
        sh.integrate_batch(depth[f0:f0 + 64], None, intr, E[f0:f0 + 64])
    out = {"scene": a.scene, "resolution": a.res, "gpus": world, "layout": sh.layout, "W": W, "H": H, "integrated_frames": a.frames}
    for F in (1, 64):
        Ef = E[:F]
        cast = lambda: sh.raycast(intr, Ef, depth_min=0.01, normals=True, colors=False)   # noqa: E731
        cast()
        ms = median_ms(cast, a.reps, dev)
        sh.raycast(intr, Ef, depth_min=0.01, normals=True, colors=False, profile=True)
        prof = dict(getattr(sh, "last_raycast_profile", {}))
        out[f"poses_{F}"] = {"ms_per_call": ms, "ms_per_pose": ms / F,
                             "split_ms_per_pose": {k: v / F for k, v in prof.items() if k != "n_rounds"}, "rounds": prof.get("n_rounds")}
    if rank == 0 and a.res <= 512:
        ref = DenseTSDFVolume(vl, trunc, a.res, origin, color=False, device=dev, unit_activation=sh.unit_activation)
        for f0 in range(0, a.frames, 64):
            ref.integrate_batch(depth[f0:f0 + 64], None, intr, E[f0:f0 + 64])
        for F in (1, 64):
            cast = lambda: ref.raycast(intr, E[:F], depth_min=0.01, normals=True, colors=False)   # noqa: E731
            cast()
            out[f"single_gpu_poses_{F}_ms_per_pose"] = median_ms(cast, a.reps, dev) / F
        del ref
    # per-frame loop: integrate one frame, ray cast its pose, track the next frame on rank 0 against the ray cast
    K3 = np.array([[K[0], 0.0, K[2]], [0.0, K[1], K[3]], [0.0, 0.0, 1.0]])
    n = min(20, a.frames - 1)
    ts = []
    d = depth[:1].clone()
    for i in range(n):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        sh.integrate_batch(d, None, intr, E[i:i + 1], broadcast_from=0)
        m = sh.raycast(intr, E[i], depth_min=0.01, colors=False, broadcast_from=0)
        if m is not None:
            rgbd_odometry_multi_scale(RGBDImage(None, depth[i + 1]), RGBDImage(None, m["depth"][0]), K3, depth_scale=1.0, method=Method.PointToPlane)
        torch.cuda.synchronize(dev)
        ts.append(1e3 * (time.perf_counter() - t0))
    out["loop_integrate_raycast_track_ms_per_frame"] = float(np.median(ts))
    if rank == 0:
        out["gpu"] = gpu_info()
        print(json.dumps(out), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
