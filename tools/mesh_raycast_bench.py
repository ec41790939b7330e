"""Mesh ray-cast measurement: one JSON line.

mesh          BASELINE configs[3] (laparoscopy512, 1000 frames) integrated in full; its marching-cubes mesh
              (`extract_triangle_mesh`, about 1 M triangles) is the scene.
build         BVH build (`RaycastingScene` commit: index check with its one synchronise, Morton keys, sort, hierarchy,
              boxes), CUDA events, median of 5 after a warm-up.
batched_64    cast_pinhole at 640 x 480 from 64 trajectory poses per call, depth + ids (no uvs / normals), 256 poses in
              all: rays/s from CUDA events.
per_pose_sync one pose per call followed by a synchronise (host clock), median and p90 ms.
traffic       inner nodes (64 B) and leaf triangles (48 B) the traversal reads per ray, counted by replaying it over a host
              copy of the BVH with the reference's rules (tests/mesh_raycast_ref.c) on 8 poses; the replay's hits must
              equal the GPU's.
cpu_baseline  the brute-force CPU reference (all host threads) on a seeded subset of 2 000 rays of one pose, rays/s;
              its outputs must equal the GPU's bit for bit.
digest        sha256 of the 256 poses' t_hit, geometry and primitive ids.
Run from the repository root: python tools/mesh_raycast_bench.py
"""
import hashlib
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

import mesh_raycast_ref as R  # noqa: E402
from bodyslam_b200 import synthetic as S  # noqa: E402
from bodyslam_b200.geometry import PinholeCameraIntrinsic  # noqa: E402
from bodyslam_b200.raycasting import RaycastingScene  # noqa: E402
from bodyslam_b200.tsdf import DenseTSDFVolume  # noqa: E402


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
    if not torch.cuda.is_available():
        raise SystemExit("mesh_raycast_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    out = {"metric": "mesh_raycast", "gpu": gpu_info()}
    cfg = S.config("laparoscopy512")
    F, W, H, K = cfg["frames"], cfg["W"], cfg["H"], cfg["K"]
    E = cfg["extrinsics"](F)
    intr = PinholeCameraIntrinsic(W, H, *K)
    depth_u16 = torch.empty((F, H, W), dtype=torch.uint16, device=dev)
    for lo in range(0, F, 100):
        depth_u16[lo:lo + 100] = S.render(cfg["surface"], E[lo:lo + 100], K=K, W=W, H=H, device=dev, with_color=False, first_frame=lo)[0]
    vol = DenseTSDFVolume(cfg["voxel_length"], cfg["sdf_trunc"], cfg["resolution"], cfg["origin"], color=False, device=dev)
    vol.integrate_u16_chunks(depth_u16, None, intr, E, vol.stream_chunks(F), 1000.0, 3.0)
    del depth_u16
    mesh = vol.extract_triangle_mesh()
    del vol
    n_tris = int(mesh.triangles.shape[0])
    out["mesh"] = {"source": f"laparoscopy512 {cfg['resolution']}^3, {F} frames, extract_triangle_mesh", "triangles": n_tris,
                   "vertices": int(mesh.vertices.shape[0])}

    # ---- build
    times = []
    for i in range(6):
        sc = RaycastingScene(dev)
        sc.add_triangles(mesh)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        bvh = sc._commit()
        b.record()
        b.synchronize()
        if i:
            times.append(a.elapsed_time(b))
    out["build"] = {"median_ms": float(np.median(times)), "bvh_bytes": int(bvh.numel())}

    # ---- cast
    poses = E[np.linspace(0, F - 1, 256).astype(int)]
    cast = lambda P: sc.cast_pinhole(intr, P, uvs=False, normals=False)     # noqa: E731
    for i in range(0, 256, 64):
        cast(poses[i:i + 64])
    torch.cuda.synchronize()
    ms = events_ms(lambda: [cast(poses[i:i + 64]) for i in range(0, 256, 64)], 5) / 4
    out["batched_64"] = {"ms_per_call": ms, "frames_per_s": 64e3 / ms, "mrays_per_s": 64 * W * H / ms / 1e3, "outputs": "t_hit + ids"}
    single = []
    for i in range(256):
        t0 = time.perf_counter()
        cast(poses[i])
        torch.cuda.synchronize()
        single.append((time.perf_counter() - t0) * 1e3)
    out["per_pose_sync"] = {"median_ms": float(np.median(single[8:])), "p90_ms": float(np.percentile(single[8:], 90))}
    res = [cast(poses[i:i + 64]) for i in range(0, 256, 64)]
    h = hashlib.sha256()
    for k in ("t_hit", "geometry_ids", "primitive_ids"):
        for r in res:
            h.update(r[k].contiguous().view(torch.int32).cpu().numpy().tobytes())
    out["digest"] = h.hexdigest()
    hit = float(torch.cat([torch.isfinite(r["t_hit"]).flatten() for r in res]).float().mean())

    # ---- traffic (replay of the traversal over the BVH) and its hits against the GPU's
    ids = np.linspace(0, 255, 8).astype(int)
    host_bvh = bvh.cpu().numpy()
    nodes = tris = 0
    replay_equal = True
    for i in ids:
        rays = R.rays_pinhole(intr.intrinsic_matrix, poses[i], W, H).reshape(-1, 6)
        rep, nn, nt = R.traverse(host_bvh, rays)
        nodes, tris = nodes + nn, tris + nt
        g = cast(poses[i])
        for k in ("t_hit", "geometry_ids", "primitive_ids"):
            replay_equal &= bool(np.array_equal(g[k].contiguous().view(torch.int32).cpu().numpy().reshape(-1), rep[k].view(np.int32)))
    n_rays = len(ids) * W * H
    bytes_per_ray = (64.0 * nodes + 48.0 * tris) / n_rays
    out["traffic"] = {"nodes_per_ray": nodes / n_rays, "triangles_per_ray": tris / n_rays, "bytes_per_ray": bytes_per_ray,
                      "algorithmic_gb_per_s_batched": bytes_per_ray * 64 * W * H / ms / 1e6, "hit_fraction": hit,
                      "replay_equals_gpu": replay_equal,
                      "bound": "latency of the dependent node gathers; the BVH is close to the 126 MB L2"}

    # ---- CPU brute force on a subset
    idx = np.random.default_rng(0).choice(W * H, 2000, replace=False)
    rays = R.rays_pinhole(intr.intrinsic_matrix, poses[0], W, H).reshape(-1, 6)[idx]
    verts, tris_np = mesh.vertices.cpu().numpy(), mesh.triangles.cpu().numpy()
    t0 = time.perf_counter()
    ref = R.cast_rays([(verts, tris_np)], rays)
    cpu_s = time.perf_counter() - t0
    g = cast(poses[0])
    equal = all(np.array_equal(g[k].contiguous().view(torch.int32).cpu().numpy().reshape(-1)[idx], ref[k].view(np.int32))
                for k in ("t_hit", "geometry_ids", "primitive_ids"))
    out["cpu_baseline"] = {"rays": len(idx), "threads": os.cpu_count(), "s": cpu_s, "rays_per_s": len(idx) / cpu_s, "equal_to_gpu": equal}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
