"""Mesh point / ray query measurement and the reconstruction-vs-truth figure: one JSON line.

scenes        recon: BASELINE configs[3] (laparoscopy512, 1000 frames) integrated in full, `extract_triangle_mesh`.
              truth: tests/meshes.icosphere(7) (327 680 triangles) with its unit vertices scaled onto Cavity().axes in
              float64, then float32.  Its vertices lie on the ellipsoid and its faces inside it; chord_bound_m bounds
              the distance between the two (a_max (1 - sqrt(1 - R^2)) over faces of planar circumradius R, plus the
              float32 rounding of the vertices).
accuracy      compute_distance of every recon vertex against truth: median / p95 / p99 / max in metres and voxels.
rates         CUDA events, median of 5 calls after a warm-up, queries/s:
              closest_recon_vertices_vs_truth   compute_closest_points of the recon vertices against truth
              closest_uniform_vs_recon          compute_closest_points of 2^24 seeded uniform points in the 512^3 box
                                                against recon (near and far queries)
              grid_vs_truth                     a 256^3 grid of voxel centres over the box against truth:
                                                compute_signed_distance (the distance kernel, then the
                                                occupancy kernel negating in place) for nsamples 1 and 3, and its
                                                two halves alone (compute_distance, compute_occupancy)
              rays_vs_recon                     count_intersections and test_occlusions (tnear 0, tfar inf) of 64
                                                pinhole poses at 640 x 480 (rays stored beforehand)
traffic       inner nodes (64 B) and leaf triangles (48 B) read per query, counted by a CPU replay of each traversal
              (tests/mesh_query_ref.c) on seeded subsets of 20 000 queries; the replays' results must equal the GPU's.
cpu_baseline  the brute-force reference (all host threads) on seeded 2 000-query subsets, queries/s; its outputs must
              equal the GPU's bit for bit.
sign_check    over the 256^3 grid, the sign of compute_signed_distance against the analytic ellipsoid test at every
              point whose distance to the ellipsoid is provably larger than chord_bound_m (|rho - 1| a_min > bound,
              rho = |p / axes|): disagreements for nsamples 1 and 3.
digest        sha256 of the accuracy distances, the uniform queries' closest points and ids, the grid's signed
              distances (nsamples 3) and the counts and occlusions.
Run from the repository root: python tools/mesh_query_bench.py
"""
import hashlib
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import mesh_query_ref as Q  # noqa: E402
from bodyslam_b200 import _lib  # noqa: E402
from bodyslam_b200 import synthetic as S  # noqa: E402
from bodyslam_b200.raycasting import RaycastingScene  # noqa: E402
from mesh_raycast_bench import gpu_info, reconstruction  # noqa: E402
from meshes import icosphere  # noqa: E402


T0 = time.perf_counter()


def progress(msg, out):
    """stage reached, elapsed seconds and the results so far (stderr)"""
    print(f"mesh_query_bench: {msg} at {time.perf_counter() - T0:.0f} s: {json.dumps(out)}", file=sys.stderr, flush=True)


def median_ms(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def i32(x):
    x = x.contiguous()
    return (x.to(torch.int32) if x.dtype == torch.bool else x.view(torch.int32)).cpu().numpy().reshape(-1)


def truth_mesh(axes):
    """icosphere(7) on the ellipsoid (float64 scale, then float32) and its chord-error bound in metres"""
    v, t = icosphere(7)
    u = v.astype(np.float64)
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    tri = u[t]
    a, b, c = tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0], tri[:, 2] - tri[:, 1]
    la, lb, lc = (np.linalg.norm(x, axis=1) for x in (a, b, c))
    area2 = np.linalg.norm(np.cross(a, b), axis=1)
    Rc = la * lb * lc / (2 * area2)                                   # planar circumradius (vertices on the unit sphere)
    sag = float(np.max(1 - np.sqrt(np.maximum(0.0, 1 - Rc * Rc))))
    verts = (u * np.asarray(axes)).astype(np.float32)
    rounding = float(np.abs(verts.astype(np.float64) - u * np.asarray(axes)).max()) * np.sqrt(3)
    return verts, t, max(axes) * sag + rounding


def pct(x, vl):
    q = {k: float(np.percentile(x, p)) for k, p in (("median", 50), ("p95", 95), ("p99", 99), ("max", 100))}
    return {"m": q, "voxels": {k: v / vl for k, v in q.items()}}


def main():
    if not torch.cuda.is_available():
        raise SystemExit("mesh_query_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    out = {"metric": "mesh_queries", "gpu": gpu_info()}
    mesh, cfg, E, intr = reconstruction(dev)
    vl, n_vox = cfg["voxel_length"], cfg["resolution"]
    lo = np.asarray(cfg["origin"], np.float64)
    hi = lo + n_vox * vl
    axes = S.Cavity().axes
    gv, gt, chord = truth_mesh(axes)
    recon = RaycastingScene(dev)
    recon.add_triangles(mesh)
    truth = RaycastingScene(dev)
    truth.add_triangles(gv, gt)
    rb, tb = recon._commit(), truth._commit()
    out["scenes"] = {"recon": {"source": f"laparoscopy512 {n_vox}^3, {cfg['frames']} frames, extract_triangle_mesh",
                               "triangles": int(mesh.triangles.shape[0]), "vertices": int(mesh.vertices.shape[0]), "bvh_bytes": int(rb.numel())},
                     "truth": {"source": f"icosphere(7) scaled onto Cavity axes {axes}", "triangles": int(len(gt)), "bvh_bytes": int(tb.numel()),
                               "chord_bound_m": chord, "chord_bound_voxels": chord / vl}}
    digest = hashlib.sha256()
    rates = out["rates"] = {}

    progress("scenes built", out)
    # ---- accuracy and closest points of the recon vertices against truth
    rv = mesh.vertices.contiguous()
    dist = truth.compute_distance(rv)
    d = dist.cpu().numpy().astype(np.float64)
    out["accuracy_recon_vertices_vs_truth"] = {"vertices": int(len(d)), **pct(d, vl), "voxel_length_m": vl,
                                               "note": "distance of every reconstruction vertex to the tessellated ellipsoid"}
    digest.update(i32(dist).tobytes())
    ms = median_ms(lambda: truth.compute_closest_points(rv))
    rates["closest_recon_vertices_vs_truth"] = {"queries": int(len(d)), "ms": ms, "mqueries_per_s": len(d) / ms / 1e3}
    ms = median_ms(lambda: truth.compute_distance(rv))
    rates["distance_recon_vertices_vs_truth"] = {"queries": int(len(d)), "ms": ms, "mqueries_per_s": len(d) / ms / 1e3}

    progress("accuracy", out)
    # ---- 2^24 uniform points against recon
    rng = np.random.default_rng(0)
    nu = 1 << 24
    uni = torch.as_tensor(rng.uniform(lo, hi, size=(nu, 3)).astype(np.float32), device=dev)
    ms = median_ms(lambda: recon.compute_closest_points(uni))
    rates["closest_uniform_vs_recon"] = {"queries": nu, "ms": ms, "mqueries_per_s": nu / ms / 1e3}
    cu = recon.compute_closest_points(uni)
    for k in ("points", "geometry_ids", "primitive_ids"):
        digest.update(i32(cu[k]).tobytes())

    progress("uniform queries", out)
    # ---- grid against truth
    ng = 256
    gx, gy, gz = (lo[k] + (np.arange(ng) + 0.5) * (hi[k] - lo[k]) / ng for k in range(3))
    X, Y, Z = np.meshgrid(gx, gy, gz, indexing="ij")
    grid_np = np.stack([X, Y, Z], -1).reshape(-1, 3).astype(np.float32)
    del X, Y, Z
    grid = torch.as_tensor(grid_np, device=dev)
    ngp = len(grid_np)
    sd = {}
    for ns in (1, 3):
        ms = median_ms(lambda: truth.compute_signed_distance(grid, nsamples=ns))
        rates[f"signed_distance_grid_vs_truth_ns{ns}"] = {"queries": ngp, "ms": ms, "mqueries_per_s": ngp / ms / 1e3}
        ms = median_ms(lambda: truth.compute_occupancy(grid, nsamples=ns))
        rates[f"occupancy_grid_vs_truth_ns{ns}"] = {"queries": ngp, "ms": ms, "mqueries_per_s": ngp / ms / 1e3}
        sd[ns] = truth.compute_signed_distance(grid, nsamples=ns).cpu().numpy()
    ms = median_ms(lambda: truth.compute_distance(grid))
    rates["distance_grid_vs_truth"] = {"queries": ngp, "ms": ms, "mqueries_per_s": ngp / ms / 1e3}
    digest.update(sd[3].view(np.int32).tobytes())
    rho = np.linalg.norm(grid_np.astype(np.float64) / np.asarray(axes), axis=1)
    decided = np.abs(rho - 1) * min(axes) > chord
    inside = rho < 1
    out["sign_check"] = {"points_decided": int(decided.sum()), "points_within_bound": int((~decided).sum()),
                         **{f"disagreements_ns{ns}": int(((sd[ns] < 0) != inside)[decided].sum()) for ns in (1, 3)}}

    progress("grid", out)
    # ---- rays of 64 poses against recon
    F, W, H = 64, cfg["W"], cfg["H"]
    poses = np.ascontiguousarray(E[np.linspace(0, cfg["frames"] - 1, F).astype(int)], dtype=np.float64)
    K = np.ascontiguousarray(intr.intrinsic_matrix, dtype=np.float64)
    rays = torch.empty((F, H, W, 6), dtype=torch.float32, device=dev)
    _lib.check(_lib.load().bslam_mesh_rays_pinhole(F, H, W, _lib.ptr(K), _lib.ptr(poses), _lib.ptr(rays), _lib.stream_ptr(dev)))
    nr = F * W * H
    ms = median_ms(lambda: recon.count_intersections(rays))
    rates["count_intersections_64_poses_vs_recon"] = {"queries": nr, "ms": ms, "mqueries_per_s": nr / ms / 1e3}
    ms = median_ms(lambda: recon.test_occlusions(rays))
    rates["test_occlusions_64_poses_vs_recon"] = {"queries": nr, "ms": ms, "mqueries_per_s": nr / ms / 1e3}
    cnt, occl = recon.count_intersections(rays), recon.test_occlusions(rays)
    digest.update(i32(cnt).tobytes())
    digest.update(i32(occl).tobytes())

    progress("rays", out)
    # ---- traffic: replays on seeded subsets, equal to the GPU
    traffic = {}
    rv_np, uni_np, rays_np = rv.cpu().numpy(), uni.cpu().numpy(), rays.reshape(-1, 6).cpu().numpy()
    replay_equal = True
    for name, bvh, sc, pts in (("closest_recon_vertices_vs_truth", tb, truth, rv_np), ("closest_uniform_vs_recon", rb, recon, uni_np),
                               ("distance_grid_vs_truth", tb, truth, grid_np)):
        idx = rng.choice(len(pts), 20_000, replace=False)
        rep, nn, nt = Q.traverse_closest(bvh.cpu().numpy(), pts[idx])
        gq = torch.as_tensor(pts[idx], device=dev)
        gp = sc.compute_closest_points(gq)
        replay_equal &= bool(np.array_equal(i32(sc.compute_distance(gq)), rep["distance"].view(np.int32)))
        for k in ("geometry_ids", "primitive_ids"):
            replay_equal &= bool(np.array_equal(i32(gp[k]), rep[k].view(np.int32)))
        traffic[name] = {"nodes_per_query": nn / len(idx), "triangles_per_query": nt / len(idx), "bytes_per_query": (64.0 * nn + 48.0 * nt) / len(idx)}
    idx = rng.choice(nr, 20_000, replace=False)
    host_rb = rb.cpu().numpy()
    for name, anyhit, gpu in (("count_intersections_64_poses_vs_recon", False, cnt), ("test_occlusions_64_poses_vs_recon", True, occl)):
        rep, nn, nt = Q.traverse_count(host_rb, rays_np[idx], 0.0, np.inf, anyhit)
        replay_equal &= bool(np.array_equal(i32(gpu)[idx], rep))
        traffic[name] = {"nodes_per_query": nn / len(idx), "triangles_per_query": nt / len(idx), "bytes_per_query": (64.0 * nn + 48.0 * nt) / len(idx)}
    traffic["replay_equals_gpu"] = replay_equal
    out["traffic"] = traffic

    progress("traffic", out)
    # ---- CPU brute force on 2 000-query subsets
    base, equal = {}, True
    truth_g, recon_g = [(gv, gt)], [(mesh.vertices.cpu().numpy(), mesh.triangles.cpu().numpy())]
    idx = rng.choice(len(rv_np), 2000, replace=False)
    t0 = time.perf_counter()
    ref = Q.closest_points(truth_g, rv_np[idx])
    base["closest_recon_vertices_vs_truth"] = 2000 / (time.perf_counter() - t0)
    gp = truth.compute_closest_points(torch.as_tensor(rv_np[idx], device=dev))
    equal &= all(np.array_equal(i32(gp[k]), ref[k].reshape(-1).view(np.int32)) for k in gp)
    idx = rng.choice(nu, 2000, replace=False)
    t0 = time.perf_counter()
    ref = Q.closest_points(recon_g, uni_np[idx])
    base["closest_uniform_vs_recon"] = 2000 / (time.perf_counter() - t0)
    gp = recon.compute_closest_points(torch.as_tensor(uni_np[idx], device=dev))
    equal &= all(np.array_equal(i32(gp[k]), ref[k].reshape(-1).view(np.int32)) for k in gp)
    idx = rng.choice(ngp, 2000, replace=False)
    t0 = time.perf_counter()
    _, ref_sd = Q.occupancy(truth_g, grid_np[idx], 3)
    base["signed_distance_grid_vs_truth_ns3"] = 2000 / (time.perf_counter() - t0)
    equal &= bool(np.array_equal(sd[3][idx].view(np.int32), ref_sd.view(np.int32)))
    idx = rng.choice(nr, 2000, replace=False)
    t0 = time.perf_counter()
    ref_c = Q.count_intersections(recon_g, rays_np[idx])
    base["count_intersections_64_poses_vs_recon"] = 2000 / (time.perf_counter() - t0)
    equal &= bool(np.array_equal(i32(cnt)[idx], ref_c)) and bool(np.array_equal(i32(occl)[idx], (ref_c > 0).astype(np.int32)))
    out["cpu_baseline"] = {"queries_per_s": base, "queries": 2000, "threads": os.cpu_count(), "equal_to_gpu": equal}
    out["digest"] = digest.hexdigest()
    out["seconds"] = time.perf_counter() - T0
    print(json.dumps(out))


if __name__ == "__main__":
    main()
