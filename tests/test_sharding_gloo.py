"""Host-side logic of the z-slab sharding over a world_size-2/3 `gloo` group (CPU tensors):
slab bounds, halo exchange, frame broadcast, variable-size mesh gather and cross-slab merge."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
from bodyslam_b200.geometry import TriangleMesh
from bodyslam_b200.sharding import (broadcast_frames, exchange_halo_color, exchange_halo_planes, gather_meshes, merge_slab_meshes, reshard_layers,
                                    reshard_plan, slab_bounds)
from util import canon_mesh


def test_slab_bounds():
    assert slab_bounds(512, 1) == [(0, 512)]
    assert slab_bounds(512, 8) == [(64 * r, 64 * (r + 1)) for r in range(8)]
    assert slab_bounds(1024, 8)[3] == (384, 512)
    b = slab_bounds(60, 3)                         # 8 bricks over 3 ranks: 3 + 3 + 2, last one ragged
    assert b == [(0, 24), (24, 48), (48, 60)]
    assert all(z0 % 8 == 0 for z0, _ in b)
    with pytest.raises(ValueError):
        slab_bounds(16, 3)


def test_reshard_plan_is_a_permutation():
    for world in (2, 4, 8):
        n = 64
        L = n // world
        plans = [reshard_plan(n, world, r) for r in range(world)]
        for q in range(world):
            got = []
            for p in range(world):
                send_pq = plans[p][0][q]                  # local interleaved indices rank p sends to q
                recv_qp = plans[q][1][p]                  # where rank q stores them
                assert len(send_pq) == len(recv_qp)
                for l, dst in zip(send_pq, recv_qp):
                    assert l * world + p == q * L + dst   # same global layer on both sides
                got += recv_qp
            assert sorted(got) == list(range(L))
    with pytest.raises(ValueError):
        reshard_plan(10, 4, 0)


def field(n=40, seed=5):
    g = (np.arange(n) + 0.5) / n - 0.5
    x, y, z = np.meshgrid(g, g, g, indexing="ij")
    rng = np.random.default_rng(seed)
    t = np.sqrt(x * x + y * y + z * z) - 0.3
    for _ in range(8):
        k = rng.normal(size=3) * 14
        t += 0.04 * rng.normal() * np.sin(k[0] * x + k[1] * y + k[2] * z)
    V = oracle.o3d.Volume(n, 0.01, 0.04, origin=(0.0, 0.1, 0.2))
    V.tsdf[:] = np.clip(t * 8, -1, 1).astype(np.float32).reshape(-1)
    V.weight[:] = 1
    return V


def split_into_slab_meshes(full, bounds, ny):
    """what each rank's bslam_mc_emit would produce: local vertex ids, local-z keys, and
    -(1 + (x*ny + y)*4 + axis) for references into the next slab's first plane"""
    keys, tz = full["keys"], full["triangle_z"]
    parts = []
    for (z0, z1) in bounds:
        own_v = np.nonzero((keys[:, 2] >= z0) & (keys[:, 2] < z1))[0]
        local = -np.ones(len(keys), np.int64)
        local[own_v] = np.arange(len(own_v))
        tri = full["triangles"][(tz >= z0) & (tz < z1)].astype(np.int64)
        out = local[tri]
        up = out < 0
        k = keys[tri[up]]
        assert np.all(k[:, 2] == z1)               # only the next slab's plane 0 can be referenced
        out[up] = -(1 + (k[:, 0].astype(np.int64) * ny + k[:, 1]) * 4 + k[:, 3])
        kk = keys[own_v].copy()
        kk[:, 2] -= z0
        parts.append(TriangleMesh(torch.from_numpy(full["vertices"][own_v].astype(np.float32)), torch.from_numpy(out.astype(np.int32)),
                                  None, torch.from_numpy(kk.astype(np.int32))))
    return parts


def test_merge_slab_meshes_single_process():
    V = field()
    full = V.extract_mesh()
    bounds = slab_bounds(40, 3)
    parts = split_into_slab_meshes(full, bounds, 40)
    assert any((p.triangles < 0).any() for p in parts[:-1])
    merged = merge_slab_meshes(parts, [b[0] for b in bounds], ny=40)
    a = canon_mesh(merged.vertices.numpy(), merged.vertex_keys.numpy(), merged.triangles.numpy(), (40,) * 3)
    b = canon_mesh(full["vertices"], full["keys"], full["triangles"], (40,) * 3)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2]) and np.abs(a[1] - b[1]).max() < 1e-6


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        V = field()
        full = V.extract_mesh()
        bounds = slab_bounds(40, world)
        mine = split_into_slab_meshes(full, bounds, 40)[rank]
        # halo exchange: every rank sends its top / bottom plane to its neighbours
        z0, z1 = bounds[rank]
        tw = np.stack([V.grid("tsdf"), V.grid("weight")], -1)
        top = torch.from_numpy(tw[:, :, z1 - 1].copy())
        bottom = torch.from_numpy(tw[:, :, z0].copy())
        lo, hi = exchange_halo_planes(top, bottom, rank, world)
        assert (lo is None) == (rank == 0) and (hi is None) == (rank == world - 1)
        if lo is not None:
            assert np.array_equal(lo.numpy(), tw[:, :, z0 - 1])
        if hi is not None:
            assert np.array_equal(hi.numpy(), tw[:, :, z1])
        # colour of the bottom plane goes to rank - 1 only (its top-plane z-edges interpolate towards it)
        rgb = np.random.default_rng(9).uniform(0, 255, size=(40, 40, 40, 3)).astype(np.float32)
        hi_col = exchange_halo_color(torch.from_numpy(rgb[:, :, z0].copy()), rank, world)
        assert (hi_col is None) == (rank == world - 1)
        if hi_col is not None:
            assert np.array_equal(hi_col.numpy(), rgb[:, :, z1])
        # frame broadcast from rank 0
        depth = torch.full((2, 4, 5), float(rank))
        color = torch.full((2, 4, 5, 3), rank, dtype=torch.uint8)
        E = torch.eye(4, dtype=torch.float64).repeat(2, 1, 1) * (rank + 1)
        broadcast_frames(depth, color, E, src=0)
        assert float(depth.max()) == 0.0 and int(color.max()) == 0 and float(E[0, 0, 0]) == 1.0
        # round-robin -> contiguous re-shard of (fake) brick layers: layer g is filled with the value g
        if 12 % world == 0:
            Lh = 12 // world
            src = torch.stack([torch.full((5,), l * world + rank, dtype=torch.uint8) for l in range(Lh)])
            dst = torch.zeros((Lh, 5), dtype=torch.uint8)
            send, recv = reshard_plan(12, world, rank)
            reshard_layers(src, dst, send, recv)
            assert dst[:, 0].tolist() == list(range(rank * Lh, (rank + 1) * Lh))
        # mesh gather + merge on rank 0
        parts = gather_meshes(mine, rank, world, dst=0)
        if rank == 0:
            merged = merge_slab_meshes(parts, [b[0] for b in bounds], ny=40)
            a = canon_mesh(merged.vertices.numpy(), merged.vertex_keys.numpy(), merged.triangles.numpy(), (40,) * 3)
            b = canon_mesh(full["vertices"], full["keys"], full["triangles"], (40,) * 3)
            ok = np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2]) and np.abs(a[1] - b[1]).max() < 1e-6
            ret.put(("ok" if ok else "mesh mismatch", len(full["triangles"])))
        else:
            assert parts is None
    except Exception as e:  # surface the failure in the parent
        ret.put((f"rank {rank}: {type(e).__name__}: {e}", 0))
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gather_and_merge_over_gloo(world):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    msg, ntri = ret.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
    assert msg == "ok", msg
    assert ntri > 3000 and all(p.exitcode == 0 for p in procs)
