"""z-slab sharding of the TSDF volume over the GPUs of one box (one process per GPU).

The reference has no multi-device code at all (SURVEY.md 2); this is the one parallel axis the
hot path offers: every voxel depends only on (its coordinates, the frame, the pose), so the grid
is cut into contiguous z-slabs, each rank integrates every frame into its own slab with NO
data-path collective, and only surface extraction exchanges data:
  * one halo plane each way between neighbouring slabs (send/recv), so cubes straddling a slab
    boundary are emitted exactly once (by the lower slab) and their shared vertices exactly once
    (by the slab owning the edge);
  * a gather of the per-slab meshes to rank 0, where vertex ids are rebased and the references
    into the next slab's first plane are resolved -- the result equals the single-GPU mesh after
    canonical ordering.
The ray cast (`ShardedTSDF.raycast`) marches every ray through the slabs in rounds: only the ray states
(an all-reduce per round), one packed halo each way and the shaded maps (a reduce to one rank) cross NVLink.
Frames reach the ranks either from each rank's own copy (synthetic / shared storage) or by a
broadcast from rank 0 (`broadcast_frames`), which is the only NCCL traffic during integration.
"""
from __future__ import annotations

import numpy as np

from .geometry import TriangleMesh

BRICK = 8


def slab_bounds(nz: int, world_size: int):
    """contiguous [z0, z1) per rank; every boundary is a multiple of the brick edge (8)."""
    nb = (nz + BRICK - 1) // BRICK
    if world_size > nb:
        raise ValueError(f"cannot cut {nz} planes into {world_size} slabs of whole bricks")
    base, extra = divmod(nb, world_size)
    out, b = [], 0
    for r in range(world_size):
        n = base + (1 if r < extra else 0)
        out.append((b * BRICK, min((b + n) * BRICK, nz)))
        b += n
    return out


def merge_slab_meshes(meshes, z_offsets, ny: int) -> TriangleMesh:
    """Concatenate per-slab meshes (ordered bottom to top) into one mesh.

    Vertex ids are rebased by the running vertex count; a negative id -(1 + (x*ny + y)*4 + axis)
    refers to the vertex on edge (x, y, z=0, axis) of the NEXT slab and is resolved through that
    slab's vertex keys.  Keys are returned with global z.  Works on torch tensors (any device); all
    slabs are handled by one set of tensor operations (one sort + one binary search for the
    cross-slab references, one host synchronisation for the consistency check).
    """
    import torch

    n = len(meshes)
    dev = meshes[0].vertices.device
    nv = torch.tensor([int(m.vertices.shape[0]) for m in meshes], dtype=torch.int64)
    nt = torch.tensor([int(m.triangles.shape[0]) for m in meshes], dtype=torch.int64)
    base = torch.cumsum(nv, 0) - nv                                          # first global id of every slab
    verts = torch.cat([m.vertices for m in meshes])
    keys = torch.cat([m.vertex_keys for m in meshes]).clone()
    slab_of_v = torch.repeat_interleave(torch.arange(n), nv).to(dev)
    local_z0 = keys[:, 2] == 0
    keys[:, 2] += torch.as_tensor(np.asarray(z_offsets, dtype=np.int64), device=dev)[slab_of_v].to(keys.dtype)
    has_col = all(m.vertex_colors is not None for m in meshes) and n > 0
    cols = torch.cat([m.vertex_colors for m in meshes]) if has_col else None
    tris = torch.cat([m.triangles for m in meshes]).to(torch.int64)
    slab_of_t = torch.repeat_interleave(torch.arange(n), nt).to(dev)
    base_d = base.to(dev)
    neg = tris < 0
    out = tris + base_d[slab_of_t][:, None]
    if int(nt.sum()) and int(nv.sum()):
        # lookup table of the vertices on every slab's plane 0: (slab, edge code) -> global id
        k64 = keys.to(torch.int64)
        M = 4 * (int(ny) + 1) * (int(k64[:, 0].max().item()) + 2)              # > any edge code
        p0 = torch.nonzero(local_z0).reshape(-1)
        code = slab_of_v[p0] * M + (k64[p0, 0] * ny + k64[p0, 1]) * 4 + k64[p0, 3]
        code_sorted, order = torch.sort(code)
        want = (slab_of_t[:, None].expand(-1, 3)[neg] + 1) * M + (-tris[neg] - 1)
        if want.numel():
            if code_sorted.numel() == 0:
                raise RuntimeError("merge_slab_meshes: unresolved cross-slab vertex reference")
            pos = torch.searchsorted(code_sorted, want).clamp_max(code_sorted.numel() - 1)
            if not bool((code_sorted[pos] == want).all()):
                raise RuntimeError("merge_slab_meshes: unresolved cross-slab vertex reference (or the top slab references a slab above it)")
            out[neg] = p0[order[pos]]
    return TriangleMesh(verts, out.to(torch.int32), cols, keys)


def broadcast_frames(depth, color, extrinsics, src: int = 0, group=None):
    """Broadcast one batch of frames from `src` to every rank (NCCL over NVLink on the GPU box).

    depth/color are pre-allocated tensors of identical shape on every rank; extrinsics a float64
    tensor [F,4,4] on the same device.  Returns the tensors (filled in place)."""
    import torch.distributed as dist

    import torch

    if depth.dtype == torch.uint16:  # NCCL has no 16-bit integer type: ship the bytes
        works = [dist.broadcast(depth.view(torch.uint8), src, group=group, async_op=True)]
    else:
        works = [dist.broadcast(depth, src, group=group, async_op=True)]
    if color is not None:
        works.append(dist.broadcast(color, src, group=group, async_op=True))
    works.append(dist.broadcast(extrinsics, src, group=group, async_op=True))
    for w in works:
        w.wait()
    return depth, color, extrinsics


def exchange_halo_planes(top_plane, bottom_plane, rank: int, world_size: int, group=None):
    """neighbour exchange: returns (halo_lo, halo_hi) = (top plane of rank-1, bottom plane of rank+1).  The "planes" are
    any per-slab tensors of one shape per side, such as the packed halos of `DenseTSDFVolume.raycast_halo`."""
    import torch
    import torch.distributed as dist

    halo_lo = torch.empty_like(top_plane) if rank > 0 else None
    halo_hi = torch.empty_like(bottom_plane) if rank + 1 < world_size else None
    ops_ = []
    if rank + 1 < world_size:
        ops_.append(dist.P2POp(dist.isend, top_plane, rank + 1, group))
        ops_.append(dist.P2POp(dist.irecv, halo_hi, rank + 1, group))
    if rank > 0:
        ops_.append(dist.P2POp(dist.isend, bottom_plane, rank - 1, group))
        ops_.append(dist.P2POp(dist.irecv, halo_lo, rank - 1, group))
    if ops_:
        for w in dist.batch_isend_irecv(ops_):
            w.wait()
    return halo_lo, halo_hi


def exchange_halo_color(bottom_color, rank: int, world_size: int, group=None):
    """colour half of the halo exchange: every rank sends the colour of its bottom plane to rank-1 and returns
    halo_hi_color = the colour of rank+1's bottom plane (None on the last rank).  Only the slab below needs it:
    a vertex on a z-edge from its top plane interpolates towards that plane's colour."""
    import torch
    import torch.distributed as dist

    halo_hi_color = torch.empty_like(bottom_color) if rank + 1 < world_size else None
    ops_ = []
    if rank + 1 < world_size:
        ops_.append(dist.P2POp(dist.irecv, halo_hi_color, rank + 1, group))
    if rank > 0:
        ops_.append(dist.P2POp(dist.isend, bottom_color, rank - 1, group))
    if ops_:
        for w in dist.batch_isend_irecv(ops_):
            w.wait()
    return halo_hi_color


def _pack_mesh(mesh: TriangleMesh):
    """vertices f32 [V,3] | keys i32 [V,4] | triangles i32 [T,3] | colours f32 [V,3] as ONE int32 buffer"""
    import torch

    parts = [mesh.vertices.contiguous().view(torch.int32).reshape(-1), mesh.vertex_keys.contiguous().to(torch.int32).reshape(-1),
             mesh.triangles.contiguous().to(torch.int32).reshape(-1)]
    if mesh.vertex_colors is not None:
        parts.append(mesh.vertex_colors.contiguous().view(torch.int32).reshape(-1))
    return torch.cat(parts) if sum(p.numel() for p in parts) else torch.empty(0, dtype=torch.int32, device=mesh.vertices.device)


def _unpack_mesh(buf, V: int, T: int, has_col: bool) -> TriangleMesh:
    import torch

    o = 0
    verts = buf[o:o + 3 * V].view(torch.float32).view(V, 3); o += 3 * V
    keys = buf[o:o + 4 * V].view(V, 4); o += 4 * V
    tris = buf[o:o + 3 * T].view(T, 3); o += 3 * T
    cols = buf[o:o + 3 * V].view(torch.float32).view(V, 3) if has_col else None
    return TriangleMesh(verts, tris, cols, keys)


def gather_meshes(mesh: TriangleMesh, rank: int, world_size: int, dst: int = 0, group=None):
    """variable-size gather of per-rank meshes to `dst` -> list of TriangleMesh (None elsewhere).
    One size exchange (all-gather of 3 integers) and ONE packed message per rank."""
    import torch
    import torch.distributed as dist

    dev = mesh.vertices.device
    has_col = mesh.vertex_colors is not None
    mine = torch.tensor([mesh.vertices.shape[0], mesh.triangles.shape[0], int(has_col)], dtype=torch.int64, device=dev)
    sizes = torch.empty(world_size * 3, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(sizes, mine, group=group)
    sizes = sizes.view(world_size, 3).tolist()
    words = lambda V, T, c: 7 * V + 3 * T + (3 * V if c else 0)
    if rank != dst:
        buf = _pack_mesh(mesh)
        if buf.numel():    # batched like the receiving side: un-batched NCCL send / recv use a separate pair communicator
            for w in dist.batch_isend_irecv([dist.P2POp(dist.isend, buf, dst, group)]):
                w.wait()
        return None
    out, ops_, bufs = [], [], {}
    for r in range(world_size):
        V, T, c = sizes[r]
        if r != dst and words(V, T, c):
            bufs[r] = torch.empty(words(V, T, c), dtype=torch.int32, device=dev)
            ops_.append(dist.P2POp(dist.irecv, bufs[r], r, group))
    if ops_:
        for w in dist.batch_isend_irecv(ops_):
            w.wait()
    for r in range(world_size):
        V, T, c = sizes[r]
        if r == dst:
            out.append(mesh)
        elif r in bufs:
            out.append(_unpack_mesh(bufs[r], V, T, bool(c)))
        else:
            out.append(TriangleMesh(torch.empty((0, 3), dtype=torch.float32, device=dev), torch.empty((0, 3), dtype=torch.int32, device=dev),
                                    torch.empty((0, 3), dtype=torch.float32, device=dev) if c else None, torch.empty((0, 4), dtype=torch.int32, device=dev)))
    return out


def reshard_plan(n_layers: int, world_size: int, rank: int):
    """Round-robin -> contiguous re-sharding of brick layers.

    Interleaved rank r holds global layers g = l * world_size + r (local index l); contiguous rank
    q holds g in [q * L, (q + 1) * L), L = n_layers / world_size.  Returns (send, recv): send[q] =
    my local interleaved indices that go to rank q (ascending); recv[p] = the local contiguous
    indices at which the layers coming from rank p land (same order as p sends them).
    """
    if n_layers % world_size:
        raise ValueError("interleaved sharding needs a brick-layer count divisible by the world size")
    L = n_layers // world_size
    send = [[l for l in range(L) if q * L <= l * world_size + rank < (q + 1) * L] for q in range(world_size)]
    recv = [[l * world_size + p - rank * L for l in range(L) if rank * L <= l * world_size + p < (rank + 1) * L]
            for p in range(world_size)]
    return send, recv


def reshard_layers(src_layers, dst_layers, send, recv, group=None):
    """all-to-all of whole brick layers: src_layers / dst_layers are [n_local_layers, bytes] uint8
    views (interleaved source, contiguous destination).  The layers a rank sends to rank q are a
    contiguous run of its local layers (ascending q = ascending local index), so the source view IS
    the send buffer of one `all_to_all_single`; the received layers land in a staging buffer ordered
    by source rank and one indexed copy scatters them (skipped when that order already is the slab's)."""
    import torch
    import torch.distributed as dist

    dev = src_layers.device
    n_in = [len(ix) for ix in send]
    n_out = [len(ix) for ix in recv]
    flat_send = [l for ix in send for l in ix]
    if flat_send != list(range(src_layers.shape[0])):
        raise ValueError("reshard_layers: the send plan must cover the local layers in ascending order")
    perm = [l for ix in recv for l in ix]
    direct = perm == list(range(dst_layers.shape[0]))
    out = dst_layers if direct else torch.empty_like(dst_layers)
    dist.all_to_all_single(out, src_layers.contiguous(), output_split_sizes=n_out, input_split_sizes=n_in, group=group)
    if not direct:
        dst_layers.index_copy_(0, torch.as_tensor(perm, dtype=torch.long, device=dev), out)


class ShardedTSDF:
    """One z-shard of a dense TSDF per rank; same surface as `TSDF` for integration, mesh on rank 0.

    layout="interleaved" (default when possible): rank r owns every world_size-th 8-voxel brick
    layer -- every rank sees the same share of any frustum, so integration scales whatever the
    camera looks at.  Extraction first re-shards the brick layers into contiguous slabs (one
    all-to-all over NVLink), then exchanges one halo plane per slab boundary.
    layout="contiguous": plain z-slabs (no re-shard, but the load follows the scene).
    Every rank calls every method (SPMD).  `integrate_batch` is collective-free; pass
    `broadcast_from=0` when only rank 0 holds the frames.
    """

    def __init__(self, voxel_length=0.001, sdf_trunc=0.1, resolution=512, origin=None, color=True, device=None,
                 rank=None, world_size=None, group=None, layout="interleaved", unit_activation=None, unit_arithmetic=False):
        """unit_activation: like `TSDF` -- True = ScalableTSDFVolume semantics (a frame integrates only the 32^3
        units its sampled points activate), False = dense UniformTSDFVolume rule, None (default) = True when the
        whole grid consists of whole units on the world unit grid.  Same default as `TSDF`, so the sharded map
        equals the single-GPU drop-in's."""
        import torch.distributed as dist

        from .tsdf import DenseTSDFVolume

        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world_size = dist.get_world_size(group) if world_size is None else world_size
        if np.isscalar(resolution):
            resolution = (int(resolution),) * 3
        self.nx, self.ny, self.nz = resolution
        self.bounds = slab_bounds(self.nz, self.world_size)
        if origin is None:
            origin = tuple(-0.5 * n * voxel_length for n in resolution)
        if unit_activation is None:
            unit_activation = DenseTSDFVolume.unit_aligned(resolution, voxel_length, origin)
        self.unit_activation = bool(unit_activation)
        # dense rule with the reference's per-unit arithmetic (see DenseTSDFVolume); ignored in unit-activation mode
        self.unit_arithmetic = bool(unit_arithmetic) and not self.unit_activation
        self._args = dict(voxel_length=voxel_length, sdf_trunc=sdf_trunc, origin=origin, color=color, device=device)
        n_layers = self.nz // BRICK
        if self.world_size == 1 or self.nz % BRICK or n_layers % self.world_size:
            layout = "contiguous"
        self.layout = layout
        if layout == "interleaved":
            self.tsdf = DenseTSDFVolume(voxel_length, sdf_trunc, (self.nx, self.ny, self.nz // self.world_size), origin, color=color,
                                        device=device, gz0=BRICK * self.rank, z_total=self.nz, z_interleave=self.world_size,
                                        unit_activation=self.unit_activation, unit_arithmetic=self.unit_arithmetic)
        else:
            z0, z1 = self.bounds[self.rank]
            self.tsdf = DenseTSDFVolume(voxel_length, sdf_trunc, (self.nx, self.ny, z1 - z0), origin, color=color, device=device,
                                        gz0=z0, z_total=self.nz, unit_activation=self.unit_activation, unit_arithmetic=self.unit_arithmetic)

    def integrate_batch(self, depth, color, intrinsic, extrinsics, broadcast_from=None):
        if broadcast_from is not None and self.world_size > 1:
            import torch

            E = torch.as_tensor(np.asarray(extrinsics, dtype=np.float64), device=depth.device).reshape(-1, 4, 4).contiguous()
            broadcast_frames(depth, color, E, broadcast_from, self.group)
            extrinsics = E.cpu().numpy()
        self.tsdf.integrate_batch(depth, color, intrinsic, extrinsics)

    @staticmethod
    def stream_ramp(world_size: int, src_on_device: bool):
        """chunk ramp of a streamed replay: host frames arrive at PCIe speed, so start with 32 frames;
        device-resident frames only have to cross NVLink (one 64-frame chunk hides the first
        broadcast); a single GPU with resident frames has nothing to overlap."""
        if world_size == 1 and src_on_device:
            return ()
        return (64,) if src_on_device else (32, 64, 128)

    def integrate_stream(self, depth_u16, intrinsic, extrinsics, src: int = 0, depth_scale: float = 1000.0, depth_trunc: float = 3.0,
                         chunk: int = 256, update_counts=None):
        """Streamed replay of F uint16 frames held by rank `src` (host memory -- ideally pinned -- or
        device memory) into every rank's shard.  Three stages overlap chunk by chunk:
            rank src: host -> device copy of chunk k+2 (copy stream)
            all     : NCCL broadcast of chunk k+1 over NVLink (NCCL's stream)
            all     : fused depth conversion + integration of chunk k (current stream)
        Every rank calls this with the same shapes; only `src` needs the data (`depth_u16` may be
        None elsewhere if `shape` = (F, H, W) is given through `extrinsics`' length and intrinsic).
        Integration itself has no data-path collective."""
        import torch
        import torch.distributed as dist

        from .geometry import to_numpy

        vol = self.tsdf
        dev = vol.device
        E = np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 4, 4)
        F = E.shape[0]
        on_dev = bool(getattr(depth_u16, "is_cuda", False))
        if self.world_size == 1:
            chunks = vol.stream_chunks(F, chunk, ramp=self.stream_ramp(1, on_dev))
            if on_dev:
                if vol.color:
                    raise RuntimeError("integrate_stream: colour volumes are not streamed yet (use integrate_batch / integrate_host)")
                vol.integrate_u16_chunks(depth_u16, None, intrinsic, E, chunks, depth_scale, depth_trunc, update_counts)
            else:
                vol.integrate_host(depth_u16, None, intrinsic, E, depth_scale, depth_trunc, chunk, update_counts)
            return
        if vol.color:
            raise RuntimeError("integrate_stream: colour volumes are not streamed yet (use integrate_batch)")
        is_src = self.rank == src
        with torch.cuda.device(dev):
            cs = vol.copy_stream()
            with torch.cuda.stream(cs):                           # poses (128 B per frame), off the compute stream
                hdr = torch.cat([torch.as_tensor(E).reshape(-1), torch.tensor([1.0 if on_dev else 0.0], dtype=torch.float64)])
                hdr = hdr.to(dev, non_blocking=True)
                dist.broadcast(hdr, src, group=self.group)
                hdr = hdr.cpu().numpy()                           # the C ABI takes the poses from host memory
            E, src_on_dev = hdr[:-1].reshape(-1, 4, 4), bool(hdr[-1] != 0.0)
            chunks = vol.stream_chunks(F, chunk, ramp=self.stream_ramp(self.world_size, src_on_dev))
            dev_src = is_src and depth_u16.is_cuda                # frames already in this rank's HBM: broadcast them in place
            if dev_src:
                cs.wait_stream(torch.cuda.current_stream(dev))    # whoever produced them did so on the current stream

            def arrive(k, stage, free):
                f0, f1 = chunks[k]
                with torch.cuda.stream(cs):
                    if dev_src:
                        u16 = depth_u16[f0:f1]
                    else:
                        u16 = stage[0][:f1 - f0]
                        cs.wait_event(free)
                        if is_src:
                            u16.copy_(depth_u16[f0:f1], non_blocking=True)
                    # the collective is enqueued behind the copy stream's work (NCCL waits for the
                    # stream that is current at the call); NCCL has no 16-bit integer type: ship bytes
                    work = dist.broadcast(u16.view(torch.uint8), src, group=self.group, async_op=True)
                return u16, None, work.wait

            vol.integrate_streamed(chunks, intrinsic, E, arrive, depth_scale, depth_trunc, update_counts)

    # ------------------------------------------------------------------ sharded ingest
    @staticmethod
    def ingest_pieces(F: int, world_size: int, chunk: int = 256):
        """Frame ownership of `integrate_stream_sharded`: per chunk (f0, f1) the list of per-rank
        frame ranges [(a_0, b_0), ..., (a_{N-1}, b_{N-1})] (contiguous, in rank order, covering the
        chunk).  -> (chunks, pieces)."""
        from .tsdf import DenseTSDFVolume

        chunks = DenseTSDFVolume.stream_chunks(F, chunk - chunk % world_size if chunk >= world_size else chunk,
                                               ramp=ShardedTSDF.stream_ramp(world_size, False), multiple_of=world_size)
        pieces = [[(f0 + (f1 - f0) * r // world_size, f0 + (f1 - f0) * (r + 1) // world_size) for r in range(world_size)]
                  for f0, f1 in chunks]
        return chunks, pieces

    @staticmethod
    def ingest_share(F: int, rank: int, world_size: int, chunk: int = 256):
        """indices of the frames rank `rank` feeds (ascending) -- what its host buffer must hold, in this order"""
        _, pieces = ShardedTSDF.ingest_pieces(F, world_size, chunk)
        return np.concatenate([np.arange(a, b) for pc in pieces for (a, b) in [pc[rank]]]) if F else np.zeros(0, np.int64)

    def integrate_stream_sharded(self, depth_u16_share, intrinsic, extrinsics, depth_scale: float = 1000.0, depth_trunc: float = 3.0,
                                 chunk: int = 256, update_counts=None):
        """Streamed replay with SHARDED INGEST: every rank feeds 1/N of each chunk from its own host
        (or device) memory over its own PCIe link -- `depth_u16_share` holds the frames
        `ingest_share(F, rank, N, chunk)` in that order -- and the pieces are exchanged over NVLink
        (NCCL all-gather, or one broadcast per piece when a chunk does not divide evenly), so that
        no single host link carries the whole stream.  `extrinsics` [F,4,4] is given on every rank.
        Same pipeline as `integrate_stream` (copy stream / NCCL stream / current stream), same result."""
        import torch
        import torch.distributed as dist

        from .geometry import to_numpy

        vol = self.tsdf
        dev = vol.device
        N, rank = self.world_size, self.rank
        E = np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 4, 4)
        F = E.shape[0]
        if N == 1:
            return self.integrate_stream(depth_u16_share, intrinsic, E, 0, depth_scale, depth_trunc, chunk, update_counts)
        if vol.color:
            raise RuntimeError("integrate_stream_sharded: colour volumes are not streamed yet (use integrate_batch)")
        chunks, pieces = self.ingest_pieces(F, N, chunk)
        if depth_u16_share.shape[0] != sum(pc[rank][1] - pc[rank][0] for pc in pieces):
            raise RuntimeError("integrate_stream_sharded: this rank's share does not match ingest_share(F, rank, world_size, chunk)")
        with torch.cuda.device(dev):
            cs = vol.copy_stream()
            if depth_u16_share.is_cuda:
                cs.wait_stream(torch.cuda.current_stream(dev))
            offs = np.concatenate([[0], np.cumsum([pc[rank][1] - pc[rank][0] for pc in pieces])])

            def arrive(k, stage, free):
                f0, f1 = chunks[k]
                u16 = stage[0][:f1 - f0]
                a, b = pieces[k][rank]
                works = []
                with torch.cuda.stream(cs):
                    cs.wait_event(free)
                    if b > a:
                        u16[a - f0:b - f0].copy_(depth_u16_share[offs[k]:offs[k + 1]], non_blocking=True)
                    sizes = {q1 - q0 for q0, q1 in pieces[k]}
                    u8 = u16.view(torch.uint8)                       # NCCL has no 16-bit integer type: ship bytes
                    if len(sizes) == 1:                              # equal pieces: one in-place all-gather
                        works.append(dist.all_gather_into_tensor(u8, u8[a - f0:b - f0], group=self.group, async_op=True))
                    else:
                        for q, (q0, q1) in enumerate(pieces[k]):
                            if q1 > q0:
                                works.append(dist.broadcast(u8[q0 - f0:q1 - f0], q, group=self.group, async_op=True))
                return u16, None, lambda: [w.wait() for w in works]

            vol.integrate_streamed(chunks, intrinsic, E, arrive, depth_scale, depth_trunc, update_counts)

    def build_3D_map(self, rgbd, intrinsic, extrinsic):
        self.tsdf.integrate(rgbd, intrinsic, extrinsic)

    def contiguous_slab(self):
        """this rank's contiguous z-slab as a DenseTSDFVolume (re-sharded copy in interleaved mode)"""
        if self.layout != "interleaved":
            return self.tsdf
        from .tsdf import DenseTSDFVolume

        z0, z1 = self.bounds[self.rank]
        a = self._args
        slab = getattr(self, "_slab", None)
        if slab is None:      # kept across calls: every brick layer (voxels, colour, flags) is overwritten by the re-shard
            slab = self._slab = DenseTSDFVolume(a["voxel_length"], a["sdf_trunc"], (self.nx, self.ny, z1 - z0), a["origin"], color=a["color"],
                                                device=self.tsdf.device, gz0=z0, z_total=self.nz, unit_activation=self.unit_activation,
                                                unit_arithmetic=self.unit_arithmetic)
        send, recv = reshard_plan(self.nz // BRICK, self.world_size, self.rank)
        src, dst = self.tsdf.storage_layers(), slab.storage_layers()
        for k in src:
            reshard_layers(src[k], dst[k], send, recv, self.group)
        return slab

    def raycast(self, intrinsic, extrinsics, depth_min: float = 0.0, depth_max: float = 3.0, depth_scale: float = 1.0,
                weight_threshold: float = 0.0, normals: bool = True, colors=None, dst: int = 0, broadcast_from=None, profile: bool = False):
        """`DenseTSDFVolume.raycast` of the whole grid, bit for bit, without gathering it: rank `dst` gets the dict, the other
        ranks None.  Every rank calls it; with `broadcast_from` only that rank needs the poses.
        The grid is cut into contiguous slabs (re-sharded in interleaved layout).  In each round every rank marches the rays
        it owns until they hit, leave the depth window or reach a sample of another slab, and an int32 all-reduce of the ray
        states hands them on; at most world_size rounds, fewer when a round hands nothing over.  Each hit is shaded by the
        slab holding its trilinear base plane (one halo plane below, two above), and the maps are summed on `dst` as
        int32 bit patterns (every pixel has one writer).  profile=True synchronises between the phases and leaves their
        wall-clock milliseconds and the round count in `self.last_raycast_profile` (measurement aid)."""
        if self.world_size == 1:
            out = self.tsdf.raycast(intrinsic, extrinsics, depth_min, depth_max, depth_scale, weight_threshold, normals, colors)
            return out if self.rank == dst else None
        import time

        import torch
        import torch.distributed as dist

        from .geometry import intrinsic_params, to_numpy

        dev, N, rank, g = self.tsdf.device, self.world_size, self.rank, self.group
        t = [time.perf_counter()]

        def mark():
            if profile:
                torch.cuda.synchronize(dev)
                t.append(time.perf_counter())

        if broadcast_from is not None:
            mine = rank == broadcast_from
            n = torch.tensor([np.asarray(to_numpy(extrinsics)).size // 16 if mine else 0], dtype=torch.int64, device=dev)
            dist.broadcast(n, broadcast_from, group=g)
            E = (torch.as_tensor(np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 4, 4), device=dev) if mine
                 else torch.empty((int(n.item()), 4, 4), dtype=torch.float64, device=dev))
            dist.broadcast(E, broadcast_from, group=g)
            extrinsics = E.cpu().numpy()
        E = np.asarray(to_numpy(extrinsics), dtype=np.float64).reshape(-1, 4, 4)
        W, H = intrinsic_params(intrinsic)[:2]
        F, n_pix = E.shape[0], E.shape[0] * H * W
        colors = self.tsdf.color if colors is None else bool(colors)
        v = self.contiguous_slab()
        mark()
        lo, hi = exchange_halo_planes(v.raycast_halo(True), v.raycast_halo(False), rank, N, g)
        mark()
        slab_z = np.asarray([b[0] for b in self.bounds] + [self.nz], dtype=np.int32)
        state = torch.empty(4 * n_pix + 1, dtype=torch.int32, device=dev)
        rounds = 0
        while F and rounds < N:
            v.raycast_segment(state, slab_z, rounds == 0, intrinsic, E, depth_min, depth_max, weight_threshold)
            dist.all_reduce(state, group=g)
            rounds += 1
            if int(state[-1].item()) == 0:
                break
        else:
            if F:
                raise RuntimeError(f"ShardedTSDF.raycast: rays still marching after {N} rounds")
        mark()
        chans = {"depth": 1, "vertex": 3}
        if normals:
            chans["normal"] = 3
        if colors:
            chans["color"] = 3
        buf = torch.empty(n_pix * sum(chans.values()), dtype=torch.int32, device=dev)
        out, o = {}, 0
        for k, c in chans.items():
            out[k] = buf[o:o + c * n_pix].view(torch.float32).view((F, H, W) + ((3,) if c == 3 else ()))
            o += c * n_pix
        v.raycast_shade(state, slab_z, lo, hi, intrinsic, E, out, depth_scale)
        if buf.numel():
            dist.reduce(buf, dst, op=dist.ReduceOp.SUM, group=g)
        mark()
        if profile:
            names = ("reshard_to_slabs", "halo_exchange", "rounds", "shade_and_composite")
            self.last_raycast_profile = {n: 1e3 * (b - a) for n, a, b in zip(names, t[:-1], t[1:])}
            self.last_raycast_profile["n_rounds"] = rounds
        return out if rank == dst else None

    def extract_mesh(self, profile: bool = False):
        """full mesh on rank 0 (None on the other ranks).  profile=True synchronises between the phases and leaves
        their wall-clock milliseconds in `self.last_extract_profile` (measurement aid)."""
        if self.world_size == 1:
            return self.tsdf.extract_triangle_mesh()
        import time

        import torch

        t = [time.perf_counter()]

        def mark():
            if profile:
                torch.cuda.synchronize(self.tsdf.device)
                t.append(time.perf_counter())

        v = self.contiguous_slab()
        mark()
        lo, hi = exchange_halo_planes(v.export_plane(v.nz - 1), v.export_plane(0), self.rank, self.world_size, self.group)
        hi_col = exchange_halo_color(v.export_plane_color(0), self.rank, self.world_size, self.group) if v.color else None
        mark()
        out = self._gather_slab_meshes(v, lo, hi, hi_col, profile_mark=mark)
        if profile:
            names = ("reshard_to_slabs", "halo_exchange", "marching_cubes_count", "sizes_allgather", "emit_and_gather", "merge")
            self.last_extract_profile = {n: 1e3 * (b - a) for n, a, b in zip(names, t[:-1], t[1:])}
        return out

    def _gather_slab_meshes(self, v, lo, hi, hi_col=None, profile_mark=lambda: None):
        """count per slab -> sizes to everybody -> rank 0 allocates the WHOLE mesh once; every slab's marching cubes
        emit straight into its rows (rank 0) or into a send buffer (others) and the pieces are received in place ->
        two small kernels (bslam_mesh_merge) rebase the vertex ids and resolve the cross-slab references."""
        import ctypes as C

        import torch
        import torch.distributed as dist

        from . import _lib

        dev, N, rank = v.device, self.world_size, self.rank
        V, T = v.mc_count(lo, hi)
        profile_mark()
        sizes = torch.empty(N * 2, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(sizes, torch.tensor([V, T], dtype=torch.int64, device=dev), group=self.group)
        sizes = sizes.view(N, 2).cpu().numpy()
        profile_mark()
        nv, nt = sizes[:, 0].copy(), sizes[:, 1].copy()
        if rank != 0:
            verts = torch.empty((V, 3), dtype=torch.float32, device=dev)
            keys = torch.empty((V, 4), dtype=torch.int32, device=dev)
            cols = torch.empty((V, 3), dtype=torch.float32, device=dev) if v.color else None
            tris = torch.empty((T, 3), dtype=torch.int32, device=dev)
            v.mc_emit(verts, keys, cols, tris, lo, hi, hi_col)
            ops_ = [dist.P2POp(dist.isend, t, 0, self.group) for t in (verts, keys, tris, cols) if t is not None and t.numel()]
            if ops_:
                for w in dist.batch_isend_irecv(ops_):
                    w.wait()
            profile_mark()
            profile_mark()
            return None
        Vt, Tt = int(nv.sum()), int(nt.sum())
        verts = torch.empty((Vt, 3), dtype=torch.float32, device=dev)
        keys = torch.empty((Vt, 4), dtype=torch.int32, device=dev)
        cols = torch.empty((Vt, 3), dtype=torch.float32, device=dev) if v.color else None
        tris = torch.empty((Tt, 3), dtype=torch.int32, device=dev)
        vb = np.concatenate([[0], np.cumsum(nv)])
        tb = np.concatenate([[0], np.cumsum(nt)])
        ops_ = []
        for r in range(1, N):
            for t, b in ((verts, vb), (keys, vb), (tris, tb), (cols, vb)):
                if t is not None and b[r + 1] > b[r]:
                    ops_.append(dist.P2POp(dist.irecv, t[b[r]:b[r + 1]], r, self.group))
        v.mc_emit(verts[:V], keys[:V], None if cols is None else cols[:V], tris[:T], lo, hi, hi_col)
        if ops_:
            for w in dist.batch_isend_irecv(ops_):
                w.wait()
        profile_mark()
        L = _lib.load()
        ws = getattr(self, "_merge_ws", None)
        need = L.bslam_mesh_merge_workspace_bytes(N, self.nx, self.ny)
        if ws is None or ws.numel() < need:
            ws = self._merge_ws = torch.empty(need, dtype=torch.uint8, device=dev)
        zoff = np.ascontiguousarray([b[0] for b in self.bounds], dtype=np.int32)
        unresolved = np.zeros(1, np.int64)
        with torch.cuda.device(dev):
            _lib.check(L.bslam_mesh_merge(N, _lib.ptr(np.ascontiguousarray(nv)), _lib.ptr(np.ascontiguousarray(nt)), _lib.ptr(zoff), self.nx, self.ny,
                                          _lib.ptr(keys), _lib.ptr(tris), _lib.ptr(ws), _lib.ptr(unresolved), _lib.stream_ptr(dev)))
        if int(unresolved[0]):
            raise RuntimeError(f"ShardedTSDF.extract_mesh: {int(unresolved[0])} unresolved cross-slab vertex references")
        profile_mark()
        return TriangleMesh(verts, tris, cols, keys)
