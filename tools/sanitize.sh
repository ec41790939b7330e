#!/bin/bash
# compute-sanitizer over the hot path (run on a GPU box):  bash tools/sanitize.sh > gpurun_out/sanitizer.log
# memcheck + racecheck + synccheck on smoke() (a4, K3 with named barriers / shared flag words / persistent
# claims, K4 marching cubes, K1, K2), on a small sharded-layout / unit-activation / colour integration, on colour
# integrations whose RGB batches end exactly where their allocations do, on unit activation with 8^3 units and two
# mask words per row, and on the image kernels at their edges.
set -u
CS=/usr/local/cuda/bin/compute-sanitizer
PY='
import sys, numpy as np, torch
sys.path.insert(0, "."); sys.path.insert(0, "tests")
import __graft_entry__ as g
g.smoke()
from util import small_scene
from bodyslam_b200 import ops, mdem
from bodyslam_b200.tsdf import DenseTSDFVolume
dev = torch.device("cuda", 0)
sc = small_scene("laparoscopy512", res=64, frames=3, W=320, H=240)
d = ops.depth_from_u16(sc["depth_u16"], 1000.0, 3.0, dev)
col = torch.from_numpy(sc["color"]).to(dev)
ul = sc["voxel_length"] * 32
org = np.floor(sc["origin"] / ul + 0.5) * ul
for kw in (dict(unit_activation=True), dict(gz0=8, z_total=64, z_interleave=2), dict()):
    for zpw in (8, 4, 2):
        res = (64, 64, 32) if "gz0" in kw else 64
        v = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], res, org, color=True, device=dev, **kw)
        v.set_z_split(zpw)
        v.integrate_batch(d, col, sc["intrinsic"], sc["E"])
        if "gz0" not in kw:
            v.extract_triangle_mesh(); v.extract_point_cloud()
# unit activation with 8^3 units and two mask words per (ux, uy) row (nuz = 64), stride 3
v = DenseTSDFVolume(sc["voxel_length"], sc["sdf_trunc"], (64, 64, 512), org, color=False, device=dev, unit_activation=True,
                    unit_resolution=8, depth_sampling_stride=3)
v.integrate_batch(d, None, sc["intrinsic"], sc["E"])
mdem.colorize(np.random.default_rng(0).uniform(0.1, 3, (120, 160)).astype(np.float32), cmap="viridis", invalid_val=0)
# image kernels at their edges: a K1 batch of 65 images of 45 x 101 px (H*W = 1 mod 4: every image after the first
# off a 16-byte boundary), a K2 call of 130 frames (three emit chunks of poses) and a K1f image holding NaN pixels
rng = np.random.default_rng(1)
ops.colorize_u16(mdem.get_cmap_lut("viridis"), depth_u16=rng.integers(0, 65536, (65, 45, 101)).astype(np.uint16), invalid_val=0)
bpd = rng.uniform(0.05, 3.0, (130, 30, 40)).astype(np.float32)
bpd[rng.uniform(size=bpd.shape) < 0.1] = 0
ops.backproject(bpd, (37.5, 36.0, 19.3, 15.1), np.eye(4)[None].repeat(130, 0), color=rng.integers(0, 256, (130, 30, 40, 3)).astype(np.uint8))
fnan = rng.uniform(0.2, 4.0, (37, 23)).astype(np.float32)
fnan.reshape(-1)[::7] = np.nan
ops.colorize_f32(mdem.get_cmap_lut("viridis"), fnan, invalid_val=0.0)
# colour gathers at the end of the RGB batch (PYTORCH_NO_CUDA_MEMORY_CACHING=1 below: every tensor is its own exactly sized
# cudaMalloc): the 512 x 512 x 144 laparoscopy slab (8 z layers per warp, no long-chain phase), then 3 frames of 333 x 201
# px, whose RGB batch (200 799 pixels) ends 3 bytes short of a 4-byte word
sl = small_scene("laparoscopy512", res=512, frames=2)
v = DenseTSDFVolume(sl["voxel_length"], sl["sdf_trunc"], (512, 512, 144), sl["origin"], color=True, device=dev, gz0=368, z_total=512)
v.integrate_batch(ops.depth_from_u16(sl["depth_u16"], 1000.0, 3.0, dev), torch.from_numpy(sl["color"]).to(dev), sl["intrinsic"], sl["E"])
od = small_scene("laparoscopy512", res=64, frames=3, W=333, H=201)
v = DenseTSDFVolume(od["voxel_length"], od["sdf_trunc"], 64, od["origin"], color=True, device=dev)
v.integrate_batch(ops.depth_from_u16(od["depth_u16"], 1000.0, 3.0, dev), torch.from_numpy(od["color"]).to(dev), od["intrinsic"], od["E"])
torch.cuda.synchronize()
print("SANITIZE_WORKLOAD_OK")
'
for tool in memcheck racecheck synccheck; do
  echo "=== compute-sanitizer --tool $tool"
  PYTORCH_NO_CUDA_MEMORY_CACHING=1 timeout 900 $CS --tool $tool --print-limit 20 python -c "$PY" 2>&1 | grep -E "SANITIZE_WORKLOAD_OK|smoke ok|ERROR SUMMARY|RACECHECK SUMMARY|Race reported|Invalid|hazard|error" | head -40
done
