// Shared host/device helpers of libbodyslam_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "bodyslam_b200.h"

namespace bslam {

void set_error(const char *fmt, ...);

#define BSLAM_CHECK_ARG(cond, ...)              \
    do {                                        \
        if (!(cond)) {                          \
            ::bslam::set_error(__VA_ARGS__);    \
            return BSLAM_E_ARG;                 \
        }                                       \
    } while (0)

#define BSLAM_CUDA(call)                                                                    \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            ::bslam::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),    \
                               __FILE__, __LINE__);                                         \
            return BSLAM_E_CUDA;                                                            \
        }                                                                                   \
    } while (0)

#define BSLAM_LAUNCH_CHECK() BSLAM_CUDA(cudaGetLastError())

constexpr int kBrick = BSLAM_BRICK;                 // 8
constexpr int kBrickVox = kBrick * kBrick * kBrick; // 512
constexpr int kNumSMsB200 = 148;                    // B200 (compile-time sizing hints only)

// SM count of `device` (cached per device, thread-safe: the cache entries are written once with the
// same value); grids of the persistent kernels are sized from it, not from a constant.
int num_sms(int device);
int current_device_sms();

// Every entry point that touches a volume runs on the volume's device and restores the caller's
// current device on the way out (torch reads it through cudaGetDevice).
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
        if (prev != device) ok = cudaSetDevice(device) == cudaSuccess; else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
};
#define BSLAM_DEVICE_GUARD(dev)                                              \
    ::bslam::DeviceGuard device_guard__(dev);                               \
    if (!device_guard__.ok) {                                               \
        ::bslam::set_error("cudaSetDevice(%d) failed (%s:%d)", (int)(dev), __FILE__, __LINE__); \
        cudaGetLastError();                                                 \
        return BSLAM_E_CUDA;                                                \
    }

// Device view of a brick-ordered volume.  Brick b = (bz*nby + by)*nbx + bx holds 512 float2
// {tsdf, weight}; in-brick index = lz*64 + lx*8 + ly  (a warp owns 32 consecutive (lx,ly)
// columns of one z layer -> one 256-byte line per access).
struct VolView {
    float2 *vox;
    float *color;        // optional: per brick 3 planes of 512 f32 (r, g, b)
    uint8_t *flags;      // per brick: bit 0 = some voxel was updated, bit 1 = some voxel holds a tsdf != 1 (or was imported)
    int nx, ny, nz, gz0; // logical box; global z of local plane z = gz0 + (z / 8) * 8 * zs + z % 8
    int zs;              // z interleave stride in brick layers (1 = contiguous slab, N = round-robin over N ranks)
    int nbx, nby, nbz;   // bricks per axis (ceil)
    float vl, half, trunc, trunc_inv;
    double ox, oy, oz;
    // ScalableTSDFVolume mode (0 = off): the box consists of whole units of unit_res^3 voxels on the
    // world unit grid, origin = u0 * unit_len; only units activated by a frame are integrated by it
    int unit_res, unit_shift, unit_stride;   // unit_res = 1 << unit_shift
    int unit_nomask;     // 1: per-unit ARITHMETIC (voxel centres, z recurrence) for every unit of the box, no activation mask
    int u0[3];
    int nux, nuy, nuz;   // units per axis (z: of the whole grid when the box is a z-shard)
    double unit_len;
    // surface-extraction flavour: a voxel is valid when weight > w_min (0: Open3D's legacy `weight != 0`; the tensor
    // pipeline of `MAP` uses weight >= 3); vertices / points sit at (index + pos_half) * voxel_length (legacy 0.5 = voxel
    // centres, tensor pipeline 0 = voxel corners)
    float w_min;
    double pos_half;
};

// world position (f32, as Open3D narrows it) of the centre of GLOBAL voxel index g along `axis`:
// dense: float(f32(half + vl * g) + origin);  unit mode: the same inside the unit that holds g
// (UniformTSDFVolume of origin = unit index * unit_len, local index g % unit_res)
template <bool UNIT>
__device__ __forceinline__ float voxel_centre(const VolView &v, int axis, int g) {
    const double o = axis == 0 ? v.ox : (axis == 1 ? v.oy : v.oz);
    if (!UNIT) return (float)((double)(v.half + v.vl * (float)g) + o);
    const int u = g >> v.unit_shift, l = g & (v.unit_res - 1);
    return (float)((double)(v.half + v.vl * (float)l) + (double)(v.u0[axis] + u) * v.unit_len);
}

__host__ __device__ inline int64_t brick_count(const VolView &v) {
    return (int64_t)v.nbx * v.nby * v.nbz;
}

__device__ __forceinline__ int64_t voxel_slot(const VolView &v, int x, int y, int z) {
    const int bx = x >> 3, by = y >> 3, bz = z >> 3;
    const int64_t b = ((int64_t)bz * v.nby + by) * v.nbx + bx;
    return b * kBrickVox + ((z & 7) << 6) + ((x & 7) << 3) + (y & 7);
}

} // namespace bslam

// host-side handle
struct bslam_volume {
    bslam::VolView v;
    int device;
    int with_color;
    int owns_storage;
    void *storage;
    size_t storage_bytes;
    double voxel_length_d, sdf_trunc_d;
    // extraction scratch (lazily sized by brick count)
    void *mc_scratch;
    size_t mc_scratch_bytes;
    // integrate scratch: active-brick list + counters
    void *int_scratch;
    size_t int_scratch_bytes;
    // optional per-launch timing of the dominant kernel (bslam_tsdf_profile)
    int batch; // frames per integrate launch (0 = default)
    int prof_enabled, prof_n;
    int zpw;                                  // z layers per integrate warp (0 = auto by shard size)
    // incremental point extraction (bslam_points_set_incremental): per-brick cache of the extracted points
    void *pts_cache;
    size_t pts_cache_bytes;
    int pts_incremental, pts_with_normals, pts_cache_valid, pts_counted;
    long long pts_last_total, pts_last_candidates, pts_last_recomputed;
    // two-stream pipeline (bslam_tsdf_prepare_u16 / bslam_tsdf_integrate_prepared): second scratch buffer, two slots
    void *int_scratch2;
    void *slot_bp[2];                         // host copies of the prepared launches' parameters (BatchP)
    cudaEvent_t slot_ready[2], slot_free[2];
    int slot_used[2], slot_prof[2], slot_tiles[2][2];
    int prep_head, prep_tail, prep_pending;
    cudaStream_t hp_stream;                   // private high-priority stream of the pipelined integration
    cudaEvent_t hp_fence;
    int clip_stride;                          // dense mode: sampling stride of the out-of-box point count (0 = off)
    int z_total;                              // planes of the whole grid when this box is a z-shard (clip check)
    static constexpr int kProfPairs = 1024;   // integrate launches timed per bslam_tsdf_profile_read
    static constexpr int kProfStages = 3;     // depth statistics (+ fused a4) | unit marks + culls + order | brick integrate
    static constexpr int kProfEvents = 5;     // per launch: prepare start / after statistics / prepare end | integrate start / end
    cudaEvent_t prof_ev[kProfEvents * kProfPairs];
    double prof_ms_accum[kProfStages];
    long long prof_launches_accum;
};

namespace bslam {

// Workspace of the VoxelBlockGrid integrator (bslam_vbg.cu), also read by its ray cast (bslam_raycast.cu): a 256-byte
// header {u64 ray points seen, u64 ray points outside the box, i32 index of the last frame of the last launch}, the
// per-block frame masks of the last launch, then the cumulative allocation bitmap (bit b: block b was activated by a
// frame integrated so far).  Blocks are numbered b = (xb * nby + yb) * nbz + zb.
constexpr int kVbgBlock = 16;
constexpr int kVbgMaxFrames = 64;
constexpr int kVbgMaskWords = kVbgMaxFrames / 32;
constexpr size_t kVbgLastFrameOffset = 16;
constexpr size_t kVbgMasksOffset = 256;
inline size_t vbg_alloc_offset(size_t n_blocks) { return kVbgMasksOffset + n_blocks * kVbgMaskWords * 4; }

// block index of the box corner on the world block grid (origin = b0 * 16 * voxel); BSLAM_E_ARG when the origin is off it
int vbg_block_origin(const bslam_volume *vol, int b0[3]);

} // namespace bslam
