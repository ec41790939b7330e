// Ray casting of the TSDF volume: rendered depth, vertex, normal and colour maps from a pose.  Tensor flavour (`MAP`,
// Open3D `t.pipelines.slam.Model.synthesize_model_frame` = VoxelBlockGrid::RayCast after EstimateRange) and legacy
// flavour (`DenseTSDFVolume`).  The semantics, including where they deliberately differ from Open3D, are written down in
// the CPU reference tests/raycast_ref.c (ref_raycast), which this file must match bit for bit (-fmad=false, IEEE `/`
// and sqrtf).
//   * one thread per ray; a warp covers an 8 x 4 pixel tile, so neighbouring rays gather from the same lines;
//     frames of one call run in gridDim.y;
//   * the march caches the current block index and its allocation bit in registers (Open3D's MiniVecCache) and
//     reads the volume through the read-only path; the call never writes the volume;
//   * templated on the flavour and on normals / colour, so a depth-only cast pays nothing for the trilinear pass.
#include <math.h>

#include "bslam_common.cuh"

namespace bslam {

constexpr int kRcMaxFrames = 64;
constexpr int kRcDown = 8;        // EstimateRange's down factor
constexpr int kRcTileW = 32, kRcTileH = 8;

struct RcFrame {
    float P[12];      // camera -> world, rows 0..2
    float E[12];      // world -> camera, rows 0..2
};
struct RcBatch {
    int F, W, H;
    float fx, fy, cx, cy;
    float depth_scale, depth_min, depth_max, w_thr, trunc, vl, bl, half;
    float org[3];                     // legacy: the float origin of the box; tensor: 0 (world block grid)
    int b0[3];                        // tensor: block index of the box corner on the world block grid; legacy: 0
    int nb[3];                        // blocks per axis (16^3 tensor blocks / 8^3 bricks)
    int n[3];                         // voxels per axis
    const unsigned int *alloc_bits;   // tensor: cumulative allocation bitmap, b = (xb * nby + yb) * nbz + zb
    const float2 *range;              // tensor: [H / 8][W / 8] {t_min, t_max}
    RcFrame fr[kRcMaxFrames];
};

template <bool TENSOR>
__device__ __forceinline__ bool rc_block_alloc(const VolView &v, const RcBatch &bp, int bx, int by, int bz) {
    if (TENSOR) {
        const int b = (bx * bp.nb[1] + by) * bp.nb[2] + bz;
        return (__ldg(bp.alloc_bits + (b >> 5)) >> (b & 31)) & 1u;
    }
    return __ldg(v.flags + ((int64_t)bz * v.nby + by) * v.nbx + bx) & 1u;     // brick flag bit 0: some voxel was updated
}

// voxel (X, Y, Z) of the box exists in the volume: inside the box and its block allocated
template <bool TENSOR>
__device__ __forceinline__ bool rc_voxel_alloc(const VolView &v, const RcBatch &bp, int X, int Y, int Z) {
    if ((unsigned)X >= (unsigned)bp.n[0] || (unsigned)Y >= (unsigned)bp.n[1] || (unsigned)Z >= (unsigned)bp.n[2]) return false;
    constexpr int S = TENSOR ? 4 : 3;
    return rc_block_alloc<TENSOR>(v, bp, X >> S, Y >> S, Z >> S);
}

template <bool TENSOR, bool NORMAL, bool COLOR>
__global__ void __launch_bounds__(256, 1) raycast_kernel(const VolView v, const __grid_constant__ RcBatch bp, float *__restrict__ out_depth,
                                                      float *__restrict__ out_vertex, float *__restrict__ out_normal, float *__restrict__ out_color) {
    constexpr int B = TENSOR ? 16 : 8;
    const int tiles_x = (bp.W + kRcTileW - 1) / kRcTileW;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int x = (blockIdx.x % tiles_x) * kRcTileW + (warp & 3) * 8 + (lane & 7);
    const int y = (blockIdx.x / tiles_x) * kRcTileH + (warp >> 2) * 4 + (lane >> 3);
    if (x >= bp.W || y >= bp.H) return;
    const int f = blockIdx.y;
    const RcFrame &fr = bp.fr[f];
    const int64_t pix = ((int64_t)f * bp.H + y) * bp.W + x;

    float t = bp.depth_min, t_max = bp.depth_max;
    if (TENSOR) {
        const int wd = bp.W / kRcDown, hd = bp.H / kRcDown;
        const int cxi = min(x / kRcDown, wd - 1), cyi = min(y / kRcDown, hd - 1);
        const float2 r = bp.range[cyi * wd + cxi];
        t = r.x; t_max = r.y;
    }
    float depth = 0.f, vert[3] = {0.f, 0.f, 0.f}, nrm[3] = {0.f, 0.f, 0.f}, col[3] = {0.f, 0.f, 0.f};
    if (t < t_max) {
        const float xc = ((float)x - bp.cx) * 1.0f / bp.fx, yc = ((float)y - bp.cy) * 1.0f / bp.fy, zc = 1.0f;
        const float o[3] = {fr.P[3], fr.P[7], fr.P[11]};
        float d[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) d[r] = (((xc * fr.P[4 * r] + yc * fr.P[4 * r + 1]) + zc * fr.P[4 * r + 2]) + fr.P[4 * r + 3]) - o[r];
        float t_prev = t, tsdf_prev = -1.0f, ts = 1.0f;
        bool hit = false;
        int cur_key = -2;          // block of the previous sample (-1 = outside the box)
        bool cur_ok = false;
        while (t < t_max) {
            int X[3], bi[3];
            bool in = true;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const float q = (o[r] + t * d[r]) - bp.org[r];
                const float bw = floorf(q / bp.bl);
                const int l = min((int)((q - bw * bp.bl) / bp.vl), B - 1);
                bi[r] = (int)bw - bp.b0[r];
                in &= (unsigned)bi[r] < (unsigned)bp.nb[r];
                X[r] = bi[r] * B + l;
            }
            const int key = in ? (bi[0] * bp.nb[1] + bi[1]) * bp.nb[2] + bi[2] : -1;
            if (key != cur_key) {
                cur_key = key;
                cur_ok = in && rc_block_alloc<TENSOR>(v, bp, bi[0], bi[1], bi[2]);
            }
            if (!cur_ok) { t_prev = t; t += bp.bl; continue; }
            const float2 tw = __ldg(v.vox + voxel_slot(v, X[0], X[1], X[2]));
            tsdf_prev = ts;
            ts = tw.x;
            if (tsdf_prev > 0.0f && (bp.w_thr > 0.0f ? tw.y >= bp.w_thr : tw.y != 0.0f) && ts <= 0.0f) { hit = true; break; }
            t_prev = t;
            const float delta = ts * bp.trunc;
            t += delta < bp.vl ? bp.vl : delta;
        }
        if (hit) {
            const float ti = (t * tsdf_prev - t_prev * ts) / (tsdf_prev - ts);
            depth = ti * bp.depth_scale;
            float p[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) p[r] = o[r] + ti * d[r];
#pragma unroll
            for (int r = 0; r < 3; ++r) vert[r] = ((fr.E[4 * r] * p[0] + fr.E[4 * r + 1] * p[1]) + fr.E[4 * r + 2] * p[2]) + fr.E[4 * r + 3];
            if (NORMAL || COLOR) {
                int base[3];
                float xv[3];
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const float q = p[r] - bp.org[r];
                    const float bw = floorf(q / bp.bl);
                    xv[r] = (q - bw * bp.bl) / bp.vl - bp.half;
                    const float fl = floorf(xv[r]);
                    base[r] = ((int)bw - bp.b0[r]) * B + (int)fl;
                    xv[r] -= fl;
                }
                float sum_r = 0.f, nacc[3] = {0.f, 0.f, 0.f}, cacc[3] = {0.f, 0.f, 0.f};
#pragma unroll 1
                for (int k = 0; k < 8; ++k) {
                    const int dk0 = k & 1, dk1 = (k >> 1) & 1, dk2 = (k >> 2) & 1;
                    const int CX = base[0] + dk0, CY = base[1] + dk1, CZ = base[2] + dk2;
                    if (!rc_voxel_alloc<TENSOR>(v, bp, CX, CY, CZ)) continue;
                    const int64_t slot = voxel_slot(v, CX, CY, CZ);
                    if (!(__ldg(v.vox + slot).y > 0.0f)) continue;
                    const float r = ((1.0f - fabsf((float)dk0 - xv[0])) * (1.0f - fabsf((float)dk1 - xv[1]))) * (1.0f - fabsf((float)dk2 - xv[2]));
                    sum_r += r;
                    if (NORMAL) {
                        const int C[3] = {CX, CY, CZ};
#pragma unroll
                        for (int a = 0; a < 3; ++a) {
                            int lo[3] = {C[0], C[1], C[2]}, hi[3] = {C[0], C[1], C[2]};
                            lo[a] -= 1; hi[a] += 1;
                            float g = 0.0f;
                            if (rc_voxel_alloc<TENSOR>(v, bp, lo[0], lo[1], lo[2]) && rc_voxel_alloc<TENSOR>(v, bp, hi[0], hi[1], hi[2]))
                                g = __ldg(v.vox + voxel_slot(v, hi[0], hi[1], hi[2])).x - __ldg(v.vox + voxel_slot(v, lo[0], lo[1], lo[2])).x;
                            nacc[a] += r * g;
                        }
                    }
                    if (COLOR) {
                        const float *cp = v.color + slot + (slot / kBrickVox) * (2 * kBrickVox);     // brick b: 3 planes of 512 at b * 1536
#pragma unroll
                        for (int c = 0; c < 3; ++c) cacc[c] += r * __ldg(cp + c * kBrickVox);
                    }
                }
                if (sum_r > 0.0f) {
                    if (COLOR) {
                        const float s = sum_r * 255.0f;
#pragma unroll
                        for (int c = 0; c < 3; ++c) col[c] = cacc[c] / s;
                    }
                    if (NORMAL) {
                        const float n2 = (nacc[0] * nacc[0] + nacc[1] * nacc[1]) + nacc[2] * nacc[2];
                        if (n2 > 0.0f) {
                            const float len = sqrtf(n2);
                            const float n[3] = {nacc[0] / len, nacc[1] / len, nacc[2] / len};
#pragma unroll
                            for (int r = 0; r < 3; ++r) nrm[r] = (fr.E[4 * r] * n[0] + fr.E[4 * r + 1] * n[1]) + fr.E[4 * r + 2] * n[2];
                        }
                    }
                }
            }
        }
    }
    out_depth[pix] = depth;
    if (out_vertex) {
#pragma unroll
        for (int r = 0; r < 3; ++r) out_vertex[3 * pix + r] = vert[r];
    }
    if (NORMAL) {
#pragma unroll
        for (int r = 0; r < 3; ++r) out_normal[3 * pix + r] = nrm[r];
    }
    if (COLOR) {
#pragma unroll
        for (int r = 0; r < 3; ++r) out_color[3 * pix + r] = col[r];
    }
}

// EstimateRange of the tensor flavour: every cell starts at [depth_max, depth_min] ...
__global__ void rc_range_init_kernel(float2 *range, int n, float depth_min, float depth_max) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) range[i] = make_float2(depth_max, depth_min);
}

// order-preserving float min / max through the integer atomics (the result does not depend on the order)
__device__ __forceinline__ void atomic_min_float(float *a, float x) {
    if (x >= 0.0f) atomicMin((int *)a, __float_as_int(x));
    else atomicMax((unsigned int *)a, __float_as_uint(x));
}
__device__ __forceinline__ void atomic_max_float(float *a, float x) {
    if (x >= 0.0f) atomicMax((int *)a, __float_as_int(x));
    else atomicMin((unsigned int *)a, __float_as_uint(x));
}

// ... then one thread per block of the box: a block the last integrated frame activated widens the cells its
// projected bounding box covers
__global__ void __launch_bounds__(256) rc_range_blocks_kernel(const __grid_constant__ RcBatch bp, const unsigned int *__restrict__ masks,
                                                              const int *__restrict__ last_frame, float2 *range) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= bp.nb[0] * bp.nb[1] * bp.nb[2]) return;
    const int lf = *last_frame;
    if (!((masks[(size_t)b * kVbgMaskWords + (lf >> 5)] >> (lf & 31)) & 1u)) return;
    const int zb = b % bp.nb[2], yb = (b / bp.nb[2]) % bp.nb[1], xb = b / (bp.nb[2] * bp.nb[1]);
    const int key[3] = {bp.b0[0] + xb, bp.b0[1] + yb, bp.b0[2] + zb};
    const float *E = bp.fr[0].E;
    const int wd = bp.W / kRcDown, hd = bp.H / kRcDown;
    int u_min = wd - 1, v_min = hd - 1, u_max = 0, v_max = 0;
    float z_min = bp.depth_max, z_max = bp.depth_min;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float xw = (float)(key[0] + ((i & 1) > 0)) * bp.bl;
        const float yw = (float)(key[1] + ((i & 2) > 0)) * bp.bl;
        const float zw = (float)(key[2] + ((i & 4) > 0)) * bp.bl;
        const float xc = ((E[0] * xw + E[1] * yw) + E[2] * zw) + E[3];
        const float yc = ((E[4] * xw + E[5] * yw) + E[6] * zw) + E[7];
        const float zc = ((E[8] * xw + E[9] * yw) + E[10] * zw) + E[11];
        if (zc <= 0.0f) continue;
        const float inv_z = 1.0f / zc;
        const float u = (bp.fx * xc * inv_z + bp.cx) / 8.0f, vv = (bp.fy * yc * inv_z + bp.cy) / 8.0f;
        v_min = min((int)floorf(vv), v_min);
        v_max = max((int)ceilf(vv), v_max);
        u_min = min((int)floorf(u), u_min);
        u_max = max((int)ceilf(u), u_max);
        z_min = fminf(z_min, zc);
        z_max = fmaxf(z_max, zc);
    }
    v_min = max(0, v_min); v_max = min(hd - 1, v_max);
    u_min = max(0, u_min); u_max = min(wd - 1, u_max);
    if (v_min >= v_max || u_min >= u_max || z_min >= z_max) return;
    for (int yy = v_min; yy <= v_max; ++yy)
        for (int xx = u_min; xx <= u_max; ++xx) {
            float2 *r = range + yy * wd + xx;
            atomic_min_float(&r->x, z_min);
            atomic_max_float(&r->y, z_max);
        }
}

static void rigid_inverse(const double *A, double *out) {
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) out[4 * i + j] = A[4 * j + i];
        out[4 * i + 3] = -(A[4 * 0 + i] * A[3] + A[4 * 1 + i] * A[7] + A[4 * 2 + i] * A[11]);
    }
}

// pose (camera -> world) or extrinsic (world -> camera) 4x4 f64 -> the frame's float P and E
static void rc_set_frame(RcFrame &fr, const double *M, bool is_pose) {
    double P[12], E[12];
    if (is_pose) { for (int i = 0; i < 12; ++i) P[i] = M[i]; rigid_inverse(M, E); }
    else { for (int i = 0; i < 12; ++i) E[i] = M[i]; rigid_inverse(M, P); }
    for (int i = 0; i < 12; ++i) { fr.P[i] = (float)P[i]; fr.E[i] = (float)E[i]; }
}

template <bool TENSOR>
static void rc_launch(const VolView &v, const RcBatch &bp, float *depth, float *vertex, float *normal, float *color, cudaStream_t st) {
    const dim3 grid(((bp.W + kRcTileW - 1) / kRcTileW) * ((bp.H + kRcTileH - 1) / kRcTileH), bp.F);
    if (normal && color) raycast_kernel<TENSOR, true, true><<<grid, 256, 0, st>>>(v, bp, depth, vertex, normal, color);
    else if (normal) raycast_kernel<TENSOR, true, false><<<grid, 256, 0, st>>>(v, bp, depth, vertex, normal, color);
    else if (color) raycast_kernel<TENSOR, false, true><<<grid, 256, 0, st>>>(v, bp, depth, vertex, normal, color);
    else raycast_kernel<TENSOR, false, false><<<grid, 256, 0, st>>>(v, bp, depth, vertex, normal, color);
}

static void rc_common(RcBatch &bp, const VolView &v, int H, int W, const double *h_K, float depth_scale, float depth_min, float depth_max,
                      float weight_threshold) {
    bp.W = W; bp.H = H;
    bp.fx = (float)h_K[0]; bp.fy = (float)h_K[1]; bp.cx = (float)h_K[2]; bp.cy = (float)h_K[3];
    bp.depth_scale = depth_scale; bp.depth_min = depth_min; bp.depth_max = depth_max; bp.w_thr = weight_threshold;
    bp.vl = v.vl;
    bp.n[0] = v.nx; bp.n[1] = v.ny; bp.n[2] = v.nz;
}

} // namespace bslam

using namespace bslam;

// n_frames == 0: the outputs are empty, so their pointers may be NULL (an empty tensor's data pointer)
#define RC_CHECK_COMMON(name, n_frames)                                                                                                \
    BSLAM_CHECK_ARG(H > 0 && W > 0, "[" name "] Unsupported image format. (H=%d W=%d)", H, W);                                          \
    BSLAM_CHECK_ARG(depth_scale > 0.f && depth_min >= 0.f && isfinite(depth_min) && isfinite(depth_max) && weight_threshold >= 0.f,     \
                    name ": depth_scale must be > 0, depth_min >= 0, depth_max finite and weight_threshold >= 0");                     \
    BSLAM_CHECK_ARG(vol && h_K && (d_depth || (n_frames) == 0), name ": NULL argument");                                            \
    BSLAM_CHECK_ARG(!(d_color && !vol->with_color), "[" name "] a colour map needs a colour volume");                                 \
    BSLAM_CHECK_ARG(vol->v.zs == 1 && vol->v.gz0 == 0 && (vol->z_total == 0 || vol->z_total == vol->v.nz),                            \
                    name ": single-box volumes only (no z-sharded or z-interleaved boxes)")

extern "C" {

int bslam_tsdf_raycast(bslam_volume *vol, int F, int H, int W, const double *h_K, const double *h_extrinsics, float depth_scale,
                       float depth_min, float depth_max, float weight_threshold, float *d_depth, float *d_vertex, float *d_normal,
                       float *d_color, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(F >= 0, "[bslam_tsdf_raycast] Unsupported image format. (F=%d)", F);
    RC_CHECK_COMMON("bslam_tsdf_raycast", F);
    BSLAM_CHECK_ARG(h_extrinsics || F == 0, "bslam_tsdf_raycast: NULL argument");
    const VolView &v = vol->v;
    BSLAM_CHECK_ARG(v.nx % kBrick == 0 && v.ny % kBrick == 0 && v.nz % kBrick == 0, "bslam_tsdf_raycast: the box must consist of whole %d^3 bricks", kBrick);
    if (F == 0) return BSLAM_OK;
    BSLAM_DEVICE_GUARD(vol->device);
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local RcBatch bp;
    rc_common(bp, v, H, W, h_K, depth_scale, depth_min, depth_max, weight_threshold);
    bp.trunc = v.trunc;
    bp.bl = v.vl * (float)kBrick;
    bp.half = 0.5f;
    bp.org[0] = (float)v.ox; bp.org[1] = (float)v.oy; bp.org[2] = (float)v.oz;
    for (int r = 0; r < 3; ++r) { bp.b0[r] = 0; bp.nb[r] = bp.n[r] / kBrick; }
    bp.alloc_bits = nullptr; bp.range = nullptr;
    const int64_t n_pix = (int64_t)W * H;
    for (int f0 = 0; f0 < F; f0 += kRcMaxFrames) {
        bp.F = F - f0 < kRcMaxFrames ? F - f0 : kRcMaxFrames;
        for (int f = 0; f < bp.F; ++f) rc_set_frame(bp.fr[f], h_extrinsics + (size_t)(f0 + f) * 16, false);
        const int64_t o = f0 * n_pix;
        rc_launch<false>(v, bp, d_depth + o, d_vertex ? d_vertex + 3 * o : nullptr, d_normal ? d_normal + 3 * o : nullptr,
                         d_color ? d_color + 3 * o : nullptr, st);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

size_t bslam_vbg_raycast_workspace_bytes(int H, int W) {
    if (H < kRcDown || W < kRcDown) return 0;
    return (size_t)(H / kRcDown) * (W / kRcDown) * sizeof(float2);
}

int bslam_vbg_raycast(bslam_volume *vol, const void *d_vbg_workspace, int H, int W, const double *h_K, const double *h_pose, float depth_scale,
                      float depth_min, float depth_max, float weight_threshold, float trunc_voxel_multiplier, float *d_depth, float *d_vertex,
                      float *d_normal, float *d_color, void *d_range_workspace, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(H >= kRcDown && W >= kRcDown, "[bslam_vbg_raycast] Unsupported image format. (H=%d W=%d; at least %d x %d)", H, W, kRcDown, kRcDown);
    RC_CHECK_COMMON("bslam_vbg_raycast", 1);
    BSLAM_CHECK_ARG(d_vbg_workspace && h_pose && d_range_workspace, "bslam_vbg_raycast: NULL argument");
    BSLAM_CHECK_ARG(trunc_voxel_multiplier > 0.f, "bslam_vbg_raycast: trunc_voxel_multiplier must be > 0");
    const VolView &v = vol->v;
    BSLAM_CHECK_ARG(!v.unit_res, "bslam_vbg_raycast: volumes without unit activation only");
    BSLAM_CHECK_ARG(v.nx % kVbgBlock == 0 && v.ny % kVbgBlock == 0 && v.nz % kVbgBlock == 0, "bslam_vbg_raycast: the box must consist of whole %d^3 blocks", kVbgBlock);
    static thread_local RcBatch bp;
    if (vbg_block_origin(vol, bp.b0) != BSLAM_OK) return BSLAM_E_ARG;
    BSLAM_DEVICE_GUARD(vol->device);
    cudaStream_t st = (cudaStream_t)stream;
    rc_common(bp, v, H, W, h_K, depth_scale, depth_min, depth_max, weight_threshold);
    bp.F = 1;
    bp.trunc = v.vl * trunc_voxel_multiplier;
    bp.bl = v.vl * (float)kVbgBlock;
    bp.half = 0.0f;
    for (int r = 0; r < 3; ++r) { bp.org[r] = 0.0f; bp.nb[r] = bp.n[r] / kVbgBlock; }
    const int n_blocks = bp.nb[0] * bp.nb[1] * bp.nb[2];
    const char *ws = (const char *)d_vbg_workspace;
    bp.alloc_bits = (const unsigned int *)(ws + vbg_alloc_offset(n_blocks));
    bp.range = (const float2 *)d_range_workspace;
    rc_set_frame(bp.fr[0], h_pose, true);
    float2 *range = (float2 *)d_range_workspace;
    const int n_cells = (H / kRcDown) * (W / kRcDown);
    rc_range_init_kernel<<<(n_cells + 255) / 256, 256, 0, st>>>(range, n_cells, depth_min, depth_max);
    BSLAM_LAUNCH_CHECK();
    rc_range_blocks_kernel<<<(n_blocks + 255) / 256, 256, 0, st>>>(bp, (const unsigned int *)(ws + kVbgMasksOffset),
                                                                   (const int *)(ws + kVbgLastFrameOffset), range);
    BSLAM_LAUNCH_CHECK();
    rc_launch<true>(v, bp, d_depth, d_vertex, d_normal, d_color, st);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

} // extern "C"
