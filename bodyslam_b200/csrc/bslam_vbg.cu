// Row f4 -- the tensor-pipeline integrator behind the reference's `MAP` class (N/3DM/tsdf.py:56-108):
// Open3D `t.pipelines.slam.Model` = VoxelBlockGrid of 16^3 blocks, `model.integrate(frame, depth_scale, depth_max,
// trunc_voxel_multiplier)`.  Restated (from knowledge of Open3D's VoxelBlockGridImpl.h, NOT pinned: Open3D is not
// installable here) in oracle/o3d_oracle.c: orc_vbg_touch / orc_vbg_integrate, which this file must match bit for bit:
//   * block activation ("depth touch"): every 4th pixel with 0 < d < depth_max is unprojected to a ray; the blocks
//     holding the ray points at depths t_min + k * (t_max - t_min) / 3, k = 0..3, t_min = max(d - trunc, 0),
//     t_max = min(d + trunc, depth_max), are activated for the frame;
//   * per voxel of an activated block: position = integer voxel coordinate * voxel_size (voxel CORNER, no half-voxel
//     offset), camera point through the extrinsic whose rotation columns are pre-scaled by voxel_size, projection
//     u = fx * x * (1/z) + cx with truncation to the pixel, PROJECTIVE sdf = depth - z (no ray-length multiplier),
//     skipped when depth <= 0, depth > depth_max, z <= 0 or sdf < -trunc; tsdf = (w * tsdf + min(sdf, trunc) / trunc)
//     * (1 / (w + 1)), colour alike, w += 1.
// The blocks live in the same brick-ordered dense box as the legacy volume (a 16^3 block = 2 x 2 x 2 bricks), so
// the K4 extraction kernels serve both (weight threshold / vertex offset set through bslam_tsdf_set_extract_flavour).
// One thread per voxel, frames in order inside the thread: simple, correct, GPU-parallel -- this second integrator is
// not on the headline path (the reference's SLAM loop does not use MAP, N/3DM/slam.py).
#include <math.h>

#include "bslam_common.cuh"

namespace bslam {

constexpr int kVbgTouchStride = 4;
constexpr int kVbgSteps = 3;
constexpr int kVbgBitmapWords = 8192;      // shared bitmap of the touch kernel: up to 262 144 blocks (1024^3 voxels)

struct VbgFrame {
    float Es[12];     // world -> camera, rows 0..2; rotation entries pre-multiplied by voxel_size (float)
    float P[12];      // camera -> world (pose), rows 0..2, float
    float depth_max;
};
struct VbgBatch {
    int F, W, H;
    float fx, fy, cx, cy;
    float depth_scale, trunc, voxel_size, block_size;
    int b0[3];        // block index of the box corner on the world block grid
    int nb[3];        // blocks per axis
    VbgFrame fr[kVbgMaxFrames];
};

__global__ void __launch_bounds__(256) vbg_touch_kernel(const __grid_constant__ VbgBatch bp, const uint16_t *__restrict__ depth, unsigned int *block_masks,
                                                        unsigned int *alloc_bits, int *last_frame, unsigned long long *clip) {
    __shared__ unsigned int s_bits[kVbgBitmapWords];
    const int f = blockIdx.x;
    const int n_blocks = bp.nb[0] * bp.nb[1] * bp.nb[2];
    const int n_words = (n_blocks + 31) >> 5;
    for (int i = threadIdx.x; i < n_words; i += blockDim.x) s_bits[i] = 0u;
    __syncthreads();
    const VbgFrame &fp = bp.fr[f];
    const int rows_s = bp.H / kVbgTouchStride, cols_s = bp.W / kVbgTouchStride;
    const uint16_t *img = depth + (int64_t)f * bp.W * bp.H;
    unsigned int n_seen = 0, n_out = 0;
    for (int q = threadIdx.x; q < rows_s * cols_s; q += blockDim.x) {
        const int y = (q / cols_s) * kVbgTouchStride, x = (q % cols_s) * kVbgTouchStride;
        const float d = (float)img[(int64_t)y * bp.W + x] / bp.depth_scale;
        if (!(d > 0.0f && d < fp.depth_max)) continue;
        // Unproject(x, y, 1) then the pose
        const float xc = ((float)x - bp.cx) * 1.0f / bp.fx, yc = ((float)y - bp.cy) * 1.0f / bp.fy, zc = 1.0f;
        const float xg = ((xc * fp.P[0] + yc * fp.P[1]) + zc * fp.P[2]) + fp.P[3];
        const float yg = ((xc * fp.P[4] + yc * fp.P[5]) + zc * fp.P[6]) + fp.P[7];
        const float zg = ((xc * fp.P[8] + yc * fp.P[9]) + zc * fp.P[10]) + fp.P[11];
        const float xo = fp.P[3], yo = fp.P[7], zo = fp.P[11];
        const float xd = xg - xo, yd = yg - yo, zd = zg - zo;
        const float t_min = fmaxf(d - bp.trunc, 0.0f), t_max = fminf(d + bp.trunc, fp.depth_max);
        const float t_step = (t_max - t_min) / (float)kVbgSteps;
        float t = t_min;
        for (int step = 0; step <= kVbgSteps; ++step) {
            const int xb = (int)floorf((xo + t * xd) / bp.block_size) - bp.b0[0];
            const int yb = (int)floorf((yo + t * yd) / bp.block_size) - bp.b0[1];
            const int zb = (int)floorf((zo + t * zd) / bp.block_size) - bp.b0[2];
            ++n_seen;
            if (xb >= 0 && yb >= 0 && zb >= 0 && xb < bp.nb[0] && yb < bp.nb[1] && zb < bp.nb[2]) {
                const int b = (xb * bp.nb[1] + yb) * bp.nb[2] + zb;
                unsigned int *wp = &s_bits[b >> 5];
                const unsigned int m = 1u << (b & 31);
                if (!(*(volatile unsigned int *)wp & m)) atomicOr(wp, m);
            } else {
                ++n_out;      // the reference's hash map is unbounded, the box is not
            }
            t += t_step;
        }
    }
    __syncthreads();
    n_seen = __reduce_add_sync(0xffffffffu, n_seen);
    n_out = __reduce_add_sync(0xffffffffu, n_out);
    if ((threadIdx.x & 31) == 0 && n_seen && clip) {
        atomicAdd(clip + 0, (unsigned long long)n_seen);
        if (n_out) atomicAdd(clip + 1, (unsigned long long)n_out);
    }
    if (threadIdx.x == 0 && f == bp.F - 1) *last_frame = f;
    for (int i = threadIdx.x; i < n_words; i += blockDim.x) {
        unsigned int m = s_bits[i];
        if (m) atomicOr(&alloc_bits[i], m);
        while (m) {
            const int b = 32 * i + __ffs(m) - 1;
            m &= m - 1;
            atomicOr(&block_masks[(size_t)b * kVbgMaskWords + (f >> 5)], 1u << (f & 31));
        }
    }
}

template <bool COLOR>
__global__ void __launch_bounds__(256) vbg_integrate_kernel(const VolView v, const __grid_constant__ VbgBatch bp, const uint16_t *__restrict__ depth,
                                                            const uint8_t *__restrict__ rgb, const unsigned int *__restrict__ block_masks,
                                                            unsigned long long *counts) {
    const int b = blockIdx.x;
    unsigned int mask[kVbgMaskWords];
    bool any = false;
#pragma unroll
    for (int k = 0; k < kVbgMaskWords; ++k) { mask[k] = block_masks[(size_t)b * kVbgMaskWords + k]; any |= mask[k] != 0u; }
    if (!any) return;
    const int zb = b % bp.nb[2], yb = (b / bp.nb[2]) % bp.nb[1], xb = b / (bp.nb[2] * bp.nb[1]);
    const int64_t n_pix = (int64_t)bp.W * bp.H;
    for (int i = threadIdx.x; i < kVbgBlock * kVbgBlock * kVbgBlock; i += blockDim.x) {
        // voxel order inside a block: y fastest (one 8-voxel brick row per 8 lanes), then x, then z
        const int ly = i & 15, lx = (i >> 4) & 15, lz = i >> 8;
        const int X = xb * kVbgBlock + lx, Y = yb * kVbgBlock + ly, Z = zb * kVbgBlock + lz;
        if (X >= v.nx || Y >= v.ny || Z >= v.nz) continue;
        // integer voxel coordinate on the world grid, as float (Open3D: static_cast<float>(x))
        const float xw = (float)(bp.b0[0] * kVbgBlock + X), yw = (float)(bp.b0[1] * kVbgBlock + Y), zw = (float)(bp.b0[2] * kVbgBlock + Z);
        const int64_t slot = voxel_slot(v, X, Y, Z);
        float2 tw = v.vox[slot];
        float c[3] = {0.f, 0.f, 0.f};
        float *cp = nullptr;
        if (COLOR) {
            cp = v.color + (slot / kBrickVox) * (3 * kBrickVox) + (slot % kBrickVox);
            c[0] = cp[0]; c[1] = cp[kBrickVox]; c[2] = cp[2 * kBrickVox];
        }
        bool dirty = false;
#pragma unroll
        for (int k = 0; k < kVbgMaskWords; ++k) {
            unsigned int m = mask[k];
            while (m) {
                const int f = 32 * k + __ffs(m) - 1;
                m &= m - 1;
                const VbgFrame &fp = bp.fr[f];
                const float xc = ((xw * fp.Es[0] + yw * fp.Es[1]) + zw * fp.Es[2]) + fp.Es[3];
                const float yc = ((xw * fp.Es[4] + yw * fp.Es[5]) + zw * fp.Es[6]) + fp.Es[7];
                const float zc = ((xw * fp.Es[8] + yw * fp.Es[9]) + zw * fp.Es[10]) + fp.Es[11];
                const float inv_z = 1.0f / zc;
                const float u = bp.fx * xc * inv_z + bp.cx, vv = bp.fy * yc * inv_z + bp.cy;
                if (!(u >= 0.0f && vv >= 0.0f && u < (float)bp.W && vv < (float)bp.H)) continue;
                const int ui = (int)u, vi = (int)vv;
                const int64_t pix = (int64_t)vi * bp.W + ui;
                const float d = (float)__ldg(depth + f * n_pix + pix) / bp.depth_scale;
                float sdf = d - zc;
                if (d <= 0.0f || d > fp.depth_max || zc <= 0.0f || sdf < -bp.trunc) continue;
                sdf = sdf < bp.trunc ? sdf : bp.trunc;
                sdf /= bp.trunc;
                const float w = tw.y;
                const float inv = 1.0f / (w + 1.0f);
                tw.x = (w * tw.x + sdf) * inv;
                if (COLOR) {
                    const uint8_t *px = rgb + (f * n_pix + pix) * 3;
#pragma unroll
                    for (int q = 0; q < 3; ++q) c[q] = (w * c[q] + (float)px[q]) * inv;
                }
                tw.y = w + 1.0f;
                dirty = true;
                if (counts) atomicAdd(counts + f, 1ull);
            }
        }
        if (dirty) {
            v.vox[slot] = tw;
            if (COLOR) { cp[0] = c[0]; cp[kBrickVox] = c[1]; cp[2 * kBrickVox] = c[2]; }
            v.flags[slot / kBrickVox] = 7;     // touched + may hold a surface (extraction candidates) + changed since the last incremental extraction
        }
    }
}

int vbg_block_origin(const bslam_volume *vol, int b0[3]) {
    const double o[3] = {vol->v.ox, vol->v.oy, vol->v.oz};
    const double bs = vol->voxel_length_d * kVbgBlock;
    for (int r = 0; r < 3; ++r) {
        const double k = nearbyint(o[r] / bs);
        BSLAM_CHECK_ARG(fabs(k * bs - o[r]) <= 1e-9 * fmax(1.0, fabs(o[r])), "origin[%d] = %.12g is not a multiple of the block length %.12g", r, o[r], bs);
        b0[r] = (int)k;
    }
    return BSLAM_OK;
}

} // namespace bslam

using namespace bslam;

extern "C" {

size_t bslam_vbg_workspace_bytes(int nx, int ny, int nz) {
    const size_t nb = (size_t)((nx + 15) / 16) * ((ny + 15) / 16) * ((nz + 15) / 16);
    return vbg_alloc_offset(nb) + (nb + 31) / 32 * 4;
}


int bslam_vbg_integrate(bslam_volume *vol, const uint16_t *d_depth_u16, const uint8_t *d_rgb, int F, int H, int W, const double *h_K,
                        const double *h_poses, const double *h_depth_max, float depth_scale, float trunc_voxel_multiplier,
                        void *d_workspace, unsigned long long *d_update_counts, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(vol && d_depth_u16 && h_K && h_poses && h_depth_max && d_workspace, "bslam_vbg_integrate: NULL argument");
    BSLAM_CHECK_ARG(F >= 0 && H > 0 && W > 0, "[bslam_vbg_integrate] Unsupported image format. (F=%d H=%d W=%d)", F, H, W);
    BSLAM_CHECK_ARG(depth_scale > 0.f && trunc_voxel_multiplier > 0.f, "bslam_vbg_integrate: depth_scale and trunc_voxel_multiplier must be > 0");
    BSLAM_CHECK_ARG(!(vol->with_color && !d_rgb), "[bslam_vbg_integrate] Unsupported image format. (colour volume needs an RGB8 image)");
    const VolView &v = vol->v;
    BSLAM_CHECK_ARG(v.zs == 1 && v.gz0 == 0 && !v.unit_res, "bslam_vbg_integrate: single-box volumes without unit activation only");
    if (F == 0) return BSLAM_OK;
    BSLAM_DEVICE_GUARD(vol->device);
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local VbgBatch bp;
    bp.W = W; bp.H = H;
    bp.fx = (float)h_K[0]; bp.fy = (float)h_K[1]; bp.cx = (float)h_K[2]; bp.cy = (float)h_K[3];
    bp.depth_scale = depth_scale;
    bp.voxel_size = v.vl;
    bp.trunc = v.vl * trunc_voxel_multiplier;
    bp.block_size = v.vl * (float)kVbgBlock;
    if (vbg_block_origin(vol, bp.b0) != BSLAM_OK) return BSLAM_E_ARG;
    bp.nb[0] = (v.nx + 15) / 16; bp.nb[1] = (v.ny + 15) / 16; bp.nb[2] = (v.nz + 15) / 16;
    const int n_blocks = bp.nb[0] * bp.nb[1] * bp.nb[2];
    BSLAM_CHECK_ARG((n_blocks + 31) / 32 <= kVbgBitmapWords, "bslam_vbg_integrate: too many blocks (%d)", n_blocks);
    unsigned int *masks = (unsigned int *)((char *)d_workspace + kVbgMasksOffset);
    unsigned int *alloc_bits = (unsigned int *)((char *)d_workspace + vbg_alloc_offset(n_blocks));
    int *last_frame = (int *)((char *)d_workspace + kVbgLastFrameOffset);
    unsigned long long *clip = (unsigned long long *)d_workspace;
    const int64_t n_pix = (int64_t)W * H;
    for (int f0 = 0; f0 < F; f0 += kVbgMaxFrames) {
        const int nf = F - f0 < kVbgMaxFrames ? F - f0 : kVbgMaxFrames;
        bp.F = nf;
        for (int f = 0; f < nf; ++f) {
            const double *P = h_poses + (size_t)(f0 + f) * 16;       // camera -> world (T_frame_to_model)
            // world -> camera: rigid inverse in f64 (Open3D: core::Tensor Inverse of the pose)
            double E[12];
            for (int i = 0; i < 3; ++i) {
                for (int j = 0; j < 3; ++j) E[4 * i + j] = P[4 * j + i];
                E[4 * i + 3] = -(P[4 * 0 + i] * P[3] + P[4 * 1 + i] * P[7] + P[4 * 2 + i] * P[11]);
            }
            VbgFrame &fp = bp.fr[f];
            for (int i = 0; i < 3; ++i) {
                for (int j = 0; j < 3; ++j) fp.Es[4 * i + j] = (float)E[4 * i + j] * v.vl;
                fp.Es[4 * i + 3] = (float)E[4 * i + 3];
            }
            for (int i = 0; i < 12; ++i) fp.P[i] = (float)P[i];
            fp.depth_max = (float)h_depth_max[f0 + f];
        }
        BSLAM_CUDA(cudaMemsetAsync(masks, 0, (size_t)n_blocks * kVbgMaskWords * 4, st));
        vbg_touch_kernel<<<nf, 256, 0, st>>>(bp, d_depth_u16 + f0 * n_pix, masks, alloc_bits, last_frame, clip);
        BSLAM_LAUNCH_CHECK();
        unsigned long long *cnt = d_update_counts ? d_update_counts + f0 : nullptr;
        if (vol->with_color)
            vbg_integrate_kernel<true><<<n_blocks, 256, 0, st>>>(v, bp, d_depth_u16 + f0 * n_pix, d_rgb + f0 * n_pix * 3, masks, cnt);
        else
            vbg_integrate_kernel<false><<<n_blocks, 256, 0, st>>>(v, bp, d_depth_u16 + f0 * n_pix, nullptr, masks, cnt);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

int bslam_vbg_stats(const void *d_workspace, unsigned long long *h_stat2, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(d_workspace && h_stat2, "bslam_vbg_stats: NULL argument");
    BSLAM_CUDA(cudaMemcpyAsync(h_stat2, d_workspace, 16, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    BSLAM_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return BSLAM_OK;
}

int bslam_tsdf_set_extract_flavour(bslam_volume *vol, float weight_threshold, double vertex_offset) {
    BSLAM_CHECK_ARG(vol != nullptr && weight_threshold >= 0.f && vertex_offset >= 0.0 && vertex_offset <= 1.0, "bslam_tsdf_set_extract_flavour: bad argument");
    // valid voxel <=> weight >= threshold (threshold 0: weight != 0, Open3D's legacy rule; weights are never negative)
    vol->v.w_min = weight_threshold > 0.f ? nextafterf(weight_threshold, 0.0f) : 0.0f;
    vol->v.pos_half = vertex_offset;
    vol->pts_cache_valid = 0;
    return BSLAM_OK;
}

} // extern "C"
