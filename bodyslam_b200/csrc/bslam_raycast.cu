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
#include <limits.h>
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

// Reads of one box (bslam_tsdf_raycast / bslam_vbg_raycast): the whole volume lives in `v`.  The march and the shading
// below are written against this interface so that a z-slab with its halo planes (RcSlabVol) can run them unchanged.
template <bool TENSOR>
struct RcBoxVol {
    const VolView &v;
    const RcBatch &bp;
    __device__ __forceinline__ bool foreign(int) const { return false; }
    __device__ __forceinline__ bool block_alloc(int bx, int by, int bz) const { return rc_block_alloc<TENSOR>(v, bp, bx, by, bz); }
    __device__ __forceinline__ bool voxel_alloc(int X, int Y, int Z) const { return rc_voxel_alloc<TENSOR>(v, bp, X, Y, Z); }
    __device__ __forceinline__ float2 voxel(int X, int Y, int Z) const { return __ldg(v.vox + voxel_slot(v, X, Y, Z)); }
    // a voxel and its colour through one slot (c-th colour channel at [c * color_stride(slot)])
    __device__ __forceinline__ int64_t slot(int X, int Y, int Z) const { return voxel_slot(v, X, Y, Z); }
    __device__ __forceinline__ float2 voxel_at(int64_t slot) const { return __ldg(v.vox + slot); }
    __device__ __forceinline__ const float *color_at(int64_t slot) const {
        return v.color + slot + (slot / kBrickVox) * (2 * kBrickVox);              // brick b: 3 planes of 512 at b * 1536
    }
    __device__ __forceinline__ int color_stride(int64_t) const { return kBrickVox; }
};

// ray of pixel (x, y): origin o and (unnormalised) direction d in world coordinates
__device__ __forceinline__ void rc_ray(const RcBatch &bp, const RcFrame &fr, int x, int y, float o[3], float d[3]) {
    const float xc = ((float)x - bp.cx) * 1.0f / bp.fx, yc = ((float)y - bp.cy) * 1.0f / bp.fy, zc = 1.0f;
    o[0] = fr.P[3]; o[1] = fr.P[7]; o[2] = fr.P[11];
#pragma unroll
    for (int r = 0; r < 3; ++r) d[r] = (((xc * fr.P[4 * r] + yc * fr.P[4 * r + 1]) + zc * fr.P[4 * r + 2]) + fr.P[4 * r + 3]) - o[r];
}

// The march's loop state between samples is (t, t_prev, ts); the block cache is a pure function of the block key.
// Marches until a zero crossing (returns true; the crossing lies between t_prev and t), t >= t_max (false), or a
// sample whose brick layer the accessor calls foreign (false with t < t_max; bz_next = that layer): that sample is not
// read, so the march resumes from the same state wherever the sample is owned.  The state is copied in and out: the
// legacy kernels compile to the same code as before the march was shared.
template <bool TENSOR, class Vol>
__device__ __forceinline__ bool rc_march(const Vol &a, const RcBatch &bp, const float o[3], const float d[3], float t_max, float &t_io, float &t_prev_io,
                                        float &tsdf_prev_io, float &ts_io, int &bz_next) {
    constexpr int B = TENSOR ? 16 : 8;
    float t = t_io, t_prev = t_prev_io, tsdf_prev = tsdf_prev_io, ts = ts_io;
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
        if (a.foreign(bi[2])) { bz_next = bi[2]; break; }
        const int key = in ? (bi[0] * bp.nb[1] + bi[1]) * bp.nb[2] + bi[2] : -1;
        if (key != cur_key) {
            cur_key = key;
            cur_ok = in && a.block_alloc(bi[0], bi[1], bi[2]);
        }
        if (!cur_ok) { t_prev = t; t += bp.bl; continue; }
        const float2 tw = a.voxel(X[0], X[1], X[2]);
        tsdf_prev = ts;
        ts = tw.x;
        if (tsdf_prev > 0.0f && (bp.w_thr > 0.0f ? tw.y >= bp.w_thr : tw.y != 0.0f) && ts <= 0.0f) { hit = true; break; }
        t_prev = t;
        const float delta = ts * bp.trunc;
        t += delta < bp.vl ? bp.vl : delta;
    }
    t_io = t; t_prev_io = t_prev; tsdf_prev_io = tsdf_prev; ts_io = ts;
    return hit;
}

// the interpolated hit distance of a march that returned kRcHit
__device__ __forceinline__ float rc_hit_t(float t, float t_prev, float tsdf_prev, float ts) {
    return (t * tsdf_prev - t_prev * ts) / (tsdf_prev - ts);
}

// trilinear base voxel (global box index) and fractions of the point p
template <bool TENSOR>
__device__ __forceinline__ void rc_trilinear_base(const RcBatch &bp, const float p[3], int base[3], float xv[3]) {
    constexpr int B = TENSOR ? 16 : 8;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float q = p[r] - bp.org[r];
        const float bw = floorf(q / bp.bl);
        xv[r] = (q - bw * bp.bl) / bp.vl - bp.half;
        const float fl = floorf(xv[r]);
        base[r] = ((int)bw - bp.b0[r]) * B + (int)fl;
        xv[r] -= fl;
    }
}

// trilinear sums at the hit point over the 8 corners of `base` and, for the normal, their +-1 neighbours, that is
// planes base[2] - 1 ... base[2] + 2: adds the weight sum, gradient (nacc) and colour (cacc) sums
template <bool NORMAL, bool COLOR, class Vol>
__device__ __forceinline__ void rc_trilinear_sums(const Vol &a, const int base[3], const float xv[3], float &sum_r, float nacc[3], float cacc[3]) {
#pragma unroll 1
    for (int k = 0; k < 8; ++k) {
        const int dk0 = k & 1, dk1 = (k >> 1) & 1, dk2 = (k >> 2) & 1;
        const int CX = base[0] + dk0, CY = base[1] + dk1, CZ = base[2] + dk2;
        if (!a.voxel_alloc(CX, CY, CZ)) continue;
        const int64_t slot = a.slot(CX, CY, CZ);
        if (!(a.voxel_at(slot).y > 0.0f)) continue;
        const float r = ((1.0f - fabsf((float)dk0 - xv[0])) * (1.0f - fabsf((float)dk1 - xv[1]))) * (1.0f - fabsf((float)dk2 - xv[2]));
        sum_r += r;
        if (NORMAL) {
            const int C[3] = {CX, CY, CZ};
#pragma unroll
            for (int ax = 0; ax < 3; ++ax) {
                int lo[3] = {C[0], C[1], C[2]}, hi[3] = {C[0], C[1], C[2]};
                lo[ax] -= 1; hi[ax] += 1;
                float g = 0.0f;
                if (a.voxel_alloc(lo[0], lo[1], lo[2]) && a.voxel_alloc(hi[0], hi[1], hi[2]))
                    g = a.voxel_at(a.slot(hi[0], hi[1], hi[2])).x - a.voxel_at(a.slot(lo[0], lo[1], lo[2])).x;
                nacc[ax] += r * g;
            }
        }
        if (COLOR) {
            const float *cp = a.color_at(slot);
#pragma unroll
            for (int c = 0; c < 3; ++c) cacc[c] += r * __ldg(cp + c * a.color_stride(slot));
        }
    }
}

// the normal (camera frame, unit) and colour in [0, 1] from the trilinear sums; unchanged where nothing is valid
template <bool NORMAL, bool COLOR>
__device__ __forceinline__ void rc_shade_finish(const RcFrame &fr, float sum_r, const float nacc[3], const float cacc[3], float nrm[3], float col[3]) {
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

// depth and vertex (camera frame) of the hit at ti; p = the world point
__device__ __forceinline__ void rc_hit_point(const RcBatch &bp, const RcFrame &fr, const float o[3], const float d[3], float ti, float p[3],
                                             float &depth, float vert[3]) {
    depth = ti * bp.depth_scale;
#pragma unroll
    for (int r = 0; r < 3; ++r) p[r] = o[r] + ti * d[r];
#pragma unroll
    for (int r = 0; r < 3; ++r) vert[r] = ((fr.E[4 * r] * p[0] + fr.E[4 * r + 1] * p[1]) + fr.E[4 * r + 2] * p[2]) + fr.E[4 * r + 3];
}

// pixel of thread: a warp covers an 8 x 4 tile; false outside the image
__device__ __forceinline__ bool rc_pixel(const RcBatch &bp, int &x, int &y) {
    const int tiles_x = (bp.W + kRcTileW - 1) / kRcTileW;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    x = (blockIdx.x % tiles_x) * kRcTileW + (warp & 3) * 8 + (lane & 7);
    y = (blockIdx.x / tiles_x) * kRcTileH + (warp >> 2) * 4 + (lane >> 3);
    return x < bp.W && y < bp.H;
}

template <bool NORMAL, bool COLOR>
__device__ __forceinline__ void rc_store(int64_t pix, float depth, const float vert[3], const float nrm[3], const float col[3], float *__restrict__ out_depth,
                                         float *__restrict__ out_vertex, float *__restrict__ out_normal, float *__restrict__ out_color) {
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

template <bool TENSOR, bool NORMAL, bool COLOR>
__global__ void __launch_bounds__(256, 1) raycast_kernel(const VolView v, const __grid_constant__ RcBatch bp, float *__restrict__ out_depth,
                                                      float *__restrict__ out_vertex, float *__restrict__ out_normal, float *__restrict__ out_color) {
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
        float o[3], d[3];
        rc_ray(bp, fr, x, y, o, d);
        float t_prev = t, tsdf_prev = -1.0f, ts = 1.0f;
        int bz_next;
        const RcBoxVol<TENSOR> a{v, bp};
        const bool hit = rc_march<TENSOR>(a, bp, o, d, t_max, t, t_prev, tsdf_prev, ts, bz_next);
        if (hit) {
            float p[3];
            rc_hit_point(bp, fr, o, d, rc_hit_t(t, t_prev, tsdf_prev, ts), p, depth, vert);
            if (NORMAL || COLOR) {
                int base[3];
                float xv[3];
                rc_trilinear_base<TENSOR>(bp, p, base, xv);
                float sum_r = 0.f, nacc[3] = {0.f, 0.f, 0.f}, cacc[3] = {0.f, 0.f, 0.f};
                rc_trilinear_sums<NORMAL, COLOR>(a, base, xv, sum_r, nacc, cacc);
                rc_shade_finish<NORMAL, COLOR>(fr, sum_r, nacc, cacc, nrm, col);
            }
        }
    }
    rc_store<NORMAL, COLOR>(pix, depth, vert, nrm, col, out_depth, out_vertex, out_normal, out_color);
}

// ------------------------------------------------------------------ z-slabs (ShardedTSDF.raycast)
// A slab [z0, z1) of a z-sharded legacy volume marches with the geometry of the whole grid (origin, brick counts), so
// every slab computes the same floats for a sample as the single box does.  A sample belongs to the slab holding its
// brick layer (layers below the grid to slab 0, above it to the last); along a ray the layer never decreases in the
// direction of d_z, so a ray visits its owners in z order and N rounds finish every ray.
constexpr int kRcMaxSlabs = 64;
constexpr int kRcMarching = 1, kRcHit = 2, kRcMiss = 3;   // low 2 bits of a ray state's code; the owner slab is code >> 2

struct RcSlabs {
    int n, me;                       // slab count, this slab
    int z0, z1;                      // this slab's global planes
    int lo_bz, hi_bz;                // brick layers whose samples this slab marches (open at the ends of the grid)
    int zb[kRcMaxSlabs + 1];         // global plane bounds of every slab
    int nxy;                         // voxels per plane
    const float2 *halo_lo_tw, *halo_hi_tw;          // plane z0 - 1 / planes z1, z1 + 1: [planes][nx][ny] {tsdf, weight}
    const float *halo_lo_rgb, *halo_hi_rgb;         // their colour [planes][nx][ny][3] (colour volumes)
    const uint8_t *halo_lo_flags, *halo_hi_flags;   // brick flags of layer z0 / 8 - 1 / z1 / 8: [nby][nbx]
};

__device__ __forceinline__ int rc_slab_of(const RcSlabs &s, int bz) {
    int k = 0;
    while (k + 1 < s.n && bz >= (s.zb[k + 1] >> 3)) ++k;
    return k;
}

// Reads of a slab and its halo: the march reads only samples of its own brick layers; the shading of a hit whose
// trilinear base plane the slab owns reads planes z0 - 1 ... z1 + 1.  A slot >= 0 is the slab's own, -1 - h the
// halo voxel h (h < nxy: plane z0 - 1, else planes z1, z1 + 1).
struct RcSlabVol {
    const VolView &v;
    const RcBatch &bp;
    const RcSlabs &s;
    __device__ __forceinline__ bool foreign(int bz) const { return bz < s.lo_bz || bz >= s.hi_bz; }
    __device__ __forceinline__ bool block_alloc(int bx, int by, int bz) const {
        return __ldg(v.flags + ((int64_t)(bz - (s.z0 >> 3)) * v.nby + by) * v.nbx + bx) & 1u;
    }
    __device__ __forceinline__ float2 voxel(int X, int Y, int Z) const { return __ldg(v.vox + voxel_slot(v, X, Y, Z - s.z0)); }
    __device__ __forceinline__ bool voxel_alloc(int X, int Y, int Z) const {
        if ((unsigned)X >= (unsigned)bp.n[0] || (unsigned)Y >= (unsigned)bp.n[1] || (unsigned)Z >= (unsigned)bp.n[2]) return false;
        const uint8_t *fl = Z < s.z0 ? s.halo_lo_flags : Z >= s.z1 ? s.halo_hi_flags : v.flags + (int64_t)((Z - s.z0) >> 3) * v.nby * v.nbx;
        return __ldg(fl + (Y >> 3) * v.nbx + (X >> 3)) & 1u;
    }
    __device__ __forceinline__ int64_t slot(int X, int Y, int Z) const {
        if (Z < s.z0) return -1 - (int64_t)(X * v.ny + Y);
        if (Z >= s.z1) return -1 - ((int64_t)(Z - s.z1 + 1) * s.nxy + X * v.ny + Y);
        return voxel_slot(v, X, Y, Z - s.z0);
    }
    __device__ __forceinline__ float2 voxel_at(int64_t slot) const {
        if (slot >= 0) return __ldg(v.vox + slot);
        const int64_t h = -1 - slot;
        return h < s.nxy ? __ldg(s.halo_lo_tw + h) : __ldg(s.halo_hi_tw + (h - s.nxy));
    }
    __device__ __forceinline__ const float *color_at(int64_t slot) const {
        if (slot >= 0) return v.color + slot + (slot / kBrickVox) * (2 * kBrickVox);
        const int64_t h = -1 - slot;
        return h < s.nxy ? s.halo_lo_rgb + 3 * h : s.halo_hi_rgb + 3 * (h - s.nxy);
    }
    __device__ __forceinline__ int color_stride(int64_t slot) const { return slot >= 0 ? kBrickVox : 1; }
};

// One round of the segment march: every ray this slab owns marches until it hits, leaves [depth_min, depth_max) or
// reaches a sample of another slab, and its state {t | ti, t_prev, ts, owner << 2 | status} is written; rays of other
// slabs are written as 0, so the sum of all slabs' states is the next round's state.  first: the state is not read;
// every slab computes each ray's first owner itself.  *handed counts the rays handed to another slab.
__global__ void __launch_bounds__(256) raycast_segment_kernel(const VolView v, const __grid_constant__ RcBatch bp, const __grid_constant__ RcSlabs s,
                                                              int first, int4 *__restrict__ state, int *__restrict__ handed) {
    int x, y;
    if (!rc_pixel(bp, x, y)) return;
    const int f = blockIdx.y;
    const RcFrame &fr = bp.fr[f];
    const int64_t pix = ((int64_t)f * bp.H + y) * bp.W + x;
    float o[3], d[3];
    rc_ray(bp, fr, x, y, o, d);
    float t, t_prev, ts;
    int owner, status;
    if (first) {
        t = t_prev = bp.depth_min;
        ts = 1.0f;
        const float q = (o[2] + t * d[2]) - bp.org[2];          // the march's first sample (rc_march)
        owner = rc_slab_of(s, (int)floorf(q / bp.bl) - bp.b0[2]);
        status = t < bp.depth_max ? kRcMarching : kRcMiss;
    } else {
        const int4 w = state[pix];
        t = __int_as_float(w.x); t_prev = __int_as_float(w.y); ts = __int_as_float(w.z);
        owner = w.w >> 2; status = w.w & 3;
    }
    const bool mine = owner == s.me;
    bool hand = false;
    if (mine && status == kRcMarching) {
        float tsdf_prev = -1.0f;
        int bz_next;
        const RcSlabVol a{v, bp, s};
        if (rc_march<false>(a, bp, o, d, bp.depth_max, t, t_prev, tsdf_prev, ts, bz_next)) {
            status = kRcHit;
            t = rc_hit_t(t, t_prev, tsdf_prev, ts);
        } else if (t < bp.depth_max) {
            owner = rc_slab_of(s, bz_next);
            hand = true;
        } else {
            status = kRcMiss;
        }
    }
    const unsigned m = __ballot_sync(__activemask(), hand);
    if (hand && (threadIdx.x & 31) == __ffs(m) - 1) atomicAdd(handed, __popc(m));
    state[pix] = mine ? make_int4(__float_as_int(t), __float_as_int(t_prev), __float_as_int(ts), owner << 2 | status) : make_int4(0, 0, 0, 0);
}

// Shading of the finished rays whose hit has its trilinear base plane in this slab (the others are written as 0):
// depth, vertex, normal and colour exactly as raycast_kernel computes them from the same ti.
template <bool NORMAL, bool COLOR>
__global__ void __launch_bounds__(256) raycast_shade_kernel(const VolView v, const __grid_constant__ RcBatch bp, const __grid_constant__ RcSlabs s,
                                                            const int4 *__restrict__ state, float *__restrict__ out_depth, float *__restrict__ out_vertex,
                                                            float *__restrict__ out_normal, float *__restrict__ out_color) {
    int x, y;
    if (!rc_pixel(bp, x, y)) return;
    const int f = blockIdx.y;
    const RcFrame &fr = bp.fr[f];
    const int64_t pix = ((int64_t)f * bp.H + y) * bp.W + x;
    float depth = 0.f, vert[3] = {0.f, 0.f, 0.f}, nrm[3] = {0.f, 0.f, 0.f}, col[3] = {0.f, 0.f, 0.f};
    const int4 w = state[pix];
    if ((w.w & 3) == kRcHit) {
        float o[3], d[3], p[3], dh, vh[3];
        rc_ray(bp, fr, x, y, o, d);
        rc_hit_point(bp, fr, o, d, __int_as_float(w.x), p, dh, vh);
        int base[3];
        float xv[3];
        rc_trilinear_base<false>(bp, p, base, xv);
        if (rc_slab_of(s, base[2] >> 3) == s.me) {
            depth = dh;
#pragma unroll
            for (int r = 0; r < 3; ++r) vert[r] = vh[r];
            if (NORMAL || COLOR) {
                const RcSlabVol a{v, bp, s};
                float sum_r = 0.f, nacc[3] = {0.f, 0.f, 0.f}, cacc[3] = {0.f, 0.f, 0.f};
                rc_trilinear_sums<NORMAL, COLOR>(a, base, xv, sum_r, nacc, cacc);
                rc_shade_finish<NORMAL, COLOR>(fr, sum_r, nacc, cacc, nrm, col);
            }
        }
    }
    rc_store<NORMAL, COLOR>(pix, depth, vert, nrm, col, out_depth, out_vertex, out_normal, out_color);
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

// the legacy batch of a slab: the geometry of the whole grid, z_total = h_slab_z[n_slabs] planes
static void rc_slab_batch(RcBatch &bp, const VolView &v, int z_total, int H, int W, const double *h_K, float depth_scale, float depth_min,
                          float depth_max, float weight_threshold) {
    rc_common(bp, v, H, W, h_K, depth_scale, depth_min, depth_max, weight_threshold);
    bp.n[2] = z_total;
    bp.trunc = v.trunc;
    bp.bl = v.vl * (float)kBrick;
    bp.half = 0.5f;
    bp.org[0] = (float)v.ox; bp.org[1] = (float)v.oy; bp.org[2] = (float)v.oz;
    for (int r = 0; r < 3; ++r) { bp.b0[r] = 0; bp.nb[r] = bp.n[r] / kBrick; }
    bp.alloc_bits = nullptr; bp.range = nullptr;
}

// checks shared by the slab entry points; fills the slab description (without halos)
static int rc_slab_check(const char *name, const bslam_volume *vol, int n_slabs, const int *h_slab_z, int F, int H, int W, const double *h_K,
                         const double *h_extrinsics, RcSlabs &s) {
    BSLAM_CHECK_ARG(F >= 0 && H > 0 && W > 0, "[%s] Unsupported image format. (F=%d H=%d W=%d)", name, F, H, W);
    BSLAM_CHECK_ARG(vol && h_K && h_slab_z && (h_extrinsics || F == 0), "%s: NULL argument", name);
    BSLAM_CHECK_ARG(n_slabs >= 1 && n_slabs <= kRcMaxSlabs, "%s: 1..%d slabs (got %d)", name, kRcMaxSlabs, n_slabs);
    const VolView &v = vol->v;
    BSLAM_CHECK_ARG(v.zs == 1, "%s: contiguous slabs only (re-shard an interleaved box first)", name);
    BSLAM_CHECK_ARG(v.nx % kBrick == 0 && v.ny % kBrick == 0 && v.nz % kBrick == 0 && v.gz0 % kBrick == 0,
                    "%s: the slab must consist of whole %d^3 bricks at a brick-aligned z", name, kBrick);
    BSLAM_CHECK_ARG(h_slab_z[0] == 0, "%s: the slab bounds must start at 0", name);
    s.n = n_slabs; s.me = -1;
    for (int k = 0; k < n_slabs; ++k) {
        BSLAM_CHECK_ARG(h_slab_z[k + 1] > h_slab_z[k] && h_slab_z[k + 1] % kBrick == 0, "%s: slab bounds must increase in whole bricks", name);
        if (h_slab_z[k] == v.gz0 && h_slab_z[k + 1] == v.gz0 + v.nz) s.me = k;
    }
    for (int k = 0; k <= n_slabs; ++k) s.zb[k] = h_slab_z[k];
    BSLAM_CHECK_ARG(s.me >= 0, "%s: the volume's planes [%d, %d) are not one of the slab bounds", name, v.gz0, v.gz0 + v.nz);
    BSLAM_CHECK_ARG(vol->z_total == 0 || vol->z_total == h_slab_z[n_slabs], "%s: the volume's z_total (%d) is not the bounds' %d planes", name,
                    vol->z_total, h_slab_z[n_slabs]);
    s.z0 = v.gz0; s.z1 = v.gz0 + v.nz;
    s.lo_bz = s.me == 0 ? INT_MIN : s.z0 / kBrick;
    s.hi_bz = s.me == n_slabs - 1 ? INT_MAX : s.z1 / kBrick;
    s.nxy = v.nx * v.ny;
    s.halo_lo_tw = s.halo_hi_tw = nullptr; s.halo_lo_rgb = s.halo_hi_rgb = nullptr; s.halo_lo_flags = s.halo_hi_flags = nullptr;
    return BSLAM_OK;
}

// packed halo of `planes` planes: {tsdf, weight} planes, colour planes (colour volumes), brick flags of one layer
static void rc_unpack_halo(const bslam_volume *vol, const void *halo, int planes, const float2 *&tw, const float *&rgb, const uint8_t *&flags) {
    const VolView &v = vol->v;
    const size_t nxy = (size_t)v.nx * v.ny;
    const char *p = (const char *)halo;
    tw = (const float2 *)p;
    p += planes * nxy * sizeof(float2);
    rgb = vol->with_color ? (const float *)p : nullptr;
    if (vol->with_color) p += planes * nxy * 3 * sizeof(float);
    flags = (const uint8_t *)p;
}

template <bool NORMAL, bool COLOR>
static void rc_shade_launch(dim3 grid, cudaStream_t st, const VolView &v, const RcBatch &bp, const RcSlabs &s, const int4 *state, float *depth,
                            float *vertex, float *normal, float *color) {
    raycast_shade_kernel<NORMAL, COLOR><<<grid, 256, 0, st>>>(v, bp, s, state, depth, vertex, normal, color);
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

size_t bslam_tsdf_raycast_halo_bytes(const bslam_volume *vol, int planes) {
    if (!vol || planes < 1) return 0;
    const size_t nxy = (size_t)vol->v.nx * vol->v.ny;
    return planes * nxy * (sizeof(float2) + (vol->with_color ? 3 * sizeof(float) : 0)) + (size_t)vol->v.nbx * vol->v.nby;
}

int bslam_tsdf_raycast_segment(bslam_volume *vol, int n_slabs, const int *h_slab_z, int first, int F, int H, int W, const double *h_K,
                               const double *h_extrinsics, float depth_min, float depth_max, float weight_threshold, int32_t *d_state,
                               bslam_stream_t stream) {
    static thread_local RcSlabs s;
    if (rc_slab_check("bslam_tsdf_raycast_segment", vol, n_slabs, h_slab_z, F, H, W, h_K, h_extrinsics, s) != BSLAM_OK) return BSLAM_E_ARG;
    BSLAM_CHECK_ARG(depth_min >= 0.f && isfinite(depth_min) && isfinite(depth_max) && weight_threshold >= 0.f,
                    "bslam_tsdf_raycast_segment: depth_min >= 0, depth_max finite and weight_threshold >= 0");
    BSLAM_CHECK_ARG(d_state || F == 0, "bslam_tsdf_raycast_segment: NULL argument");
    if (F == 0) return BSLAM_OK;
    BSLAM_DEVICE_GUARD(vol->device);
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local RcBatch bp;
    rc_slab_batch(bp, vol->v, h_slab_z[n_slabs], H, W, h_K, 1.0f, depth_min, depth_max, weight_threshold);
    const int64_t n_pix = (int64_t)W * H;
    int *handed = d_state + 4 * (int64_t)F * n_pix;
    BSLAM_CUDA(cudaMemsetAsync(handed, 0, sizeof(int), st));
    for (int f0 = 0; f0 < F; f0 += kRcMaxFrames) {
        bp.F = F - f0 < kRcMaxFrames ? F - f0 : kRcMaxFrames;
        for (int f = 0; f < bp.F; ++f) rc_set_frame(bp.fr[f], h_extrinsics + (size_t)(f0 + f) * 16, false);
        const dim3 grid(((W + kRcTileW - 1) / kRcTileW) * ((H + kRcTileH - 1) / kRcTileH), bp.F);
        raycast_segment_kernel<<<grid, 256, 0, st>>>(vol->v, bp, s, first, (int4 *)d_state + f0 * n_pix, handed);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

int bslam_tsdf_raycast_shade(bslam_volume *vol, int n_slabs, const int *h_slab_z, const void *d_halo_lo, const void *d_halo_hi, int F, int H, int W,
                             const double *h_K, const double *h_extrinsics, float depth_scale, const int32_t *d_state, float *d_depth, float *d_vertex,
                             float *d_normal, float *d_color, bslam_stream_t stream) {
    static thread_local RcSlabs s;
    if (rc_slab_check("bslam_tsdf_raycast_shade", vol, n_slabs, h_slab_z, F, H, W, h_K, h_extrinsics, s) != BSLAM_OK) return BSLAM_E_ARG;
    BSLAM_CHECK_ARG(depth_scale > 0.f, "bslam_tsdf_raycast_shade: depth_scale must be > 0");
    BSLAM_CHECK_ARG((d_state && d_depth) || F == 0, "bslam_tsdf_raycast_shade: NULL argument");
    BSLAM_CHECK_ARG(!(d_color && !vol->with_color), "[bslam_tsdf_raycast_shade] a colour map needs a colour volume");
    BSLAM_CHECK_ARG((d_halo_lo != nullptr) == (s.me > 0), "bslam_tsdf_raycast_shade: the halo below is required exactly when a slab lies below");
    BSLAM_CHECK_ARG((d_halo_hi != nullptr) == (s.me < n_slabs - 1), "bslam_tsdf_raycast_shade: the halo above is required exactly when a slab lies above");
    if (F == 0) return BSLAM_OK;
    if (d_halo_lo) rc_unpack_halo(vol, d_halo_lo, 1, s.halo_lo_tw, s.halo_lo_rgb, s.halo_lo_flags);
    if (d_halo_hi) rc_unpack_halo(vol, d_halo_hi, 2, s.halo_hi_tw, s.halo_hi_rgb, s.halo_hi_flags);
    BSLAM_DEVICE_GUARD(vol->device);
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local RcBatch bp;
    rc_slab_batch(bp, vol->v, h_slab_z[n_slabs], H, W, h_K, depth_scale, 0.0f, 0.0f, 0.0f);
    const int64_t n_pix = (int64_t)W * H;
    for (int f0 = 0; f0 < F; f0 += kRcMaxFrames) {
        bp.F = F - f0 < kRcMaxFrames ? F - f0 : kRcMaxFrames;
        for (int f = 0; f < bp.F; ++f) rc_set_frame(bp.fr[f], h_extrinsics + (size_t)(f0 + f) * 16, false);
        const dim3 grid(((W + kRcTileW - 1) / kRcTileW) * ((H + kRcTileH - 1) / kRcTileH), bp.F);
        const int64_t o = f0 * n_pix;
        const int4 *sp = (const int4 *)d_state + o;
        float *dp = d_depth + o, *vp = d_vertex ? d_vertex + 3 * o : nullptr, *np = d_normal ? d_normal + 3 * o : nullptr, *cp = d_color ? d_color + 3 * o : nullptr;
        if (np && cp) rc_shade_launch<true, true>(grid, st, vol->v, bp, s, sp, dp, vp, np, cp);
        else if (np) rc_shade_launch<true, false>(grid, st, vol->v, bp, s, sp, dp, vp, np, cp);
        else if (cp) rc_shade_launch<false, true>(grid, st, vol->v, bp, s, sp, dp, vp, np, cp);
        else rc_shade_launch<false, false>(grid, st, vol->v, bp, s, sp, dp, vp, np, cp);
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
