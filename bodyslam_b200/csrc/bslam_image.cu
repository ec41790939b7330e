// K1 (metric scaling + colorize), a4 (3DM depth scaling) and K2 (back-projection + SE(3))
// for sm_100a.  All three are pure HBM streaming: 128-bit loads/stores, grids sized in
// multiples of the SM count, no tensor cores (nothing here is a contraction).
//
// Semantics (checked against oracle/mdem.py and oracle/o3d_oracle.c):
//   K1  R/examples/depth_estimation/depth_map_scaling.py:12-45  (colorize)
//       + ZoeDepth infer_pil tail (R/src/depth_estimation/interface.py:61)
//   a4  N/3DM/slam_utils.py:212-220,231-233
//   K2  N/3DM/scaling_system.py:72-77, N/3DM/mapping_module.py:37,41
#include <math.h>

#include "bslam_common.cuh"

namespace bslam {

constexpr int kBins = 65536;

// per-image workspace: [hist u32 x 65536][index table u8 x 65536][stats]
struct ImgStats {
    double vmin, vmax;
    unsigned long long n_valid;
    unsigned int vmin_u, vmax_u; // min / max valid value (minmax path)
};
constexpr size_t kWsPerImage = kBins * 4 + kBins + 256;

__device__ __forceinline__ unsigned int *ws_hist(void *ws, int b) { return (unsigned int *)((char *)ws + (size_t)b * kWsPerImage); }
__device__ __forceinline__ uint8_t *ws_table(void *ws, int b) { return (uint8_t *)((char *)ws + (size_t)b * kWsPerImage + kBins * 4); }
__device__ __forceinline__ ImgStats *ws_stats(void *ws, int b) { return (ImgStats *)((char *)ws + (size_t)b * kWsPerImage + kBins * 4 + kBins); }

__device__ __forceinline__ unsigned int to_u16_sat(float m, float scale_mul) {
    // numpy: (metres * 256).astype(uint16) -- f32 multiply, truncation toward zero.
    // one saturating conversion (round toward zero; negative and NaN -> 0) and an integer clamp
    return min(__float2uint_rz(m * scale_mul), 65535u);
}

// ---------------------------------------------------------------- K1 pass A: scale + histogram
// Each block owns kPxPerBlock consecutive pixels of one image, keeps them in registers,
// histograms into a shared window anchored at the block minimum and flushes the non-empty bins.
constexpr int kHistThreads = 256;
constexpr int kPxPerThread = 16;
constexpr int kPxPerBlock = kHistThreads * kPxPerThread;
constexpr int kWindow = 4096;

// Equal values are combined before they reach the shared-memory atomics (<= 2 lanes per cycle and SM, so smooth images must
// not spend one atomic per pixel): a 4-pixel group whose pixels are equal adds once, and the equal groups of a warp that hold
// the same value are combined with match.any into one atomic per distinct value and warp.  The window is zeroed and
// flushed 16 bytes at a time.  The run-length merge and the group merge without match.any measured slower:
// profiles/r02_k1_hist_merge.md.
template <bool FROM_FLOAT>
__global__ void __launch_bounds__(kHistThreads) scale_hist_kernel(const float *__restrict__ depth_m, const uint16_t *__restrict__ u16_in,
                                                                   uint16_t *__restrict__ u16_out, int64_t n_per_image, float scale_mul,
                                                                   int has_invalid, unsigned int invalid_val, void *ws) {
    __shared__ __align__(16) unsigned int s_hist[kWindow];
    __shared__ unsigned int s_min;
    const int b = blockIdx.y;
    const int64_t start = (int64_t)blockIdx.x * kPxPerBlock;
    unsigned int *hist = ws_hist(ws, b);
    for (int i = threadIdx.x; i < kWindow / 4; i += kHistThreads) reinterpret_cast<uint4 *>(s_hist)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) s_min = 0xffffffffu;
    __syncthreads();

    unsigned int val[kPxPerThread];
    unsigned int tmin = 0xffffffffu;
    const int64_t img_off = (int64_t)b * n_per_image;
    // a value no pixel can hold when there is no invalid marker: one compare + select per pixel either way
    const unsigned int inv = has_invalid ? invalid_val : 0xfffffffeu;
    // thread t handles 4 groups of 4 consecutive pixels, groups strided by 1024 -> 16-byte accesses
    if (start + kPxPerBlock <= n_per_image && ((img_off + start) & 3) == 0) {
        // the whole block lies inside the image and its rows of 4 are 16-byte aligned: no per-group tests
        const int64_t q = img_off + start + threadIdx.x * 4;
#pragma unroll
        for (int g = 0; g < kPxPerThread / 4; ++g) {
            if (FROM_FLOAT) {
                const float4 d = *reinterpret_cast<const float4 *>(depth_m + q + g * (kHistThreads * 4));
                val[4 * g + 0] = to_u16_sat(d.x, scale_mul); val[4 * g + 1] = to_u16_sat(d.y, scale_mul);
                val[4 * g + 2] = to_u16_sat(d.z, scale_mul); val[4 * g + 3] = to_u16_sat(d.w, scale_mul);
                if (u16_out)
                    *reinterpret_cast<ushort4 *>(u16_out + q + g * (kHistThreads * 4)) =
                        make_ushort4((unsigned short)val[4 * g], (unsigned short)val[4 * g + 1], (unsigned short)val[4 * g + 2], (unsigned short)val[4 * g + 3]);
            } else {
                const ushort4 d = *reinterpret_cast<const ushort4 *>(u16_in + q + g * (kHistThreads * 4));
                val[4 * g + 0] = d.x; val[4 * g + 1] = d.y; val[4 * g + 2] = d.z; val[4 * g + 3] = d.w;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                unsigned int &x = val[4 * g + j];
                x = (x == inv) ? 0xffffffffu : x;
                tmin = min(tmin, x);
            }
        }
    } else {
#pragma unroll
    for (int g = 0; g < kPxPerThread / 4; ++g) {
        const int64_t p = start + (int64_t)g * (kHistThreads * 4) + threadIdx.x * 4;
        if (p + 3 < n_per_image && ((img_off + p) & 3) == 0) {
            if (FROM_FLOAT) {
                const float4 d = *reinterpret_cast<const float4 *>(depth_m + img_off + p);
                val[4 * g + 0] = to_u16_sat(d.x, scale_mul); val[4 * g + 1] = to_u16_sat(d.y, scale_mul);
                val[4 * g + 2] = to_u16_sat(d.z, scale_mul); val[4 * g + 3] = to_u16_sat(d.w, scale_mul);
                if (u16_out) {
                    ushort4 o = make_ushort4((unsigned short)val[4 * g], (unsigned short)val[4 * g + 1],
                                             (unsigned short)val[4 * g + 2], (unsigned short)val[4 * g + 3]);
                    *reinterpret_cast<ushort4 *>(u16_out + img_off + p) = o;
                }
            } else {
                const ushort4 d = *reinterpret_cast<const ushort4 *>(u16_in + img_off + p);
                val[4 * g + 0] = d.x; val[4 * g + 1] = d.y; val[4 * g + 2] = d.z; val[4 * g + 3] = d.w;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                unsigned int x = 0xffffffffu; // out of range marker
                if (p + j < n_per_image) {
                    if (FROM_FLOAT) {
                        x = to_u16_sat(depth_m[img_off + p + j], scale_mul);
                        if (u16_out) u16_out[img_off + p + j] = (unsigned short)x;
                    } else {
                        x = u16_in[img_off + p + j];
                    }
                }
                val[4 * g + j] = x;
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            unsigned int &x = val[4 * g + j];
            x = (x == inv) ? 0xffffffffu : x;
            tmin = min(tmin, x);
        }
    }
    }
    for (int o = 16; o; o >>= 1) tmin = min(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
    if ((threadIdx.x & 31) == 0 && tmin != 0xffffffffu) atomicMin(&s_min, tmin);
    __syncthreads();
    const unsigned int base = s_min;
    if (base == 0xffffffffu) return; // no valid pixel in this block
    // the marker 0xffffffff never lands in the window (base <= 65535), so only the global path tests for it
    auto add = [&](unsigned int x, unsigned int n) {
        const unsigned int rel = x - base;
        if (rel < kWindow) atomicAdd(&s_hist[rel], n);
        else if (x != 0xffffffffu) atomicAdd(&hist[x], n);
    };
    // the increment of the per-pixel path is kept opaque: with a literal 1 ptxas emits ATOMS.POPC.INC, which matches addresses
    // across the warp first and runs at half the rate of ATOMS.ADD when the addresses are spread (white noise: 1.07 vs 0.50 ms)
    // (n_per_image >= 1 here, so this is 1 -- but ptxas cannot know; an empty asm barrier is not enough, it leaves no PTX behind)
    const unsigned int one = (unsigned int)min(n_per_image, (int64_t)1);
#pragma unroll
    for (int g = 0; g < kPxPerThread / 4; ++g) {
        const unsigned int a = val[4 * g], c1 = val[4 * g + 1], c2 = val[4 * g + 2], c3 = val[4 * g + 3];
        const bool uni = (a == c1) & (c1 == c2) & (c2 == c3);
        // lanes whose group is equal AND holds the same value elect their lowest lane; a mixed group matches nobody
        const unsigned int peers = __match_any_sync(0xffffffffu, uni ? a : (0xffff0000u | (threadIdx.x & 31)));
        if (uni) {
            if ((threadIdx.x & 31) == __ffs(peers) - 1) add(a, 4u * __popc(peers));
            continue;
        }
        add(a, one); add(c1, one); add(c2, one); add(c3, one);
    }
    __syncthreads();
    // flush: 16-byte reads find the (on depth images: few) occupied bins.  Where a warp's 128-bin segment is densely
    // occupied it is re-read word-interleaved, so that one global reduction covers 32 consecutive bins = 4 sectors; with
    // the 16-byte ownership every reduction would touch 16 sectors, 2 bins each, and the L2 atomic units take a dense
    // window (white noise) at a quarter of the rate: 1.07 instead of 0.50 ms per 64 x 1080p.
    const int lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < kWindow / 4; i += kHistThreads) {   // same trip count for every thread
        const uint4 c = reinterpret_cast<const uint4 *>(s_hist)[i];
        const bool nz = (c.x | c.y | c.z | c.w) != 0;
        if (__popc(__ballot_sync(0xffffffffu, nz)) > 8) {
            const int seg = 4 * (i - lane);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const unsigned int w = s_hist[seg + 32 * k + lane];
                if (w) atomicAdd(&hist[base + seg + 32 * k + lane], w);
            }
        } else if (nz) {
            if (c.x) atomicAdd(&hist[base + 4 * i + 0], c.x);
            if (c.y) atomicAdd(&hist[base + 4 * i + 1], c.y);
            if (c.z) atomicAdd(&hist[base + 4 * i + 2], c.z);
            if (c.w) atomicAdd(&hist[base + 4 * i + 3], c.w);
        }
    }
}

// ---------------------------------------------------------------- K1 pass B: order statistics + index table
__device__ double numpy_lerp(double a, double b, double t) {
    // numpy.lib._function_base_impl._lerp
    const double diff = b - a;
    double r = a + diff * t;
    if (t >= 0.5) r = b - diff * (1.0 - t);
    return r;
}

// mode 0: percentile colorize table; mode 1: min-max uint8 table; mode 2: median only
// grid = (images, kTableSlices): every CTA of an image recomputes the image's order statistics
// from the 256 KB histogram (L2-resident; each thread keeps its 64 bins in registers) and then
// builds only its own 1/kTableSlices of the 65 536-entry index table -- the 65 536 f64 divisions
// per image are the long pole, so they are spread over kTableSlices SMs.
constexpr int kTableSlices = 8;

// phase 0: statistics + table in one launch (every slice CTA recomputes the statistics);  phase 1: statistics only
// (grid (images, 1)) -> ImgStats;  phase 2: table only (grid (images, kTableSlices)) from the stored vmin / vmax.
// The colorize / min-max paths launch phase 1 then phase 2: with phase 0 all 8 slice CTAs of an image re-read its
// 256 KB histogram (134 MB of L2 traffic per 64 images, most of the pass's 49 us).
__global__ void __launch_bounds__(1024) stats_table_kernel(void *ws, double p_lo, double p_hi, const double *vmin_vmax_override /*device*/,
                                                           double *vmin_vmax_out, double *median_out, int mode,
                                                           const uint8_t *table_override, int phase) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_before[4];
    __shared__ int s_owner[4];
    __shared__ double s_vals[4];
    __shared__ unsigned int s_mm[2];
    const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, wid = t >> 5;
    const int slice = blockIdx.y, n_slices = gridDim.y;
    const int i_begin = (int)((int64_t)kBins * slice / n_slices), i_end = (int)((int64_t)kBins * (slice + 1) / n_slices);
    const unsigned int *hist = ws_hist(ws, b);
    uint8_t *table = ws_table(ws, b);
    ImgStats *st = ws_stats(ws, b);
    if (table_override) { // value_transform path: the host supplies the table
        if (phase != 1)
            for (int i = i_begin + t; i < i_end; i += 1024) table[i] = table_override[(size_t)b * kBins + i];
        return;
    }
    if (phase == 2) {     // table only: the statistics were stored by the phase-1 launch
        if (t == 0) {
            s_vals[0] = st->vmin; s_vals[1] = st->vmax;
            if (mode == 1) { s_vals[0] = (double)st->vmin_u; s_vals[1] = (double)st->vmax_u; }
        }
        __syncthreads();
    }
    if (phase != 2) {
    constexpr int kPer = kBins / 1024; // 64 consecutive bins per thread, fetched as 16-byte words
    unsigned long long local = 0;
    unsigned int lmin = 0xffffffffu, lmax = 0;
#pragma unroll 4
    for (int i = 0; i < kPer / 4; ++i) {
        const uint4 c4 = reinterpret_cast<const uint4 *>(hist + t * kPer)[i];
        const unsigned int c[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            local += c[j];
            if (c[j]) { lmin = min(lmin, (unsigned int)(t * kPer + 4 * i + j)); lmax = max(lmax, (unsigned int)(t * kPer + 4 * i + j)); }
        }
    }
    if (t == 0) { s_mm[0] = 0xffffffffu; s_mm[1] = 0; }
    // inclusive scan of the 1024 partial sums: warp shuffles, then the 32 warp totals
    unsigned long long inc = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        lmin = min(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    }
    if (lane == 0 && lmin != 0xffffffffu) { atomicMin(&s_mm[0], lmin); atomicMax(&s_mm[1], lmax); }
    if (wid == 0) {
        const unsigned long long w = s_warp[lane];
        unsigned long long winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long up = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += up;
        }
        s_warp[lane] = winc;   // inclusive over warps
    }
    __syncthreads();
    const unsigned long long n = s_warp[31];
    const unsigned long long before = (wid ? s_warp[wid - 1] : 0ull) + inc - local; // exclusive prefix of this thread's bins
    // wanted sorted positions: floor((n-1)*q) and +1 for both quantiles (and the medians).  The thread
    // whose 64 bins hold a wanted position publishes itself; warp j then finds position j's bin with
    // two coalesced loads per lane and a warp scan (a serial walk over the 64 bins costs 64 L2 round trips)
    unsigned long long want[4] = {0, 0, 0, 0};
    if (n > 0) {
        double q[2] = {p_lo / 100.0, p_hi / 100.0};
        if (mode == 2) { q[0] = 0.5; q[1] = 0.5; }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const double virt = (double)(n - 1) * q[k];
            const unsigned long long i0 = (unsigned long long)floor(virt);
            want[2 * k] = i0;
            want[2 * k + 1] = (i0 + 1 > n - 1) ? n - 1 : i0 + 1;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (want[j] >= before && want[j] < before + local) { s_owner[j] = t; s_before[j] = before; }
    }
    __syncthreads();
    if (n > 0 && wid < 4) {
        const int owner = s_owner[wid];
        const unsigned long long rel = want[wid] - s_before[wid];      // 0 <= rel < the owner's 64-bin total
        const unsigned int c0 = hist[owner * kPer + lane], c1 = hist[owner * kPer + 32 + lane];
        unsigned long long a0 = c0, a1 = c1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u0 = __shfl_up_sync(0xffffffffu, a0, o), u1 = __shfl_up_sync(0xffffffffu, a1, o);
            if (lane >= o) { a0 += u0; a1 += u1; }
        }
        a1 += __shfl_sync(0xffffffffu, a0, 31);
        const unsigned int m0 = __ballot_sync(0xffffffffu, a0 > rel), m1 = __ballot_sync(0xffffffffu, a1 > rel);
        if (lane == 0) s_vals[wid] = (double)(owner * kPer + (m0 ? __ffs(m0) - 1 : 32 + __ffs(m1) - 1));
    }
    __syncthreads();
    if (t == 0) {
        double vmin = 0.0, vmax = 0.0;
        if (n > 0) {
            if (mode == 2) {
                // numpy median: mean of the two middle elements (they coincide for odd n)
                const bool odd = (n & 1ull) != 0;
                vmin = vmax = odd ? s_vals[0] : (s_vals[0] + s_vals[1]) / 2.0;
            } else {
                const double v0 = (double)(n - 1) * (p_lo / 100.0), v1 = (double)(n - 1) * (p_hi / 100.0);
                vmin = numpy_lerp(s_vals[0], s_vals[1], v0 - floor(v0));
                vmax = numpy_lerp(s_vals[2], s_vals[3], v1 - floor(v1));
            }
        }
        if (mode == 1) { vmin = (double)s_mm[0]; vmax = (double)s_mm[1]; }
        if (vmin_vmax_override) {
            const double a = vmin_vmax_override[2 * b], c = vmin_vmax_override[2 * b + 1];
            if (a == a) vmin = a;
            if (c == c) vmax = c;
        }
        if (slice == 0) {
            st->vmin = vmin; st->vmax = vmax; st->n_valid = n; st->vmin_u = s_mm[0]; st->vmax_u = s_mm[1];
            if (vmin_vmax_out) { vmin_vmax_out[2 * b] = vmin; vmin_vmax_out[2 * b + 1] = vmax; }
            if (median_out) median_out[b] = vmin;
        }
        s_vals[0] = vmin; s_vals[1] = vmax;
    }
    __syncthreads();
    }   // phase != 2
    if (mode == 2 || phase == 1) return;
    const double vmin = s_vals[0], vmax = s_vals[1];
    for (int i = i_begin + t; i < i_end; i += 1024) {
        unsigned int idx;
        if (mode == 0) {
            // colorize: x = (value - vmin)/(vmax - vmin) (f64), matplotlib: trunc(x*256) with
            // x<0 -> under (row 0), x*256 == 256 -> 255, > 255 -> over (row 255)
            double x = (vmin != vmax) ? ((double)i - vmin) / (vmax - vmin) : (double)i * 0.0;
            x *= 256.0;
            if (x < 0.0) idx = 0;
            else if (x >= 256.0) idx = 255;
            else idx = (unsigned int)x;
        } else {
            // np.uint8(255 * (d - min) / (max - min))
            const double x = 255.0 * ((double)i - vmin) / (vmax - vmin);
            idx = (x >= 0.0 && x < 256.0) ? (unsigned int)x : 0u; // values outside [min,max] never occur
        }
        table[i] = (uint8_t)idx;
    }
}

// ---------------------------------------------------------------- K1 pass C: LUT application
template <int OUT_CH> // 4: RGBA (colorize), 3: 3-byte colour (+ gray) for the min-max path
__global__ void __launch_bounds__(256) apply_table_kernel(const uint16_t *__restrict__ u16, int64_t n_per_image, const uint8_t *__restrict__ lut,
                                                          int has_invalid, unsigned int invalid_val, uint32_t bg, uint8_t *__restrict__ out,
                                                          uint8_t *__restrict__ gray, void *ws) {
    __shared__ uint32_t s_lut[256];
    const int b = blockIdx.y;
    if (lut) {
        if (OUT_CH == 4) s_lut[threadIdx.x] = reinterpret_cast<const uint32_t *>(lut)[threadIdx.x];
        else s_lut[threadIdx.x] = lut[3 * threadIdx.x] | (lut[3 * threadIdx.x + 1] << 8) | (lut[3 * threadIdx.x + 2] << 16);
    }
    __syncthreads();
    const uint8_t *table = ws_table(ws, b);
    const int64_t img_off = (int64_t)b * n_per_image;
    for (int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; p < n_per_image; p += (int64_t)gridDim.x * blockDim.x * 4) {
        unsigned int v[4];
        const bool vec = (p + 3 < n_per_image) && (((img_off + p) & 3) == 0);
        if (vec) {
            const ushort4 d = *reinterpret_cast<const ushort4 *>(u16 + img_off + p);
            v[0] = d.x; v[1] = d.y; v[2] = d.z; v[3] = d.w;
        } else {
            for (int j = 0; j < 4; ++j) v[j] = (p + j < n_per_image) ? u16[img_off + p + j] : 0u;
        }
        uint32_t c[4]; uint8_t g[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            g[j] = __ldg(table + v[j]);
            c[j] = (has_invalid && v[j] == invalid_val) ? bg : s_lut[g[j]];
        }
        if (OUT_CH == 4) {
            if (vec) {
                *reinterpret_cast<uint4 *>(out + (img_off + p) * 4) = make_uint4(c[0], c[1], c[2], c[3]);
            } else {
                for (int j = 0; j < 4 && p + j < n_per_image; ++j) reinterpret_cast<uint32_t *>(out)[img_off + p + j] = c[j];
            }
        } else {
            for (int j = 0; j < 4 && p + j < n_per_image; ++j) {
                if (gray) gray[img_off + p + j] = g[j];
                if (out) {
                    uint8_t *o = out + (img_off + p + j) * 3;
                    o[0] = c[j] & 0xff; o[1] = (c[j] >> 8) & 0xff; o[2] = (c[j] >> 16) & 0xff;
                }
            }
        }
    }
}

__global__ void scale_u16_kernel(const float *__restrict__ in, int64_t n, float scale_mul, uint16_t *__restrict__ out) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
    for (int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; p < n; p += stride) {
        if (p + 3 < n) {
            const float4 d = *reinterpret_cast<const float4 *>(in + p);
            *reinterpret_cast<ushort4 *>(out + p) = make_ushort4((unsigned short)to_u16_sat(d.x, scale_mul), (unsigned short)to_u16_sat(d.y, scale_mul),
                                                                 (unsigned short)to_u16_sat(d.z, scale_mul), (unsigned short)to_u16_sat(d.w, scale_mul));
        } else {
            for (int j = 0; p + j < n; ++j) out[p + j] = (unsigned short)to_u16_sat(in[p + j], scale_mul);
        }
    }
}

// ---------------------------------------------------------------- a4: u16 -> metres
__device__ __forceinline__ float depth_cvt(unsigned int u, float scale, float trunc) {
    float p = (float)u / scale; // IEEE division, like Open3D's `*p /= (float)depth_scale`
    if (trunc > 0.0f && p >= trunc) p = 0.0f;
    return p;
}
__global__ void depth_from_u16_kernel(const uint16_t *__restrict__ in, int64_t n, float scale, float trunc, float *__restrict__ out) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
    for (int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; p < n; p += stride) {
        if (p + 3 < n) {
            const ushort4 d = *reinterpret_cast<const ushort4 *>(in + p);
            *reinterpret_cast<float4 *>(out + p) = make_float4(depth_cvt(d.x, scale, trunc), depth_cvt(d.y, scale, trunc),
                                                               depth_cvt(d.z, scale, trunc), depth_cvt(d.w, scale, trunc));
        } else {
            for (int j = 0; p + j < n; ++j) out[p + j] = depth_cvt(in[p + j], scale, trunc);
        }
    }
}

// ---------------------------------------------------------------- K2: back-projection + SE(3)
// Order-preserving compaction in three launches, none of which has a cross-CTA dependency:
//   bp_count_kernel : streams the depth once; a warp owns "warp tiles" of 256 visited pixels and
//                     writes each tile's valid count as an offset inside its CTA (32 tiles) plus
//                     the CTA total.
//   bp_scan_kernel  : one CTA turns the CTA totals into i64 bases and the per-image row counts.
//   bp_emit_kernel  : streams the depth again; every warp works alone (no block barrier): ballots
//                     rank its tile's valid pixels in row-major order, points are staged in the
//                     warp's 3 KB of shared memory and leave as fully coalesced 4-byte words.
// (A single-pass decoupled look-back version was measured first: its CTAs spend their life in four
//  barrier-separated global round trips -- ticket, depth, look-back, write -- and reached 1.1 TB/s.)
constexpr int kBpMaxImages = 64;       // poses per emit launch, passed by value -> constant bank
constexpr int kBpThreads = 256;
constexpr int kBpWarps = kBpThreads / 32;
constexpr int kBpTilePx = 256;         // visited pixels per warp tile (8 per lane)
constexpr int kBpTilesPerWarp = 4;
constexpr int kBpTilesPerCta = kBpWarps * kBpTilesPerWarp;   // 32

struct BackprojP {
    float fx, fy, cx, cy, inv_fx, inv_fy;
    int H, W, Hs, Ws, stride;
    int tiles_per_image, ctas_per_image;
    int img0, n_images;      // images of this launch (poses below are for img0 .. img0 + n_images - 1)
    float pose[kBpMaxImages][12];
};

struct BackprojWs {
    int *tile_off;           // [B * ctas_per_image * 32] exclusive offset of a tile inside its CTA
    int *cta_total;          // [B * ctas_per_image]
    long long *cta_base;     // [B * ctas_per_image] exclusive prefix over all CTAs (row index of the CTA's first point)
};

// visited pixel q of the strided grid -> (row v, column u) of the image: float estimate + exact correction
__device__ __forceinline__ void bp_pixel(const BackprojP &bp, float inv_ws, unsigned int q, int &u, int &v) {
    int r = (int)((float)q * inv_ws);
    int c = (int)q - r * bp.Ws;
    r += (c >= bp.Ws) - (c < 0);
    c = (int)q - r * bp.Ws;
    v = r * bp.stride; u = c * bp.stride;
}

__global__ void __launch_bounds__(kBpThreads) bp_count_kernel(const __grid_constant__ BackprojP bp, const float *__restrict__ depth, int valid_only,
                                                              BackprojWs ws) {
    __shared__ int s_cnt[kBpTilesPerCta];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned int img = blockIdx.x / (unsigned int)bp.ctas_per_image;
    const unsigned int cta_in_img = blockIdx.x - img * (unsigned int)bp.ctas_per_image;
    const unsigned int n_vis = (unsigned int)(bp.Hs * bp.Ws);
    const float *dimg = depth + (int64_t)img * bp.H * bp.W;
    const float inv_ws = 1.0f / (float)bp.Ws;
    const bool vec = (bp.stride == 1) && ((reinterpret_cast<uintptr_t>(dimg) & 15) == 0);
    int cnt[kBpTilesPerWarp];
#pragma unroll
    for (int t = 0; t < kBpTilesPerWarp; ++t) {
        const unsigned int tile = cta_in_img * kBpTilesPerCta + wid * kBpTilesPerWarp + t;
        const unsigned int q0 = tile * kBpTilePx;
        int c = 0;
        if (vec && q0 + kBpTilePx <= n_vis) {            // whole tile, contiguous pixels: two 16-byte loads per lane
            const float4 a = __ldg(reinterpret_cast<const float4 *>(dimg + q0) + lane);
            const float4 b = __ldg(reinterpret_cast<const float4 *>(dimg + q0) + 32 + lane);
            c = (a.x > 0.f) + (a.y > 0.f) + (a.z > 0.f) + (a.w > 0.f) + (b.x > 0.f) + (b.y > 0.f) + (b.z > 0.f) + (b.w > 0.f);
            if (!valid_only) c = 8;
        } else {
#pragma unroll
            for (int j = 0; j < kBpTilePx / 32; ++j) {
                const unsigned int q = q0 + j * 32 + lane;
                if (q < n_vis) {
                    int u, v;
                    bp_pixel(bp, inv_ws, q, u, v);
                    c += valid_only ? (__ldg(dimg + v * bp.W + u) > 0.f) : 1;
                }
            }
        }
        cnt[t] = __reduce_add_sync(0xffffffffu, c);
    }
    if (lane == 0) {
#pragma unroll
        for (int t = 0; t < kBpTilesPerWarp; ++t) s_cnt[wid * kBpTilesPerWarp + t] = cnt[t];
    }
    __syncthreads();
    if (wid == 0) {
        const int c = s_cnt[lane];
        int inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        ws.tile_off[(size_t)blockIdx.x * kBpTilesPerCta + lane] = inc - c;
        if (lane == 31) ws.cta_total[blockIdx.x] = inc;
    }
}

// exclusive i64 scan of the CTA totals (one CTA; n is a few thousand) + per-image row counts
__global__ void __launch_bounds__(1024) bp_scan_kernel(BackprojWs ws, int n_ctas, int ctas_per_image, int B, long long *counts /*[B+1]*/) {
    __shared__ long long s_warp[32];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n_ctas; base += 1024) {
        const int i = base + threadIdx.x;
        const long long c = (i < n_ctas) ? ws.cta_total[i] : 0;
        long long inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) s_warp[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            const long long w = s_warp[lane];
            long long winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long t = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o) winc += t;
            }
            s_warp[lane] = winc - w;     // exclusive over warps
        }
        __syncthreads();
        const long long carry = s_carry;
        if (i < n_ctas) ws.cta_base[i] = carry + s_warp[wid] + inc - c;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + s_warp[31] + inc;
        __syncthreads();
    }
    // rows of image k = base of the first CTA of image k+1 (or the grand total) - base of its own first CTA
    for (int k = threadIdx.x; k < B; k += 1024) {
        const long long lo = ws.cta_base[(size_t)k * ctas_per_image];
        const long long hi = (k + 1 < B) ? ws.cta_base[(size_t)(k + 1) * ctas_per_image] : s_carry;
        counts[k] = hi - lo;
    }
    if (threadIdx.x == 0) counts[B] = s_carry;
}

__device__ __forceinline__ float3 backproject_px(const BackprojP &bp, int img, int u, int v, float d) {
    // pixel_to_3d (scaling_system.py:72-77): x = (u - cx) * depth / fx ; then the rigid transform
    // (f32; the f64 reference value is matched to ~2 ulp either way: reciprocal multiply instead of two IEEE divisions)
    const float x = ((float)u - bp.cx) * d * bp.inv_fx;
    const float y = ((float)v - bp.cy) * d * bp.inv_fy;
    const float *M = bp.pose[img];
    float3 p;
    p.x = fmaf(M[0], x, fmaf(M[1], y, fmaf(M[2], d, M[3])));
    p.y = fmaf(M[4], x, fmaf(M[5], y, fmaf(M[6], d, M[7])));
    p.z = fmaf(M[8], x, fmaf(M[9], y, fmaf(M[10], d, M[11])));
    return p;
}

template <bool WITH_RGB>
__global__ void __launch_bounds__(kBpThreads) bp_emit_kernel(const __grid_constant__ BackprojP bp, const float *__restrict__ depth,
                                                             const uint8_t *__restrict__ rgb_u8, int valid_only,
                                                             float *__restrict__ xyz, float *__restrict__ rgb, int64_t capacity,
                                                             BackprojWs ws) {
    __shared__ float s_xyz[kBpWarps][kBpTilePx * 3];
    __shared__ float s_rgb[WITH_RGB ? kBpWarps : 1][WITH_RGB ? kBpTilePx * 3 : 1];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned int gcta = (unsigned int)bp.img0 * bp.ctas_per_image + blockIdx.x;   // CTA index of the count pass
    const unsigned int img = gcta / (unsigned int)bp.ctas_per_image;
    const unsigned int cta_in_img = gcta - img * (unsigned int)bp.ctas_per_image;
    const int img_local = (int)img - bp.img0;
    const unsigned int n_vis = (unsigned int)(bp.Hs * bp.Ws);
    const float *dimg = depth + (int64_t)img * bp.H * bp.W;
    const float inv_ws = 1.0f / (float)bp.Ws;
    const long long cta_base = ws.cta_base[gcta];
    float *sx = s_xyz[wid], *sc = s_rgb[WITH_RGB ? wid : 0];
#pragma unroll 1
    for (int t = 0; t < kBpTilesPerWarp; ++t) {
        const unsigned int tile_in_cta = wid * kBpTilesPerWarp + t;
        const unsigned int q0 = (cta_in_img * kBpTilesPerCta + tile_in_cta) * kBpTilePx;
        if (q0 >= n_vis) break;
        const long long base = cta_base + ws.tile_off[(size_t)gcta * kBpTilesPerCta + tile_in_cta];
        // addresses, then all eight loads back to back, then the ballots (a ballot is a convergence
        // point: fused into one loop the loads would be issued one DRAM round trip after the other)
        int off[kBpTilePx / 32];
        unsigned int uv[kBpTilePx / 32];
        float d[kBpTilePx / 32];
#pragma unroll
        for (int j = 0; j < kBpTilePx / 32; ++j) {
            const unsigned int q = q0 + j * 32 + lane;     // lane-consecutive pixels
            int u, v;
            bp_pixel(bp, inv_ws, q, u, v);
            uv[j] = ((unsigned int)v << 16) | (unsigned int)u;
            off[j] = (q < n_vis) ? v * bp.W + u : -1;
        }
#pragma unroll
        for (int j = 0; j < kBpTilePx / 32; ++j) d[j] = (off[j] >= 0) ? __ldg(dimg + off[j]) : -1.0f;   // -1: not visited
        int n = 0;                                           // points staged so far (warp-uniform)
#pragma unroll
        for (int j = 0; j < kBpTilePx / 32; ++j) {
            const bool visited = off[j] >= 0;
            const bool valid = d[j] > 0.0f;
            const bool emit = visited && (valid || !valid_only);
            const unsigned int bal = __ballot_sync(0xffffffffu, emit);
            if (emit) {
                const int o = n + __popc(bal & ((1u << lane) - 1u));
                const int v = (int)(uv[j] >> 16), u = (int)(uv[j] & 0xffffu);
                float3 p = make_float3(NAN, NAN, NAN);
                if (valid) p = backproject_px(bp, img_local, u, v, d[j]);
                sx[3 * o + 0] = p.x; sx[3 * o + 1] = p.y; sx[3 * o + 2] = p.z;
                if (WITH_RGB) {
                    const uint8_t *c = rgb_u8 + ((int64_t)img * bp.H * bp.W + off[j]) * 3;
                    sc[3 * o + 0] = valid ? c[0] / 255.0f : NAN;
                    sc[3 * o + 1] = valid ? c[1] / 255.0f : NAN;
                    sc[3 * o + 2] = valid ? c[2] / 255.0f : NAN;
                }
            }
            n += __popc(bal);
        }
        __syncwarp();
        const long long room = capacity - base;
        const int n_write = (int)max(0ll, min((long long)n, room));
        float *dst = xyz + 3 * base;
        for (int i = lane; i < 3 * n_write; i += 32) dst[i] = sx[i];
        if (WITH_RGB) {
            float *dstc = rgb + 3 * base;
            for (int i = lane; i < 3 * n_write; i += 32) dstc[i] = sc[i];
        }
        __syncwarp();
    }
}

static int grid_for(int64_t work_items, int per_block) {
    int64_t g = (work_items + per_block - 1) / per_block;
    const int64_t cap = (int64_t)current_device_sms() * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

} // namespace bslam

using namespace bslam;

extern "C" {

int bslam_scale_u16(const float *d_depth, int64_t n, float scale_mul, uint16_t *d_out, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(d_depth && d_out && n >= 0, "bslam_scale_u16: bad argument");
    BSLAM_CHECK_ARG(((uintptr_t)d_depth & 15) == 0 && ((uintptr_t)d_out & 7) == 0, "bslam_scale_u16: buffers must be 16-byte aligned");
    if (n == 0) return BSLAM_OK;
    scale_u16_kernel<<<grid_for(n, 1024), 256, 0, (cudaStream_t)stream>>>(d_depth, n, scale_mul, d_out);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

size_t bslam_colorize_workspace_bytes(int B) { return B > 0 ? (size_t)B * kWsPerImage + (size_t)B * 16 : 0; }

static int run_hist(const float *d_depth_m, const uint16_t *d_u16_in, int B, int64_t n, float scale_mul, uint16_t *d_u16_out,
                    int has_invalid, uint16_t invalid_val, void *ws, cudaStream_t st) {
    BSLAM_CUDA(cudaMemsetAsync(ws, 0, bslam_colorize_workspace_bytes(B), st));
    const dim3 grid((unsigned)((n + kPxPerBlock - 1) / kPxPerBlock), (unsigned)B);
    if (d_depth_m) scale_hist_kernel<true><<<grid, kHistThreads, 0, st>>>(d_depth_m, nullptr, d_u16_out, n, scale_mul, has_invalid, invalid_val, ws);
    else scale_hist_kernel<false><<<grid, kHistThreads, 0, st>>>(nullptr, d_u16_in, nullptr, n, scale_mul, has_invalid, invalid_val, ws);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

int bslam_colorize(const float *d_depth_m, const uint16_t *d_u16_in, int B, int H, int W, float scale_mul, uint16_t *d_u16_out,
                   uint8_t *d_rgba, const uint8_t *d_lut, double p_lo, double p_hi, int has_invalid, uint16_t invalid_val,
                   uint32_t bg_rgba, const double *h_vmin_vmax, double *d_vmin_vmax_out, const uint8_t *d_table_override,
                   void *d_workspace, bslam_stream_t stream) {
    BSLAM_CHECK_ARG((d_depth_m != nullptr) != (d_u16_in != nullptr), "bslam_colorize: give exactly one of d_depth_m / d_u16_in");
    BSLAM_CHECK_ARG(B > 0 && H > 0 && W > 0 && B <= 65535, "bslam_colorize: bad shape B=%d H=%d W=%d", B, H, W);
    BSLAM_CHECK_ARG(d_rgba && d_lut && d_workspace, "bslam_colorize: NULL output / lut / workspace");
    BSLAM_CHECK_ARG(!(d_depth_m && !d_u16_out), "bslam_colorize: float input needs d_u16_out (the metric-scaled image)");
    BSLAM_CHECK_ARG(p_lo >= 0 && p_lo <= 100 && p_hi >= 0 && p_hi <= 100, "bslam_colorize: percentiles must be in [0,100]");
    // the kernels read 4 pixels per access: float4 / ushort4 / uchar4 x 4
    BSLAM_CHECK_ARG(((uintptr_t)d_depth_m & 15) == 0 && ((uintptr_t)d_u16_in & 7) == 0 && ((uintptr_t)d_u16_out & 7) == 0 && ((uintptr_t)d_rgba & 15) == 0,
                    "bslam_colorize: depth / rgba buffers must be 16-byte aligned, u16 buffers 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = (int64_t)H * W;
    int rc = run_hist(d_depth_m, d_u16_in, B, n, scale_mul, d_u16_out, has_invalid, invalid_val, d_workspace, st);
    if (rc) return rc;
    double *d_override = nullptr;
    if (h_vmin_vmax) {
        d_override = (double *)((char *)d_workspace + (size_t)B * kWsPerImage);
        BSLAM_CUDA(cudaMemcpyAsync(d_override, h_vmin_vmax, (size_t)B * 16, cudaMemcpyHostToDevice, st));
    }
    stats_table_kernel<<<dim3((unsigned)B, 1), 1024, 0, st>>>(d_workspace, p_lo, p_hi, d_override, d_vmin_vmax_out, nullptr, 0, d_table_override, 1);
    BSLAM_LAUNCH_CHECK();
    stats_table_kernel<<<dim3((unsigned)B, kTableSlices), 1024, 0, st>>>(d_workspace, p_lo, p_hi, d_override, nullptr, nullptr, 0, d_table_override, 2);
    BSLAM_LAUNCH_CHECK();
    const uint16_t *src = d_depth_m ? d_u16_out : d_u16_in;
    const dim3 grid((unsigned)grid_for(n, 1024 * 4), (unsigned)B);
    apply_table_kernel<4><<<grid, 256, 0, st>>>(src, n, d_lut, has_invalid, invalid_val, bg_rgba, d_rgba, nullptr, d_workspace);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

int bslam_minmax_u8(const uint16_t *d_u16, int B, int H, int W, uint8_t *d_gray, uint8_t *d_rgb, const uint8_t *d_lut3,
                    void *d_workspace, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(d_u16 && d_workspace && B > 0 && H > 0 && W > 0 && B <= 65535, "bslam_minmax_u8: bad argument");
    BSLAM_CHECK_ARG(d_gray || d_rgb, "bslam_minmax_u8: no output requested");
    BSLAM_CHECK_ARG(!(d_rgb && !d_lut3), "bslam_minmax_u8: colour output needs a 256x3 LUT");
    BSLAM_CHECK_ARG(((uintptr_t)d_u16 & 7) == 0, "bslam_minmax_u8: the u16 buffer must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = (int64_t)H * W;
    int rc = run_hist(nullptr, d_u16, B, n, 1.0f, nullptr, 0, 0, d_workspace, st);
    if (rc) return rc;
    stats_table_kernel<<<dim3((unsigned)B, 1), 1024, 0, st>>>(d_workspace, 0, 100, nullptr, nullptr, nullptr, 1, nullptr, 1);
    BSLAM_LAUNCH_CHECK();
    stats_table_kernel<<<dim3((unsigned)B, kTableSlices), 1024, 0, st>>>(d_workspace, 0, 100, nullptr, nullptr, nullptr, 1, nullptr, 2);
    BSLAM_LAUNCH_CHECK();
    const dim3 grid((unsigned)grid_for(n, 1024 * 4), (unsigned)B);
    apply_table_kernel<3><<<grid, 256, 0, st>>>(d_u16, n, d_lut3, 0, 0, 0, d_rgb, d_gray, d_workspace);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

int bslam_median_u16(const uint16_t *d_u16, int B, int64_t n_per_image, int has_invalid, uint16_t invalid_val, double *d_out,
                     void *d_workspace, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(d_u16 && d_out && d_workspace && B > 0 && B <= 65535 && n_per_image > 0, "bslam_median_u16: bad argument");
    BSLAM_CHECK_ARG(((uintptr_t)d_u16 & 7) == 0, "bslam_median_u16: the u16 buffer must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = run_hist(nullptr, d_u16, B, n_per_image, 1.0f, nullptr, has_invalid, invalid_val, d_workspace, st);
    if (rc) return rc;
    stats_table_kernel<<<dim3((unsigned)B, 1), 1024, 0, st>>>(d_workspace, 50, 50, nullptr, nullptr, d_out, 2, nullptr, 0);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

int bslam_depth_from_u16(const uint16_t *d_in, int64_t n, float depth_scale, float depth_trunc, float *d_out, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(d_in && d_out && n >= 0 && depth_scale > 0, "bslam_depth_from_u16: bad argument");
    BSLAM_CHECK_ARG(((uintptr_t)d_in & 7) == 0 && ((uintptr_t)d_out & 15) == 0, "bslam_depth_from_u16: buffers must be 16-byte aligned");
    if (n == 0) return BSLAM_OK;
    depth_from_u16_kernel<<<grid_for(n, 1024), 256, 0, (cudaStream_t)stream>>>(d_in, n, depth_scale, depth_trunc, d_out);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

static int bp_tiles_per_image(int H, int W, int stride) {
    const int64_t n_vis = (int64_t)((H + stride - 1) / stride) * ((W + stride - 1) / stride);
    return (int)((n_vis + kBpTilePx - 1) / kBpTilePx);
}
static int bp_ctas_per_image(int H, int W, int stride) { return (bp_tiles_per_image(H, W, stride) + kBpTilesPerCta - 1) / kBpTilesPerCta; }

size_t bslam_backproject_workspace_bytes(int B, int H, int W, int stride) {
    if (B <= 0 || H <= 0 || W <= 0 || stride <= 0) return 0;
    const size_t n_ctas = (size_t)B * bp_ctas_per_image(H, W, stride);
    return n_ctas * kBpTilesPerCta * 4 + n_ctas * 4 + n_ctas * 8 + 3 * 256;
}

int bslam_backproject(const float *d_depth, const uint8_t *d_rgb_u8, int B, int H, int W, int stride, const float *h_K,
                      const float *h_cam_to_world, int valid_only, float *d_xyz, float *d_rgb, int64_t capacity,
                      int64_t *d_counts, void *d_workspace, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(d_depth && h_K && h_cam_to_world && d_xyz && d_counts && d_workspace, "bslam_backproject: NULL argument");
    BSLAM_CHECK_ARG(B > 0 && H > 0 && W > 0 && stride > 0, "bslam_backproject: bad shape");
    BSLAM_CHECK_ARG(!(d_rgb && !d_rgb_u8), "bslam_backproject: colour output needs the RGB8 image");
    BSLAM_CHECK_ARG(H <= 65535 && W <= 65535 && (int64_t)H * W < (1ll << 31), "bslam_backproject: image too large");
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local BackprojP bp;
    bp.fx = h_K[0]; bp.fy = h_K[1]; bp.cx = h_K[2]; bp.cy = h_K[3];
    bp.inv_fx = (float)(1.0 / (double)h_K[0]); bp.inv_fy = (float)(1.0 / (double)h_K[1]);
    bp.H = H; bp.W = W; bp.stride = stride;
    bp.Hs = (H + stride - 1) / stride; bp.Ws = (W + stride - 1) / stride;
    bp.tiles_per_image = bp_tiles_per_image(H, W, stride);
    bp.ctas_per_image = bp_ctas_per_image(H, W, stride);
    const int64_t n_ctas = (int64_t)B * bp.ctas_per_image;
    BSLAM_CHECK_ARG(n_ctas < (1ll << 31), "bslam_backproject: too many tiles");
    BackprojWs ws;
    char *w = (char *)d_workspace;
    ws.cta_base = (long long *)w;  w += ((size_t)n_ctas * 8 + 255) / 256 * 256;
    ws.tile_off = (int *)w;        w += ((size_t)n_ctas * kBpTilesPerCta * 4 + 255) / 256 * 256;
    ws.cta_total = (int *)w;
    bp.img0 = 0; bp.n_images = B;
    bp_count_kernel<<<(unsigned)n_ctas, kBpThreads, 0, st>>>(bp, d_depth, valid_only, ws);
    BSLAM_LAUNCH_CHECK();
    bp_scan_kernel<<<1, 1024, 0, st>>>(ws, (int)n_ctas, bp.ctas_per_image, B, (long long *)d_counts);
    BSLAM_LAUNCH_CHECK();
    for (int i0 = 0; i0 < B; i0 += kBpMaxImages) {
        const int nb = (B - i0 < kBpMaxImages) ? B - i0 : kBpMaxImages;
        bp.img0 = i0; bp.n_images = nb;
        memcpy(bp.pose, h_cam_to_world + (size_t)i0 * 12, (size_t)nb * 12 * sizeof(float));
        const unsigned grid = (unsigned)(nb * bp.ctas_per_image);
        if (d_rgb && d_rgb_u8) bp_emit_kernel<true><<<grid, kBpThreads, 0, st>>>(bp, d_depth, d_rgb_u8, valid_only, d_xyz, d_rgb, capacity, ws);
        else bp_emit_kernel<false><<<grid, kBpThreads, 0, st>>>(bp, d_depth, nullptr, valid_only, d_xyz, nullptr, capacity, ws);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

} // extern "C"
