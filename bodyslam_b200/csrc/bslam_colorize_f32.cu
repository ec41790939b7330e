// K1, float flavour -- `colorize(value, ...)` of R/examples/depth_estimation/depth_map_scaling.py:12-45 for a
// FLOAT32 image (metres from ZoeDepth, a torch tensor or a numpy array -- the reference accepts both, :14-15),
// where the 65 536-bin histogram of the uint16 path does not apply.
//
// NumPy semantics reproduced (NumPy 2.x, float32 input -> everything stays float32):
//   n      = number of valid pixels (value != invalid_val)
//   q      = float32(p) / float32(100);  virt = float32(n - 1) * q            (float32 products)
//   i0     = floor(virt), i1 = min(i0 + 1, n - 1), gamma = virt - i0           (float32)
//   vmin   = lerp(sorted[i0], sorted[i1], gamma)  with numpy's _lerp           (float32)
//            NaN when any valid pixel is NaN (np.percentile propagates NaN), so every valid pixel gets the bad colour
//   x      = (value - vmin) / (vmax - vmin)   (float32)   or   value * 0  when vmin == vmax
//            with both bounds explicit (Python floats) `vmin != vmax` and `vmax - vmin` are evaluated in double,
//            and the difference meets the float32 array rounded to float32 (NEP 50)
//   index  = matplotlib Colormap.__call__(x, bytes=True): x * 256, < 0 -> 0, == 256 -> 255, > 255 -> 255, trunc
// The four order statistics come from an exact two-level radix select on the order-preserving 32-bit key of
// the float: a 65 536-bin histogram of the key's high half, then -- for the (at most four) bins that hold a
// wanted rank -- a 65 536-bin histogram of the low half.  No sort, no library call.
#include <math.h>

#include "bslam_common.cuh"

namespace bslam {

constexpr int kFBins = 65536;
// per-image workspace: hi histogram | 4 lo histograms | select state
struct FSel {
    unsigned int n_valid;
    unsigned int n_nan;         // valid pixels that are NaN (counted by the level-0 histogram pass)
    unsigned int want[4];       // wanted sorted positions
    unsigned int hi_bin[4];     // high half of the key holding each wanted position
    unsigned int before[4];     // valid pixels with a smaller high half
    float gamma[2];
    float vmin, vmax;
    float den;                  // vmax - vmin as the normalisation divides by it
    unsigned int flat;          // vmin == vmax: x = value * 0
};
constexpr size_t kFWsPerImage = (size_t)kFBins * 4 * 5 + 256;

__device__ __forceinline__ unsigned int *f_hist_hi(void *ws, int b) { return (unsigned int *)((char *)ws + (size_t)b * kFWsPerImage); }
__device__ __forceinline__ unsigned int *f_hist_lo(void *ws, int b, int j) { return f_hist_hi(ws, b) + (size_t)(1 + j) * kFBins; }
__device__ __forceinline__ FSel *f_sel(void *ws, int b) { return (FSel *)((char *)ws + (size_t)b * kFWsPerImage + (size_t)kFBins * 4 * 5); }

// order-preserving key: a < b (as floats, -0 < +0, NaNs at the ends)  <=>  key(a) < key(b)
__device__ __forceinline__ unsigned int fkey(float v) {
    const unsigned int u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(unsigned int k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// one atomic per distinct bin per warp (depth images are smooth: neighbouring pixels share a bin)
__device__ __forceinline__ void warp_hist_add(unsigned int *hist, unsigned int bin, bool valid) {
    const unsigned int act = __ballot_sync(0xffffffffu, valid);
    if (!valid) return;
    const unsigned int peers = __match_any_sync(act, bin);
    if ((__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(hist + bin, (unsigned int)__popc(peers));
}

template <int LEVEL>
__global__ void __launch_bounds__(256) fkey_hist_kernel(const float *__restrict__ value, int64_t n_per_image, int has_invalid, float invalid_val, void *ws) {
    const int b = blockIdx.y;
    const float *img = value + (int64_t)b * n_per_image;
    unsigned int *hi = f_hist_hi(ws, b);
    FSel *sel = f_sel(ws, b);
    unsigned int tgt[4] = {0, 0, 0, 0};
    if (LEVEL == 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) tgt[j] = sel->hi_bin[j];
    }
    const int64_t per_iter = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_round = (n_per_image + per_iter - 1) / per_iter * per_iter;   // whole warps stay converged for the ballots
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_round; p += per_iter) {
        float v = 0.f;
        bool ok = p < n_per_image;
        if (ok) {
            v = __ldg(img + p);
            ok = !(has_invalid && v == invalid_val);
        }
        const unsigned int k = fkey(v);
        if (LEVEL == 0) {
            warp_hist_add(hi, k >> 16, ok);
            const unsigned int nan = __ballot_sync(0xffffffffu, ok && v != v);
            if (nan && (threadIdx.x & 31) == 0) atomicAdd(&sel->n_nan, (unsigned int)__popc(nan));
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                bool dup = false;       // identical target bins share histogram j' < j
#pragma unroll
                for (int i = 0; i < j; ++i) dup |= tgt[i] == tgt[j];
                if (!dup) warp_hist_add(f_hist_lo(ws, b, j), k & 0xffffu, ok && (k >> 16) == tgt[j]);
            }
        }
    }
}

// exclusive block scan over 65 536 bins held 64 per thread (1024 threads) -> (bin, count before the bin) of `want`
__device__ void find_rank(const unsigned int *hist, const unsigned int *want, int n_want, unsigned int *out_bin, unsigned int *out_before,
                          unsigned int *total_out) {
    __shared__ unsigned int s_warp[32];
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    constexpr int kPer = kFBins / 1024;
    unsigned int local = 0;
    for (int i = 0; i < kPer / 4; ++i) {
        const uint4 c = reinterpret_cast<const uint4 *>(hist + t * kPer)[i];
        local += c.x + c.y + c.z + c.w;
    }
    unsigned int inc = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
    }
    __syncthreads();
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        unsigned int w = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int up = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += up;
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    const unsigned int before = (wid ? s_warp[wid - 1] : 0u) + inc - local;
    if (total_out && t == 0) *total_out = s_warp[31];
    for (int j = 0; j < n_want; ++j) {
        const unsigned int w = want[j];
        if (w >= before && w < before + local) {        // exactly one thread owns the rank: walk its 64 bins
            unsigned int acc = before;
            for (int i = 0; i < kPer; ++i) {
                const unsigned int c = hist[t * kPer + i];
                if (w < acc + c) { out_bin[j] = (unsigned int)(t * kPer + i); out_before[j] = acc; break; }
                acc += c;
            }
        }
    }
    __syncthreads();
}

// level 0: n, wanted ranks (NumPy float32 arithmetic) and the high-half bins holding them
__global__ void __launch_bounds__(1024) fkey_select_hi_kernel(void *ws, float p_lo, float p_hi) {
    __shared__ unsigned int s_n;
    __shared__ unsigned int s_want[4];
    __shared__ unsigned int s_bin[4], s_before[4];
    const int b = blockIdx.x;
    FSel *s = f_sel(ws, b);
    const unsigned int *hist = f_hist_hi(ws, b);
    // total first (a scan with no wanted rank), then the ranks
    find_rank(hist, s_want, 0, s_bin, s_before, &s_n);
    __syncthreads();
    const unsigned int n = s_n;
    if (threadIdx.x == 0) {
        s->n_valid = n;
        const float p[2] = {p_lo, p_hi};
        for (int k = 0; k < 2; ++k) {
            unsigned int i0 = 0, i1 = 0;
            float g = 0.f;
            if (n > 0) {
                const float q = p[k] / 100.0f;                  // np.true_divide(q, float32(100))
                const float virt = (float)(n - 1) * q;          // (n - 1) * quantiles, float32
                float fl = floorf(virt);
                if (fl > (float)(n - 1)) fl = (float)(n - 1);   // _get_indexes clips
                i0 = (unsigned int)fl;
                i1 = (i0 + 1 > n - 1) ? n - 1 : i0 + 1;
                g = virt - fl;
            }
            s_want[2 * k] = i0; s_want[2 * k + 1] = i1;
            s->want[2 * k] = i0; s->want[2 * k + 1] = i1;
            s->gamma[k] = g;
        }
    }
    __syncthreads();
    if (n == 0) {
        if (threadIdx.x < 4) { s->hi_bin[threadIdx.x] = 0; s->before[threadIdx.x] = 0; }
        return;
    }
    find_rank(hist, s_want, 4, s_bin, s_before, nullptr);
    if (threadIdx.x < 4) { s->hi_bin[threadIdx.x] = s_bin[threadIdx.x]; s->before[threadIdx.x] = s_before[threadIdx.x]; }
}

__device__ __forceinline__ float numpy_lerp_f32(float a, float b, float t) {
    const float diff = b - a;
    float r = a + diff * t;
    if (t >= 0.5f) r = b - diff * (1.0f - t);
    return r;
}

// level 1: the low halves -> the four order statistics -> vmin / vmax (float32 lerp)
__global__ void __launch_bounds__(1024) fkey_select_lo_kernel(void *ws, const double *vmin_vmax_override, double *vmin_vmax_out) {
    __shared__ unsigned int s_want[1], s_bin[1], s_before[1];
    __shared__ float s_val[4];
    const int b = blockIdx.x;
    FSel *s = f_sel(ws, b);
    const unsigned int n = s->n_valid;
    for (int j = 0; j < 4 && n > 0; ++j) {
        int src = j;                                   // duplicates were accumulated into the first histogram with that bin
        for (int i = j - 1; i >= 0; --i)
            if (s->hi_bin[i] == s->hi_bin[j]) src = i;
        if (threadIdx.x == 0) s_want[0] = s->want[j] - s->before[j];
        __syncthreads();
        find_rank(f_hist_lo(ws, b, src), s_want, 1, s_bin, s_before, nullptr);
        if (threadIdx.x == 0) s_val[j] = fkey_inv((s->hi_bin[j] << 16) | s_bin[0]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        float vmin = 0.f, vmax = 0.f;
        if (n > 0) {
            vmin = numpy_lerp_f32(s_val[0], s_val[1], s->gamma[0]);
            vmax = numpy_lerp_f32(s_val[2], s_val[3], s->gamma[1]);
            if (s->n_nan) vmin = vmax = __int_as_float(0x7fffffff);   // np.percentile of data holding a NaN
        }
        const double a = vmin_vmax_override ? vmin_vmax_override[2 * b] : NAN, c = vmin_vmax_override ? vmin_vmax_override[2 * b + 1] : NAN;
        if (a == a) vmin = (float)a;        // explicit vmin / vmax: a Python float meets a float32 array -> float32 (NEP 50)
        if (c == c) vmax = (float)c;
        bool flat = vmin == vmax;
        float den = vmax - vmin;
        if (a == a && c == c) {             // two Python floats: compared and subtracted in double
            flat = a == c;
            den = (float)(c - a);
        }
        s->vmin = vmin; s->vmax = vmax; s->den = den; s->flat = flat;
        if (vmin_vmax_out) { vmin_vmax_out[2 * b] = (double)vmin; vmin_vmax_out[2 * b + 1] = (double)vmax; }
    }
}

__global__ void __launch_bounds__(256) apply_f32_kernel(const float *__restrict__ value, int64_t n_per_image, const uint8_t *__restrict__ lut,
                                                        int has_invalid, float invalid_val, uint32_t bg, uint8_t *__restrict__ out, void *ws) {
    __shared__ uint32_t s_lut[256];
    const int b = blockIdx.y;
    s_lut[threadIdx.x] = reinterpret_cast<const uint32_t *>(lut)[threadIdx.x];
    __syncthreads();
    const FSel *s = f_sel(ws, b);
    const float vmin = s->vmin, den = s->den;
    const bool flat = s->flat != 0;
    const int64_t img_off = (int64_t)b * n_per_image;
    uint32_t *o32 = reinterpret_cast<uint32_t *>(out) + img_off;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_per_image; p += (int64_t)gridDim.x * blockDim.x) {
        const float v = __ldg(value + img_off + p);
        uint32_t c;
        if (has_invalid && v == invalid_val) {
            c = bg;
        } else {
            float x = flat ? v * 0.0f : (v - vmin) / den;      // float32, like numpy
            x *= 256.0f;                                        // xa *= N
            unsigned int idx;
            if (!(x == x)) idx = 0xffffffffu;                   // NaN -> the colormap's "bad" colour (0, 0, 0, 0)
            else if (x < 0.0f) idx = 0;
            else if (x >= 256.0f) idx = 255;
            else idx = (unsigned int)x;
            c = idx == 0xffffffffu ? 0u : s_lut[idx];
        }
        o32[p] = c;
    }
}

} // namespace bslam

using namespace bslam;

extern "C" {

size_t bslam_colorize_f32_workspace_bytes(int B) { return B > 0 ? (size_t)B * kFWsPerImage + (size_t)B * 16 : 0; }

int bslam_colorize_f32(const float *d_value, int B, int H, int W, uint8_t *d_rgba, const uint8_t *d_lut, double p_lo, double p_hi,
                       int has_invalid, float invalid_val, uint32_t bg_rgba, const double *h_vmin_vmax, double *d_vmin_vmax_out,
                       void *d_workspace, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(d_value && d_rgba && d_lut && d_workspace, "bslam_colorize_f32: NULL argument");
    BSLAM_CHECK_ARG(B > 0 && H > 0 && W > 0 && B <= 65535 && (int64_t)H * W < (1ll << 32), "bslam_colorize_f32: bad shape B=%d H=%d W=%d", B, H, W);
    BSLAM_CHECK_ARG(p_lo >= 0 && p_lo <= 100 && p_hi >= 0 && p_hi <= 100, "bslam_colorize_f32: percentiles must be in [0,100]");
    BSLAM_CHECK_ARG(((uintptr_t)d_rgba & 3) == 0, "bslam_colorize_f32: the RGBA image must be 4-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = (int64_t)H * W;
    BSLAM_CUDA(cudaMemsetAsync(d_workspace, 0, bslam_colorize_f32_workspace_bytes(B), st));
    int gx = (int)((n + 256 * 8 - 1) / (256 * 8));
    const int cap = current_device_sms() * 8;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    const dim3 grid((unsigned)gx, (unsigned)B);
    fkey_hist_kernel<0><<<grid, 256, 0, st>>>(d_value, n, has_invalid, invalid_val, d_workspace);
    BSLAM_LAUNCH_CHECK();
    fkey_select_hi_kernel<<<B, 1024, 0, st>>>(d_workspace, (float)p_lo, (float)p_hi);
    BSLAM_LAUNCH_CHECK();
    fkey_hist_kernel<1><<<grid, 256, 0, st>>>(d_value, n, has_invalid, invalid_val, d_workspace);
    BSLAM_LAUNCH_CHECK();
    double *d_override = nullptr;
    if (h_vmin_vmax) {
        d_override = (double *)((char *)d_workspace + (size_t)B * kFWsPerImage);
        BSLAM_CUDA(cudaMemcpyAsync(d_override, h_vmin_vmax, (size_t)B * 16, cudaMemcpyHostToDevice, st));
    }
    fkey_select_lo_kernel<<<B, 1024, 0, st>>>(d_workspace, d_override, d_vmin_vmax_out);
    BSLAM_LAUNCH_CHECK();
    apply_f32_kernel<<<grid, 256, 0, st>>>(d_value, n, d_lut, has_invalid, invalid_val, bg_rgba, d_rgba, d_workspace);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

} // extern "C"
