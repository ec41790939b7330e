// Multi-scale RGB-D odometry: Open3D's tensor `rgbd_odometry_multi_scale` (point-to-plane, intensity, hybrid), which
// `t.pipelines.slam.Model.track_frame_to_model` runs with the ray-cast model frame as the target.  The semantics are
// written down in the CPU reference tests/odometry_ref.c, which this file must match: the prepared maps bit for bit
// (-fmad=false, IEEE `/` and sqrtf), the 29 float64 sums of a linearisation up to their summation order.  Parity with
// Open3D itself is unpinned.
//   * frame preparation: depth / intensity conversion, both pyramids, vertex, normal and Sobel maps of F frames into a
//     caller-owned buffer (layout in bodyslam_b200.h); a frame shared by two pairs is prepared once;
//   * odom_reduce_kernel<method>: kOdThreads threads per CTA, each over kOdPerThread source pixels, grid = tiles x pairs; every
//     CTA writes its 29 float64 partial sums to its own slot -- no float atomics, so a pair's sums are bit-reproducible
//     and do not depend on the other pairs of the launch;
//   * odom_solve_kernel: one CTA per pair sums the partials in a fixed order, solves the 6x6 system in float64, updates
//     T and decides convergence; a converged or singular pair is skipped by the later launches of its level;
//   * no host synchronisation and no copies inside the loop: poses and pair indices enter through kernel parameters.
#include <math.h>

#include "bslam_common.cuh"

namespace bslam {

constexpr int kOdPlanes = 12;         // depth, intensity, vertex xyz, normal xyz, Sobel x/y of depth, Sobel x/y of intensity
constexpr int kOdDepth = 0, kOdInt = 1, kOdVx = 2, kOdNx = 5, kOdDdx = 8, kOdDdy = 9, kOdDix = 10, kOdDiy = 11;
constexpr int kOdSums = 29;           // upper triangle of J^T J (21), J^T huber'(r) (6), sum huber(r), inlier count
constexpr int kOdThreads = 256;
constexpr int kOdPerThread = 4;
constexpr int kOdTile = kOdThreads * kOdPerThread;
constexpr int kOdMaxLevels = 16;
constexpr int kOdMaxGridY = 65535;    // frames per prepare call and pairs per track / linearize call (they run in gridDim.y)
constexpr int kOdInitPairs = 128;     // pairs per init launch (their poses travel as kernel parameters)
enum { kPointToPlane = 0, kIntensity = 1, kHybrid = 2 };

// Open3D's hybrid weights sqrt(lambda) (lambda_depth = 0.968, lambda_intensity = 0.032; recalled, as in the reference)
constexpr float kSqrtLambdaDepth = 0.98386991f;
constexpr float kSqrtLambdaIntensity = 0.17888544f;

__device__ __forceinline__ float od_nan() { return __int_as_float(0x7fc00000); }

__host__ __device__ inline int64_t od_level_offset(int H, int W, int l) {
    int64_t o = 0;
    for (int k = 0; k < l; ++k) o += (int64_t)kOdPlanes * (H >> k) * (W >> k);
    return o;
}

struct OdK {
    float fx, fy, cx, cy;
};
static OdK od_level_k(const double *h_K, int l) {
    const float s = 1.0f / (float)(1 << l);
    return OdK{(float)h_K[0] * s, (float)h_K[1] * s, (float)h_K[2] * s, (float)h_K[3] * s};
}

// per-pair state of a track / linearize call (the pose itself lives in the caller's d_T)
struct OdPair {
    float Tf[12];                 // T rounded to float32, rows 0..2: what the pixel kernel uses
    double prev_fit, prev_rmse;
    int src, tgt;
    int done_level;               // level at which the pair converged (-1: none)
    int status;                   // 0 = ok, 1 = singular system
    int pad[2];
};
static size_t od_pairs_bytes(int P) { return ((size_t)P * sizeof(OdPair) + 255) & ~(size_t)255; }

// ------------------------------------------------------------------------------------------------ frame preparation
__global__ void odom_convert_kernel(const void *__restrict__ depth, int depth_dtype, const void *__restrict__ color, int color_dtype, int H,
                                    int W, int64_t frame_floats, float depth_scale, float depth_max, float *__restrict__ frames) {
    const int64_t n = (int64_t)H * W;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t f = blockIdx.y;
    float *fr = frames + f * frame_floats;
    const float raw = depth_dtype == 0 ? (float)((const uint16_t *)depth)[f * n + i] : ((const float *)depth)[f * n + i];
    const float d = raw / depth_scale;
    fr[kOdDepth * n + i] = (d <= 0.0f || d >= depth_max) ? od_nan() : d;
    float I = od_nan();
    if (color) {
        float c[3];
#pragma unroll
        for (int k = 0; k < 3; ++k)
            c[k] = color_dtype == 0 ? (float)((const uint8_t *)color)[(f * n + i) * 3 + k] : ((const float *)color)[(f * n + i) * 3 + k];
        I = (0.299f * c[0] + 0.587f * c[1]) + 0.114f * c[2];
        if (color_dtype == 0) I = I / 255.0f;
    }
    fr[kOdInt * n + i] = I;
}

__constant__ float c_od_gauss[5] = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};

// level l - 1 -> level l: PyrDownDepth (Gaussian mean of the valid neighbours within thr of the centre) and PyrDown of
// the intensity (replicated borders)
__global__ void odom_pyrdown_kernel(int H, int W, int l, int64_t frame_floats, float thr, float *__restrict__ frames) {
    const int Hs = H >> (l - 1), Ws = W >> (l - 1), Hd = H >> l, Wd = W >> l;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Hd * Wd) return;
    const int y = i / Wd, x = i % Wd;
    float *fr = frames + (int64_t)blockIdx.y * frame_floats;
    const float *sd = fr + od_level_offset(H, W, l - 1) + (int64_t)kOdDepth * Hs * Ws;
    const float *si = fr + od_level_offset(H, W, l - 1) + (int64_t)kOdInt * Hs * Ws;
    float *dd = fr + od_level_offset(H, W, l) + (int64_t)kOdDepth * Hd * Wd;
    float *di = fr + od_level_offset(H, W, l) + (int64_t)kOdInt * Hd * Wd;
    const float c = sd[(2 * y) * Ws + 2 * x];
    float sw = 0.0f, sv = 0.0f, si_acc = 0.0f;
    for (int dy = -2; dy <= 2; ++dy)
        for (int dx = -2; dx <= 2; ++dx) {
            const int yy = 2 * y + dy, xx = 2 * x + dx;
            const float w = c_od_gauss[dy + 2] * c_od_gauss[dx + 2];
            const int yc = yy < 0 ? 0 : (yy >= Hs ? Hs - 1 : yy), xc = xx < 0 ? 0 : (xx >= Ws ? Ws - 1 : xx);
            si_acc += w * si[yc * Ws + xc];
            if (yy < 0 || yy >= Hs || xx < 0 || xx >= Ws) continue;
            const float d = sd[yy * Ws + xx];
            if (!(fabsf(d - c) < thr)) continue;
            sw += w;
            sv += w * d;
        }
    dd[y * Wd + x] = isnan(c) ? od_nan() : sv / sw;
    di[y * Wd + x] = si_acc;
}

__device__ __forceinline__ void od_vertex(float d, int x, int y, const OdK &k, float *v) {
    v[0] = (((float)x - k.cx) * d) / k.fx;
    v[1] = (((float)y - k.cy) * d) / k.fy;
    v[2] = d;
}

__device__ __forceinline__ void od_sobel(const float *p, int H, int W, int x, int y, float *dx, float *dy) {
    const int xm = x > 0 ? x - 1 : 0, xp = x < W - 1 ? x + 1 : W - 1, ym = y > 0 ? y - 1 : 0, yp = y < H - 1 ? y + 1 : H - 1;
    const float a00 = p[ym * W + xm], a01 = p[ym * W + x], a02 = p[ym * W + xp];
    const float a10 = p[y * W + xm], a12 = p[y * W + xp];
    const float a20 = p[yp * W + xm], a21 = p[yp * W + x], a22 = p[yp * W + xp];
    *dx = ((a02 - a00) + 2.0f * (a12 - a10)) + (a22 - a20);
    *dy = ((a20 - a00) + 2.0f * (a21 - a01)) + (a22 - a02);
}

// vertex, normal and Sobel maps of one level
__global__ void odom_maps_kernel(int H, int W, int l, int64_t frame_floats, OdK k, float *__restrict__ frames) {
    const int Hl = H >> l, Wl = W >> l;
    const int64_t n = (int64_t)Hl * Wl;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int y = i / Wl, x = i % Wl;
    float *L = frames + (int64_t)blockIdx.y * frame_floats + od_level_offset(H, W, l);
    const float *D = L + kOdDepth * n;
    float v[3];
    od_vertex(D[i], x, y, k, v);
    const bool ok = !isnan(D[i]);
#pragma unroll
    for (int c = 0; c < 3; ++c) L[(kOdVx + c) * n + i] = ok ? v[c] : od_nan();
    float nr[3] = {od_nan(), od_nan(), od_nan()};
    if (x < Wl - 1 && y < Hl - 1 && ok && !isnan(D[i + 1]) && !isnan(D[i + Wl])) {
        float v10[3], v01[3];
        od_vertex(D[i + 1], x + 1, y, k, v10);
        od_vertex(D[i + Wl], x, y + 1, k, v01);
        const float a[3] = {v10[0] - v[0], v10[1] - v[1], v10[2] - v[2]};
        const float b[3] = {v01[0] - v[0], v01[1] - v[1], v01[2] - v[2]};
        const float c[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
        const float len = sqrtf((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2]);
#pragma unroll
        for (int q = 0; q < 3; ++q) nr[q] = c[q] / len;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) L[(kOdNx + c) * n + i] = nr[c];
    od_sobel(D, Hl, Wl, x, y, &L[kOdDdx * n + i], &L[kOdDdy * n + i]);
    od_sobel(L + kOdInt * n, Hl, Wl, x, y, &L[kOdDix * n + i], &L[kOdDiy * n + i]);
}

// ------------------------------------------------------------------------------------------------ linearisation
struct OdLevel {
    int H, W, Hl, Wl, level, n_tiles, tiles_cap;
    int64_t frame_floats, level_offset;
    OdK k;
    float trunc, depth_huber, intensity_huber;
};

__device__ __forceinline__ float od_huber(float r, float d) {
    const float a = fabsf(r);
    return a <= d ? 0.5f * r * r : d * (a - 0.5f * d);
}
__device__ __forceinline__ float od_huber_deriv(float r, float d) { return fabsf(r) <= d ? r : (r > 0.0f ? d : -d); }

// residuals and Jacobians of one source pixel (tests/odometry_ref.c pixel_terms); 0 = rejected
template <int METHOD>
__device__ __forceinline__ int od_pixel_terms(const float *__restrict__ S, const float *__restrict__ Tg, const OdLevel &lv, const float *Tf,
                                              int64_t i, int x, int y, float J[2][6], float r[2]) {
    const int64_t n = (int64_t)lv.Hl * lv.Wl;
    const float v[3] = {S[(kOdVx + 0) * n + i], S[(kOdVx + 1) * n + i], S[(kOdVx + 2) * n + i]};
    if (isnan(v[2])) return 0;
    const float Is = METHOD != kPointToPlane ? S[kOdInt * n + i] : 0.0f;
    if (METHOD != kPointToPlane && isnan(Is)) return 0;
    float vs[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) vs[q] = ((Tf[4 * q] * v[0] + Tf[4 * q + 1] * v[1]) + Tf[4 * q + 2] * v[2]) + Tf[4 * q + 3];
    if (vs[2] <= 0.0f) return 0;
    const float uf = (lv.k.fx * vs[0]) / vs[2] + lv.k.cx, vf = (lv.k.fy * vs[1]) / vs[2] + lv.k.cy;
    if (!(uf > -1.0f && uf < (float)lv.Wl && vf > -1.0f && vf < (float)lv.Hl)) return 0;
    const int u = (int)roundf(uf), w = (int)roundf(vf);
    if (u < 0 || u >= lv.Wl || w < 0 || w >= lv.Hl) return 0;
    const int64_t j = (int64_t)w * lv.Wl + u;
    if (METHOD == kPointToPlane) {
        const float vt[3] = {__ldg(Tg + (kOdVx + 0) * n + j), __ldg(Tg + (kOdVx + 1) * n + j), __ldg(Tg + (kOdVx + 2) * n + j)};
        const float nt[3] = {__ldg(Tg + (kOdNx + 0) * n + j), __ldg(Tg + (kOdNx + 1) * n + j), __ldg(Tg + (kOdNx + 2) * n + j)};
        if (isnan(vt[2]) || isnan(nt[0]) || isnan(nt[1]) || isnan(nt[2])) return 0;
        const float res = ((vs[0] - vt[0]) * nt[0] + (vs[1] - vt[1]) * nt[1]) + (vs[2] - vt[2]) * nt[2];
        if (fabsf(res) > lv.trunc) return 0;
        J[0][0] = vs[1] * nt[2] - vs[2] * nt[1];
        J[0][1] = vs[2] * nt[0] - vs[0] * nt[2];
        J[0][2] = vs[0] * nt[1] - vs[1] * nt[0];
        J[0][3] = nt[0]; J[0][4] = nt[1]; J[0][5] = nt[2];
        r[0] = res;
        return 1;
    }
    const float Dt = __ldg(Tg + kOdDepth * n + j);
    if (isnan(Dt) || !(fabsf(Dt - vs[2]) <= lv.trunc)) return 0;
    const float dIx = 0.125f * __ldg(Tg + kOdDix * n + j), dIy = 0.125f * __ldg(Tg + kOdDiy * n + j);
    if (isnan(dIx) || isnan(dIy)) return 0;
    float dDx = 0.0f, dDy = 0.0f;
    if (METHOD == kHybrid) {
        dDx = 0.125f * __ldg(Tg + kOdDdx * n + j);
        dDy = 0.125f * __ldg(Tg + kOdDdy * n + j);
        if (isnan(dDx) || isnan(dDy)) return 0;
    }
    const float invz = 1.0f / vs[2];
    const float c0 = (dIx * lv.k.fx) * invz, c1 = (dIy * lv.k.fy) * invz, c2 = -((c0 * vs[0] + c1 * vs[1]) * invz);
    const float wI = METHOD == kHybrid ? kSqrtLambdaIntensity : 1.0f;
    J[0][0] = wI * (vs[1] * c2 - vs[2] * c1);
    J[0][1] = wI * (vs[2] * c0 - vs[0] * c2);
    J[0][2] = wI * (vs[0] * c1 - vs[1] * c0);
    J[0][3] = wI * c0; J[0][4] = wI * c1; J[0][5] = wI * c2;
    r[0] = wI * (__ldg(Tg + kOdInt * n + j) - Is);
    if (METHOD != kHybrid) return 1;
    const float d0 = (dDx * lv.k.fx) * invz, d1 = (dDy * lv.k.fy) * invz, d2 = -((d0 * vs[0] + d1 * vs[1]) * invz);
    const float wD = kSqrtLambdaDepth;
    J[1][0] = wD * ((vs[1] * d2 - vs[2] * d1) - vs[1]);
    J[1][1] = wD * ((vs[2] * d0 - vs[0] * d2) + vs[0]);
    J[1][2] = wD * (vs[0] * d1 - vs[1] * d0);
    J[1][3] = wD * d0; J[1][4] = wD * d1; J[1][5] = wD * (d2 - 1.0f);
    r[1] = wD * (Dt - vs[2]);
    return 2;
}

// sum of v over the CTA in a fixed order (shuffle tree within each warp, then the warps in order); valid in thread 0..
// of `out` (shared, kOdSums doubles) after the call
__device__ __forceinline__ void od_block_sum(double *acc, double (*s_warp)[kOdSums], double *out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < kOdSums; ++k) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) s_warp[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < kOdSums) {
        double v = 0.0;
        for (int w = 0; w < kOdThreads / 32; ++w) v += s_warp[w][threadIdx.x];
        out[threadIdx.x] = v;
    }
    __syncthreads();
}

__device__ __forceinline__ bool od_active(const OdPair &p, int level) { return p.status == 0 && p.done_level != level; }

template <int METHOD>
__global__ void __launch_bounds__(kOdThreads) odom_reduce_kernel(const float *__restrict__ frames, const OdPair *__restrict__ pairs,
                                                                 const __grid_constant__ OdLevel lv, double *__restrict__ partials) {
    const int p = blockIdx.y;
    const OdPair &st = pairs[p];
    if (!od_active(st, lv.level)) return;
    __shared__ double s_warp[kOdThreads / 32][kOdSums];
    __shared__ double s_out[kOdSums];
    float Tf[12];
#pragma unroll
    for (int q = 0; q < 12; ++q) Tf[q] = st.Tf[q];
    const float *S = frames + (int64_t)st.src * lv.frame_floats + lv.level_offset;
    const float *Tg = frames + (int64_t)st.tgt * lv.frame_floats + lv.level_offset;
    const float dI = METHOD == kPointToPlane ? lv.depth_huber : lv.intensity_huber;
    double acc[kOdSums];
#pragma unroll
    for (int k = 0; k < kOdSums; ++k) acc[k] = 0.0;
    const int64_t n = (int64_t)lv.Hl * lv.Wl;
#pragma unroll 1
    for (int q = 0; q < kOdPerThread; ++q) {
        const int64_t i = (int64_t)blockIdx.x * kOdTile + q * kOdThreads + threadIdx.x;
        if (i >= n) break;
        float J[2][6], r[2];
        const int nres = od_pixel_terms<METHOD>(S, Tg, lv, Tf, i, (int)(i % lv.Wl), (int)(i / lv.Wl), J, r);
        if (!nres) continue;
        const float hp0 = od_huber_deriv(r[0], dI);
        const float hp1 = METHOD == kHybrid ? od_huber_deriv(r[1], lv.depth_huber) : 0.0f;
        int k = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
            for (int b = a; b < 6; ++b, ++k) {
                double v = (double)J[0][a] * (double)J[0][b];
                if (METHOD == kHybrid) v += (double)J[1][a] * (double)J[1][b];
                acc[k] += v;
            }
#pragma unroll
        for (int a = 0; a < 6; ++a) {
            double v = (double)J[0][a] * (double)hp0;
            if (METHOD == kHybrid) v += (double)J[1][a] * (double)hp1;
            acc[21 + a] += v;
        }
        double loss = (double)od_huber(r[0], dI);
        if (METHOD == kHybrid) loss += (double)od_huber(r[1], lv.depth_huber);
        acc[27] += loss;
        acc[28] += 1.0;
    }
    od_block_sum(acc, s_warp, s_out);
    if (threadIdx.x < kOdSums) partials[((int64_t)p * lv.tiles_cap + blockIdx.x) * kOdSums + threadIdx.x] = s_out[threadIdx.x];
}

// ------------------------------------------------------------------------------------------------ solve and update
__device__ bool od_solve6(const double *S, double *x) {
    if (!(S[28] >= 6.0)) return false;
    double A[6][6], L[6][6], y[6];
    int k = 0;
    for (int a = 0; a < 6; ++a)
        for (int b = a; b < 6; ++b, ++k) A[a][b] = A[b][a] = S[k];
    for (int j = 0; j < 6; ++j) {
        double s = A[j][j];
        for (int q = 0; q < j; ++q) s -= L[j][q] * L[j][q];
        if (!(s > 0.0)) return false;
        L[j][j] = sqrt(s);
        for (int i = j + 1; i < 6; ++i) {
            double t = A[i][j];
            for (int q = 0; q < j; ++q) t -= L[i][q] * L[j][q];
            L[i][j] = t / L[j][j];
        }
    }
    for (int i = 0; i < 6; ++i) {
        double t = -S[21 + i];
        for (int q = 0; q < i; ++q) t -= L[i][q] * y[q];
        y[i] = t / L[i][i];
    }
    for (int i = 5; i >= 0; --i) {
        double t = y[i];
        for (int q = i + 1; q < 6; ++q) t -= L[q][i] * x[q];
        x[i] = t / L[i][i];
    }
    return true;
}

// T <- DeltaT(x) * T, DeltaT = [Rz(gamma) Ry(beta) Rx(alpha) | t]
__device__ void od_update_pose(double *T, const double *x) {
    const double ca = cos(x[0]), sa = sin(x[0]), cb = cos(x[1]), sb = sin(x[1]), cg = cos(x[2]), sg = sin(x[2]);
    const double D[16] = {cg * cb, -sg * ca + (cg * sb) * sa, sg * sa + (cg * sb) * ca, x[3],
                          sg * cb, cg * ca + (sg * sb) * sa, -cg * sa + (sg * sb) * ca, x[4],
                          -sb, cb * sa, cb * ca, x[5],
                          0.0, 0.0, 0.0, 1.0};
    double N[16];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j)
            N[4 * i + j] = ((D[4 * i] * T[j] + D[4 * i + 1] * T[4 + j]) + D[4 * i + 2] * T[8 + j]) + D[4 * i + 3] * T[12 + j];
    for (int i = 0; i < 16; ++i) T[i] = N[i];
}

struct OdSolve {
    int level, crit, n_levels;
    double rel_fitness, rel_rmse;
    int first;                      // first iteration of the level: no previous fitness
};

// one CTA per pair.  sums != NULL (bslam_odom_linearize): write the 29 sums and stop.
__global__ void __launch_bounds__(kOdThreads) odom_solve_kernel(OdPair *__restrict__ pairs, const __grid_constant__ OdLevel lv, OdSolve sv,
                                                                const double *__restrict__ partials, double *__restrict__ sums,
                                                                double *__restrict__ d_T, double *__restrict__ d_rmse_fitness,
                                                                int *__restrict__ d_iters, int *__restrict__ d_status) {
    const int p = blockIdx.x;
    OdPair &st = pairs[p];
    if (!od_active(st, lv.level)) return;
    __shared__ double s_warp[kOdThreads / 32][kOdSums];
    __shared__ double s_out[kOdSums];
    double acc[kOdSums];
#pragma unroll
    for (int k = 0; k < kOdSums; ++k) acc[k] = 0.0;
    for (int t = threadIdx.x; t < lv.n_tiles; t += kOdThreads) {
        const double *src = partials + ((int64_t)p * lv.tiles_cap + t) * kOdSums;
#pragma unroll
        for (int k = 0; k < kOdSums; ++k) acc[k] += src[k];
    }
    od_block_sum(acc, s_warp, s_out);
    if (sums) {
        if (threadIdx.x < kOdSums) sums[(int64_t)p * kOdSums + threadIdx.x] = s_out[threadIdx.x];
        return;
    }
    if (threadIdx.x != 0) return;
    const double *S = s_out;
    const double fit = S[28] / ((double)lv.Hl * (double)lv.Wl);
    const double rmse = S[28] > 0.0 ? sqrt(S[27] / S[28]) : 0.0;
    d_rmse_fitness[2 * p] = rmse;
    d_rmse_fitness[2 * p + 1] = fit;
    d_iters[(int64_t)p * sv.n_levels + sv.crit] += 1;
    double x[6];
    if (!od_solve6(S, x)) {
        st.status = 1;
        d_status[p] = 1;
        return;
    }
    double *T = d_T + (int64_t)p * 16;
    od_update_pose(T, x);
    for (int q = 0; q < 12; ++q) st.Tf[q] = (float)T[q];
    const double pf = sv.first ? 0.0 : st.prev_fit, pr = sv.first ? 0.0 : st.prev_rmse;
    if (pf != 0.0 && fabs(fit - pf) / pf < sv.rel_fitness && fabs(rmse - pr) / pr < sv.rel_rmse) st.done_level = lv.level;
    st.prev_fit = fit;
    st.prev_rmse = rmse;
}

// pair state from the host's poses and indices (kernel parameters: no copy); T is written to d_T
struct OdInit {
    int n;
    int src[kOdInitPairs], tgt[kOdInitPairs];
    double T[kOdInitPairs][16];
};
__global__ void odom_init_kernel(const __grid_constant__ OdInit in, int p0, int n_levels, OdPair *__restrict__ pairs, double *__restrict__ d_T,
                                 double *__restrict__ d_rmse_fitness, int *__restrict__ d_iters, int *__restrict__ d_status) {
    const int i = threadIdx.x;
    if (i >= in.n) return;
    const int p = p0 + i;
    OdPair &st = pairs[p];
    for (int q = 0; q < 12; ++q) st.Tf[q] = (float)in.T[i][q];
    st.prev_fit = st.prev_rmse = 0.0;
    st.src = in.src[i];
    st.tgt = in.tgt[i];
    st.done_level = -1;
    st.status = 0;
    if (d_T)
        for (int q = 0; q < 16; ++q) d_T[(int64_t)p * 16 + q] = in.T[i][q];
    if (d_rmse_fitness) d_rmse_fitness[2 * p] = d_rmse_fitness[2 * p + 1] = 0.0;
    if (d_iters)
        for (int q = 0; q < n_levels; ++q) d_iters[(int64_t)p * n_levels + q] = 0;
    if (d_status) d_status[p] = 0;
}

static int od_tiles(int H, int W, int l) { return (int)(((int64_t)(H >> l) * (W >> l) + kOdTile - 1) / kOdTile); }

static OdLevel od_level(int H, int W, int levels, int l, const double *h_K, float trunc, float dh, float ih) {
    OdLevel lv;
    lv.H = H; lv.W = W; lv.Hl = H >> l; lv.Wl = W >> l; lv.level = l;
    lv.n_tiles = od_tiles(H, W, l);
    lv.tiles_cap = od_tiles(H, W, 0);
    lv.frame_floats = od_level_offset(H, W, levels);
    lv.level_offset = od_level_offset(H, W, l);
    lv.k = od_level_k(h_K, l);
    lv.trunc = trunc; lv.depth_huber = dh; lv.intensity_huber = ih;
    return lv;
}

static void od_launch_reduce(int method, const float *frames, const OdPair *pairs, const OdLevel &lv, int P, double *partials, cudaStream_t st) {
    const dim3 grid(lv.n_tiles, P);
    if (method == kPointToPlane) odom_reduce_kernel<kPointToPlane><<<grid, kOdThreads, 0, st>>>(frames, pairs, lv, partials);
    else if (method == kIntensity) odom_reduce_kernel<kIntensity><<<grid, kOdThreads, 0, st>>>(frames, pairs, lv, partials);
    else odom_reduce_kernel<kHybrid><<<grid, kOdThreads, 0, st>>>(frames, pairs, lv, partials);
}

static int od_init(const int *h_pairs, const double *h_T, int P, int n_levels, OdPair *pairs, double *d_T, double *d_rmse_fitness, int *d_iters,
                   int *d_status, cudaStream_t st) {
    static thread_local OdInit in;
    for (int p0 = 0; p0 < P; p0 += kOdInitPairs) {
        in.n = P - p0 < kOdInitPairs ? P - p0 : kOdInitPairs;
        for (int i = 0; i < in.n; ++i) {
            in.src[i] = h_pairs[2 * (p0 + i)];
            in.tgt[i] = h_pairs[2 * (p0 + i) + 1];
            memcpy(in.T[i], h_T + (size_t)(p0 + i) * 16, 16 * sizeof(double));
        }
        odom_init_kernel<<<1, kOdInitPairs, 0, st>>>(in, p0, n_levels, pairs, d_T, d_rmse_fitness, d_iters, d_status);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

} // namespace bslam

using namespace bslam;

#define OD_CHECK_SHAPE(name)                                                                                                          \
    BSLAM_CHECK_ARG(H > 0 && W > 0 && levels >= 1 && levels <= kOdMaxLevels && (H >> (levels - 1)) >= 1 && (W >> (levels - 1)) >= 1, \
                    "[" name "] Unsupported image format. (H=%d W=%d levels=%d: every level must be at least 1 x 1)", H, W, levels)

#define OD_CHECK_PAIRS(name)                                                                                                          \
    BSLAM_CHECK_ARG(F >= 0 && P >= 0 && P <= kOdMaxGridY, name ": F must be >= 0 and P in [0, %d]", kOdMaxGridY);               \
    BSLAM_CHECK_ARG(method >= kPointToPlane && method <= kHybrid, name ": method must be 0 (PointToPlane), 1 (Intensity) or 2 (Hybrid)"); \
    BSLAM_CHECK_ARG(h_K, name ": NULL argument");                                                                                   \
    for (int i = 0; i < 2 * P && h_pairs; ++i)                                                                                      \
        BSLAM_CHECK_ARG(h_pairs[i] >= 0 && h_pairs[i] < F, name ": pair index %d out of range [0, %d)", h_pairs[i], F)

extern "C" {

size_t bslam_odom_frame_bytes(int H, int W, int levels) {
    if (H <= 0 || W <= 0 || levels < 1 || levels > kOdMaxLevels || (H >> (levels - 1)) < 1 || (W >> (levels - 1)) < 1) return 0;
    return (size_t)od_level_offset(H, W, levels) * sizeof(float);
}

int bslam_odom_prepare(const void *d_depth, int depth_dtype, const void *d_color, int color_dtype, int F, int H, int W, int levels,
                       const double *h_K, float depth_scale, float depth_max, float depth_outlier_trunc, float *d_frames, bslam_stream_t stream) {
    OD_CHECK_SHAPE("bslam_odom_prepare");
    BSLAM_CHECK_ARG(F >= 0 && F <= kOdMaxGridY, "bslam_odom_prepare: F must be in [0, %d]", kOdMaxGridY);
    BSLAM_CHECK_ARG((depth_dtype == 0 || depth_dtype == 1) && (color_dtype == 0 || color_dtype == 1),
                    "bslam_odom_prepare: depth_dtype must be 0 (uint16) or 1 (float32), color_dtype 0 (uint8) or 1 (float32)");
    BSLAM_CHECK_ARG(depth_scale > 0.f && depth_max > 0.f && depth_outlier_trunc >= 0.f,
                    "bslam_odom_prepare: depth_scale and depth_max must be > 0, depth_outlier_trunc >= 0");
    BSLAM_CHECK_ARG(h_K && ((d_depth && d_frames) || F == 0), "bslam_odom_prepare: NULL argument");
    if (F == 0) return BSLAM_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t ff = od_level_offset(H, W, levels);
    const int64_t n0 = (int64_t)H * W;
    odom_convert_kernel<<<dim3((unsigned)((n0 + 255) / 256), F), 256, 0, st>>>(d_depth, depth_dtype, d_color, color_dtype, H, W, ff, depth_scale,
                                                                               depth_max, d_frames);
    BSLAM_LAUNCH_CHECK();
    for (int l = 1; l < levels; ++l) {
        const int64_t n = (int64_t)(H >> l) * (W >> l);
        odom_pyrdown_kernel<<<dim3((unsigned)((n + 255) / 256), F), 256, 0, st>>>(H, W, l, ff, 2.0f * depth_outlier_trunc, d_frames);
        BSLAM_LAUNCH_CHECK();
    }
    for (int l = 0; l < levels; ++l) {
        const int64_t n = (int64_t)(H >> l) * (W >> l);
        odom_maps_kernel<<<dim3((unsigned)((n + 255) / 256), F), 256, 0, st>>>(H, W, l, ff, od_level_k(h_K, l), d_frames);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

size_t bslam_odom_workspace_bytes(int P, int H, int W, int levels) {
    if (P <= 0 || bslam_odom_frame_bytes(H, W, levels) == 0) return 0;
    return od_pairs_bytes(P) + (size_t)P * od_tiles(H, W, 0) * kOdSums * sizeof(double);
}

int bslam_odom_track(const float *d_frames, int F, const int *h_pairs, int P, int H, int W, int levels, const double *h_K, int method,
                     const int *h_max_iter, const double *h_rel_fitness, const double *h_rel_rmse, float depth_outlier_trunc,
                     float depth_huber_delta, float intensity_huber_delta, const double *h_init, double *d_T, double *d_rmse_fitness,
                     int *d_iters, int *d_status, void *d_workspace, bslam_stream_t stream) {
    OD_CHECK_SHAPE("bslam_odom_track");
    OD_CHECK_PAIRS("bslam_odom_track");
    BSLAM_CHECK_ARG(h_max_iter && h_rel_fitness && h_rel_rmse, "bslam_odom_track: NULL argument");
    for (int c = 0; c < levels; ++c) BSLAM_CHECK_ARG(h_max_iter[c] >= 0, "bslam_odom_track: max_iteration must be >= 0");
    BSLAM_CHECK_ARG(depth_outlier_trunc >= 0.f && depth_huber_delta >= 0.f && intensity_huber_delta >= 0.f,
                    "bslam_odom_track: depth_outlier_trunc and the Huber deltas must be >= 0");
    if (P == 0) return BSLAM_OK;
    BSLAM_CHECK_ARG(d_frames && h_pairs && h_init && d_T && d_rmse_fitness && d_iters && d_status && d_workspace, "bslam_odom_track: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    OdPair *pairs = (OdPair *)d_workspace;
    double *partials = (double *)((char *)d_workspace + od_pairs_bytes(P));
    if (od_init(h_pairs, h_init, P, levels, pairs, d_T, d_rmse_fitness, d_iters, d_status, st) != BSLAM_OK) return BSLAM_E_CUDA;
    for (int c = 0; c < levels; ++c) {
        const int l = levels - 1 - c;
        const OdLevel lv = od_level(H, W, levels, l, h_K, depth_outlier_trunc, depth_huber_delta, intensity_huber_delta);
        for (int it = 0; it < h_max_iter[c]; ++it) {
            od_launch_reduce(method, d_frames, pairs, lv, P, partials, st);
            BSLAM_LAUNCH_CHECK();
            const OdSolve sv{l, c, levels, h_rel_fitness[c], h_rel_rmse[c], it == 0};
            odom_solve_kernel<<<P, kOdThreads, 0, st>>>(pairs, lv, sv, partials, nullptr, d_T, d_rmse_fitness, d_iters, d_status);
            BSLAM_LAUNCH_CHECK();
        }
    }
    return BSLAM_OK;
}

int bslam_odom_linearize(const float *d_frames, int F, const int *h_pairs, int P, int H, int W, int levels, int level, const double *h_K,
                         int method, float depth_outlier_trunc, float depth_huber_delta, float intensity_huber_delta, const double *h_T,
                         double *d_sums, void *d_workspace, bslam_stream_t stream) {
    OD_CHECK_SHAPE("bslam_odom_linearize");
    OD_CHECK_PAIRS("bslam_odom_linearize");
    BSLAM_CHECK_ARG(level >= 0 && level < levels, "bslam_odom_linearize: level %d out of range [0, %d)", level, levels);
    if (P == 0) return BSLAM_OK;
    BSLAM_CHECK_ARG(d_frames && h_pairs && h_T && d_sums && d_workspace, "bslam_odom_linearize: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    OdPair *pairs = (OdPair *)d_workspace;
    double *partials = (double *)((char *)d_workspace + od_pairs_bytes(P));
    if (od_init(h_pairs, h_T, P, levels, pairs, nullptr, nullptr, nullptr, nullptr, st) != BSLAM_OK) return BSLAM_E_CUDA;
    const OdLevel lv = od_level(H, W, levels, level, h_K, depth_outlier_trunc, depth_huber_delta, intensity_huber_delta);
    od_launch_reduce(method, d_frames, pairs, lv, P, partials, st);
    BSLAM_LAUNCH_CHECK();
    const OdSolve sv{level, 0, levels, 0.0, 0.0, 1};
    odom_solve_kernel<<<P, kOdThreads, 0, st>>>(pairs, lv, sv, partials, d_sums, nullptr, nullptr, nullptr, nullptr);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

} // extern "C"
