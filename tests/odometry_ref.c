/* CPU reference of the multi-scale RGB-D odometry (TEST INFRASTRUCTURE, like oracle/): the semantics that
 * csrc/bslam_odometry.cu must match.  Open3D's tensor odometry (t.pipelines.odometry.rgbd_odometry_multi_scale, and
 * t.pipelines.slam.Model.track_frame_to_model, which calls it with the ray-cast model frame as the target) is restated
 * here from knowledge of RGBDOdometry.cpp / RGBDOdometryImpl.h / RGBDOdometryJacobianImpl.h, not from its source:
 * parity with Open3D itself is UNPINNED, and where a detail was uncertain this file decides (DESIGN.md section 7 lists
 * those details as hypotheses).
 *
 * Per-pixel arithmetic is float32 evaluated left to right (-ffp-contract=off; the library builds with -fmad=false);
 * the 29 sums of a linearisation are float64 (a product of two float32 values is exact in float64, so only the order
 * of the summation differs between this file and the GPU; Open3D sums in float32 with atomics).  The 6x6 solve and
 * the pose are float64.
 *
 * Prepared frame layout (shared with the library): per frame, per level l (H_l = H >> l, W_l = W >> l, coarser
 * levels after finer ones) 12 planes of H_l * W_l float32: depth (metres, NaN = invalid), intensity, vertex x, y, z,
 * normal x, y, z, Sobel_x(depth), Sobel_y(depth), Sobel_x(intensity), Sobel_y(intensity) (unscaled 3x3 Sobel). */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define API __attribute__((visibility("default")))

enum { M_POINT_TO_PLANE = 0, M_INTENSITY = 1, M_HYBRID = 2 };
enum { P_DEPTH = 0, P_INT = 1, P_VX = 2, P_NX = 5, P_DDX = 8, P_DDY = 9, P_DIX = 10, P_DIY = 11, N_PLANES = 12 };
enum { N_SUMS = 29 };

/* Open3D's hybrid weights, sqrt(lambda): lambda_depth = 0.968 and lambda_intensity = 1 - 0.968 (recalled) */
static const float kSqrtLambdaDepth = 0.98386991f;
static const float kSqrtLambdaIntensity = 0.17888544f;
static const float kGauss[5] = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};

static int64_t level_offset(int H, int W, int l) {
    int64_t o = 0;
    for (int k = 0; k < l; ++k) o += (int64_t)N_PLANES * (H >> k) * (W >> k);
    return o;
}

API int64_t ref_odom_frame_floats(int H, int W, int levels) { return level_offset(H, W, levels); }

static float huber(float r, float d) {
    const float a = fabsf(r);
    return a <= d ? 0.5f * r * r : d * (a - 0.5f * d);
}
static float huber_deriv(float r, float d) { return fabsf(r) <= d ? r : (r > 0.0f ? d : -d); }

static void sobel(const float *p, int H, int W, int x, int y, float *dx, float *dy) {
    const int xm = x > 0 ? x - 1 : 0, xp = x < W - 1 ? x + 1 : W - 1, ym = y > 0 ? y - 1 : 0, yp = y < H - 1 ? y + 1 : H - 1;
    const float a00 = p[ym * W + xm], a01 = p[ym * W + x], a02 = p[ym * W + xp];
    const float a10 = p[y * W + xm], a12 = p[y * W + xp];
    const float a20 = p[yp * W + xm], a21 = p[yp * W + x], a22 = p[yp * W + xp];
    *dx = ((a02 - a00) + 2.0f * (a12 - a10)) + (a22 - a20);
    *dy = ((a20 - a00) + 2.0f * (a21 - a01)) + (a22 - a02);
}

static void vertex(float d, int x, int y, float fx, float fy, float cx, float cy, float *v) {
    v[0] = (((float)x - cx) * d) / fx;
    v[1] = (((float)y - cy) * d) / fy;
    v[2] = d;
}

/* depth: [F][H][W] uint16 (depth_dtype 0) or float32 (1); color: NULL or [F][H][W][3] uint8 (color_dtype 0) or float32
 * in [0, 1] (1); K = fx, fy, cx, cy of level 0; out: F * ref_odom_frame_floats(H, W, levels) floats */
API void ref_odom_prepare(const void *depth, int depth_dtype, const void *color, int color_dtype, int F, int H, int W, int levels,
                          const double *K, float depth_scale, float depth_max, float depth_outlier_trunc, float *out) {
    const int64_t ff = ref_odom_frame_floats(H, W, levels);
    for (int f = 0; f < F; ++f) {
        float *fr = out + f * ff;
        const int64_t n = (int64_t)H * W;
        for (int64_t i = 0; i < n; ++i) {
            const float raw = depth_dtype == 0 ? (float)((const uint16_t *)depth)[f * n + i] : ((const float *)depth)[f * n + i];
            const float d = raw / depth_scale;
            fr[P_DEPTH * n + i] = (d <= 0.0f || d >= depth_max) ? NAN : d;
            float I = NAN;
            if (color) {
                float c[3];
                for (int k = 0; k < 3; ++k)
                    c[k] = color_dtype == 0 ? (float)((const uint8_t *)color)[(f * n + i) * 3 + k] : ((const float *)color)[(f * n + i) * 3 + k];
                I = (0.299f * c[0] + 0.587f * c[1]) + 0.114f * c[2];
                if (color_dtype == 0) I = I / 255.0f;
            }
            fr[P_INT * n + i] = I;
        }
        const float thr = 2.0f * depth_outlier_trunc;
        for (int l = 1; l < levels; ++l) {
            const int Hs = H >> (l - 1), Ws = W >> (l - 1), Hd = H >> l, Wd = W >> l;
            const float *sd = fr + level_offset(H, W, l - 1) + P_DEPTH * (int64_t)Hs * Ws;
            const float *si = fr + level_offset(H, W, l - 1) + P_INT * (int64_t)Hs * Ws;
            float *dd = fr + level_offset(H, W, l) + P_DEPTH * (int64_t)Hd * Wd;
            float *di = fr + level_offset(H, W, l) + P_INT * (int64_t)Hd * Wd;
            for (int y = 0; y < Hd; ++y)
                for (int x = 0; x < Wd; ++x) {
                    /* PyrDownDepth: Gaussian mean of the valid neighbours within thr of the centre; NaN centre -> NaN */
                    const float c = sd[(2 * y) * Ws + 2 * x];
                    float sw = 0.0f, sv = 0.0f, si_acc = 0.0f;
                    for (int dy = -2; dy <= 2; ++dy)
                        for (int dx = -2; dx <= 2; ++dx) {
                            const int yy = 2 * y + dy, xx = 2 * x + dx;
                            const float w = kGauss[dy + 2] * kGauss[dx + 2];
                            /* PyrDown of the intensity: replicated borders */
                            const int yc = yy < 0 ? 0 : (yy >= Hs ? Hs - 1 : yy), xc = xx < 0 ? 0 : (xx >= Ws ? Ws - 1 : xx);
                            si_acc += w * si[yc * Ws + xc];
                            if (yy < 0 || yy >= Hs || xx < 0 || xx >= Ws) continue;
                            const float d = sd[yy * Ws + xx];
                            if (!(fabsf(d - c) < thr)) continue;
                            sw += w;
                            sv += w * d;
                        }
                    dd[y * Wd + x] = isnan(c) ? NAN : sv / sw;
                    di[y * Wd + x] = si_acc;
                }
        }
        for (int l = 0; l < levels; ++l) {
            const int Hl = H >> l, Wl = W >> l;
            const int64_t n = (int64_t)Hl * Wl;
            const float s = 1.0f / (float)(1 << l);
            const float fx = (float)K[0] * s, fy = (float)K[1] * s, cx = (float)K[2] * s, cy = (float)K[3] * s;
            float *L = fr + level_offset(H, W, l);
            const float *D = L + P_DEPTH * n;
            for (int y = 0; y < Hl; ++y)
                for (int x = 0; x < Wl; ++x) {
                    const int64_t i = (int64_t)y * Wl + x;
                    float v[3];
                    vertex(D[i], x, y, fx, fy, cx, cy, v);
                    for (int k = 0; k < 3; ++k) L[(P_VX + k) * n + i] = isnan(D[i]) ? NAN : v[k];
                    float nr[3] = {NAN, NAN, NAN};
                    if (x < Wl - 1 && y < Hl - 1 && !isnan(D[i]) && !isnan(D[i + 1]) && !isnan(D[i + Wl])) {
                        float v10[3], v01[3];
                        vertex(D[i + 1], x + 1, y, fx, fy, cx, cy, v10);
                        vertex(D[i + Wl], x, y + 1, fx, fy, cx, cy, v01);
                        const float a[3] = {v10[0] - v[0], v10[1] - v[1], v10[2] - v[2]};
                        const float b[3] = {v01[0] - v[0], v01[1] - v[1], v01[2] - v[2]};
                        const float c[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
                        const float len = sqrtf((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2]);
                        for (int k = 0; k < 3; ++k) nr[k] = c[k] / len;
                    }
                    for (int k = 0; k < 3; ++k) L[(P_NX + k) * n + i] = nr[k];
                    sobel(D, Hl, Wl, x, y, &L[P_DDX * n + i], &L[P_DDY * n + i]);
                    sobel(L + P_INT * n, Hl, Wl, x, y, &L[P_DIX * n + i], &L[P_DIY * n + i]);
                }
        }
    }
}

typedef struct {
    const float *s, *t;     /* source / target frame, this level */
    int H, W;
    float fx, fy, cx, cy, trunc;
    int method;
} Level;

static Level level_of(const float *frames, int64_t ff, int src, int tgt, int H, int W, int l, const double *K, int method, float trunc) {
    Level L;
    const int64_t o = level_offset(H, W, l);
    L.s = frames + src * ff + o;
    L.t = frames + tgt * ff + o;
    L.H = H >> l;
    L.W = W >> l;
    const float s = 1.0f / (float)(1 << l);
    L.fx = (float)K[0] * s; L.fy = (float)K[1] * s; L.cx = (float)K[2] * s; L.cy = (float)K[3] * s;
    L.trunc = trunc;
    L.method = method;
    return L;
}

/* residuals r[0..nres-1] and their Jacobians J[k][6] (x = rotation alpha, beta, gamma, translation) of source pixel
 * (x, y) under the source -> target transform Tf (rows 0..2, float32); 0 = the pixel is rejected */
static int pixel_terms(const Level *L, const float *Tf, int x, int y, float J[2][6], float r[2], int *nres) {
    const int64_t n = (int64_t)L->H * L->W, i = (int64_t)y * L->W + x;
    const float v[3] = {L->s[(P_VX + 0) * n + i], L->s[(P_VX + 1) * n + i], L->s[(P_VX + 2) * n + i]};
    if (isnan(v[2])) return 0;
    const float Is = L->s[P_INT * n + i];
    if (L->method != M_POINT_TO_PLANE && isnan(Is)) return 0;
    float vs[3];
    for (int k = 0; k < 3; ++k) vs[k] = ((Tf[4 * k] * v[0] + Tf[4 * k + 1] * v[1]) + Tf[4 * k + 2] * v[2]) + Tf[4 * k + 3];
    if (vs[2] <= 0.0f) return 0;
    const float uf = (L->fx * vs[0]) / vs[2] + L->cx, vf = (L->fy * vs[1]) / vs[2] + L->cy;
    if (!(uf > -1.0f && uf < (float)L->W && vf > -1.0f && vf < (float)L->H)) return 0;
    const int u = (int)roundf(uf), w = (int)roundf(vf);
    if (u < 0 || u >= L->W || w < 0 || w >= L->H) return 0;
    const int64_t j = (int64_t)w * L->W + u;
    if (L->method == M_POINT_TO_PLANE) {
        const float vt[3] = {L->t[(P_VX + 0) * n + j], L->t[(P_VX + 1) * n + j], L->t[(P_VX + 2) * n + j]};
        const float nt[3] = {L->t[(P_NX + 0) * n + j], L->t[(P_NX + 1) * n + j], L->t[(P_NX + 2) * n + j]};
        if (isnan(vt[2]) || isnan(nt[0]) || isnan(nt[1]) || isnan(nt[2])) return 0;
        const float res = ((vs[0] - vt[0]) * nt[0] + (vs[1] - vt[1]) * nt[1]) + (vs[2] - vt[2]) * nt[2];
        if (fabsf(res) > L->trunc) return 0;
        J[0][0] = vs[1] * nt[2] - vs[2] * nt[1];
        J[0][1] = vs[2] * nt[0] - vs[0] * nt[2];
        J[0][2] = vs[0] * nt[1] - vs[1] * nt[0];
        J[0][3] = nt[0]; J[0][4] = nt[1]; J[0][5] = nt[2];
        r[0] = res;
        *nres = 1;
        return 1;
    }
    const float Dt = L->t[P_DEPTH * n + j];
    if (isnan(Dt) || !(fabsf(Dt - vs[2]) <= L->trunc)) return 0;
    const float dIx = 0.125f * L->t[P_DIX * n + j], dIy = 0.125f * L->t[P_DIY * n + j];
    if (isnan(dIx) || isnan(dIy)) return 0;
    const float dDx = 0.125f * L->t[P_DDX * n + j], dDy = 0.125f * L->t[P_DDY * n + j];
    if (L->method == M_HYBRID && (isnan(dDx) || isnan(dDy))) return 0;
    const float invz = 1.0f / vs[2];
    const float c0 = (dIx * L->fx) * invz, c1 = (dIy * L->fy) * invz, c2 = -((c0 * vs[0] + c1 * vs[1]) * invz);
    const float wI = L->method == M_HYBRID ? kSqrtLambdaIntensity : 1.0f;
    J[0][0] = wI * (vs[1] * c2 - vs[2] * c1);
    J[0][1] = wI * (vs[2] * c0 - vs[0] * c2);
    J[0][2] = wI * (vs[0] * c1 - vs[1] * c0);
    J[0][3] = wI * c0; J[0][4] = wI * c1; J[0][5] = wI * c2;
    r[0] = wI * (L->t[P_INT * n + j] - Is);
    *nres = 1;
    if (L->method == M_HYBRID) {
        const float d0 = (dDx * L->fx) * invz, d1 = (dDy * L->fy) * invz, d2 = -((d0 * vs[0] + d1 * vs[1]) * invz);
        const float wD = kSqrtLambdaDepth;
        J[1][0] = wD * ((vs[1] * d2 - vs[2] * d1) - vs[1]);
        J[1][1] = wD * ((vs[2] * d0 - vs[0] * d2) + vs[0]);
        J[1][2] = wD * (vs[0] * d1 - vs[1] * d0);
        J[1][3] = wD * d0; J[1][4] = wD * d1; J[1][5] = wD * (d2 - 1.0f);
        r[1] = wD * (Dt - vs[2]);
        *nres = 2;
    }
    return 1;
}

/* adds one inlier pixel's terms to the 29 sums: upper triangle of J^T J (row-major), J^T huber'(r), sum huber(r), count */
static void accumulate(double *S, float J[2][6], const float r[2], int nres, int method, float depth_huber_delta, float intensity_huber_delta) {
    const float delta0 = method == M_POINT_TO_PLANE ? depth_huber_delta : intensity_huber_delta;
    const float hp0 = huber_deriv(r[0], delta0), hp1 = nres > 1 ? huber_deriv(r[1], depth_huber_delta) : 0.0f;
    int k = 0;
    for (int a = 0; a < 6; ++a)
        for (int b = a; b < 6; ++b, ++k) {
            double v = (double)J[0][a] * (double)J[0][b];
            if (nres > 1) v += (double)J[1][a] * (double)J[1][b];
            S[k] += v;
        }
    for (int a = 0; a < 6; ++a) {
        double v = (double)J[0][a] * (double)hp0;
        if (nres > 1) v += (double)J[1][a] * (double)hp1;
        S[21 + a] += v;
    }
    double loss = (double)huber(r[0], delta0);
    if (nres > 1) loss += (double)huber(r[1], depth_huber_delta);
    S[27] += loss;
    S[28] += 1.0;
}

static void to_f32(const double *T, float *Tf) {
    for (int i = 0; i < 12; ++i) Tf[i] = (float)T[i];
}

static void linearize(const Level *L, const float *Tf, float dhd, float ihd, double *S) {
    double *rows = calloc((size_t)L->H * N_SUMS, sizeof(double));
#pragma omp parallel for schedule(static)
    for (int y = 0; y < L->H; ++y) {
        double *R = rows + (size_t)y * N_SUMS;
        for (int x = 0; x < L->W; ++x) {
            float J[2][6], r[2];
            int nres;
            if (pixel_terms(L, Tf, x, y, J, r, &nres)) accumulate(R, J, r, nres, L->method, dhd, ihd);
        }
    }
    memset(S, 0, N_SUMS * sizeof(double));
    for (int y = 0; y < L->H; ++y)
        for (int k = 0; k < N_SUMS; ++k) S[k] += rows[(size_t)y * N_SUMS + k];
    free(rows);
}

/* AtA x = -Atb by Cholesky; 0 = singular (fewer than 6 inliers or a non-positive pivot) */
static int solve6(const double *S, double *x) {
    if (!(S[28] >= 6.0)) return 0;
    double A[6][6], L[6][6], y[6];
    int k = 0;
    for (int a = 0; a < 6; ++a)
        for (int b = a; b < 6; ++b, ++k) A[a][b] = A[b][a] = S[k];
    for (int j = 0; j < 6; ++j) {
        double s = A[j][j];
        for (int q = 0; q < j; ++q) s -= L[j][q] * L[j][q];
        if (!(s > 0.0)) return 0;
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
    return 1;
}

/* T <- DeltaT(x) * T, DeltaT = [Rz(gamma) Ry(beta) Rx(alpha) | t] */
static void update_pose(double *T, const double *x) {
    const double ca = cos(x[0]), sa = sin(x[0]), cb = cos(x[1]), sb = sin(x[1]), cg = cos(x[2]), sg = sin(x[2]);
    const double D[16] = {cg * cb, -sg * ca + (cg * sb) * sa, sg * sa + (cg * sb) * ca, x[3],
                          sg * cb, cg * ca + (sg * sb) * sa, -cg * sa + (sg * sb) * ca, x[4],
                          -sb, cb * sa, cb * ca, x[5],
                          0.0, 0.0, 0.0, 1.0};
    double N[16];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j)
            N[4 * i + j] = ((D[4 * i] * T[j] + D[4 * i + 1] * T[4 + j]) + D[4 * i + 2] * T[8 + j]) + D[4 * i + 3] * T[12 + j];
    memcpy(T, N, sizeof(N));
}

/* the 29 sums of pair (src, tgt) at `level` under T [16] (row-major source -> target) */
API void ref_odom_linearize(const float *frames, int src, int tgt, int H, int W, int levels, int level, const double *K, int method,
                            float depth_outlier_trunc, float depth_huber_delta, float intensity_huber_delta, const double *T, double *sums) {
    const Level L = level_of(frames, ref_odom_frame_floats(H, W, levels), src, tgt, H, W, level, K, method, depth_outlier_trunc);
    float Tf[12];
    to_f32(T, Tf);
    linearize(&L, Tf, depth_huber_delta, intensity_huber_delta, sums);
}

/* one source pixel's terms (the Jacobian tests): returns the number of residuals, 0 = rejected */
API int ref_odom_pixel(const float *frames, int src, int tgt, int H, int W, int levels, int level, const double *K, int method,
                       float depth_outlier_trunc, const double *T, int x, int y, float *J12, float *r2) {
    const Level L = level_of(frames, ref_odom_frame_floats(H, W, levels), src, tgt, H, W, level, K, method, depth_outlier_trunc);
    float Tf[12], J[2][6], r[2];
    int nres = 0;
    to_f32(T, Tf);
    if (!pixel_terms(&L, Tf, x, y, J, r, &nres)) return 0;
    memcpy(J12, J, nres * 6 * sizeof(float));
    memcpy(r2, r, nres * sizeof(float));
    return nres;
}

/* the multi-scale loop, levels coarsest first (max_iter[0], rel_fitness[0], rel_rmse[0] belong to level levels - 1).
 * T [16]: in = init, out = result; rmse_fitness [2] of the last evaluation; iters [levels] evaluations per criteria
 * entry.  Returns 0, or 1 when a singular system ended the pair. */
API int ref_odom_track(const float *frames, int src, int tgt, int H, int W, int levels, const double *K, int method, const int *max_iter,
                       const double *rel_fitness, const double *rel_rmse, float depth_outlier_trunc, float depth_huber_delta,
                       float intensity_huber_delta, double *T, double *rmse_fitness, int *iters) {
    const int64_t ff = ref_odom_frame_floats(H, W, levels);
    rmse_fitness[0] = rmse_fitness[1] = 0.0;
    for (int c = 0; c < levels; ++c) iters[c] = 0;
    for (int c = 0; c < levels; ++c) {
        const int l = levels - 1 - c;
        const Level L = level_of(frames, ff, src, tgt, H, W, l, K, method, depth_outlier_trunc);
        double prev_fit = 0.0, prev_rmse = 0.0;
        for (int it = 0; it < max_iter[c]; ++it) {
            float Tf[12];
            double S[N_SUMS], x[6];
            to_f32(T, Tf);
            linearize(&L, Tf, depth_huber_delta, intensity_huber_delta, S);
            iters[c] += 1;
            const double fit = S[28] / ((double)L.H * (double)L.W);
            const double rmse = S[28] > 0.0 ? sqrt(S[27] / S[28]) : 0.0;
            rmse_fitness[0] = rmse;
            rmse_fitness[1] = fit;
            if (!solve6(S, x)) return 1;
            update_pose(T, x);
            if (prev_fit != 0.0 && fabs(fit - prev_fit) / prev_fit < rel_fitness[c] && fabs(rmse - prev_rmse) / prev_rmse < rel_rmse[c]) break;
            prev_fit = fit;
            prev_rmse = rmse;
        }
    }
    return 0;
}
