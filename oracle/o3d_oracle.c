/*
 * oracle/o3d_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement of the arithmetic behind BodySLAM's 3DM hot path.  The
 * reference delegates every one of these steps to Open3D (unpinned in
 * N/requirements.txt:12, not vendored under /root/reference, not installable
 * offline), so this file restates Open3D's legacy-pipeline semantics
 * (SURVEY.md Appendix A) and anchors on the reference's own call sites:
 *
 *   orc_depth_from_u16   <- RGBDImage.create_from_color_and_depth(depth_scale, depth_trunc)
 *                           N/3DM/slam_utils.py:212-220            (Appendix A.1)
 *   orc_backproject      <- PointCloud.create_from_depth_image / pixel_to_3d
 *                           N/3DM/mapping_module.py:37,41 ; N/3DM/scaling_system.py:72-77 (A.2)
 *   orc_tsdf_integrate   <- TSDF.build_3D_map -> volume.integrate   N/3DM/tsdf.py:14-22 (A.3)
 *   orc_scalable_integrate <- the same through ScalableTSDFVolume (unit activation, A.3 step 7)
 *   orc_extract_mesh     <- TSDF.extract_mesh                       N/3DM/tsdf.py:42-43 (A.4)
 *   orc_extract_points   <- TSDF.extract_pcd                        N/3DM/tsdf.py:39-40 (A.5)
 *
 * PARITY STATUS: *unpinned* against real Open3D for these five functions -- the
 * reference holds no test, fixture or recorded output for them (SURVEY.md 8c)
 * and Open3D cannot be imported here.  The oracle therefore DEFINES the order of
 * floating point operations (no FMA contraction: build with -ffp-contract=off).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference legs may load this library.
 *
 * Volume layout: dense box of nx*ny*nz voxels, Open3D order  idx = (x*ny + y)*nz + z.
 * The box may be a z-slab of a larger grid: local z maps to global z = gz0 + z.
 * World position of global voxel (X,Y,Z) centre = origin + (X+0.5, Y+0.5, Z+0.5)*voxel_length.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif
#include "mc_tables.h"

#define ORC_API __attribute__((visibility("default")))

ORC_API int orc_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

ORC_API void orc_set_num_threads(int n) {
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
#else
    (void)n;
#endif
}

/* ------------------------------------------------------------------ A.1 */
/* u16 -> f32 plain cast, divide by (float)depth_scale, zero when >= depth_trunc. */
ORC_API void orc_depth_from_u16(const uint16_t *in, size_t n, double depth_scale,
                                double depth_trunc, float *out) {
    const float scale_f = (float)depth_scale;
    for (size_t i = 0; i < n; ++i) {
        float p = (float)in[i];
        p /= scale_f;
        if ((double)p >= depth_trunc) p = 0.0f;
        out[i] = p;
    }
}

/* ------------------------------------------------------------------ A.2 */
/* cam_to_world = inverse(extrinsic) (row-major 4x4, f64), K = {fx, fy, cx, cy}.
 * Row-major scan, step `stride`; d > 0 pixels are emitted in order.  With
 * valid_only == 0 every visited pixel produces a row (NaN for d <= 0).
 * rgb (H*W*3 u8) may be NULL; colours are c/255 as f64.  Returns the number of rows. */
ORC_API int64_t orc_backproject(const float *depth, const uint8_t *rgb, int W, int H,
                                const double *K, const double *cam_to_world, int stride,
                                int valid_only, double *out_xyz, double *out_rgb) {
    const double fx = K[0], fy = K[1], cx = K[2], cy = K[3];
    const double *M = cam_to_world;
    int64_t n = 0;
    for (int i = 0; i < H; i += stride) {
        for (int j = 0; j < W; j += stride) {
            const float p = depth[(size_t)i * W + j];
            if (p > 0) {
                const double z = (double)p;
                const double x = (j - cx) * z / fx;
                const double y = (i - cy) * z / fy;
                for (int r = 0; r < 3; ++r)
                    out_xyz[3 * n + r] = ((M[4 * r + 0] * x + M[4 * r + 1] * y) + M[4 * r + 2] * z) + M[4 * r + 3];
                if (rgb && out_rgb)
                    for (int c = 0; c < 3; ++c)
                        out_rgb[3 * n + c] = rgb[((size_t)i * W + j) * 3 + c] / 255.0;
                ++n;
            } else if (!valid_only) {
                for (int r = 0; r < 3; ++r) out_xyz[3 * n + r] = NAN;
                if (rgb && out_rgb)
                    for (int c = 0; c < 3; ++c) out_rgb[3 * n + c] = NAN;
                ++n;
            }
        }
    }
    return n;
}

/* ------------------------------------------------------------------ A.3 */
/*
 * One frame into the dense box.  z_restart R: the float32 camera-space point of a
 * voxel column is evaluated directly (E*p) at every GLOBAL z that is a multiple
 * of R and advanced by the float32 increment E[:,2]*voxel_length in between;
 * R <= 0 is Open3D's literal loop (direct evaluation at global z = 0 only).
 * color: optional nx*ny*nz*3 f32 running mean of rgb (Open3D keeps f64; the
 * product keeps f32 -- see DESIGN.md), rgb: optional H*W*3 u8.
 * Returns the number of voxels updated by this frame (U_f of SURVEY.md 8d).
 */
ORC_API int64_t orc_tsdf_integrate(float *tsdf, float *weight, float *color, int nx, int ny,
                                   int nz, int gz0, double voxel_length, double sdf_trunc,
                                   const double *origin, const float *depth, const uint8_t *rgb,
                                   int W, int H, const double *K, const double *extrinsic,
                                   int z_restart) {
    const float fx = (float)K[0], fy = (float)K[1], cx = (float)K[2], cy = (float)K[3];
    float E[16];
    for (int i = 0; i < 16; ++i) E[i] = (float)extrinsic[i];
    const float vl = (float)voxel_length;
    const float half = vl * 0.5f;
    const float trunc_f = (float)sdf_trunc;
    const float trunc_inv = 1.0f / trunc_f;
    const float dzx = E[2] * vl, dzy = E[6] * vl, dzz = E[10] * vl; /* E_scaled(:,2) */
    const float safe_w = W - 0.0001f, safe_h = H - 0.0001f;
    const float fxi = 1.0f / fx, fyi = 1.0f / fy;
    int64_t updated = 0;

#pragma omp parallel for schedule(static) reduction(+ : updated)
    for (int x = 0; x < nx; ++x) {
        for (int y = 0; y < ny; ++y) {
            const float px = (float)((double)(half + vl * (float)x) + origin[0]);
            const float py = (float)((double)(half + vl * (float)y) + origin[1]);
            float pcx = 0.f, pcy = 0.f, pcz = 0.f;
            /* literal mode: march from global z = 0 up to the slab base */
            int need_direct = 1;
            int gz_begin = gz0;
            if (z_restart <= 0 && gz0 > 0) gz_begin = 0;
            for (int gz = gz_begin; gz < gz0 + nz; ++gz) {
                if (need_direct || (z_restart > 0 && gz % z_restart == 0)) {
                    const float pz = (float)((double)(half + vl * (float)gz) + origin[2]);
                    pcx = ((E[0] * px + E[1] * py) + E[2] * pz) + E[3];
                    pcy = ((E[4] * px + E[5] * py) + E[6] * pz) + E[7];
                    pcz = ((E[8] * px + E[9] * py) + E[10] * pz) + E[11];
                    need_direct = 0;
                }
                const float cxp = pcx, cyp = pcy, czp = pcz;
                pcx += dzx; pcy += dzy; pcz += dzz; /* value for gz+1 */
                if (gz < gz0) continue;
                if (czp <= 0) continue;
                const float u_f = cxp * fx / czp + cx + 0.5f;
                const float v_f = cyp * fy / czp + cy + 0.5f;
                if (!(u_f >= 0.0001f && u_f < safe_w && v_f >= 0.0001f && v_f < safe_h)) continue;
                const int u = (int)u_f, v = (int)v_f;
                const float d = depth[(size_t)v * W + u];
                if (d <= 0.0f) continue;
                const float xx = ((float)u - cx) * fxi, yy = ((float)v - cy) * fyi;
                const float mult = sqrtf((xx * xx + yy * yy) + 1.0f);
                const float sdf = (d - czp) * mult;
                if (sdf > -trunc_f) {
                    const size_t idx = ((size_t)x * ny + y) * nz + (gz - gz0);
                    const float t = fminf(1.0f, sdf * trunc_inv);
                    const float w = weight[idx];
                    if (color && rgb) {
                        const uint8_t *c = rgb + ((size_t)v * W + u) * 3;
                        for (int k = 0; k < 3; ++k)
                            color[3 * idx + k] = (color[3 * idx + k] * w + (float)c[k]) / (w + 1.0f);
                    }
                    tsdf[idx] = (tsdf[idx] * w + t) / (w + 1.0f);
                    weight[idx] = w + 1.0f;
                    ++updated;
                }
            }
        }
    }
    return updated;
}

/* Eigen's Matrix4d::inverse() is the cofactor (adjugate / determinant) formula; row-major f64 */
ORC_API void orc_invert4x4(const double *a, double *out) {
    double c[16];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {
            /* minor of (j, i) -> adjugate entry (i, j) */
            double m[9];
            int k = 0;
            for (int r = 0; r < 4; ++r) {
                if (r == j) continue;
                for (int q = 0; q < 4; ++q) {
                    if (q == i) continue;
                    m[k++] = a[4 * r + q];
                }
            }
            const double det3 = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
            c[4 * i + j] = ((i + j) & 1) ? -det3 : det3;
        }
    const double det = a[0] * c[0] + a[1] * c[4] + a[2] * c[8] + a[3] * c[12];
    for (int i = 0; i < 16; ++i) out[i] = c[i] / det;
}

/* ------------------------------------------------------------------ A.3 step 7 */
/*
 * ScalableTSDFVolume::Integrate (the volume `TSDF.__init__` literally builds, N/3DM/tsdf.py:7-12:
 * volume_unit_resolution = 32, depth_sampling_stride = 8), restated on a dense box made of whole
 * units: the box origin is unit0 * unit_length (unit_length = voxel_length * unit_res, f64) and
 * nx, ny, nz are multiples of unit_res.  Units outside the box are ignored (the reference's
 * volume is unbounded; the build's is not).
 *   1. points = CreateFromDepthImage(depth f32, K, extrinsic, stride) in world space, f64 (A.2);
 *   2. every unit with index in floor((p - trunc) / unit_length) .. floor((p + trunc) / unit_length)
 *      (inclusive, per axis) is opened and integrated ONCE for this frame;
 *   3. a unit is a UniformTSDFVolume(length = unit_length, resolution = unit_res,
 *      origin = index * unit_length): A.3 steps 2-6 with x, y, z local to the unit.
 * z_restart as in orc_tsdf_integrate (applied to the unit-local z; unit_res is a multiple of 8).
 * touched_out: optional [nux*nuy*nuz] bytes ((ux*nuy + uy)*nuz + uz), 1 = integrated this frame.
 * Threading follows g_scalable_schedule (orc_set_scalable_schedule): 0 = Open3D's own -- the touched
 * units are integrated one after the other and only the x loop INSIDE a unit is an OpenMP
 * `parallel for` (UniformTSDFVolume::IntegrateWithDepthToCameraDistanceMultiplier); 1 = the units
 * themselves are spread over the threads (more parallel than the reference; same result).
 * Returns the number of voxels updated.
 */
static int g_scalable_schedule = 1;
ORC_API void orc_set_scalable_schedule(int s) { g_scalable_schedule = s; }
/* 1: every unit of the box is integrated by every frame (no activation test) -- the "dense box with the reference's
 * per-unit arithmetic" mode of the product (bslam_tsdf_set_unit_activation with stride -1) */
static int g_scalable_all_units = 0;
ORC_API void orc_set_scalable_all_units(int a) { g_scalable_all_units = a; }

ORC_API int64_t orc_scalable_integrate(float *tsdf, float *weight, float *color, int nx, int ny, int nz,
                                       const int *unit0, int unit_res, int stride, double voxel_length,
                                       double sdf_trunc, const float *depth, const uint8_t *rgb, int W, int H,
                                       const double *K, const double *extrinsic, const double *cam_to_world,
                                       int z_restart, uint8_t *touched_out) {
    const int nux = nx / unit_res, nuy = ny / unit_res, nuz = nz / unit_res;
    const double unit_length = voxel_length * (double)unit_res;
    uint8_t *touched = (uint8_t *)calloc((size_t)nux * nuy * nuz, 1);
    if (g_scalable_all_units) {
        memset(touched, 1, (size_t)nux * nuy * nuz);
    } else {
        const double fxd = K[0], fyd = K[1], cxd = K[2], cyd = K[3];
        const double *M = cam_to_world;
        for (int i = 0; i < H; i += stride)
            for (int j = 0; j < W; j += stride) {
                const float p = depth[(size_t)i * W + j];
                if (!(p > 0)) continue;
                const double z = (double)p;
                const double x = (j - cxd) * z / fxd;
                const double y = (i - cyd) * z / fyd;
                double w[3];
                int finite = 1;
                for (int r = 0; r < 3; ++r) {
                    w[r] = ((M[4 * r + 0] * x + M[4 * r + 1] * y) + M[4 * r + 2] * z) + M[4 * r + 3];
                    finite &= isfinite(w[r]) != 0;
                }
                /* not finite: Open3D's (int) conversion gives the INT_MIN unit, outside every box */
                if (!finite) continue;
                const int n[3] = {nux, nuy, nuz};
                int lo[3], hi[3];
                for (int r = 0; r < 3; ++r) {
                    /* floor clamped to +-2^40 before the conversion, offset and clamp to the box in 64 bits: no UB for huge depths */
                    const long long l = (long long)fmin(fmax(floor((w[r] - sdf_trunc) / unit_length), -1099511627776.0), 1099511627776.0) - unit0[r];
                    const long long h = (long long)fmin(fmax(floor((w[r] + sdf_trunc) / unit_length), -1099511627776.0), 1099511627776.0) - unit0[r];
                    lo[r] = (int)(l < 0 ? 0 : (l > n[r] ? n[r] : l));
                    hi[r] = (int)(h > n[r] - 1 ? n[r] - 1 : (h < -1 ? -1 : h));
                }
                for (int ux = lo[0]; ux <= hi[0]; ++ux)
                    for (int uy = lo[1]; uy <= hi[1]; ++uy)
                        for (int uz = lo[2]; uz <= hi[2]; ++uz) touched[((size_t)ux * nuy + uy) * nuz + uz] = 1;
            }
    }
    const float fx = (float)K[0], fy = (float)K[1], cx = (float)K[2], cy = (float)K[3];
    float E[16];
    for (int i = 0; i < 16; ++i) E[i] = (float)extrinsic[i];
    const float vl = (float)voxel_length;
    const float half = vl * 0.5f;
    const float trunc_f = (float)sdf_trunc;
    const float trunc_inv = 1.0f / trunc_f;
    const float dzx = E[2] * vl, dzy = E[6] * vl, dzz = E[10] * vl;
    const float safe_w = W - 0.0001f, safe_h = H - 0.0001f;
    const float fxi = 1.0f / fx, fyi = 1.0f / fy;
    int64_t updated = 0;
    const int n_units = nux * nuy * nuz;
    const int par_units = g_scalable_schedule != 0;
#pragma omp parallel for schedule(dynamic) reduction(+ : updated) if (par_units)
    for (int u = 0; u < n_units; ++u) {
        if (!touched[u]) continue;
        const int uz = u % nuz, uy = (u / nuz) % nuy, ux = u / (nuz * nuy);
        const double org[3] = {(double)(unit0[0] + ux) * unit_length, (double)(unit0[1] + uy) * unit_length,
                               (double)(unit0[2] + uz) * unit_length};
#pragma omp parallel for schedule(static) reduction(+ : updated) if (!par_units)
        for (int x = 0; x < unit_res; ++x)
            for (int y = 0; y < unit_res; ++y) {
                const float px = (float)((double)(half + vl * (float)x) + org[0]);
                const float py = (float)((double)(half + vl * (float)y) + org[1]);
                float pcx = 0.f, pcy = 0.f, pcz = 0.f;
                for (int z = 0; z < unit_res; ++z) {
                    if (z == 0 || (z_restart > 0 && z % z_restart == 0)) {
                        const float pz = (float)((double)(half + vl * (float)z) + org[2]);
                        pcx = ((E[0] * px + E[1] * py) + E[2] * pz) + E[3];
                        pcy = ((E[4] * px + E[5] * py) + E[6] * pz) + E[7];
                        pcz = ((E[8] * px + E[9] * py) + E[10] * pz) + E[11];
                    }
                    const float cxp = pcx, cyp = pcy, czp = pcz;
                    pcx += dzx; pcy += dzy; pcz += dzz;
                    if (czp <= 0) continue;
                    const float u_f = cxp * fx / czp + cx + 0.5f;
                    const float v_f = cyp * fy / czp + cy + 0.5f;
                    if (!(u_f >= 0.0001f && u_f < safe_w && v_f >= 0.0001f && v_f < safe_h)) continue;
                    const int uu = (int)u_f, vv = (int)v_f;
                    const float d = depth[(size_t)vv * W + uu];
                    if (d <= 0.0f) continue;
                    const float xx = ((float)uu - cx) * fxi, yy = ((float)vv - cy) * fyi;
                    const float mult = sqrtf((xx * xx + yy * yy) + 1.0f);
                    const float sdf = (d - czp) * mult;
                    if (sdf > -trunc_f) {
                        const size_t idx = ((size_t)(ux * unit_res + x) * ny + (uy * unit_res + y)) * nz + (uz * unit_res + z);
                        const float t = fminf(1.0f, sdf * trunc_inv);
                        const float w = weight[idx];
                        if (color && rgb) {
                            const uint8_t *c = rgb + ((size_t)vv * W + uu) * 3;
                            for (int k = 0; k < 3; ++k) color[3 * idx + k] = (color[3 * idx + k] * w + (float)c[k]) / (w + 1.0f);
                        }
                        tsdf[idx] = (tsdf[idx] * w + t) / (w + 1.0f);
                        weight[idx] = w + 1.0f;
                        ++updated;
                    }
                }
            }
    }
    if (touched_out) memcpy(touched_out, touched, (size_t)n_units);
    free(touched);
    return updated;
}

/* Surface-extraction flavour (row f4): a voxel is valid when weight >= g_w_thr (0: the legacy rule weight != 0),
 * vertices / points sit at (index + g_pos_half) * voxel_length.  Legacy Open3D: 0 / 0.5; the tensor pipeline behind
 * `MAP` (N/3DM/tsdf.py:85-89: voxel_grid.extract_triangle_mesh() / extract_point_cloud(), weight_threshold = 3): 3 / 0. */
static float g_w_thr = 0.0f;
static double g_pos_half = 0.5;
ORC_API void orc_set_extract_flavour(double weight_threshold, double pos_half) { g_w_thr = (float)weight_threshold; g_pos_half = pos_half; }
static int orc_valid_w(float w) { return g_w_thr > 0.0f ? (w >= g_w_thr) : (w != 0.0f); }

/* ------------------------------------------------------------------ A.4 */
typedef struct {
    uint64_t *keys;
    int32_t *vals;
    size_t cap, n;
} orc_map;

static void map_init(orc_map *m, size_t cap) {
    m->cap = cap; m->n = 0;
    m->keys = (uint64_t *)malloc(cap * sizeof(uint64_t));
    m->vals = (int32_t *)malloc(cap * sizeof(int32_t));
    memset(m->keys, 0xff, cap * sizeof(uint64_t));
}
static size_t map_slot(const orc_map *m, uint64_t k) {
    uint64_t h = k * 0x9E3779B97F4A7C15ull;
    size_t i = (size_t)(h >> 20) & (m->cap - 1);
    while (m->keys[i] != UINT64_MAX && m->keys[i] != k) i = (i + 1) & (m->cap - 1);
    return i;
}
static void map_grow(orc_map *m) {
    orc_map n; map_init(&n, m->cap * 2);
    for (size_t i = 0; i < m->cap; ++i)
        if (m->keys[i] != UINT64_MAX) {
            size_t s = map_slot(&n, m->keys[i]);
            n.keys[s] = m->keys[i]; n.vals[s] = m->vals[i]; n.n++;
        }
    free(m->keys); free(m->vals); *m = n;
}

/*
 * Serial marching cubes over cubes based at x in [0,nx-2], y in [0,ny-2], z in [0,nz-2]
 * (x outer, z inner).  Vertices are shared through the edge key (x,y,z,axis) and
 * numbered in first-seen order; triangles are (e[t0], e[t2], e[t1]).
 * Outputs (capacity cap_v / cap_t rows; rows beyond capacity are counted, not written):
 *   out_v   [V,3] f64 world position,   out_key [V,4] i32 (x,y,z,axis) local voxel coords,
 *   out_c   [V,3] f64 colour in [0,1] (if color != NULL), out_t [T,3] i32,
 *   out_tz  [T] i32 local z of the emitting cube (optional; lets tests split a mesh into z-slabs).
 * counts[0] = V, counts[1] = T.
 */
ORC_API void orc_extract_mesh(const float *tsdf, const float *weight, const float *color, int nx,
                              int ny, int nz, int gz0, double voxel_length, const double *origin,
                              double *out_v, int32_t *out_key, double *out_c, int64_t cap_v,
                              int32_t *out_t, int32_t *out_tz, int64_t cap_t, int64_t *counts) {
    const double half = voxel_length * g_pos_half;
    orc_map map; map_init(&map, 1u << 16);
    int64_t nv = 0, nt = 0;
    for (int x = 0; x < nx - 1; ++x)
        for (int y = 0; y < ny - 1; ++y)
            for (int z = 0; z < nz - 1; ++z) {
                int cube_index = 0, ok = 1;
                float f[8]; size_t id[8];
                for (int i = 0; i < 8; ++i) {
                    id[i] = ((size_t)(x + orc_shift[i][0]) * ny + (y + orc_shift[i][1])) * nz + (z + orc_shift[i][2]);
                    if (!orc_valid_w(weight[id[i]])) { ok = 0; break; }
                    f[i] = tsdf[id[i]];
                    if (f[i] < 0.0f) cube_index |= (1 << i);
                }
                if (!ok || cube_index == 0 || cube_index == 255) continue;
                const int em = orc_edge_table(cube_index);
                int32_t e2v[12];
                for (int e = 0; e < 12; ++e) {
                    e2v[e] = -1;
                    if (!(em & (1 << e))) continue;
                    const int ex = x + orc_edge_shift[e][0], ey = y + orc_edge_shift[e][1],
                              ez = z + orc_edge_shift[e][2], ax = orc_edge_shift[e][3];
                    const uint64_t key = ((((uint64_t)ex * (uint64_t)ny + (uint64_t)ey) * (uint64_t)nz + (uint64_t)ez) << 2) | (uint64_t)ax;
                    size_t s = map_slot(&map, key);
                    if (map.keys[s] == UINT64_MAX) {
                        if ((map.n + 1) * 2 > map.cap) { map_grow(&map); s = map_slot(&map, key); }
                        map.keys[s] = key; map.vals[s] = (int32_t)nv; map.n++;
                        const int i0 = orc_edge_to_vert[e][0], i1 = orc_edge_to_vert[e][1];
                        const double f0 = fabs((double)f[i0]), f1 = fabs((double)f[i1]);
                        if (nv < cap_v) {
                            double pt[3] = {half + voxel_length * ex, half + voxel_length * ey,
                                            half + voxel_length * (ez + gz0)};
                            pt[ax] += f0 * voxel_length / (f0 + f1);
                            for (int k = 0; k < 3; ++k) out_v[3 * nv + k] = pt[k] + origin[k];
                            out_key[4 * nv + 0] = ex; out_key[4 * nv + 1] = ey;
                            out_key[4 * nv + 2] = ez; out_key[4 * nv + 3] = ax;
                            if (color && out_c)
                                for (int k = 0; k < 3; ++k)
                                    out_c[3 * nv + k] = ((f1 * (double)color[3 * id[i0] + k] + f0 * (double)color[3 * id[i1] + k]) / (f0 + f1)) / 255.0;
                        }
                        e2v[e] = (int32_t)nv++;
                    } else {
                        e2v[e] = map.vals[s];
                    }
                }
                for (int i = 0; orc_tri_table[cube_index][i] != -1; i += 3) {
                    if (nt < cap_t) {
                        out_t[3 * nt + 0] = e2v[orc_tri_table[cube_index][i]];
                        out_t[3 * nt + 1] = e2v[orc_tri_table[cube_index][i + 2]];
                        out_t[3 * nt + 2] = e2v[orc_tri_table[cube_index][i + 1]];
                        if (out_tz) out_tz[nt] = z; /* local z of the cube that emitted the triangle */
                    }
                    ++nt;
                }
            }
    free(map.keys); free(map.vals);
    counts[0] = nv; counts[1] = nt;
}

/* ------------------------------------------------------------------ A.5 */
static double tsdf_at(const float *tsdf, int ny, int nz, double voxel_length, const double *p) {
    int idx[3]; double r[3];
    for (int i = 0; i < 3; ++i) {
        const double g = p[i] / voxel_length - g_pos_half;
        idx[i] = (int)floor(g);
        r[i] = g - (double)idx[i];
    }
#define TS(a, b, c) ((double)tsdf[((size_t)(idx[0] + a) * ny + (idx[1] + b)) * nz + (idx[2] + c)])
    double t = 0;
    t += (1 - r[0]) * (1 - r[1]) * (1 - r[2]) * TS(0, 0, 0);
    t += (1 - r[0]) * (1 - r[1]) * r[2] * TS(0, 0, 1);
    t += (1 - r[0]) * r[1] * (1 - r[2]) * TS(0, 1, 0);
    t += (1 - r[0]) * r[1] * r[2] * TS(0, 1, 1);
    t += r[0] * (1 - r[1]) * (1 - r[2]) * TS(1, 0, 0);
    t += r[0] * (1 - r[1]) * r[2] * TS(1, 0, 1);
    t += r[0] * r[1] * (1 - r[2]) * TS(1, 1, 0);
    t += r[0] * r[1] * r[2] * TS(1, 1, 1);
#undef TS
    return t;
}

/*
 * Surface points: interior voxels x,y,z in [1, n-2] (serial x,y,z order, then axis).
 * Local coordinates are relative to the box (single-box volumes only: gz0 shifts the
 * emitted position, the trilinear normal lookup stays inside the box).
 * out_p [P,3] f64, out_n [P,3] f64 (unit normal, 0.99*voxel central difference of the
 * trilinear TSDF at the point), out_c [P,3] f64 if color != NULL, out_key [P,4] i32.
 */
ORC_API int64_t orc_extract_points(const float *tsdf, const float *weight, const float *color,
                                   int nx, int ny, int nz, int gz0, double voxel_length,
                                   const double *origin, double *out_p, double *out_n,
                                   double *out_c, int32_t *out_key, int64_t cap) {
    const double half = voxel_length * g_pos_half;
    const double half_gap = 0.99 * voxel_length;
    const int n[3] = {nx, ny, nz};
    int64_t np = 0;
    for (int x = 1; x < nx - 1; ++x)
        for (int y = 1; y < ny - 1; ++y)
            for (int z = 1; z < nz - 1; ++z) {
                const int idx0[3] = {x, y, z};
                const size_t i0 = ((size_t)x * ny + y) * nz + z;
                const float w0 = weight[i0], f0 = tsdf[i0];
                if (!(orc_valid_w(w0) && f0 < 0.98f && f0 >= -0.98f)) continue;
                const double p0[3] = {half + voxel_length * x, half + voxel_length * y, half + voxel_length * z};
                for (int i = 0; i < 3; ++i) {
                    int idx1[3] = {x, y, z};
                    idx1[i] += 1;
                    if (!(idx1[i] < n[i] - 1)) continue;
                    const size_t i1 = ((size_t)idx1[0] * ny + idx1[1]) * nz + idx1[2];
                    const float w1 = weight[i1], f1 = tsdf[i1];
                    if (!(orc_valid_w(w1) && f1 < 0.98f && f1 >= -0.98f && f0 * f1 < 0)) continue;
                    const float r0 = fabsf(f0), r1 = fabsf(f1);
                    double p[3] = {p0[0], p0[1], p0[2]};
                    const double p1i = p0[i] + voxel_length;
                    p[i] = (p0[i] * r1 + p1i * r0) / (r0 + r1);
                    if (np < cap) {
                        for (int k = 0; k < 3; ++k) out_p[3 * np + k] = p[k] + origin[k];
                        out_p[3 * np + 2] += voxel_length * gz0;
                        if (color && out_c)
                            for (int k = 0; k < 3; ++k)
                                out_c[3 * np + k] = (((double)color[3 * i0 + k] * r1 + (double)color[3 * i1 + k] * r0) / (r0 + r1)) / 255.0;
                        if (out_n) {
                            double nn[3];
                            for (int k = 0; k < 3; ++k) {
                                double q0[3] = {p[0], p[1], p[2]}, q1[3] = {p[0], p[1], p[2]};
                                q0[k] -= half_gap; q1[k] += half_gap;
                                nn[k] = tsdf_at(tsdf, ny, nz, voxel_length, q1) - tsdf_at(tsdf, ny, nz, voxel_length, q0);
                            }
                            const double len = sqrt(nn[0] * nn[0] + nn[1] * nn[1] + nn[2] * nn[2]);
                            for (int k = 0; k < 3; ++k) out_n[3 * np + k] = len > 0 ? nn[k] / len : nn[k];
                        }
                        if (out_key) {
                            out_key[4 * np + 0] = idx0[0]; out_key[4 * np + 1] = idx0[1];
                            out_key[4 * np + 2] = idx0[2]; out_key[4 * np + 3] = i;
                        }
                    }
                    ++np;
                }
            }
    return np;
}

/* ------------------------------------------------------------------ A.6 (row f4)
 * `MAP.integrate` (N/3DM/tsdf.py:71-83) = Open3D t.pipelines.slam.Model.integrate on a VoxelBlockGrid of 16^3 blocks,
 * restated on a bounded dense box whose origin is block0 * block_size (block_size = 16 * voxel_size); PARITY UNPINNED
 * (written from knowledge of Open3D's VoxelBlockGridImpl.h: DepthTouch + Integrate; float32 tsdf / weight / colour).
 *   pose         camera -> world 4x4 f64 (T_frame_to_model); the extrinsic is its rigid inverse (f64), cast to
 *                float with the rotation entries pre-multiplied by voxel_size (TransformIndexer(.., voxel_size))
 *   touch        every 4th pixel, d = (float)u16 / depth_scale, 0 < d < depth_max: ray through Unproject(x, y, 1)
 *                and the pose; blocks at t = t_min + k * (t_max - t_min) / 3, k = 0..3
 *   integrate    voxel position = integer voxel coordinate (world grid) as float; u = fx * x * (1/z) + cx, truncation;
 *                sdf = depth - z (projective); skip depth <= 0, depth > depth_max, z <= 0, sdf < -trunc;
 *                tsdf = (w * tsdf + min(sdf, trunc) / trunc) * (1 / (w + 1)); colour alike; w += 1
 * touched_out: optional [nbx*nby*nbz] bytes ((xb * nby + yb) * nbz + zb).  Returns the number of voxels updated.
 */
ORC_API int64_t orc_vbg_integrate(float *tsdf, float *weight, float *color, int nx, int ny, int nz, const int *block0,
                                  double voxel_size, double trunc_voxel_multiplier, const uint16_t *depth, const uint8_t *rgb,
                                  int W, int H, const double *K, const double *pose, double depth_scale_d, double depth_max_d,
                                  uint8_t *touched_out) {
    const int B = 16;
    const int nbx = (nx + B - 1) / B, nby = (ny + B - 1) / B, nbz = (nz + B - 1) / B;
    const float fx = (float)K[0], fy = (float)K[1], cx = (float)K[2], cy = (float)K[3];
    const float vs = (float)voxel_size, depth_scale = (float)depth_scale_d, depth_max = (float)depth_max_d;
    const float trunc = vs * (float)trunc_voxel_multiplier, block_size = vs * (float)B;
    double E[12];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) E[4 * i + j] = pose[4 * j + i];
        E[4 * i + 3] = -(pose[4 * 0 + i] * pose[3] + pose[4 * 1 + i] * pose[7] + pose[4 * 2 + i] * pose[11]);
    }
    float Es[12], P[12];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) Es[4 * i + j] = (float)E[4 * i + j] * vs;
        Es[4 * i + 3] = (float)E[4 * i + 3];
    }
    for (int i = 0; i < 12; ++i) P[i] = (float)pose[i];
    uint8_t *touched = (uint8_t *)calloc((size_t)nbx * nby * nbz, 1);
    for (int y = 0; y + 0 < (H / 4) * 4; y += 4)
        for (int x = 0; x < (W / 4) * 4; x += 4) {
            const float d = (float)depth[(size_t)y * W + x] / depth_scale;
            if (!(d > 0.0f && d < depth_max)) continue;
            const float xc = ((float)x - cx) * 1.0f / fx, yc = ((float)y - cy) * 1.0f / fy, zc = 1.0f;
            const float xg = ((xc * P[0] + yc * P[1]) + zc * P[2]) + P[3];
            const float yg = ((xc * P[4] + yc * P[5]) + zc * P[6]) + P[7];
            const float zg = ((xc * P[8] + yc * P[9]) + zc * P[10]) + P[11];
            const float xo = P[3], yo = P[7], zo = P[11];
            const float xd = xg - xo, yd = yg - yo, zd = zg - zo;
            const float t_min = fmaxf(d - trunc, 0.0f), t_max = fminf(d + trunc, depth_max);
            const float t_step = (t_max - t_min) / 3.0f;
            float t = t_min;
            for (int step = 0; step <= 3; ++step) {
                const int xb = (int)floorf((xo + t * xd) / block_size) - block0[0];
                const int yb = (int)floorf((yo + t * yd) / block_size) - block0[1];
                const int zb = (int)floorf((zo + t * zd) / block_size) - block0[2];
                if (xb >= 0 && yb >= 0 && zb >= 0 && xb < nbx && yb < nby && zb < nbz) touched[((size_t)xb * nby + yb) * nbz + zb] = 1;
                t += t_step;
            }
        }
    int64_t updated = 0;
    const int n_blocks = nbx * nby * nbz;
#pragma omp parallel for schedule(dynamic) reduction(+ : updated)
    for (int b = 0; b < n_blocks; ++b) {
        if (!touched[b]) continue;
        const int zb = b % nbz, yb = (b / nbz) % nby, xb = b / (nbz * nby);
        for (int lx = 0; lx < B; ++lx)
            for (int ly = 0; ly < B; ++ly)
                for (int lz = 0; lz < B; ++lz) {
                    const int X = xb * B + lx, Y = yb * B + ly, Z = zb * B + lz;
                    if (X >= nx || Y >= ny || Z >= nz) continue;
                    const float xw = (float)(block0[0] * B + X), yw = (float)(block0[1] * B + Y), zw = (float)(block0[2] * B + Z);
                    const float xc = ((xw * Es[0] + yw * Es[1]) + zw * Es[2]) + Es[3];
                    const float yc = ((xw * Es[4] + yw * Es[5]) + zw * Es[6]) + Es[7];
                    const float zc = ((xw * Es[8] + yw * Es[9]) + zw * Es[10]) + Es[11];
                    const float inv_z = 1.0f / zc;
                    const float u = fx * xc * inv_z + cx, v = fy * yc * inv_z + cy;
                    if (!(u >= 0.0f && v >= 0.0f && u < (float)W && v < (float)H)) continue;
                    const int ui = (int)u, vi = (int)v;
                    const float d = (float)depth[(size_t)vi * W + ui] / depth_scale;
                    float sdf = d - zc;
                    if (d <= 0.0f || d > depth_max || zc <= 0.0f || sdf < -trunc) continue;
                    sdf = sdf < trunc ? sdf : trunc;
                    sdf /= trunc;
                    const size_t idx = ((size_t)X * ny + Y) * nz + Z;
                    const float w = weight[idx];
                    const float inv = 1.0f / (w + 1.0f);
                    tsdf[idx] = (w * tsdf[idx] + sdf) * inv;
                    if (color && rgb) {
                        const uint8_t *c = rgb + ((size_t)vi * W + ui) * 3;
                        for (int k = 0; k < 3; ++k) color[3 * idx + k] = (w * color[3 * idx + k] + (float)c[k]) * inv;
                    }
                    weight[idx] = w + 1.0f;
                    ++updated;
                }
    }
    if (touched_out) memcpy(touched_out, touched, (size_t)n_blocks);
    free(touched);
    return updated;
}

/* occupancy helper for the parity tests: number of voxels with weight != 0 */
ORC_API int64_t orc_count_occupied(const float *weight, size_t n) {
    int64_t c = 0;
    for (size_t i = 0; i < n; ++i) c += weight[i] != 0.0f;
    return c;
}
