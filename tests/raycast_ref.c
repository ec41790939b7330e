/*
 * tests/raycast_ref.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE: the CPU reference of the ray cast
 * (csrc/bslam_raycast.cu must match it bit for bit).  Built by tests/raycast_ref.py with
 * -ffp-contract=off, like the oracle library: this file DEFINES the order of floating point operations.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define REF_API __attribute__((visibility("default")))

/* Ray cast (row f4 + legacy volumes)
 * `t.pipelines.slam.Model.synthesize_model_frame` = VoxelBlockGrid::RayCast after EstimateRange, restated from knowledge
 * of Open3D's VoxelBlockGridImpl.h (RayCastCPU / EstimateRangeCPU), in the style of oracle/o3d_oracle.c.  PARITY WITH
 * OPEN3D UNPINNED: no Open3D output is recorded for it.  Grids (tsdf, weight, colour [.., 3]) are dense nx*ny*nz boxes in
 * Open3D order idx = (x*ny + y)*nz + z, as the oracle's Volume keeps them.  One call = one frame.  flavour 1 (tensor, `MAP`): 16^3 blocks on the world block grid (box origin = block0 * 16 *
 * voxel), samples on voxel corners; flavour 0 (legacy dense box, `DenseTSDFVolume`): 8^3 bricks relative to the float
 * origin, samples at voxel centres (the trilinear part uses index + 0.5).  Box dims must be multiples of the block edge.
 * Per ray (integer pixel x, y, no +0.5; pose and intrinsics narrowed to float):
 *   dir = P * Unproject(x, y, 1) - o (vbg_touch's operation order), o = translation of P (camera -> world);
 *   [t, t_max] = range of the ray; t >= t_max: miss;  t_prev = t, tsdf_prev = -1, tsdf = 1;
 *   march: p = o + t * dir;  block of p outside the box or unallocated: t_prev = t, t += block_len;  else tsdf_prev = tsdf,
 *     (tsdf, w) = voxel holding p;  tsdf_prev > 0 && valid(w) && tsdf <= 0: hit;  t_prev = t, t += max(tsdf * sdf_trunc, voxel);
 *   hit: t_i = (t * tsdf_prev - t_prev * tsdf) / (tsdf_prev - tsdf), depth = t_i * depth_scale, p_i = o + t_i * dir,
 *     vertex = E * p_i (camera frame); over the 8 trilinear corners k of p_i with weight > 0 (and in the box / allocated):
 *     colour = sum r_k c_k / (255 sum r_k), normal = normalise(sum r_k grad_k) rotated by E, grad_k = central tsdf
 *     differences at corner k, a component dropped when a neighbour is outside the box or unallocated;
 *   miss: all outputs 0.
 * Deliberate choices of this restatement:
 *   - valid(w): w >= thr for thr > 0, w != 0 for thr == 0 (the oracle's orc_valid_w); Open3D accepts w = 0 samples at threshold 0;
 *   - the in-block voxel index is clamped to block_edge - 1: rounding of (p - b * block_len) / voxel can give
 *     block_edge, where Open3D would index past the block;
 *   - "normalise" divides by sqrtf(|n|^2) when it is > 0 (no epsilon);
 *   - tensor flavour: "allocated" = every block activated by any frame so far (`allocated`, the hash map's blocks);
 *     the range comes from EstimateRange with down factor 8 over the blocks the LAST frame activated (`range_blocks`):
 *     per block, the 8 world corners through the float world -> camera transform (corners with z <= 0 skipped),
 *     u = fx * x * (1 / z) + cx, / 8, box = floor / ceil clamped to the down-sampled image (initial u_min = w/8 - 1,
 *     u_max = 0, likewise v), z_min = min(depth_max, z), z_max = max(depth_min, z), degenerate boxes dropped; every cell
 *     starts at [depth_max, depth_min]; ray (x, y) reads cell (min(x/8, w/8 - 1), min(y/8, h/8 - 1));
 *   - legacy flavour: Open3D's legacy volumes have no ray cast; the range is [depth_min, depth_max] for every ray and
 *     "allocated" = the brick holds a weight != 0 (the product's brick flag bit 0, equivalent for integrated volumes);
 *     the extrinsic's rigid inverse (f64) is the pose.
 * `pose_or_extrinsic`: 4x4 f64, camera -> world for flavour 1, world -> camera for flavour 0.  `sdf_trunc`: flavour 1
 * takes the trunc_voxel_multiplier (sdf_trunc = (float)voxel * (float)multiplier, as the integrator).  Outputs [H*W] / [H*W*3]
 * f32, each optional except depth.  Returns the number of voxel samples the march read (all rays).
 */
static void rigid_inverse(const double *A, double *out) {
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) out[4 * i + j] = A[4 * j + i];
        out[4 * i + 3] = -(A[4 * 0 + i] * A[3] + A[4 * 1 + i] * A[7] + A[4 * 2 + i] * A[11]);
    }
}

typedef struct {
    const float *tsdf, *weight, *color;
    const uint8_t *alloc;   /* per block ((xb * nby + yb) * nbz + zb) */
    int n[3], nb[3], b0[3], B;
    float vl, bl, half, org[3];
} rc_vol;

static int rc_alloc(const rc_vol *v, int X, int Y, int Z) {
    if (X < 0 || Y < 0 || Z < 0 || X >= v->n[0] || Y >= v->n[1] || Z >= v->n[2]) return 0;
    return v->alloc[((size_t)(X / v->B) * v->nb[1] + Y / v->B) * v->nb[2] + Z / v->B];
}
static size_t rc_idx(const rc_vol *v, int X, int Y, int Z) { return ((size_t)X * v->n[1] + Y) * v->n[2] + Z; }

REF_API int64_t ref_raycast(const float *tsdf, const float *weight, const float *color, int nx, int ny, int nz, double voxel_length,
                            double sdf_trunc, const double *origin, int flavour, const uint8_t *allocated, const uint8_t *range_blocks,
                            int W, int H, const double *K, const double *pose_or_extrinsic, double depth_scale_d, double depth_min_d,
                            double depth_max_d, double weight_threshold, float *out_depth, float *out_vertex, float *out_normal,
                            float *out_color) {
    rc_vol v;
    v.tsdf = tsdf; v.weight = weight; v.color = color;
    v.n[0] = nx; v.n[1] = ny; v.n[2] = nz;
    v.B = flavour ? 16 : 8;
    v.vl = (float)voxel_length;
    v.bl = v.vl * (float)v.B;
    v.half = flavour ? 0.0f : 0.5f;
    for (int r = 0; r < 3; ++r) v.nb[r] = v.n[r] / v.B;
    uint8_t *alloc_legacy = NULL;
    if (flavour) {
        const double bs = voxel_length * 16.0;
        for (int r = 0; r < 3; ++r) { v.b0[r] = (int)nearbyint(origin[r] / bs); v.org[r] = 0.0f; }
        v.alloc = allocated;
    } else {
        for (int r = 0; r < 3; ++r) { v.b0[r] = 0; v.org[r] = (float)origin[r]; }
        const size_t nbt = (size_t)v.nb[0] * v.nb[1] * v.nb[2];
        alloc_legacy = (uint8_t *)calloc(nbt, 1);
        for (int X = 0; X < nx; ++X)
            for (int Y = 0; Y < ny; ++Y)
                for (int Z = 0; Z < nz; ++Z)
                    if (weight[rc_idx(&v, X, Y, Z)] != 0.0f) alloc_legacy[((size_t)(X / 8) * v.nb[1] + Y / 8) * v.nb[2] + Z / 8] = 1;
        v.alloc = alloc_legacy;
    }
    double P[12], E[12];
    if (flavour) { for (int i = 0; i < 12; ++i) P[i] = pose_or_extrinsic[i]; rigid_inverse(pose_or_extrinsic, E); }
    else { for (int i = 0; i < 12; ++i) E[i] = pose_or_extrinsic[i]; rigid_inverse(pose_or_extrinsic, P); }
    float Pf[12], Ef[12];
    for (int i = 0; i < 12; ++i) { Pf[i] = (float)P[i]; Ef[i] = (float)E[i]; }
    const float fx = (float)K[0], fy = (float)K[1], cx = (float)K[2], cy = (float)K[3];
    const float depth_scale = (float)depth_scale_d, depth_min = (float)depth_min_d, depth_max = (float)depth_max_d;
    const float thr = (float)weight_threshold, trunc = flavour ? v.vl * (float)sdf_trunc : (float)sdf_trunc;

    /* range map (tensor flavour) */
    const int wd = W / 8, hd = H / 8;
    float *range = NULL;
    if (flavour) {
        range = (float *)malloc((size_t)(wd > 0 ? wd : 1) * (hd > 0 ? hd : 1) * 2 * sizeof(float));
        for (int i = 0; i < wd * hd; ++i) { range[2 * i] = depth_max; range[2 * i + 1] = depth_min; }
        for (int xb = 0; xb < v.nb[0]; ++xb)
            for (int yb = 0; yb < v.nb[1]; ++yb)
                for (int zb = 0; zb < v.nb[2]; ++zb) {
                    if (!range_blocks[((size_t)xb * v.nb[1] + yb) * v.nb[2] + zb]) continue;
                    const int key[3] = {v.b0[0] + xb, v.b0[1] + yb, v.b0[2] + zb};
                    int u_min = wd - 1, v_min = hd - 1, u_max = 0, v_max = 0;
                    float z_min = depth_max, z_max = depth_min;
                    for (int i = 0; i < 8; ++i) {
                        const float xw = (float)(key[0] + ((i & 1) > 0)) * v.bl;
                        const float yw = (float)(key[1] + ((i & 2) > 0)) * v.bl;
                        const float zw = (float)(key[2] + ((i & 4) > 0)) * v.bl;
                        const float xc = ((Ef[0] * xw + Ef[1] * yw) + Ef[2] * zw) + Ef[3];
                        const float yc = ((Ef[4] * xw + Ef[5] * yw) + Ef[6] * zw) + Ef[7];
                        const float zc = ((Ef[8] * xw + Ef[9] * yw) + Ef[10] * zw) + Ef[11];
                        if (zc <= 0.0f) continue;
                        const float inv_z = 1.0f / zc;
                        const float u = (fx * xc * inv_z + cx) / 8.0f, vv = (fy * yc * inv_z + cy) / 8.0f;
                        const int vf = (int)floorf(vv), vc = (int)ceilf(vv), uf = (int)floorf(u), uc = (int)ceilf(u);
                        if (vf < v_min) v_min = vf;
                        if (vc > v_max) v_max = vc;
                        if (uf < u_min) u_min = uf;
                        if (uc > u_max) u_max = uc;
                        z_min = fminf(z_min, zc);
                        z_max = fmaxf(z_max, zc);
                    }
                    if (v_min < 0) v_min = 0;
                    if (v_max > hd - 1) v_max = hd - 1;
                    if (u_min < 0) u_min = 0;
                    if (u_max > wd - 1) u_max = wd - 1;
                    if (v_min >= v_max || u_min >= u_max || z_min >= z_max) continue;
                    for (int y = v_min; y <= v_max; ++y)
                        for (int x = u_min; x <= u_max; ++x) {
                            float *r = range + 2 * ((size_t)y * wd + x);
                            r[0] = fminf(r[0], z_min);
                            r[1] = fmaxf(r[1], z_max);
                        }
                }
    }

    int64_t samples = 0;
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : samples)
    for (int y = 0; y < H; ++y)
        for (int x = 0; x < W; ++x) {
            const size_t pix = (size_t)y * W + x;
            out_depth[pix] = 0.0f;
            for (int k = 0; k < 3; ++k) {
                if (out_vertex) out_vertex[3 * pix + k] = 0.0f;
                if (out_normal) out_normal[3 * pix + k] = 0.0f;
                if (out_color) out_color[3 * pix + k] = 0.0f;
            }
            float t = depth_min, t_max = depth_max;
            if (flavour) {
                const int cxi = x / 8 < wd - 1 ? x / 8 : wd - 1, cyi = y / 8 < hd - 1 ? y / 8 : hd - 1;
                t = range[2 * ((size_t)cyi * wd + cxi)];
                t_max = range[2 * ((size_t)cyi * wd + cxi) + 1];
            }
            if (t >= t_max) continue;
            const float xc = ((float)x - cx) * 1.0f / fx, yc = ((float)y - cy) * 1.0f / fy, zc = 1.0f;
            const float o[3] = {Pf[3], Pf[7], Pf[11]};
            float d[3];
            for (int r = 0; r < 3; ++r) d[r] = (((xc * Pf[4 * r] + yc * Pf[4 * r + 1]) + zc * Pf[4 * r + 2]) + Pf[4 * r + 3]) - o[r];
            float t_prev = t, tsdf_prev = -1.0f, ts = 1.0f;
            int hit = 0;
            while (t < t_max) {
                int Xv[3], in = 1;
                for (int r = 0; r < 3; ++r) {
                    const float q = (o[r] + t * d[r]) - v.org[r];
                    const float bw = floorf(q / v.bl);
                    int l = (int)((q - bw * v.bl) / v.vl);
                    if (l > v.B - 1) l = v.B - 1;
                    const int b = (int)bw - v.b0[r];
                    if (b < 0 || b >= v.nb[r]) in = 0;
                    Xv[r] = b * v.B + l;
                }
                if (!in || !rc_alloc(&v, Xv[0], Xv[1], Xv[2])) { t_prev = t; t += v.bl; continue; }
                const size_t i = rc_idx(&v, Xv[0], Xv[1], Xv[2]);
                tsdf_prev = ts;
                ts = tsdf[i];
                const float w = weight[i];
                ++samples;
                if (tsdf_prev > 0.0f && (thr > 0.0f ? w >= thr : w != 0.0f) && ts <= 0.0f) { hit = 1; break; }
                t_prev = t;
                const float delta = ts * trunc;
                t += delta < v.vl ? v.vl : delta;
            }
            if (!hit) continue;
            const float ti = (t * tsdf_prev - t_prev * ts) / (tsdf_prev - ts);
            out_depth[pix] = ti * depth_scale;
            float p[3];
            for (int r = 0; r < 3; ++r) p[r] = o[r] + ti * d[r];
            if (out_vertex)
                for (int r = 0; r < 3; ++r) out_vertex[3 * pix + r] = ((Ef[4 * r] * p[0] + Ef[4 * r + 1] * p[1]) + Ef[4 * r + 2] * p[2]) + Ef[4 * r + 3];
            if (!out_normal && !out_color) continue;
            int base[3];
            float xv[3];
            for (int r = 0; r < 3; ++r) {
                const float q = p[r] - v.org[r];
                const float bw = floorf(q / v.bl);
                xv[r] = (q - bw * v.bl) / v.vl - v.half;
                const float fl = floorf(xv[r]);
                base[r] = ((int)bw - v.b0[r]) * v.B + (int)fl;
                xv[r] -= fl;      /* position relative to the corner base */
            }
            float sum_r = 0.0f, nacc[3] = {0.f, 0.f, 0.f}, cacc[3] = {0.f, 0.f, 0.f};
            for (int k = 0; k < 8; ++k) {
                const int dk[3] = {k & 1, (k >> 1) & 1, (k >> 2) & 1};
                const int X = base[0] + dk[0], Y = base[1] + dk[1], Z = base[2] + dk[2];
                if (!rc_alloc(&v, X, Y, Z)) continue;
                const size_t ik = rc_idx(&v, X, Y, Z);
                if (!(weight[ik] > 0.0f)) continue;
                const float r = ((1.0f - fabsf((float)dk[0] - xv[0])) * (1.0f - fabsf((float)dk[1] - xv[1]))) * (1.0f - fabsf((float)dk[2] - xv[2]));
                sum_r += r;
                if (out_normal) {
                    const int C0[3] = {X, Y, Z};
                    for (int a = 0; a < 3; ++a) {
                        int lo[3] = {C0[0], C0[1], C0[2]}, hi[3] = {C0[0], C0[1], C0[2]};
                        lo[a] -= 1; hi[a] += 1;
                        float g = 0.0f;
                        if (rc_alloc(&v, lo[0], lo[1], lo[2]) && rc_alloc(&v, hi[0], hi[1], hi[2]))
                            g = tsdf[rc_idx(&v, hi[0], hi[1], hi[2])] - tsdf[rc_idx(&v, lo[0], lo[1], lo[2])];
                        nacc[a] += r * g;
                    }
                }
                if (out_color && color)
                    for (int c = 0; c < 3; ++c) cacc[c] += r * color[3 * ik + c];
            }
            if (!(sum_r > 0.0f)) continue;
            if (out_color && color) {
                const float s = sum_r * 255.0f;
                for (int c = 0; c < 3; ++c) out_color[3 * pix + c] = cacc[c] / s;
            }
            if (out_normal) {
                const float n2 = (nacc[0] * nacc[0] + nacc[1] * nacc[1]) + nacc[2] * nacc[2];
                if (n2 > 0.0f) {
                    const float len = sqrtf(n2);
                    const float n[3] = {nacc[0] / len, nacc[1] / len, nacc[2] / len};
                    for (int r = 0; r < 3; ++r) out_normal[3 * pix + r] = (Ef[4 * r] * n[0] + Ef[4 * r + 1] * n[1]) + Ef[4 * r + 2] * n[2];
                }
            }
        }
    free(range);
    free(alloc_legacy);
    return samples;
}
