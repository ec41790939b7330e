/* Brute-force CPU reference of the mesh ray cast (csrc/bslam_mesh_raycast.cu, `RaycastingScene`): every ray is tested
 * against every triangle.  TEST INFRASTRUCTURE, like oracle/: it defines the semantics the GPU must equal bit for bit.
 * Built by tests/mesh_raycast_ref.py with gcc -ffp-contract=off (no contraction, like the library's -fmad=false).
 *
 *   scene      geometries g = 0..G-1 (one per add_triangles call), primitive p = row of the triangle in its geometry;
 *              a triangle with a non-finite coordinate or a float32 normal n with n . n == 0 (not > 0) is not in it
 *   ray        {o, d} float32, hit point o + t d for t in [0, +inf); a ray with a non-finite component or d = 0 misses
 *   test       watertight (Woop, Benthin and Wald, JCGT 2013) in float32, U, V, W recomputed in float64 when one of
 *              them is exactly 0; no backface culling; u = V / det (weight of v1), v = W / det (weight of v2)
 *   box rule   a hit counts only if t lies in box_interval of the triangle's own bounding box (see the .cu for why the
 *              BVH cast then equals this brute force exactly)
 *   closest    the lexicographic minimum of (t, g, p) over the accepted triangles
 *   outputs    t_hit (+inf on a miss), g / p (0xFFFFFFFF), uv (0), unit normal (v1 - v0) x (v2 - v0) / sqrtf(n . n) (0)
 *   pinhole    M = R^T K^-1 (float64, K^-1 by cofactors like Eigen), cast to float32; origin -R^T t; direction
 *              M (x + 0.5, y + 0.5, 1) in float32 as (m0 px + m1 py) + m2
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define API __attribute__((visibility("default")))
#define EPS (1.0f / 65536.0f)
#define INVALID 0xFFFFFFFFu

static void box_interval(const float lo[3], const float hi[3], const float o[3], const float d[3], float *t0, float *t1) {
    float a = -INFINITY, b = INFINITY;
    for (int k = 0; k < 3; ++k) {
        if (d[k] == 0.0f) {
            if (!(lo[k] <= o[k] && o[k] <= hi[k])) { a = INFINITY; b = -INFINITY; }
        } else {
            float ta = (lo[k] - o[k]) / d[k], tb = (hi[k] - o[k]) / d[k];
            if (ta > tb) { const float s = ta; ta = tb; tb = s; }
            a = ta > a ? ta : a;
            b = tb < b ? tb : b;
        }
    }
    float m = -a > b ? -a : b;
    m = m > 0.0f ? m : 0.0f;
    const float w = EPS * m;
    *t0 = a - w;
    *t1 = b + w;
}

typedef struct {
    float o[3], d[3];
    int kx, ky, kz;
    float Sx, Sy, Sz;
} Ray;

static int ray_setup(const float r[6], Ray *ray) {
    int ok = 1, nz = 0;
    for (int k = 0; k < 6; ++k) ok &= isfinite(r[k]) != 0;
    for (int k = 0; k < 3; ++k) { ray->o[k] = r[k]; ray->d[k] = r[3 + k]; nz |= r[3 + k] != 0.0f; }
    if (!(ok && nz)) return 0;
    int kz = 0;
    if (fabsf(ray->d[1]) > fabsf(ray->d[kz])) kz = 1;
    if (fabsf(ray->d[2]) > fabsf(ray->d[kz])) kz = 2;
    int kx = kz == 2 ? 0 : kz + 1, ky = kx == 2 ? 0 : kx + 1;
    const float dz = ray->d[kz];
    if (dz < 0.0f) { const int s = kx; kx = ky; ky = s; }
    ray->kx = kx; ray->ky = ky; ray->kz = kz;
    ray->Sx = ray->d[kx] / dz;
    ray->Sy = ray->d[ky] / dz;
    ray->Sz = 1.0f / dz;
    return 1;
}

static int tri_hit(const Ray *ray, const float v[9], float *t, float *u, float *w2) {
    float A[3], B[3], C[3];
    for (int k = 0; k < 3; ++k) { A[k] = v[k] - ray->o[k]; B[k] = v[3 + k] - ray->o[k]; C[k] = v[6 + k] - ray->o[k]; }
    const float Akz = A[ray->kz], Bkz = B[ray->kz], Ckz = C[ray->kz];
    const float Ax = A[ray->kx] - ray->Sx * Akz, Ay = A[ray->ky] - ray->Sy * Akz;
    const float Bx = B[ray->kx] - ray->Sx * Bkz, By = B[ray->ky] - ray->Sy * Bkz;
    const float Cx = C[ray->kx] - ray->Sx * Ckz, Cy = C[ray->ky] - ray->Sy * Ckz;
    float U = Cx * By - Cy * Bx, V = Ax * Cy - Ay * Cx, W = Bx * Ay - By * Ax;
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
        V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
        W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return 0;
    const float det = (U + V) + W;
    if (det == 0.0f) return 0;
    const float T = ((U * (ray->Sz * Akz)) + V * (ray->Sz * Bkz)) + W * (ray->Sz * Ckz);
    if (det > 0.0f ? T < 0.0f : T > 0.0f) return 0;
    *t = T / det;
    float lo[3], hi[3], t0, t1;
    for (int k = 0; k < 3; ++k) {
        const float a = v[k], b = v[3 + k], c = v[6 + k];
        lo[k] = a < b ? (a < c ? a : c) : (b < c ? b : c);
        hi[k] = a > b ? (a > c ? a : c) : (b > c ? b : c);
    }
    box_interval(lo, hi, ray->o, ray->d, &t0, &t1);
    if (!(t0 <= *t && *t <= t1 && *t < INFINITY)) return 0;
    *u = V / det;
    *w2 = W / det;
    return 1;
}

static void tri_normal(const float v[9], float n[3], float *nn) {
    const float e1[3] = {v[3] - v[0], v[4] - v[1], v[5] - v[2]}, e2[3] = {v[6] - v[0], v[7] - v[1], v[8] - v[2]};
    n[0] = e1[1] * e2[2] - e1[2] * e2[1];
    n[1] = e1[2] * e2[0] - e1[0] * e2[2];
    n[2] = e1[0] * e2[1] - e1[1] * e2[0];
    *nn = (n[0] * n[0] + n[1] * n[1]) + n[2] * n[2];
}

/* 1 when the triangle is part of the scene */
static int tri_in_scene(const float v[9]) {
    for (int k = 0; k < 9; ++k)
        if (!isfinite(v[k])) return 0;
    float n[3], nn;
    tri_normal(v, n, &nn);
    return nn > 0.0f;
}

static int64_t g_verts_first(const int64_t *geom, int g) { return geom[2 * g + 1]; }

/* verts [n_verts][3] f32, tris [n_tris][3] i32 local to their geometry, geom [n_geoms + 1][2] {first triangle, first
 * vertex} (indices must be in range: the caller checks them); rays [n][6]; uv / nrm may be NULL */
API void ref_mesh_cast(const float *verts, const int32_t *tris, const int64_t *geom, int n_geoms, const float *rays, int64_t n, float *t_hit,
                       uint32_t *geom_ids, uint32_t *prim_ids, float *uv, float *nrm) {
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t i = 0; i < n; ++i) {
        Ray ray;
        float tb = INFINITY, ub = 0.0f, vb = 0.0f, vbest[9] = {0};
        uint32_t gb = INVALID, pb = INVALID;
        if (ray_setup(rays + 6 * i, &ray)) {
            for (int g = 0; g < n_geoms; ++g) {
                const int64_t vf = g_verts_first(geom, g);
                for (int64_t j = geom[2 * g]; j < geom[2 * g + 2]; ++j) {
                    float v[9], t, u, w2;
                    for (int c = 0; c < 3; ++c)
                        for (int k = 0; k < 3; ++k) v[3 * c + k] = verts[3 * (vf + tris[3 * j + c]) + k];
                    if (!tri_in_scene(v) || !tri_hit(&ray, v, &t, &u, &w2)) continue;
                    const uint32_t p = (uint32_t)(j - geom[2 * g]);
                    /* (g, p) grow with the scan, so among equal t the first accepted triangle wins */
                    if (t < tb) { tb = t; ub = u; vb = w2; gb = (uint32_t)g; pb = p; memcpy(vbest, v, sizeof v); }
                }
            }
        }
        t_hit[i] = tb;
        geom_ids[i] = gb;
        prim_ids[i] = pb;
        if (uv) { uv[2 * i] = ub; uv[2 * i + 1] = vb; }
        if (nrm) {
            float nv[3] = {0.0f, 0.0f, 0.0f}, nn;
            if (gb != INVALID) {
                tri_normal(vbest, nv, &nn);
                const float len = sqrtf(nn);
                for (int k = 0; k < 3; ++k) nv[k] = nv[k] / len;
            }
            for (int k = 0; k < 3; ++k) nrm[3 * i + k] = nv[k];
        }
    }
}

/* K 3x3 row-major f64, E 4x4 row-major f64 world -> camera -> rays [H][W][6] */
API void ref_mesh_rays_pinhole(const double *K, const double *E, int W, int H, float *rays) {
    double cof[3][3], Ki[9];
    float M[9], c[3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
            cof[i][j] = K[3 * i1 + j1] * K[3 * i2 + j2] - K[3 * i1 + j2] * K[3 * i2 + j1];
        }
    const double det = (cof[0][0] * K[0] + cof[1][0] * K[3]) + cof[2][0] * K[6];
    const double inv = 1.0 / det;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) Ki[3 * j + i] = cof[i][j] * inv;
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) M[3 * i + j] = (float)((E[0 * 4 + i] * Ki[0 * 3 + j] + E[1 * 4 + i] * Ki[1 * 3 + j]) + E[2 * 4 + i] * Ki[2 * 3 + j]);
        c[i] = (float)((E[0 * 4 + i] * -E[3] + E[1 * 4 + i] * -E[7]) + E[2 * 4 + i] * -E[11]);
    }
    for (int y = 0; y < H; ++y)
        for (int x = 0; x < W; ++x) {
            float *r = rays + 6 * ((int64_t)y * W + x);
            const float px = (float)x + 0.5f, py = (float)y + 0.5f;
            for (int i = 0; i < 3; ++i) {
                r[i] = c[i];
                r[3 + i] = (M[3 * i] * px + M[3 * i + 1] * py) + M[3 * i + 2];
            }
        }
}

/* Reads of the device BVH (a host copy of bslam_mesh_build's output) by the cast's traversal, replayed on the CPU with
 * the same pruning rule: out[0] += inner nodes read (64 B each), out[1] += leaf triangles read (48 B each; the winner's
 * normal re-read is not counted).  Also returns the hit (t, g, p) so the replay can be checked against the brute force. */
API void ref_mesh_traverse(const void *bvh, const float *rays, int64_t n, float *t_hit, uint32_t *geom_ids, uint32_t *prim_ids, int64_t *out) {
    const char *base = (const char *)bvh;
    int n_leaf;
    memcpy(&n_leaf, base, 4);
    const char *nodes = base + 64, *leaves = base + 64 + 64 * (int64_t)(n_leaf > 1 ? n_leaf - 1 : 0);
    int64_t n_nodes = 0, n_tris = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : n_nodes, n_tris)
    for (int64_t i = 0; i < n; ++i) {
        Ray ray;
        float tb = INFINITY;
        uint64_t kb = ~(uint64_t)0;
        int best = -1;
        if (n_leaf > 0 && ray_setup(rays + 6 * i, &ray)) {
            int stack[64], sp = 0, node = n_leaf > 1 ? 0 : ~0;
            stack[sp++] = INT32_MIN;
            while (node != INT32_MIN) {
                while (node >= 0) {
                    float b[12], a0, b0, a1, b1;
                    int c[2];
                    memcpy(b, nodes + 64 * (int64_t)node, 48);
                    memcpy(c, nodes + 64 * (int64_t)node + 48, 8);
                    ++n_nodes;
                    box_interval(b, b + 3, ray.o, ray.d, &a0, &b0);
                    box_interval(b + 6, b + 9, ray.o, ray.d, &a1, &b1);
                    const int h0 = !(a0 > tb) && !(b0 < 0.0f), h1 = !(a1 > tb) && !(b1 < 0.0f);
                    if (h0 && h1) {
                        const int first0 = !(a1 < a0);
                        stack[sp++] = first0 ? c[1] : c[0];
                        node = first0 ? c[0] : c[1];
                    } else if (h0 || h1) {
                        node = h0 ? c[0] : c[1];
                    } else {
                        node = stack[--sp];
                    }
                }
                if (node != INT32_MIN) {
                    const int li = ~node;
                    float v[9], t, u, w2;
                    uint32_t gp[2];
                    memcpy(v, leaves + 48 * (int64_t)li, 36);
                    memcpy(gp, leaves + 48 * (int64_t)li + 36, 8);
                    ++n_tris;
                    if (tri_hit(&ray, v, &t, &u, &w2)) {
                        const uint64_t key = (uint64_t)gp[0] << 32 | gp[1];
                        if (t < tb || (t == tb && key < kb)) { tb = t; kb = key; best = li; }
                    }
                    node = stack[--sp];
                }
            }
        }
        t_hit[i] = tb;
        geom_ids[i] = best >= 0 ? (uint32_t)(kb >> 32) : INVALID;
        prim_ids[i] = best >= 0 ? (uint32_t)kb : INVALID;
    }
    out[0] += n_nodes;
    out[1] += n_tris;
}
