/* Brute-force CPU reference of the mesh point and ray queries (csrc/bslam_mesh_raycast.cu, `RaycastingScene`'s
 * compute_closest_points, compute_distance, compute_occupancy, compute_signed_distance, count_intersections,
 * test_occlusions): every query is tested against every triangle.  TEST INFRASTRUCTURE, like oracle/: it defines the
 * semantics the GPU must equal bit for bit.  Built by tests/mesh_query_ref.py with gcc -ffp-contract=off.
 *
 * The scene rules, the ray set-up, the watertight test with its box rule and the normal are the cast's: this file
 * includes tests/mesh_raycast_ref.c and uses its functions, so both references share one definition of them. */
#include "mesh_raycast_ref.c"

#include "../bodyslam_b200/csrc/bslam_mesh_dirs.h"   /* the occupancy directions, shared with the library */

/* ------------------------------------------------------------------ point and ray queries
 *
 *   closest    Ericson's ClosestPtPointTriangle (Real-Time Collision Detection 5.1.5) in float32, regions tested in the
 *              order v0, v1, edge v0v1, v2, edge v0v2, edge v1v2, face; dots summed (x + y) + z.  When c or its weights
 *              are not finite (a region's 0 / 0, an overflow), the triangle's nearest vertex stands in (first of v0, v1,
 *              v2 on a tie).  d^2 = |c - p|^2 (+inf when it overflows: the triangle still competes).
 *   key        max(d^2, lb(own box, p)) with lb = (g0^2 + g1^2) + g2^2, g_k = max(lo_k - p_k, p_k - hi_k, 0): the
 *              nearest triangle is the lexicographic minimum of (key, g, p); the BVH prunes by lb, see the .cu.
 *   outputs    closest point, ids, uv = weights of v1 and v2, the cast's unit normal; distance sqrtf(d^2)
 *   undefined  a query point with a non-finite component, or an empty scene: distance +inf, ids 0xFFFFFFFF, point, uv,
 *              normal and occupancy 0 (this project's choice; Open3D's behaviour there is unpinned)
 *   count      the number of triangles tri_hit accepts (t >= 0 under the box rule, as the cast): a ray through an
 *              edge shared by two triangles counts both
 *   occlusion  some accepted hit with tnear <= t <= tfar, both ends inclusive
 *   occupancy  rays from p along the first nsamples directions of bslam_mesh_direction_set (odd, <= 31); 1 when more
 *              than half of them have an odd count; signed distance = the distance, negated when the occupancy is 1
 */

static float dot3(const float a[3], const float b[3]) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }

static float box_lb(const float lo[3], const float hi[3], const float q[3]) {
    float g[3];
    for (int k = 0; k < 3; ++k) {
        const float a = lo[k] - q[k], b = q[k] - hi[k];
        const float m = b > a ? b : a;
        g[k] = m > 0.0f ? m : 0.0f;
    }
    return (g[0] * g[0] + g[1] * g[1]) + g[2] * g[2];
}

static float closest_tri(const float p[3], const float v[9], float c[3], float *u, float *w) {
    const float *a = v, *b = v + 3, *cc = v + 6;
    float ab[3], ac[3], ap[3], bp[3], cp[3];
    for (int k = 0; k < 3; ++k) { ab[k] = b[k] - a[k]; ac[k] = cc[k] - a[k]; ap[k] = p[k] - a[k]; bp[k] = p[k] - b[k]; cp[k] = p[k] - cc[k]; }
    const float d1 = dot3(ab, ap), d2 = dot3(ac, ap), d3 = dot3(ab, bp), d4 = dot3(ac, bp), d5 = dot3(ab, cp), d6 = dot3(ac, cp);
    const float vc = d1 * d4 - d3 * d2, vb = d5 * d2 - d1 * d6, va = d3 * d6 - d5 * d4;
    int ok = 1;
    float s = 0.0f, t = 0.0f;
    if (d1 <= 0.0f && d2 <= 0.0f) {                                       /* vertex v0 */
        for (int k = 0; k < 3; ++k) c[k] = a[k];
        *u = 0.0f; *w = 0.0f;
    } else if (d3 >= 0.0f && d4 <= d3) {                                  /* vertex v1 */
        for (int k = 0; k < 3; ++k) c[k] = b[k];
        *u = 1.0f; *w = 0.0f;
    } else if (vc <= 0.0f && d1 >= 0.0f && d3 <= 0.0f) {                  /* edge v0 v1 */
        s = d1 / (d1 - d3);
        for (int k = 0; k < 3; ++k) c[k] = a[k] + s * ab[k];
        *u = s; *w = 0.0f;
    } else if (d6 >= 0.0f && d5 <= d6) {                                  /* vertex v2 */
        for (int k = 0; k < 3; ++k) c[k] = cc[k];
        *u = 0.0f; *w = 1.0f;
    } else if (vb <= 0.0f && d2 >= 0.0f && d6 <= 0.0f) {                  /* edge v0 v2 */
        t = d2 / (d2 - d6);
        for (int k = 0; k < 3; ++k) c[k] = a[k] + t * ac[k];
        *u = 0.0f; *w = t;
    } else if (va <= 0.0f && (d4 - d3) >= 0.0f && (d5 - d6) >= 0.0f) {   /* edge v1 v2 */
        t = (d4 - d3) / ((d4 - d3) + (d5 - d6));
        for (int k = 0; k < 3; ++k) c[k] = b[k] + t * (cc[k] - b[k]);
        *u = 1.0f - t; *w = t;
    } else {                                                              /* face */
        const float den = 1.0f / ((va + vb) + vc);
        s = vb * den;
        t = vc * den;
        for (int k = 0; k < 3; ++k) c[k] = (a[k] + ab[k] * s) + ac[k] * t;
        *u = s; *w = t;
    }
    for (int k = 0; k < 3; ++k) ok &= isfinite(c[k]) != 0;
    ok &= isfinite(*u) != 0 && isfinite(*w) != 0;
    if (!ok) {
        float best = INFINITY;
        int j = 0;
        for (int m = 0; m < 3; ++m) {
            float e[3];
            for (int k = 0; k < 3; ++k) e[k] = v[3 * m + k] - p[k];
            const float dd = dot3(e, e);
            if (m == 0 || dd < best) { best = dd; j = m; }
        }
        for (int k = 0; k < 3; ++k) c[k] = v[3 * j + k];
        *u = j == 1 ? 1.0f : 0.0f;
        *w = j == 2 ? 1.0f : 0.0f;
    }
    float e[3];
    for (int k = 0; k < 3; ++k) e[k] = c[k] - p[k];
    return dot3(e, e);
}

static void tri_box(const float v[9], float lo[3], float hi[3]) {
    for (int k = 0; k < 3; ++k) {
        const float a = v[k], b = v[3 + k], c = v[6 + k];
        lo[k] = a < b ? (a < c ? a : c) : (b < c ? b : c);
        hi[k] = a > b ? (a > c ? a : c) : (b > c ? b : c);
    }
}

static void load_tri(const float *verts, const int32_t *tris, int64_t vf, int64_t j, float v[9]) {
    for (int c = 0; c < 3; ++c)
        for (int k = 0; k < 3; ++k) v[3 * c + k] = verts[3 * (vf + tris[3 * j + c]) + k];
}

/* nearest triangle of one point by brute force -> d^2 (+inf and g = INVALID when there is none) */
static float closest_one(const float *verts, const int32_t *tris, const int64_t *geom, int n_geoms, const float p[3], float c[3], float *u, float *w,
                         uint32_t *gb, uint32_t *pb, float vbest[9]) {
    float keyb = INFINITY, d2b = INFINITY;
    *gb = INVALID; *pb = INVALID; *u = 0.0f; *w = 0.0f;
    c[0] = c[1] = c[2] = 0.0f;
    if (!(isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]))) return INFINITY;
    for (int g = 0; g < n_geoms; ++g) {
        const int64_t vf = g_verts_first(geom, g);
        for (int64_t j = geom[2 * g]; j < geom[2 * g + 2]; ++j) {
            float v[9], cj[3], uj, wj, lo[3], hi[3];
            load_tri(verts, tris, vf, j, v);
            if (!tri_in_scene(v)) continue;
            const float d2 = closest_tri(p, v, cj, &uj, &wj);
            tri_box(v, lo, hi);
            const float lb = box_lb(lo, hi, p);
            const float key = d2 > lb ? d2 : lb;
            /* (g, p) grow with the scan, so among equal keys the first triangle wins */
            if (key < keyb || (*gb == INVALID && key == keyb)) {
                keyb = key; d2b = d2; *u = uj; *w = wj; *gb = (uint32_t)g; *pb = (uint32_t)(j - geom[2 * g]);
                memcpy(c, cj, sizeof cj);
                memcpy(vbest, v, 9 * sizeof(float));
            }
        }
    }
    return d2b;
}

/* points [n][3]; every output may be NULL */
API void ref_mesh_closest(const float *verts, const int32_t *tris, const int64_t *geom, int n_geoms, const float *pts, int64_t n, float *dist,
                          float *points, uint32_t *geom_ids, uint32_t *prim_ids, float *uv, float *nrm) {
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t i = 0; i < n; ++i) {
        float c[3], u, w, vbest[9] = {0};
        uint32_t g, p;
        const float d2 = closest_one(verts, tris, geom, n_geoms, pts + 3 * i, c, &u, &w, &g, &p, vbest);
        if (dist) dist[i] = sqrtf(d2);
        if (points) for (int k = 0; k < 3; ++k) points[3 * i + k] = c[k];
        if (geom_ids) geom_ids[i] = g;
        if (prim_ids) prim_ids[i] = p;
        if (uv) { uv[2 * i] = u; uv[2 * i + 1] = w; }
        if (nrm) {
            float nv[3] = {0.0f, 0.0f, 0.0f}, nn;
            if (g != INVALID) {
                tri_normal(vbest, nv, &nn);
                const float len = sqrtf(nn);
                for (int k = 0; k < 3; ++k) nv[k] = nv[k] / len;
            }
            for (int k = 0; k < 3; ++k) nrm[3 * i + k] = nv[k];
        }
    }
}

static int count_one(const float *verts, const int32_t *tris, const int64_t *geom, int n_geoms, const float r[6], float tnear, float tfar) {
    Ray ray;
    int count = 0;
    if (!ray_setup(r, &ray)) return 0;
    for (int g = 0; g < n_geoms; ++g) {
        const int64_t vf = g_verts_first(geom, g);
        for (int64_t j = geom[2 * g]; j < geom[2 * g + 2]; ++j) {
            float v[9], t, u, w2;
            load_tri(verts, tris, vf, j, v);
            if (tri_in_scene(v) && tri_hit(&ray, v, &t, &u, &w2) && tnear <= t && t <= tfar) ++count;
        }
    }
    return count;
}

/* accepted hits with tnear <= t <= tfar of each ray: count_intersections is (0, +inf), test_occlusions is count > 0 */
API void ref_mesh_count(const float *verts, const int32_t *tris, const int64_t *geom, int n_geoms, const float *rays, int64_t n, float tnear, float tfar,
                        int32_t *counts) {
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t i = 0; i < n; ++i) counts[i] = count_one(verts, tris, geom, n_geoms, rays + 6 * i, tnear, tfar);
}

API void ref_mesh_directions(int n, float *dirs) { bslam_mesh_direction_set(n, dirs); }

/* occupancy / signed distance (either may be NULL); nsamples odd in [1, BSLAM_MESH_MAX_SAMPLES]: returns 0, else -1 */
API int ref_mesh_occupancy(const float *verts, const int32_t *tris, const int64_t *geom, int n_geoms, const float *pts, int64_t n, int nsamples,
                           float *occupancy, float *sdist) {
    if (nsamples < 1 || nsamples > BSLAM_MESH_MAX_SAMPLES || nsamples % 2 == 0) return -1;
    float dirs[BSLAM_MESH_MAX_SAMPLES][3];
    bslam_mesh_direction_set(nsamples, &dirs[0][0]);
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t i = 0; i < n; ++i) {
        const float *p = pts + 3 * i;
        int inside = 0;
        for (int s = 0; s < nsamples; ++s) {
            const float r[6] = {p[0], p[1], p[2], dirs[s][0], dirs[s][1], dirs[s][2]};
            inside += count_one(verts, tris, geom, n_geoms, r, 0.0f, INFINITY) & 1;
        }
        const int occ = 2 * inside > nsamples;
        if (occupancy) occupancy[i] = occ ? 1.0f : 0.0f;
        if (sdist) {
            float c[3], u, w, vb[9];
            uint32_t g, pr;
            const float d = sqrtf(closest_one(verts, tris, geom, n_geoms, p, c, &u, &w, &g, &pr, vb));
            sdist[i] = occ ? -d : d;
        }
    }
    return 0;
}

/* Replays of the BVH traversals of the queries over a host copy of the BVH, with the kernels' rules: out[0] += inner
 * nodes read (64 B), out[1] += leaf triangles read (48 B; the winner's normal re-read is not counted). */
API void ref_mesh_traverse_closest(const void *bvh, const float *pts, int64_t n, float *dist, uint32_t *geom_ids, uint32_t *prim_ids, int64_t *out) {
    const char *base = (const char *)bvh;
    int n_leaf;
    memcpy(&n_leaf, base, 4);
    const char *nodes = base + 64, *leaves = base + 64 + 64 * (int64_t)(n_leaf > 1 ? n_leaf - 1 : 0);
    int64_t n_nodes = 0, n_tris = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : n_nodes, n_tris)
    for (int64_t i = 0; i < n; ++i) {
        const float *p = pts + 3 * i;
        float keyb = INFINITY, d2b = INFINITY;
        uint64_t kb = ~(uint64_t)0;
        int best = -1;
        if (n_leaf > 0 && isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2])) {
            int stack[64], sp = 0, node = n_leaf > 1 ? 0 : ~0;
            stack[sp++] = INT32_MIN;
            while (node != INT32_MIN) {
                while (node >= 0) {
                    float b[12];
                    int c[2];
                    memcpy(b, nodes + 64 * (int64_t)node, 48);
                    memcpy(c, nodes + 64 * (int64_t)node + 48, 8);
                    ++n_nodes;
                    const float l0 = box_lb(b, b + 3, p), l1 = box_lb(b + 6, b + 9, p);
                    const int h0 = !(l0 > keyb), h1 = !(l1 > keyb);
                    if (h0 && h1) {
                        const int first0 = !(l1 < l0);
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
                    float v[9], cj[3], u, w, lo[3], hi[3];
                    uint32_t gp[2];
                    memcpy(v, leaves + 48 * (int64_t)li, 36);
                    memcpy(gp, leaves + 48 * (int64_t)li + 36, 8);
                    ++n_tris;
                    const float d2 = closest_tri(p, v, cj, &u, &w);
                    tri_box(v, lo, hi);
                    const float lb = box_lb(lo, hi, p);
                    const float key = d2 > lb ? d2 : lb;
                    const uint64_t gk = (uint64_t)gp[0] << 32 | gp[1];
                    if (key < keyb || (key == keyb && gk < kb)) { keyb = key; kb = gk; best = li; d2b = d2; }
                    node = stack[--sp];
                }
            }
        }
        dist[i] = sqrtf(d2b);
        geom_ids[i] = best >= 0 ? (uint32_t)(kb >> 32) : INVALID;
        prim_ids[i] = best >= 0 ? (uint32_t)kb : INVALID;
    }
    out[0] += n_nodes;
    out[1] += n_tris;
}

/* any = 0: counts of accepted hits in [tnear, tfar]; any = 1: 0 / 1, stopping at the first */
API void ref_mesh_traverse_count(const void *bvh, const float *rays, int64_t n, float tnear, float tfar, int any, int32_t *counts, int64_t *out) {
    const char *base = (const char *)bvh;
    int n_leaf;
    memcpy(&n_leaf, base, 4);
    const char *nodes = base + 64, *leaves = base + 64 + 64 * (int64_t)(n_leaf > 1 ? n_leaf - 1 : 0);
    int64_t n_nodes = 0, n_tris = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : n_nodes, n_tris)
    for (int64_t i = 0; i < n; ++i) {
        Ray ray;
        int count = 0;
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
                    const int h0 = !(a0 > tfar) && !(b0 < tnear) && !(a0 > b0), h1 = !(a1 > tfar) && !(b1 < tnear) && !(a1 > b1);
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
                    float v[9], t, u, w2;
                    memcpy(v, leaves + 48 * (int64_t)~node, 36);
                    ++n_tris;
                    if (tri_hit(&ray, v, &t, &u, &w2) && tnear <= t && t <= tfar) {
                        ++count;
                        if (any) break;
                    }
                    node = stack[--sp];
                }
            }
        }
        counts[i] = count;
    }
    out[0] += n_nodes;
    out[1] += n_tris;
}
