// Mesh ray casting (Open3D `t.geometry.RaycastingScene.cast_rays`, the reference's synthetic depth generator): closest
// hits of rays against triangle meshes through an LBVH built on the device.  The semantics are written down in the
// brute-force CPU reference tests/mesh_raycast_ref.c (every ray against every triangle), which this file must match bit
// for bit (-fmad=false, IEEE `/` and sqrtf):
//   * the watertight ray/triangle test of Woop, Benthin and Wald (JCGT 2013) in float32, float64 fall-back when an edge
//     function is exactly 0; no backface culling; t in [0, +inf);
//   * a hit counts only if its t lies in mr_box_interval of the triangle's own bounding box;
//   * the closest hit is the lexicographic minimum of (t, geometry, primitive), so the result does not depend on the
//     traversal order;
//   * triangles with a non-finite coordinate or a zero float32 normal (n . n == 0) are not part of the scene; rays with a
//     non-finite component or d = 0 miss.
// Build: 64-bit keys (30-bit Morton code of the centroid, triangle index) sorted with CUB, Karras's (2012) split search,
// boxes fitted bottom-up with arrival counters.  Cast: one thread per ray, nearest child first, 64-entry stack.
#include <float.h>
#include <limits.h>
#include <math.h>

#include <cub/device/device_radix_sort.cuh>

#include "bslam_common.cuh"

namespace bslam {

constexpr float kMrEps = 1.0f / 65536.0f;            // widening of every box interval, relative to its magnitude
constexpr int kMrStack = 64;                          // unique 64-bit keys: the tree is at most 64 levels deep
constexpr int kMrMaxFrames = 64;
constexpr int kMrTileW = 32, kMrTileH = 8;
constexpr int kMrEmpty = INT_MIN;                     // stack sentinel (leaf refs are ~i >= -(2^31 - 1))
constexpr uint32_t kMrInvalid = 0xFFFFFFFFu;
constexpr unsigned long long kMrOut = 1ull << 62;     // key flag: triangle left out of the scene, sorted after the rest

// 64 B: both child boxes {lo xyz, hi xyz} and both child references (>= 0: internal node, < 0: ~leaf)
struct __align__(16) MrNode {
    float b[2][6];
    int child[2];
    int pad[2];
};
// 48 B, in leaf order: the three vertices and the ids, so that traversal never follows an index
struct __align__(16) MrTri {
    float v[9];
    uint32_t g, p, out;
};
constexpr size_t kMrHeader = 64;                      // {int n_leaf}

__host__ __device__ inline size_t mr_nodes_offset() { return kMrHeader; }
__host__ __device__ inline size_t mr_leaves_offset(int64_t n) { return kMrHeader + sizeof(MrNode) * (size_t)(n > 1 ? n - 1 : 0); }

// Slab interval [t0, t1] of the ray o + t d through the box [lo, hi], widened by kMrEps of its magnitude.
// Exactness: a hit is accepted only if its t lies in the interval of the triangle's own box, and a node is pruned only
// if its interval misses [0, t_best].  Node boxes are exact min / max unions, so along every axis parent.lo <= child.lo
// and parent.hi >= child.hi.  Each step below is monotone in the box, rounding included (x - o, x / d, max, min, the
// products and sums of the widening): for d_k > 0 the entry value ta grows with lo_k and tb with hi_k, for d_k < 0 the
// roles swap; an axis with d_k == 0 is unbounded or empty, and the parent's slab contains o_k whenever the child's
// does (an empty axis sets a = +inf, b = -inf, m = 0: rejected and pruned).  Hence a <= a_child and b >= b_child, so
// m = max(-a, b, 0) >= m_child and t0 <= t0_child, t1 >= t1_child: the interval of a node contains the intervals of all
// triangles below it, and a triangle whose t is accepted (t0_tri <= t <= t_best, t <= t1_tri) never sits below a pruned
// node.  With o and d finite, no NaN arises before the widening; an infinite a and m make t0 NaN, which rejects a
// triangle (t0 <= t is false) and never prunes a node (t0 > t_best is false), so the property holds there too.
__host__ __device__ __forceinline__ void mr_box_interval(const float lo[3], const float hi[3], const float o[3], const float d[3], float &t0,
                                                         float &t1) {
    float a = -INFINITY, b = INFINITY;
#pragma unroll
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
    const float w = kMrEps * m;
    t0 = a - w;
    t1 = b + w;
}

// per-ray constants of the watertight test
struct MrRay {
    float o[3], d[3];
    int kx, ky, kz;
    float Sx, Sy, Sz;
};

__host__ __device__ __forceinline__ float mr_sel(const float a[3], int k) { return k == 0 ? a[0] : (k == 1 ? a[1] : a[2]); }

// false: the ray misses everything (a non-finite component, or d = 0)
__host__ __device__ __forceinline__ bool mr_ray_setup(const float r[6], MrRay &ray) {
    bool ok = true, nz = false;
    for (int k = 0; k < 6; ++k) ok &= isfinite(r[k]) != 0;
    for (int k = 0; k < 3; ++k) { ray.o[k] = r[k]; ray.d[k] = r[3 + k]; nz |= r[3 + k] != 0.0f; }
    if (!(ok && nz)) return false;
    int kz = 0;
    if (fabsf(ray.d[1]) > fabsf(ray.d[kz])) kz = 1;
    if (fabsf(ray.d[2]) > fabsf(ray.d[kz])) kz = 2;
    int kx = kz == 2 ? 0 : kz + 1, ky = kx == 2 ? 0 : kx + 1;
    const float dz = mr_sel(ray.d, kz);
    if (dz < 0.0f) { const int s = kx; kx = ky; ky = s; }
    ray.kx = kx; ray.ky = ky; ray.kz = kz;
    ray.Sx = mr_sel(ray.d, kx) / dz;
    ray.Sy = mr_sel(ray.d, ky) / dz;
    ray.Sz = 1.0f / dz;
    return true;
}

// Woop-Benthin-Wald test plus the box rule; t, u (weight of v1), v (weight of v2) when the hit counts
__host__ __device__ __forceinline__ bool mr_tri_hit(const MrRay &ray, const float v[9], float &t, float &u, float &w2) {
    float A[3], B[3], C[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { A[k] = v[k] - ray.o[k]; B[k] = v[3 + k] - ray.o[k]; C[k] = v[6 + k] - ray.o[k]; }
    const float Akz = mr_sel(A, ray.kz), Bkz = mr_sel(B, ray.kz), Ckz = mr_sel(C, ray.kz);
    const float Ax = mr_sel(A, ray.kx) - ray.Sx * Akz, Ay = mr_sel(A, ray.ky) - ray.Sy * Akz;
    const float Bx = mr_sel(B, ray.kx) - ray.Sx * Bkz, By = mr_sel(B, ray.ky) - ray.Sy * Bkz;
    const float Cx = mr_sel(C, ray.kx) - ray.Sx * Ckz, Cy = mr_sel(C, ray.ky) - ray.Sy * Ckz;
    float U = Cx * By - Cy * Bx, V = Ax * Cy - Ay * Cx, W = Bx * Ay - By * Ax;
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
        V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
        W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
    const float det = (U + V) + W;
    if (det == 0.0f) return false;
    const float T = ((U * (ray.Sz * Akz)) + V * (ray.Sz * Bkz)) + W * (ray.Sz * Ckz);
    if (det > 0.0f ? T < 0.0f : T > 0.0f) return false;
    t = T / det;
    float lo[3], hi[3], t0, t1;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float a = v[k], b = v[3 + k], c = v[6 + k];
        lo[k] = a < b ? (a < c ? a : c) : (b < c ? b : c);
        hi[k] = a > b ? (a > c ? a : c) : (b > c ? b : c);
    }
    mr_box_interval(lo, hi, ray.o, ray.d, t0, t1);
    if (!(t0 <= t && t <= t1 && t < INFINITY)) return false;
    u = V / det;
    w2 = W / det;
    return true;
}

// unit normal (v1 - v0) x (v2 - v0) / sqrtf(n . n); nn = n . n (a triangle with !(nn > 0) is left out of the scene)
__host__ __device__ __forceinline__ void mr_normal(const float v[9], float n[3], float &nn) {
    const float e1[3] = {v[3] - v[0], v[4] - v[1], v[5] - v[2]}, e2[3] = {v[6] - v[0], v[7] - v[1], v[8] - v[2]};
    n[0] = e1[1] * e2[2] - e1[2] * e2[1];
    n[1] = e1[2] * e2[0] - e1[0] * e2[2];
    n[2] = e1[0] * e2[1] - e1[1] * e2[0];
    nn = (n[0] * n[0] + n[1] * n[1]) + n[2] * n[2];
}

// ray of pixel (x, y) of a pinhole frame Mc = {M row-major (3x3), camera centre}
__host__ __device__ __forceinline__ void mr_pinhole_ray(const float Mc[12], int x, int y, float r[6]) {
    const float px = (float)x + 0.5f, py = (float)y + 0.5f;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        r[i] = Mc[9 + i];
        r[3 + i] = (Mc[3 * i] * px + Mc[3 * i + 1] * py) + Mc[3 * i + 2];
    }
}

// M = R^T K^-1 (K^-1 by cofactors, Eigen's 3x3 inverse) and the camera centre -R^T t, in float64, cast to float32
static void mr_pinhole_frame(const double *K, const double *E, float Mc[12]) {
    double Ki[9];
    double cof[3][3];
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
        for (int j = 0; j < 3; ++j) Mc[3 * i + j] = (float)((E[0 * 4 + i] * Ki[0 * 3 + j] + E[1 * 4 + i] * Ki[1 * 3 + j]) + E[2 * 4 + i] * Ki[2 * 3 + j]);
        Mc[9 + i] = (float)((E[0 * 4 + i] * -E[3] + E[1 * 4 + i] * -E[7]) + E[2 * 4 + i] * -E[11]);
    }
}

struct MrPinhole {
    int F, W, H;
    float Mc[kMrMaxFrames][12];
};

// ------------------------------------------------------------------ cast

__device__ __forceinline__ void mr_load_tri(const MrTri *leaves, int i, float v[9], uint32_t &g, uint32_t &p) {
    const float4 *q = reinterpret_cast<const float4 *>(leaves + i);
    const float4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w; v[8] = c.x;
    g = __float_as_uint(c.y);
    p = __float_as_uint(c.z);
}

template <bool UV, bool NRM>
__device__ __forceinline__ void mr_trace(const char *__restrict__ bvh, const float r[6], int64_t i, float *__restrict__ t_hit,
                                         uint32_t *__restrict__ geom_ids, uint32_t *__restrict__ prim_ids, float *__restrict__ uvs,
                                         float *__restrict__ normals) {
    const int n_leaf = __ldg(reinterpret_cast<const int *>(bvh));
    const MrNode *nodes = reinterpret_cast<const MrNode *>(bvh + mr_nodes_offset());
    const MrTri *leaves = reinterpret_cast<const MrTri *>(bvh + mr_leaves_offset(n_leaf));
    float tb = INFINITY, ub = 0.0f, vb = 0.0f;
    unsigned long long kb = ~0ull;
    int best = -1;
    MrRay ray;
    if (n_leaf > 0 && mr_ray_setup(r, ray)) {
        int stack[kMrStack];
        int sp = 0;
        int node = n_leaf > 1 ? 0 : ~0;
        stack[sp++] = kMrEmpty;
        while (node != kMrEmpty) {
            while (node >= 0) {           // inner nodes: descend, nearest child first
                const float4 *q = reinterpret_cast<const float4 *>(nodes + node);
                const float4 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);
                const float lo0[3] = {q0.x, q0.y, q0.z}, hi0[3] = {q0.w, q1.x, q1.y};
                const float lo1[3] = {q1.z, q1.w, q2.x}, hi1[3] = {q2.y, q2.z, q2.w};
                float a0, b0, a1, b1;
                mr_box_interval(lo0, hi0, ray.o, ray.d, a0, b0);
                mr_box_interval(lo1, hi1, ray.o, ray.d, a1, b1);
                const bool h0 = !(a0 > tb) && !(b0 < 0.0f), h1 = !(a1 > tb) && !(b1 < 0.0f);
                const int c0 = __float_as_int(q3.x), c1 = __float_as_int(q3.y);
                if (h0 && h1) {
                    const bool first0 = !(a1 < a0);
                    stack[sp++] = first0 ? c1 : c0;
                    node = first0 ? c0 : c1;
                } else if (h0 || h1) {
                    node = h0 ? c0 : c1;
                } else {
                    node = stack[--sp];
                }
            }
            if (node != kMrEmpty) {       // a leaf
                const int li = ~node;
                float v[9], t, u, w2;
                uint32_t g, p;
                mr_load_tri(leaves, li, v, g, p);
                if (mr_tri_hit(ray, v, t, u, w2)) {
                    const unsigned long long key = (unsigned long long)g << 32 | p;
                    if (t < tb || (t == tb && key < kb)) { tb = t; kb = key; ub = u; vb = w2; best = li; }
                }
                node = stack[--sp];
            }
        }
    }
    t_hit[i] = tb;
    geom_ids[i] = best >= 0 ? (uint32_t)(kb >> 32) : kMrInvalid;
    prim_ids[i] = best >= 0 ? (uint32_t)kb : kMrInvalid;
    if (UV) { uvs[2 * i] = ub; uvs[2 * i + 1] = vb; }
    if (NRM) {
        float n[3] = {0.0f, 0.0f, 0.0f};
        if (best >= 0) {
            float v[9], nn;
            uint32_t g, p;
            mr_load_tri(leaves, best, v, g, p);
            mr_normal(v, n, nn);
            const float len = sqrtf(nn);
#pragma unroll
            for (int k = 0; k < 3; ++k) n[k] = n[k] / len;
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) normals[3 * i + k] = n[k];
    }
}

template <bool UV, bool NRM>
__global__ void __launch_bounds__(256) mesh_cast_rays_kernel(const char *__restrict__ bvh, const float *__restrict__ rays, int64_t n, float *__restrict__ t_hit,
                                                             uint32_t *__restrict__ geom_ids, uint32_t *__restrict__ prim_ids, float *__restrict__ uvs,
                                                             float *__restrict__ normals) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float r[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) r[k] = __ldg(rays + 6 * i + k);
    mr_trace<UV, NRM>(bvh, r, i, t_hit, geom_ids, prim_ids, uvs, normals);
}

// pixel of thread: a warp covers an 8 x 4 tile (as raycast_kernel); frames in gridDim.y
__device__ __forceinline__ bool mr_pixel(const MrPinhole &ph, int &x, int &y) {
    const int tiles_x = (ph.W + kMrTileW - 1) / kMrTileW;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    x = (blockIdx.x % tiles_x) * kMrTileW + (warp & 3) * 8 + (lane & 7);
    y = (blockIdx.x / tiles_x) * kMrTileH + (warp >> 2) * 4 + (lane >> 3);
    return x < ph.W && y < ph.H;
}

template <bool UV, bool NRM>
__global__ void __launch_bounds__(256) mesh_cast_pinhole_kernel(const char *__restrict__ bvh, const __grid_constant__ MrPinhole ph, float *__restrict__ t_hit,
                                                                uint32_t *__restrict__ geom_ids, uint32_t *__restrict__ prim_ids, float *__restrict__ uvs,
                                                                float *__restrict__ normals) {
    int x, y;
    if (!mr_pixel(ph, x, y)) return;
    const int f = blockIdx.y;
    float r[6];
    mr_pinhole_ray(ph.Mc[f], x, y, r);
    mr_trace<UV, NRM>(bvh, r, ((int64_t)f * ph.H + y) * ph.W + x, t_hit, geom_ids, prim_ids, uvs, normals);
}

__global__ void __launch_bounds__(256) mesh_rays_pinhole_kernel(const __grid_constant__ MrPinhole ph, float *__restrict__ rays) {
    int x, y;
    if (!mr_pixel(ph, x, y)) return;
    float r[6];
    mr_pinhole_ray(ph.Mc[blockIdx.y], x, y, r);
    const int64_t i = ((int64_t)blockIdx.y * ph.H + y) * ph.W + x;
#pragma unroll
    for (int k = 0; k < 6; ++k) rays[6 * i + k] = r[k];
}

// ------------------------------------------------------------------ build

struct MrStatus {
    int bad;              // smallest triangle index with a vertex index out of range (INT_MAX: none)
    int n_in;             // triangles in the scene
    int bounds[6];        // centroid bounds of those triangles, order-preserving int images of floats (lo xyz, hi xyz)
};

__device__ __forceinline__ int mr_ord(float x) { const int b = __float_as_int(x); return b >= 0 ? b : b ^ 0x7FFFFFFF; }
__device__ __forceinline__ float mr_unord(int b) { return __int_as_float(b >= 0 ? b : b ^ 0x7FFFFFFF); }

__device__ __forceinline__ void mr_centroid(const float v[9], float c[3]) {
    // scaled by 3/4 (exact powers of two, no overflow): the Morton code is invariant under the scale
#pragma unroll
    for (int k = 0; k < 3; ++k) c[k] = (v[k] * 0.25f + v[3 + k] * 0.25f) + v[6 + k] * 0.25f;
}

__global__ void __launch_bounds__(256) mesh_prep_kernel(const float *__restrict__ verts, const int32_t *__restrict__ tris, int n,
                                                        const long long *__restrict__ geom, int n_geoms, MrTri *__restrict__ recs, MrStatus *st) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int lo = 0, hi = n_geoms;         // the last geometry whose first triangle is <= i
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(geom + 2 * mid) <= i) lo = mid; else hi = mid;
    }
    const long long vf = __ldg(geom + 2 * lo + 1), nv = __ldg(geom + 2 * lo + 3) - vf;
    MrTri t;
    bool in = true;
    for (int c = 0; c < 3; ++c) {
        const int idx = __ldg(tris + 3 * (int64_t)i + c);
        if (idx < 0 || idx >= nv) { atomicMin(&st->bad, i); in = false; break; }
        for (int k = 0; k < 3; ++k) t.v[3 * c + k] = __ldg(verts + 3 * (vf + idx) + k);
    }
    if (in) {
        for (int k = 0; k < 9; ++k) in &= isfinite(t.v[k]) != 0;
    }
    if (in) {
        float nrm[3], nn;
        mr_normal(t.v, nrm, nn);
        in = nn > 0.0f;
    }
    t.g = (uint32_t)lo;
    t.p = (uint32_t)(i - __ldg(geom + 2 * lo));
    t.out = in ? 0u : 1u;
    recs[i] = t;
    if (!in) return;
    atomicAdd(&st->n_in, 1);
    float c[3];
    mr_centroid(t.v, c);
    for (int k = 0; k < 3; ++k) {
        atomicMin(&st->bounds[k], mr_ord(c[k]));
        atomicMax(&st->bounds[3 + k], mr_ord(c[k]));
    }
}

__device__ __forceinline__ unsigned int mr_expand10(unsigned int x) {
    x &= 0x3FFu;
    x = (x | (x << 16)) & 0x030000FFu;
    x = (x | (x << 8)) & 0x0300F00Fu;
    x = (x | (x << 4)) & 0x030C30C3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}

__global__ void __launch_bounds__(256) mesh_morton_kernel(const MrTri *__restrict__ recs, int n, const MrStatus *__restrict__ st,
                                                          unsigned long long *__restrict__ keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const MrTri t = recs[i];
    if (t.out) { keys[i] = kMrOut | (unsigned)i; return; }
    float c[3];
    mr_centroid(t.v, c);
    unsigned int code = 0;
    for (int k = 0; k < 3; ++k) {
        const double lo = mr_unord(st->bounds[k]), hi = mr_unord(st->bounds[3 + k]);
        const double q = hi > lo ? ((double)c[k] - lo) / (hi - lo) * 1024.0 : 0.0;
        const unsigned int b = q < 0.0 ? 0u : (q > 1023.0 ? 1023u : (unsigned int)q);
        code |= mr_expand10(b) << (2 - k);
    }
    keys[i] = (unsigned long long)code << 32 | (unsigned)i;
}

__device__ __forceinline__ int mr_delta(const unsigned long long *keys, int n, int i, long long j) {
    if (j < 0 || j >= n) return -1;
    return __clzll(keys[i] ^ keys[j]);
}

// Karras (2012): internal node i of n leaves; parents are stored as (parent << 1 | side)
__global__ void __launch_bounds__(256) mesh_hierarchy_kernel(const unsigned long long *__restrict__ keys, int n, char *__restrict__ bvh,
                                                             int *__restrict__ parent_in, int *__restrict__ parent_leaf) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *reinterpret_cast<int *>(bvh) = n;
    if (i >= n - 1) return;
    MrNode *nodes = reinterpret_cast<MrNode *>(bvh + mr_nodes_offset());
    const int d = mr_delta(keys, n, i, i + 1) - mr_delta(keys, n, i, i - 1) > 0 ? 1 : -1;
    const int dmin = mr_delta(keys, n, i, (long long)i - d);
    long long lmax = 2;
    while (mr_delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    long long l = 0;
    for (long long t = lmax >> 1; t >= 1; t >>= 1)
        if (mr_delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const int j = (int)(i + l * d);
    const int dnode = mr_delta(keys, n, i, j);
    long long s = 0, t = l;
    do {
        t = (t + 1) >> 1;
        if (mr_delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    const int gamma = (int)(i + s * d + (d < 0 ? -1 : 0));
    const int lo = i < j ? i : j, hi = i < j ? j : i;
    const int c0 = lo == gamma ? ~gamma : gamma, c1 = hi == gamma + 1 ? ~(gamma + 1) : gamma + 1;
    nodes[i].child[0] = c0;
    nodes[i].child[1] = c1;
    nodes[i].pad[0] = nodes[i].pad[1] = 0;
    if (c0 < 0) parent_leaf[~c0] = i << 1; else parent_in[c0] = i << 1;
    if (c1 < 0) parent_leaf[~c1] = i << 1 | 1; else parent_in[c1] = i << 1 | 1;
}

// leaves in key order, then the boxes bottom-up: the second thread to arrive at a node fits it and climbs on
__global__ void __launch_bounds__(256) mesh_fit_kernel(const unsigned long long *__restrict__ keys, int n, const MrTri *__restrict__ recs, char *bvh,
                                                       const int *__restrict__ parent_in, const int *__restrict__ parent_leaf, int *arrivals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    MrNode *nodes = reinterpret_cast<MrNode *>(bvh + mr_nodes_offset());
    MrTri *leaves = reinterpret_cast<MrTri *>(bvh + mr_leaves_offset(n));
    const MrTri t = recs[(unsigned)keys[i]];
    leaves[i] = t;
    if (n < 2) return;
    float b[6];
    for (int k = 0; k < 3; ++k) {
        const float a = t.v[k], c = t.v[3 + k], e = t.v[6 + k];
        b[k] = fminf(fminf(a, c), e);
        b[3 + k] = fmaxf(fmaxf(a, c), e);
    }
    int up = parent_leaf[i];
    while (true) {
        const int node = up >> 1, side = up & 1;
        for (int k = 0; k < 6; ++k) nodes[node].b[side][k] = b[k];
        __threadfence();
        if (atomicAdd(arrivals + node, 1) == 0) return;
        __threadfence();
        for (int k = 0; k < 3; ++k) {
            const float l0 = __ldcg(&nodes[node].b[0][k]), l1 = __ldcg(&nodes[node].b[1][k]);
            const float h0 = __ldcg(&nodes[node].b[0][3 + k]), h1 = __ldcg(&nodes[node].b[1][3 + k]);
            b[k] = fminf(l0, l1);
            b[3 + k] = fmaxf(h0, h1);
        }
        if (node == 0) return;
        up = parent_in[node];
    }
}

static size_t mr_align(size_t x) { return (x + 255) & ~(size_t)255; }

struct MrWorkspace {
    size_t status, geom, recs, keys_in, keys_out, parent_in, parent_leaf, arrivals, sort, sort_bytes, total;
};

static int mr_sort_bytes(int n, size_t &bytes) {
    bytes = 0;
    if (n == 0) return BSLAM_OK;
    BSLAM_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, bytes, (const unsigned long long *)nullptr, (unsigned long long *)nullptr, n, 0, 63));
    return BSLAM_OK;
}

static int mr_workspace(int n, int n_geoms, MrWorkspace &w) {
    size_t o = 0;
    w.status = o; o += mr_align(sizeof(MrStatus));
    w.geom = o; o += mr_align(sizeof(long long) * 2 * ((size_t)n_geoms + 1));
    w.recs = o; o += mr_align(sizeof(MrTri) * (size_t)n);
    w.keys_in = o; o += mr_align(8 * (size_t)n);
    w.keys_out = o; o += mr_align(8 * (size_t)n);
    w.parent_in = o; o += mr_align(4 * (size_t)n);
    w.parent_leaf = o; o += mr_align(4 * (size_t)n);
    w.arrivals = o; o += mr_align(4 * (size_t)n);
    w.sort = o;
    if (mr_sort_bytes(n, w.sort_bytes) != BSLAM_OK) return BSLAM_E_CUDA;
    o += mr_align(w.sort_bytes);
    w.total = o;
    return BSLAM_OK;
}

template <bool UV, bool NRM>
static void mr_launch_rays(const char *bvh, const float *rays, int64_t n, float *t, uint32_t *g, uint32_t *p, float *uv, float *nrm, cudaStream_t st) {
    mesh_cast_rays_kernel<UV, NRM><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(bvh, rays, n, t, g, p, uv, nrm);
}

template <bool UV, bool NRM>
static void mr_launch_pinhole(dim3 grid, const char *bvh, const MrPinhole &ph, float *t, uint32_t *g, uint32_t *p, float *uv, float *nrm, cudaStream_t st) {
    mesh_cast_pinhole_kernel<UV, NRM><<<grid, 256, 0, st>>>(bvh, ph, t, g, p, uv, nrm);
}

static dim3 mr_grid(int W, int H, int F) { return dim3(((W + kMrTileW - 1) / kMrTileW) * ((H + kMrTileH - 1) / kMrTileH), F); }

} // namespace bslam

using namespace bslam;

extern "C" {

size_t bslam_mesh_bvh_bytes(int64_t n_tris) {
    if (n_tris < 0 || n_tris >= INT_MAX) return 0;
    return mr_leaves_offset(n_tris) + sizeof(MrTri) * (size_t)n_tris;
}

size_t bslam_mesh_build_workspace_bytes(int64_t n_tris, int n_geoms) {
    if (n_tris < 0 || n_tris >= INT_MAX || n_geoms < 0) return 0;
    MrWorkspace w;
    if (mr_workspace((int)n_tris, n_geoms, w) != BSLAM_OK) return 0;
    return w.total;
}

int bslam_mesh_build(const float *d_verts, int64_t n_verts, const int32_t *d_tris, int64_t n_tris, const int64_t *h_geom, int n_geoms, void *d_bvh,
                     void *d_workspace, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(n_verts >= 0 && n_tris >= 0 && n_tris < INT_MAX && n_geoms >= 0, "bslam_mesh_build: bad sizes (n_verts=%lld n_tris=%lld n_geoms=%d)",
                    (long long)n_verts, (long long)n_tris, n_geoms);
    BSLAM_CHECK_ARG(d_bvh && h_geom && (d_workspace || n_tris == 0), "bslam_mesh_build: NULL argument");
    BSLAM_CHECK_ARG((d_verts || n_verts == 0) && (d_tris || n_tris == 0), "bslam_mesh_build: NULL argument");
    BSLAM_CHECK_ARG(h_geom[0] == 0 && h_geom[1] == 0 && h_geom[2 * n_geoms] == n_tris && h_geom[2 * n_geoms + 1] == n_verts,
                    "bslam_mesh_build: the geometry table must run from {0, 0} to {n_tris, n_verts}");
    for (int g = 0; g < n_geoms; ++g)
        BSLAM_CHECK_ARG(h_geom[2 * g + 2] >= h_geom[2 * g] && h_geom[2 * g + 3] >= h_geom[2 * g + 1], "bslam_mesh_build: the geometry table must not decrease");
    cudaStream_t st = (cudaStream_t)stream;
    const int n = (int)n_tris;
    if (n == 0) {
        BSLAM_CUDA(cudaMemsetAsync(d_bvh, 0, kMrHeader, st));
        return BSLAM_OK;
    }
    MrWorkspace w;
    if (mr_workspace(n, n_geoms, w) != BSLAM_OK) return BSLAM_E_CUDA;
    char *ws = (char *)d_workspace;
    MrStatus *status = (MrStatus *)(ws + w.status);
    MrStatus init;
    init.bad = INT_MAX;
    init.n_in = 0;
    for (int k = 0; k < 3; ++k) { init.bounds[k] = INT_MAX; init.bounds[3 + k] = INT_MIN; }
    BSLAM_CUDA(cudaMemcpyAsync(status, &init, sizeof(init), cudaMemcpyHostToDevice, st));
    BSLAM_CUDA(cudaMemcpyAsync(ws + w.geom, h_geom, sizeof(long long) * 2 * ((size_t)n_geoms + 1), cudaMemcpyHostToDevice, st));
    MrTri *recs = (MrTri *)(ws + w.recs);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    mesh_prep_kernel<<<blocks, 256, 0, st>>>(d_verts, d_tris, n, (const long long *)(ws + w.geom), n_geoms, recs, status);
    BSLAM_LAUNCH_CHECK();
    MrStatus host;
    BSLAM_CUDA(cudaMemcpyAsync(&host, status, sizeof(host), cudaMemcpyDeviceToHost, st));
    BSLAM_CUDA(cudaStreamSynchronize(st));
    if (host.bad != INT_MAX) {
        int g = 0;
        while (g + 1 < n_geoms && h_geom[2 * (g + 1)] <= host.bad) ++g;
        BSLAM_CHECK_ARG(false, "bslam_mesh_build: triangle %lld of geometry %d has a vertex index out of range [0, %lld)",
                        (long long)(host.bad - h_geom[2 * g]), g, (long long)(h_geom[2 * g + 3] - h_geom[2 * g + 1]));
    }
    unsigned long long *keys_in = (unsigned long long *)(ws + w.keys_in), *keys_out = (unsigned long long *)(ws + w.keys_out);
    mesh_morton_kernel<<<blocks, 256, 0, st>>>(recs, n, status, keys_in);
    BSLAM_LAUNCH_CHECK();
    size_t sort_bytes = w.sort_bytes;
    BSLAM_CUDA(cub::DeviceRadixSort::SortKeys(ws + w.sort, sort_bytes, keys_in, keys_out, n, 0, 63, st));
    const int n_leaf = host.n_in;
    int *parent_in = (int *)(ws + w.parent_in), *parent_leaf = (int *)(ws + w.parent_leaf), *arrivals = (int *)(ws + w.arrivals);
    BSLAM_CUDA(cudaMemsetAsync(arrivals, 0, 4 * (size_t)n, st));
    mesh_hierarchy_kernel<<<(unsigned)((n_leaf + 255) / 256) + 1, 256, 0, st>>>(keys_out, n_leaf, (char *)d_bvh, parent_in, parent_leaf);
    BSLAM_LAUNCH_CHECK();
    if (n_leaf > 0) {
        mesh_fit_kernel<<<(unsigned)((n_leaf + 255) / 256), 256, 0, st>>>(keys_out, n_leaf, recs, (char *)d_bvh, parent_in, parent_leaf, arrivals);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

int bslam_mesh_cast_rays(const void *d_bvh, const float *d_rays, int64_t n, float *d_t_hit, uint32_t *d_geom_ids, uint32_t *d_prim_ids, float *d_uvs,
                         float *d_normals, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(n >= 0, "bslam_mesh_cast_rays: n = %lld < 0", (long long)n);
    if (n == 0) return BSLAM_OK;
    BSLAM_CHECK_ARG(d_bvh && d_rays && d_t_hit && d_geom_ids && d_prim_ids, "bslam_mesh_cast_rays: NULL argument");
    BSLAM_CHECK_ARG(n <= (int64_t)INT_MAX * 256, "bslam_mesh_cast_rays: too many rays (%lld)", (long long)n);
    cudaStream_t st = (cudaStream_t)stream;
    const char *bvh = (const char *)d_bvh;
    if (d_uvs && d_normals) mr_launch_rays<true, true>(bvh, d_rays, n, d_t_hit, d_geom_ids, d_prim_ids, d_uvs, d_normals, st);
    else if (d_uvs) mr_launch_rays<true, false>(bvh, d_rays, n, d_t_hit, d_geom_ids, d_prim_ids, d_uvs, d_normals, st);
    else if (d_normals) mr_launch_rays<false, true>(bvh, d_rays, n, d_t_hit, d_geom_ids, d_prim_ids, d_uvs, d_normals, st);
    else mr_launch_rays<false, false>(bvh, d_rays, n, d_t_hit, d_geom_ids, d_prim_ids, d_uvs, d_normals, st);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

int bslam_mesh_rays_pinhole(int F, int H, int W, const double *h_K, const double *h_extrinsics, float *d_rays, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(F >= 0 && H >= 0 && W >= 0, "[bslam_mesh_rays_pinhole] Unsupported image format. (F=%d H=%d W=%d)", F, H, W);
    if ((int64_t)F * H * W == 0) return BSLAM_OK;
    BSLAM_CHECK_ARG(h_K && h_extrinsics && d_rays, "bslam_mesh_rays_pinhole: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local MrPinhole ph;
    ph.W = W; ph.H = H;
    const int64_t n_pix = (int64_t)W * H;
    for (int f0 = 0; f0 < F; f0 += kMrMaxFrames) {
        ph.F = F - f0 < kMrMaxFrames ? F - f0 : kMrMaxFrames;
        for (int f = 0; f < ph.F; ++f) mr_pinhole_frame(h_K, h_extrinsics + (size_t)(f0 + f) * 16, ph.Mc[f]);
        mesh_rays_pinhole_kernel<<<mr_grid(W, H, ph.F), 256, 0, st>>>(ph, d_rays + 6 * f0 * n_pix);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

int bslam_mesh_cast_pinhole(const void *d_bvh, int F, int H, int W, const double *h_K, const double *h_extrinsics, float *d_t_hit, uint32_t *d_geom_ids,
                            uint32_t *d_prim_ids, float *d_uvs, float *d_normals, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(F >= 0 && H >= 0 && W >= 0, "[bslam_mesh_cast_pinhole] Unsupported image format. (F=%d H=%d W=%d)", F, H, W);
    if ((int64_t)F * H * W == 0) return BSLAM_OK;
    BSLAM_CHECK_ARG(d_bvh && h_K && h_extrinsics && d_t_hit && d_geom_ids && d_prim_ids, "bslam_mesh_cast_pinhole: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    const char *bvh = (const char *)d_bvh;
    static thread_local MrPinhole ph;
    ph.W = W; ph.H = H;
    const int64_t n_pix = (int64_t)W * H;
    for (int f0 = 0; f0 < F; f0 += kMrMaxFrames) {
        ph.F = F - f0 < kMrMaxFrames ? F - f0 : kMrMaxFrames;
        for (int f = 0; f < ph.F; ++f) mr_pinhole_frame(h_K, h_extrinsics + (size_t)(f0 + f) * 16, ph.Mc[f]);
        const dim3 grid = mr_grid(W, H, ph.F);
        const int64_t o = f0 * n_pix;
        float *t = d_t_hit + o, *uv = d_uvs ? d_uvs + 2 * o : nullptr, *nrm = d_normals ? d_normals + 3 * o : nullptr;
        uint32_t *g = d_geom_ids + o, *p = d_prim_ids + o;
        if (uv && nrm) mr_launch_pinhole<true, true>(grid, bvh, ph, t, g, p, uv, nrm, st);
        else if (uv) mr_launch_pinhole<true, false>(grid, bvh, ph, t, g, p, uv, nrm, st);
        else if (nrm) mr_launch_pinhole<false, true>(grid, bvh, ph, t, g, p, uv, nrm, st);
        else mr_launch_pinhole<false, false>(grid, bvh, ph, t, g, p, uv, nrm, st);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

} // extern "C"
