// K4 -- surface extraction (marching cubes + point cloud) for sm_100a.
//
// Semantics: Open3D extract_triangle_mesh / extract_point_cloud as reached from
// TSDF.extract_mesh / TSDF.extract_pcd (N/3DM/tsdf.py:39-43); restated in SURVEY.md
// Appendix A.4/A.5 and checked against oracle/o3d_oracle.c.
//
// One CTA pass per 8^3 brick (512 threads, one per voxel), and only for SURFACE CANDIDATES: bricks
// that may hold a tsdf < 1 (flag bit 1, set by the band path of the integration) or whose +x/+y/+z
// neighbours do -- a cube or an edge with a sign change has a negative corner, and that corner lies
// in such a brick.  The candidates are compacted in brick order (deterministic output) and walked by
// a persistent grid, so the cost follows the surface (~10^4 bricks at 512^3), not the volume
// (2.6 * 10^5), and is low enough for the reference's extract-every-frame cadence
// (N/3DM/slam.py:126,195).  Compaction is count -> prefix sum -> emit:
//   * warp ballots give, per 32-voxel chunk and axis, the mask of edges that own a vertex;
//     popc prefixes of the 48 mask words number the vertices inside a brick;
//   * a prefix sum over bricks gives each brick's vertex / triangle base;
//   * triangle corners are resolved to vertex ids with  base[b'] + prefix[b'][w] + popc(mask & lt)
//     of the OWNING brick b' -- no hash map, no atomics, deterministic output order.
#include <math.h>

#include "bslam_common.cuh"
#include "mc_tables.cuh"

namespace bslam {

constexpr int kMaskWordsPerBrick = 48; // 16 chunks of 32 voxels x 3 axes
constexpr int kR = 10;                 // staged region edge: voxels -1 .. 8 of the brick

struct McScratch {
    uint32_t *vmask;     // [nb][48]
    uint16_t *vprefix;   // [nb][48] exclusive popc prefix inside the brick
    uint32_t *nvert;     // [nb]
    uint32_t *ntri;      // [nb]
    uint32_t *vbase;     // [nb] exclusive prefix over bricks
    uint32_t *tbase;     // [nb]
    uint32_t *cand;      // [nb] 1 = surface candidate
    uint32_t *cbase;     // [nb] exclusive prefix of cand
    uint32_t *list;      // [nb] candidate bricks, ascending
    unsigned long long *totals; // [4]: vertices, triangles, candidates, -
    unsigned long long *scan_ws; // [2 * kScanMaxCtas] CTA totals / bases of the multi-CTA prefix sums
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static size_t mc_scratch_bytes(size_t nb) {
    return align_up(nb * kMaskWordsPerBrick * 4, 256) + align_up(nb * kMaskWordsPerBrick * 2, 256) + 7 * align_up(nb * 4, 256) + 256 + 2 * 2048 * 8;
}

static McScratch carve_mc(void *p0, size_t nb) {
    char *p = (char *)p0;
    McScratch s;
    s.vmask = (uint32_t *)p; p += align_up(nb * kMaskWordsPerBrick * 4, 256);
    s.vprefix = (uint16_t *)p; p += align_up(nb * kMaskWordsPerBrick * 2, 256);
    s.nvert = (uint32_t *)p; p += align_up(nb * 4, 256);
    s.ntri = (uint32_t *)p; p += align_up(nb * 4, 256);
    s.vbase = (uint32_t *)p; p += align_up(nb * 4, 256);
    s.tbase = (uint32_t *)p; p += align_up(nb * 4, 256);
    s.cand = (uint32_t *)p; p += align_up(nb * 4, 256);
    s.cbase = (uint32_t *)p; p += align_up(nb * 4, 256);
    s.list = (uint32_t *)p; p += align_up(nb * 4, 256);
    s.totals = (unsigned long long *)p; p += 256;
    s.scan_ws = (unsigned long long *)p;
    return s;
}

// {tsdf, weight} of local voxel (x,y,z); outside the box -> weight 0; z = -1 / nz -> halo planes
__device__ __forceinline__ float2 fetch_voxel(const VolView &v, const float2 *halo_lo, const float2 *halo_hi, int x, int y, int z) {
    if (x < 0 || y < 0 || x >= v.nx || y >= v.ny || z < -1 || z > v.nz) return make_float2(0.f, 0.f);
    if (z == -1) return halo_lo ? halo_lo[(int64_t)x * v.ny + y] : make_float2(0.f, 0.f);
    if (z == v.nz) return halo_hi ? halo_hi[(int64_t)x * v.ny + y] : make_float2(0.f, 0.f);
    return v.vox[voxel_slot(v, x, y, z)];
}

struct BrickClass {
    bool cube_valid;
    int cube_index;
    unsigned int vbits; // bit a: the edge from this voxel towards +axis a owns a vertex
};

__device__ __forceinline__ int ridx(int rx, int ry, int rz) { return (rz * kR + rx) * kR + ry; }

// Stage the 10^3 neighbourhood of brick (bx,by,bz) and classify the calling thread's voxel.
__device__ __forceinline__ BrickClass classify_brick(const VolView &v, const float2 *halo_lo, const float2 *halo_hi, int bx, int by, int bz,
                                                     float *s_t, uint8_t *s_ok, uint8_t *s_cv) {
    const int tid = threadIdx.x;
    for (int i = tid; i < kR * kR * kR; i += kBrickVox) {
        const int ry = i % kR, rx = (i / kR) % kR, rz = i / (kR * kR);
        const float2 t = fetch_voxel(v, halo_lo, halo_hi, bx * 8 - 1 + rx, by * 8 - 1 + ry, bz * 8 - 1 + rz);
        s_t[i] = t.x;
        s_ok[i] = t.y > v.w_min;
    }
    __syncthreads();
    // cube validity for the 9^3 cubes based at region coords [0,9)^3
    for (int i = tid; i < 9 * 9 * 9; i += kBrickVox) {
        const int cy = i % 9, cx = (i / 9) % 9, cz = i / 81;
        uint8_t ok = 1;
#pragma unroll
        for (int k = 0; k < 8; ++k) ok &= s_ok[ridx(cx + ((k & 1) ? 1 : 0), cy + ((k & 2) ? 1 : 0), cz + ((k & 4) ? 1 : 0))];
        s_cv[(cz * 9 + cx) * 9 + cy] = ok;
    }
    __syncthreads();
    const int ly = tid & 7, lx = (tid >> 3) & 7, lz = tid >> 6;
    const int rx = lx + 1, ry = ly + 1, rz = lz + 1;
    BrickClass c;
    c.cube_valid = s_cv[(rz * 9 + rx) * 9 + ry] != 0 && (bz * 8 + lz < v.nz); // cubes based on the halo_hi plane belong to the slab above
    c.cube_index = 0;
    if (c.cube_valid) {
        // Open3D corner order: (0,0,0),(1,0,0),(1,1,0),(0,1,0),(0,0,1),(1,0,1),(1,1,1),(0,1,1)
        const int sx[8] = {0, 1, 1, 0, 0, 1, 1, 0}, sy[8] = {0, 0, 1, 1, 0, 0, 1, 1}, sz[8] = {0, 0, 0, 0, 1, 1, 1, 1};
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (s_t[ridx(rx + sx[k], ry + sy[k], rz + sz[k])] < 0.0f) c.cube_index |= 1 << k;
    }
    c.vbits = 0;
    const bool own = (bx * 8 + lx < v.nx) && (by * 8 + ly < v.ny) && (bz * 8 + lz < v.nz) && s_ok[ridx(rx, ry, rz)];
    if (own) {
        const bool neg0 = s_t[ridx(rx, ry, rz)] < 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const int nx_ = rx + (a == 0), ny_ = ry + (a == 1), nz_ = rz + (a == 2);
            if (!s_ok[ridx(nx_, ny_, nz_)]) continue;
            if ((s_t[ridx(nx_, ny_, nz_)] < 0.0f) == neg0) continue;
            // the 4 cubes sharing this edge: base = voxel - {0,1} along the two other axes
            bool any = false;
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                int qx = rx, qy = ry, qz = rz;
                const int d0 = d & 1, d1 = d >> 1;
                if (a == 0) { qy -= d0; qz -= d1; }
                if (a == 1) { qx -= d0; qz -= d1; }
                if (a == 2) { qx -= d0; qy -= d1; }
                // cubes based on the halo_hi plane do not exist for this slab's vertices either:
                // they can only be reached from voxels of that plane, which are not owned here
                any |= s_cv[(qz * 9 + qx) * 9 + qy] != 0;
            }
            if (any) c.vbits |= 1u << a;
        }
    }
    return c;
}

template <bool EMIT>
__global__ void __launch_bounds__(kBrickVox) mc_brick_kernel(const VolView v, double vld, const float2 *halo_lo, const float2 *halo_hi,
                                                              const float *halo_hi_color, McScratch sc, float *vertices, int32_t *keys, float *colors, int64_t cap_v,
                                                              int32_t *tris, int64_t cap_t) {
    __shared__ float s_t[kR * kR * kR];
    __shared__ uint8_t s_ok[kR * kR * kR];
    __shared__ uint8_t s_cv[9 * 9 * 9];
    __shared__ uint32_t s_mask[kMaskWordsPerBrick];
    __shared__ uint32_t s_pref[kMaskWordsPerBrick];
    __shared__ uint32_t s_wtri[16];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned int n_cand = (unsigned int)sc.totals[2];
  for (unsigned int ci = blockIdx.x; ci < n_cand; ci += gridDim.x) {      // persistent grid over the candidate list
    __syncthreads();                                                       // shared buffers of the previous brick are free
    const int64_t b = sc.list[ci];
    if (EMIT && sc.nvert[b] == 0 && sc.ntri[b] == 0) continue;
    const int bx = (int)(b % v.nbx), by = (int)((b / v.nbx) % v.nby), bz = (int)(b / ((int64_t)v.nbx * v.nby));
    const BrickClass c = classify_brick(v, halo_lo, halo_hi, bx, by, bz, s_t, s_ok, s_cv);

    // vertex masks: word 3*chunk + axis, chunk == warp id (in-brick index == tid)
    unsigned int bal[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        bal[a] = __ballot_sync(0xffffffffu, (c.vbits >> a) & 1u);
        if (lane == 0) s_mask[3 * wid + a] = bal[a];
    }
    int ntri = c.cube_valid ? (int)kNumTris[c.cube_index] : 0;
    // block scan of triangle counts (exclusive) -- warp scan + warp totals
    int inc = ntri;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_wtri[wid] = inc;
    __syncthreads();
    if (tid == 0) {
        uint32_t acc = 0;
        for (int w = 0; w < kMaskWordsPerBrick; ++w) { s_pref[w] = acc; acc += __popc(s_mask[w]); }
        uint32_t tacc = 0;
        for (int w = 0; w < 16; ++w) { const uint32_t t = s_wtri[w]; s_wtri[w] = tacc; tacc += t; }
        if (!EMIT) { sc.nvert[b] = acc; sc.ntri[b] = tacc; }
    }
    __syncthreads();
    if (!EMIT) {
        if (tid < kMaskWordsPerBrick) {
            sc.vmask[b * kMaskWordsPerBrick + tid] = s_mask[tid];
            sc.vprefix[b * kMaskWordsPerBrick + tid] = (uint16_t)s_pref[tid];
        }
        continue;
    }
    // ---------------- emit vertices
    const int ly = tid & 7, lx = (tid >> 3) & 7, lz = tid >> 6;
    const int X = bx * 8 + lx, Y = by * 8 + ly, Z = bz * 8 + lz;
    const uint32_t vb = sc.vbase[b];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        if (!((c.vbits >> a) & 1u)) continue;
        const int64_t id = (int64_t)vb + s_pref[3 * wid + a] + __popc(bal[a] & ((1u << lane) - 1u));
        if (id >= cap_v) continue;
        const int rx = lx + 1, ry = ly + 1, rz = lz + 1;
        const double f0 = fabs((double)s_t[ridx(rx, ry, rz)]);
        const double f1 = fabs((double)s_t[ridx(rx + (a == 0), ry + (a == 1), rz + (a == 2))]);
        // Open3D: pt = half + vl * (x,y,z) (f64); pt[axis] += f0 * vl / (f0 + f1); + origin
        double pt[3] = {v.pos_half * vld + vld * X, v.pos_half * vld + vld * Y, v.pos_half * vld + vld * (Z + v.gz0)};
        pt[a] += f0 * vld / (f0 + f1);
        vertices[3 * id + 0] = (float)(pt[0] + v.ox);
        vertices[3 * id + 1] = (float)(pt[1] + v.oy);
        vertices[3 * id + 2] = (float)(pt[2] + v.oz);
        if (keys) { keys[4 * id + 0] = X; keys[4 * id + 1] = Y; keys[4 * id + 2] = Z; keys[4 * id + 3] = a; }
        if (colors && v.color) {
            const int64_t s0 = voxel_slot(v, X, Y, Z);
            const int X1 = X + (a == 0), Y1 = Y + (a == 1), Z1 = Z + (a == 2);
            // the far end of a z-edge from the top plane lies on the halo_hi plane: its colour comes from the slab above
            const bool hi = Z1 >= v.nz;
            const int64_t s1 = hi ? 0 : voxel_slot(v, X1, Y1, Z1);
            for (int k = 0; k < 3; ++k) {
                const double c0 = v.color[(s0 / kBrickVox) * (3 * kBrickVox) + k * kBrickVox + (s0 % kBrickVox)];
                const double c1 = hi ? halo_hi_color[((int64_t)X1 * v.ny + Y1) * 3 + k]
                                     : v.color[(s1 / kBrickVox) * (3 * kBrickVox) + k * kBrickVox + (s1 % kBrickVox)];
                colors[3 * id + k] = (float)(((f1 * c0 + f0 * c1) / (f0 + f1)) / 255.0);
            }
        }
    }
    // ---------------- emit triangles
    if (ntri) {
        int64_t t_out = (int64_t)sc.tbase[b] + s_wtri[wid] + (inc - ntri);
        const int8_t *row = kTriTable + c.cube_index * 16;
        for (int i = 0; i < ntri; ++i, ++t_out) {
            if (t_out >= cap_t) break;
            int32_t ids[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int e = row[3 * i + k];
                const int ox_ = X + kEdgeShift[4 * e + 0], oy_ = Y + kEdgeShift[4 * e + 1], oz_ = Z + kEdgeShift[4 * e + 2];
                const int ax = kEdgeShift[4 * e + 3];
                if (oz_ >= v.nz) { // owned by the first plane of the slab above
                    ids[k] = -(1 + (ox_ * v.ny + oy_) * 4 + ax);
                    continue;
                }
                const int64_t ob = ((int64_t)(oz_ >> 3) * v.nby + (oy_ >> 3)) * v.nbx + (ox_ >> 3);
                const int in = ((oz_ & 7) << 6) + ((ox_ & 7) << 3) + (oy_ & 7);
                const int w = 3 * (in >> 5) + ax;
                const uint32_t m = sc.vmask[ob * kMaskWordsPerBrick + w];
                ids[k] = (int32_t)(sc.vbase[ob] + sc.vprefix[ob * kMaskWordsPerBrick + w] + __popc(m & ((1u << (in & 31)) - 1u)));
            }
            // Open3D pushes (e[t0], e[t2], e[t1])
            tris[3 * t_out + 0] = ids[0];
            tris[3 * t_out + 1] = ids[2];
            tris[3 * t_out + 2] = ids[1];
        }
    }
  }
}

// exclusive prefix sums over bricks of up to two arrays, three small launches:
//   scan_partial_kernel : every CTA scans its own 8192 entries (8 per thread: warp-shuffle scan + 32 warp totals),
//                         writes the CTA-local exclusive prefixes and the CTA totals;
//   scan_totals_kernel  : one CTA scans the (<= 2048) CTA totals -> CTA bases + grand totals;
//   scan_add_kernel     : adds the CTA base to every entry.
// (The single-CTA scan this replaces took 220 - 380 us for the 262 144 bricks of a 512^3 volume -- 40 % of a
// per-frame extract_pcd at the SLAM loop's cadence; the three launches take ~10 us together.)
constexpr int kScanPer = 8;
constexpr int kScanChunk = 1024 * kScanPer;
constexpr int kScanMaxCtas = 2048;     // 16.7 M bricks

__global__ void __launch_bounds__(1024) scan_partial_kernel(const uint32_t *a, const uint32_t *b, uint32_t *abase, uint32_t *bbase, int64_t n,
                                                            unsigned long long *cta_tot) {
    __shared__ unsigned long long s_wa[32], s_wb[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t i0 = (int64_t)blockIdx.x * kScanChunk + (int64_t)threadIdx.x * kScanPer;
    uint32_t va[kScanPer], vb[kScanPer];
    unsigned long long la = 0, lb = 0;
#pragma unroll
    for (int k = 0; k < kScanPer; ++k) {
        va[k] = (i0 + k < n) ? a[i0 + k] : 0u;
        vb[k] = (b && i0 + k < n) ? b[i0 + k] : 0u;
        la += va[k]; lb += vb[k];
    }
    unsigned long long ia = la, ib = lb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += ta; ib += tb; }
    }
    if (lane == 31) { s_wa[wid] = ia; s_wb[wid] = ib; }
    __syncthreads();
    if (wid == 0) {
        const unsigned long long wa = s_wa[lane], wb = s_wb[lane];
        unsigned long long xa = wa, xb = wb;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long ta = __shfl_up_sync(0xffffffffu, xa, o), tb = __shfl_up_sync(0xffffffffu, xb, o);
            if (lane >= o) { xa += ta; xb += tb; }
        }
        s_wa[lane] = xa - wa; s_wb[lane] = xb - wb;     // exclusive over warps
        if (lane == 31) { cta_tot[2 * blockIdx.x] = xa; cta_tot[2 * blockIdx.x + 1] = xb; }
    }
    __syncthreads();
    unsigned long long ea = s_wa[wid] + ia - la, eb = s_wb[wid] + ib - lb;
#pragma unroll
    for (int k = 0; k < kScanPer; ++k) {
        if (i0 + k < n) {
            abase[i0 + k] = (uint32_t)ea;
            if (b) bbase[i0 + k] = (uint32_t)eb;
        }
        ea += va[k]; eb += vb[k];
    }
}

__global__ void __launch_bounds__(1024) scan_totals_kernel(unsigned long long *cta_tot, int n_ctas, unsigned long long *totals) {
    __shared__ unsigned long long s_wa[32], s_wb[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // two CTA totals per thread
    unsigned long long a[2] = {0, 0}, b[2] = {0, 0};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int i = 2 * threadIdx.x + k;
        if (i < n_ctas) { a[k] = cta_tot[2 * i]; b[k] = cta_tot[2 * i + 1]; }
    }
    unsigned long long ia = a[0] + a[1], ib = b[0] + b[1];
    const unsigned long long la = ia, lb = ib;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += ta; ib += tb; }
    }
    if (lane == 31) { s_wa[wid] = ia; s_wb[wid] = ib; }
    __syncthreads();
    if (wid == 0) {
        const unsigned long long wa = s_wa[lane], wb = s_wb[lane];
        unsigned long long xa = wa, xb = wb;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long ta = __shfl_up_sync(0xffffffffu, xa, o), tb = __shfl_up_sync(0xffffffffu, xb, o);
            if (lane >= o) { xa += ta; xb += tb; }
        }
        s_wa[lane] = xa - wa; s_wb[lane] = xb - wb;
        if (lane == 31) { totals[0] = xa; totals[1] = xb; }
    }
    __syncthreads();
    unsigned long long ea = s_wa[wid] + ia - la, eb = s_wb[wid] + ib - lb;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int i = 2 * threadIdx.x + k;
        if (i < n_ctas) { cta_tot[2 * i] = ea; cta_tot[2 * i + 1] = eb; }     // in place: totals -> exclusive bases
        ea += a[k]; eb += b[k];
    }
}

__global__ void __launch_bounds__(1024) scan_add_kernel(uint32_t *abase, uint32_t *bbase, int64_t n, const unsigned long long *cta_base) {
    if (blockIdx.x == 0) return;       // base 0
    const uint32_t ba = (uint32_t)cta_base[2 * blockIdx.x], bb = (uint32_t)cta_base[2 * blockIdx.x + 1];
    const int64_t i0 = (int64_t)blockIdx.x * kScanChunk + (int64_t)threadIdx.x * kScanPer;
#pragma unroll
    for (int k = 0; k < kScanPer; ++k)
        if (i0 + k < n) {
            abase[i0 + k] += ba;
            if (bbase) bbase[i0 + k] += bb;
        }
}

// a, b (optional) -> exclusive prefixes abase, bbase; totals[0..1] = grand totals.  scan_ws: 2 * kScanMaxCtas u64.
static int brick_scan(const uint32_t *a, const uint32_t *b, uint32_t *abase, uint32_t *bbase, int64_t n, unsigned long long *totals,
                      unsigned long long *scan_ws, cudaStream_t st) {
    const int n_ctas = (int)((n + kScanChunk - 1) / kScanChunk);
    BSLAM_CHECK_ARG(n_ctas <= kScanMaxCtas, "surface extraction: too many bricks (%lld)", (long long)n);
    scan_partial_kernel<<<n_ctas, 1024, 0, st>>>(a, b, abase, bbase, n, scan_ws);
    BSLAM_LAUNCH_CHECK();
    scan_totals_kernel<<<1, 1024, 0, st>>>(scan_ws, n_ctas, totals);
    BSLAM_LAUNCH_CHECK();
    if (n_ctas > 1) {
        scan_add_kernel<<<n_ctas, 1024, 0, st>>>(abase, b ? bbase : nullptr, n, scan_ws);
        BSLAM_LAUNCH_CHECK();
    }
    return BSLAM_OK;
}

// surface candidates: brick b is looked at if any of the 8 bricks b + {0,1}^3 may hold a tsdf < 1
// (flag bit 1); with a halo plane above, the top brick layer is kept whenever it was touched at
// all (the slab above keeps its own flags).  Also clears the per-brick counts of the others.
__global__ void mc_mark_kernel(const VolView v, int have_halo_hi, McScratch sc) {
    const int64_t nb = brick_count(v);
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (int64_t)gridDim.x * blockDim.x) {
        const int bx = (int)(b % v.nbx), by = (int)((b / v.nbx) % v.nby), bz = (int)(b / ((int64_t)v.nbx * v.nby));
        unsigned int any = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int x = bx + (k & 1), y = by + ((k >> 1) & 1), z = bz + (k >> 2);
            if (x < v.nbx && y < v.nby && z < v.nbz) any |= v.flags[((int64_t)z * v.nby + y) * v.nbx + x] & 2u;
        }
        if (have_halo_hi && bz == v.nbz - 1) any |= v.flags[b] & 1u;
        sc.cand[b] = any ? 1u : 0u;
        sc.nvert[b] = 0; sc.ntri[b] = 0;
    }
}

__global__ void mc_list_kernel(int64_t nb, McScratch sc) {
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (int64_t)gridDim.x * blockDim.x)
        if (sc.cand[b]) sc.list[sc.cbase[b]] = (uint32_t)b;
}

// ---------------------------------------------------------------- incremental point extraction (row f1)
// The SLAM loop extracts the point cloud after EVERY frame (N/3DM/slam.py:126,195) while a frame only changes the bricks
// it sees.  K3 raises flag bit 2 ("changed since the last incremental extraction") on every brick it updates; a brick's
// points depend on its own voxels and on its 26 neighbours' (the +1 voxel of an edge, the -1 .. +2 stencil of the
// normals), so a brick is RE-EXTRACTED when any brick of its 3 x 3 x 3 neighbourhood carries the bit; every other
// candidate brick's points are copied from a per-brick cache slot (<= 128 points; larger bricks are always recomputed).
// The output is the same array, in the same order, as the full extraction's.
constexpr uint32_t kNone = 0xffffffffu;
constexpr int kSlotPts = 128;
constexpr int kSlotWords = 13 * kSlotPts;      // xyz | normal | rgb | key(4) per point, structure of arrays inside a slot
struct PtsCache {
    uint32_t *slot;    // [nb] cache slot of the brick, kNone = none
    uint32_t *cnt;     // [nb] cached point count, kNone = unknown / not cached -> recomputed every time
    uint32_t *need;    // [nb] 1 = recompute in this extraction
    uint32_t *used;    // [1] slots handed out so far
    float *pool;       // [n_slots][kSlotWords]
    uint32_t n_slots;
};

__global__ void pts_need_kernel(const VolView v, McScratch sc, PtsCache pc, int valid) {
    const int64_t nb = brick_count(v);
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (int64_t)gridDim.x * blockDim.x) {
        const bool cand = sc.cand[b] != 0;
        bool need = false;
        if (cand) {
            need = !valid || pc.cnt[b] == kNone;
            if (!need) {
                const int bx = (int)(b % v.nbx), by = (int)((b / v.nbx) % v.nby), bz = (int)(b / ((int64_t)v.nbx * v.nby));
                unsigned int any = 0;
                for (int dz = -1; dz <= 1; ++dz)
                    for (int dy = -1; dy <= 1; ++dy)
                        for (int dx = -1; dx <= 1; ++dx) {
                            const int x = bx + dx, y = by + dy, z = bz + dz;
                            if (x >= 0 && y >= 0 && z >= 0 && x < v.nbx && y < v.nby && z < v.nbz) any |= v.flags[((int64_t)z * v.nby + y) * v.nbx + x] & 4u;
                        }
                need = any != 0;
            }
        }
        pc.need[b] = need ? 1u : 0u;
        sc.nvert[b] = (cand && !need) ? pc.cnt[b] : 0u;     // clean bricks keep their cached count; the count pass fills the others
        if (need) atomicAdd(sc.totals + 3, 1ull);           // statistics: bricks recomputed by this extraction
    }
}

__global__ void pts_clear_dirty_kernel(const VolView v) {
    const int64_t nb = brick_count(v);
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (int64_t)gridDim.x * blockDim.x)
        if (v.flags[b] & 4u) v.flags[b] &= (uint8_t)~4u;
}

// ---------------------------------------------------------------- surface points (A.5)
__device__ __forceinline__ bool pt_ok(const VolView &v, float2 t) { return t.y > v.w_min && t.x < 0.98f && t.x >= -0.98f; }

__device__ double tsdf_at(const VolView &v, double vl, const double *p) {
    int idx[3]; double r[3];
    for (int i = 0; i < 3; ++i) {
        const double g = p[i] / vl - v.pos_half;
        idx[i] = (int)floor(g);
        r[i] = g - (double)idx[i];
    }
    double t = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { // Open3D term order: (0,0,0),(0,0,1),(0,1,0),(0,1,1),(1,0,0),...
        const int a = (k >> 2) & 1, b = (k >> 1) & 1, c = k & 1;
        const double wgt = (a ? r[0] : 1 - r[0]) * (b ? r[1] : 1 - r[1]) * (c ? r[2] : 1 - r[2]);
        t += wgt * (double)v.vox[voxel_slot(v, idx[0] + a, idx[1] + b, idx[2] + c)].x;
    }
    return t;
}

// trilinear TSDF at local position p from the staged (11^3) neighbourhood of the brick: voxels -1 .. 9 per axis
// (a point of voxel X along axis a needs X - 1 .. X + 2, see A.5), same term order as tsdf_at
constexpr int kPR = 11;
__device__ __forceinline__ double tsdf_at_staged(const float *s_t, double vl, double pos_half, int bx8, int by8, int bz8, const double *p) {
    int idx[3]; double r[3];
    for (int i = 0; i < 3; ++i) {
        const double g = p[i] / vl - pos_half;
        idx[i] = (int)floor(g);
        r[i] = g - (double)idx[i];
    }
    const int rx = idx[0] - bx8 + 1, ry = idx[1] - by8 + 1, rz = idx[2] - bz8 + 1;
    double t = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { // Open3D term order: (0,0,0),(0,0,1),(0,1,0),(0,1,1),(1,0,0),...
        const int a = (k >> 2) & 1, b = (k >> 1) & 1, c = k & 1;
        const double wgt = (a ? r[0] : 1 - r[0]) * (b ? r[1] : 1 - r[1]) * (c ? r[2] : 1 - r[2]);
        t += wgt * (double)s_t[((rz + c) * kPR + (rx + a)) * kPR + (ry + b)];
    }
    return t;
}

// pc.need != NULL: incremental mode (see above) -- the count pass only visits the bricks to recompute, the emit pass
// recomputes those (and refreshes their cache slot) and copies the others from the cache
template <bool EMIT>
__global__ void __launch_bounds__(kBrickVox) points_brick_kernel(const VolView v, double vl, McScratch sc, float *points, float *normals,
                                                                  float *colors, int32_t *keys, int64_t cap, PtsCache pc) {
    __shared__ uint32_t s_w[16];
    __shared__ float s_t[EMIT ? kPR * kPR * kPR : 1];
    __shared__ uint32_t s_slot;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned int n_cand = (unsigned int)sc.totals[2];
  for (unsigned int ci = blockIdx.x; ci < n_cand; ci += gridDim.x) {      // persistent grid over the candidate list
    __syncthreads();
    const int64_t b = sc.list[ci];
    const bool incremental = pc.need != nullptr;
    if (incremental && !pc.need[b]) {
        if (!EMIT) continue;
        // clean brick: its points come from the cache, in the order they were emitted
        const uint32_t n = sc.nvert[b], sl = pc.slot[b];
        if (n == 0 || sl == kNone) continue;
        const float *src = pc.pool + (size_t)sl * kSlotWords;
        const int64_t o0 = (int64_t)sc.vbase[b];
        for (uint32_t i = tid; i < n; i += kBrickVox) {
            const int64_t o = o0 + i;
            if (o >= cap) continue;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                points[3 * o + k] = src[k * kSlotPts + i];
                if (normals) normals[3 * o + k] = src[(3 + k) * kSlotPts + i];
                if (colors && v.color) colors[3 * o + k] = src[(6 + k) * kSlotPts + i];
            }
            if (keys)
#pragma unroll
                for (int k = 0; k < 4; ++k) keys[4 * o + k] = __float_as_int(src[(9 + k) * kSlotPts + i]);
        }
        continue;
    }
    if (EMIT && sc.nvert[b] == 0) continue;
    const int bx = (int)(b % v.nbx), by = (int)((b / v.nbx) % v.nby), bz = (int)(b / ((int64_t)v.nbx * v.nby));
    if (EMIT && normals) {
        // the tsdf of voxels -1 .. 9 of the brick per axis (0 outside the box; never read for a valid point)
        for (int i = tid; i < kPR * kPR * kPR; i += kBrickVox) {
            const int ry = i % kPR, rx = (i / kPR) % kPR, rz = i / (kPR * kPR);
            const int x = bx * 8 - 1 + rx, y = by * 8 - 1 + ry, z = bz * 8 - 1 + rz;
            s_t[i] = (x >= 0 && y >= 0 && z >= 0 && x < v.nx && y < v.ny && z < v.nz) ? v.vox[voxel_slot(v, x, y, z)].x : 0.0f;
        }
    }
    const int ly = tid & 7, lx = (tid >> 3) & 7, lz = tid >> 6;
    const int X = bx * 8 + lx, Y = by * 8 + ly, Z = bz * 8 + lz;
    const int n[3] = {v.nx, v.ny, v.nz};
    unsigned int bits = 0;
    float2 t0 = make_float2(0.f, 0.f), t1[3];
    if (X >= 1 && Y >= 1 && Z >= 1 && X < v.nx - 1 && Y < v.ny - 1 && Z < v.nz - 1) {
        t0 = v.vox[b * kBrickVox + tid];
        if (pt_ok(v, t0)) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const int c1[3] = {X + (a == 0), Y + (a == 1), Z + (a == 2)};
                if (!(c1[a] < n[a] - 1)) continue;
                t1[a] = v.vox[voxel_slot(v, c1[0], c1[1], c1[2])];
                if (pt_ok(v, t1[a]) && t0.x * t1[a].x < 0) bits |= 1u << a;
            }
        }
    }
    const int cnt = __popc(bits);
    int inc = cnt;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_w[wid] = inc;
    __syncthreads();
    if (tid == 0) {
        uint32_t acc = 0;
        for (int w = 0; w < 16; ++w) { const uint32_t t = s_w[w]; s_w[w] = acc; acc += t; }
        if (!EMIT) {
            sc.nvert[b] = acc;
            if (incremental && acc == 0) pc.cnt[b] = 0;      // nothing to cache: clean until a neighbour changes
        } else if (incremental) {
            // cache slot for the recomputed brick (kept if it has one; a new one while the pool lasts; none if too large)
            uint32_t sl = kNone;
            if (acc <= (uint32_t)kSlotPts) {
                sl = pc.slot[b];
                if (sl == kNone) {
                    const uint32_t got = atomicAdd(pc.used, 1u);
                    if (got < pc.n_slots) { sl = got; pc.slot[b] = sl; }
                }
            }
            s_slot = sl;
            pc.cnt[b] = (sl != kNone) ? acc : kNone;
        }
    }
    __syncthreads();
    if (!EMIT || !cnt) continue;
    const int64_t li0 = (int64_t)s_w[wid] + (inc - cnt);        // index of this voxel's first point inside the brick
    float *cache = (incremental && s_slot != kNone) ? pc.pool + (size_t)s_slot * kSlotWords : nullptr;
    int64_t li = li0;
    int64_t o = (int64_t)sc.vbase[b] + li0;
    const double half = vl * v.pos_half, half_gap = 0.99 * vl;
    const double p0[3] = {half + vl * X, half + vl * Y, half + vl * Z};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        if (!((bits >> a) & 1u)) continue;
        if (o < cap) {
            const float r0 = fabsf(t0.x), r1 = fabsf(t1[a].x);
            double p[3] = {p0[0], p0[1], p0[2]};
            p[a] = (p0[a] * r1 + (p0[a] + vl) * r0) / (r0 + r1);
            points[3 * o + 0] = (float)(p[0] + v.ox);
            points[3 * o + 1] = (float)(p[1] + v.oy);
            points[3 * o + 2] = (float)(p[2] + v.oz + vl * v.gz0);
            if (keys) { keys[4 * o + 0] = X; keys[4 * o + 1] = Y; keys[4 * o + 2] = Z; keys[4 * o + 3] = a; }
            if (cache) {
                cache[0 * kSlotPts + li] = points[3 * o + 0]; cache[1 * kSlotPts + li] = points[3 * o + 1]; cache[2 * kSlotPts + li] = points[3 * o + 2];
                cache[9 * kSlotPts + li] = __int_as_float(X); cache[10 * kSlotPts + li] = __int_as_float(Y);
                cache[11 * kSlotPts + li] = __int_as_float(Z); cache[12 * kSlotPts + li] = __int_as_float(a);
            }
            if (normals) {
                double nn[3];
                for (int k = 0; k < 3; ++k) {
                    double q0[3] = {p[0], p[1], p[2]}, q1[3] = {p[0], p[1], p[2]};
                    q0[k] -= half_gap; q1[k] += half_gap;
                    nn[k] = tsdf_at_staged(s_t, vl, v.pos_half, bx * 8, by * 8, bz * 8, q1) - tsdf_at_staged(s_t, vl, v.pos_half, bx * 8, by * 8, bz * 8, q0);
                }
                const double len = sqrt(nn[0] * nn[0] + nn[1] * nn[1] + nn[2] * nn[2]);
                for (int k = 0; k < 3; ++k) {
                    normals[3 * o + k] = (float)(len > 0 ? nn[k] / len : nn[k]);
                    if (cache) cache[(3 + k) * kSlotPts + li] = normals[3 * o + k];
                }
            }
            if (colors && v.color) {
                const int64_t s0 = b * kBrickVox + tid;
                const int64_t s1 = voxel_slot(v, X + (a == 0), Y + (a == 1), Z + (a == 2));
                for (int k = 0; k < 3; ++k) {
                    const double c0 = v.color[(s0 / kBrickVox) * (3 * kBrickVox) + k * kBrickVox + (s0 % kBrickVox)];
                    const double c1 = v.color[(s1 / kBrickVox) * (3 * kBrickVox) + k * kBrickVox + (s1 % kBrickVox)];
                    colors[3 * o + k] = (float)(((c0 * r1 + c1 * r0) / (r0 + r1)) / 255.0);
                    if (cache) cache[(6 + k) * kSlotPts + li] = colors[3 * o + k];
                }
            }
        }
        ++o; ++li;
    }
  }
}

// candidate list of the volume -> sc.list / sc.totals[2] (shared by marching cubes and point extraction)
static int build_candidates(bslam_volume *vol, const McScratch &sc, int have_halo_hi, cudaStream_t st) {
    const int64_t nb = brick_count(vol->v);
    mc_mark_kernel<<<num_sms(vol->device) * 4, 256, 0, st>>>(vol->v, have_halo_hi, sc);
    BSLAM_LAUNCH_CHECK();
    const int rc = brick_scan(sc.cand, nullptr, sc.cbase, nullptr, nb, sc.totals + 2, sc.scan_ws, st);
    if (rc) return rc;
    mc_list_kernel<<<num_sms(vol->device) * 4, 256, 0, st>>>(nb, sc);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}
#define kExtractGrid (num_sms(vol->device) * 3)   /* persistent CTAs of 512 threads (3 resident per SM) */

// ---------------------------------------------------------------- gather-side merge of per-slab meshes
// The slabs' vertex keys / triangles are concatenated (bottom slab first).  Pass 1 (vertices): global z of
// the key, and the vertices on every slab's plane 0 are entered into a per-slab table indexed by the edge code
// (x * ny + y) * 4 + axis.  Pass 2 (triangle corners): local id -> + slab base; a negative id
// -(1 + code) refers to the vertex on edge `code` of the NEXT slab's plane 0 (bslam_mc_emit) -> table.
constexpr int kMaxSlabs = 64;
struct MergeP {
    int n;
    long long vend[kMaxSlabs];   // exclusive end of slab s in the vertex array (vend[s-1] = its base)
    long long tend[kMaxSlabs];
    int zoff[kMaxSlabs];
};

__device__ __forceinline__ int slab_of(const long long *end, int n, long long i) {
    int s = 0;
    while (s < n - 1 && i >= end[s]) ++s;
    return s;
}

__global__ void merge_vertices_kernel(const __grid_constant__ MergeP mp, int32_t *keys, long long nv, int ny, long long table_stride, int32_t *table) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nv) return;
    const int s = slab_of(mp.vend, mp.n, i);
    int4 k = reinterpret_cast<int4 *>(keys)[i];
    if (k.z == 0) table[(long long)s * table_stride + ((long long)k.x * ny + k.y) * 4 + k.w] = (int32_t)i;
    k.z += mp.zoff[s];
    reinterpret_cast<int4 *>(keys)[i] = k;
}

__global__ void merge_triangles_kernel(const __grid_constant__ MergeP mp, int32_t *tris, long long nt, long long table_stride, const int32_t *table,
                                       unsigned int *unresolved) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nt) return;
    const int s = slab_of(mp.tend, mp.n, i);
    const long long base = s ? mp.vend[s - 1] : 0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int32_t id = tris[3 * i + c];
        int32_t out;
        if (id >= 0) {
            out = (int32_t)(id + base);
        } else {
            const long long code = -(long long)id - 1;
            out = (s + 1 < mp.n && code < table_stride) ? table[(long long)(s + 1) * table_stride + code] : -1;
            if (out < 0) atomicAdd(unresolved, 1u);
        }
        tris[3 * i + c] = out;
    }
}

static int ensure_mc_scratch(bslam_volume *vol) {
    const size_t nb = (size_t)brick_count(vol->v);
    const size_t need = mc_scratch_bytes(nb);
    if (vol->mc_scratch && vol->mc_scratch_bytes >= need) return BSLAM_OK;
    if (vol->mc_scratch) cudaFree(vol->mc_scratch);
    vol->mc_scratch = nullptr;
    BSLAM_CUDA(cudaMalloc(&vol->mc_scratch, need));
    vol->mc_scratch_bytes = need;
    return BSLAM_OK;
}

static uint32_t pts_cache_slots(size_t nb) { return (uint32_t)(nb < 49152 ? nb : 49152); }
static size_t pts_cache_bytes(size_t nb) {
    return 3 * align_up(nb * 4, 256) + 256 + (size_t)pts_cache_slots(nb) * kSlotWords * sizeof(float);
}
static PtsCache carve_pts(void *p0, size_t nb) {
    char *p = (char *)p0;
    PtsCache c;
    c.slot = (uint32_t *)p; p += align_up(nb * 4, 256);
    c.cnt = (uint32_t *)p; p += align_up(nb * 4, 256);
    c.need = (uint32_t *)p; p += align_up(nb * 4, 256);
    c.used = (uint32_t *)p; p += 256;
    c.pool = (float *)p;
    c.n_slots = pts_cache_slots(nb);
    return c;
}
static PtsCache no_cache() {
    PtsCache c;
    memset(&c, 0, sizeof(c));
    return c;
}

} // namespace bslam

using namespace bslam;

extern "C" {

int bslam_points_set_incremental(bslam_volume *vol, int enable, int with_normals) {
    BSLAM_CHECK_ARG(vol != nullptr, "bslam_points_set_incremental: vol is NULL");
    BSLAM_CHECK_ARG(!enable || (vol->v.gz0 == 0 && vol->v.zs == 1), "bslam_points_set_incremental: single-box volumes only");
    vol->pts_incremental = enable ? 1 : 0;
    vol->pts_with_normals = with_normals ? 1 : 0;
    vol->pts_cache_valid = 0;
    return BSLAM_OK;
}

int bslam_points_last_stats(const bslam_volume *vol, long long *h_stat2) {
    BSLAM_CHECK_ARG(vol && h_stat2, "bslam_points_last_stats: NULL argument");
    h_stat2[0] = vol->pts_last_candidates;
    h_stat2[1] = vol->pts_last_recomputed;
    return BSLAM_OK;
}

int bslam_mc_count(bslam_volume *vol, const float *d_halo_lo, const float *d_halo_hi, int64_t *h_counts, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(vol && h_counts, "bslam_mc_count: NULL argument");
    BSLAM_CHECK_ARG(vol->v.zs == 1, "bslam_mc_count: interleaved slabs must be re-sharded to contiguous ones first");
    BSLAM_DEVICE_GUARD(vol->device);
    int rc = ensure_mc_scratch(vol);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nb = brick_count(vol->v);
    const McScratch sc = carve_mc(vol->mc_scratch, (size_t)nb);
    rc = build_candidates(vol, sc, d_halo_hi != nullptr, st);
    if (rc) return rc;
    mc_brick_kernel<false><<<kExtractGrid, kBrickVox, 0, st>>>(vol->v, vol->voxel_length_d, (const float2 *)d_halo_lo, (const float2 *)d_halo_hi, nullptr, sc,
                                                               nullptr, nullptr, nullptr, 0, nullptr, 0);
    BSLAM_LAUNCH_CHECK();
    rc = brick_scan(sc.nvert, sc.ntri, sc.vbase, sc.tbase, nb, sc.totals, sc.scan_ws, st);
    if (rc) return rc;
    unsigned long long tot[2];
    BSLAM_CUDA(cudaMemcpyAsync(tot, sc.totals, 16, cudaMemcpyDeviceToHost, st));
    BSLAM_CUDA(cudaStreamSynchronize(st));
    h_counts[0] = (int64_t)tot[0];
    h_counts[1] = (int64_t)tot[1];
    return BSLAM_OK;
}

int bslam_mc_emit(bslam_volume *vol, const float *d_halo_lo, const float *d_halo_hi, const float *d_halo_hi_color, float *d_vertices,
                  int32_t *d_keys, float *d_colors, int64_t cap_v, int32_t *d_tri, int64_t cap_t, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(vol && vol->mc_scratch, "bslam_mc_emit: call bslam_mc_count first");
    BSLAM_CHECK_ARG((d_vertices || cap_v == 0) && (d_tri || cap_t == 0), "bslam_mc_emit: NULL output");
    BSLAM_CHECK_ARG(!(d_colors && vol->v.color && d_halo_hi && !d_halo_hi_color),
                    "bslam_mc_emit: colours with a halo_hi plane need its colour plane (bslam_tsdf_export_plane_color)");
    BSLAM_DEVICE_GUARD(vol->device);
    const int64_t nb = brick_count(vol->v);
    const McScratch sc = carve_mc(vol->mc_scratch, (size_t)nb);
    mc_brick_kernel<true><<<kExtractGrid, kBrickVox, 0, (cudaStream_t)stream>>>(vol->v, vol->voxel_length_d, (const float2 *)d_halo_lo, (const float2 *)d_halo_hi,
                                                                                 d_halo_hi_color, sc, d_vertices, d_keys, d_colors, cap_v, d_tri, cap_t);
    BSLAM_LAUNCH_CHECK();
    return BSLAM_OK;
}

size_t bslam_mesh_merge_workspace_bytes(int n_slabs, int nx, int ny) {
    if (n_slabs <= 0 || nx <= 0 || ny <= 0) return 0;
    return (size_t)n_slabs * (size_t)nx * (size_t)ny * 4 * sizeof(int32_t) + 256;
}

int bslam_mesh_merge(int n_slabs, const int64_t *h_nv, const int64_t *h_nt, const int32_t *h_z_offsets, int nx, int ny, int32_t *d_keys,
                     int32_t *d_tris, void *d_workspace, int64_t *h_unresolved, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(n_slabs >= 1 && n_slabs <= kMaxSlabs && h_nv && h_nt && h_z_offsets && d_workspace, "bslam_mesh_merge: bad argument (1..%d slabs)", kMaxSlabs);
    BSLAM_CHECK_ARG(((uintptr_t)d_keys & 15) == 0, "bslam_mesh_merge: keys must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    MergeP mp;
    memset(&mp, 0, sizeof(mp));
    mp.n = n_slabs;
    long long nv = 0, nt = 0;
    for (int s = 0; s < n_slabs; ++s) {
        nv += h_nv[s]; nt += h_nt[s];
        mp.vend[s] = nv; mp.tend[s] = nt; mp.zoff[s] = h_z_offsets[s];
    }
    BSLAM_CHECK_ARG(nv < (1ll << 31), "bslam_mesh_merge: more than 2^31 vertices");
    const long long stride = (long long)nx * ny * 4;
    unsigned int *d_unres = (unsigned int *)d_workspace;
    int32_t *table = (int32_t *)((char *)d_workspace + 256);
    BSLAM_CUDA(cudaMemsetAsync(d_workspace, 0, 256, st));
    BSLAM_CUDA(cudaMemsetAsync(table, 0xff, (size_t)n_slabs * stride * sizeof(int32_t), st));
    if (nv) merge_vertices_kernel<<<(unsigned)((nv + 255) / 256), 256, 0, st>>>(mp, d_keys, nv, ny, stride, table);
    BSLAM_LAUNCH_CHECK();
    if (nt) merge_triangles_kernel<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(mp, d_tris, nt, stride, table, d_unres);
    BSLAM_LAUNCH_CHECK();
    if (h_unresolved) {
        unsigned int u = 0;
        BSLAM_CUDA(cudaMemcpyAsync(&u, d_unres, 4, cudaMemcpyDeviceToHost, st));
        BSLAM_CUDA(cudaStreamSynchronize(st));
        *h_unresolved = u;
    }
    return BSLAM_OK;
}

int bslam_points_count(bslam_volume *vol, int64_t *h_count, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(vol && h_count, "bslam_points_count: NULL argument");
    BSLAM_CHECK_ARG(vol->v.gz0 == 0 && vol->v.zs == 1, "bslam_points_count: single-box volumes only (gz0 must be 0)");
    BSLAM_DEVICE_GUARD(vol->device);
    int rc = ensure_mc_scratch(vol);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nb = brick_count(vol->v);
    const McScratch sc = carve_mc(vol->mc_scratch, (size_t)nb);
    rc = build_candidates(vol, sc, 0, st);
    if (rc) return rc;
    PtsCache pc = no_cache();
    if (vol->pts_incremental) {
        const size_t need_bytes = pts_cache_bytes((size_t)nb);
        if (!vol->pts_cache || vol->pts_cache_bytes < need_bytes) {
            if (vol->pts_cache) cudaFree(vol->pts_cache);
            vol->pts_cache = nullptr;
            BSLAM_CUDA(cudaMalloc(&vol->pts_cache, need_bytes));
            vol->pts_cache_bytes = need_bytes;
            vol->pts_cache_valid = 0;
        }
        pc = carve_pts(vol->pts_cache, (size_t)nb);
        if (!vol->pts_cache_valid) {    // slots, counts (0xffffffff = none / unknown) and the slot counter start over
            BSLAM_CUDA(cudaMemsetAsync(vol->pts_cache, 0xff, 2 * align_up((size_t)nb * 4, 256), st));
            BSLAM_CUDA(cudaMemsetAsync(pc.used, 0, 4, st));
        }
        const int g = num_sms(vol->device) * 4;
        BSLAM_CUDA(cudaMemsetAsync(sc.totals + 3, 0, 8, st));
        pts_need_kernel<<<g, 256, 0, st>>>(vol->v, sc, pc, vol->pts_cache_valid);
        BSLAM_LAUNCH_CHECK();
        pts_clear_dirty_kernel<<<g, 256, 0, st>>>(vol->v);
        BSLAM_LAUNCH_CHECK();
        vol->pts_cache_valid = 0;      // until the emit pass has refreshed the recomputed bricks' slots
        vol->pts_counted = 1;
    }
    points_brick_kernel<false><<<kExtractGrid, kBrickVox, 0, st>>>(vol->v, vol->voxel_length_d, sc, nullptr, nullptr, nullptr, nullptr, 0, pc);
    BSLAM_LAUNCH_CHECK();
    rc = brick_scan(sc.nvert, nullptr, sc.vbase, nullptr, nb, sc.totals, sc.scan_ws, st);
    if (rc) return rc;
    unsigned long long tot[4];
    BSLAM_CUDA(cudaMemcpyAsync(tot, sc.totals, 32, cudaMemcpyDeviceToHost, st));
    BSLAM_CUDA(cudaStreamSynchronize(st));
    *h_count = (int64_t)tot[0];
    vol->pts_last_total = (long long)tot[0];
    vol->pts_last_candidates = (long long)tot[2];
    vol->pts_last_recomputed = vol->pts_incremental ? (long long)tot[3] : (long long)tot[2];
    return BSLAM_OK;
}

int bslam_points_emit(bslam_volume *vol, float *d_points, float *d_normals, float *d_colors, int32_t *d_keys, int64_t cap, bslam_stream_t stream) {
    BSLAM_CHECK_ARG(vol && vol->mc_scratch, "bslam_points_emit: call bslam_points_count first");
    BSLAM_CHECK_ARG(d_points || cap == 0, "bslam_points_emit: NULL output");
    BSLAM_DEVICE_GUARD(vol->device);
    const int64_t nb = brick_count(vol->v);
    const McScratch sc = carve_mc(vol->mc_scratch, (size_t)nb);
    PtsCache pc = no_cache();
    if (vol->pts_incremental) {
        BSLAM_CHECK_ARG(vol->pts_cache && vol->pts_counted, "bslam_points_emit: incremental mode needs bslam_points_count before every emit");
        BSLAM_CHECK_ARG(cap >= vol->pts_last_total, "bslam_points_emit: incremental mode needs room for all %lld points", vol->pts_last_total);
        BSLAM_CHECK_ARG((d_normals != nullptr) == (vol->pts_with_normals != 0), "bslam_points_emit: incremental extraction was enabled %s normals",
                        vol->pts_with_normals ? "with" : "without");
        BSLAM_CHECK_ARG(!(vol->v.color && !d_colors), "bslam_points_emit: incremental extraction of a colour volume needs the colour output");
        pc = carve_pts(vol->pts_cache, (size_t)nb);
    }
    points_brick_kernel<true><<<kExtractGrid, kBrickVox, 0, (cudaStream_t)stream>>>(vol->v, vol->voxel_length_d, sc, d_points, d_normals, d_colors,
                                                                                     d_keys, cap, pc);
    BSLAM_LAUNCH_CHECK();
    if (vol->pts_incremental) { vol->pts_cache_valid = 1; vol->pts_counted = 0; }
    return BSLAM_OK;
}

} // extern "C"
