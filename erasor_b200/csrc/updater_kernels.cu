// updater_kernels.cu -- device versions of the caller-side steps either side of the R-POD -> SRT -> R-GPF path
// (SURVEY.md section 8f, rows 1-3), so that the map never leaves HBM between frames:
//
//   U1  stable partition of the map by a per-point predicate, with the float affine of pcl::transformPointCloud
//       fused into the copy of the selected side:
//         * OfflineMapUpdater::fetch_VoI  ("naive" mode)          reference OfflineMapUpdater.cpp:381-438
//         * OfflineMapUpdater::set_submap (large-scale window)    reference OfflineMapUpdater.cpp:360-379
//   U2  affine copy (body2origin, lidar2body: pcl::transformPointCloud)             :240, :286-288, :441-449
//   U3  erasor_utils::voxelize_preserving_labels for clouds of any size             erasor_utils.cpp:80-114
//       (pcl::VoxelGrid keys -> stable global radix sort -> centroids -> exact 1-NN label restore);
//       used on the query scan (:238) and by save_static_map (:186)
//
// Arithmetic is spelled with round-to-nearest intrinsics (no FMA contraction), exactly as restated in oracle/.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cstdint>

#include "updater_kernels.h"

namespace erasor {

#define FULL_MASK 0xFFFFFFFFu
#define FM(a, b) __fmul_rn((a), (b))
#define FA(a, b) __fadd_rn((a), (b))
#define FS(a, b) __fsub_rn((a), (b))
#define FD(a, b) __fdiv_rn((a), (b))

// pcl::transformPointCloud, PCL 1.8 scalar path: ((m0*x + m1*y) + m2*z) + m3, float, no contraction
__device__ __forceinline__ float4 affine(const Mat4& T, float4 p) {
    float4 o;
    o.x = FA(FA(FA(FM(T.m[0], p.x), FM(T.m[1], p.y)), FM(T.m[2], p.z)), T.m[3]);
    o.y = FA(FA(FA(FM(T.m[4], p.x), FM(T.m[5], p.y)), FM(T.m[6], p.z)), T.m[7]);
    o.z = FA(FA(FA(FM(T.m[8], p.x), FM(T.m[9], p.y)), FM(T.m[10], p.z)), T.m[11]);
    o.w = p.w;
    return o;
}

__device__ __forceinline__ bool part_pred(const PartPred& P, float4 p) {
    if (P.kind == PART_RADIUS) {
        // double dist_square = pow(pt.x - x_criterion, 2) + pow(pt.y - y_criterion, 2); dist_square < max_dist_square
        const double dx = __dsub_rn((double)p.x, P.x), dy = __dsub_rn((double)p.y, P.y);
        const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        return d2 < P.limit;
    }
    if (P.kind == PART_NOT_NEAR) {
        // mapgen's vehicle-body cut (src/mapgen/mapgen.hpp:218-229): dist_square = pow(pt.x, 2) + pow(pt.y, 2) in double;
        // points with dist_square < max_dist_square are dropped, everything else (NaN included) is kept
        const double xd = (double)p.x, yd = (double)p.y;
        const double d2 = __dadd_rn(__dmul_rn(xd, xd), __dmul_rn(yd, yd));
        return !(d2 < P.limit);
    }
    // set_submap: fabs(x - pt.x) < submap_size && fabs(y - pt.y) < submap_size
    const double dx = fabs(__dsub_rn(P.x, (double)p.x)), dy = fabs(__dsub_rn(P.y, (double)p.y));
    return (dx < P.limit) && (dy < P.limit);
}

constexpr int PART_CHUNK = 4096;          // points per partition / head-count chunk (one virtual block)

__global__ void k_affine_copy(Mat4 T, int do_transform, const float4* in, float4* out, uint32_t n) {   // in may alias out
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = do_transform ? affine(T, in[i]) : in[i];
}
__global__ void __launch_bounds__(256) k_copy_segments(Mat4 T, CopySeg s0, CopySeg s1, CopySeg s2, CopySeg s3) {
    const CopySeg segs[4] = {s0, s1, s2, s3};
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t blocks = (segs[k].n + 255u) / 256u * 256u;     // segments start on block boundaries: no divergence inside a warp
        if (i < blocks) {
            if (i < segs[k].n) { const float4 p = segs[k].src[i]; segs[k].dst[i] = segs[k].xform ? affine(T, p) : p; }
            return;
        }
        i -= blocks;
    }
}
cudaError_t launch_copy_segments(cudaStream_t st, const Mat4& T, const CopySeg* segs, int n_segs) {
    CopySeg s[4] = {{nullptr, nullptr, 0u, 0}, {nullptr, nullptr, 0u, 0}, {nullptr, nullptr, 0u, 0}, {nullptr, nullptr, 0u, 0}};
    uint32_t blocks = 0;
    for (int k = 0; k < n_segs && k < 4; ++k) { s[k] = segs[k]; blocks += (segs[k].n + 255u) / 256u; }
    if (blocks == 0) return cudaSuccess;
    k_copy_segments<<<blocks, 256, 0, st>>>(T, s[0], s[1], s[2], s[3]);
    return cudaGetLastError();
}
cudaError_t launch_affine_copy(cudaStream_t st, const Mat4& T, bool do_transform, const float4* in, float4* out, uint32_t n) {
    if (n == 0) return cudaSuccess;
    k_affine_copy<<<(n + 255) / 256, 256, 0, st>>>(T, do_transform ? 1 : 0, in, out, n);
    return cudaGetLastError();
}

// ============================================================================================
// U3  voxelize_preserving_labels
// ============================================================================================
__device__ __forceinline__ uint32_t f2ord(float f) { const uint32_t u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float ord2f(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o); }

// Radix-sort segment = the run of points one warp ranks (stably, match.any) in a pass.  The walk is a serial chain of rows, so
// segments are as short as the counter matrices allow: 8 rows of 32 up to 2 M points, longer beyond (<= 8192 segments).
constexpr uint32_t RS_ROWS_MIN = 8, RS_MAX_SEGS = 8192;
constexpr int      RB = 9;                  // radix digit: 9 bits -- a LiDAR scan's 27-bit voxel keys sort in three passes
constexpr uint32_t RD = 1u << RB;
__host__ __device__ inline uint32_t rs_seg_len(uint32_t n) {
    uint32_t rows = (uint32_t)(((unsigned long long)n + 32ull * RS_MAX_SEGS - 1ull) / (32ull * RS_MAX_SEGS));
    rows = (rows + RS_ROWS_MIN - 1u) / RS_ROWS_MIN * RS_ROWS_MIN;
    return 32u * (rows < RS_ROWS_MIN ? RS_ROWS_MIN : rows);
}

// pcl::CentroidPoint: float sums over the voxel's members in cloud order, divided by float(count)
__device__ __forceinline__ float4 vox_centroid_of(const float4* __restrict__ in, const uint32_t* __restrict__ sidx, const uint32_t* __restrict__ vox_start, uint32_t v) {
    const uint32_t a = vox_start[v], e = vox_start[v + 1];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    for (uint32_t k = a; k < e; ++k) {
        const float4 p = in[sidx[k]];
        sx = FA(sx, p.x); sy = FA(sy, p.y); sz = FA(sz, p.z); si = FA(si, p.w);
    }
    const float cn = (float)(e - a);
    return make_float4(FD(sx, cn), FD(sy, cn), FD(sz, cn), FD(si, cn));
}

// Conservative distance along one axis from coordinate x to the voxel cell with (absolute) index `cell`, which lies `off` cells
// away from x's own cell (off < 0: below, > 0: above, 0: the same slab).  A point is assigned to `cell` when
// floorf(x * (1 / leaf)) == cell in float arithmetic, so the cell's faces sit within a few ulp of cell * leaf and (cell + 1) * leaf;
// `slack` covers that and the rounding of this expression, so the returned gap never exceeds the true one.
__device__ __forceinline__ float cell_gap(float x, int cell, int off, float leaf, float slack) {
    if (off == 0) return 0.0f;
    const float g = (off > 0) ? ((float)cell * leaf - x) : (x - (float)(cell + 1) * leaf);
    return fmaxf(g - slack, 0.0f);
}

// exact 1-NN of a centroid into the source cloud through the voxel grid itself (cells = voxels): grow the Chebyshev shell
// until nothing unseen can be closer; ties go to the lowest cloud index.  Mirrors oracle/ line by line.
__device__ __noinline__ float4 vox_label_of(const float4* __restrict__ in, const uint32_t* __restrict__ sidx, const uint32_t* __restrict__ vox_start,
                                            const uint32_t* __restrict__ vox_key, const VoxGrid* __restrict__ g, uint32_t nv, float4 c) {
    if (g->overflow) return c;         // every point is its own voxel: the nearest point is itself (or an identical earlier one)
    const float inv = g->inv, leaf = g->leaf;
    const int d0 = g->div[0], d1 = g->div[1], d2 = g->div[2];
    const int ci = (int)FS(floorf(FM(c.x, inv)), (float)g->min_b[0]);
    const int cj = (int)FS(floorf(FM(c.y, inv)), (float)g->min_b[1]);
    const int ck = (int)FS(floorf(FM(c.z, inv)), (float)g->min_b[2]);
    float best_d = __int_as_float(0x7f800000);
    uint32_t best_i = 0xFFFFFFFFu;
    const float slack = 1.0e-3f * leaf + 4.0e-6f * fmaxf(fabsf(c.x), fmaxf(fabsf(c.y), fabsf(c.z)));
    int rad = 0;
    while (true) {
        // scan the shell of Chebyshev radius `rad`
        for (int a = -rad; a <= rad; ++a) {
            const int ii = ci + a;
            if (ii < 0 || ii >= d0) continue;
            for (int b = -rad; b <= rad; ++b) {
                const int jj = cj + b;
                if (jj < 0 || jj >= d1) continue;
                for (int cc = -rad; cc <= rad; ++cc) {
                    if (max(abs(a), max(abs(b), abs(cc))) != rad) continue;
                    const int kk = ck + cc;
                    if (kk < 0 || kk >= d2) continue;
                    // Skip the cell when even its nearest corner is provably farther than the best so far (strictly: no tie can hide
                    // there).  The gaps are shortened by more than the float error of the cell assignment, so this only drops work.
                    if (rad > 0) {
                        const float gx = cell_gap(c.x, ci + a + g->min_b[0], a, leaf, slack);
                        const float gy = cell_gap(c.y, cj + b + g->min_b[1], b, leaf, slack);
                        const float gz = cell_gap(c.z, ck + cc + g->min_b[2], cc, leaf, slack);
                        if (0.999f * (gx * gx + gy * gy + gz * gz) > best_d) continue;
                    }
                    const uint32_t key = (uint32_t)(ii + jj * d0 + kk * d0 * d1);
                    uint32_t lo = 0, hi = nv;                 // first voxel with vox_key >= key
                    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (vox_key[mid] < key) lo = mid + 1; else hi = mid; }
                    if (lo >= nv || vox_key[lo] != key) continue;
                    for (uint32_t k = vox_start[lo]; k < vox_start[lo + 1]; ++k) {
                        const uint32_t i = sidx[k];
                        const float4 p = in[i];
                        const float dx = FS(c.x, p.x), dy = FS(c.y, p.y), dz = FS(c.z, p.z);
                        const float d = FA(FA(FM(dx, dx), FM(dy, dy)), FM(dz, dz));
                        if (d < best_d || (d == best_d && i < best_i)) { best_d = d; best_i = i; }
                    }
                }
            }
        }
        const float reach = FM(FM((float)rad, leaf), 0.9999f);
        if (best_i != 0xFFFFFFFFu && best_d < FM(reach, reach)) break;
        ++rad;
        if (rad > 64 && best_i != 0xFFFFFFFFu) break;
        if (rad > 4096) break;
    }
    if (best_i != 0xFFFFFFFFu) c.w = in[best_i].w;
    return c;
}

// ============================================================================================
// Fused form: one cooperative launch per node (grid-wide barriers between the phases above)
// ============================================================================================
// The per-node prologue of OfflineMapUpdater::callback_node is 25 small dependent kernels in the stepwise form (U3: 22,
// U1: 3) and is bound by launch latency, not by work.  k_node_fused runs the same phases -- same arithmetic, same
// order, bit-identical results -- as ONE cooperative kernel: every phase is a loop over the virtual blocks of the stepwise
// kernel, phases are separated by grid.sync().  The fetch_VoI partition of the map (U1) is independent of the scan's
// voxelisation (U3), so its three phases ride in U3's first three.  The radix sort runs only the passes the key width
// needs (the stepwise form always runs four).
namespace cg = cooperative_groups;
constexpr int FT = 1024;                 // threads per CTA
constexpr int FW = FT / 32;

// exclusive scan of v[0..n) in place by one CTA of FT threads; *total (nullable) receives the sum
__device__ void cta_scan_u32(uint32_t* __restrict__ v, uint32_t n, uint32_t* __restrict__ total, uint32_t* s_part /*[34]*/) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t seg = (n + FT - 1u) / FT;
    const uint32_t b0 = min(n, tid * seg), b1 = min(n, b0 + seg);
    uint32_t sum = 0;
    for (uint32_t i = b0; i < b1; ++i) sum += v[i];
    uint32_t incl = sum;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += t; }
    __syncthreads();
    if (lane == 31) s_part[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = s_part[lane];
        uint32_t wi = w;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(FULL_MASK, wi, o); if (lane >= o) wi += t; }
        s_part[lane] = wi - w;
        if (lane == 31) s_part[33] = wi;
    }
    __syncthreads();
    uint32_t run = s_part[warp] + incl - sum;
    for (uint32_t i = b0; i < b1; ++i) { const uint32_t t = v[i]; v[i] = run; run += t; }
    if (tid == 0 && total) *total = s_part[33];
    __syncthreads();
}

// rank of the flagged threads of one FT-wide row in thread order: `before` = flagged threads in front of this one, `round` = all
__device__ __forceinline__ void cta_rank(bool flag, uint32_t* s_w /*[FW]*/, uint32_t& before, uint32_t& round) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned bal = __ballot_sync(FULL_MASK, flag);
    if (lane == 0) s_w[warp] = __popc(bal);
    __syncthreads();
    uint32_t b = 0, r = 0;
#pragma unroll
    for (int w = 0; w < FW; ++w) { const uint32_t c = s_w[w]; b += (w < warp) ? c : 0u; r += c; }
    before = b + __popc(bal & ((1u << lane) - 1u));
    round = r;
    __syncthreads();
}
__device__ __forceinline__ uint32_t cta_sum(uint32_t c, uint32_t* s_w /*[FW]*/) {
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL_MASK, c, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
    __syncthreads();
    uint32_t t = 0;
#pragma unroll
    for (int w = 0; w < FW; ++w) t += s_w[w];
    __syncthreads();
    return t;
}

// batched U3: the cloud that point (or sorted position) e belongs to = the first f with off[f + 1] > e (empty clouds are skipped)
__device__ __forceinline__ uint32_t cloud_of(const uint32_t* __restrict__ off, uint32_t F, uint32_t e) {
    uint32_t lo = 0, hi = F;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (off[mid + 1] <= e) lo = mid + 1; else hi = mid; }
    return lo;
}
// first index in a[0..n) with a[i] >= x (a ascending)
__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t* __restrict__ a, uint32_t n, uint32_t x) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (a[mid] < x) lo = mid + 1; else hi = mid; }
    return lo;
}

// getMinMax3D of in[b0..b1) by the whole grid: this CTA's partial (order-preserving encodings, min x y z then max x y z) to out6
__device__ __forceinline__ void cta_minmax(const float4* __restrict__ in, uint32_t b0, uint32_t b1, uint32_t* s_c, uint32_t* out6) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t mn[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, mx[3] = {0u, 0u, 0u};
    for (uint32_t i = b0 + blockIdx.x * FT + tid; i < b1; i += gridDim.x * FT) {
        const float4 p = in[i];
        const uint32_t a = f2ord(p.x + 0.0f), b = f2ord(p.y + 0.0f), c = f2ord(p.z + 0.0f);
        mn[0] = min(mn[0], a); mx[0] = max(mx[0], a);
        mn[1] = min(mn[1], b); mx[1] = max(mx[1], b);
        mn[2] = min(mn[2], c); mx[2] = max(mx[2], c);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const uint32_t a = __reduce_min_sync(FULL_MASK, mn[k]), b = __reduce_max_sync(FULL_MASK, mx[k]);
        if (lane == 0) { s_c[warp * 6 + k] = a; s_c[warp * 6 + 3 + k] = b; }
    }
    __syncthreads();
    if (tid < 6) {
        uint32_t r = (tid < 3) ? 0xFFFFFFFFu : 0u;
        for (int w = 0; w < FW; ++w) r = (tid < 3) ? min(r, s_c[w * 6 + tid]) : max(r, s_c[w * 6 + tid]);
        out6[tid] = r;
    }
    __syncthreads();
}

// pcl::VoxelGrid set-up of one cloud of n points from its min / max (s_w[0..6), order-preserving encodings); one thread
__device__ void vox_grid_setup(VoxGrid* g, float leaf, uint32_t n, const uint32_t* s_w) {
    g->n_vox = 0; g->overflow = 0; g->npass = 0;
    const float inv = FD(1.0f, leaf);
    g->leaf = leaf; g->inv = inv;
    if (n == 0) {
        for (int k = 0; k < 3; ++k) { g->mn[k] = 0xFFFFFFFFu; g->mx[k] = 0u; g->div[k] = 1; g->min_b[k] = 0; }
        return;
    }
    float mnf[3], mxf[3];
    for (int k = 0; k < 3; ++k) {
        g->mn[k] = s_w[k]; g->mx[k] = s_w[3 + k];
        mnf[k] = ord2f(s_w[k]); mxf[k] = ord2f(s_w[3 + k]);
    }
    const long long dx = (long long)FM(FS(mxf[0], mnf[0]), inv) + 1;
    const long long dy = (long long)FM(FS(mxf[1], mnf[1]), inv) + 1;
    const long long dz = (long long)FM(FS(mxf[2], mnf[2]), inv) + 1;
    const int ovf = (dx * dy * dz) > 2147483647LL ? 1 : 0;
    g->overflow = ovf;
    unsigned long long cells = 1ull;
    for (int k = 0; k < 3; ++k) {
        g->min_b[k] = (int)floorf(FM(mnf[k], inv));
        const int max_b = (int)floorf(FM(mxf[k], inv));
        g->div[k] = max_b - g->min_b[k] + 1;
        cells *= (unsigned long long)(unsigned)g->div[k];
    }
    // radix passes the keys need: keys are < cells (int32 arithmetic as in PCL), or < n in the overflow case
    unsigned long long lim = ovf ? (unsigned long long)n : cells;
    int bits = 32;
    if (lim <= 0x80000000ull) { bits = 1; while ((1ull << bits) < lim) ++bits; }
    g->npass = (bits + RB - 1) / RB;
}

// pcl::VoxelGrid key of point p (local: its index within its cloud, the key of the overflow case)
__device__ __forceinline__ uint32_t vox_key(int ovf, float inv, float mb0, float mb1, float mb2, int d0, int d01, float4 p, uint32_t local) {
    if (ovf) return local;      // "Leaf size is too small": output = input, one point per voxel in cloud order
    const int ijk0 = (int)FS(floorf(FM(p.x, inv)), mb0);
    const int ijk1 = (int)FS(floorf(FM(p.y, inv)), mb1);
    const int ijk2 = (int)FS(floorf(FM(p.z, inv)), mb2);
    return (uint32_t)(ijk0 + ijk1 * d0 + ijk2 * d01);
}

struct VoxPlan {                          // carve-up of the voxeliser's scratch (host and device agree through this one function)
    uint32_t *key_a, *idx_a, *key_b, *idx_b, *cnt_x, *cnt_y, *tot, *chunk, *vstart, *vkey, *partial, *cvox;
    uint32_t seg, nseg;
};
__host__ __device__ inline VoxPlan vox_plan(void* tmp, uint32_t n, uint32_t n_clouds = 1) {
    VoxPlan p;
    uint32_t* w = reinterpret_cast<uint32_t*>(tmp);
    p.seg  = rs_seg_len(n);
    p.nseg = (n + p.seg - 1) / p.seg;
    p.key_a = w;            p.idx_a = p.key_a + n;
    p.key_b = p.idx_a + n;  p.idx_b = p.key_b + n;
    p.cnt_x = p.idx_b + n;                                            // [RD][nseg] digit histogram per segment (even passes)
    p.cnt_y = p.cnt_x + (size_t)RD * (p.nseg + 1);                    // ... (odd passes)
    p.tot   = p.cnt_y + (size_t)RD * (p.nseg + 1);                    // [RD] points per digit
    p.chunk = p.tot + RD;                                            // (n + PART_CHUNK - 1) / PART_CHUNK + 1
    p.vstart = p.chunk + ((size_t)(n + PART_CHUNK - 1) / PART_CHUNK + 1);   // n + 2
    p.vkey   = p.vstart + ((size_t)n + 2);                            // n + 2
    p.partial = p.vkey + ((size_t)n + 2);                             // 6 * kFusedMaxGrid per cloud
    p.cvox    = p.partial + (size_t)6 * kFusedMaxGrid * n_clouds;     // batched: first voxel of every non-empty cloud
    return p;
}

// BATCH = false: one cloud (FusedJob.vin[0..vn)) plus the optional U1 partition -- the sequential updater's form.
// BATCH = true:  FusedJob.n_clouds clouds in one launch.  The phases are the same; per cloud they keep their own min / max,
// grid and key, and after the key passes the stable radix sort runs the cloud id as its most significant digit(s), so
// every cloud's points end up contiguous, in ascending key, members in cloud order -- what one call per cloud gives.
template <bool BATCH>
__global__ void __launch_bounds__(FT, 1) k_node_fused(FusedJob J) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ uint32_t s_c[];        // [FW][RD] next free destination per digit, one row per warp (also the min/max staging)
    __shared__ uint32_t s_w[FW];
    __shared__ uint32_t s_part[34];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t G = gridDim.x, bid = blockIdx.x;
    const uint32_t n = J.vn, pn = J.pn;
    const uint32_t NC = BATCH ? J.n_clouds : 1u;
    const uint32_t* __restrict__ coff = J.cloud_off;
    const bool has_part = !BATCH && J.has_part;
    const VoxPlan vp = vox_plan(J.vtmp, n, NC);
    const uint32_t nseg = vp.nseg, SEG = vp.seg;
    VoxGrid* g = J.grid;
    const uint32_t pchunks = (pn + PART_CHUNK - 1) / PART_CHUNK;
    // phase profile of CTA 0 (nanoseconds, %globaltimer): read back by erasor_updater_get_fused_profile
#define PH(slot) do { if (bid == 0 && tid == 0) { unsigned long long t__; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t__)); g->prof[slot] = t__; } } while (0)
    PH(0);

    // ---- phase 0: getMinMax3D partials per CTA | partition: selected points per chunk ----
    if (n) {
        for (uint32_t i = bid * FT + tid; i < 2u * RD * (nseg + 1u); i += G * FT) vp.cnt_x[i] = 0u;      // both histogram matrices (contiguous)
        if (!BATCH) {
            cta_minmax(J.vin, 0u, n, s_c, vp.partial + bid * 6);
        } else {
            for (uint32_t f = 0; f < NC; ++f) {                                                  // per cloud: partial [f][bid][6]
                const uint32_t o0 = coff[f], o1 = coff[f + 1];
                if (o0 < o1) cta_minmax(J.vin, o0, o1, s_c, vp.partial + ((size_t)f * G + bid) * 6);
            }
        }
    }
    if (BATCH) {
        for (uint32_t f = bid * FT + tid; f < NC; f += G * FT) J.cloud_nvox[f] = 0u;
    }
    if (has_part) {
        for (uint32_t vb = bid; vb < pchunks; vb += G) {
            const uint32_t b0 = vb * PART_CHUNK, b1 = min(pn, b0 + PART_CHUNK);
            uint32_t c = 0;
            for (uint32_t i = b0 + tid; i < b1; i += FT) c += part_pred(J.P, J.pin[i]) ? 1u : 0u;
            const uint32_t t = cta_sum(c, s_w);
            if (tid == 0) J.chunk_tmp[vb] = t;
        }
    }
    grid.sync();
    PH(1);

    // ---- phase 1: VoxelGrid set-up (CTA 0) | partition: chunk offsets (last CTA) ----
    for (uint32_t f = bid; f < NC; f += G) {      // (one cloud: CTA 0)
        const uint32_t nf = BATCH ? coff[f + 1] - coff[f] : n;
        if (nf && warp < 6) {                   // reduce the per-CTA partials: warp k < 3 the minimum of axis k, warps 3..5 the maxima
            const uint32_t* part = vp.partial + (size_t)f * G * 6;
            uint32_t r = (warp < 3) ? 0xFFFFFFFFu : 0u;
            for (uint32_t c = lane; c < G; c += 32) r = (warp < 3) ? min(r, part[c * 6 + warp]) : max(r, part[c * 6 + warp]);
            r = (warp < 3) ? __reduce_min_sync(FULL_MASK, r) : __reduce_max_sync(FULL_MASK, r);
            if (lane == 0) s_w[warp] = r;
        }
        __syncthreads();
        if (tid == 0) {
            vox_grid_setup(g + f, J.leaf, nf, s_w);
            if (n == 0 && f == 0) *J.d_n_out = 0u;
        }
        __syncthreads();
    }
    if (has_part && bid == G - 1) cta_scan_u32(J.chunk_tmp, pchunks, J.d_total_sel, s_part);
    grid.sync();
    PH(2);

    // ---- phase 2: voxel keys + digit-0 histogram, one warp per 1024-point segment | partition: stable scatter ----
    // batched: the key passes every cloud needs, then the cloud id's digits
    int npk = 0, npass = 0;
    if (!BATCH) {
        npass = n ? g->npass : 0;
        npk = npass;
    } else if (n) {
        for (uint32_t f = lane; f < NC; f += 32) npk = max(npk, g[f].npass);
        npk = __reduce_max_sync(FULL_MASK, npk);
        const int cbits = NC > 1 ? 32 - __clz(NC - 1) : 0;
        npass = npk + (cbits + RB - 1) / RB;
    }
    uint32_t* const my_c = s_c + warp * RD;
    if (n && !BATCH) {
        const int ovf = g->overflow;
        const float inv = g->inv;
        const float mb0 = (float)g->min_b[0], mb1 = (float)g->min_b[1], mb2 = (float)g->min_b[2];
        const int d0 = g->div[0], d01 = g->div[0] * g->div[1];
        for (uint32_t e = bid * FT + tid; e < n; e += G * FT) {
            const uint32_t k = vox_key(ovf, inv, mb0, mb1, mb2, d0, d01, J.vin[e], e);
            vp.key_a[e] = k; vp.idx_a[e] = e;
            atomicAdd(&vp.cnt_x[(size_t)(k & (RD - 1u)) * nseg + e / SEG], 1u);      // pass 0's histogram (counts: order-free)
        }
    } else if (n) {
        for (uint32_t e = bid * FT + tid; e < n; e += G * FT) {
            const uint32_t f = cloud_of(coff, NC, e);
            const VoxGrid* gf = g + f;
            const uint32_t k = vox_key(gf->overflow, gf->inv, (float)gf->min_b[0], (float)gf->min_b[1], (float)gf->min_b[2], gf->div[0],
                                       gf->div[0] * gf->div[1], J.vin[e], e - coff[f]);
            vp.key_a[e] = k; vp.idx_a[e] = e;
            atomicAdd(&vp.cnt_x[(size_t)(k & (RD - 1u)) * nseg + e / SEG], 1u);
        }
    }
    if (has_part) {
        for (uint32_t vb = bid; vb < pchunks; vb += G) {
            const uint32_t b0 = vb * PART_CHUNK, b1 = min(pn, b0 + PART_CHUNK);
            uint32_t sel_base = J.chunk_tmp[vb];
            uint32_t rest_base = b0 - sel_base;
            for (uint32_t r0 = b0; r0 < b1; r0 += FT) {
                const uint32_t i = r0 + tid;
                const bool ok = i < b1;
                const float4 p = ok ? J.pin[i] : make_float4(0.f, 0.f, 0.f, 0.f);
                const bool s = ok && part_pred(J.P, p);
                uint32_t rank_sel, round;
                cta_rank(s, s_w, rank_sel, round);
                if (ok) {
                    if (s) J.out_sel[sel_base + rank_sel] = J.xform_sel ? affine(J.T_sel, p) : p;
                    else   J.out_rest[rest_base + (i - r0) - rank_sel] = p;
                }
                const uint32_t valid = min((uint32_t)FT, b1 - r0);
                sel_base += round;
                rest_base += valid - round;
            }
        }
    }
    grid.sync();
    PH(3);

    // ---- stable LSD radix sort of (key, cloud index), 9-bit digits, only the passes the key width needs.  Per pass:
    //   (a) one warp per digit scans its row of per-segment counts in place (exclusive) and leaves the digit's total;
    //   (b) one warp per segment ranks its points stably (match.any) behind base[digit] + row prefix and scatters them;
    //       on the way it counts the NEXT pass's digits per destination segment with RED (counts are order-free),
    //       so there is no separate histogram phase.
    for (int pass = 0; pass < npass; ++pass) {
        const uint32_t* ki = (pass & 1) ? vp.key_b : vp.key_a;  const uint32_t* ii = (pass & 1) ? vp.idx_b : vp.idx_a;
        uint32_t* ko = (pass & 1) ? vp.key_a : vp.key_b;        uint32_t* io = (pass & 1) ? vp.idx_a : vp.idx_b;
        uint32_t* cnt  = (pass & 1) ? vp.cnt_y : vp.cnt_x;     // this pass's histogram
        uint32_t* cntn = (pass & 1) ? vp.cnt_x : vp.cnt_y;     // the next pass's (zero on entry to (b))
        const int shift = pass * RB;
        const bool more = pass + 1 < npass;
        // (a)
        if (pass > 0 && more) for (uint32_t i = bid * FT + tid; i < RD * nseg; i += G * FT) cntn[i] = 0u;      // consumed two phases ago
        for (uint32_t d = (uint32_t)warp * G + bid; d < RD; d += G * FW) {
            uint32_t* row = cnt + (size_t)d * nseg;
            uint32_t carry = 0u;
            for (uint32_t c0 = 0; c0 < nseg; c0 += 512u) {              // 16 consecutive counters per lane and round, loaded together
                const uint32_t a = c0 + (uint32_t)lane * 16u;
                uint32_t v[16], sum = 0u;
#pragma unroll
                for (int j = 0; j < 16; ++j) { v[j] = (a + j < nseg) ? row[a + j] : 0u; }
#pragma unroll
                for (int j = 0; j < 16; ++j) { const uint32_t t = v[j]; v[j] = sum; sum += t; }
                uint32_t incl = sum;
                for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += t; }
                const uint32_t base = carry + incl - sum;
#pragma unroll
                for (int j = 0; j < 16; ++j) { if (a + j < nseg) row[a + j] = base + v[j]; }
                carry += __shfl_sync(FULL_MASK, incl, 31);
            }
            if (lane == 0) vp.tot[d] = carry;
        }
        grid.sync();
        PH(4 + 2 * pass);
        // (b)
        for (uint32_t seg = (uint32_t)warp * G + bid; seg < nseg; seg += G * FW) {     // consecutive segments on different SMs (match.any is a per-SM unit)
            const uint32_t b0 = seg * SEG, b1 = min(n, b0 + SEG);
            {   // next free destination per digit: points of smaller digits + points of this digit in earlier segments
                constexpr int DL = RD / 32;            // digits per lane
                uint32_t t[DL], c[DL], sum = 0u;
#pragma unroll
                for (int j = 0; j < DL; ++j) { t[j] = vp.tot[lane * DL + j]; }
#pragma unroll
                for (int j = 0; j < DL; ++j) { c[j] = cnt[(size_t)(lane * DL + j) * nseg + seg]; }
#pragma unroll
                for (int j = 0; j < DL; ++j) { const uint32_t x = t[j]; t[j] = sum; sum += x; }
                uint32_t incl = sum;
                for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += x; }
#pragma unroll
                for (int j = 0; j < DL; ++j) my_c[lane * DL + j] = incl - sum + t[j] + c[j];
            }
            __syncwarp();
            for (uint32_t r0 = b0; r0 < b1; r0 += 32u * RS_ROWS_MIN) {       // blocks of 8 rows: keys and indices loaded together, then ranked row by row
                uint32_t kk[RS_ROWS_MIN], vv[RS_ROWS_MIN];
#pragma unroll
                for (int r = 0; r < (int)RS_ROWS_MIN; ++r) {
                    const uint32_t e = r0 + (uint32_t)r * 32u + lane;
                    kk[r] = (e < b1) ? ki[e] : 0u; vv[r] = (e < b1) ? ii[e] : 0u;
                }
#pragma unroll
                for (int r = 0; r < (int)RS_ROWS_MIN; ++r) {
                    const uint32_t e = r0 + (uint32_t)r * 32u + lane;
                    const bool valid = e < b1;
                    const unsigned vm = __ballot_sync(FULL_MASK, valid);
                    unsigned my_peers = 0u;
                    uint32_t dst_o = 0u;
                    if (valid) {
                        const uint32_t d = (!BATCH || pass < npk) ? (kk[r] >> shift) & (RD - 1u)
                                                                  : (cloud_of(coff, NC, vv[r]) >> ((pass - npk) * RB)) & (RD - 1u);
                        const unsigned peers = __match_any_sync(vm, d);
                        const uint32_t base = my_c[d];
                        __syncwarp(vm);
                        if (lane == __ffs(peers) - 1) my_c[d] = base + __popc(peers);
                        const uint32_t o = base + __popc(peers & ((1u << lane) - 1u));
                        ko[o] = kk[r]; io[o] = vv[r];
                        my_peers = peers; dst_o = o;
                    }
                    if (more) {
                        // next pass's histogram: one RED per run of equal digits when the whole run lands in one counter (the usual
                        // case -- neighbouring voxels share their upper key bits), else one per point
                        uint32_t nd = 0u;
                        if (valid) nd = (!BATCH || pass + 1 < npk) ? (kk[r] >> (shift + RB)) & (RD - 1u)
                                                                   : (cloud_of(coff, NC, vv[r]) >> ((pass + 1 - npk) * RB)) & (RD - 1u);
                        const uint32_t slot = valid ? nd * nseg + dst_o / SEG : 0xFFFFFFFFu;
                        const int      lead = valid ? __ffs(my_peers) - 1 : lane;
                        const uint32_t lslot = __shfl_sync(FULL_MASK, slot, lead);
                        const unsigned differ = __ballot_sync(FULL_MASK, valid && slot != lslot);
                        if (valid) {
                            if ((my_peers & differ) == 0u) { if (lane == lead) atomicAdd(&cntn[slot], (uint32_t)__popc(my_peers)); }
                            else atomicAdd(&cntn[slot], 1u);
                        }
                    }
                    __syncwarp();
                }
            }
            __syncwarp();
        }
        grid.sync();
        PH(4 + 2 * pass + 1);
    }
    PH(12);
    if (n == 0) return;                                   // (grid-uniform)
    const uint32_t* skey = (npass & 1) ? vp.key_b : vp.key_a;
    const uint32_t* sidx = (npass & 1) ? vp.idx_b : vp.idx_a;

    // ---- heads of equal-key runs: count per chunk, offsets, ordered scatter ----
    const uint32_t hchunks = (n + PART_CHUNK - 1) / PART_CHUNK;
    for (uint32_t vb = bid; vb < hchunks; vb += G) {
        const uint32_t b0 = vb * PART_CHUNK, b1 = min(n, b0 + PART_CHUNK);
        uint32_t c = 0;
        for (uint32_t i = b0 + tid; i < b1; i += FT)
            c += (i == 0 || skey[i] != skey[i - 1] || (BATCH && cloud_of(coff, NC, i) != cloud_of(coff, NC, i - 1))) ? 1u : 0u;
        const uint32_t t = cta_sum(c, s_w);
        if (tid == 0) vp.chunk[vb] = t;
    }
    grid.sync();
    if (bid == 0) cta_scan_u32(vp.chunk, hchunks, J.d_n_out, s_part);
    grid.sync();
    PH(13);
    const uint32_t n_vox = *J.d_n_out;
    if (bid == 0 && tid == 0) { if (!BATCH) g->n_vox = n_vox; vp.vstart[n_vox] = n; }
    for (uint32_t vb = bid; vb < hchunks; vb += G) {
        const uint32_t b0 = vb * PART_CHUNK, b1 = min(n, b0 + PART_CHUNK);
        uint32_t base = vp.chunk[vb];
        for (uint32_t r0 = b0; r0 < b1; r0 += FT) {
            const uint32_t i = r0 + tid;
            // (batched: the sort left cloud f at positions [cloud_off[f], cloud_off[f + 1]), so a cloud's first point is a head too)
            const uint32_t cf = (BATCH && i < b1) ? cloud_of(coff, NC, i) : 0u;
            const bool first = BATCH && i < b1 && (i == 0 || cf != cloud_of(coff, NC, i - 1));
            const bool hd = (i < b1) && (i == 0 || skey[i] != skey[i - 1] || first);
            uint32_t before, round;
            cta_rank(hd, s_w, before, round);
            if (hd) { vp.vstart[base + before] = i; vp.vkey[base + before] = skey[i]; }
            if (first) vp.cvox[cf] = base + before;
            base += round;
        }
    }
    grid.sync();

    // ---- centroids (pcl::CentroidPoint, members in cloud order), exact 1-NN label, optional affine on the way out ----
    PH(14);
    for (uint32_t v0 = ((uint32_t)warp * G + bid) * 32u; v0 < n_vox; v0 += G * FT) {     // 32 consecutive voxels per warp, warps dealt round-robin over the SMs
        const uint32_t v = v0 + lane;
        if (v >= n_vox) continue;
        float4 c = vox_centroid_of(J.vin, sidx, vp.vstart, v);
        if (!BATCH) {
            c = vox_label_of(J.vin, sidx, vp.vstart, vp.vkey, g, n_vox, c);
            J.vout[v] = J.xform_out ? affine(J.T_out, c) : c;
        } else {
            // cloud f's voxels are [vo, vo + nvf) of the global list; the label search stays inside them
            const uint32_t f = cloud_of(coff, NC, vp.vstart[v]);
            const uint32_t vo = vp.cvox[f], o1 = coff[f + 1];
            const bool last = v + 1 == n_vox || vp.vstart[v + 1] >= o1;
            if (J.restore_labels) {
                const uint32_t nvf = last ? v + 1 - vo : lower_bound_u32(vp.vstart + v + 1, n_vox - v - 1, o1) + v + 1 - vo;
                c = vox_label_of(J.vin, sidx, vp.vstart + vo, vp.vkey + vo, g + f, nvf, c);
            }
            J.vout[coff[f] + (v - vo)] = J.xform_out ? affine(J.T_out, c) : c;
            if (last) J.cloud_nvox[f] = v + 1 - vo;
        }
    }
    PH(15);
#undef PH
}

size_t partition_tmp_words(uint32_t n) { return (size_t)(n + PART_CHUNK - 1) / PART_CHUNK + 1; }

size_t voxelize_tmp_bytes(uint32_t n, uint32_t n_clouds) {
    const size_t nseg = ((size_t)n + rs_seg_len(n) - 1) / rs_seg_len(n) + 1;
    const size_t nc = n_clouds < 1 ? 1 : n_clouds;
    // key/idx ping-pong (4 arrays), two digit-histogram matrices + digit totals, head-chunk counters, voxel starts/keys, per-CTA
    // min/max partials per cloud, first voxel per cloud (batched)
    return sizeof(uint32_t) * ((size_t)4 * n + 2 * (size_t)RD * nseg + RD + partition_tmp_words(n) + 2 * ((size_t)n + 2) + 64 +
                               6 * (size_t)kFusedMaxGrid * nc + (n_clouds ? nc : 0));
}

cudaError_t launch_node_fused(cudaStream_t st, const FusedJob& J, int sm_count, int max_ctas) {
    constexpr size_t SMEM = sizeof(uint32_t) * FW * RD;
    const bool batch = J.n_clouds > 0;
    const void* kern = batch ? (const void*)k_node_fused<true> : (const void*)k_node_fused<false>;
    static int max_ctas_per_sm[2] = {-1, -1};
    int& mc = max_ctas_per_sm[batch ? 1 : 0];
    if (mc < 0) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
        if (e != cudaSuccess) return e;
        int v = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, kern, FT, SMEM);
        if (e != cudaSuccess) return e;
        mc = v;
    }
    const int max_ctas_per_sm_ = mc;
    if (max_ctas_per_sm_ < 1) return cudaErrorLaunchOutOfResources;
    if (batch && (J.has_part || !J.cloud_off || !J.cloud_nvox || !J.d_n_out)) return cudaErrorInvalidValue;
    const uint32_t work = J.vn > J.pn || batch ? J.vn : J.pn;
    uint32_t G = (work + FT - 1) / FT;
    const uint32_t cap = (uint32_t)std::min<long long>((long long)sm_count * max_ctas_per_sm_, (long long)kFusedMaxGrid);
    G = G < 1u ? 1u : (G > cap ? cap : G);
    if (max_ctas > 0 && G > (uint32_t)max_ctas) G = (uint32_t)max_ctas;      // look-ahead jobs leave most SMs to the current node's path
    FusedJob jj = J;
    void* args[] = {&jj};
    return cudaLaunchCooperativeKernel(kern, dim3(G), dim3(FT), args, SMEM, st);
}

__global__ void k_expand_xyz(const float* __restrict__ in, float4* __restrict__ out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_float4(in[3 * (size_t)i], in[3 * (size_t)i + 1], in[3 * (size_t)i + 2], 0.0f);
}
cudaError_t launch_expand_xyz(cudaStream_t st, const float* in, float4* out, uint32_t n) {
    if (n == 0) return cudaSuccess;
    k_expand_xyz<<<(n + 255) / 256, 256, 0, st>>>(in, out, n);
    return cudaGetLastError();
}

// stable compaction by a keep byte: kept points per chunk, chunk offsets (one CTA), ordered scatter
__global__ void __launch_bounds__(FT) k_keep_count(const uint8_t* __restrict__ keep, uint32_t n, uint32_t* __restrict__ chunk) {
    __shared__ uint32_t s_w[FW];
    const uint32_t b0 = blockIdx.x * PART_CHUNK, b1 = min(n, b0 + PART_CHUNK);
    uint32_t c = 0;
    for (uint32_t i = b0 + threadIdx.x; i < b1; i += FT) c += keep[i] ? 1u : 0u;
    const uint32_t t = cta_sum(c, s_w);
    if (threadIdx.x == 0) chunk[blockIdx.x] = t;
}
__global__ void __launch_bounds__(FT) k_keep_scan(uint32_t* chunk, uint32_t n_chunks, uint32_t* total) {
    __shared__ uint32_t s_part[34];
    cta_scan_u32(chunk, n_chunks, total, s_part);
}
__global__ void __launch_bounds__(FT) k_keep_scatter(const float4* __restrict__ pts, const uint8_t* __restrict__ keep, uint32_t n,
                                                     const uint32_t* __restrict__ chunk, float4* __restrict__ out) {
    __shared__ uint32_t s_w[FW];
    const uint32_t b0 = blockIdx.x * PART_CHUNK, b1 = min(n, b0 + PART_CHUNK);
    uint32_t base = chunk[blockIdx.x];
    for (uint32_t r0 = b0; r0 < b1; r0 += FT) {
        const uint32_t i = r0 + threadIdx.x;
        const bool k = i < b1 && keep[i];
        uint32_t before, round;
        cta_rank(k, s_w, before, round);
        if (k) out[base + before] = pts[i];
        base += round;
    }
}
cudaError_t launch_compact_keep(cudaStream_t st, const float4* pts, const uint8_t* keep, uint32_t n, float4* out, uint32_t* d_n, uint32_t* tmp) {
    const uint32_t chunks = (n + PART_CHUNK - 1) / PART_CHUNK;
    if (chunks == 0) return cudaMemsetAsync(d_n, 0, sizeof(uint32_t), st);
    k_keep_count<<<chunks, FT, 0, st>>>(keep, n, tmp);
    k_keep_scan<<<1, FT, 0, st>>>(tmp, chunks, d_n);
    k_keep_scatter<<<chunks, FT, 0, st>>>(pts, keep, n, tmp, out);
    return cudaGetLastError();
}

}  // namespace erasor
