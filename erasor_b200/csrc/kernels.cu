// kernels.cu -- the sm_100a kernels of the R-POD -> Scan Ratio Test -> R-GPF path.
//
//   K1  k1_rpod_bin     polar index + per-bin min/max z and count, query and map in one launch
//                       (ERASOR::voi2r_pod x2 + pt2r_pod, reference erasor.cpp:87-144)
//   K3  k3_srt          per-bin totals, Scan Ratio Test, status / action codes, v3 neighbour pass,
//                       scatter offsets, flagged-bin work list
//                       (compare_vois_and_revert_ground[_w_block], erasor.cpp:346-427, 448-563, 573-595)
//   K2  k2_scatter[_mw] stable counting-sort scatter of points into bin order (the per-bin
//                       pcl::PointCloud push_back, erasor.cpp:89) -- all bins (cloud mode) or flagged bins only (mask mode)
//   K4  k4_rgpf         Region-wise Ground Plane Fitting per flagged bin
//                       (extract_ground / extract_initial_seeds_ / estimate_plane_, erasor.cpp:183-294)
//   K5  k5_plan/k5_copy output assembly in the reference's order (r_pod2pc, get_static_estimate,
//                       get_outliers, erasor.cpp:309-327, 612-626)
//
// No tensor cores anywhere: the path is bandwidth-bound indexing and reduction (DESIGN.md section 5).
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>

#include "device_types.h"
#include "kernels.h"

#include <algorithm>
#include <mutex>
#include <unordered_map>

namespace erasor {

#define FULL_MASK 0xFFFFFFFFu

// cudaFuncSetAttribute costs a few microseconds per call; the dynamic shared-memory ceiling of a kernel only ever has
// to grow, so remember the largest value set per kernel and skip the call otherwise.
template <class K>
static cudaError_t ensure_dyn_smem(K kern, size_t bytes) {
    static std::mutex mu;
    static std::unordered_map<const void*, size_t> seen;
    std::lock_guard<std::mutex> lock(mu);
    const void* key = reinterpret_cast<const void*>(kern);
    auto it = seen.find(key);
    if (it != seen.end() && it->second >= bytes) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) seen[key] = bytes;
    return e;
}

__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// ============================================================================================
// K1
// ============================================================================================
// Warp-level pre-aggregation of (bin, z) into the CTA's shared tables.  Input clouds are spatially
// coherent (voxel-key order, or bin order after the first frame), so most warps hold 1-3 runs of equal bins:
// one REDUX pair + three shared atomics per run instead of three atomics per point.
__device__ __forceinline__ void k1_aggregate(int key, uint32_t zenc, int lane, uint32_t* s_cnt, uint32_t* s_mn, uint32_t* s_mx, int B) {
    // key: bin id in [0,B), B for "not binned", -2 for an out-of-range lane
    const int key0 = __shfl_sync(FULL_MASK, key, 0);
    if (__all_sync(FULL_MASK, key == key0)) {
        if (key0 >= 0) {
            if (key0 < B) {
                const uint32_t mn = __reduce_min_sync(FULL_MASK, zenc);
                const uint32_t mx = __reduce_max_sync(FULL_MASK, zenc);
                if (lane == 0) {
                    atomicMin(&s_mn[key0], mn);
                    atomicMax(&s_mx[key0], mx);
                    atomicAdd(&s_cnt[key0], 32u);
                }
            } else if (lane == 0) {
                atomicAdd(&s_cnt[B], 32u);
            }
        }
        return;
    }
    // Mixed warp (in node mode a third of the lanes of a typical row lie outside the VoI, so runs of equal bins are short):
    // per-lane shared-memory atomics, but only where they can change something -- a bin's min / max settle after its
    // first few points, and a plain (possibly stale) read is a safe filter because the values only move one way.
    // (A segmented shuffle scan over the runs was measured at 68 instructions per row here, ncu r02; this is ~14.)
    if (key >= 0) {
        if (key < B) {
            if (zenc < s_mn[key]) atomicMin(&s_mn[key], zenc);
            if (zenc > s_mx[key]) atomicMax(&s_mx[key], zenc);
        }
        atomicAdd(&s_cnt[key], 1u);          // key == B: the complement's count
    }
}

__device__ __forceinline__ float rsqrt_ftz(float v) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
__device__ __forceinline__ float div_ftz(float a, float b) { float r; asm("div.approx.ftz.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }

// the exact path of binning.h, kept out of line: it is taken by ~1e-4 of the points
__device__ __noinline__ int bin_exact(const BinTablesView& T, float x, float y, float z, BinFenceCounters* fc) {
    return bin_of_point(T, T.ring_thr, x, y, z, fc);
}

// Branch-free fast path of binning.h's bin_of_point for the device, float arithmetic only: returns the bin, -1 (not
// binned) or -3 when the point needs the exact path (r^2 inside the guard band of s_max or of a ring threshold, ring guess
// off, sector coordinate inside its guard band, y == 0).  Every decision taken here is one the exact path would take too:
// the float r^2 is compared against thresholds widened by its own worst-case error (binning_tables.cpp).
__device__ __forceinline__ int bin_fast(float x, float y, float z, float z_lo, float z_hi, float smax_lo, float smax_hi, float inv_ring, float inv_ss,
                                        float eps_q, int R, int S, const float2* __restrict__ s_ringf) {
    const float sf   = fmaf(y, y, x * x);
    const bool  zin  = (z < z_hi) && (z > z_lo);
    const bool  in_sure  = sf <= smax_lo;
    const bool  out_sure = !(sf <= smax_hi);                  // also NaN
    const float sfc = fmaxf(sf, 1e-30f);
    int g = (int)(sfc * rsqrt_ftz(sfc) * inv_ring);
    g = min(g, R - 1);
    const float2 t0 = s_ringf[g], t1 = s_ringf[g + 1];         // {up, dn} of thresholds g and g + 1
    const bool ring_ok = (sf >= t0.x) && (sf < t1.y);
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    float a = atan_unit(div_ftz(mn, mx));
    if (ay > ax)  a = 1.57079637f - a;
    if (x < 0.0f) a = 3.14159274f - a;
    if (y < 0.0f) a = 6.28318548f - a;
    const float q  = a * inv_ss;
    const int   k  = (int)q;
    const float fr = q - (float)k;
    const bool sec_ok = (fr >= eps_q) && (fr <= 1.0f - eps_q) && (ay != 0.0f);
    if (!zin || out_sure) return -1;
    if (!(in_sure && ring_ok && sec_ok)) return -3;
    return min(k, S - 1) * R + g;
}

// pcl::transformPointCloud, PCL 1.8 scalar path: ((m0*x + m1*y) + m2*z) + m3 in float, no contraction -- the same
// association as updater_kernels.cu::affine and oracle transform_point_cloud (OfflineMapUpdater.cpp:436)
__device__ __forceinline__ float4 affine12(const float* __restrict__ T, float4 p) {
    float4 o;
    o.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[0], p.x), __fmul_rn(T[1], p.y)), __fmul_rn(T[2], p.z)), T[3]);
    o.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[4], p.x), __fmul_rn(T[5], p.y)), __fmul_rn(T[6], p.z)), T[7]);
    o.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[8], p.x), __fmul_rn(T[9], p.y)), __fmul_rn(T[10], p.z)), T[11]);
    o.w = p.w;
    return o;
}
// OfflineMapUpdater::fetch_VoI's cut (OfflineMapUpdater.cpp:394-396): pow(pt.x - x, 2) + pow(pt.y - y, 2) < max_dist_square in
// double on float differences.  A float evaluation decides every point outside a 1e-6 band around the limit (its error is
// below 2.4e-7 relative); points inside the band get the reference's double expression.
__device__ __forceinline__ bool in_voi_radius(const NodePose& P, float x, float y) {
    const float dxf = x - P.pxf, dyf = y - P.pyf;
    const float d2f = fmaf(dyf, dyf, dxf * dxf);
    if (d2f < P.lim_lo) return true;
    if (d2f > P.lim_hi) return false;
    const double dx = __dsub_rn((double)x, P.px), dy = __dsub_rn((double)y, P.py);
    return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < P.limit;
}

// NODE: the map cloud is the resident global map in the origin frame; every frame's chunks scan it, keep the points
// inside the frame's radius (fetch_VoI) and bin their origin -> body transforms.  Points outside the VoI get no bin id
// and are not counted anywhere (they are the reference's map_outskirts_, which never reach ERASOR).
template <int THREADS, int UNROLL, bool ROWS, bool NODE>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 4 : 1)      // four 8-warp CTAs per SM (64 registers) or one 32-warp CTA
k1_rpod_bin(BinTablesView T, const float4* __restrict__ map_pts, const float4* __restrict__ qry_pts,
            const ChunkDesc* __restrict__ chunks, uint16_t* __restrict__ bin_map, uint16_t* __restrict__ bin_qry,
            uint32_t* __restrict__ ch_cnt, uint32_t* __restrict__ zmin, uint32_t* __restrict__ zmax, uint32_t* __restrict__ cnt_tab,
            int B, int F, unsigned long long* __restrict__ fence, const NodePose* __restrict__ poses,
            uint32_t* __restrict__ list_idx, uint32_t* __restrict__ list_cnt, int qry_xyz /*query cloud packed x y z (12 bytes per point)*/) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2*   s_ring = reinterpret_cast<float2*>(smem_raw);               // {up, dn} guard thresholds of r^2 per ring boundary
    uint32_t* s_cnt  = reinterpret_cast<uint32_t*>(s_ring + ((T.R + 2) & ~1));
    uint32_t* s_mn   = s_cnt + (B + 1);
    uint32_t* s_mx   = s_mn + B;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = THREADS / 32;
    const ChunkDesc cd = chunks[blockIdx.x];
    __shared__ NodePose s_pose;
    const bool node_map = NODE && cd.cloud == 0;          // CTA-uniform

    for (int i = tid; i <= T.R; i += THREADS) s_ring[i] = make_float2(T.ring_guard[2 * i], T.ring_guard[2 * i + 1]);
    for (int i = tid; i <= B; i += THREADS) s_cnt[i] = 0u;
    for (int i = tid; i < B; i += THREADS) { s_mn[i] = 0xFFFFFFFFu; s_mx[i] = 0u; }
    if (NODE && tid == 0) s_pose = poses[cd.frame];
    __syncthreads();

    const float4* __restrict__ src = (cd.cloud == 0 ? map_pts : qry_pts) + cd.begin;
    uint16_t* __restrict__     dst = (cd.cloud == 0 ? bin_map : bin_qry) + cd.bin_begin;
    BinFenceCounters fc{0u, 0u, 0u};
    const float  z_lo = T.z_lo, z_hi = T.z_hi, inv_ring = T.inv_ring, inv_ss = T.inv_ss, eps_q = T.eps_q;
    const float  smax_lo = T.smax_lo, smax_hi = T.smax_hi;
    const int    R = T.R, S = T.S;

    if (node_map) {
        // ---- node mode, map cloud: fetch_VoI fused in.  Every warp streams its own contiguous sub-range of the chunk (four
        // float4 loads in flight per lane, no block-wide barrier) and compacts the points inside the VoI, in order, into a
        // 64-entry ring in shared memory; whenever the ring holds a full row the warp runs the expensive part on it --
        // origin -> body transform, polar bin, table update -- with all 32 lanes busy (in map order a third of the lanes of a
        // mixed row lie outside the radius, ncu r02), and appends (bin id, map index) to its dense list.  K2 walks those
        // lists, warp by warp in the same split, instead of every map point.
        __shared__ float4 s_ring_q[NODE ? NW * 64 : 1];
        float4* __restrict__ q = s_ring_q + warp * 64;
        const uint32_t sub = (((cd.len + NW - 1) / NW) + 31u) & ~31u;
        const uint32_t w0 = min(cd.len, (uint32_t)warp * sub), w1 = min(cd.len, w0 + sub);
        uint16_t* __restrict__ lbin = bin_map + cd.bin_begin + w0;
        uint32_t* __restrict__ lidx = list_idx + cd.bin_begin + w0;
        uint32_t qh = 0, qt = 0;                       // ring head / tail as running counts (qt - qh < 64)
        auto dense_row = [&](uint32_t n) {             // the first n (<= 32) entries of the ring
            const bool ok = (uint32_t)lane < n;
            const float4 e = q[(qh + lane) & 63u];
            const float4 pp = affine12(s_pose.T, e);
            int b = bin_fast(pp.x, pp.y, pp.z, z_lo, z_hi, smax_lo, smax_hi, inv_ring, inv_ss, eps_q, R, S, s_ring);
            if (__any_sync(FULL_MASK, ok && b == -3)) {
                if (ok && b == -3) b = bin_exact(T, pp.x, pp.y, pp.z, &fc);   // exact path (rare)
            }
            int key = -2;
            if (ok) {
                lbin[qh + lane] = (b < 0) ? kNoBin16 : (uint16_t)b;
                lidx[qh + lane] = cd.begin + __float_as_uint(e.w);              // index in the resident map
                key = (b < 0) ? B : b;
            }
            k1_aggregate(key, float_to_ordered(pp.z), lane, s_cnt, s_mn, s_mx, B);
            qh += n;
            __syncwarp();                              // the row's ring slots may be overwritten from here on
        };
        // (the resident map carries kMapPad points of slack, so the loads need no bounds checks: positions >= w1 are masked below)
        for (uint32_t base = w0; base < w1; base += 32u * UNROLL) {
            float4 p[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) p[u] = ld_stream_f4(src + (base + u * 32u + lane));
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const uint32_t i = base + u * 32u + lane;
                const bool in = (i < w1) && in_voi_radius(s_pose, p[u].x, p[u].y);
                const unsigned bal = __ballot_sync(FULL_MASK, in);
                if (bal == 0u) continue;                                         // warp-uniform
                if (in) q[(qt + __popc(bal & ((1u << lane) - 1u))) & 63u] = make_float4(p[u].x, p[u].y, p[u].z, __uint_as_float(i));
                qt += __popc(bal);
                __syncwarp();
                if (qt - qh >= 32u) dense_row(32u);
            }
        }
        if (qt != qh) dense_row(qt - qh);
        if (lane == 0) list_cnt[(size_t)blockIdx.x * kListWarps + warp] = qt;
    } else
    for (uint32_t base = warp * (32u * UNROLL); base < cd.len; base += NW * (32u * UNROLL)) {
        float4 p[UNROLL];
        const bool full = base + 32u * UNROLL <= cd.len;          // warp-uniform
        if (qry_xyz && cd.cloud == 1) {                            // CTA-uniform: packed x y z, three coalesced 4-byte loads per point
            const float* __restrict__ q3 = reinterpret_cast<const float*>(qry_pts) + (size_t)cd.begin * 3u;
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const uint32_t i = base + u * 32u + lane;
                p[u] = (full || i < cd.len) ? make_float4(__ldg(q3 + 3u * (size_t)i), __ldg(q3 + 3u * (size_t)i + 1u), __ldg(q3 + 3u * (size_t)i + 2u), 0.f)
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        } else {
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const uint32_t i = base + u * 32u + lane;
            p[u] = (full || i < cd.len) ? ld_stream_f4(src + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const uint32_t i = base + u * 32u + lane;
            const bool ok = full || i < cd.len;
            const float4 pp = p[u];
            int b = bin_fast(pp.x, pp.y, pp.z, z_lo, z_hi, smax_lo, smax_hi, inv_ring, inv_ss, eps_q, R, S, s_ring);
            if (__any_sync(FULL_MASK, ok && b == -3)) {
                if (ok && b == -3) b = bin_exact(T, pp.x, pp.y, pp.z, &fc);   // exact path (rare)
            }
            int key = -2;
            if (ok) {
                dst[i] = (b < 0) ? kNoBin16 : (uint16_t)b;
                key = (b < 0) ? B : b;
            }
            k1_aggregate(key, float_to_ordered(pp.z), lane, s_cnt, s_mn, s_mx, B);
        }
    }
    __syncthreads();

    // flush: per-bin count / min / max by RED to the frame tables (non-empty bins only); in cloud mode also the dense
    // per-chunk count row that K3 turns into prefixes for K2's stable scatter
    uint32_t* __restrict__ row = ROWS ? ch_cnt + (size_t)blockIdx.x * (B + 1) : nullptr;
    const size_t ft = ((size_t)cd.cloud * F + cd.frame) * B;
    const size_t ct = ((size_t)cd.cloud * F + cd.frame) * (B + 1);
    for (int i = tid; i <= B; i += THREADS) {
        const uint32_t c = s_cnt[i];
        if (ROWS) row[i] = c;
        if (c != 0u) {
            atomicAdd(&cnt_tab[ct + i], c);
            if (i < B) {
                atomicMin(&zmin[ft + i], s_mn[i]);
                atomicMax(&zmax[ft + i], s_mx[i]);
            }
        }
    }
    if (fc.negzero) atomicAdd(&fence[0], (unsigned long long)fc.negzero);
    if (fc.ambiguous) atomicAdd(&fence[2], (unsigned long long)fc.ambiguous);
    if (fc.slow) atomicAdd(&fence[3], (unsigned long long)fc.slow);
}

bool k1_big_tables(int R, int B) { return k1_smem_bytes(R, B) > 56 * 1024; }

size_t k1_smem_bytes(int R, int B) {
    return sizeof(float2) * ((R + 2) & ~1) + sizeof(uint32_t) * ((size_t)(B + 1) + 2 * (size_t)B);
}

cudaError_t launch_k1(cudaStream_t st, const BinTablesView& T, const float4* map_pts, const float4* qry_pts,
                      const ChunkDesc* chunks, int n_chunks, uint16_t* bin_map, uint16_t* bin_qry, uint32_t* ch_cnt,
                      uint32_t* zmin, uint32_t* zmax, uint32_t* cnt_tab, int B, int F, unsigned long long* fence, const NodePose* poses,
                      uint32_t* list_idx, uint32_t* list_cnt, bool qry_xyz) {
    if (n_chunks == 0) return cudaSuccess;
    const int qx = qry_xyz ? 1 : 0;
    constexpr int UNROLL = 4;
    const size_t smem = k1_smem_bytes(T.R, B);
    cudaError_t e;
    // Bin tables beyond ~56 KB (40 x 360 bins: 173 KB) leave one CTA per SM: give that CTA 32 warps instead of 8, the
    // kernel needs ~32 resident warps per SM to cover its latencies (measured: 1 / 2 / 4 CTAs of 8 warps -> 128 / 75 / 62 us).
    if (k1_big_tables(T.R, B)) {
        constexpr int THREADS = 1024;
        if (poses) {
            auto kern = k1_rpod_bin<THREADS, UNROLL, true, true>;
            if ((e = ensure_dyn_smem(kern, smem)) != cudaSuccess) return e;
            kern<<<n_chunks, THREADS, smem, st>>>(T, map_pts, qry_pts, chunks, bin_map, bin_qry, ch_cnt, zmin, zmax, cnt_tab, B, F, fence, poses, list_idx, list_cnt, qx);
        } else {
            auto kern = k1_rpod_bin<THREADS, UNROLL, true, false>;
            if ((e = ensure_dyn_smem(kern, smem)) != cudaSuccess) return e;
            kern<<<n_chunks, THREADS, smem, st>>>(T, map_pts, qry_pts, chunks, bin_map, bin_qry, ch_cnt, zmin, zmax, cnt_tab, B, F, fence, nullptr, nullptr, nullptr, qx);
        }
        return cudaGetLastError();
    }
    constexpr int THREADS = 256;
    if (poses) {
        auto kern = k1_rpod_bin<THREADS, UNROLL, true, true>;
        if ((e = ensure_dyn_smem(kern, smem)) != cudaSuccess) return e;
        kern<<<n_chunks, THREADS, smem, st>>>(T, map_pts, qry_pts, chunks, bin_map, bin_qry, ch_cnt, zmin, zmax, cnt_tab, B, F, fence, poses, list_idx, list_cnt, qx);
    } else {
        auto kern = k1_rpod_bin<THREADS, UNROLL, true, false>;
        if ((e = ensure_dyn_smem(kern, smem)) != cudaSuccess) return e;
        kern<<<n_chunks, THREADS, smem, st>>>(T, map_pts, qry_pts, chunks, bin_map, bin_qry, ch_cnt, zmin, zmax, cnt_tab, B, F, fence, nullptr, nullptr, nullptr, qx);
    }
    return cudaGetLastError();
}

// ============================================================================================
// K3
// ============================================================================================
// exclusive scan of in[0..n) into out[0..n) (may alias); every thread returns the total.
__device__ uint32_t block_excl_scan(const uint32_t* in, uint32_t* out, int n, uint32_t* s_part /*[34]*/) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    const int seg = (n + nt - 1) / nt;
    const int b0 = min(n, tid * seg), b1 = min(n, b0 + seg);
    uint32_t sum = 0;
    for (int i = b0; i < b1; ++i) sum += in[i];
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(FULL_MASK, incl, o);
        if (lane >= o) incl += v;
    }
    __syncthreads();                     // s_part may still be read from a previous call
    if (lane == 31) s_part[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = lane < nw ? s_part[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(FULL_MASK, wi, o);
            if (lane >= o) wi += v;
        }
        if (lane < nw) s_part[lane] = wi - w;
        if (lane == 31) s_part[33] = wi;
    }
    __syncthreads();
    uint32_t run = s_part[warp] + incl - sum;
    const uint32_t total = s_part[33];
    for (int i = b0; i < b1; ++i) {
        const uint32_t v = in[i];
        out[i] = run;
        run += v;
    }
    __syncthreads();
    return total;
}

__device__ __forceinline__ double std_min_d(double a, double b) { return (b < a) ? b : a; }   // std::min, NaN-faithful (App. B-4)

// Does the Scan Ratio Test hand this bin to R-GPF?  The same decisions as k3_srt's status passes, reduced to the one bit
// the scatter needs: version 3 -- MAP_IS_HIGHER in pass 1 and map_dh > 0.5 in pass 2 (erasor.cpp:448-486, 507-511; the
// neighbour test of pass 2 only relabels MERGE_BINS as BLOCKED); version 2 -- MAP_IS_HIGHER and map.max_h > th_bin_max_h
// (erasor.cpp:346-389).
__device__ __forceinline__ bool srt_is_flagged(const SrtParams& P, uint32_t mc, uint32_t qc, uint32_t zmx_m, uint32_t zmn_m, uint32_t zmx_q, uint32_t zmn_q) {
    if (mc == 0u || qc == 0u || P.minimum_num_pts < 0 || qc < (uint32_t)P.minimum_num_pts) return false;
    const double map_max = (double)ordered_to_float(zmx_m);
    const double map_dh  = map_max - (double)ordered_to_float(zmn_m);
    const double curr_dh = (double)ordered_to_float(zmx_q) - (double)ordered_to_float(zmn_q);
    const double ratio   = std_min_d(map_dh / curr_dh, curr_dh / map_dh);
    if (!(ratio < P.scan_ratio_threshold) || !(map_dh >= curr_dh)) return false;
    return (P.version == 3) ? (map_dh > 0.5) : (map_max > P.th_bin_max_h);
}

__global__ void __launch_bounds__(1024)
k3_srt(SrtParams P, int F, const uint32_t* __restrict__ chunk_range /*[2][F+1]*/, uint32_t* __restrict__ ch_cnt,
       const uint32_t* __restrict__ zmin, const uint32_t* __restrict__ zmax, const uint32_t* __restrict__ frame_off /*[2][F+1]*/,
       const uint32_t* __restrict__ cnt /*[2][F][B+1]*/, uint32_t* __restrict__ dst_start /*[2][F][B+2]*/,
       uint8_t* __restrict__ status /*[F][B]*/, uint8_t* __restrict__ action /*[F][B]*/,
       uint32_t* __restrict__ flag_slot /*[F][B]*/, uint32_t* __restrict__ n_flagged /*[F]*/, uint32_t* __restrict__ frame_rec_base /*[F]*/,
       FlagRec* __restrict__ recs, uint32_t* __restrict__ n_recs, uint32_t rec_capacity,
       uint32_t* __restrict__ queue /*[kQueueWords]*/, uint32_t* __restrict__ bucket_list /*[kNumBuckets][rec_capacity]*/) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int B = P.B, R = P.R, S = P.S;
    uint32_t* s_sz   = reinterpret_cast<uint32_t*>(smem_raw);          // B+2
    uint32_t* s_part = s_sz + (B + 2);                                 // 34
    uint8_t*  s_st   = reinterpret_cast<uint8_t*>(s_part + 34);        // B
    __shared__ uint32_t s_rec_base;
    const int f = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;

    const uint32_t* cm = cnt + ((size_t)0 * F + f) * (B + 1);
    const uint32_t* cq = cnt + ((size_t)1 * F + f) * (B + 1);
    const uint32_t* mnm = zmin + ((size_t)0 * F + f) * B; const uint32_t* mxm = zmax + ((size_t)0 * F + f) * B;
    const uint32_t* mnq = zmin + ((size_t)1 * F + f) * B; const uint32_t* mxq = zmax + ((size_t)1 * F + f) * B;
    uint8_t* st_out  = status + (size_t)f * B;
    uint8_t* act_out = action + (size_t)f * B;
    const bool min_pts_neg = P.minimum_num_pts < 0;     // size_t < int comparison wraps (App. B-9)
    long long t_prev = clock64();                       // phase profile of frame 0 (erasor_get_srt_profile)
#define K3_TICK(slot) do { if (f == 0 && tid == 0) { const long long t__ = clock64(); queue[20 + (slot)] = (uint32_t)(t__ - t_prev); t_prev = t__; } } while (0)

    if (P.version == 3) {
        // pass 1 (erasor.cpp:448-486)
        for (int b = tid; b < B; b += nt) {
            const uint32_t mc = cm[b], qc = cq[b];
            const uint32_t zmx_m = mxm[b], zmn_m = mnm[b], zmx_q = mxq[b], zmn_q = mnq[b];   // one round trip for all six tables
            uint8_t st = ST_LITTLE;
            if (mc != 0u && !(min_pts_neg || qc < (uint32_t)P.minimum_num_pts)) {
                // empty curr bin keeps the reference's sentinels: max_h = -INF, min_h = +INF (erasor.h:3)
                const double map_dh  = (double)ordered_to_float(zmx_m) - (double)ordered_to_float(zmn_m);
                const double curr_dh = (qc != 0u) ? (double)ordered_to_float(zmx_q) - (double)ordered_to_float(zmn_q)
                                                  : (-10000000000000.0 - 10000000000000.0);
                const double ratio   = std_min_d(map_dh / curr_dh, curr_dh / map_dh);
                if (qc != 0u) {
                    if (ratio < P.scan_ratio_threshold) {
                        if (map_dh >= curr_dh) st = ST_MAP_HIGH;
                        else if (map_dh <= curr_dh) st = ST_CURR_HIGH;
                    } else {
                        st = ST_MERGE;
                    }
                }
            }
            s_st[b] = st;
        }
        __syncthreads();
        // pass 2 (erasor.cpp:493-563)
        for (int b = tid; b < B; b += nt) {
            const int theta = b / R, r = b - theta * R;
            const uint8_t s1 = s_st[b];
            uint8_t st = s1, act = ACT_MAP;
            if (s1 == ST_MAP_HIGH) {
                const double map_dh = (double)ordered_to_float(mxm[b]) - (double)ordered_to_float(mnm[b]);
                if (map_dh > 0.5) act = ACT_FLAG; else st = ST_LITTLE;       // NOT_ASSIGNED == 0.0 == LITTLE_NUM
            } else if (s1 == ST_MERGE) {
                // is_dynamic_obj_close(r_pod_selected, r, theta, 1, 1), wrap with num_rings (sic, App. B-2)
                bool close = false;
                for (int j = theta - 1; j <= theta + 1; ++j) {
                    int tj = j;
                    if (j < 0) tj = j + R; else if (j >= S) tj = j - R;
                    if (tj < 0 || tj >= S) continue;                       // fence: reference indexes out of range here
                    const int r0 = max(0, r - 1), r1 = min(r + 1, R - 1);
                    for (int rr = r0; rr <= r1; ++rr) {
                        if (rr == r && tj == theta) continue;
                        if (s_st[tj * R + rr] == ST_CURR_HIGH) close = true;
                    }
                }
                st = close ? ST_BLOCKED : ST_MERGE;
            }
            st_out[b] = st; act_out[b] = act;
        }
    } else {
        // version 2 (erasor.cpp:346-427)
        for (int b = tid; b < B; b += nt) {
            const uint32_t mc = cm[b], qc = cq[b];
            uint8_t st = ST_LITTLE, act = ACT_NONE;
            if (min_pts_neg || qc < (uint32_t)P.minimum_num_pts) {
                act = ACT_MAP; st = ST_LITTLE;
            } else if (qc != 0u && mc != 0u) {
                const double map_max = (double)ordered_to_float(mxm[b]), cur_max = (double)ordered_to_float(mxq[b]);
                const double map_dh  = map_max - (double)ordered_to_float(mnm[b]);
                const double curr_dh = cur_max - (double)ordered_to_float(mnq[b]);
                const double ratio   = std_min_d(map_dh / curr_dh, curr_dh / map_dh);
                if (ratio < P.scan_ratio_threshold) {
                    if (map_dh >= curr_dh) {
                        st = ST_MAP_HIGH;
                        act = (map_max > P.th_bin_max_h) ? ACT_FLAG : ACT_MAP;
                    } else if (map_dh <= curr_dh) {
                        st = ST_CURR_HIGH;
                        act = ACT_MAP;
                        if (cur_max > P.th_bin_max_h) act |= ACT_CURR_REJECTED_BIT;
                    }
                } else {
                    st = ST_MERGE; act = ACT_MERGE;
                }
            } else if (qc != 0u) {
                act = ACT_CURR;
            } else if (mc != 0u) {
                act = ACT_MAP;
            }
            st_out[b] = st; act_out[b] = act;
        }
    }
    __syncthreads();
    K3_TICK(0);

    // in-place exclusive prefix of the per-chunk count rows over the frame's chunks, for the bins K2 will scatter:
    // every bin of both clouds in cloud mode, the flagged map bins only in mask mode (the per-bin totals themselves
    // were accumulated by K1 into cnt[])
    for (int c = 0; c < 2; ++c) {
        if (c == 1 && P.scatter_mode != 0) break;
        const uint32_t c0 = chunk_range[c * (F + 1) + f], c1 = chunk_range[c * (F + 1) + f + 1];
        for (int b = tid; b <= B; b += nt) {
            const bool take = (P.scatter_mode == 0) || (b < B && (act_out[b] & 0x0F) == ACT_FLAG);
            if (!take) continue;
            // eight rows per round trip: the loads of a batch are independent, only the running sum is serial
            uint32_t run = 0;
            for (uint32_t k0 = c0; k0 < c1; k0 += 8u) {
                uint32_t v[8];
#pragma unroll
                for (uint32_t u = 0; u < 8u; ++u) v[u] = (k0 + u < c1) ? ch_cnt[(size_t)(k0 + u) * (B + 1) + b] : 0u;
#pragma unroll
                for (uint32_t u = 0; u < 8u; ++u) {
                    if (k0 + u < c1) { ch_cnt[(size_t)(k0 + u) * (B + 1) + b] = run; run += v[u]; }
                }
            }
        }
    }
    __syncthreads();
    K3_TICK(1);
    // flagged bins, in bin order
    uint32_t* slot_out = flag_slot + (size_t)f * B;
    for (int b = tid; b < B; b += nt) s_sz[b] = ((act_out[b] & 0x0F) == ACT_FLAG) ? 1u : 0u;
    __syncthreads();
    const uint32_t nflag = block_excl_scan(s_sz, s_sz, B, s_part);
    uint32_t rec_base_reg = 0u;      // thread 0: the atomic's round trip overlaps the map-offset scan below
    if (tid == 0) {
        n_flagged[f] = nflag;
        rec_base_reg = nflag ? atomicAdd(n_recs, nflag) : 0u;
    }
    for (int b = tid; b < B; b += nt) slot_out[b] = ((act_out[b] & 0x0F) == ACT_FLAG) ? s_sz[b] : kSkip;
    __syncthreads();
    K3_TICK(2);

    // scatter offsets, map cloud: every bin + complement (mode 0) or flagged bins only (mode 1)
    uint32_t* dsm = dst_start + ((size_t)0 * F + f) * (B + 2);
    uint32_t* dsq = dst_start + ((size_t)1 * F + f) * (B + 2);
    for (int b = tid; b <= B; b += nt) {
        const bool take = (P.scatter_mode == 0) || (b < B && (act_out[b] & 0x0F) == ACT_FLAG);
        s_sz[b] = take ? cm[b] : 0u;
    }
    __syncthreads();
    const uint32_t tot_m = block_excl_scan(s_sz, s_sz, B + 1, s_part);
    for (int b = tid; b <= B; b += nt) {
        const bool take = (P.scatter_mode == 0) || (b < B && (act_out[b] & 0x0F) == ACT_FLAG);
        dsm[b] = take ? s_sz[b] : kSkip;
    }
    if (tid == 0) { dsm[B + 1] = tot_m; s_rec_base = rec_base_reg; frame_rec_base[f] = rec_base_reg; }
    __syncthreads();
    const uint32_t rec_base = s_rec_base;
    K3_TICK(3);
    // flagged-bin records for K4
    for (int b = tid; b < B; b += nt) {
        if ((act_out[b] & 0x0F) == ACT_FLAG) {
            const uint32_t slot = slot_out[b];
            const uint32_t ri   = rec_base + slot;
            if (ri < rec_capacity) {
                FlagRec& rc = recs[ri];
                rc.frame = f; rc.bin = b; rc.slot = slot; rc.n_points = cm[b];
                rc.src_begin = frame_off[f] + s_sz[b];
                rc.n_seeds = 0; rc.n_empty_fits = 0; rc.n_ground_final = 0; rc.lpr_height = 0.0; rc.cursor = 0u; rc.n_rejected = 0u;
                if (cm[b] != 0u) {   // hand the record to the R-GPF size bucket (order inside a bucket is irrelevant: bins are independent)
                    const int bk = rgpf_bucket_of(cm[b]);
                    bucket_list[(size_t)bk * rec_capacity + atomicAdd(&queue[bk], 1u)] = ri;
                }
            }
        }
    }
    __syncthreads();
    K3_TICK(4);
    // query cloud: all binned points (mode 0) or nothing (mode 1)
    if (P.scatter_mode == 0) {
        for (int b = tid; b <= B; b += nt) s_sz[b] = (b < B) ? cq[b] : 0u;
        __syncthreads();
        const uint32_t tot_q = block_excl_scan(s_sz, s_sz, B + 1, s_part);
        for (int b = tid; b <= B; b += nt) dsq[b] = (b < B) ? s_sz[b] : kSkip;
        if (tid == 0) dsq[B + 1] = tot_q;
    } else {
        for (int b = tid; b <= B; b += nt) dsq[b] = kSkip;
        if (tid == 0) dsq[B + 1] = 0u;
    }
    K3_TICK(5);
#undef K3_TICK
}

size_t k3_smem_bytes(int B) { return sizeof(uint32_t) * ((size_t)B + 2 + 34) + (size_t)B + 16; }

cudaError_t launch_k3(cudaStream_t st, const SrtParams& P, int F, const uint32_t* chunk_range, uint32_t* ch_cnt,
                      const uint32_t* zmin, const uint32_t* zmax, const uint32_t* frame_off, const uint32_t* cnt, uint32_t* dst_start,
                      uint8_t* status, uint8_t* action, uint32_t* flag_slot, uint32_t* n_flagged, uint32_t* frame_rec_base,
                      FlagRec* recs, uint32_t* n_recs, uint32_t rec_capacity, uint32_t* queue, uint32_t* bucket_list) {
    const size_t smem = k3_smem_bytes(P.B);
    cudaError_t e = ensure_dyn_smem(k3_srt, smem);
    if (e != cudaSuccess) return e;
    k3_srt<<<F, 1024, smem, st>>>(P, F, chunk_range, ch_cnt, zmin, zmax, frame_off, cnt, dst_start, status, action,
                                  flag_slot, n_flagged, frame_rec_base, recs, n_recs, rec_capacity, queue, bucket_list);
    return cudaGetLastError();
}

// ============================================================================================
// K2
// ============================================================================================
// Stable counting-sort scatter of the points of the "scattered" bins into bin-contiguous storage, source order kept
// inside every bin (the per-bin pcl::PointCloud push_back of erasor.cpp:89).  Scattered bins are numbered by dense
// SLOTS in bin order: every bin plus the complement (cloud mode: slot == bin, B + 1 slots) or the flagged bins only
// (mask mode: K3's flag_slot, n_flagged[frame] slots -- a few per cent of the bins).
//
// One CTA of W warps per chunk; the warps split the chunk into W contiguous sub-ranges.  Pass A counts each sub-range
// per slot into the warp's own shared-memory row (match_any dedups a 32-point step, so no atomics); a column scan
// turns the rows into absolute destinations (dst_start + earlier chunks of the frame + earlier warps); pass B re-walks
// the sub-range in order.  The rows cover a WINDOW of SW slots; a frame with more slots than fit in shared memory
// (40 x 360 bins in cloud mode) takes several window passes over the chunk's bin ids, so there is no bin-count limit
// and no slow fallback.  NODE: points are read from the resident map and moved origin -> body on the way (fetch_VoI's
// transform, OfflineMapUpdater.cpp:436), the source index is the global map index.
// pass A of one window: per-slot counts of the warp's sub-range [s0, s1) into its own row
__device__ __forceinline__ void k2_count_pass(const uint16_t* __restrict__ ids, uint32_t s0, uint32_t s1, const uint16_t* __restrict__ s_slot,
                                              uint32_t win0, uint32_t ns, uint32_t* __restrict__ mine, int B, int lane) {
    // Both passes walk the sub-range 256 points (8 steps of 32) at a time; the bin ids of the next block are loaded while
    // the current one is processed, so that no step waits on global memory.  Only points of the window's slots take part
    // in the match_any ranking.
    // (the id arrays carry kIdPad entries of slack, so the loads need no bounds checks: positions >= s1 are masked by `take`)
    uint32_t cur[8], nxt[8];
    const uint16_t* __restrict__ pb = ids + (size_t)s0 + lane;      // one 64-bit base per block, constant offsets per load
#pragma unroll
    for (int u = 0; u < 8; ++u) cur[u] = pb[u * 32];
    for (uint32_t i0 = s0; i0 < s1; i0 += 256u, pb += 256) {
#pragma unroll
        for (int u = 0; u < 8; ++u) nxt[u] = pb[256 + u * 32];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint32_t i = i0 + (uint32_t)u * 32u + lane;
            const int      key  = (int)min(cur[u], (uint32_t)B);      // kNoBin16 -> B; also fences whatever the unchecked prefetch read behind the chunk
            const uint32_t sl   = (uint32_t)s_slot[key] - win0;                 // 0xFFFF (not scattered) and other windows: >= ns
            const bool     take = (i < s1) && (sl < ns);
            const unsigned tmask = __ballot_sync(FULL_MASK, take);
            if (take) {
                const unsigned peers = __match_any_sync(tmask, sl);
                if (lane == __ffs(peers) - 1) mine[sl] += __popc(peers);
            }
            __syncwarp();
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) cur[u] = nxt[u];
    }
}

// pass B of one window: re-walk the sub-range in order; mine[] holds the absolute destination of the next point per slot
template <bool NODE>
__device__ __forceinline__ void k2_scatter_pass(const uint16_t* __restrict__ ids, uint32_t s0, uint32_t s1, const uint16_t* __restrict__ s_slot,
                                                uint32_t win0, uint32_t ns, uint32_t* __restrict__ mine, int B, int lane,
                                                const float4* __restrict__ src, const float* __restrict__ s_T, uint32_t out_base, uint32_t local0,
                                                float4* __restrict__ out_pts, uint32_t* __restrict__ out_src, const uint32_t* __restrict__ lidx) {
    uint32_t cur[8], nxt[8];
    const uint16_t* __restrict__ pb = ids + (size_t)s0 + lane;      // one 64-bit base per block, constant offsets per load
#pragma unroll
    for (int u = 0; u < 8; ++u) cur[u] = pb[u * 32];
    for (uint32_t i0 = s0; i0 < s1; i0 += 256u, pb += 256) {
#pragma unroll
        for (int u = 0; u < 8; ++u) nxt[u] = pb[256 + u * 32];
        uint32_t dst[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint32_t i = i0 + (uint32_t)u * 32u + lane;
            const int      key  = (int)min(cur[u], (uint32_t)B);      // kNoBin16 -> B; also fences whatever the unchecked prefetch read behind the chunk
            const uint32_t sl   = (uint32_t)s_slot[key] - win0;
            const bool     take = (i < s1) && (sl < ns);
            const uint32_t base = take ? mine[sl] : 0u;
            const unsigned tmask = __ballot_sync(FULL_MASK, take);      // also orders the reads of mine[] before the updates below
            dst[u] = kSkip;
            if (take) {
                const unsigned peers = __match_any_sync(tmask, sl);
                if (lane == __ffs(peers) - 1) mine[sl] = base + __popc(peers);
                dst[u] = base + __popc(peers & ((1u << lane) - 1u));
            }
            __syncwarp();
        }
        // the copies of the block, four at a time: all loads of a group in flight before its first store
#pragma unroll
        for (int g = 0; g < 8; g += 4) {
            float4 pv[4];
            uint32_t si[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {                       // NODE: the chunk's list holds the map index of every entry
                si[u] = local0 + i0 + (uint32_t)(g + u) * 32u + lane;
                if (NODE && dst[g + u] != kSkip) si[u] = lidx[i0 + (uint32_t)(g + u) * 32u + lane];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (dst[g + u] != kSkip) pv[u] = NODE ? src[si[u]] : src[i0 + (uint32_t)(g + u) * 32u + lane];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (dst[g + u] != kSkip) {
                    const size_t o = (size_t)out_base + dst[g + u];
                    out_pts[o] = NODE ? affine12(s_T, pv[u]) : pv[u];
                    out_src[o] = si[u];
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) cur[u] = nxt[u];
    }
}

// DUAL (cloud mode): one launch scatters both clouds -- CTAs [0, second.first_row) take the map cloud's chunks with the
// arguments below, the rest the query cloud's with `second` (chunk rows are numbered map first, then query).
struct K2Second { uint32_t first_row; const uint16_t* bin_ids; const float4* pts; const uint32_t* dst_start; float4* out_pts; uint32_t* out_src; };

template <int W, bool NODE, bool DUAL>
__global__ void __launch_bounds__(W * 32, 4)      // 4 CTAs per SM: the chunking aims at one wave of sm_count * 4 CTAs
k2_scatter_win(const ChunkDesc* __restrict__ chunks, uint32_t chunk_base, const uint16_t* __restrict__ bin_ids,
               const float4* __restrict__ pts, const NodePose* __restrict__ poses, const uint32_t* __restrict__ ch_cnt,
               const uint32_t* __restrict__ dst_start /*[F][B+2] of this cloud*/, const uint32_t* __restrict__ flag_slot /*[F][B]; null: every bin + complement*/,
               const uint32_t* __restrict__ n_flagged /*[F]*/, float4* __restrict__ out_pts, uint32_t* __restrict__ out_src, int B, uint32_t SW,
               const uint32_t* __restrict__ list_idx, const uint32_t* __restrict__ list_cnt, int k1_warps, K2Second second) {
    extern __shared__ uint32_t s_tab[];   // [W][ns] per-warp counters / destinations | [SW] bases | u16 slot of every bin [B+1]
    __shared__ float s_T[12];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t row = chunk_base + blockIdx.x;
    if (DUAL && row >= second.first_row) {        // CTA-uniform
        bin_ids = second.bin_ids; pts = second.pts; dst_start = second.dst_start; out_pts = second.out_pts; out_src = second.out_src;
    }
    const ChunkDesc cd = chunks[row];
    const uint32_t* ds   = dst_start + (size_t)cd.frame * (B + 2);
    const uint32_t* pref = ch_cnt + (size_t)row * (B + 1);
    uint32_t* s_base = s_tab + (size_t)W * SW;
    uint16_t* s_slot = reinterpret_cast<uint16_t*>(s_base + SW);
    const uint32_t n_slots = flag_slot ? n_flagged[cd.frame] : (uint32_t)(B + 1);
    if (flag_slot) {
        const uint32_t* fs = flag_slot + (size_t)cd.frame * B;
        for (int b = tid; b <= B; b += W * 32) { const uint32_t v = (b < B) ? fs[b] : kSkip; s_slot[b] = (v == kSkip) ? (uint16_t)0xFFFFu : (uint16_t)v; }
    } else {
        for (int b = tid; b <= B; b += W * 32) s_slot[b] = (ds[b] == kSkip) ? (uint16_t)0xFFFFu : (uint16_t)b;   // (the query cloud's complement is not scattered)
    }
    if (NODE && tid < 12) s_T[tid] = poses[cd.frame].T[tid];
    // this warp's part of the chunk: a contiguous sub-range of its points -- or, in node mode, the dense VoI lists that
    // k1_warps / W of K1's warps left for their sub-ranges (same split, same order)
    const int      nseg = NODE ? k1_warps / W : 1;
    const uint32_t sub  = (((cd.len + (NODE ? k1_warps : W) - 1) / (NODE ? k1_warps : W)) + 31u) & ~31u;
    auto seg_range = [&](int g, uint32_t& s0, uint32_t& s1) {
        const uint32_t kw = (uint32_t)warp * nseg + g;
        s0 = min(cd.len, kw * sub);
        s1 = NODE ? s0 + list_cnt[(size_t)row * kListWarps + kw] : min(cd.len, s0 + sub);
    };
    const uint16_t* ids = bin_ids + cd.bin_begin;
    const uint32_t local0 = cd.begin - cd.frame_begin;
    const float4* src = NODE ? pts : pts + cd.begin;
    const uint32_t* lidx = NODE ? list_idx + cd.bin_begin : nullptr;

    for (uint32_t win0 = 0; win0 < n_slots; win0 += SW) {
        const uint32_t ns = min(SW, n_slots - win0);          // row stride of this window
        uint32_t* mine = s_tab + (size_t)warp * ns;
        __syncthreads();                                      // slot table ready / previous window's rows consumed
        for (uint32_t i = tid; i < (uint32_t)W * ns; i += W * 32) s_tab[i] = 0u;
        __syncthreads();
        for (int g = 0; g < nseg; ++g) { uint32_t s0, s1; seg_range(g, s0, s1); k2_count_pass(ids, s0, s1, s_slot, win0, ns, mine, B, lane); }
        // bases of the window's slots: dst_start + points of the bin in earlier chunks of the frame
        for (int b = tid; b <= B; b += W * 32) {
            const uint32_t sl = (uint32_t)s_slot[b] - win0;
            if (sl < ns) s_base[sl] = ds[b] + pref[b];
        }
        __syncthreads();
        for (uint32_t j = tid; j < ns; j += W * 32) {
            uint32_t run = s_base[j];
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const uint32_t c = s_tab[(size_t)w * ns + j];
                s_tab[(size_t)w * ns + j] = run;
                run += c;
            }
        }
        __syncthreads();
        for (int g = 0; g < nseg; ++g) {
            uint32_t s0, s1; seg_range(g, s0, s1);
            k2_scatter_pass<NODE>(ids, s0, s1, s_slot, win0, ns, mine, B, lane, src, s_T, cd.out_base, local0, out_pts, out_src, lidx);
        }
    }
}

// Mask modes: the Scan Ratio Test folded into the scatter (no k3_srt launch, no dependent round trip between them).
// Every CTA (one per map chunk) recomputes its frame's flagged set from K1's R-POD tables -- B cheap FP64 decisions, the
// tables sit in L2 -- numbers the flagged bins (slots, bin order), and per window of slots derives
//   destination = (points of earlier flagged bins of the frame) + (points of the bin in earlier chunks of the frame) + earlier warps.
// The first chunk of each frame is its LEADER: it also publishes n_flagged[frame] and the flagged-bin records + size
// buckets R-GPF consumes (what k3_srt does in cloud mode).
template <int W, bool NODE>
__global__ void __launch_bounds__(W * 32, 4)
k2_srt_scatter(SrtParams P, int F, const ChunkDesc* __restrict__ chunks, const uint32_t* __restrict__ chunk_range /*[2][F+1]*/,
               const uint16_t* __restrict__ bin_ids, const float4* __restrict__ pts, const NodePose* __restrict__ poses,
               const uint32_t* __restrict__ ch_cnt /*raw per-chunk counts*/, const uint32_t* __restrict__ zmin, const uint32_t* __restrict__ zmax,
               const uint32_t* __restrict__ cnt /*[2][F][B+1]*/, const uint32_t* __restrict__ frame_off /*[2][F+1]*/,
               uint32_t* __restrict__ n_flagged /*[F]*/, FlagRec* __restrict__ recs, uint32_t* __restrict__ n_recs, uint32_t rec_capacity,
               uint32_t* __restrict__ queue, uint32_t* __restrict__ bucket_list,
               float4* __restrict__ out_pts, uint32_t* __restrict__ out_src, uint32_t SW,
               const uint32_t* __restrict__ list_idx, const uint32_t* __restrict__ list_cnt, int k1_warps) {
    extern __shared__ uint32_t s_tab[];   // [W][ns] rows | [SW] bases | u16 slot of every bin [B+1]
    __shared__ float    s_T[12];
    __shared__ uint32_t s_part[34];
    __shared__ uint32_t s_bcast[2];
    constexpr int NT = W * 32;
    const int B = P.B;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t row = blockIdx.x;
    const ChunkDesc cd = chunks[row];
    const int f = (int)cd.frame;
    const uint32_t row0 = chunk_range[f];                    // first chunk of the frame's map cloud
    const bool leader = row == row0;
    uint32_t* s_base = s_tab + (size_t)W * SW;
    uint16_t* s_slot = reinterpret_cast<uint16_t*>(s_base + SW);
    const uint32_t* cm = cnt + ((size_t)0 * F + f) * (B + 1);
    const uint32_t* cq = cnt + ((size_t)1 * F + f) * (B + 1);
    const uint32_t* mnm = zmin + ((size_t)0 * F + f) * B; const uint32_t* mxm = zmax + ((size_t)0 * F + f) * B;
    const uint32_t* mnq = zmin + ((size_t)1 * F + f) * B; const uint32_t* mxq = zmax + ((size_t)1 * F + f) * B;

    // ---- Scan Ratio Test: flagged bit per bin (coalesced over the tables) ----
    for (int b = tid; b <= B; b += NT) {
        bool fl = false;
        if (b < B) {
            const uint32_t mc = cm[b], qc = cq[b];
            if (mc != 0u && qc != 0u) fl = srt_is_flagged(P, mc, qc, mxm[b], mnm[b], mxq[b], mnq[b]);
        }
        s_slot[b] = fl ? (uint16_t)0u : (uint16_t)0xFFFFu;
    }
    if (NODE && tid < 12) s_T[tid] = poses[f].T[tid];
    __syncthreads();
    // ---- slots: rank of every flagged bin, in bin order (each thread numbers a contiguous range of bins) ----
    const int seg = (B + NT - 1) / NT;
    const int b0 = min(B, tid * seg), b1 = min(B, b0 + seg);
    uint32_t mycnt = 0;
    for (int b = b0; b < b1; ++b) mycnt += (s_slot[b] == 0u) ? 1u : 0u;
    uint32_t incl = mycnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_part[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = lane < W ? s_part[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(FULL_MASK, wi, o); if (lane >= o) wi += v; }
        if (lane < W) s_part[lane] = wi - w;
        if (lane == 31) s_part[33] = wi;
    }
    __syncthreads();
    const uint32_t n_slots = s_part[33];
    {
        uint32_t run = s_part[warp] + incl - mycnt;
        for (int b = b0; b < b1; ++b) if (s_slot[b] == 0u) s_slot[b] = (uint16_t)(run++);
    }
    if (leader && tid == 0) {
        n_flagged[f] = n_slots;
        s_bcast[0] = n_slots ? atomicAdd(n_recs, n_slots) : 0u;
    }
    __syncthreads();
    const uint32_t rec_base = leader ? s_bcast[0] : 0u;

    // this warp's part of the chunk: a contiguous sub-range of its points -- or, in node mode, the dense VoI lists that
    // k1_warps / W of K1's warps left for their sub-ranges (same split, same order)
    const int      nseg = NODE ? k1_warps / W : 1;
    const uint32_t sub  = (((cd.len + (NODE ? k1_warps : W) - 1) / (NODE ? k1_warps : W)) + 31u) & ~31u;
    auto seg_range = [&](int g, uint32_t& s0, uint32_t& s1) {
        const uint32_t kw = (uint32_t)warp * nseg + g;
        s0 = min(cd.len, kw * sub);
        s1 = NODE ? s0 + list_cnt[(size_t)row * kListWarps + kw] : min(cd.len, s0 + sub);
    };
    const uint16_t* ids = bin_ids + cd.bin_begin;
    const uint32_t local0 = cd.begin - cd.frame_begin;
    const float4* src = NODE ? pts : pts + cd.begin;
    const uint32_t* lidx = NODE ? list_idx + cd.bin_begin : nullptr;
    const uint32_t fbase = frame_off[f];
    uint32_t win_carry = 0u;                                  // points of the flagged bins of earlier windows

    for (uint32_t win0 = 0; win0 < n_slots; win0 += SW) {
        const uint32_t ns = min(SW, n_slots - win0);
        uint32_t* mine = s_tab + (size_t)warp * ns;
        uint32_t* s_bin = s_tab;                              // [ns] bin of every slot of the window   (rows are not in use yet)
        uint32_t* s_pf  = s_tab + ns;                         // [ns] points of the bin in earlier chunks of the frame
        __syncthreads();
        for (int b = tid; b < B; b += NT) {
            const uint32_t sl = (uint32_t)s_slot[b] - win0;
            if (sl < ns) s_bin[sl] = (uint32_t)b;
        }
        __syncthreads();
        // sizes -> s_base, earlier-chunk prefixes -> s_pf
        for (uint32_t j = tid; j < ns; j += NT) {
            const uint32_t b = s_bin[j];
            s_base[j] = cm[b];
            uint32_t pf = 0u;
            for (uint32_t k0 = row0; k0 < row; k0 += 8u) {    // eight rows per round trip
                uint32_t v[8];
#pragma unroll
                for (uint32_t u = 0; u < 8u; ++u) v[u] = (k0 + u < row) ? ch_cnt[(size_t)(k0 + u) * (B + 1) + b] : 0u;
#pragma unroll
                for (uint32_t u = 0; u < 8u; ++u) pf += v[u];
            }
            s_pf[j] = pf;
        }
        __syncthreads();
        const uint32_t win_total = block_excl_scan(s_base, s_base, (int)ns, s_part);     // offsets of the window's bins inside the frame's region
        if (leader) {
            // flagged-bin records for K4 (slot order == bin order) and their size buckets
            for (uint32_t j = tid; j < ns; j += NT) {
                const uint32_t b = s_bin[j], slot = win0 + j, ri = rec_base + slot, sz = cm[b];
                if (ri < rec_capacity) {
                    FlagRec& rc = recs[ri];
                    rc.frame = (uint32_t)f; rc.bin = b; rc.slot = slot; rc.n_points = sz;
                    rc.src_begin = fbase + win_carry + s_base[j];
                    rc.n_seeds = 0; rc.n_empty_fits = 0; rc.n_ground_final = 0; rc.lpr_height = 0.0; rc.cursor = 0u; rc.n_rejected = 0u;
                    if (sz != 0u) {
                        const int bk = rgpf_bucket_of(sz);
                        bucket_list[(size_t)bk * rec_capacity + atomicAdd(&queue[bk], 1u)] = ri;
                    }
                }
            }
        }
        __syncthreads();
        // absolute base per slot, then the rows can be zeroed (s_bin / s_pf live in them)
        for (uint32_t j = tid; j < ns; j += NT) s_base[j] = win_carry + s_base[j] + s_pf[j];
        __syncthreads();
        for (uint32_t i = tid; i < (uint32_t)W * ns; i += NT) s_tab[i] = 0u;
        __syncthreads();
        for (int g = 0; g < nseg; ++g) { uint32_t s0, s1; seg_range(g, s0, s1); k2_count_pass(ids, s0, s1, s_slot, win0, ns, mine, B, lane); }
        __syncthreads();
        for (uint32_t j = tid; j < ns; j += NT) {
            uint32_t run = s_base[j];
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const uint32_t c = s_tab[(size_t)w * ns + j];
                s_tab[(size_t)w * ns + j] = run;
                run += c;
            }
        }
        __syncthreads();
        for (int g = 0; g < nseg; ++g) {
            uint32_t s0, s1; seg_range(g, s0, s1);
            k2_scatter_pass<NODE>(ids, s0, s1, s_slot, win0, ns, mine, B, lane, src, s_T, cd.out_base, local0, out_pts, out_src, lidx);
        }
        win_carry += win_total;
    }
}

static void k2_smem_plan(int B, bool with_complement, uint32_t& SW, size_t& smem) {
    constexpr int W = 8;
    const size_t fixed  = ((sizeof(uint16_t) * ((size_t)B + 2)) + 15) & ~(size_t)15;
    // one window over all slots while that leaves two CTAs per SM; beyond that (40 x 360 bins) the largest window that does:
    // mask mode rarely has more flagged bins per frame than it holds, cloud mode takes ceil((B + 1) / window) passes
    const uint32_t n_slots_max = with_complement ? (uint32_t)B + 1u : (uint32_t)B;
    const size_t full = sizeof(uint32_t) * (size_t)(W + 1) * n_slots_max + fixed;
    const size_t two_per_sm = 111 * 1024;                 // two CTAs per SM: (227 KB - static shared memory) / 2
    const size_t budget = full <= two_per_sm ? full : two_per_sm;      // 40 x 360: 2356-slot windows (config 5 flags ~2060 bins per frame)
    SW   = (uint32_t)std::min<size_t>(std::max<uint32_t>(n_slots_max, 1u), std::max<size_t>(1, (budget - fixed) / (sizeof(uint32_t) * (W + 1))));
    smem = sizeof(uint32_t) * (size_t)(W + 1) * SW + fixed;
}

cudaError_t launch_k2_srt(cudaStream_t st, const SrtParams& P, int F, const ChunkDesc* chunks, const uint32_t* chunk_range, uint32_t n_chunks_map,
                          const uint16_t* bin_ids, const float4* pts, const NodePose* poses, const uint32_t* ch_cnt, const uint32_t* zmin,
                          const uint32_t* zmax, const uint32_t* cnt, const uint32_t* frame_off, uint32_t* n_flagged, FlagRec* recs, uint32_t* n_recs,
                          uint32_t rec_capacity, uint32_t* queue, uint32_t* bucket_list, float4* out_pts, uint32_t* out_src,
                          const uint32_t* list_idx, const uint32_t* list_cnt) {
    if (n_chunks_map == 0) return cudaSuccess;
    constexpr int W = 8;
    const int k1_warps = k1_big_tables(P.R, P.B) ? 32 : 8;       // the split K1 compacted the chunk's VoI points in
    uint32_t SW; size_t smem;
    k2_smem_plan(P.B, false, SW, smem);
    cudaError_t e;
    if (poses) {
        auto kern = k2_srt_scatter<W, true>;
        if ((e = ensure_dyn_smem(kern, smem)) != cudaSuccess) return e;
        kern<<<n_chunks_map, W * 32, smem, st>>>(P, F, chunks, chunk_range, bin_ids, pts, poses, ch_cnt, zmin, zmax, cnt, frame_off, n_flagged, recs, n_recs,
                                                 rec_capacity, queue, bucket_list, out_pts, out_src, SW, list_idx, list_cnt, k1_warps);
    } else {
        auto kern = k2_srt_scatter<W, false>;
        if ((e = ensure_dyn_smem(kern, smem)) != cudaSuccess) return e;
        kern<<<n_chunks_map, W * 32, smem, st>>>(P, F, chunks, chunk_range, bin_ids, pts, nullptr, ch_cnt, zmin, zmax, cnt, frame_off, n_flagged, recs, n_recs,
                                                 rec_capacity, queue, bucket_list, out_pts, out_src, SW, list_idx, list_cnt, k1_warps);
    }
    return cudaGetLastError();
}

cudaError_t launch_k2(cudaStream_t st, const ChunkDesc* chunks, uint32_t chunk_base, uint32_t n_chunks,
                      const uint16_t* bin_ids, const float4* pts, const NodePose* poses, const uint32_t* ch_cnt, const uint32_t* dst_start,
                      const uint32_t* flag_slot, const uint32_t* n_flagged, float4* out_pts, uint32_t* out_src, int B,
                      const uint32_t* list_idx, const uint32_t* list_cnt, int k1_warps) {
    if (n_chunks == 0) return cudaSuccess;
    constexpr int W = 8;
    uint32_t SW; size_t smem;
    k2_smem_plan(B, flag_slot == nullptr, SW, smem);
    cudaError_t e;
    const K2Second none{0u, nullptr, nullptr, nullptr, nullptr, nullptr};
    if (poses) {
        auto kern = k2_scatter_win<W, true, false>;
        if ((e = ensure_dyn_smem(kern, smem)) != cudaSuccess) return e;
        kern<<<n_chunks, W * 32, smem, st>>>(chunks, chunk_base, bin_ids, pts, poses, ch_cnt, dst_start, flag_slot, n_flagged, out_pts, out_src, B, SW, list_idx, list_cnt, k1_warps, none);
    } else {
        auto kern = k2_scatter_win<W, false, false>;
        if ((e = ensure_dyn_smem(kern, smem)) != cudaSuccess) return e;
        kern<<<n_chunks, W * 32, smem, st>>>(chunks, chunk_base, bin_ids, pts, nullptr, ch_cnt, dst_start, flag_slot, n_flagged, out_pts, out_src, B, SW, nullptr, nullptr, W, none);
    }
    return cudaGetLastError();
}

// cloud mode: the map cloud's chunks (rows [0, n_chunks_map)) and the query cloud's (the n_chunks_qry rows behind them) in one launch
cudaError_t launch_k2_both(cudaStream_t st, const ChunkDesc* chunks, uint32_t n_chunks_map, uint32_t n_chunks_qry, const uint32_t* ch_cnt, int B,
                           const uint16_t* bin_map, const float4* map_pts, const uint32_t* dst_start_map, float4* out_map, uint32_t* src_map,
                           const uint16_t* bin_qry, const float4* qry_pts, const uint32_t* dst_start_qry, float4* out_qry, uint32_t* src_qry) {
    if (n_chunks_map + n_chunks_qry == 0) return cudaSuccess;
    constexpr int W = 8;
    uint32_t SW; size_t smem;
    k2_smem_plan(B, true, SW, smem);
    auto kern = k2_scatter_win<W, false, true>;
    cudaError_t e = ensure_dyn_smem(kern, smem);
    if (e != cudaSuccess) return e;
    const K2Second second{n_chunks_map, bin_qry, qry_pts, dst_start_qry, out_qry, src_qry};
    kern<<<n_chunks_map + n_chunks_qry, W * 32, smem, st>>>(chunks, 0u, bin_map, map_pts, nullptr, ch_cnt, dst_start_map, nullptr, nullptr, out_map, src_map, B, SW,
                                                             nullptr, nullptr, W, second);
    return cudaGetLastError();
}

// ============================================================================================
// K4  R-GPF
// ============================================================================================
// All float arithmetic below is spelled with round-to-nearest intrinsics so that nvcc cannot contract
// a*b+c into an FMA: the reference's x86-64 build (no -march, CMakeLists.txt:3-4) has none, and the
// unshifted covariance of PCL<=1.10 is so ill-conditioned that a single different rounding moves the plane.
#define FM(a, b) __fmul_rn((a), (b))
#define FA(a, b) __fadd_rn((a), (b))
#define FS(a, b) __fsub_rn((a), (b))
#define FD(a, b) __fdiv_rn((a), (b))
#define FSQ(a)   __fsqrt_rn((a))

struct Rot { float c, s; };

// internal::apply_rotation_in_the_plane on (x, y) pairs held in registers
#define ROT2(X_, Y_, J_)                                            \
    do {                                                            \
        const float xi__ = (X_), yi__ = (Y_);                       \
        (X_) = FA(FM((J_).c, xi__), FM((J_).s, yi__));              \
        (Y_) = FA(FM(-(J_).s, xi__), FM((J_).c, yi__));             \
    } while (0)

// Eigen 3.3 JacobiSVD<MatrixXf>(A, ComputeFullU) on a 3x3 (two-sided Jacobi, no preconditioner); returns U.col(2).
// Everything stays in registers: the (p,q) sweep is unrolled so that all matrix indices are compile-time.
__device__ __forceinline__ uint32_t jacobi_svd_normal(const float (&A)[9], float (&normal)[3]) {
    const float precision = 2.0f * FLT_EPSILON, considerAsZero = FLT_MIN;
    float W[9], U[9];
    float scale = 0.0f;
#pragma unroll
    for (int i = 0; i < 9; ++i) { const float a = fabsf(A[i]); scale = (a > scale) ? a : scale; }
    if (scale == 0.0f) scale = 1.0f;
#pragma unroll
    for (int i = 0; i < 9; ++i) W[i] = FD(A[i], scale);
#pragma unroll
    for (int i = 0; i < 9; ++i) U[i] = (i % 4 == 0) ? 1.0f : 0.0f;
    float maxDiag = 0.0f;
#pragma unroll
    for (int i = 0; i < 3; ++i) { const float a = fabsf(W[i * 4]); maxDiag = (a > maxDiag) ? a : maxDiag; }
    bool finished = false;
    int sweeps = 0;
    while (!finished && sweeps < 1000) {
        finished = true;
        ++sweeps;
#pragma unroll
        for (int p = 1; p < 3; ++p) {
#pragma unroll
            for (int q = 0; q < p; ++q) {
                const float pm = FM(precision, maxDiag);
                const float threshold = (considerAsZero < pm) ? pm : considerAsZero;     // std::max(considerAsZero, pm)
                if (fabsf(W[p * 3 + q]) > threshold || fabsf(W[q * 3 + p]) > threshold) {
                    finished = false;
                    // real_2x2_jacobi_svd
                    float m00 = W[p * 3 + p], m01 = W[p * 3 + q], m10 = W[q * 3 + p], m11 = W[q * 3 + q];
                    Rot rot1;
                    const float t = FA(m00, m11);
                    const float d = FS(m10, m01);
                    if (fabsf(d) < FLT_MIN) {
                        rot1.s = 0.0f; rot1.c = 1.0f;
                    } else {
                        const float u   = FD(t, d);
                        const float tmp = FSQ(FA(1.0f, FM(u, u)));
                        rot1.s = FD(1.0f, tmp);
                        rot1.c = FD(u, tmp);
                    }
                    if (!(rot1.c == 1.0f && rot1.s == 0.0f)) { ROT2(m00, m10, rot1); ROT2(m01, m11, rot1); }   // m.applyOnTheLeft(0,1,rot1)
                    Rot jr;
                    {   // makeJacobi(m00, m01, m11)
                        const float deno = FM(2.0f, fabsf(m01));
                        if (deno < FLT_MIN) {
                            jr.c = 1.0f; jr.s = 0.0f;
                        } else {
                            const float tau = FD(FS(m00, m11), deno);
                            const float w   = FSQ(FA(FM(tau, tau), 1.0f));
                            float tt;
                            if (tau > 0.0f) tt = FD(1.0f, FA(tau, w));
                            else            tt = FD(1.0f, FS(tau, w));
                            const float sign_t = tt > 0.0f ? 1.0f : -1.0f;
                            const float n = FD(1.0f, FSQ(FA(FM(tt, tt), 1.0f)));
                            jr.s = FM(FM(FM(-sign_t, FD(m01, fabsf(m01))), fabsf(tt)), n);
                            jr.c = n;
                        }
                    }
                    // j_left = rot1 * j_right.transpose()
                    const Rot jrt{jr.c, -jr.s};
                    const Rot jl{FS(FM(rot1.c, jrt.c), FM(rot1.s, jrt.s)), FA(FM(rot1.c, jrt.s), FM(rot1.s, jrt.c))};
                    if (!(jl.c == 1.0f && jl.s == 0.0f)) {
#pragma unroll
                        for (int i = 0; i < 3; ++i) ROT2(W[p * 3 + i], W[q * 3 + i], jl);      // W.applyOnTheLeft(p,q,j_left)
#pragma unroll
                        for (int i = 0; i < 3; ++i) ROT2(U[i * 3 + p], U[i * 3 + q], jl);      // U.applyOnTheRight(p,q,j_left.transpose())
                    }
                    if (!(jrt.c == 1.0f && jrt.s == 0.0f)) {
#pragma unroll
                        for (int i = 0; i < 3; ++i) ROT2(W[i * 3 + p], W[i * 3 + q], jrt);     // W.applyOnTheRight(p,q,j_right)
                    }
                    const float a = fabsf(W[p * 4]), b = fabsf(W[q * 4]);
                    const float ab = (a < b) ? b : a;
                    maxDiag = (maxDiag < ab) ? ab : maxDiag;
                }
            }
        }
    }
    float sv[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float a = W[i * 4];
        sv[i] = fabsf(a);
        if (a < 0.0f) { U[0 * 3 + i] = -U[0 * 3 + i]; U[1 * 3 + i] = -U[1 * 3 + i]; U[2 * 3 + i] = -U[2 * 3 + i]; }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) sv[i] = FM(sv[i], scale);
    // descending selection sort with "first maximum", stopping at the first zero remainder; only the column that
    // ends up at position 2 is needed, so track the column permutation in three scalars.
    int c0 = 0, c1 = 1, c2 = 2;
    {
        // i = 0: first maximum of sv[0..2]
        int pos = 0; float mx = sv[0];
        if (sv[1] > mx) { mx = sv[1]; pos = 1; }
        if (sv[2] > mx) { mx = sv[2]; pos = 2; }
        if (mx != 0.0f) {
            if (pos == 1) { const float t0 = sv[0]; sv[0] = sv[1]; sv[1] = t0; const int tc = c0; c0 = c1; c1 = tc; }
            if (pos == 2) { const float t0 = sv[0]; sv[0] = sv[2]; sv[2] = t0; const int tc = c0; c0 = c2; c2 = tc; }
            // i = 1: first maximum of sv[1..2]
            if (sv[2] > sv[1]) {
                if (sv[2] != 0.0f) { const float t1 = sv[1]; sv[1] = sv[2]; sv[2] = t1; const int tc = c1; c1 = c2; c2 = tc; }
            }
            // (if max(sv[1], sv[2]) == 0 the loop breaks without swapping: both are 0, so no swap happens above either)
        }
    }
    (void)c0; (void)c1;
    normal[0] = (c2 == 0) ? U[0] : (c2 == 1) ? U[1] : U[2];
    normal[1] = (c2 == 0) ? U[3] : (c2 == 1) ? U[4] : U[5];
    normal[2] = (c2 == 0) ? U[6] : (c2 == 1) ? U[7] : U[8];
    return (uint32_t)sweeps;
}

constexpr uint32_t K4_PAD = 0xFFFFFFFFu;

// A "group" is the set of threads that cooperates on one flagged bin: a whole CTA (G == blockDim.x) for large
// bins, one warp (G == 32) for small ones -- the plane fit is serial in one warp, so small bins are better served
// by many independent warps than by CTAs whose other warps wait at a barrier.
template <int G> __device__ __forceinline__ void group_sync() { if (G == 32) __syncwarp(); else __syncthreads(); }
template <int G> __device__ __forceinline__ int  group_tid() { return (G == 32) ? (threadIdx.x & 31) : threadIdx.x; }

// ordered compaction of indices i in [0,n) with pred(i) into out[]; returns count (all threads of the group).
template <int G, class Pred>
__device__ __forceinline__ uint32_t k4_compact(uint32_t n, uint32_t* out, uint32_t* s_warp /*[G/32 + 1], unused for G == 32*/, Pred pred) {
    const int tid = group_tid<G>(), lane = tid & 31, warp = tid >> 5;
    constexpr int NW = G / 32;
    uint32_t total = 0;
    for (uint32_t base = 0; base < n; base += G) {
        const uint32_t i = base + tid;
        const bool g = (i < n) && pred(i);
        const unsigned bal = __ballot_sync(FULL_MASK, g);
        if (G == 32) {
            if (g) out[total + __popc(bal & ((1u << lane) - 1u))] = i;
            total += __popc(bal);
            __syncwarp();
        } else {
            if (lane == 0) s_warp[warp] = __popc(bal);
            __syncthreads();
            uint32_t off = total, round = 0;
#pragma unroll
            for (int w = 0; w < NW; ++w) { const uint32_t c = s_warp[w]; off += (w < warp) ? c : 0u; round += c; }
            if (g) out[off + __popc(bal & ((1u << lane) - 1u))] = i;
            total += round;
            __syncthreads();
        }
    }
    return total;
}

// exclusive scan of 8*G counters by the group (8 per thread); s_part: G/32 + 2 words of scratch
template <int G>
__device__ __forceinline__ void group_excl_scan8(uint32_t* CNT, uint32_t* s_part) {
    const int tid = group_tid<G>(), lane = tid & 31, warp = tid >> 5;
    constexpr int NW = G / 32;
    uint32_t v[8], sum = 0;
#pragma unroll
    for (int u = 0; u < 8; ++u) { v[u] = CNT[tid * 8 + u]; sum += v[u]; }
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL_MASK, incl, o);
        if (lane >= o) incl += t;
    }
    uint32_t excl = incl - sum;
    if (G != 32) {
        if (lane == 31) s_part[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const uint32_t w = lane < NW ? s_part[lane] : 0u;
            uint32_t wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(FULL_MASK, wi, o);
                if (lane >= o) wi += t;
            }
            if (lane < NW) s_part[lane] = wi - w;
        }
        __syncthreads();
        excl += s_part[warp];
    }
    uint32_t run = excl;
#pragma unroll
    for (int u = 0; u < 8; ++u) { CNT[tid * 8 + u] = run; run += v[u]; }
    group_sync<G>();
}

// Stable LSD radix sort (8-bit digits) of the n values in A by key(value); Bf is an n-word ping-pong buffer,
// CNT 8*G counters laid out [digit][warp].  Each warp owns a contiguous segment of the input: it histograms the
// segment (match_any dedups equal digits inside a 32-element step, so no atomics), and after the group-wide scan
// re-walks the segment in order handing out destinations -- which is what makes the sort stable.  Returns the
// buffer (A or Bf) that holds the result.  ~35 warp instructions per 32 elements per pass: about 8x fewer than
// the shared-memory bitonic network this replaced (profiles/README.md, R-GPF section).
template <int G, class KeyF>
__device__ __forceinline__ uint32_t* group_radix_sort(uint32_t* A, uint32_t* Bf, uint32_t n, uint32_t* CNT, uint32_t* s_part,
                                                      int key_bits, KeyF key) {
    constexpr int NW = G / 32;
    const int tid = group_tid<G>(), lane = tid & 31, warp = tid >> 5;
    const uint32_t seg = (((n + NW - 1) / NW) + 31u) & ~31u;
    const uint32_t s0 = min(n, (uint32_t)warp * seg), s1 = min(n, s0 + seg);
    uint32_t* src = A;
    uint32_t* dst = Bf;
    for (int shift = 0; shift < key_bits; shift += 8) {
#pragma unroll
        for (int u = 0; u < 8; ++u) CNT[tid + u * G] = 0u;
        group_sync<G>();
        for (uint32_t e0 = s0; e0 < s1; e0 += 32) {
            const uint32_t e = e0 + lane;
            const bool valid = e < s1;
            const unsigned vmask = __ballot_sync(FULL_MASK, valid);
            if (valid) {
                const uint32_t d = (key(src[e]) >> shift) & 255u;
                const unsigned peers = __match_any_sync(vmask, d);
                if (lane == __ffs(peers) - 1) CNT[d * NW + warp] += __popc(peers);
            }
            __syncwarp();
        }
        group_sync<G>();
        group_excl_scan8<G>(CNT, s_part);
        for (uint32_t e0 = s0; e0 < s1; e0 += 32) {
            const uint32_t e = e0 + lane;
            const bool valid = e < s1;
            const unsigned vmask = __ballot_sync(FULL_MASK, valid);
            if (valid) {
                const uint32_t id = src[e];
                const uint32_t d  = (key(id) >> shift) & 255u;
                const unsigned peers = __match_any_sync(vmask, d);
                const uint32_t base  = CNT[d * NW + warp];
                __syncwarp(vmask);
                if (lane == __ffs(peers) - 1) CNT[d * NW + warp] = base + __popc(peers);
                dst[base + __popc(peers & ((1u << lane) - 1u))] = id;
            }
            __syncwarp();
        }
        group_sync<G>();
        uint32_t* t = src; src = dst; dst = t;
    }
    return src;
}

// order-preserving 32-bit encoding of z for the R-GPF sort (-0.0 folded onto +0.0: a.z < b.z treats them as equal)
__device__ __forceinline__ uint32_t z_sort_key(float z) {
    uint32_t u = __float_as_uint(z);
    if (u == 0x80000000u) u = 0u;
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// Bitonic sorting network over NW*32*E 64-bit values held in registers, position p = gtid*E + r (gtid = thread of the
// group).  Stages with j < E are compare-exchanges between registers of one thread, stages with E <= j < 32E go
// through shuffles, and (NW > 1) stages with j >= 32E exchange through shared memory, half of the registers at a
// time so that the exchange buffer (32*NW*E/2 values) fits in the bin's 8n-byte order area.  Register indices are
// compile-time constants throughout (the per-warp network is straight-line code; only the cross-warp levels loop).
// Values are (z key << 32 | source index): distinct, so the unstable network yields the stable order std::sort by z
// would give with ties in source order (sort_mode 1).
// compare-exchange as min / max with a selectable direction (IMNMX with a predicate operand for 32-bit values)
#define K4_CMPX(a_, b_, asc_) do { const auto lo__ = min((a_), (b_)); const auto hi__ = max((a_), (b_)); \
                                   (a_) = (asc_) ? lo__ : hi__; (b_) = (asc_) ? hi__ : lo__; } while (0)

// stages j = E/2 .. 1 inside the thread, block direction asc
template <int E, class T>
__device__ __forceinline__ void bitonic_lane_stages(T (&v)[E], bool asc) {
#pragma unroll
    for (int j = E >> 1; j > 0; j >>= 1) {
#pragma unroll
        for (int r = 0; r < E; ++r) {
            if ((r & j) == 0) K4_CMPX(v[r], v[r | j], asc);
        }
    }
}
// stages j = DMAX*E .. E across lanes (d = j / E), block direction asc
template <int E, int DMAX, class T>
__device__ __forceinline__ void bitonic_shfl_stages(T (&v)[E], int lane, bool asc) {
#pragma unroll
    for (int d = DMAX; d > 0; d >>= 1) {
        const bool keep_min = ((lane & d) == 0) == asc;
#pragma unroll
        for (int r = 0; r < E; ++r) {
            const T o = __shfl_xor_sync(FULL_MASK, v[r], d);
            v[r] = keep_min ? min(v[r], o) : max(v[r], o);
        }
    }
}
// full sort of the warp's 32E positions; the top-level direction is asc_top, lower levels follow the network
template <int E, class T>
__device__ __forceinline__ void bitonic_warp_sort(T (&v)[E], int lane, bool asc_top) {
    // k < E: inside the thread, direction from the register index
#pragma unroll
    for (int k = 2; k < E; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int r = 0; r < E; ++r) {
                if ((r & j) == 0) K4_CMPX(v[r], v[r | j], (r & k) == 0);
            }
        }
    }
    // k = E .. 32E: direction from the lane (top level: asc_top)
    bitonic_lane_stages<E>(v, (lane & 1) == 0);                                                     // k = E
    bitonic_shfl_stages<E, 1>(v, lane, (lane & 2) == 0);  bitonic_lane_stages<E>(v, (lane & 2) == 0);    // k = 2E
    bitonic_shfl_stages<E, 2>(v, lane, (lane & 4) == 0);  bitonic_lane_stages<E>(v, (lane & 4) == 0);    // k = 4E
    bitonic_shfl_stages<E, 4>(v, lane, (lane & 8) == 0);  bitonic_lane_stages<E>(v, (lane & 8) == 0);    // k = 8E
    bitonic_shfl_stages<E, 8>(v, lane, (lane & 16) == 0); bitonic_lane_stages<E>(v, (lane & 16) == 0);   // k = 16E
    bitonic_shfl_stages<E, 16>(v, lane, asc_top);         bitonic_lane_stages<E>(v, asc_top);            // k = 32E
}
// the whole group's network: per-warp sort, then (NW > 1) the cross-warp levels through xbuf (32*NW*E/2 values of T)
template <int E, int NW, class T>
__device__ __forceinline__ void bitonic_group_sort(T (&v)[E], T* xbuf) {
    const int gtid = (NW == 1) ? (threadIdx.x & 31) : threadIdx.x;
    const int lane = gtid & 31, warp = gtid >> 5;
    bitonic_warp_sort<E>(v, lane, (NW == 1) ? true : ((warp & 1) == 0));
    if (NW > 1) {
        constexpr int H = E / 2;
#pragma unroll 1
        for (int lvl = 2; lvl <= NW; lvl <<= 1) {            // k = 32E * lvl; block direction of the level: warp bit `lvl`
            const bool asc = (warp & lvl) == 0;              // (lvl == NW: always ascending)
#pragma unroll 1
            for (int dw = lvl >> 1; dw > 0; dw >>= 1) {      // stages j = 32E * dw: partner warp = warp ^ dw
                const bool keep_min = ((warp & dw) == 0) == asc;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
#pragma unroll
                    for (int r = 0; r < H; ++r) xbuf[(warp * H + r) * 32 + lane] = v[h * H + r];
                    __syncthreads();
#pragma unroll
                    for (int r = 0; r < H; ++r) {
                        const T o = xbuf[((warp ^ dw) * H + r) * 32 + lane];
                        v[h * H + r] = keep_min ? min(v[h * H + r], o) : max(v[h * H + r], o);
                    }
                    __syncthreads();
                }
            }
            bitonic_shfl_stages<E, 16>(v, lane, asc);
            bitonic_lane_stages<E>(v, asc);
        }
    }
}

// z-sort, exact 64-bit version: values (z key << 32 | source index).  ORD[0..n) <- source indices in (z, index) order.
// Requires n <= NW*32*E.  For NW > 1, ORD must start an 8-byte aligned area of at least 8n bytes (the exchange buffer).
// Not inlined: one copy of each network serves the shared-memory and the global-scratch variants of the caller.
template <int E, int NW>
__device__ __noinline__ void group_bitonic_zsort(const float* Z, uint32_t* ORD, uint32_t n) {
    constexpr int G = NW * 32;
    const int gtid = (NW == 1) ? (threadIdx.x & 31) : threadIdx.x;
    unsigned long long v[E];
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const uint32_t e = (uint32_t)r * G + gtid;       // any placement works: the network sorts positions, ties carry the index
        v[r] = (e < n) ? (((unsigned long long)z_sort_key(Z[e]) << 32) | e) : ~0ull;
    }
    bitonic_group_sort<E, NW>(v, reinterpret_cast<unsigned long long*>(ORD));
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const uint32_t pos = (uint32_t)gtid * E + r;
        if (pos < n) ORD[pos] = (uint32_t)v[r];
    }
    if (NW == 1) __syncwarp(); else __syncthreads();
}

// z-sort, packed 32-bit version (4x fewer instructions than the 64-bit network).  Each point becomes one word
//   (q << IB) | source index,   q = min(uint((z - zmin) * QMAX / (zmax - zmin)), QMAX)   (23 bits for a warp, 20 for a CTA):
// q is monotone in z, so after sorting the words the order is exact except inside runs of equal q, which are still in
// source-index order.  Those runs are short (q resolves the bin's z range to 2^-23 / 2^-20, about one float ulp) and
// are finished by an odd-even transposition on the full (z key, index) pairs, restricted to the listed positions p
// with q[p] == q[p+1].  More than list_cap such positions: returns false and the caller runs the 64-bit network.
// s_red: 2*NW + 2 words of scratch (CTA groups).
template <int E, int NW>
__device__ __noinline__ bool group_packed_zsort(const float* Z, uint32_t* ORD, uint32_t n, uint32_t* list, uint32_t list_cap, uint32_t* s_red) {
    constexpr int G  = NW * 32;
    constexpr int IB = (NW == 1) ? 9 : 12;
    constexpr uint32_t QMAX = (1u << (32 - IB)) - 1u, IMASK = (1u << IB) - 1u;
    const int gtid = (NW == 1) ? (threadIdx.x & 31) : threadIdx.x;
    const int lane = gtid & 31, warp = gtid >> 5;
    float z[E];
    float mn = __int_as_float(0x7f800000), mx = __int_as_float(0xff800000);
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const uint32_t e = (uint32_t)r * G + gtid;
        z[r] = (e < n) ? Z[e] : 0.0f;
        if (e < n) { mn = fminf(mn, z[r]); mx = fmaxf(mx, z[r]); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { mn = fminf(mn, __shfl_xor_sync(FULL_MASK, mn, o)); mx = fmaxf(mx, __shfl_xor_sync(FULL_MASK, mx, o)); }
    if (NW > 1) {
        if (lane == 0) { s_red[warp] = __float_as_uint(mn); s_red[NW + warp] = __float_as_uint(mx); }
        if (gtid == 0) s_red[2 * NW] = 0u;
        __syncthreads();
#pragma unroll
        for (int w = 0; w < NW; ++w) { mn = fminf(mn, __uint_as_float(s_red[w])); mx = fmaxf(mx, __uint_as_float(s_red[NW + w])); }
    }
    const float D = __fsub_rn(mx, mn);
    float scale = (D > 0.0f) ? __fdiv_rn((float)QMAX, D) : 0.0f;
    if (!(scale <= 3.0e38f)) scale = 0.0f;
    auto q_of = [&](float zz) -> uint32_t { return min(__float2uint_rz(__fmul_rn(__fsub_rn(zz, mn), scale)), QMAX); };
    uint32_t v[E];
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const uint32_t e = (uint32_t)r * G + gtid;
        v[r] = (e < n) ? ((q_of(z[r]) << IB) | e) : 0xFFFFFFFFu;      // a pad equals a real word only when no pad exists (n == 32*NW*E)
    }
    bitonic_group_sort<E, NW>(v, ORD);
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const uint32_t pos = (uint32_t)gtid * E + r;
        if (pos < n) ORD[pos] = v[r] & IMASK;
    }
    if (NW == 1) __syncwarp(); else __syncthreads();
    // positions whose successor shares q
    uint32_t cnt = 0;
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const uint32_t pos = (uint32_t)gtid * E + r;
        bool same = false;
        if (pos + 1u < n) {
            const uint32_t qn = (r + 1 < E) ? (v[(r + 1 < E) ? r + 1 : r] >> IB) : q_of(Z[ORD[pos + 1u]]);
            same = (v[r] >> IB) == qn;
        }
        if (NW == 1) {
            const unsigned bal = __ballot_sync(FULL_MASK, same);
            if (same) { const uint32_t s = cnt + __popc(bal & ((1u << lane) - 1u)); if (s < list_cap) list[s] = pos; }
            cnt += __popc(bal);
        } else if (same) {
            const uint32_t s = atomicAdd(&s_red[2 * NW], 1u);
            if (s < list_cap) list[s] = pos;
        }
    }
    if (NW == 1) __syncwarp(); else { __syncthreads(); cnt = s_red[2 * NW]; }
    if (cnt > list_cap) return false;
    if (cnt == 0u) return true;
    for (;;) {
        bool swapped = false;
#pragma unroll 1
        for (uint32_t phase = 0; phase < 2u; ++phase) {
            for (uint32_t t = gtid; t < cnt; t += G) {
                const uint32_t pp = list[t];
                if ((pp & 1u) == phase) {
                    const uint32_t ia = ORD[pp], ib = ORD[pp + 1u];
                    const uint32_t ka = z_sort_key(Z[ia]), kb = z_sort_key(Z[ib]);
                    if (ka > kb || (ka == kb && ia > ib)) { ORD[pp] = ib; ORD[pp + 1u] = ia; swapped = true; }
                }
            }
            if (NW == 1) __syncwarp(); else __syncthreads();
        }
        const bool any = (NW == 1) ? (__any_sync(FULL_MASK, swapped) != 0) : (__syncthreads_or(swapped ? 1 : 0) != 0);
        if (!any) break;
    }
    return true;
}

struct K4Shared {
    float    normal[3];
    uint32_t pad_;
    double   thd;
    double   seed_thr;
    uint32_t warp[34];
};

// One flagged bin, handled by one group.  X/Y/Z/ORD/FLG live in shared memory or in the bin's slice of the global scratch.
template <int G, bool kShared>
__device__ __forceinline__ void k4_process_bin(const GpfParams& P, FlagRec& rc, unsigned char* base, float* prd, uint32_t* cnt_scratch, K4Shared& sh,
                                               const float4* __restrict__ sorted_pts, uint32_t* __restrict__ sorted_src,
                                               const float4* __restrict__ in_pts, const uint32_t* __restrict__ frame_off,
                                               float4* __restrict__ part_pts, uint8_t* __restrict__ keep_mask,
                                               uint8_t* __restrict__ ground_mask, uint32_t* __restrict__ frame_rejected,
                                               unsigned long long* __restrict__ fence, const K4Fold& fold) {
    const int tid = group_tid<G>(), lane = tid & 31, warp = tid >> 5;
    const uint32_t n = rc.n_points, src_begin = rc.src_begin;
    const uint32_t fbase = frame_off[rc.frame];
    // slice layout: [ORD n u32][TMP n u32 (CTA groups only)][X][Y][Z n f32 each][FLG n u8]; ORD|TMP is also the 8n-byte
    // exchange area of the class-B sort, hence first (the slice base is 16-byte aligned)
    uint32_t* ORD = reinterpret_cast<uint32_t*>(base);
    uint32_t* TMP = ORD + n;
    float*    X   = reinterpret_cast<float*>((G == 32) ? TMP : TMP + n);
    float*    Y   = X + n;
    float*    Z   = Y + n;
    uint8_t*  FLG = reinterpret_cast<uint8_t*>(Z + n);
    constexpr int HT = (G == 32) ? 32 : (G == 128 ? 96 : 128);      // half tile of the covariance accumulation (CTA groups: the threads beyond warp 0 stage it)
    constexpr int PB = 9 * (HT + 1);
    float*    PRD = prd;                          // two buffers of 9 x (HT + 1) floats, always shared memory
    long long t_prev = clock64();
    uint32_t prof[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define K4_TICK(slot) do { const long long t_now__ = clock64(); prof[slot] += (uint32_t)(t_now__ - t_prev); t_prev = t_now__; } while (0)

    // K2 placed the bin's points contiguously in source order (all bins in cloud mode, flagged bins only in mask mode)
    for (uint32_t i0 = tid; i0 < n; i0 += 4u * G) {
        float4 p[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {                      // four independent loads in flight per thread
            const uint32_t i = i0 + (uint32_t)u * G;
            if (i < n) p[u] = sorted_pts[src_begin + i];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t i = i0 + (uint32_t)u * G;
            if (i < n) {
                X[i] = p[u].x; Y[i] = p[u].y; Z[i] = p[u].z;
                if (G > 256 || (G == 128 && n > 2048u)) ORD[i] = i;      // the radix sort permutes an index list
            }
        }
    }
    group_sync<G>();
    K4_TICK(0);

    // std::sort by z (erasor.cpp:240), ties in source order: stable radix sort on the order-preserving encoding of z
    // (-0.0 is folded onto +0.0 first: the comparator a.z < b.z treats them as equal)
    if constexpr (G == 32) {
        // class A (n <= 512): the warp sorts in registers; the collision list lives in the (still unused) product tile
        uint32_t* lst = reinterpret_cast<uint32_t*>(PRD);
        if (n <= 128u)      { if (!group_packed_zsort<4, 1>(Z, ORD, n, lst, 256u, sh.warp))  group_bitonic_zsort<4, 1>(Z, ORD, n); }
        else if (n <= 256u) { if (!group_packed_zsort<8, 1>(Z, ORD, n, lst, 256u, sh.warp))  group_bitonic_zsort<8, 1>(Z, ORD, n); }
        else                { if (!group_packed_zsort<16, 1>(Z, ORD, n, lst, 256u, sh.warp)) group_bitonic_zsort<16, 1>(Z, ORD, n); }
    } else if constexpr (G == 128) {
        // class B (512 < n <= 2560): four warps -- half the registers per bin of the eight-warp form (a bin keeps them for its
        // whole serial chain, and registers are what limits how many chains of overlapped submissions an SM holds); cross-warp
        // stages through the ORD|TMP area; the few bins beyond 16 keys per lane take the radix sort
        uint32_t* lst = reinterpret_cast<uint32_t*>(PRD);
        if (n <= 512u)       { if (!group_packed_zsort<4, 4>(Z, ORD, n, lst, 1024u, sh.warp))  group_bitonic_zsort<4, 4>(Z, ORD, n); }
        else if (n <= 1024u) { if (!group_packed_zsort<8, 4>(Z, ORD, n, lst, 1024u, sh.warp))  group_bitonic_zsort<8, 4>(Z, ORD, n); }
        else if (n <= 2048u) { if (!group_packed_zsort<16, 4>(Z, ORD, n, lst, 1024u, sh.warp)) group_bitonic_zsort<16, 4>(Z, ORD, n); }
        else {
            uint32_t* zs = group_radix_sort<G>(ORD, TMP, n, cnt_scratch, sh.warp, 32, [&](uint32_t id) { return z_sort_key(Z[id]); });
            if (zs != ORD) { TMP = ORD; ORD = zs; }
        }
    } else {
        uint32_t* zs = group_radix_sort<G>(ORD, TMP, n, cnt_scratch, sh.warp, 32, [&](uint32_t id) { return z_sort_key(Z[id]); });
        if (zs != ORD) { TMP = ORD; ORD = zs; }
    }
    K4_TICK(1);

    // extract_initial_seeds_ (erasor.cpp:204-231)
    if (tid == 0) {
        double sum = 0.0;
        int    cnt = 0;
        if (P.num_lowest_pts >= 0) {
            for (uint32_t i = (uint32_t)P.num_lowest_pts; i < n && cnt < P.num_lpr; ++i) { sum += (double)Z[ORD[i]]; ++cnt; }
        }
        const double lpr = cnt != 0 ? sum / cnt : 0.0;
        rc.lpr_height = lpr;
        sh.seed_thr   = lpr + P.th_seeds;
    }
    group_sync<G>();
    const double seed_thr = sh.seed_thr;
    uint32_t m;   // seeds = sorted prefix with z < lpr + th_seeds
    {
        uint32_t c = 0;
        for (uint32_t i = tid; i < n; i += G) c += ((double)Z[ORD[i]] < seed_thr) ? 1u : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL_MASK, c, o);
        if (G == 32) {
            m = c;
        } else {
            if (lane == 0) sh.warp[warp] = c;
            __syncthreads();
            m = 0;
#pragma unroll
            for (int ww = 0; ww < G / 32; ++ww) m += sh.warp[ww];
            __syncthreads();
        }
    }
    if (tid == 0) rc.n_seeds = m;
    K4_TICK(2);

    uint32_t n_empty = 0;
    for (int it = 0; it < P.iters; ++it) {
        // ---- estimate_plane_ over ORD[0..m) (erasor.cpp:183-198) ----
        // pcl::computeMeanAndCovarianceMatrix: nine float accumulators walked in list order.  The nine products of a
        // half tile of list elements are staged in shared memory (row stride HT+1: conflict-free for the nine summing
        // lanes), then lane L of warp 0 adds row L in order: the serial FADD chain is fed by independent, prefetchable
        // shared-memory loads (4-5 cycles per element instead of a dependent gather).
        float K0 = 0.0f, K1 = 0.0f, K2 = 0.0f;
        if (P.cov_mode == 1 && m > 0) { const uint32_t f0 = ORD[0]; K0 = X[f0]; K1 = Y[f0]; K2 = Z[f0]; }
        float acc = 0.0f;
        if (m > 0) {
            // PRD holds two buffers of 9 x (HT + 1): while the nine lanes add the rows of one buffer in order, the next
            // HT list elements are staged into the other.  A warp group does both in one instruction stream (the staging
            // loads are in flight under the serial FADD chain; every lane runs the chain, lanes >= 9 on a copy of row 8,
            // so that there is no branch between the two); in a CTA group warp 0 adds and the next 128 threads stage.
            auto stage_prod = [&](float x, float y, float z, float* buf, uint32_t k) {
                x = FS(x, K0); y = FS(y, K1); z = FS(z, K2);
                buf[0 * (HT + 1) + k] = FM(x, x);
                buf[1 * (HT + 1) + k] = FM(x, y);
                buf[2 * (HT + 1) + k] = FM(x, z);
                buf[3 * (HT + 1) + k] = FM(y, y);
                buf[4 * (HT + 1) + k] = FM(y, z);
                buf[5 * (HT + 1) + k] = FM(z, z);
                buf[6 * (HT + 1) + k] = x;
                buf[7 * (HT + 1) + k] = y;
                buf[8 * (HT + 1) + k] = z;
            };
            auto chain = [&](const float* buf, uint32_t cntk) {
                const float* row = buf + min(lane, 8) * (HT + 1);
                if (cntk == (uint32_t)HT) {
#pragma unroll
                    for (int k = 0; k < HT; k += 16) {
                        float q[16];
#pragma unroll
                        for (int u = 0; u < 16; ++u) q[u] = row[k + u];
#pragma unroll
                        for (int u = 0; u < 16; ++u) acc = FA(acc, q[u]);
                    }
                } else {
                    for (uint32_t k = 0; k < cntk; k += 16u) {
                        float q[16];
#pragma unroll
                        for (uint32_t u = 0; u < 16u; ++u) q[u] = row[min(k + u, (uint32_t)HT)];
#pragma unroll
                        for (uint32_t u = 0; u < 16u; ++u) { if (k + u < cntk) acc = FA(acc, q[u]); }
                    }
                }
            };
            {   // prologue: list elements [0, HT) -> buffer 0
                const uint32_t k = (G == 32) ? (uint32_t)lane : (uint32_t)tid;
                if (k < (uint32_t)HT) { const uint32_t idx = ORD[min(k, m - 1u)]; stage_prod(X[idx], Y[idx], Z[idx], PRD, k); }
            }
            group_sync<G>();
            uint32_t t = 0;
            for (uint32_t base_i = 0; base_i < m; base_i += HT, ++t) {
                float* cur = PRD + (t & 1u) * PB;
                float* nxt = PRD + ((t & 1u) ^ 1u) * PB;
                const uint32_t cntk = min((uint32_t)HT, m - base_i);
                const bool more = base_i + HT < m;                      // group-uniform
                if (G == 32) {
                    float sx = 0.0f, sy = 0.0f, sz = 0.0f;
                    if (more) { const uint32_t idx = ORD[min(base_i + HT + lane, m - 1u)]; sx = X[idx]; sy = Y[idx]; sz = Z[idx]; }
                    chain(cur, cntk);
                    if (more) stage_prod(sx, sy, sz, nxt, (uint32_t)lane);
                    __syncwarp();
                } else {
                    if (warp == 0) {
                        chain(cur, cntk);
                    } else if (more && tid - 32 < HT) {
                        const uint32_t k = (uint32_t)tid - 32u;
                        const uint32_t idx = ORD[min(base_i + HT + k, m - 1u)];
                        stage_prod(X[idx], Y[idx], Z[idx], nxt, k);
                    }
                    __syncthreads();
                }
            }
        }
        if (warp == 0) {
            if (lane < 9 && m != 0) acc = FD(acc, (float)m);
            K4_TICK(3);
            float a[9];
#pragma unroll
            for (int k = 0; k < 9; ++k) a[k] = __shfl_sync(FULL_MASK, acc, k);
            if (lane == 0) {
                float cov[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, mean[3] = {0, 0, 0};
                if (m != 0) {
                    mean[0] = (P.cov_mode == 1) ? FA(a[6], K0) : a[6];
                    mean[1] = (P.cov_mode == 1) ? FA(a[7], K1) : a[7];
                    mean[2] = (P.cov_mode == 1) ? FA(a[8], K2) : a[8];
                    cov[0] = FS(a[0], FM(a[6], a[6]));
                    cov[1] = FS(a[1], FM(a[6], a[7]));
                    cov[2] = FS(a[2], FM(a[6], a[8]));
                    cov[4] = FS(a[3], FM(a[7], a[7]));
                    cov[5] = FS(a[4], FM(a[7], a[8]));
                    cov[8] = FS(a[5], FM(a[8], a[8]));
                    cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
                }
                float nrm[3];
                prof[7] += jacobi_svd_normal(cov, nrm);
                const float dot = FA(FA(FM(nrm[0], mean[0]), FM(nrm[1], mean[1])), FM(nrm[2], mean[2]));
                const double d  = (double)(-dot);
                sh.normal[0] = nrm[0]; sh.normal[1] = nrm[1]; sh.normal[2] = nrm[2];
                sh.thd = P.th_dist - d;
                if (it < kMaxIter) {
                    rc.normal_d[it][0] = nrm[0]; rc.normal_d[it][1] = nrm[1]; rc.normal_d[it][2] = nrm[2]; rc.normal_d[it][3] = d;
                }
            }
        }
        if (m == 0) ++n_empty;
        group_sync<G>();
        K4_TICK(4);
        const float n0 = sh.normal[0], n1 = sh.normal[1], n2 = sh.normal[2];
        const double thd = sh.thd;
        // ---- classify every point of the bin in source order (erasor.cpp:265-281) ----
        // (classification fused into the stable compaction: one pass over the bin instead of two)
        m = k4_compact<G>(n, ORD, sh.warp, [&](uint32_t i) {
            const float r = FA(FA(FM(X[i], n0), FM(Y[i], n1)), FM(Z[i], n2));
            const bool  g = (double)r < thd;
            FLG[i] = g ? 1 : 0;
            return g;
        });
        if (tid == 0 && it < kMaxIter) rc.n_ground[it] = m;
        K4_TICK(5);
    }
    // gf_iter == 0: the reference returns the seeds as ground and fills no outliers (erasor.cpp:260-285)
    if (P.iters <= 0) {
        for (uint32_t i = tid; i < n; i += G) FLG[i] = 0;
        group_sync<G>();
        for (uint32_t i = tid; i < m; i += G) FLG[ORD[i]] = 1;
        group_sync<G>();
    }
    if (tid == 0) {
        rc.n_ground_final = m; rc.n_empty_fits = n_empty; rc.n_rejected = (P.iters > 0) ? n - m : 0u;
        if (n_empty) atomicAdd(&fence[1], (unsigned long long)n_empty);
        if (frame_rejected) atomicAdd(&frame_rejected[rc.frame], n - m);
    }

    // ---- outputs ----
    if (keep_mask || ground_mask || fold.keep) {
        for (uint32_t i0 = tid; i0 < n; i0 += 4u * G) {
            uint32_t s[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {                  // four independent index loads in flight per thread
                const uint32_t i = i0 + (uint32_t)u * G;
                s[u] = (i < n) ? sorted_src[src_begin + i] : 0u;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t i = i0 + (uint32_t)u * G;
                if (i < n) {
                    if (keep_mask && !FLG[i]) keep_mask[fbase + s[u]] = 0;      // not in the selected bin any more (gf_iter == 0: dropped silently)
                    if (ground_mask && FLG[i]) ground_mask[fbase + s[u]] = 1;
                    if (fold.keep && !FLG[i]) {
                        // the multi-GPU fold, in the epilogue: a global map point survives unless some frame rejected it.
                        // Only zeros are ever written, so concurrent bins / frames / handles need no atomics.
                        const uint32_t g = fold.index ? fold.index[fbase + s[u]] : s[u];
                        if (g < fold.n) fold.keep[g] = 0;
                    }
                }
            }
        }
    }
    if (part_pts) {
        // partitioned copy of the bin: [ground, source order][non-ground, source order]
        for (uint32_t i = tid; i < m; i += G) part_pts[src_begin + i] = sorted_pts[src_begin + ORD[i]];
        group_sync<G>();
        const uint32_t m2 = k4_compact<G>(n, ORD, sh.warp, [&](uint32_t i) { return FLG[i] == 0; });
        for (uint32_t i = tid; i < m2; i += G) part_pts[src_begin + m + i] = sorted_pts[src_begin + ORD[i]];
    }
    group_sync<G>();
    K4_TICK(6);
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) rc.prof[k] = prof[k];
    }
#undef K4_TICK
}

// One launch per size class.  Groups pull records of the class from the bucketed queue (largest bins first) through
// an atomic cursor until the class is drained.
// G == 32: every warp of the CTA is a group with its own shared-memory slice (slice_bytes).
// G == THREADS: the CTA is the group; bins above smem_cap_points work in their slice of the global scratch.
template <int THREADS, int G>
__global__ void __launch_bounds__(THREADS, (THREADS == 256) ? 3 : (THREADS == 128 ? 6 : 1))
k4_rgpf(GpfParams P, FlagRec* __restrict__ recs, uint32_t* __restrict__ queue, const uint32_t* __restrict__ bucket_list,
        uint32_t rec_capacity, int bk0, int bk1, int cls, const float4* __restrict__ sorted_pts, uint32_t* __restrict__ sorted_src,
        const float4* __restrict__ in_pts, const uint32_t* __restrict__ frame_off /*map cloud [F+1]*/,
        float4* __restrict__ part_pts /*nullable*/, uint8_t* __restrict__ keep_mask /*nullable*/,
        uint8_t* __restrict__ ground_mask /*nullable*/, uint32_t* __restrict__ frame_rejected /*[F] nullable*/,
        unsigned char* __restrict__ gscratch, uint32_t smem_cap_points, uint32_t slice_bytes,
        unsigned long long* __restrict__ fence, K4Fold fold) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NG = THREADS / G;
    constexpr int HT = (G == 32) ? 32 : (G == 128 ? 96 : 128);
    constexpr int NCNT = (G >= 128) ? 8 * G : 1;         // radix counters: class C, and class B's bins beyond 2048 points
    __shared__ K4Shared sh[NG];
    __shared__ float    s_prd[NG][2 * 9 * (HT + 1)];
    __shared__ uint32_t s_cnt[NG][NCNT];
    __shared__ uint32_t s_fetch;
    const int grp = (G == 32) ? (threadIdx.x >> 5) : 0;
    uint32_t bcnt[4] = {0u, 0u, 0u, 0u}, total = 0u;     // a class spans at most four buckets
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (bk0 + k < bk1) { bcnt[k] = min(queue[bk0 + k], rec_capacity); total += bcnt[k]; }
    }
    for (;;) {
        uint32_t i;
        if (G == 32) {
            i = 0u;
            if ((threadIdx.x & 31) == 0) i = atomicAdd(&queue[kQueueCursor + cls], 1u);
            i = __shfl_sync(FULL_MASK, i, 0);
        } else {
            if (threadIdx.x == 0) s_fetch = atomicAdd(&queue[kQueueCursor + cls], 1u);
            __syncthreads();
            i = s_fetch;
            __syncthreads();
        }
        if (i >= total) break;
        int bk = bk0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            if (bk == bk0 + k && i >= bcnt[k]) { i -= bcnt[k]; ++bk; }
        }
        const uint32_t w = bucket_list[(size_t)bk * rec_capacity + i];
        FlagRec& rc = recs[w];
        const uint32_t n = rc.n_points;
        if constexpr (G <= 256) {
            // classes A and B: the launch sizes the slices for the class maximum (kClassAMax / kClassBMax), so the bin always fits
            k4_process_bin<G, true>(P, rc, smem_raw + (size_t)grp * slice_bytes, s_prd[grp], s_cnt[grp], sh[grp], sorted_pts, sorted_src, in_pts,
                                    frame_off, part_pts, keep_mask, ground_mask, frame_rejected, fence, fold);
        } else if (n <= smem_cap_points) {
            k4_process_bin<G, true>(P, rc, smem_raw + (size_t)grp * slice_bytes, s_prd[grp], s_cnt[grp], sh[grp], sorted_pts, sorted_src, in_pts,
                                    frame_off, part_pts, keep_mask, ground_mask, frame_rejected, fence, fold);
        } else {
            k4_process_bin<G, false>(P, rc, gscratch + (size_t)rc.src_begin * 24u, s_prd[grp], s_cnt[grp], sh[grp], sorted_pts, sorted_src, in_pts,
                                     frame_off, part_pts, keep_mask, ground_mask, frame_rejected, fence, fold);
        }
    }
}

template <int THREADS, int G>
static cudaError_t launch_k4_class(cudaStream_t st, const GpfParams& P, FlagRec* recs, uint32_t* queue, const uint32_t* bucket_list,
                                   uint32_t rec_capacity, int bk0, int bk1, int cls, uint32_t smem_bytes, const float4* sorted_pts,
                                   uint32_t* sorted_src, const float4* in_pts, const uint32_t* frame_off, float4* part_pts,
                                   uint8_t* keep_mask, uint8_t* ground_mask, uint32_t* frame_rejected, unsigned char* gscratch, int grid,
                                   unsigned long long* fence, const K4Fold& fold) {
    // per bin: 12 n (xyz) + 4 n (order) + n (flags) = 17 n for warp groups, + 4 n (second half of the order / exchange area) = 21 n
    constexpr int NG = THREADS / G;
    constexpr uint32_t per_pt = (G == 32) ? 17u : 21u;
    const uint32_t slice = (smem_bytes / NG) & ~15u;
    const uint32_t cap = (slice - 32) / per_pt;
    if ((G == 32 && cap < kClassAMax) || (G == 128 && cap < kClassBMax)) return cudaErrorInvalidConfiguration;   // A / B have no scratch path
    auto kern = k4_rgpf<THREADS, G>;
    cudaError_t e = ensure_dyn_smem(kern, smem_bytes);
    if (e != cudaSuccess) return e;
    kern<<<grid, THREADS, smem_bytes, st>>>(P, recs, queue, bucket_list, rec_capacity, bk0, bk1, cls, sorted_pts, sorted_src, in_pts, frame_off,
                                            part_pts, keep_mask, ground_mask, frame_rejected, gscratch, cap, slice, fence, fold);
    return cudaGetLastError();
}

int k4_num_launches(bool with_class_c) { return with_class_c ? 3 : 2; }

cudaError_t launch_k4(cudaStream_t st, cudaStream_t st_b, cudaStream_t st_c, const GpfParams& P, FlagRec* recs, uint32_t* queue,
                      const uint32_t* bucket_list, uint32_t rec_capacity, const float4* sorted_pts, uint32_t* sorted_src, const float4* in_pts,
                      const uint32_t* frame_off, float4* part_pts, uint8_t* keep_mask, uint8_t* ground_mask, uint32_t* frame_rejected,
                      unsigned char* gscratch, int sm_count, unsigned long long* fence, const K4Fold& fold, int classes) {
    // The three size classes touch disjoint bins, so they run concurrently on three streams (the caller forks / joins).
    // Shared memory: A  8 x 8.75 KB slices + 18.7 KB products ~ 90 KB per CTA (8 bins);  B  52.6 KB + 11 KB products / radix counters ~ 64 KB
    // per CTA (1 bin, 4 warps).  Registers (80 per thread): A 20 K per 8 bins, B 10 K per bin.
    // Class C wants most of an SM: it is issued first so that its CTAs (which exit at once when the class is empty, the
    // usual case for KITTI-sized maps) do not have to wait for shared memory held by A and B.
    static_assert(kClassAMax <= 512 && kClassBMax <= 4096, "sort networks: 16 keys per lane");
    cudaError_t e;
    // class C: n > 2560, one 1024-thread CTA with most of an SM's shared memory; beyond ~8.7 k points global scratch.
    // Each of its CTAs needs a whole SM's registers just to find its queue empty, which stalls behind (and in front of) the
    // kernels of overlapped submissions: the caller leaves it out (classes & 4 == 0) while no such bin has been seen, and
    // runs it afterwards (classes == 4) if one turns up.
    if (classes & 4) {
        e = launch_k4_class<1024, 1024>(st_c, P, recs, queue, bucket_list, rec_capacity, kBucketC0, kBucketB0, 2, 180 * 1024, sorted_pts, sorted_src,
                                        in_pts, frame_off, part_pts, keep_mask, ground_mask, frame_rejected, gscratch, sm_count, fence, fold);
        if (e != cudaSuccess) return e;
    }
    if (!(classes & 3)) return cudaSuccess;
    // class B: 512 < n <= 2560, one 128-thread CTA per bin
    e = launch_k4_class<128, 128>(st_b, P, recs, queue, bucket_list, rec_capacity, kBucketB0, kBucketA0, 1, 21 * kClassBMax + 64, sorted_pts,
                                  sorted_src, in_pts, frame_off, part_pts, keep_mask, ground_mask, frame_rejected, gscratch, sm_count * 3, fence, fold);
    if (e != cudaSuccess) return e;
    // class A: n <= 512, one warp per bin, 8 warps per CTA
    // (two CTAs per SM fit by shared memory: with tens of thousands of small flagged bins per step -- 40 x 360 bins, 2 M-point map --
    //  R-GPF is bound by resident chains per SM, and CTAs that find the queue empty exit at once)
    return launch_k4_class<256, 32>(st, P, recs, queue, bucket_list, rec_capacity, kBucketA0, kNumBuckets, 0, 8 * (17 * kClassAMax + 48), sorted_pts,
                                    sorted_src, in_pts, frame_off, part_pts, keep_mask, ground_mask, frame_rejected, gscratch, sm_count * 2, fence, fold);
}

// ============================================================================================
// K4b  in-bin voxelize_preserving_labels of version 3 (erasor.cpp:526-528, erasor_utils.cpp:80-114):
//      pcl::VoxelGrid (centroid of all four fields per 'map_voxel_size' voxel, ascending voxel key) followed by
//      an exact 1-NN into the un-voxelised points to restore an un-averaged label in `intensity`.
//      Input of a flagged bin = bin_curr's points (source order) then the R-GPF ground points (source order).
//      Unpinned third-party choices, fixed the same way in the oracle: members of one voxel are summed in input
//      order; 1-NN ties go to the lowest input index.
// ============================================================================================
constexpr int K4B_THREADS = 512;      // one CTA per flagged bin; the per-bin chain (sort, heads, centroids, 1-NN) is what a launch lasts

// conservative distance along one axis from x to the voxel cell `cell` lying `off` cells away from x's own (see
// updater_kernels.cu::cell_gap): never more than the true gap, so a cell is only skipped when it cannot hold the nearest point
__device__ __forceinline__ float k4b_cell_gap(float x, int cell, int off, float leaf, float slack) {
    if (off == 0) return 0.0f;
    const float g = (off > 0) ? ((float)cell * leaf - x) : (x - (float)(cell + 1) * leaf);
    return fmaxf(g - slack, 0.0f);
}

__global__ void __launch_bounds__(K4B_THREADS)
k4b_voxelize(float leaf_f, int B, const FlagRec* __restrict__ recs, const uint32_t* __restrict__ n_recs, uint32_t rec_capacity,
             const uint32_t* __restrict__ cnt /*[2][1][B+1]*/, const uint32_t* __restrict__ dst_start /*[2][1][B+2]*/,
             const float4* __restrict__ qry_sorted, const float4* __restrict__ part_pts,
             float4* __restrict__ vox_pts, uint32_t* __restrict__ vox_cnt, uint32_t* __restrict__ vox_start,
             unsigned char* __restrict__ gscratch, uint32_t smem_cap_points) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ uint32_t s_warp[K4B_THREADS / 32 + 1];
    __shared__ float    s_red[6][K4B_THREADS / 32];
    __shared__ float    s_minmax[6];
    __shared__ uint32_t s_hist[K4B_THREADS / 32][256];      // radix sort: per-warp digit counts / running offsets
    __shared__ uint32_t s_tot[256];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t nrec = min(*n_recs, rec_capacity);
    const float inv = FD(1.0f, leaf_f);
    const uint32_t* cq  = cnt + (B + 1);
    const uint32_t* dsm = dst_start;
    const uint32_t* dsq = dst_start + (B + 2);

    for (uint32_t w = blockIdx.x; w < nrec; w += gridDim.x) {
        const FlagRec& rc = recs[w];
        const uint32_t b = rc.bin, qc = cq[b], ng = rc.n_ground_final, n = qc + ng;
        const uint32_t region = dsq[b] + dsm[b];
        unsigned char* base = (n <= smem_cap_points) ? smem_raw : (gscratch + (size_t)region * 36u);
        float*    X   = reinterpret_cast<float*>(base);
        float*    Y   = X + n;
        float*    Z   = Y + n;
        float*    I   = Z + n;
        uint32_t* KEY = reinterpret_cast<uint32_t*>(I + n);
        uint32_t* VST = KEY + n;                  // voxel start positions (<= n entries) + 1
        uint32_t* ORD = VST + n + 1;              // point order, ping ...
        uint32_t* ORD2 = ORD + n;                 // ... pong of the radix sort
        uint32_t* VK  = ORD2 + n;                 // voxel key per voxel, ascending (<= n entries)
        if (n == 0) {
            if (tid == 0) { vox_cnt[rc.slot] = 0u; vox_start[rc.slot] = region; }
            continue;
        }
        for (uint32_t i = tid; i < n; i += K4B_THREADS) {
            const float4 p = (i < qc) ? qry_sorted[dsq[b] + i] : part_pts[rc.src_begin + (i - qc)];
            X[i] = p.x; Y[i] = p.y; Z[i] = p.z; I[i] = p.w; ORD[i] = i;
        }
        __syncthreads();
        // getMinMax3D
        {
            float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
            for (uint32_t i = tid; i < n; i += K4B_THREADS) {
                mn[0] = fminf(mn[0], X[i]); mx[0] = fmaxf(mx[0], X[i]);
                mn[1] = fminf(mn[1], Y[i]); mx[1] = fmaxf(mx[1], Y[i]);
                mn[2] = fminf(mn[2], Z[i]); mx[2] = fmaxf(mx[2], Z[i]);
            }
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                for (int o = 16; o > 0; o >>= 1) {
                    mn[a] = fminf(mn[a], __shfl_xor_sync(FULL_MASK, mn[a], o));
                    mx[a] = fmaxf(mx[a], __shfl_xor_sync(FULL_MASK, mx[a], o));
                }
                if (lane == 0) { s_red[a][warp] = mn[a]; s_red[3 + a][warp] = mx[a]; }
            }
            __syncthreads();
            if (tid < 6) {
                float v = s_red[tid][0];
                for (int ww = 1; ww < K4B_THREADS / 32; ++ww) v = (tid < 3) ? fminf(v, s_red[tid][ww]) : fmaxf(v, s_red[tid][ww]);
                s_minmax[tid] = v;
            }
            __syncthreads();
        }
        const float mnx = s_minmax[0], mny = s_minmax[1], mnz = s_minmax[2];
        const float mxx = s_minmax[3], mxy = s_minmax[4], mxz = s_minmax[5];
        const long long dx = (long long)FM(FS(mxx, mnx), inv) + 1;
        const long long dy = (long long)FM(FS(mxy, mny), inv) + 1;
        const long long dz = (long long)FM(FS(mxz, mnz), inv) + 1;
        const bool overflow = (dx * dy * dz) > 2147483647LL;
        uint32_t nv;
        float4* out = vox_pts + region;
        // pcl::VoxelGrid's cell grid of this bin (meaningful when !overflow)
        const int g_mb0 = (int)floorf(FM(mnx, inv)), g_mb1 = (int)floorf(FM(mny, inv)), g_mb2 = (int)floorf(FM(mnz, inv));
        const int g_div0 = (int)floorf(FM(mxx, inv)) - g_mb0 + 1, g_div1 = (int)floorf(FM(mxy, inv)) - g_mb1 + 1, g_div2 = (int)floorf(FM(mxz, inv)) - g_mb2 + 1;
        if (overflow) {
            // "Leaf size is too small for the input dataset": output = input
            nv = n;
            for (uint32_t i = tid; i < n; i += K4B_THREADS) out[i] = make_float4(X[i], Y[i], Z[i], I[i]);
            __syncthreads();
        } else {
            const int mb0 = (int)floorf(FM(mnx, inv)), mb1 = (int)floorf(FM(mny, inv)), mb2 = (int)floorf(FM(mnz, inv));
            const int Mb0 = (int)floorf(FM(mxx, inv)), Mb1 = (int)floorf(FM(mxy, inv));
            const int div0 = Mb0 - mb0 + 1, div1 = Mb1 - mb1 + 1;
            const int mul1 = div0, mul2 = div0 * div1;
            for (uint32_t i = tid; i < n; i += K4B_THREADS) {
                const int ijk0 = (int)FS(floorf(FM(X[i], inv)), (float)mb0);
                const int ijk1 = (int)FS(floorf(FM(Y[i], inv)), (float)mb1);
                const int ijk2 = (int)FS(floorf(FM(Z[i], inv)), (float)mb2);
                KEY[i] = (uint32_t)(ijk0 + ijk1 * mul1 + ijk2 * mul2);
            }
            __syncthreads();
            // stable LSD radix sort of the point order by voxel key (ties keep cloud order, like the index-tie-broken network it
            // replaces -- measured at 57 k cycles for 512 points, r02): 8-bit digits, as many passes as the bin's cell count needs;
            // every warp ranks a contiguous run of points with match.any, a column scan over the warps' rows makes the ranks global
            {
                constexpr int NW = K4B_THREADS / 32;
                const uint32_t cells = (uint32_t)((long long)g_div0 * g_div1 * g_div2);       // < 2^31: the overflow case went the other way
                int bits = 1; while (bits < 31 && (1u << bits) < cells) ++bits;
                const int npass = (bits + 7) / 8;
                const uint32_t chunk = ((n + NW * 32u - 1u) / (NW * 32u)) * 32u;
                const uint32_t w0 = min(n, (uint32_t)warp * chunk), w1 = min(n, w0 + chunk);
                uint32_t* src = ORD; uint32_t* dst = ORD2;
                uint32_t* mine = &s_hist[warp][0];
                for (int pass = 0; pass < npass; ++pass) {
                    const int shift = pass * 8;
                    for (int i = tid; i < NW * 256; i += K4B_THREADS) (&s_hist[0][0])[i] = 0u;
                    __syncthreads();
                    for (uint32_t i0 = w0; i0 < w1; i0 += 32u) {
                        const uint32_t i = i0 + lane;
                        const bool valid = i < w1;
                        const unsigned vm = __ballot_sync(FULL_MASK, valid);
                        if (valid) {
                            const uint32_t d = (KEY[src[i]] >> shift) & 255u;
                            const unsigned peers = __match_any_sync(vm, d);
                            if (lane == __ffs(peers) - 1) mine[d] += __popc(peers);
                        }
                        __syncwarp();
                    }
                    __syncthreads();
                    if (tid < 256) {                      // column scan over the warps' rows; the digit's total
                        uint32_t run = 0u;
#pragma unroll
                        for (int w = 0; w < NW; ++w) { const uint32_t c = s_hist[w][tid]; s_hist[w][tid] = run; run += c; }
                        s_tot[tid] = run;
                    }
                    __syncthreads();
                    if (warp == 0) {                      // exclusive scan of the 256 digit totals
                        uint32_t t[8], sum = 0u;
#pragma unroll
                        for (int j = 0; j < 8; ++j) { t[j] = s_tot[lane * 8 + j]; }
#pragma unroll
                        for (int j = 0; j < 8; ++j) { const uint32_t x = t[j]; t[j] = sum; sum += x; }
                        uint32_t incl = sum;
                        for (int o = 1; o < 32; o <<= 1) { const uint32_t x = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += x; }
#pragma unroll
                        for (int j = 0; j < 8; ++j) s_tot[lane * 8 + j] = incl - sum + t[j];
                    }
                    __syncthreads();
                    for (uint32_t i0 = w0; i0 < w1; i0 += 32u) {
                        const uint32_t i = i0 + lane;
                        const bool valid = i < w1;
                        const unsigned vm = __ballot_sync(FULL_MASK, valid);
                        if (valid) {
                            const uint32_t q = src[i];
                            const uint32_t d = (KEY[q] >> shift) & 255u;
                            const unsigned peers = __match_any_sync(vm, d);
                            const uint32_t off = mine[d];
                            __syncwarp(vm);
                            if (lane == __ffs(peers) - 1) mine[d] = off + __popc(peers);
                            dst[s_tot[d] + off + __popc(peers & ((1u << lane) - 1u))] = q;
                        }
                        __syncwarp();
                    }
                    __syncthreads();
                    uint32_t* t = src; src = dst; dst = t;
                }
                ORD = src;
            }
            // voxel heads in sorted order
            nv = k4_compact<K4B_THREADS>(n, VST, s_warp, [&](uint32_t i) { return i == 0 || KEY[ORD[i]] != KEY[ORD[i - 1]]; });
            if (tid == 0) VST[nv] = n;
            __syncthreads();
            // centroids: float sums in member order, divided by float(count)  (pcl::CentroidPoint)
            for (uint32_t v = tid; v < nv; v += K4B_THREADS) {
                const uint32_t a = VST[v], e = VST[v + 1];
                float sx = 0.0f, sy = 0.0f, sz = 0.0f, si = 0.0f;
                for (uint32_t li = a; li < e; ++li) {
                    const uint32_t q = ORD[li];
                    sx = FA(sx, X[q]); sy = FA(sy, Y[q]); sz = FA(sz, Z[q]); si = FA(si, I[q]);
                }
                const float cn = (float)(e - a);
                out[v] = make_float4(FD(sx, cn), FD(sy, cn), FD(sz, cn), FD(si, cn));
            }
            __syncthreads();
        }
        // exact 1-NN of every centroid into the bin's points (ties to the lowest index); copy that point's intensity.
        // Through the voxel grid itself: the centroid's own cell first, then the 26 around it -- each skipped when even its
        // nearest corner is provably farther than the best so far -- and further shells only while something unseen could
        // still be closer.  Same result as comparing against every point (the fallback for the overflow case and for
        // non-finite centroids), at a few cells per centroid instead of n distance evaluations.
        if (!overflow) {
            for (uint32_t v = tid; v < nv; v += K4B_THREADS) VK[v] = KEY[ORD[VST[v]]];
            __syncthreads();
        }
        for (uint32_t v = tid; v < nv; v += K4B_THREADS) {
            const float4 c = out[v];
            float best = __int_as_float(0x7f800000);
            uint32_t bi = 0xFFFFFFFFu;
            const bool finite = (fabsf(c.x) < 3.0e38f) && (fabsf(c.y) < 3.0e38f) && (fabsf(c.z) < 3.0e38f);
            if (!overflow && finite) {
                const int ci = (int)FS(floorf(FM(c.x, inv)), (float)g_mb0), cj = (int)FS(floorf(FM(c.y, inv)), (float)g_mb1), ck = (int)FS(floorf(FM(c.z, inv)), (float)g_mb2);
                const float slack = 1.0e-3f * leaf_f + 4.0e-6f * fmaxf(fabsf(c.x), fmaxf(fabsf(c.y), fabsf(c.z)));
                int rad = 0;
                while (true) {
                    for (int a = -rad; a <= rad; ++a) {
                        const int ii = ci + a;
                        if (ii < 0 || ii >= g_div0) continue;
                        for (int bb = -rad; bb <= rad; ++bb) {
                            const int jj = cj + bb;
                            if (jj < 0 || jj >= g_div1) continue;
                            for (int cc = -rad; cc <= rad; ++cc) {
                                if (max(abs(a), max(abs(bb), abs(cc))) != rad) continue;
                                const int kk = ck + cc;
                                if (kk < 0 || kk >= g_div2) continue;
                                if (rad > 0) {
                                    const float gx = k4b_cell_gap(c.x, ii + g_mb0, a, leaf_f, slack);
                                    const float gy = k4b_cell_gap(c.y, jj + g_mb1, bb, leaf_f, slack);
                                    const float gz = k4b_cell_gap(c.z, kk + g_mb2, cc, leaf_f, slack);
                                    if (0.999f * (gx * gx + gy * gy + gz * gz) > best) continue;
                                }
                                const uint32_t key = (uint32_t)(ii + jj * g_div0 + kk * g_div0 * g_div1);
                                uint32_t lo = 0, hi = nv;                 // first voxel with key >= `key`
                                while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (VK[mid] < key) lo = mid + 1; else hi = mid; }
                                if (lo >= nv || VK[lo] != key) continue;
                                for (uint32_t li = VST[lo]; li < VST[lo + 1]; ++li) {
                                    const uint32_t q = ORD[li];
                                    const float ddx = FS(c.x, X[q]), ddy = FS(c.y, Y[q]), ddz = FS(c.z, Z[q]);
                                    const float d = FA(FA(FM(ddx, ddx), FM(ddy, ddy)), FM(ddz, ddz));
                                    if (d < best || (d == best && q < bi)) { best = d; bi = q; }
                                }
                            }
                        }
                    }
                    const float reach = FM(FM((float)rad, leaf_f), 0.9999f);
                    if (bi != 0xFFFFFFFFu && best < FM(reach, reach)) break;
                    ++rad;
                    if (rad > 4096) break;
                }
            }
            if (bi == 0xFFFFFFFFu) {
                bi = 0;
                for (uint32_t i = 0; i < n; ++i) {
                    const float ddx = FS(c.x, X[i]), ddy = FS(c.y, Y[i]), ddz = FS(c.z, Z[i]);
                    const float d = FA(FA(FM(ddx, ddx), FM(ddy, ddy)), FM(ddz, ddz));
                    if (d < best) { best = d; bi = i; }
                }
            }
            out[v].w = I[bi];
        }
        if (tid == 0) { vox_cnt[rc.slot] = nv; vox_start[rc.slot] = region; }
        __syncthreads();
    }
}

cudaError_t launch_k4b(cudaStream_t st, float leaf, int B, const FlagRec* recs, const uint32_t* n_recs, uint32_t rec_capacity,
                       const uint32_t* cnt, const uint32_t* dst_start, const float4* qry_sorted, const float4* part_pts,
                       float4* vox_pts, uint32_t* vox_cnt, uint32_t* vox_start, unsigned char* gscratch, int grid) {
    constexpr uint32_t SMEM_BYTES = 160 * 1024;     // one CTA per SM (a frame flags a few dozen bins): bins up to ~4500 points stay in shared memory
    // 16 n (xyzi) + 4 n (key) + 4 (n+1) (voxel starts) + 2 x 4 n (point order, ping-pong) + 4 n (voxel keys) = 36 n + 4
    const uint32_t cap = (SMEM_BYTES - 64) / 36u;
    cudaError_t e = ensure_dyn_smem(k4b_voxelize, SMEM_BYTES);
    if (e != cudaSuccess) return e;
    k4b_voxelize<<<grid, K4B_THREADS, SMEM_BYTES, st>>>(leaf, B, recs, n_recs, rec_capacity, cnt, dst_start, qry_sorted, part_pts,
                                                       vox_pts, vox_cnt, vox_start, gscratch, cap);
    return cudaGetLastError();
}

// ============================================================================================
// K5  output assembly (single-frame cloud mode)
// ============================================================================================
// Plan: sizes per bin -> exclusive scans -> copy jobs.  Job slots: [0,2B) selected bins (two sources each),
// [2B,3B) ground_viz per flagged slot, [3B,4B) map_rejected per flagged slot, [4B,5B) curr_rejected per bin.
__global__ void __launch_bounds__(1024)
k5_plan(int B, int version, int skip_voxelize, const uint32_t* __restrict__ cnt /*[2][1][B+1]*/,
        const uint32_t* __restrict__ dst_start /*[2][1][B+2]*/, const uint8_t* __restrict__ action,
        const uint32_t* __restrict__ flag_slot, const FlagRec* __restrict__ recs, const uint32_t* __restrict__ n_recs,
        const uint32_t* __restrict__ vox_cnt /*per slot, nullable*/, const uint32_t* __restrict__ vox_start /*per slot*/,
        const float4* __restrict__ map_sorted, const float4* __restrict__ qry_sorted, const float4* __restrict__ part_pts,
        const float4* __restrict__ vox_pts,
        float4* __restrict__ arranged, float4* __restrict__ map_rej, float4* __restrict__ curr_rej,
        CopyJob* __restrict__ jobs, uint32_t* __restrict__ out_sizes /*[4]: arranged, complement, map_rej, curr_rej*/,
        uint32_t* __restrict__ tmp /*[3*(B+1)]*/) {
    __shared__ uint32_t s_part[34];
    const int tid = threadIdx.x, nt = blockDim.x;
    const uint32_t* cm = cnt;
    const uint32_t* cq = cnt + (B + 1);
    const uint32_t* dsm = dst_start;
    const uint32_t* dsq = dst_start + (B + 2);
    uint32_t* sel = tmp;                 // selected size / start per bin
    uint32_t* gv  = tmp + (B + 1);       // ground size / start per flagged slot
    uint32_t* rj  = tmp + 2 * (B + 1);   // rejected size / start per flagged slot
    const uint32_t nflag = *n_recs;      // single frame: records are this frame's, indexed by slot
    const bool vox = (version == 3) && !skip_voxelize;

    for (int b = tid; b < B; b += nt) {
        const uint8_t a = action[b] & 0x0F;
        uint32_t sz = 0;
        if (a == ACT_MAP) sz = cm[b];
        else if (a == ACT_FLAG) sz = vox ? vox_cnt[flag_slot[b]] : cq[b] + recs[flag_slot[b]].n_ground_final;
        else if (a == ACT_MERGE) sz = cq[b] + cm[b];
        else if (a == ACT_CURR) sz = cq[b];
        sel[b] = sz;
    }
    for (uint32_t s = tid; s < (uint32_t)B; s += nt) {
        gv[s] = (s < nflag) ? recs[s].n_ground_final : 0u;
        rj[s] = (s < nflag) ? recs[s].n_rejected : 0u;
    }
    __syncthreads();
    const uint32_t sel_total = block_excl_scan(sel, sel, B, s_part);
    const uint32_t gv_total  = block_excl_scan(gv, gv, B, s_part);
    const uint32_t rj_total  = block_excl_scan(rj, rj, B, s_part);
    // selected bins
    for (int b = tid; b < B; b += nt) {
        const uint8_t a = action[b] & 0x0F;
        CopyJob j0{nullptr, nullptr, 0u, 0u}, j1{nullptr, nullptr, 0u, 0u};
        float4* dst = arranged + sel[b];
        if (a == ACT_MAP) {
            j0 = CopyJob{map_sorted + dsm[b], dst, cm[b], 0u};
        } else if (a == ACT_FLAG) {
            const uint32_t slot = flag_slot[b];
            if (vox) {
                j0 = CopyJob{vox_pts + vox_start[slot], dst, vox_cnt[slot], 0u};
            } else {
                j0 = CopyJob{qry_sorted + dsq[b], dst, cq[b], 0u};                                           // bin_curr
                j1 = CopyJob{part_pts + recs[slot].src_begin, dst + cq[b], recs[slot].n_ground_final, 0u};   // += piecewise_ground_
            }
        } else if (a == ACT_MERGE) {
            j0 = CopyJob{qry_sorted + dsq[b], dst, cq[b], 0u};                 // merge_bins: curr first,
            j1 = CopyJob{map_sorted + dsm[b], dst + cq[b], cm[b], 0u};         // then map (erasor.cpp:301-306)
        } else if (a == ACT_CURR) {
            j0 = CopyJob{qry_sorted + dsq[b], dst, cq[b], 0u};
        }
        jobs[2 * b] = j0; jobs[2 * b + 1] = j1;
    }
    // ground_viz (appended to arranged, erasor.cpp:616) and map_rejected, per flagged slot in processing order
    for (uint32_t s = tid; s < (uint32_t)B; s += nt) {
        CopyJob jg{nullptr, nullptr, 0u, 0u}, jr{nullptr, nullptr, 0u, 0u};
        if (s < nflag) {
            const FlagRec& rc = recs[s];
            jg = CopyJob{part_pts + rc.src_begin, arranged + sel_total + gv[s], rc.n_ground_final, 0u};
            jr = CopyJob{part_pts + rc.src_begin + rc.n_ground_final, map_rej + rj[s], rc.n_rejected, 0u};
        }
        jobs[2 * B + s] = jg; jobs[3 * B + s] = jr;
    }
    __syncthreads();
    // curr_rejected (version 2 only, erasor.cpp:405-408)
    for (int b = tid; b < B; b += nt) sel[b] = (action[b] & ACT_CURR_REJECTED_BIT) ? cq[b] : 0u;
    __syncthreads();
    const uint32_t cr_total = block_excl_scan(sel, sel, B, s_part);
    for (int b = tid; b < B; b += nt) {
        CopyJob j{nullptr, nullptr, 0u, 0u};
        if (action[b] & ACT_CURR_REJECTED_BIT) j = CopyJob{qry_sorted + dsq[b], curr_rej + sel[b], cq[b], 0u};
        jobs[4 * B + b] = j;
    }
    if (tid == 0) {
        out_sizes[0] = sel_total + gv_total;
        out_sizes[1] = cm[B];
        out_sizes[2] = rj_total;
        out_sizes[3] = cr_total;
        out_sizes[4] = gv_total;          // ground_viz = the tail of arranged (erasor.cpp:616)
    }
}

__global__ void __launch_bounds__(128) k5_copy(const CopyJob* __restrict__ jobs, uint32_t n_jobs) {
    for (uint32_t j = blockIdx.x; j < n_jobs; j += gridDim.x) {
        const CopyJob jb = jobs[j];
        for (uint32_t i = threadIdx.x; i < jb.n; i += 128) jb.dst[i] = jb.src[i];
    }
}

cudaError_t launch_k5(cudaStream_t st, int B, int version, int skip_voxelize, const uint32_t* cnt, const uint32_t* dst_start,
                      const uint8_t* action, const uint32_t* flag_slot, const FlagRec* recs, const uint32_t* n_recs,
                      const uint32_t* vox_cnt, const uint32_t* vox_start, const float4* map_sorted, const float4* qry_sorted,
                      const float4* part_pts, const float4* vox_pts, float4* arranged, float4* map_rej, float4* curr_rej,
                      CopyJob* jobs, uint32_t* out_sizes, uint32_t* tmp, int copy_grid) {
    k5_plan<<<1, 1024, 0, st>>>(B, version, skip_voxelize, cnt, dst_start, action, flag_slot, recs, n_recs, vox_cnt, vox_start,
                                map_sorted, qry_sorted, part_pts, vox_pts, arranged, map_rej, curr_rej, jobs, out_sizes, tmp);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    k5_copy<<<copy_grid, 128, 0, st>>>(jobs, 5u * (uint32_t)B);
    return cudaGetLastError();
}

// ============================================================================================
// small utilities
// ============================================================================================
__global__ void k_init_tables(uint32_t* zmin, uint32_t* zmax, size_t n, uint32_t* cnt, size_t n_cnt, uint32_t* n_recs,
                              uint32_t* frame_rejected, uint32_t* n_flagged, int F, uint32_t* queue) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (size_t)kQueueWords) queue[i] = 0u;
    if (i < n) { zmin[i] = 0xFFFFFFFFu; zmax[i] = 0u; }
    if (i < n_cnt) cnt[i] = 0u;
    if (i == 0) *n_recs = 0u;
    if (frame_rejected && i < (size_t)F) frame_rejected[i] = 0u;
    if (n_flagged && i < (size_t)F) n_flagged[i] = 0u;      // (a frame without map points has no chunk, hence no leader CTA to write it)
}
cudaError_t launch_init_tables(cudaStream_t st, uint32_t* zmin, uint32_t* zmax, size_t n, uint32_t* cnt, size_t n_cnt, uint32_t* n_recs,
                               uint32_t* frame_rejected, uint32_t* n_flagged, int F, uint32_t* queue) {
    size_t m = n > (size_t)F ? n : (size_t)F;
    m = m > n_cnt ? m : n_cnt;
    const int blocks = (int)((m + 255) / 256);
    k_init_tables<<<blocks > 0 ? blocks : 1, 256, 0, st>>>(zmin, zmax, n, cnt, n_cnt, n_recs, frame_rejected, n_flagged, F, queue);
    return cudaGetLastError();
}

// fold per-frame keep masks onto the global map: a map point survives unless some frame rejected it.
// Only zeros are written, so concurrent writers need no atomics; the mask ACCUMULATES over calls (reset it with
// launch_fill_u8 / erasor_reset_keep_mask at the start of a job).  Indices beyond the mask are dropped.
__global__ void k_fold_keep(const uint8_t* __restrict__ keep, const uint32_t* __restrict__ voi_index, size_t n, uint8_t* __restrict__ global_keep, uint32_t n_global) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && keep[i] == 0) {
        const uint32_t g = voi_index[i];
        if (g < n_global) global_keep[g] = 0;
    }
}
cudaError_t launch_fold_keep(cudaStream_t st, const uint8_t* keep, const uint32_t* voi_index, size_t n, uint8_t* global_keep, size_t n_global) {
    if (n == 0) return cudaSuccess;
    k_fold_keep<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(keep, voi_index, n, global_keep, (uint32_t)n_global);
    return cudaGetLastError();
}

// ---- the exchange step of the frame-sharded job: bit-packed masks (8x fewer bytes over NVLink), AND over the ranks -----
// keep[0..n) bytes (0 / non-0) -> bits, one 32-bit word per warp step (ballot); the tail word is padded with ones.
__global__ void __launch_bounds__(256) k_pack_keep_bits(const uint8_t* __restrict__ keep, size_t n, uint32_t* __restrict__ words, size_t n_words) {
    const size_t w0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const size_t stride = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t w = w0; w < n_words; w += stride) {
        const size_t i = w * 32 + lane;
        const bool k = (i < n) ? (keep[i] != 0) : true;
        const unsigned bal = __ballot_sync(FULL_MASK, k);
        if (lane == 0) words[w] = bal;
    }
}
// gathered[r][w], r < n_ranks: AND over the ranks, unpacked back into one byte per map point
__global__ void __launch_bounds__(256) k_and_unpack_keep(const uint32_t* __restrict__ gathered, int n_ranks, size_t n_words, size_t n, uint8_t* __restrict__ keep) {
    const size_t w0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const size_t stride = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t w = w0; w < n_words; w += stride) {
        uint32_t v = 0xFFFFFFFFu;
        for (int r = lane; r < n_ranks; r += 32) v &= gathered[(size_t)r * n_words + w];
        v = __reduce_and_sync(FULL_MASK, v);
        const size_t i = w * 32 + lane;
        if (i < n) keep[i] = (uint8_t)((v >> lane) & 1u);
    }
}
cudaError_t launch_pack_keep_bits(cudaStream_t st, const uint8_t* keep, size_t n, uint32_t* words) {
    const size_t n_words = (n + 31) / 32;
    if (n_words == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)std::min<size_t>((n_words + 7) / 8, 148 * 8);
    k_pack_keep_bits<<<blocks, 256, 0, st>>>(keep, n, words, n_words);
    return cudaGetLastError();
}
cudaError_t launch_and_unpack_keep(cudaStream_t st, const uint32_t* gathered, int n_ranks, size_t n, uint8_t* keep) {
    const size_t n_words = (n + 31) / 32;
    if (n_words == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)std::min<size_t>((n_words + 7) / 8, 148 * 8);
    k_and_unpack_keep<<<blocks, 256, 0, st>>>(gathered, n_ranks, n_words, n, keep);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) k_fill_u8(uint8_t* __restrict__ p, size_t n, uint8_t v) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
cudaError_t launch_fill_u8(cudaStream_t st, uint8_t* p, size_t n, uint8_t v) {
    if (n == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)std::min<size_t>((n + 255) / 256, 148 * 8);
    k_fill_u8<<<blocks, 256, 0, st>>>(p, n, v);
    return cudaGetLastError();
}

// erasor_process_scans: the query chunks were cut on the host from the raw scan sizes (an upper bound of the voxel counts);
// set every query chunk's length from its full length (pad_) and the frame's voxel count written by the batched voxeliser
__global__ void __launch_bounds__(256) k_clamp_query_chunks(ChunkDesc* __restrict__ chunks, uint32_t first, uint32_t n, const uint32_t* __restrict__ count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ChunkDesc& d = chunks[first + i];
    const uint32_t c = count[d.frame], s = d.begin - d.frame_begin;
    d.len = c > s ? min(d.pad_, c - s) : 0u;
}
cudaError_t launch_clamp_query_chunks(cudaStream_t st, ChunkDesc* chunks, uint32_t first, uint32_t n, const uint32_t* count) {
    if (n == 0) return cudaSuccess;
    k_clamp_query_chunks<<<(n + 255) / 256, 256, 0, st>>>(chunks, first, n, count);
    return cudaGetLastError();
}

}  // namespace erasor
