// device_types.h -- shared host/device structs of the path's HBM layout (see DESIGN.md section 3).
#pragma once
#include <cstdint>

#include "binning.h"

namespace erasor {

constexpr uint32_t kSkip      = 0xFFFFFFFFu;   // dst_start value of a bin that is not scattered
constexpr uint16_t kNoBin16   = 0xFFFFu;       // bin id of a point that failed the z window / range test
constexpr uint32_t kIdPad     = 1024;          // slack entries behind the bin-id arrays: K2 prefetches ids without bounds checks
constexpr uint32_t kMapPad    = 256;           // slack points behind the resident map: node-mode K1 streams it without bounds checks
constexpr int      kListWarps = 32;            // node mode: per-chunk stride of the per-warp VoI list counters (K1 runs 8 or 32 warps)
constexpr int      kMaxIter   = 8;             // gf_iter upper bound for the tap arrays

// status codes held on the device (values published through erasor_get_status)
enum : uint8_t { ST_LITTLE = 0, ST_MERGE = 1, ST_MAP_HIGH = 2, ST_BLOCKED = 3, ST_CURR_HIGH = 4 };
// what the selected bin is made of (erasor.cpp:493-563 / 346-427)
enum : uint8_t { ACT_MAP = 0, ACT_FLAG = 1, ACT_MERGE = 2, ACT_CURR = 3, ACT_NONE = 4, ACT_CURR_REJECTED_BIT = 0x10 };

// One contiguous run of points of one cloud of one frame, processed by one CTA of K1 / one warp of K2.
struct ChunkDesc {
    uint32_t begin;        // first point (index into the source cloud array: the concatenated batch clouds, or the resident global map in node mode)
    uint32_t len;          // points in this chunk
    uint32_t frame;        // frame index
    uint32_t cloud;        // 0 map, 1 query
    uint32_t frame_begin;  // source index of the frame's first point (node mode, map cloud: 0 -- every frame scans the whole map)
    uint32_t bin_begin;    // index of the chunk's first point in the bin-id array (batch mode: == begin; node mode: frame * n_map + begin)
    uint32_t out_base;     // base of the frame's region in the scattered arrays and the per-frame masks (batch: frame_begin; node: frame * n_map)
    uint32_t pad_;         // (erasor_process_scans, query chunks: the chunk's full length, len being clamped on the device)
};

// Node mode (map resident in HBM, erasor_process_nodes): what OfflineMapUpdater::fetch_VoI needs per frame
// (reference OfflineMapUpdater.cpp:381-438): the radius cut around the body position, in double on float
// differences, and the origin -> body affine (float, pcl::transformPointCloud association, no contraction).
struct NodePose {
    double px, py;         // tf_body2origin(0,3), (1,3) as the reference reads them (:246-247)
    double limit;          // pow(max_range, 2)
    float  T[12];          // rows 0..2 of tf_body2origin.inverse()
    float  pxf, pyf;       // px, py as floats (they are floats widened to double, so this is exact)
    float  lim_lo, lim_hi; // float guard band around limit: d2f < lim_lo => inside for sure, d2f > lim_hi => outside for sure
};

struct SrtParams {
    double scan_ratio_threshold;
    double th_bin_max_h;
    int    minimum_num_pts;
    int    version;
    int    R, S, B;
    int    scatter_mode;       // 0: every bin (cloud outputs), 1: flagged bins only (mask outputs)
};

struct GpfParams {
    double th_dist;            // gf_dist_thr
    double th_seeds;           // gf_th_seeds_height
    int    num_lowest_pts;
    int    num_lpr;
    int    iters;
    int    cov_mode;
};

// The multi-GPU fold, done in K4's epilogue: global_keep[index ? index[frame_base + src] : src] = 0 for every rejected point.
struct K4Fold {
    uint8_t*        keep;      // global keep mask of the map (null: no fold)
    const uint32_t* index;     // per-VoI-point global index (batch mode); null: the source index is the global index (node mode)
    uint32_t        n;         // size of the global mask (writes beyond it are dropped)
    uint32_t        pad_;
};

// R-GPF work queue.  K3 appends every flagged-bin record to the bucket of its size; K4's three size classes
// (A: one warp per bin, B: one 256-thread CTA per bin, C: one 1024-thread CTA per bin) walk their buckets from the
// largest bins to the smallest through an atomic cursor, so the long bins start first and no group idles while
// records of its class remain.
constexpr uint32_t kClassAMax   = 512;     // class A: n <= 512          (register bitonic sort, 16 keys per lane)
constexpr uint32_t kClassBMax   = 2560;    // class B: 512 < n <= 2560   (8 warps x 512 keys)
constexpr int      kNumBuckets  = 9;       // 0: C | 1-4: B | 5-8: A
constexpr int      kBucketC0 = 0, kBucketB0 = 1, kBucketA0 = 5;
constexpr int      kQueueCursor = 16;      // queue[kQueueCursor + class] : next virtual index of the class (0 A, 1 B, 2 C)
constexpr int      kQueueWords  = 32;      // queue[0 .. kNumBuckets) : records per bucket
ERASOR_HD int rgpf_bucket_of(uint32_t n) {
    if (n > kClassBMax) return 0;
    if (n > 2048u) return 1;
    if (n > 1536u) return 2;
    if (n > 1024u) return 3;
    if (n > kClassAMax) return 4;
    if (n > 384u) return 5;
    if (n > 256u) return 6;
    if (n > 128u) return 7;
    return 8;
}

// Per flagged bin record written by K3 and completed by K4
struct FlagRec {
    uint32_t frame;
    uint32_t bin;
    uint32_t slot;             // index among the frame's flagged bins (bin order)
    uint32_t n_points;
    uint32_t src_begin;        // offset of the bin's points in the scattered map array (absolute)
    uint32_t n_seeds;
    uint32_t n_empty_fits;
    uint32_t n_ground_final;
    uint32_t cursor;           // reserved
    uint32_t n_rejected;       // points handed to map_rejected (0 when gf_iter == 0: the reference fills no outliers then)
    double   lpr_height;
    double   normal_d[kMaxIter][4];
    uint32_t n_ground[kMaxIter];
    uint32_t prof[8];          // SM cycles per phase (thread 0): load+idx sort, z sort, seeds, accumulate, svd, classify+compact, outputs, sweeps
};

}  // namespace erasor
