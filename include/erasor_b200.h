/* ============================================================================
 * erasor_b200.h -- C ABI of the B200-native R-POD -> Scan Ratio Test -> R-GPF path
 *
 * This is the drop-in boundary for the reference's `class ERASOR`
 * (reference include/erasor/erasor.h:43-147, src/offline_map_updater/src/erasor.cpp)
 * as used by its single caller OfflineMapUpdater::callback_node
 * (src/offline_map_updater/src/OfflineMapUpdater.cpp:266-284).  The reference has no
 * FFI layer of its own; each entry point below names the C++ member it replaces.
 *
 * Conventions
 *   - plain C types only; clouds are float[n][4] = x, y, z, intensity (pcl::PointXYZI's
 *     four used floats; on the device this is one float4 per point, 16-byte aligned);
 *   - every function returns 0 (ERASOR_OK) or a negative error code and never throws;
 *     erasor_last_error() gives the text;
 *   - one handle <-> one CUDA device + one stream; a handle is not thread-safe, but distinct handles may be driven from
 *     distinct host threads, and several handles on one device overlap on the GPU (the *_async entry points);
 *   - device buffers are owned by the handle, caller buffers by the caller;
 *     `ptr_kind` says whether caller buffers are host (pageable or pinned) or device memory;
 *   - bins are indexed  bin = sector * num_rings + ring  (theta outer, r inner: the order
 *     in which the reference walks and flattens its R-POD, erasor.cpp:309-320);
 *   - there is no CPU fallback: without a CUDA device erasor_create fails with ERASOR_E_CUDA.
 * ========================================================================== */
#ifndef ERASOR_B200_H
#define ERASOR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ERASOR_B200_ABI_VERSION 2

typedef struct erasor_ctx* erasor_handle_t;

/* The 15 keys ERASOR's constructor reads from /erasor/ (erasor.h:47-61), /erasor/version
 * (OfflineMapUpdater.cpp:81) and three mode switches that pin choices the reference leaves
 * to its third-party libraries. */
typedef struct {
    double max_range;              /* /erasor/max_range             erasor.h:47 */
    double min_h;                  /* /erasor/min_h                 erasor.h:51 */
    double max_h;                  /* /erasor/max_h                 erasor.h:50 */
    double th_bin_max_h;           /* /erasor/th_bin_max_h          erasor.h:52 (v2 only) */
    double scan_ratio_threshold;   /* /erasor/scan_ratio_threshold  erasor.h:53 */
    double rejection_ratio;        /* /erasor/rejection_ratio       erasor.h:56 (unused by the path) */
    double gf_dist_thr;            /* /erasor/gf_dist_thr           erasor.h:57 */
    double gf_th_seeds_height;     /* /erasor/gf_th_seeds_height    erasor.h:60 */
    double map_voxel_size;         /* /erasor/map_voxel_size        erasor.h:61 */
    int    num_rings;              /* /erasor/num_rings             erasor.h:48 */
    int    num_sectors;            /* /erasor/num_sectors           erasor.h:49 */
    int    num_lowest_pts;         /* /erasor/num_lowest_pts        erasor.h:54 */
    int    minimum_num_pts;        /* /erasor/minimum_num_pts       erasor.h:55 */
    int    gf_iter;                /* /erasor/gf_iter               erasor.h:58 */
    int    gf_num_lpr;             /* /erasor/gf_num_lpr            erasor.h:59 */
    int    version;                /* /erasor/version               OfflineMapUpdater.cpp:81 */
    int    cov_mode;               /* 0: pcl::computeMeanAndCovarianceMatrix of PCL<=1.10 (default), 1: PCL>=1.11 (shifted) */
    int    sort_mode;              /* must be 1: R-GPF z-sort ties in source order (std::sort's tie order is unspecified) */
    int    skip_voxelize;          /* 1: leave out v3's in-bin voxelize_preserving_labels (erasor.cpp:526-528) */
} erasor_params_t;

enum { ERASOR_PTR_HOST = 0, ERASOR_PTR_DEVICE = 1,
       /* OR-able onto either, mask modes only (erasor_process_frames* / erasor_process_nodes*): the QUERY cloud is packed
        * x y z, three floats per point.  The masks never read the query's intensity (it only travels into the cloud outputs,
        * erasor.cpp:526-563), and a caller that repacks pcl::PointXYZI (32 bytes) anyway ships a quarter less over PCIe. */
       ERASOR_PTR_QUERY_XYZ = 16 };
enum { ERASOR_CLOUD_MAP = 0, ERASOR_CLOUD_QUERY = 1 };

enum {
    ERASOR_OK            = 0,
    ERASOR_E_INVALID     = -1,   /* bad argument / parameter */
    ERASOR_E_CUDA        = -2,   /* CUDA runtime error, or no device */
    ERASOR_E_STATE       = -3,   /* call order violated (set_inputs -> compare -> get_*) */
    ERASOR_E_CAPACITY    = -4,   /* caller buffer too small */
    ERASOR_E_UNSUPPORTED = -5    /* e.g. num_rings*num_sectors beyond the shared-memory table limit */
};

/* status values, as the reference publishes them (erasor.h:12-18) */
#define ERASOR_STATUS_LITTLE_NUM     0.0f
#define ERASOR_STATUS_MERGE_BINS     0.25f
#define ERASOR_STATUS_MAP_IS_HIGHER  0.5f
#define ERASOR_STATUS_BLOCKED        0.8f
#define ERASOR_STATUS_CURR_IS_HIGHER 1.0f

/* ---- lifetime --------------------------------------------------------------------------- */
/* replaces ERASOR::ERASOR(ros::NodeHandle*) (erasor.h:46-103): parameters are fixed here. */
int  erasor_create(const erasor_params_t* params, int device, erasor_handle_t* out);
void erasor_destroy(erasor_handle_t h);
const char* erasor_last_error(erasor_handle_t h);   /* h may be NULL: error of the last failed erasor_create */
int  erasor_abi_version(void);
/* the handle's CUDA stream (cudaStream_t as void*), so callers can order their own work after it */
void* erasor_stream(erasor_handle_t h);
int  erasor_synchronize(erasor_handle_t h);

/* ---- the per-frame path, in the reference's call order ------------------------------------ */
/* replaces ERASOR::set_inputs(map_voi, query_voi) (erasor.cpp:57-85): both clouds already in the
 * egocentric body frame.  Builds both R-PODs (bin of every point, per-bin min/max z and count). */
int erasor_set_inputs(erasor_handle_t h, const float* map_voi_xyzi, size_t n_map,
                      const float* query_voi_xyzi, size_t n_query, int ptr_kind);
/* replaces compare_vois_and_revert_ground(frame) [version 2, erasor.cpp:332-434] and
 * compare_vois_and_revert_ground_w_block(frame) [version 3, erasor.cpp:438-571]:
 * Scan Ratio Test, status per bin, R-GPF on the flagged bins, selection. */
int erasor_compare(erasor_handle_t h, int version, int frame);
/* sizes of the four output clouds of the last compare (so the caller can allocate) */
int erasor_get_output_sizes(erasor_handle_t h, size_t* n_arranged, size_t* n_complement,
                            size_t* n_map_rejected, size_t* n_curr_rejected);
/* replaces ERASOR::get_static_estimate(arranged, complement) (erasor.cpp:612-626); output in the
 * reference's order: selected bins theta-major / r-minor, then ground_viz; complement in source order. */
int erasor_get_static_estimate(erasor_handle_t h, float* arranged_xyzi, size_t cap_arranged, size_t* n_arranged,
                               float* complement_xyzi, size_t cap_complement, size_t* n_complement, int ptr_kind);
/* replaces ERASOR::get_outliers(map_rejected, curr_rejected) (erasor.cpp:322-327) */
int erasor_get_outliers(erasor_handle_t h, float* map_rejected_xyzi, size_t cap_map, size_t* n_map_rejected,
                        float* curr_rejected_xyzi, size_t cap_curr, size_t* n_curr_rejected, int ptr_kind);
/* ERASOR::ground_viz (public member, erasor.h:127): ground points of the flagged bins, the tail of `arranged`.
 * ground_xyzi may be NULL to query *n_ground. */
int erasor_get_ground_viz(erasor_handle_t h, float* ground_xyzi, size_t cap, size_t* n_ground, int ptr_kind);
/* Device-resident callers (the OfflineMapUpdater mirror, erasor_updater_*): device pointers to the four output clouds of the
 * last compare, in place -- no copy, no synchronisation.  Sizes: erasor_get_output_sizes.  They live in the handle's own
 * buffers on erasor_stream(h) and are valid until the next erasor_set_inputs / batch call on this handle; work that reads
 * them must be ordered on that stream.  Any pointer may be NULL. */
int erasor_device_outputs(erasor_handle_t h, const float** arranged, const float** complement, const float** map_rejected,
                          const float** curr_rejected);
/* replaces ERASOR::get_max_range() (erasor.cpp:628) */
double erasor_get_max_range(erasor_handle_t h);

/* ---- parity taps (the reference exposes these only as public members / rviz topics) --------- */
/* r_pod_map / r_pod_curr (erasor.h:143-144): bin of every input point (-1: complement / dropped),
 * per-bin min z, max z (NaN where the bin is empty) and count.  Any pointer may be NULL. Host buffers. */
int erasor_get_bins(erasor_handle_t h, int which_cloud, int32_t* bin_of_point, float* min_h, float* max_h, uint32_t* count);
/* per-bin status of the last compare as published on /SCDR/debug/polygons_marker (erasor.cpp:439-441,570) */
int erasor_get_status(erasor_handle_t h, float* status);
/* R-GPF taps: for each bin that ran extract_ground (processing order), its bin id, point count, seed count,
 * LPR height, and per iteration the plane (nx,ny,nz,d) and the ground count.  *n_planes in: capacity, out: count. */
int erasor_get_planes(erasor_handle_t h, int32_t* bin_ids, int32_t* n_points, int32_t* n_seeds, double* lpr_height,
                      double* normal_d /* [n][gf_iter][4] */, int32_t* n_ground /* [n][gf_iter] */, size_t* n_planes);
/* per map_voi point (source order): keep_map = 0 where the point is rejected as dynamic (non-ground point of a
 * flagged bin), is_ground = 1 where R-GPF retained it as ground.  Host buffers, either may be NULL. */
int erasor_get_static_mask(erasor_handle_t h, uint8_t* keep_map, uint8_t* is_ground);
/* events the reference would have thrown / invoked UB on (SURVEY App. B-1, B-3): points with y == -0.0f and
 * x <= -0 (fenced to y = +0), plane fits on an empty set (fenced to normal (0,0,1), d = 0), and sector decisions
 * that stayed ambiguous after double-double arithmetic (never observed). */
int erasor_get_fence_counts(erasor_handle_t h, uint64_t* negzero_points, uint64_t* empty_plane_fits, uint64_t* ambiguous_sector);

/* ---- frame-independent batch mode (north_star: frames shard across GPUs, masks all-gathered) --- */
/* Runs the whole path on n_frames independent (map_voi, query_voi) pairs and writes, for every map point of
 * every frame, keep = 0 where the frame rejects it.  Frame f's map points are
 * map_xyzi[map_offsets[f] .. map_offsets[f+1]) (offsets in points, n_frames+1 entries, host memory);
 * likewise the queries.  keep_mask has map_offsets[n_frames] bytes.  Clouds / mask: host or device (ptr_kind).
 * A batch too large for one submission (more than 2^32 points, or more flagged-bin records than the work queue holds)
 * is split into consecutive sub-batches internally. */
int erasor_process_frames(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets,
                          const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                          uint8_t* keep_mask, int ptr_kind);
/* Same, returning as soon as the work is enqueued on the handle's stream; erasor_wait(h) completes it (and reports its
 * error, if any).  Host buffers must stay valid and -- to actually be asynchronous -- be pinned.  Two or three handles
 * fed round-robin overlap consecutive batches on the GPU (one batch's R-GPF runs under the next one's binning). */
int erasor_process_frames_async(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets,
                                const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                                uint8_t* keep_mask, int ptr_kind);
int erasor_wait(erasor_handle_t h);
/* Multi-GPU exchange helper: fold per-frame keep masks onto the global map (a point survives unless some frame
 * rejected it): global_keep[voi_index[i]] = 0 where keep_mask[i] == 0.  The mask ACCUMULATES over calls -- start a job
 * with erasor_reset_keep_mask.  Indices >= n_global are ignored.  DEVICE pointers; asynchronous on the handle's stream. */
int erasor_fold_keep_masks(erasor_handle_t h, const uint8_t* keep_mask, const uint32_t* voi_index, size_t n, uint8_t* global_keep, size_t n_global);
int erasor_reset_keep_mask(erasor_handle_t h, uint8_t* global_keep, size_t n_global);   /* global_keep[] = 1; DEVICE pointer, asynchronous */
/* erasor_process_frames with the fold done in R-GPF's epilogue (no extra pass over the masks): what a rank of the
 * frame-sharded job runs per batch.  voi_index (global index of every VoI point, map_offsets[n_frames] entries) and
 * global_keep: DEVICE.  global_keep accumulates (see erasor_reset_keep_mask). */
int erasor_process_frames_fold(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets,
                               const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                               uint8_t* keep_mask, int ptr_kind,
                               const uint32_t* voi_index, uint8_t* global_keep, size_t n_global);
int erasor_process_frames_fold_async(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets,
                                     const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                                     uint8_t* keep_mask, int ptr_kind,
                                     const uint32_t* voi_index, uint8_t* global_keep, size_t n_global);
/* per-frame counters of the last erasor_process_frames / erasor_process_nodes: flagged bins and rejected points (host arrays of n_frames) */
int erasor_get_frame_stats(erasor_handle_t h, uint32_t* n_flagged_bins, uint32_t* n_rejected_points);

/* ---- map-resident frame-independent mode: the global map is uploaded once, per node only pose + query cross PCIe ---- */
/* The initial map of OfflineMapUpdater::load_global_map (OfflineMapUpdater.cpp:107-167), origin frame, resident in HBM,
 * together with its global keep mask (one byte per map point, 1 = static so far).  One map may be attached to any
 * number of handles on the same device. */
typedef struct erasor_map_ctx* erasor_map_t;
int    erasor_map_create(const float* map_xyzi, size_t n_map, int ptr_kind, int device, erasor_map_t* out);
void   erasor_map_destroy(erasor_map_t m);
size_t erasor_map_size(erasor_map_t m);
int    erasor_map_reset_keep(erasor_map_t m);                              /* keep[] = 1 (synchronous) */
int    erasor_map_get_keep(erasor_map_t m, uint8_t* keep, int ptr_kind);   /* synchronous copy; wait for the handles first */
uint8_t*     erasor_map_keep_device(erasor_map_t m);                       /* the mask in HBM (n_map bytes) */
const float* erasor_map_points_device(erasor_map_t m);
int    erasor_attach_map(erasor_handle_t h, erasor_map_t m);
/* n_frames nodes against the attached map, every one tested against the same (initial) map.  For node f:
 *   poses7[7 f .. 7 f + 7) = msg->odom, body -> origin, x y z qx qy qz qw (HOST memory; OfflineMapUpdater.cpp:219);
 *   query cloud = query_xyzi[query_offsets[f] .. query_offsets[f+1]): the scan as callback_node hands it to
 *   ERASOR::set_inputs, i.e. voxelised and in the body frame (OfflineMapUpdater.cpp:237-241).
 * On the device, per node: fetch_VoI (OfflineMapUpdater.cpp:381-438: radius cut at voi_max_range around the body position
 * in double, origin -> body transform; <= 0 selects /erasor/max_range) fused into the polar binning, then SRT and R-GPF
 * as in erasor_process_frames.  Results:
 *   - the map's keep mask &= this batch's verdicts (always; written by R-GPF's epilogue);
 *   - frame_keep (nullable): n_frames x n_map bytes, frame f's keep mask over the GLOBAL map indices
 *     (1 also for points outside the node's VoI);
 *   - keep_out (nullable): copy of the map's keep mask after this batch (n_map bytes).
 * query_xyzi / frame_keep / keep_out: host or device (ptr_kind); host buffers should be pinned.  With ERASOR_PTR_QUERY_XYZ
 * in ptr_kind, query_xyzi holds 3 floats per point. */
int erasor_process_nodes(erasor_handle_t h, const double* poses7, const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                         double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind);
int erasor_process_nodes_async(erasor_handle_t h, const double* poses7, const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                               double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind);
/* per-node counters of the last erasor_process_nodes / erasor_process_scans: points inside the VoI (|map_voi_|), flagged
 * bins, rejected points */
int erasor_get_node_stats(erasor_handle_t h, uint32_t* n_voi_points, uint32_t* n_flagged_bins, uint32_t* n_rejected_points);

/* Node mode on raw scans.  What callback_node does to a scan before ERASOR::set_inputs (OfflineMapUpdater.cpp:237-241),
 * on the device and for the whole batch in one launch: query_f = transform(voxelize_preserving_labels(scan_f,
 * query_voxel_size), lidar2body), each scan on its own pcl::VoxelGrid (a scan whose grid overflows int32 passes unfiltered,
 * an empty scan gives an empty query).  Then exactly erasor_process_nodes on those queries: same outputs, same counters.
 *   scans[scan_offsets[f] .. scan_offsets[f+1]): scan f in the LiDAR frame, x y z i (16 bytes per point), or packed x y z
 *   (12 bytes) with ERASOR_PTR_QUERY_XYZ in ptr_kind.  The masks never read a query's intensity, so labels are not restored.
 * The step needs no device -> host read-back of the voxel counts: the host cuts the query work from the raw scan sizes,
 * the device clamps it to the counts.  Invalid voxel size, poses or offsets: ERASOR_E_INVALID. */
typedef struct {
    double query_voxel_size;       /* /erasor/query_voxel_size (> 0) */
    double lidar2body[7];          /* /tf/lidar2body: x y z qx qy qz qw */
} erasor_scan_params_t;
int erasor_process_scans(erasor_handle_t h, const erasor_scan_params_t* sp, const double* poses7, const float* scans,
                         const uint64_t* scan_offsets, int n_frames, double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind);
int erasor_process_scans_async(erasor_handle_t h, const erasor_scan_params_t* sp, const double* poses7, const float* scans,
                               const uint64_t* scan_offsets, int n_frames, double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out,
                               int ptr_kind);
/* The voxelised body-frame queries of the last erasor_process_scans submission (its last sub-batch when the batch was split),
 * x y z per point (HOST, 3 floats each), frame after frame, each in voxel-key order; offsets[0 .. n + 1) receives the
 * per-frame starts (n = frames of that submission; HOST, n + 1 entries).  xyz == NULL: offsets only.  Synchronous. */
int erasor_get_scan_queries(erasor_handle_t h, float* xyz, size_t cap, uint64_t* offsets);
/* OfflineMapUpdater::save_static_map for the attached map (OfflineMapUpdater.cpp:174-196, no file): voxelize_preserving_labels
 * of the map points whose keep byte is 1, in map order, at voxel_size, labels restored (HOST out_xyzi, x y z i).  *n receives
 * the size; out_xyzi == NULL (or cap < *n with ERASOR_E_CAPACITY) is the size query.  Synchronous. */
int erasor_save_static_map(erasor_handle_t h, float voxel_size, float* out_xyzi, size_t cap, size_t* n);

/* ---- the path's single collective, behind the C ABI (north_star: one NCCL all-gather of the static masks) ------------ */
/* A communicator owned by the handle (NCCL is loaded with dlopen("libnccl.so.2") on first use).  Rank 0 calls
 * erasor_comm_unique_id and ships the 128 bytes to the other ranks by whatever means the host program has
 * (MPI, torch.distributed, a file); every rank then calls erasor_comm_init (collective). */
#define ERASOR_COMM_ID_BYTES 128
int erasor_comm_unique_id(uint8_t* id128);
int erasor_comm_init(erasor_handle_t h, const uint8_t* id128, int n_ranks, int rank);
int erasor_comm_destroy(erasor_handle_t h);
/* global_keep (DEVICE, n_global bytes, this rank's folded mask) <- AND over all ranks: the bytes are packed to bits
 * (8x less traffic), all-gathered with ONE ncclAllGather over NVLink and AND-ed + unpacked by a library kernel.
 * Asynchronous on the handle's stream.  Without a communicator (single GPU) it is a no-op. */
int erasor_allgather_and_keep(erasor_handle_t h, uint8_t* global_keep, size_t n_global);
/* The local half of that exchange on its own: out[i] = AND over r of masks[r][i] (DEVICE, contiguous [n_masks][n] bytes),
 * through the same bit-pack / AND / unpack kernels.  For callers with their own transport, and for single-GPU tests. */
int erasor_and_keep_masks(erasor_handle_t h, const uint8_t* masks, int n_masks, size_t n, uint8_t* out);

/* ---- instrumentation ---------------------------------------------------------------------- */
/* per flagged bin of the last run: point count and SM cycles per R-GPF phase (load + index sort, z sort, seeds,
 * accumulate, SVD + plane, classify + compact, outputs) plus the Jacobi sweep count in slot 7.  *n in: capacity, out: count. */
int erasor_get_rgpf_profile(erasor_handle_t h, uint32_t* n_points, uint32_t* prof8, size_t* n);
/* SM cycles per phase of the SRT kernel (K3), frame 0 of the last run: status passes, chunk-row prefixes, flagged-bin scan +
 * record base, map scatter offsets, records + R-GPF queue, query scatter offsets; slots 6-7 reserved (host array of 8). */
int erasor_get_srt_profile(erasor_handle_t h, uint32_t* cycles8);
/* number of kernels this library launched on the handle since creation */
uint64_t erasor_kernel_launch_count(erasor_handle_t h);
/* CUDA-event time (ms) spent in the binning kernel (K1) since the last reset, and its launch count */
int erasor_get_kernel_time_ms(erasor_handle_t h, int kernel_id, double* total_ms, uint64_t* launches);
int erasor_reset_kernel_times(erasor_handle_t h, int enable_timing);

/* ============================================================================================
 * The caller, device-resident: erasor::OfflineMapUpdater (reference include/erasor/OfflineMapUpdater.h,
 * src/offline_map_updater/src/OfflineMapUpdater.cpp) with ROS stripped -- SURVEY.md section 8f rows 1-3.
 * The global map lives in HBM; per node only the raw scan and the pose cross PCIe.
 * ========================================================================================== */
typedef struct erasor_updater_ctx* erasor_updater_t;

typedef struct {
    double query_voxel_size;   /* /MapUpdater/query_voxel_size   OfflineMapUpdater.cpp:66 */
    double map_voxel_size;     /* /MapUpdater/map_voxel_size     :67 (unused by the path) */
    int    removal_interval;   /* /MapUpdater/removal_interval   :69 */
    int    is_large_scale;     /* /large_scale/is_large_scale    :75 */
    double submap_size;        /* /large_scale/submap_size       :76 */
    double max_range;          /* /erasor/max_range as read by the updater, default 60.0  :78 */
    int    version;            /* /erasor/version                :81 */
    int    pad_;
    double lidar2body[7];      /* /tf/lidar2body  x y z qx qy qz qw   :89-104 */
} erasor_updater_params_t;

/* replaces OfflineMapUpdater::OfflineMapUpdater() = set_params + load_global_map + new ERASOR (:5-32, 63-167);
 * the initial map is handed over as a host cloud instead of a PCD path. */
int  erasor_updater_create(const erasor_updater_params_t* up, const erasor_params_t* ep, const float* initial_map_xyzi, size_t n_map,
                           int device, erasor_updater_t* out);
void erasor_updater_destroy(erasor_updater_t u);
/* load_global_map again (:107-167) on a live updater: new initial map, counters reset, device buffers kept */
int  erasor_updater_reset(erasor_updater_t u, const float* initial_map_xyzi, size_t n_map);
const char* erasor_updater_last_error(erasor_updater_t u);
/* replaces OfflineMapUpdater::callback_node(msg) (:203-330): seq = msg->header.seq, odom7 = msg->odom as x y z qx qy qz qw
 * (body -> origin), lidar = msg->lidar in the LIDAR frame.  *processed = 1 when the node was processed (every
 * removal_interval-th call), 0 for the reference's "PASS!". */
int  erasor_updater_process_node(erasor_updater_t u, int seq, const double* odom7, const float* lidar_xyzi, size_t n_lidar, int ptr_kind,
                                 int* processed);
/* Optional look-ahead for callers that know the coming nodes' scans (file-based / offline runs: the reference replays a rosbag,
 * OfflineMapUpdater.cpp:203): starts a scan's upload, voxelize_preserving_labels and lidar -> body (:237-241) on a second stream,
 * so that it runs under the path of the node being processed.  Two look-aheads can be pending: hand in node k + 1's scan, then
 * call erasor_updater_process_node for node k.  A process_node call given the same (pointer, n, ptr_kind) consumes the
 * look-ahead -- results are identical with and without; one that matches nothing runs the usual way.  The scan buffer must
 * stay valid and unchanged until it has been consumed; a DEVICE scan must be complete (its producer synchronised) before the
 * call, because the look-ahead reads it on the updater's own second stream. */
int  erasor_updater_prefetch_scan(erasor_updater_t u, const float* lidar_xyzi, size_t n_lidar, int ptr_kind);
int  erasor_updater_map_size(erasor_updater_t u, size_t* n);
/* clouds of the last processed node (parity taps): 0 map_arranged_, 1 map_voi_ (body), 2 query_voi_ (body),
 * 5 map_rejected_ (origin), 7 map_outskirts_, 8 map_arranged_complement_ (large-scale).  xyzi may be NULL to query *n. */
int  erasor_updater_get_cloud(erasor_updater_t u, int which, float* xyzi, size_t cap, size_t* n, int ptr_kind);
/* replaces OfflineMapUpdater::save_static_map(voxel_size) minus the PCD write (:174-196) */
int  erasor_updater_save_static_map(erasor_updater_t u, float voxel_size, float* out_xyzi, size_t cap, size_t* n);
/* erasor_utils::voxelize_preserving_labels on a free-standing host cloud (erasor_utils.cpp:80-114) */
int  erasor_updater_voxelize(erasor_updater_t u, const float* xyzi, size_t n_in, float leaf, float* out_xyzi, size_t cap, size_t* n);
/* mapgen's per-node producer on the device (reference src/mapgen/mapgen.hpp:198-239): 2.7 m vehicle-body cut, 1.73 m lift,
 * pose transform, voxelize_preserving_labels at 0.2 m -> cloud_curr.  out_xyzi needs room for n_lidar points (cap). */
int  erasor_updater_mapgen_node(erasor_updater_t u, const double* odom7, const float* lidar_xyzi, size_t n_lidar, int ptr_kind,
                                float* out_xyzi, size_t cap, size_t* n);
/* the ERASOR handle inside the updater (for the parity taps above) */
erasor_handle_t erasor_updater_erasor(erasor_updater_t u);
uint64_t erasor_updater_kernel_launch_count(erasor_updater_t u);
/* phase boundaries (ns, %globaltimer of CTA 0) of the last fused prologue launch -- the per-node cooperative kernel that
 * voxelises the scan and cuts the VoI: [0] start, [1] min/max + partition count, [2] set-up + chunk offsets, [3] keys + partition
 * scatter, [4+2p] histogram + offsets of radix pass p, [5+2p] its scatter, [12] sort done, [13] run heads counted, [14] heads
 * scattered, [15] centroids + labels written. */
int erasor_updater_get_fused_profile(erasor_updater_t u, uint64_t* ns16);

#ifdef __cplusplus
}
#endif
#endif /* ERASOR_B200_H */
