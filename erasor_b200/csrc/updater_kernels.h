// updater_kernels.h -- launch wrappers of the caller-side device steps (definitions in updater_kernels.cu)
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace erasor {

struct Mat4 { float m[16]; };            // row-major 4x4, like Eigen::Matrix4f(r, c) = m[4 r + c]

enum { PART_RADIUS = 0, PART_SUBMAP = 1, PART_NOT_NEAR = 2 };
struct PartPred {
    int    kind;
    int    pad_;
    double x, y;                         // criterion point
    double limit;                        // PART_RADIUS: max_dist_square; PART_SUBMAP: submap_size; PART_NOT_NEAR: squared vehicle-body radius
};

struct VoxGrid {                         // pcl::VoxelGrid state of one filter call, kept on the device
    uint32_t mn[3], mx[3];               // order-preserving encodings of the cloud's min / max
    float    leaf, inv;
    int      min_b[3], div[3];
    uint32_t n_vox;
    int      overflow;
    int      npass;                      // 8-bit radix passes the key width needs
    unsigned long long prof[16];         // phase boundaries of the fused kernel's CTA 0 (ns, %globaltimer)
};

constexpr int kFusedMaxGrid = 1024;      // CTAs of the fused kernel (one per SM in practice); sizes the per-CTA min/max partials

// One cooperative launch = erasor_utils::voxelize_preserving_labels of one cloud (U3) and, optionally and independently, one
// stable partition of another (U1: fetch_VoI / set_submap / mapgen's body cut).  Either job may be empty.
struct FusedJob {
    // U3: vout[0..*d_n_out) = voxelised vin[0..vn) in ascending voxel key, labels restored by exact 1-NN, then (xform_out) T_out
    const float4* vin; uint32_t vn; float leaf; VoxGrid* grid; void* vtmp /*voxelize_tmp_bytes(vn)*/; float4* vout; uint32_t* d_n_out;
    Mat4 T_out; int xform_out;
    // U1: pred-true points of pin[0..pn) (optionally through the affine T_sel) to out_sel, the rest to out_rest, both in source
    // order; *d_total_sel receives the number selected
    int has_part; PartPred P; Mat4 T_sel; int xform_sel; const float4* pin; uint32_t pn; uint32_t* chunk_tmp /*partition_tmp_words(pn)*/;
    uint32_t* d_total_sel; float4* out_sel; float4* out_rest;
    // Batched U3 (n_clouds > 0; no U1 job): vin[cloud_off[f] .. cloud_off[f + 1]) for f < n_clouds are independent clouds, each
    // voxelised on its own grid grid[f] exactly as one call would; cloud f's voxels go to vout[cloud_off[f] ..) in ascending
    // key, their number to cloud_nvox[f]; *d_n_out receives the total.  cloud_off lives in device memory.  restore_labels = 0
    // skips the 1-NN label restore (the centroid keeps the averaged fourth component).  n_clouds = 0: the single-cloud job above.
    uint32_t n_clouds = 0; const uint32_t* cloud_off = nullptr; uint32_t* cloud_nvox = nullptr; int restore_labels = 1;
};
size_t partition_tmp_words(uint32_t n);
size_t voxelize_tmp_bytes(uint32_t n, uint32_t n_clouds = 1);
cudaError_t launch_node_fused(cudaStream_t st, const FusedJob& job, int sm_count, int max_ctas = 0 /*0: as many as the job wants, up to one per SM*/);

cudaError_t launch_affine_copy(cudaStream_t st, const Mat4& T, bool do_transform, const float4* in, float4* out, uint32_t n);
// packed x y z (12 bytes per point) -> float4 with w = 0
cudaError_t launch_expand_xyz(cudaStream_t st, const float* in, float4* out, uint32_t n);
// stable compaction: out[0..*d_n) = the points of pts[0..n) whose keep byte is nonzero, in order; tmp: partition_tmp_words(n)
cudaError_t launch_compact_keep(cudaStream_t st, const float4* pts, const uint8_t* keep, uint32_t n, float4* out, uint32_t* d_n, uint32_t* tmp);

// epilogue of callback_node (OfflineMapUpdater.cpp:281-290) in one launch: up to four copy segments, each optionally through
// the float affine T (pcl::transformPointCloud)
struct CopySeg { const float4* src; float4* dst; uint32_t n; int xform; };
cudaError_t launch_copy_segments(cudaStream_t st, const Mat4& T, const CopySeg* segs, int n_segs);

}  // namespace erasor
