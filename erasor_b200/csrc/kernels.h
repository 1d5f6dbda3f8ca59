// kernels.h -- launch wrappers of the path's kernels (definitions in kernels.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

#include "device_types.h"

namespace erasor {

struct CopyJob {
    const float4* src;
    float4*       dst;
    uint32_t      n;
    uint32_t      pad_;
};

size_t k1_smem_bytes(int R, int B);
bool   k1_big_tables(int R, int B);      // one 1024-thread CTA per SM instead of four 256-thread ones
size_t k3_smem_bytes(int B);

cudaError_t launch_init_tables(cudaStream_t st, uint32_t* zmin, uint32_t* zmax, size_t n, uint32_t* cnt, size_t n_cnt, uint32_t* n_recs,
                               uint32_t* frame_rejected, uint32_t* n_flagged, int F, uint32_t* queue);

// poses != null: node mode (the map cloud is the resident global map; fetch_VoI's cut + transform fused into the binning)
cudaError_t launch_k1(cudaStream_t st, const BinTablesView& T, const float4* map_pts, const float4* qry_pts,
                      const ChunkDesc* chunks, int n_chunks, uint16_t* bin_map, uint16_t* bin_qry, uint32_t* ch_cnt,
                      uint32_t* zmin, uint32_t* zmax, uint32_t* cnt_tab, int B, int F, unsigned long long* fence, const NodePose* poses,
                      uint32_t* list_idx /*node mode: map index of every VoI point, per chunk*/, uint32_t* list_cnt /*node mode: VoI points per chunk*/,
                      bool qry_xyz = false /*the query cloud is packed x y z, 12 bytes per point (mask modes)*/);

cudaError_t launch_k3(cudaStream_t st, const SrtParams& P, int F, const uint32_t* chunk_range, uint32_t* ch_cnt,
                      const uint32_t* zmin, const uint32_t* zmax, const uint32_t* frame_off, const uint32_t* cnt, uint32_t* dst_start,
                      uint8_t* status, uint8_t* action, uint32_t* flag_slot, uint32_t* n_flagged, uint32_t* frame_rec_base,
                      FlagRec* recs, uint32_t* n_recs, uint32_t rec_capacity, uint32_t* queue, uint32_t* bucket_list);

// mask modes: Scan Ratio Test + stable scatter of the flagged bins + R-GPF records / queue in one kernel (no k3_srt launch);
// ch_cnt holds K1's raw per-chunk counts
cudaError_t launch_k2_srt(cudaStream_t st, const SrtParams& P, int F, const ChunkDesc* chunks, const uint32_t* chunk_range, uint32_t n_chunks_map,
                          const uint16_t* bin_ids, const float4* pts, const NodePose* poses, const uint32_t* ch_cnt, const uint32_t* zmin,
                          const uint32_t* zmax, const uint32_t* cnt, const uint32_t* frame_off, uint32_t* n_flagged, FlagRec* recs, uint32_t* n_recs,
                          uint32_t rec_capacity, uint32_t* queue, uint32_t* bucket_list, float4* out_pts, uint32_t* out_src,
                          const uint32_t* list_idx, const uint32_t* list_cnt);

// flag_slot == null: every bin of dst_start's cloud that has an offset is scattered (cloud mode); otherwise the flagged bins only
cudaError_t launch_k2(cudaStream_t st, const ChunkDesc* chunks, uint32_t chunk_base, uint32_t n_chunks,
                      const uint16_t* bin_ids, const float4* pts, const NodePose* poses, const uint32_t* ch_cnt, const uint32_t* dst_start,
                      const uint32_t* flag_slot, const uint32_t* n_flagged, float4* out_pts, uint32_t* out_src, int B,
                      const uint32_t* list_idx, const uint32_t* list_cnt, int k1_warps /*warps of the K1 launch that wrote the lists (8 or 32)*/);

// cloud mode: both clouds' stable scatters in one launch (chunk rows: map first, then query)
cudaError_t launch_k2_both(cudaStream_t st, const ChunkDesc* chunks, uint32_t n_chunks_map, uint32_t n_chunks_qry, const uint32_t* ch_cnt, int B,
                           const uint16_t* bin_map, const float4* map_pts, const uint32_t* dst_start_map, float4* out_map, uint32_t* src_map,
                           const uint16_t* bin_qry, const float4* qry_pts, const uint32_t* dst_start_qry, float4* out_qry, uint32_t* src_qry);

int k4_num_launches(bool with_class_c);
// sorted_pts / sorted_src: K2's output (bins contiguous in source order + source index of every slot); in_pts is unused
// since K2 also serves mask mode, kept in the signature for ABI stability of the launch wrapper.
// queue / bucket_list: the size-bucketed work queue K3 filled (device_types.h).
cudaError_t launch_k4(cudaStream_t st, cudaStream_t st_b, cudaStream_t st_c, const GpfParams& P, FlagRec* recs, uint32_t* queue,
                      const uint32_t* bucket_list, uint32_t rec_capacity, const float4* sorted_pts, uint32_t* sorted_src, const float4* in_pts, const uint32_t* frame_off,
                      float4* part_pts, uint8_t* keep_mask, uint8_t* ground_mask, uint32_t* frame_rejected, unsigned char* gscratch,
                      int sm_count, unsigned long long* fence, const K4Fold& fold, int classes /*bit 0|1: A and B, bit 2: C*/);

cudaError_t launch_k4b(cudaStream_t st, float leaf, int B, const FlagRec* recs, const uint32_t* n_recs, uint32_t rec_capacity,
                       const uint32_t* cnt, const uint32_t* dst_start, const float4* qry_sorted, const float4* part_pts,
                       float4* vox_pts, uint32_t* vox_cnt, uint32_t* vox_start, unsigned char* gscratch, int grid);

cudaError_t launch_k5(cudaStream_t st, int B, int version, int skip_voxelize, const uint32_t* cnt, const uint32_t* dst_start,
                      const uint8_t* action, const uint32_t* flag_slot, const FlagRec* recs, const uint32_t* n_recs,
                      const uint32_t* vox_cnt, const uint32_t* vox_start, const float4* map_sorted, const float4* qry_sorted,
                      const float4* part_pts, const float4* vox_pts, float4* arranged, float4* map_rej, float4* curr_rej,
                      CopyJob* jobs, uint32_t* out_sizes, uint32_t* tmp, int copy_grid);

cudaError_t launch_fold_keep(cudaStream_t st, const uint8_t* keep, const uint32_t* voi_index, size_t n, uint8_t* global_keep, size_t n_global);
cudaError_t launch_fill_u8(cudaStream_t st, uint8_t* p, size_t n, uint8_t v);
// chunks[first .. first + n): len = min(full length in pad_, what is left of count[frame] from the chunk's start)
cudaError_t launch_clamp_query_chunks(cudaStream_t st, ChunkDesc* chunks, uint32_t first, uint32_t n, const uint32_t* count);
// exchange step of the frame-sharded job: pack the keep bytes into bits, AND the all-gathered words of every rank, unpack
cudaError_t launch_pack_keep_bits(cudaStream_t st, const uint8_t* keep, size_t n, uint32_t* words);
cudaError_t launch_and_unpack_keep(cudaStream_t st, const uint32_t* gathered, int n_ranks, size_t n, uint8_t* keep);

}  // namespace erasor
