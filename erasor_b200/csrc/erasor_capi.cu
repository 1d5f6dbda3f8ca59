// erasor_capi.cu -- the extern "C" boundary (include/erasor_b200.h): context, HBM buffers, launch order.
// There is no host compute path in this file: every entry point either launches the sm_100a kernels of
// kernels.cu or fails with an error code.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>      // types only: the library is loaded with dlopen on first use (erasor_comm_*)

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "../../include/erasor_b200.h"
#include "binning_tables.h"
#include "device_types.h"
#include "kernels.h"
#include "pose_math.h"

using namespace erasor;

namespace {

thread_local std::string g_create_error;

struct DevBuf {
    void*     p = nullptr;
    size_t    cap = 0;
    uint64_t* epoch = nullptr;   // the owning handle's allocation epoch: bumped on every (re)allocation, captured graphs hold raw pointers
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (epoch) ++*epoch;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = want;
        return cudaSuccess;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinnedBuf {
    void*  p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = want;
        return cudaSuccess;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

constexpr int kNumTimers = 6;   // 0 whole pipeline, 1..5 = K1..K5
constexpr size_t kMaxRecords = (size_t)1 << 21;   // flagged-bin records of one submission (larger batches are split)

struct Timer {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    double   total_ms = 0;
    uint64_t launches = 0;
};

}  // namespace

struct erasor_map_ctx {
    int          device = 0;
    float4*      d_pts = nullptr;
    uint8_t*     d_keep = nullptr;
    size_t       n = 0;
    cudaStream_t st = nullptr;
    std::string  err;
};

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char*  (*GetErrorString)(ncclResult_t) = nullptr;
};

struct erasor_ctx {
    erasor_params_t p{};
    int             device = 0;
    cudaStream_t    stream = nullptr, stream_a = nullptr, stream_b = nullptr, stream_c = nullptr;   // a/b/c: concurrent R-GPF size classes (high priority)
    cudaEvent_t     ev_fork = nullptr, ev_join_a = nullptr, ev_join_b = nullptr, ev_join_c = nullptr;
    int             sm_count = 148;
    std::string     err;
    HostBinTables   tables;
    DevBuf          d_ring, d_pos, d_neg, d_guard;
    BinTablesView   view{};
    int             B = 0;
    uint64_t        alloc_epoch = 0;           // bumped by every DevBuf (re)allocation of this handle

    // per-batch buffers
    DevBuf d_map_in, d_qry_in;                 // staging when the caller's clouds are host memory
    DevBuf d_bin_map, d_bin_qry;               // uint16 bin id per point
    DevBuf d_chunks, d_chunk_range, d_frame_off;
    DevBuf d_chcnt, d_zmin, d_zmax, d_cnt, d_dst_start, d_status, d_action, d_flag_slot, d_nflag;
    DevBuf d_recs, d_nrecs, d_frame_rej, d_frame_rec_base, d_queue, d_bucket;
    DevBuf d_map_sorted, d_map_src, d_qry_sorted, d_qry_src, d_part, d_scratch;
    DevBuf d_keep, d_ground;
    DevBuf d_arranged, d_map_rej, d_curr_rej, d_jobs, d_out_sizes, d_k5tmp;
    DevBuf d_vox, d_vox_cnt, d_vox_start, d_vox_scratch;
    DevBuf d_fence;                            // 4 x u64: negzero, empty fits, ambiguous, slow-path points
    DevBuf d_poses;                            // node mode: NodePose per frame
    DevBuf d_list_idx, d_list_cnt;             // node mode: per chunk, the map index of every VoI point (dense, map order) and their number
    DevBuf d_pack, d_gather;                   // exchange step: packed keep bits of this rank / of every rank
    DevBuf d_scan_f4, d_scan_q, d_scan_grid, d_scan_tmp, d_scan_cnt;   // erasor_process_scans: scans widened to float4 (packed x y z input),
                                                                       // voxelised body-frame queries (at the raw scans' offsets), per-scan
                                                                       // VoxelGrid state, voxeliser scratch, voxels per scan (+ total)
    DevBuf d_sv_pts, d_sv_tmp, d_sv_out, d_sv_grid, d_sv_vtmp;        // erasor_save_static_map: kept points, compaction / voxeliser state
    PinnedBuf h_stage, h_pose, h_words;        // h_words: small device -> host read-backs of a submission (pinned: an asynchronous copy into
                                               // pageable memory blocks the launching thread until the whole stream has drained, which
                                               // serialised overlapped handles)
    std::vector<DevBuf*> all_bufs() {
        return {&d_ring, &d_pos, &d_neg, &d_guard, &d_map_in, &d_qry_in, &d_bin_map, &d_bin_qry, &d_chunks, &d_chunk_range, &d_frame_off, &d_chcnt, &d_zmin,
                &d_zmax, &d_cnt, &d_dst_start, &d_status, &d_action, &d_flag_slot, &d_nflag, &d_recs, &d_nrecs, &d_queue, &d_bucket, &d_frame_rej,
                &d_map_sorted, &d_map_src, &d_qry_sorted, &d_qry_src, &d_part, &d_scratch, &d_keep, &d_ground, &d_arranged, &d_map_rej, &d_curr_rej,
                &d_jobs, &d_out_sizes, &d_k5tmp, &d_fence, &d_vox, &d_vox_cnt, &d_vox_start, &d_vox_scratch, &d_frame_rec_base, &d_poses, &d_list_idx, &d_list_cnt, &d_pack,
                &d_gather, &d_scan_f4, &d_scan_q, &d_scan_grid, &d_scan_tmp, &d_scan_cnt, &d_sv_pts, &d_sv_tmp, &d_sv_out, &d_sv_grid, &d_sv_vtmp};
    }

    // batch geometry of the last run
    int      F = 0;
    size_t   NM = 0, NQ = 0;                   // points of the map-side arrays (node mode: F * n_map) / of the queries
    uint32_t n_chunks_map = 0, n_chunks_qry = 0;
    uint32_t rec_capacity = 0;
    const float4* cur_map = nullptr;
    const float4* cur_qry = nullptr;
    bool     qry_xyz = false;                  // the staged query cloud is packed x y z (ERASOR_PTR_QUERY_XYZ, mask modes)
    std::vector<uint64_t> map_off, qry_off;
    int      desc_mode = -1;                   // mode the uploaded chunk descriptors were built for (-1: none; 0 cloud, 1 batch masks, 2 node masks,
                                               // 3 node masks on raw scans: query chunks clamped on the device)
    uint64_t desc_epoch = 0;                   // bumped whenever the descriptors are rebuilt (invalidates cached graphs)
    int      stat_F = 0;                       // frames of the last batch call (all its sub-batches): extent of the per-frame counters
    int      f0 = 0;                           // first frame of the sub-batch being submitted
    struct StepGraph { const void* ptr[8]; size_t fold_n; int kind, mode, f0; uint64_t epoch, alloc; double scan[8]; cudaGraphExec_t exec; };
    std::vector<StepGraph> graphs;             // captured mask-mode steps, one per (pointers, geometry)
    bool     use_graphs = true;
    int      ctas_per_sm = 4;                  // K1 / K2 grid target: one wave of sm_count * ctas_per_sm CTAs (ERASOR_B200_CTAS_PER_SM)
    bool     fused_srt = true;                 // mask modes: Scan Ratio Test inside the scatter kernel (ERASOR_B200_UNFUSED_SRT=1: separate k3_srt)
    uint64_t graph_kernel_nodes = 0;
    bool     pending = false;                  // an asynchronous submission has not been waited for yet
    // R-GPF class C (bins beyond 2560 points) is launched only while such bins are being seen (its CTAs need whole SMs even to
    // find their queue empty, which serialises overlapped submissions); if one turns up unannounced, erasor_wait runs the class.
    int      class_c_state = -1;               // -1 unknown (launch it), 0 none in the last run, > 0 seen
    uint32_t class_c_count_host = 0;           // queue[kBucketC0] of the submission in flight
    struct { bool with_c = true, host = false; int mode = 1; uint8_t* d_keep = nullptr; uint8_t* user_keep = nullptr; size_t n_keep = 0;
             uint8_t* keep_out = nullptr; size_t n_map_global = 0; K4Fold fold{nullptr, nullptr, 0u, 0u}; } last;

    // node mode
    erasor_map_ctx* map = nullptr;
    int      scan_F = 0;                       // frames of the last submission if it came from erasor_process_scans (0: it did not)

    // exchange
    ncclComm_t comm = nullptr;
    int        comm_ranks = 1, comm_rank = 0;

    // single-frame state machine
    int      stage = 0;                        // 0: nothing, 1: inputs set, 2: compared
    uint32_t out_sizes[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // arranged, complement, map_rejected, curr_rejected, ground_viz
    uint32_t complement_start = 0;
    uint32_t n_recs_host = 0;                  // (cloud mode; the mask modes read back into h_words)
    volatile uint32_t* words() { return h_words.as<volatile uint32_t>(); }   // [0] flagged-bin records, [1] class-C bins of the submission in flight

    uint64_t launches = 0;
    bool     timing = false;
    Timer    timers[kNumTimers];
};

namespace {

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e__);                          \
            return ERASOR_E_CUDA;                                                                  \
        }                                                                                          \
    } while (0)

// NCCL is bound at run time: single-GPU users need no libnccl, and inside a torch process dlopen returns the copy torch
// already loaded (same soname), so the process keeps exactly one NCCL.
NcclApi* nccl_api(std::string& err) {
    static NcclApi api;
    static bool tried = false;
    if (api.lib) return &api;
    if (tried) { err = "libnccl.so.2 could not be loaded"; return nullptr; }
    tried = true;
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) { err = std::string("dlopen(libnccl.so.2): ") + dlerror(); return nullptr; }
    api.GetUniqueId    = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(lib, "ncclGetUniqueId"));
    api.CommInitRank   = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(lib, "ncclCommInitRank"));
    api.CommDestroy    = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(lib, "ncclCommDestroy"));
    api.AllGather      = reinterpret_cast<decltype(api.AllGather)>(dlsym(lib, "ncclAllGather"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(lib, "ncclGetErrorString"));
    if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllGather || !api.GetErrorString) { err = "libnccl.so.2 lacks a required symbol"; return nullptr; }
    api.lib = lib;
    return &api;
}

struct Scope {   // optional CUDA-event bracket around a kernel (timing == true only)
    erasor_ctx* h; int id; cudaEvent_t a = nullptr, b = nullptr;
    Scope(erasor_ctx* h_, int id_) : h(h_), id(id_) {
        if (h->timing) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, h->stream); }
    }
    ~Scope() {
        if (h->timing) { cudaEventRecord(b, h->stream); h->timers[id].pending.emplace_back(a, b); }
    }
};

void drain_timers(erasor_ctx* h) {
    for (int i = 0; i < kNumTimers; ++i) {
        for (auto& pr : h->timers[i].pending) {
            cudaEventSynchronize(pr.second);
            float ms = 0;
            cudaEventElapsedTime(&ms, pr.first, pr.second);
            h->timers[i].total_ms += ms;
            h->timers[i].launches += 1;
            cudaEventDestroy(pr.first); cudaEventDestroy(pr.second);
        }
        h->timers[i].pending.clear();
    }
}

uint32_t choose_chunk(const erasor_ctx* h, const uint64_t* map_off, const uint64_t* qry_off, int F) {
    // Chunk = one CTA of K1 and of K2.  Aim at ONE wave of CTAs (4 resident per SM for both kernels): a second, nearly empty
    // wave costs a whole CTA latency.  Frames are chunked separately, so the count is taken over the real frame sizes.
    // The dense per-chunk count rows cost 4*(B+1) bytes each: keep the chunk at >= 5*B points (<= 5 % extra traffic).
    const size_t total = (size_t)(map_off[F] + qry_off[F]);
    const size_t slots = (size_t)h->sm_count * (k1_big_tables(h->p.num_rings, h->B) ? 1 : h->ctas_per_sm);
    auto count = [&](size_t ch) {
        size_t n = 0;
        for (int f = 0; f < F; ++f) n += (size_t)((map_off[f + 1] - map_off[f] + ch - 1) / ch) + (size_t)((qry_off[f + 1] - qry_off[f] + ch - 1) / ch);
        return n;
    };
    const size_t cap = 65536;
    size_t ch = std::max<size_t>(total / slots + 1, std::max<size_t>(2048, (size_t)5 * h->B));
    ch = std::min<size_t>((ch + 127) & ~(size_t)127, cap);
    if (count(cap) <= slots) {
        while (ch < cap && count(ch) > slots) ch = std::min<size_t>(cap, (ch + std::max<size_t>(128, ch / 64) + 127) & ~(size_t)127);
    } else {
        ch = cap;      // several waves anyway
    }
    return (uint32_t)ch;
}

// Build chunk descriptors + per-frame chunk ranges + frame offsets, upload them, size every buffer.
// mode 0: single frame, cloud outputs; 1: batch of (map_voi, query_voi) pairs, masks; 2: node mode -- map_off is
// {0, n_map, 2 n_map, ...}: every frame scans the whole resident map (fetch_VoI fused into K1), masks on global indices.
int prepare_batch(erasor_ctx* h, const uint64_t* map_off, const uint64_t* qry_off, int F, int mode) {
    if (F <= 0) { h->err = "n_frames must be positive"; return ERASOR_E_INVALID; }
    const size_t NM = map_off[F], NQ = qry_off[F];
    if (NM >= 0xFFFFFFF0ull || NQ >= 0xFFFFFFF0ull) { h->err = "batch exceeds 2^32 points; split it"; return ERASOR_E_INVALID; }
    for (int f = 0; f < F; ++f)
        if (map_off[f + 1] < map_off[f] || qry_off[f + 1] < qry_off[f]) { h->err = "offsets must be non-decreasing"; return ERASOR_E_INVALID; }
    const int B = h->B;
    // per-frame counters span the caller's whole batch (all its sub-batches), so they are sized before the shortcut below
    CK(h->d_nflag.ensure(sizeof(uint32_t) * (size_t)std::max(h->stat_F, h->f0 + F)));
    CK(h->d_frame_rej.ensure(sizeof(uint32_t) * (size_t)std::max(h->stat_F, h->f0 + F)));
    // same batch geometry as the previous call (the usual case when a caller streams equally-shaped batches):
    // the chunk descriptors already on the device are still valid -- skip rebuild, upload and the staging sync
    if (h->desc_mode == mode && h->F == F && h->map_off.size() == (size_t)F + 1 && h->qry_off.size() == (size_t)F + 1 &&
        std::equal(map_off, map_off + F + 1, h->map_off.begin()) && std::equal(qry_off, qry_off + F + 1, h->qry_off.begin()))
        return ERASOR_OK;
    h->desc_mode = -1;
    h->F = F; h->NM = NM; h->NQ = NQ;
    h->map_off.assign(map_off, map_off + F + 1);
    h->qry_off.assign(qry_off, qry_off + F + 1);
    const uint32_t CH = choose_chunk(h, map_off, qry_off, F);
    const bool node = mode >= 2;

    std::vector<ChunkDesc> chunks;
    std::vector<uint32_t>  range(2 * (size_t)(F + 1)), foff(2 * (size_t)(F + 1));
    chunks.reserve((NM + NQ) / CH + 2 * (size_t)F + 2);
    for (int c = 0; c < 2; ++c) {
        const uint64_t* off = c == 0 ? map_off : qry_off;
        for (int f = 0; f < F; ++f) {
            range[(size_t)c * (F + 1) + f] = (uint32_t)chunks.size();
            foff[(size_t)c * (F + 1) + f]  = (uint32_t)off[f];
            for (uint64_t b = off[f]; b < off[f + 1]; b += CH) {
                ChunkDesc d{};
                d.len = (uint32_t)std::min<uint64_t>(CH, off[f + 1] - b);
                d.frame = (uint32_t)f; d.cloud = (uint32_t)c;
                d.bin_begin = (uint32_t)b; d.out_base = (uint32_t)off[f];
                d.pad_ = d.len;
                if (node && c == 0) { d.begin = (uint32_t)(b - off[f]); d.frame_begin = 0u; }      // source = the resident map itself
                else                { d.begin = (uint32_t)b; d.frame_begin = (uint32_t)off[f]; }
                chunks.push_back(d);
            }
        }
        range[(size_t)c * (F + 1) + F] = (uint32_t)chunks.size();
        foff[(size_t)c * (F + 1) + F]  = (uint32_t)off[F];
        if (c == 0) h->n_chunks_map = (uint32_t)chunks.size();
    }
    h->n_chunks_qry = (uint32_t)chunks.size() - h->n_chunks_map;
    const size_t n_chunks = chunks.size();

    // device buffers
    CK(h->d_chunks.ensure(sizeof(ChunkDesc) * std::max<size_t>(n_chunks, 1)));
    CK(h->d_chunk_range.ensure(sizeof(uint32_t) * range.size()));
    CK(h->d_frame_off.ensure(sizeof(uint32_t) * foff.size()));
    CK(h->d_bin_map.ensure(sizeof(uint16_t) * (NM + kIdPad)));      // + slack: K2 prefetches ids past a chunk's end unchecked
    CK(h->d_bin_qry.ensure(sizeof(uint16_t) * (NQ + kIdPad)));
    CK(h->d_chcnt.ensure(sizeof(uint32_t) * std::max<size_t>(n_chunks, 1) * (B + 1)));
    CK(h->d_map_sorted.ensure(sizeof(float4) * std::max<size_t>(NM, 1)));
    CK(h->d_zmin.ensure(sizeof(uint32_t) * 2 * (size_t)F * B));
    CK(h->d_zmax.ensure(sizeof(uint32_t) * 2 * (size_t)F * B));
    CK(h->d_cnt.ensure(sizeof(uint32_t) * 2 * (size_t)F * (B + 1)));
    CK(h->d_dst_start.ensure(sizeof(uint32_t) * 2 * (size_t)F * (B + 2)));
    CK(h->d_status.ensure((size_t)F * B));
    CK(h->d_action.ensure((size_t)F * B));
    CK(h->d_flag_slot.ensure(sizeof(uint32_t) * (size_t)F * B));
    CK(h->d_frame_rec_base.ensure(sizeof(uint32_t) * (size_t)F));
    h->rec_capacity = (uint32_t)std::min<size_t>((size_t)F * B, kMaxRecords);
    CK(h->d_recs.ensure(sizeof(FlagRec) * (size_t)h->rec_capacity));
    CK(h->d_nrecs.ensure(sizeof(uint32_t) * 4));
    CK(h->d_queue.ensure(sizeof(uint32_t) * kQueueWords));
    CK(h->d_bucket.ensure(sizeof(uint32_t) * (size_t)kNumBuckets * h->rec_capacity));
    CK(h->d_map_src.ensure(sizeof(uint32_t) * std::max<size_t>(NM, 1)));
    CK(h->d_scratch.ensure((size_t)24 * std::max<size_t>(NM, 1) + 64));
    if (node) {
        CK(h->d_poses.ensure(sizeof(NodePose) * (size_t)F));
        CK(h->d_list_idx.ensure(sizeof(uint32_t) * (NM + kIdPad)));
        CK(h->d_list_cnt.ensure(sizeof(uint32_t) * kListWarps * std::max<size_t>(n_chunks, 1)));
    }
    if (mode == 0) {
        CK(h->d_qry_sorted.ensure(sizeof(float4) * std::max<size_t>(NQ, 1)));
        CK(h->d_qry_src.ensure(sizeof(uint32_t) * std::max<size_t>(NQ, 1)));
        CK(h->d_part.ensure(sizeof(float4) * std::max<size_t>(NM, 1)));
    }

    // upload descriptors through pinned staging
    const size_t b0 = sizeof(ChunkDesc) * n_chunks, b1 = sizeof(uint32_t) * range.size(), b2 = sizeof(uint32_t) * foff.size();
    CK(cudaStreamSynchronize(h->stream));   // staging may still be in flight from the previous call
    CK(h->h_stage.ensure(b0 + b1 + b2 + 64));
    unsigned char* st = h->h_stage.as<unsigned char>();
    if (b0) std::memcpy(st, chunks.data(), b0);
    std::memcpy(st + b0, range.data(), b1);
    std::memcpy(st + b0 + b1, foff.data(), b2);
    if (b0) CK(cudaMemcpyAsync(h->d_chunks.p, st, b0, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_chunk_range.p, st + b0, b1, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_frame_off.p, st + b0 + b1, b2, cudaMemcpyHostToDevice, h->stream));
    h->desc_mode = mode;
    h->desc_epoch++;
    return ERASOR_OK;
}

// one caller cloud -> device pointer (staged through `stage` when it lives in host memory)
int stage_cloud(erasor_ctx* h, DevBuf& stage, const float* xyzi, size_t n, int ptr_kind, const float4** out, size_t bytes_per_point = sizeof(float4)) {
    if (ptr_kind == ERASOR_PTR_DEVICE) {
        const uintptr_t align = bytes_per_point == sizeof(float4) ? 15 : 3;
        if (n && (reinterpret_cast<uintptr_t>(xyzi) & align)) { h->err = "device clouds must be 16-byte aligned (float4; packed xyz: 4-byte)"; return ERASOR_E_INVALID; }
        *out = reinterpret_cast<const float4*>(xyzi);
        return ERASOR_OK;
    }
    CK(stage.ensure(sizeof(float4) * std::max<size_t>(n, 1)));
    if (n) CK(cudaMemcpyAsync(stage.p, xyzi, bytes_per_point * n, cudaMemcpyHostToDevice, h->stream));
    *out = stage.as<float4>();
    return ERASOR_OK;
}

int stage_inputs(erasor_ctx* h, const float* map_xyzi, const float* qry_xyzi, int ptr_kind) {
    int rc;
    if ((rc = stage_cloud(h, h->d_map_in, map_xyzi, h->NM, ptr_kind, &h->cur_map))) return rc;
    return stage_cloud(h, h->d_qry_in, qry_xyzi, h->NQ, ptr_kind, &h->cur_qry, h->qry_xyz ? 3 * sizeof(float) : sizeof(float4));
}

int run_k1(erasor_ctx* h, int mode) {
    const int B = h->B, F = h->F;
    {
        h->launches++;
        CK(launch_init_tables(h->stream, h->d_zmin.as<uint32_t>(), h->d_zmax.as<uint32_t>(), 2 * (size_t)F * B,
                              h->d_cnt.as<uint32_t>(), 2 * (size_t)F * (B + 1), h->d_nrecs.as<uint32_t>(), h->d_frame_rej.as<uint32_t>() + h->f0,
                              h->d_nflag.as<uint32_t>() + h->f0, F, h->d_queue.as<uint32_t>()));
    }
    {
        Scope s(h, 1);
        if (h->n_chunks_map + h->n_chunks_qry) h->launches++;
        CK(launch_k1(h->stream, h->view, h->cur_map, h->cur_qry, h->d_chunks.as<ChunkDesc>(), (int)(h->n_chunks_map + h->n_chunks_qry),
                     h->d_bin_map.as<uint16_t>(), h->d_bin_qry.as<uint16_t>(), h->d_chcnt.as<uint32_t>(), h->d_zmin.as<uint32_t>(),
                     h->d_zmax.as<uint32_t>(), h->d_cnt.as<uint32_t>(), B, F, h->d_fence.as<unsigned long long>(),
                     mode == 2 ? h->d_poses.as<NodePose>() : nullptr, mode == 2 ? h->d_list_idx.as<uint32_t>() : nullptr,
                     mode == 2 ? h->d_list_cnt.as<uint32_t>() : nullptr, mode != 0 && h->qry_xyz));
    }
    return ERASOR_OK;
}

// K3 -> K2 -> K4 ; mode 0: every bin scattered + partitioned copies (cloud outputs), mode 1 / 2: flagged only + masks
// classes: which R-GPF size classes to launch (bits 0|1: A and B, bit 2: C); 0x8 alone = R-GPF only, for the class-C fix-up
int run_compare(erasor_ctx* h, int version, int mode, uint8_t* keep_mask, uint8_t* ground_mask, const K4Fold& fold, int classes = 7, bool only_rgpf = false) {
    const int B = h->B, F = h->F;
    const NodePose* poses = mode == 2 ? h->d_poses.as<NodePose>() : nullptr;
    uint32_t* nflag = h->d_nflag.as<uint32_t>() + h->f0;
    SrtParams sp{};
    sp.scan_ratio_threshold = h->p.scan_ratio_threshold;
    sp.th_bin_max_h = h->p.th_bin_max_h;
    sp.minimum_num_pts = h->p.minimum_num_pts;
    sp.version = version; sp.R = h->p.num_rings; sp.S = h->p.num_sectors; sp.B = B; sp.scatter_mode = mode == 0 ? 0 : 1;
    const bool fused = mode != 0 && h->fused_srt;      // mask modes: SRT inside the scatter kernel
    if (!fused && !only_rgpf) {
        Scope s(h, 3);
        h->launches++;
        CK(launch_k3(h->stream, sp, F, h->d_chunk_range.as<uint32_t>(), h->d_chcnt.as<uint32_t>(), h->d_zmin.as<uint32_t>(),
                     h->d_zmax.as<uint32_t>(), h->d_frame_off.as<uint32_t>(), h->d_cnt.as<uint32_t>(), h->d_dst_start.as<uint32_t>(),
                     h->d_status.as<uint8_t>(), h->d_action.as<uint8_t>(), h->d_flag_slot.as<uint32_t>(), nflag,
                     h->d_frame_rec_base.as<uint32_t>(), h->d_recs.as<FlagRec>(), h->d_nrecs.as<uint32_t>(), h->rec_capacity,
                     h->d_queue.as<uint32_t>(), h->d_bucket.as<uint32_t>()));
    }
    if (!only_rgpf) {
        Scope s(h, 2);
        if (mode == 0) {
            if (h->n_chunks_map + h->n_chunks_qry) h->launches++;
            CK(launch_k2_both(h->stream, h->d_chunks.as<ChunkDesc>(), h->n_chunks_map, h->n_chunks_qry, h->d_chcnt.as<uint32_t>(), B,
                              h->d_bin_map.as<uint16_t>(), h->cur_map, h->d_dst_start.as<uint32_t>(), h->d_map_sorted.as<float4>(), h->d_map_src.as<uint32_t>(),
                              h->d_bin_qry.as<uint16_t>(), h->cur_qry, h->d_dst_start.as<uint32_t>() + (size_t)F * (B + 2), h->d_qry_sorted.as<float4>(),
                              h->d_qry_src.as<uint32_t>()));
        } else if (fused) {
            if (h->n_chunks_map) h->launches++;
            CK(launch_k2_srt(h->stream, sp, F, h->d_chunks.as<ChunkDesc>(), h->d_chunk_range.as<uint32_t>(), h->n_chunks_map, h->d_bin_map.as<uint16_t>(),
                             h->cur_map, poses, h->d_chcnt.as<uint32_t>(), h->d_zmin.as<uint32_t>(), h->d_zmax.as<uint32_t>(), h->d_cnt.as<uint32_t>(),
                             h->d_frame_off.as<uint32_t>(), nflag, h->d_recs.as<FlagRec>(), h->d_nrecs.as<uint32_t>(), h->rec_capacity,
                             h->d_queue.as<uint32_t>(), h->d_bucket.as<uint32_t>(), h->d_map_sorted.as<float4>(), h->d_map_src.as<uint32_t>(),
                             poses ? h->d_list_idx.as<uint32_t>() : nullptr, poses ? h->d_list_cnt.as<uint32_t>() : nullptr));
        } else {
            // mask modes, unfused (ERASOR_B200_UNFUSED_SRT=1): the same stable scatter, restricted to the flagged bins (K3's dense slots)
            if (h->n_chunks_map) h->launches++;
            CK(launch_k2(h->stream, h->d_chunks.as<ChunkDesc>(), 0u, h->n_chunks_map, h->d_bin_map.as<uint16_t>(), h->cur_map, poses,
                         h->d_chcnt.as<uint32_t>(), h->d_dst_start.as<uint32_t>(), h->d_flag_slot.as<uint32_t>(), nflag,
                         h->d_map_sorted.as<float4>(), h->d_map_src.as<uint32_t>(), B,
                         poses ? h->d_list_idx.as<uint32_t>() : nullptr, poses ? h->d_list_cnt.as<uint32_t>() : nullptr,
                         k1_big_tables(h->p.num_rings, B) ? 32 : 8));
        }
    }
    {
        Scope s(h, 4);
        GpfParams gp{};
        gp.th_dist = h->p.gf_dist_thr; gp.th_seeds = h->p.gf_th_seeds_height; gp.num_lowest_pts = h->p.num_lowest_pts;
        gp.num_lpr = h->p.gf_num_lpr; gp.iters = std::min(h->p.gf_iter, kMaxIter); gp.cov_mode = h->p.cov_mode;
        const bool with_c = (classes & 4) != 0;
        h->launches += k4_num_launches(with_c);
        CK(cudaEventRecord(h->ev_fork, h->stream));
        CK(cudaStreamWaitEvent(h->stream_a, h->ev_fork, 0));
        CK(cudaStreamWaitEvent(h->stream_b, h->ev_fork, 0));
        if (with_c) CK(cudaStreamWaitEvent(h->stream_c, h->ev_fork, 0));
        CK(launch_k4(h->stream_a, h->stream_b, h->stream_c, gp, h->d_recs.as<FlagRec>(), h->d_queue.as<uint32_t>(), h->d_bucket.as<uint32_t>(), h->rec_capacity,
                     h->d_map_sorted.as<float4>(), h->d_map_src.as<uint32_t>(), h->cur_map,
                     h->d_frame_off.as<uint32_t>(), mode == 0 ? h->d_part.as<float4>() : nullptr, keep_mask, ground_mask,
                     h->d_frame_rej.as<uint32_t>() + h->f0, h->d_scratch.as<unsigned char>(), h->sm_count, h->d_fence.as<unsigned long long>(), fold, classes));
        CK(cudaEventRecord(h->ev_join_a, h->stream_a));
        CK(cudaEventRecord(h->ev_join_b, h->stream_b));
        if (with_c) CK(cudaEventRecord(h->ev_join_c, h->stream_c));
        CK(cudaStreamWaitEvent(h->stream, h->ev_join_a, 0));
        CK(cudaStreamWaitEvent(h->stream, h->ev_join_b, 0));
        if (with_c) CK(cudaStreamWaitEvent(h->stream, h->ev_join_c, 0));
    }
    return ERASOR_OK;
}

int copy_out(erasor_ctx* h, const void* dev_src, void* user_dst, size_t bytes, int ptr_kind) {
    if (!bytes) return ERASOR_OK;
    CK(cudaMemcpyAsync(user_dst, dev_src, bytes, ptr_kind == ERASOR_PTR_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
    return ERASOR_OK;
}

float status_value(uint8_t code) {
    switch (code) {
        case ST_MERGE: return ERASOR_STATUS_MERGE_BINS;
        case ST_MAP_HIGH: return ERASOR_STATUS_MAP_IS_HIGHER;
        case ST_BLOCKED: return ERASOR_STATUS_BLOCKED;
        case ST_CURR_HIGH: return ERASOR_STATUS_CURR_IS_HIGHER;
        default: return ERASOR_STATUS_LITTLE_NUM;
    }
}

}  // namespace

extern "C" {

int erasor_abi_version(void) { return ERASOR_B200_ABI_VERSION; }

const char* erasor_last_error(erasor_handle_t h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int erasor_create(const erasor_params_t* params, int device, erasor_handle_t* out) {
    if (!params || !out) { g_create_error = "null argument"; return ERASOR_E_INVALID; }
    *out = nullptr;
    const erasor_params_t& p = *params;
    const long long Bll = (long long)p.num_rings * (long long)p.num_sectors;
    if (p.num_rings < 1 || p.num_sectors < 1 || Bll > 65534) { g_create_error = "num_rings*num_sectors must be in [1, 65534]"; return ERASOR_E_INVALID; }
    if (p.version != 2 && p.version != 3) { g_create_error = "Other version is not implemented!"; return ERASOR_E_INVALID; }   // OfflineMapUpdater.cpp:274
    if (p.sort_mode != 1) { g_create_error = "sort_mode must be 1 (stable z order)"; return ERASOR_E_UNSUPPORTED; }
    if (p.gf_iter > kMaxIter) { g_create_error = "gf_iter above the tap capacity (8)"; return ERASOR_E_UNSUPPORTED; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                         " (this library has no CPU path)";
        return ERASOR_E_CUDA;
    }
    if (device < 0 || device >= ndev) { g_create_error = "bad device index"; return ERASOR_E_INVALID; }
    erasor_ctx* h = new erasor_ctx();
    h->p = p; h->device = device; h->B = (int)Bll;
    for (DevBuf* b : h->all_bufs()) b->epoch = &h->alloc_epoch;
    if (const char* ng = std::getenv("ERASOR_B200_NO_GRAPH")) h->use_graphs = !(ng[0] == '1');
    if (const char* uf = std::getenv("ERASOR_B200_UNFUSED_SRT")) h->fused_srt = !(uf[0] == '1');
    if (const char* cs = std::getenv("ERASOR_B200_CTAS_PER_SM")) h->ctas_per_sm = std::max(1, std::min(8, std::atoi(cs)));
    std::string terr;
    if (build_bin_tables(p, h->tables, terr) != 0) { g_create_error = terr; delete h; return ERASOR_E_INVALID; }
    auto fail = [&](const char* what, cudaError_t ce) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(ce);
        erasor_destroy(h);
        return ERASOR_E_CUDA;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail("cudaGetDeviceProperties", e);
    h->sm_count = prop.multiProcessorCount;
    const size_t need = std::max(k1_smem_bytes(p.num_rings, h->B), k3_smem_bytes(h->B));
    if (need > (size_t)prop.sharedMemPerBlockOptin) {
        g_create_error = "num_rings*num_sectors too large for the per-CTA shared-memory bin table";
        erasor_destroy(h);
        return ERASOR_E_UNSUPPORTED;
    }
    // R-GPF's bins are long serial chains: its CTAs go first whenever SM resources free up (highest stream priority), the
    // bandwidth / issue-bound kernels of this and of overlapped handles fill in around them
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (const char* np = std::getenv("ERASOR_B200_NO_PRIORITY")) { if (np[0] == '1') prio_hi = prio_lo; }
    if ((e = cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio_lo)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithPriority(&h->stream_a, cudaStreamNonBlocking, prio_hi)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithPriority(&h->stream_b, cudaStreamNonBlocking, prio_hi)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithPriority(&h->stream_c, cudaStreamNonBlocking, prio_hi)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaEventCreateWithFlags(&h->ev_join_a, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&h->ev_join_b, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&h->ev_join_c, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    const size_t rb = sizeof(double) * h->tables.ring_thr.size(), sb = sizeof(SectorBoundary) * h->tables.sec_pos.size();
    if ((e = h->h_words.ensure(128)) != cudaSuccess) return fail("cudaMallocHost", e);
    std::memset(h->h_words.p, 0, 128);
    const size_t gb = sizeof(float) * h->tables.ring_guard.size();
    if ((e = h->d_guard.ensure(gb)) != cudaSuccess) return fail("cudaMalloc", e);
    if ((e = cudaMemcpy(h->d_guard.p, h->tables.ring_guard.data(), gb, cudaMemcpyHostToDevice)) != cudaSuccess) return fail("cudaMemcpy", e);
    if ((e = h->d_ring.ensure(rb)) != cudaSuccess || (e = h->d_pos.ensure(sb)) != cudaSuccess || (e = h->d_neg.ensure(sb)) != cudaSuccess ||
        (e = h->d_fence.ensure(sizeof(unsigned long long) * 4)) != cudaSuccess)
        return fail("cudaMalloc", e);
    if ((e = cudaMemcpy(h->d_ring.p, h->tables.ring_thr.data(), rb, cudaMemcpyHostToDevice)) != cudaSuccess) return fail("cudaMemcpy", e);
    if ((e = cudaMemcpy(h->d_pos.p, h->tables.sec_pos.data(), sb, cudaMemcpyHostToDevice)) != cudaSuccess) return fail("cudaMemcpy", e);
    if ((e = cudaMemcpy(h->d_neg.p, h->tables.sec_neg.data(), sb, cudaMemcpyHostToDevice)) != cudaSuccess) return fail("cudaMemcpy", e);
    if ((e = cudaMemset(h->d_fence.p, 0, sizeof(unsigned long long) * 4)) != cudaSuccess) return fail("cudaMemset", e);
    h->view = h->tables.view(h->d_ring.as<double>(), h->d_pos.as<SectorBoundary>(), h->d_neg.as<SectorBoundary>(), h->d_guard.as<float>());
    *out = h;
    return ERASOR_OK;
}

void erasor_destroy(erasor_handle_t h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    drain_timers(h);
    for (auto& g : h->graphs) cudaGraphExecDestroy(g.exec);
    h->graphs.clear();
    if (h->comm) { NcclApi* api = nccl_api(h->err); if (api) api->CommDestroy(h->comm); h->comm = nullptr; }
    for (DevBuf* b : h->all_bufs()) b->release();
    h->h_pose.release();
    h->h_words.release();
    h->h_stage.release();
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join_a) cudaEventDestroy(h->ev_join_a);
    if (h->ev_join_b) cudaEventDestroy(h->ev_join_b);
    if (h->ev_join_c) cudaEventDestroy(h->ev_join_c);
    if (h->stream_a) cudaStreamDestroy(h->stream_a);
    if (h->stream_b) cudaStreamDestroy(h->stream_b);
    if (h->stream_c) cudaStreamDestroy(h->stream_c);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

void* erasor_stream(erasor_handle_t h) { return h ? (void*)h->stream : nullptr; }

int erasor_synchronize(erasor_handle_t h) {
    if (!h) return ERASOR_E_INVALID;
    CK(cudaStreamSynchronize(h->stream));
    return ERASOR_OK;
}

double erasor_get_max_range(erasor_handle_t h) { return h ? h->p.max_range : 0.0; }

int erasor_set_inputs(erasor_handle_t h, const float* map_voi_xyzi, size_t n_map, const float* query_voi_xyzi, size_t n_query, int ptr_kind) {
    if (!h) return ERASOR_E_INVALID;
    if ((n_map && !map_voi_xyzi) || (n_query && !query_voi_xyzi)) { h->err = "null cloud"; return ERASOR_E_INVALID; }
    CK(cudaSetDevice(h->device));
    int rc;
    if (h->pending && (rc = erasor_wait(h))) return rc;
    h->stage = 0;
    h->f0 = 0; h->stat_F = 1;
    h->qry_xyz = false;
    if (ptr_kind != ERASOR_PTR_HOST && ptr_kind != ERASOR_PTR_DEVICE) { h->err = "erasor_set_inputs: ptr_kind must be HOST or DEVICE (the cloud outputs carry the query's intensity)"; return ERASOR_E_INVALID; }
    const uint64_t mo[2] = {0, n_map}, qo[2] = {0, n_query};
    rc = prepare_batch(h, mo, qo, 1, 0);
    if (rc) return rc;
    if ((rc = stage_inputs(h, map_voi_xyzi, query_voi_xyzi, ptr_kind))) return rc;
    if ((rc = run_k1(h, 0))) return rc;
    h->stage = 1;
    return ERASOR_OK;
}

int erasor_compare(erasor_handle_t h, int version, int frame) {
    (void)frame;   // the reference uses it only for a commented-out csv dump (erasor.cpp:341-343)
    if (!h) return ERASOR_E_INVALID;
    if (h->stage < 1) { h->err = "erasor_compare before erasor_set_inputs"; return ERASOR_E_STATE; }
    if (h->stage > 1) { h->err = "erasor_compare called twice: set_inputs -> exactly one compare (OfflineMapUpdater.cpp:266-272)"; return ERASOR_E_STATE; }
    if (version != 2 && version != 3) { h->err = "Other version is not implemented!"; return ERASOR_E_INVALID; }
    CK(cudaSetDevice(h->device));
    const int B = h->B;
    const size_t NM = h->NM, NQ = h->NQ;
    CK(h->d_keep.ensure(std::max<size_t>(NM, 1)));
    CK(h->d_ground.ensure(std::max<size_t>(NM, 1)));
    CK(cudaMemsetAsync(h->d_keep.p, 1, std::max<size_t>(NM, 1), h->stream));
    CK(cudaMemsetAsync(h->d_ground.p, 0, std::max<size_t>(NM, 1), h->stream));
    // R-GPF class C (bins beyond 2560 points, 1024-thread CTAs) is launched only while such bins are being seen; if one turns up
    // unannounced the class runs after the fact and the output assembly is repeated (same policy as the mask modes, erasor_wait)
    const bool with_c = h->class_c_state != 0;
    int rc = run_compare(h, version, 0, h->d_keep.as<uint8_t>(), h->d_ground.as<uint8_t>(), K4Fold{nullptr, nullptr, 0u, 0u}, with_c ? 7 : 3);
    if (rc) return rc;
    const bool vox = (version == 3) && !h->p.skip_voxelize;
    if (vox) {
        CK(h->d_vox.ensure(sizeof(float4) * (NM + NQ + 1)));
        CK(h->d_vox_cnt.ensure(sizeof(uint32_t) * (size_t)B));
        CK(h->d_vox_start.ensure(sizeof(uint32_t) * (size_t)B));
        CK(h->d_vox_scratch.ensure((size_t)36 * (NM + NQ + 1) + 64));
    }
    CK(h->d_arranged.ensure(sizeof(float4) * (2 * NM + NQ + 1)));
    CK(h->d_map_rej.ensure(sizeof(float4) * std::max<size_t>(NM, 1)));
    CK(h->d_curr_rej.ensure(sizeof(float4) * std::max<size_t>(NQ, 1)));
    CK(h->d_jobs.ensure(sizeof(CopyJob) * 5 * (size_t)B));
    CK(h->d_out_sizes.ensure(sizeof(uint32_t) * 8));
    CK(h->d_k5tmp.ensure(sizeof(uint32_t) * 3 * (size_t)(B + 1)));
    // in-bin voxelisation (v3) + output assembly + the sizes the caller needs, read back through pinned memory
    auto assemble = [&]() -> int {
        if (vox) {
            Scope s(h, 4);
            h->launches++;
            CK(launch_k4b(h->stream, (float)h->p.map_voxel_size, B, h->d_recs.as<FlagRec>(), h->d_nrecs.as<uint32_t>(), h->rec_capacity,
                          h->d_cnt.as<uint32_t>(), h->d_dst_start.as<uint32_t>(), h->d_qry_sorted.as<float4>(), h->d_part.as<float4>(),
                          h->d_vox.as<float4>(), h->d_vox_cnt.as<uint32_t>(), h->d_vox_start.as<uint32_t>(),
                          h->d_vox_scratch.as<unsigned char>(), h->sm_count));
        }
        {
            Scope s(h, 5);
            h->launches += 2;
            CK(launch_k5(h->stream, B, version, h->p.skip_voxelize, h->d_cnt.as<uint32_t>(), h->d_dst_start.as<uint32_t>(), h->d_action.as<uint8_t>(),
                         h->d_flag_slot.as<uint32_t>(), h->d_recs.as<FlagRec>(), h->d_nrecs.as<uint32_t>(),
                         vox ? h->d_vox_cnt.as<uint32_t>() : nullptr, vox ? h->d_vox_start.as<uint32_t>() : nullptr,
                         h->d_map_sorted.as<float4>(), h->d_qry_sorted.as<float4>(), h->d_part.as<float4>(),
                         vox ? h->d_vox.as<float4>() : nullptr, h->d_arranged.as<float4>(),
                         h->d_map_rej.as<float4>(), h->d_curr_rej.as<float4>(), h->d_jobs.as<CopyJob>(), h->d_out_sizes.as<uint32_t>(),
                         h->d_k5tmp.as<uint32_t>(), h->sm_count * 4));
        }
        uint32_t* w = h->h_words.as<uint32_t>();
        CK(cudaMemcpyAsync(w + 4, h->d_out_sizes.p, sizeof(uint32_t) * 5, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(w + 9, h->d_dst_start.as<uint32_t>() + B, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(w + 10, h->d_nrecs.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(w + 11, h->d_queue.as<uint32_t>() + kBucketC0, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return ERASOR_OK;
    };
    if ((rc = assemble())) return rc;
    const uint32_t n_class_c = h->words()[11];
    if (!with_c && n_class_c > 0) {
        if ((rc = run_compare(h, version, 0, h->d_keep.as<uint8_t>(), h->d_ground.as<uint8_t>(), K4Fold{nullptr, nullptr, 0u, 0u}, 4, true))) return rc;
        if ((rc = assemble())) return rc;
    }
    h->class_c_state = (int)std::min<uint32_t>(n_class_c, 0x7FFFFFFFu);
    for (int i = 0; i < 5; ++i) h->out_sizes[i] = h->words()[4 + i];
    h->complement_start = h->words()[9];
    h->n_recs_host = h->words()[10];
    h->stage = 2;
    return ERASOR_OK;
}

int erasor_get_output_sizes(erasor_handle_t h, size_t* n_arranged, size_t* n_complement, size_t* n_map_rejected, size_t* n_curr_rejected) {
    if (!h) return ERASOR_E_INVALID;
    if (h->stage < 2) { h->err = "no compare result"; return ERASOR_E_STATE; }
    if (n_arranged) *n_arranged = h->out_sizes[0];
    if (n_complement) *n_complement = h->out_sizes[1];
    if (n_map_rejected) *n_map_rejected = h->out_sizes[2];
    if (n_curr_rejected) *n_curr_rejected = h->out_sizes[3];
    return ERASOR_OK;
}

int erasor_get_static_estimate(erasor_handle_t h, float* arranged_xyzi, size_t cap_arranged, size_t* n_arranged,
                               float* complement_xyzi, size_t cap_complement, size_t* n_complement, int ptr_kind) {
    if (!h) return ERASOR_E_INVALID;
    if (h->stage < 2) { h->err = "erasor_get_static_estimate before erasor_compare"; return ERASOR_E_STATE; }
    if (n_arranged) *n_arranged = h->out_sizes[0];
    if (n_complement) *n_complement = h->out_sizes[1];
    if ((arranged_xyzi && cap_arranged < h->out_sizes[0]) || (complement_xyzi && cap_complement < h->out_sizes[1])) {
        h->err = "output buffer too small"; return ERASOR_E_CAPACITY;
    }
    CK(cudaSetDevice(h->device));
    int rc;
    if (arranged_xyzi && (rc = copy_out(h, h->d_arranged.p, arranged_xyzi, sizeof(float4) * h->out_sizes[0], ptr_kind))) return rc;
    if (complement_xyzi && (rc = copy_out(h, h->d_map_sorted.as<float4>() + h->complement_start, complement_xyzi,
                                          sizeof(float4) * h->out_sizes[1], ptr_kind))) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return ERASOR_OK;
}

int erasor_get_outliers(erasor_handle_t h, float* map_rejected_xyzi, size_t cap_map, size_t* n_map_rejected,
                        float* curr_rejected_xyzi, size_t cap_curr, size_t* n_curr_rejected, int ptr_kind) {
    if (!h) return ERASOR_E_INVALID;
    if (h->stage < 2) { h->err = "erasor_get_outliers before erasor_compare"; return ERASOR_E_STATE; }
    if (n_map_rejected) *n_map_rejected = h->out_sizes[2];
    if (n_curr_rejected) *n_curr_rejected = h->out_sizes[3];
    if ((map_rejected_xyzi && cap_map < h->out_sizes[2]) || (curr_rejected_xyzi && cap_curr < h->out_sizes[3])) {
        h->err = "output buffer too small"; return ERASOR_E_CAPACITY;
    }
    CK(cudaSetDevice(h->device));
    int rc;
    if (map_rejected_xyzi && (rc = copy_out(h, h->d_map_rej.p, map_rejected_xyzi, sizeof(float4) * h->out_sizes[2], ptr_kind))) return rc;
    if (curr_rejected_xyzi && (rc = copy_out(h, h->d_curr_rej.p, curr_rejected_xyzi, sizeof(float4) * h->out_sizes[3], ptr_kind))) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return ERASOR_OK;
}

int erasor_device_outputs(erasor_handle_t h, const float** arranged, const float** complement, const float** map_rejected, const float** curr_rejected) {
    if (!h) return ERASOR_E_INVALID;
    if (h->stage < 2) { h->err = "erasor_device_outputs before erasor_compare"; return ERASOR_E_STATE; }
    if (arranged) *arranged = h->d_arranged.as<float>();
    if (complement) *complement = reinterpret_cast<const float*>(h->d_map_sorted.as<float4>() + h->complement_start);
    if (map_rejected) *map_rejected = h->d_map_rej.as<float>();
    if (curr_rejected) *curr_rejected = h->d_curr_rej.as<float>();
    return ERASOR_OK;
}

// ERASOR::ground_viz (public member, erasor.h:127): the R-GPF ground points of the flagged bins of the last compare, in
// processing order -- the tail get_static_estimate appends to `arranged` (erasor.cpp:616)
int erasor_get_ground_viz(erasor_handle_t h, float* ground_xyzi, size_t cap, size_t* n_ground, int ptr_kind) {
    if (!h) return ERASOR_E_INVALID;
    if (h->stage < 2) { h->err = "erasor_get_ground_viz before erasor_compare"; return ERASOR_E_STATE; }
    const size_t n = h->out_sizes[4];
    if (n_ground) *n_ground = n;
    if (!ground_xyzi) return ERASOR_OK;
    if (cap < n) { h->err = "output buffer too small"; return ERASOR_E_CAPACITY; }
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = copy_out(h, h->d_arranged.as<float4>() + (h->out_sizes[0] - n), ground_xyzi, sizeof(float4) * n, ptr_kind))) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return ERASOR_OK;
}

int erasor_get_bins(erasor_handle_t h, int which_cloud, int32_t* bin_of_point, float* min_h, float* max_h, uint32_t* count) {
    if (!h) return ERASOR_E_INVALID;
    if (h->stage < 1 || h->F != 1) { h->err = "erasor_get_bins needs a single-frame erasor_set_inputs"; return ERASOR_E_STATE; }
    if (which_cloud != 0 && which_cloud != 1) { h->err = "which_cloud"; return ERASOR_E_INVALID; }
    CK(cudaSetDevice(h->device));
    const int B = h->B;
    const size_t n = which_cloud == 0 ? h->NM : h->NQ;
    CK(cudaStreamSynchronize(h->stream));
    if (bin_of_point && n) {
        std::vector<uint16_t> tmp(n);
        CK(cudaMemcpy(tmp.data(), which_cloud == 0 ? h->d_bin_map.p : h->d_bin_qry.p, sizeof(uint16_t) * n, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < n; ++i) bin_of_point[i] = tmp[i] == kNoBin16 ? -1 : (int32_t)tmp[i];
    }
    if (min_h || max_h || count) {
        std::vector<uint32_t> mn(B), mx(B);
        CK(cudaMemcpy(mn.data(), h->d_zmin.as<uint32_t>() + (size_t)which_cloud * B, sizeof(uint32_t) * B, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(mx.data(), h->d_zmax.as<uint32_t>() + (size_t)which_cloud * B, sizeof(uint32_t) * B, cudaMemcpyDeviceToHost));
        std::vector<uint32_t> c(B, 0);
        CK(cudaMemcpy(c.data(), h->d_cnt.as<uint32_t>() + (size_t)which_cloud * (B + 1), sizeof(uint32_t) * B, cudaMemcpyDeviceToHost));
        const float nan = std::numeric_limits<float>::quiet_NaN();
        for (int b = 0; b < B; ++b) {
            const bool empty = mn[b] == 0xFFFFFFFFu && mx[b] == 0u;
            if (min_h) min_h[b] = empty ? nan : ordered_to_float(mn[b]);
            if (max_h) max_h[b] = empty ? nan : ordered_to_float(mx[b]);
            if (count) count[b] = c[b];
        }
    }
    return ERASOR_OK;
}

int erasor_get_status(erasor_handle_t h, float* status) {
    if (!h || !status) return ERASOR_E_INVALID;
    if (h->stage < 2) { h->err = "erasor_get_status before erasor_compare"; return ERASOR_E_STATE; }
    CK(cudaSetDevice(h->device));
    std::vector<uint8_t> st(h->B);
    CK(cudaMemcpy(st.data(), h->d_status.p, h->B, cudaMemcpyDeviceToHost));
    for (int b = 0; b < h->B; ++b) status[b] = status_value(st[b]);
    return ERASOR_OK;
}

int erasor_get_planes(erasor_handle_t h, int32_t* bin_ids, int32_t* n_points, int32_t* n_seeds, double* lpr_height,
                      double* normal_d, int32_t* n_ground, size_t* n_planes) {
    if (!h || !n_planes) return ERASOR_E_INVALID;
    if (h->stage < 2) { h->err = "erasor_get_planes before erasor_compare"; return ERASOR_E_STATE; }
    CK(cudaSetDevice(h->device));
    const size_t n = h->n_recs_host, cap = *n_planes;
    *n_planes = n;
    if (!bin_ids && !n_points && !n_seeds && !lpr_height && !normal_d && !n_ground) return ERASOR_OK;
    if (cap < n) { h->err = "plane buffer too small"; return ERASOR_E_CAPACITY; }
    std::vector<FlagRec> recs(n);
    if (n) CK(cudaMemcpy(recs.data(), h->d_recs.p, sizeof(FlagRec) * n, cudaMemcpyDeviceToHost));
    const int it = std::min(h->p.gf_iter, kMaxIter);
    for (size_t i = 0; i < n; ++i) {
        const FlagRec& r = recs[i];   // single frame: record index == slot == processing order (bin order)
        if (bin_ids) bin_ids[i] = (int32_t)r.bin;
        if (n_points) n_points[i] = (int32_t)r.n_points;
        if (n_seeds) n_seeds[i] = (int32_t)r.n_seeds;
        if (lpr_height) lpr_height[i] = r.lpr_height;
        for (int k = 0; k < it; ++k) {
            if (normal_d) for (int c = 0; c < 4; ++c) normal_d[(i * it + k) * 4 + c] = r.normal_d[k][c];
            if (n_ground) n_ground[i * it + k] = (int32_t)r.n_ground[k];
        }
    }
    return ERASOR_OK;
}

int erasor_get_static_mask(erasor_handle_t h, uint8_t* keep_map, uint8_t* is_ground) {
    if (!h) return ERASOR_E_INVALID;
    if (h->stage < 2) { h->err = "erasor_get_static_mask before erasor_compare"; return ERASOR_E_STATE; }
    CK(cudaSetDevice(h->device));
    if (keep_map && h->NM) CK(cudaMemcpy(keep_map, h->d_keep.p, h->NM, cudaMemcpyDeviceToHost));
    if (is_ground && h->NM) CK(cudaMemcpy(is_ground, h->d_ground.p, h->NM, cudaMemcpyDeviceToHost));
    return ERASOR_OK;
}

int erasor_get_fence_counts(erasor_handle_t h, uint64_t* negzero_points, uint64_t* empty_plane_fits, uint64_t* ambiguous_sector) {
    if (!h) return ERASOR_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    unsigned long long v[4];
    CK(cudaMemcpy(v, h->d_fence.p, sizeof(v), cudaMemcpyDeviceToHost));
    if (negzero_points) *negzero_points = v[0];
    if (empty_plane_fits) *empty_plane_fits = v[1];
    if (ambiguous_sector) *ambiguous_sector = v[2];
    return ERASOR_OK;
}

namespace {

// One submission of a mask mode: a batch of (map_voi, query_voi) pairs (mode 1) or of nodes against the resident map (mode 2).
struct Submit {
    int mode = 1;
    const float*    map_xyzi = nullptr;     // mode 1
    const uint64_t* map_off = nullptr;      // mode 1: caller's offsets; mode 2: {0, n_map, 2 n_map, ...}
    const float*    qry_xyzi = nullptr;
    const uint64_t* qry_off = nullptr;
    int             F = 0;
    uint8_t*        keep_mask = nullptr;    // mode 1: one byte per VoI point; mode 2: frame_keep [F][n_map] (nullable)
    int             ptr_kind = ERASOR_PTR_HOST;
    bool            qry_xyz = false;        // the query cloud is packed x y z (ERASOR_PTR_QUERY_XYZ)
    const uint32_t* fold_index = nullptr;   // mode 1 fold (nullable)
    uint8_t*        fold_global = nullptr;
    size_t          fold_n = 0;
    const NodePose* poses = nullptr;        // mode 2: host array [F]
    uint8_t*        keep_out = nullptr;     // mode 2 (nullable)
    int             f0 = 0;                 // index of the first frame within the caller's batch (per-frame counters)
    const erasor_scan_params_t* scan = nullptr;   // mode 2 on raw scans (erasor_process_scans): qry_xyzi holds the scans
    bool            scan_xyz = false;       // ... packed x y z
};

bool is_pinned_host(const void* p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// Enqueue one submission on the handle's stream (CUDA graph when possible) and return without waiting.
// The whole step (copies, memset, K1, K3, K2, the three concurrent K4 classes with the fold in their epilogue, mask /
// counter read-back) is a fixed launch sequence once the batch geometry and the buffers are known: it is captured into a
// CUDA graph the first time and replayed afterwards (one launch instead of ~15 API calls).
int submit(erasor_ctx* h, const Submit& S) {
    int rc;
    CK(cudaSetDevice(h->device));
    if (h->pending && (rc = erasor_wait(h))) return rc;      // one submission in flight per handle (buffers and staging are reused)
    h->stage = 0;
    h->f0 = S.f0;
    h->qry_xyz = S.qry_xyz;
    if ((rc = prepare_batch(h, S.map_off, S.qry_off, S.F, S.scan ? 3 : S.mode))) return rc;
    const bool host = S.ptr_kind != ERASOR_PTR_DEVICE;
    Mat4 T_l2b{};
    if (S.scan) {
        Mat4 G{}, I{};                                          // tf_lidar2body_ = geoPose2eigen(pose) * Identity, as the updater builds it
        pose_to_mat(S.scan->lidar2body, G);
        for (int i = 0; i < 4; ++i) I.m[5 * i] = 1.0f;
        mat_mul(G, I, T_l2b);
        CK(h->d_scan_q.ensure(sizeof(float4) * std::max<size_t>(h->NQ, 1)));
        CK(h->d_scan_grid.ensure(sizeof(VoxGrid) * (size_t)S.F));
        CK(h->d_scan_tmp.ensure(voxelize_tmp_bytes((uint32_t)h->NQ, (uint32_t)S.F)));
        CK(h->d_scan_cnt.ensure(sizeof(uint32_t) * ((size_t)S.F + 1)));
        if (S.scan_xyz) CK(h->d_scan_f4.ensure(sizeof(float4) * std::max<size_t>(h->NQ, 1)));
    }
    const size_t n_keep = S.keep_mask ? h->NM : 0;          // bytes of the per-frame mask output
    const size_t n_map_global = S.mode == 2 ? h->map->n : 0;
    if (S.mode == 1 && ((h->NM && !S.map_xyzi) || (h->NQ && !S.qry_xyzi))) { h->err = "null cloud"; return ERASOR_E_INVALID; }
    if (S.mode == 2 && h->NQ && !S.qry_xyzi) { h->err = "null cloud"; return ERASOR_E_INVALID; }
    if (host) {
        if (n_keep) CK(h->d_keep.ensure(std::max<size_t>(n_keep, 1)));
        if (S.mode == 1) CK(h->d_map_in.ensure(sizeof(float4) * std::max<size_t>(h->NM, 1)));
        CK(h->d_qry_in.ensure(sizeof(float4) * std::max<size_t>(h->NQ, 1)));
    }
    if (S.mode == 2) {
        if (sizeof(NodePose) * (size_t)S.F > h->h_pose.cap) h->alloc_epoch++;      // captured graphs copy from this staging buffer
        CK(h->h_pose.ensure(sizeof(NodePose) * (size_t)S.F));
        std::memcpy(h->h_pose.p, S.poses, sizeof(NodePose) * (size_t)S.F);
    }
    const bool with_c = h->class_c_state != 0;
    auto enqueue = [&]() -> int {
        int r;
        if (S.mode == 1) {
            if ((r = stage_inputs(h, S.map_xyzi, S.qry_xyzi, S.ptr_kind))) return r;
        } else {
            h->cur_map = reinterpret_cast<const float4*>(h->map->d_pts);
            if (!S.scan) {
                if ((r = stage_cloud(h, h->d_qry_in, S.qry_xyzi, h->NQ, S.ptr_kind, &h->cur_qry, S.qry_xyz ? 3 * sizeof(float) : sizeof(float4)))) return r;
            } else {
                // raw scans -> voxelised body-frame queries, all frames in one cooperative launch; frame f's voxels land at its raw
                // offset, their number in d_scan_cnt[f], and the query chunks (cut from the raw sizes) are clamped to it on the device
                const float4* raw = nullptr;
                if ((r = stage_cloud(h, h->d_qry_in, S.qry_xyzi, h->NQ, S.ptr_kind, &raw, S.scan_xyz ? 3 * sizeof(float) : sizeof(float4)))) return r;
                if (S.scan_xyz) {
                    h->launches++;
                    CK(launch_expand_xyz(h->stream, reinterpret_cast<const float*>(raw), h->d_scan_f4.as<float4>(), (uint32_t)h->NQ));
                    raw = h->d_scan_f4.as<float4>();
                }
                FusedJob J{};
                J.vin = raw; J.vn = (uint32_t)h->NQ; J.leaf = (float)S.scan->query_voxel_size; J.grid = h->d_scan_grid.as<VoxGrid>();
                J.vtmp = h->d_scan_tmp.p; J.vout = h->d_scan_q.as<float4>(); J.d_n_out = h->d_scan_cnt.as<uint32_t>() + S.F;
                J.T_out = T_l2b; J.xform_out = 1;
                J.n_clouds = (uint32_t)S.F; J.cloud_off = h->d_frame_off.as<uint32_t>() + (S.F + 1); J.cloud_nvox = h->d_scan_cnt.as<uint32_t>();
                J.restore_labels = 0;
                h->launches += 2;
                CK(launch_node_fused(h->stream, J, h->sm_count));
                CK(launch_clamp_query_chunks(h->stream, h->d_chunks.as<ChunkDesc>(), h->n_chunks_map, h->n_chunks_qry, h->d_scan_cnt.as<uint32_t>()));
                h->cur_qry = h->d_scan_q.as<float4>();
            }
            CK(cudaMemcpyAsync(h->d_poses.p, h->h_pose.p, sizeof(NodePose) * (size_t)S.F, cudaMemcpyHostToDevice, h->stream));
        }
        uint8_t* d_keep = nullptr;
        if (n_keep) {
            d_keep = host ? h->d_keep.as<uint8_t>() : S.keep_mask;
            CK(cudaMemsetAsync(d_keep, 1, n_keep, h->stream));
        }
        if ((r = run_k1(h, S.mode))) return r;
        K4Fold fold{nullptr, nullptr, 0u, 0u};
        if (S.mode == 2)        fold = K4Fold{h->map->d_keep, nullptr, (uint32_t)n_map_global, 0u};
        else if (S.fold_global) fold = K4Fold{S.fold_global, S.fold_index, (uint32_t)std::min<size_t>(S.fold_n, 0xFFFFFFFFu), 0u};
        if ((r = run_compare(h, h->p.version, S.mode, d_keep, nullptr, fold, with_c ? 7 : 3))) return r;
        h->last.with_c = with_c; h->last.host = host; h->last.mode = S.mode; h->last.d_keep = d_keep; h->last.user_keep = S.keep_mask; h->last.n_keep = n_keep;
        h->last.keep_out = S.keep_out; h->last.n_map_global = n_map_global; h->last.fold = fold;
        CK(cudaMemcpyAsync(h->h_words.as<uint32_t>() + 1, h->d_queue.as<uint32_t>() + kBucketC0, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
        if (host && n_keep) CK(cudaMemcpyAsync(S.keep_mask, d_keep, n_keep, cudaMemcpyDeviceToHost, h->stream));
        if (S.keep_out && n_map_global)
            CK(cudaMemcpyAsync(S.keep_out, h->map->d_keep, n_map_global, host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
        CK(cudaMemcpyAsync(h->h_words.as<uint32_t>(), h->d_nrecs.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
        return ERASOR_OK;
    };
    bool graphable = h->use_graphs && !h->timing;
    if (graphable && host) {
        // host buffers must be pinned for copies to be capturable
        if (S.mode == 1 && h->NM && !is_pinned_host(S.map_xyzi)) graphable = false;
        if (h->NQ && !is_pinned_host(S.qry_xyzi)) graphable = false;
        if (n_keep && !is_pinned_host(S.keep_mask)) graphable = false;
        if (S.keep_out && n_map_global && !is_pinned_host(S.keep_out)) graphable = false;
    }
    if (graphable) {
        erasor_ctx::StepGraph key{};
        key.ptr[0] = S.map_xyzi; key.ptr[1] = S.qry_xyzi; key.ptr[2] = S.keep_mask; key.ptr[3] = S.fold_index; key.ptr[4] = S.fold_global;
        key.ptr[5] = S.keep_out; key.ptr[6] = S.mode == 2 ? (const void*)h->map : nullptr; key.ptr[7] = with_c ? (const void*)h : nullptr;
        key.fold_n = S.fold_n; key.kind = S.ptr_kind | (S.qry_xyz || S.scan_xyz ? ERASOR_PTR_QUERY_XYZ : 0); key.mode = S.scan ? 3 : S.mode; key.f0 = S.f0;
        key.epoch = h->desc_epoch; key.alloc = h->alloc_epoch;
        for (int i = 0; i < 8; ++i) key.scan[i] = S.scan ? (i == 0 ? S.scan->query_voxel_size : S.scan->lidar2body[i - 1]) : 0.0;   // baked into the voxeliser's launch
        auto same = [&](const erasor_ctx::StepGraph& g) {
            return std::equal(g.ptr, g.ptr + 8, key.ptr) && g.fold_n == key.fold_n && g.kind == key.kind && g.mode == key.mode && g.f0 == key.f0 &&
                   g.epoch == key.epoch && g.alloc == key.alloc && std::equal(g.scan, g.scan + 8, key.scan);
        };
        cudaGraphExec_t exec = nullptr;
        for (auto& g : h->graphs) if (same(g)) exec = g.exec;
        if (!exec) {
            // drop graphs of older geometries, bound the cache
            for (size_t i = 0; i < h->graphs.size();) {
                if (h->graphs[i].epoch != h->desc_epoch || h->graphs[i].alloc != h->alloc_epoch || h->graphs.size() > 64) { cudaGraphExecDestroy(h->graphs[i].exec); h->graphs.erase(h->graphs.begin() + i); }
                else ++i;
            }
            cudaGraph_t graph = nullptr;
            const uint64_t launches_before = h->launches;
            CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeRelaxed));
            rc = enqueue();
            h->graph_kernel_nodes = h->launches - launches_before;
            h->launches = launches_before;                              // captured, not launched
            cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
            if (rc == ERASOR_OK && ce == cudaSuccess && graph && h->alloc_epoch == key.alloc) {
                ce = cudaGraphInstantiate(&exec, graph, 0);
                cudaGraphDestroy(graph);
                if (ce == cudaSuccess) { key.exec = exec; h->graphs.push_back(key); }
                else exec = nullptr;
            } else {
                if (graph) cudaGraphDestroy(graph);
                exec = nullptr;
            }
            if (!exec) { cudaGetLastError(); h->use_graphs = false; }      // capture not possible here: fall back to plain launches for good
        }
        if (exec) {
            CK(cudaGraphLaunch(exec, h->stream));
            h->launches += h->graph_kernel_nodes;                        // kernel nodes of the graph: init, K1, K3, K2, K4 classes
        } else if ((rc = enqueue())) {
            return rc;
        }
    } else {
        Scope whole(h, 0);
        if ((rc = enqueue())) return rc;
    }
    {   // what erasor_wait needs for the class-C fix-up (set here as well: a replayed graph does not run enqueue())
        const bool hst = S.ptr_kind != ERASOR_PTR_DEVICE;
        h->last.with_c = with_c; h->last.host = hst; h->last.mode = S.mode; h->last.user_keep = S.keep_mask; h->last.n_keep = n_keep;
        h->last.d_keep = n_keep ? (hst ? h->d_keep.as<uint8_t>() : S.keep_mask) : nullptr;
        h->last.keep_out = S.keep_out; h->last.n_map_global = n_map_global;
        if (S.mode == 2)        h->last.fold = K4Fold{h->map->d_keep, nullptr, (uint32_t)n_map_global, 0u};
        else if (S.fold_global) h->last.fold = K4Fold{S.fold_global, S.fold_index, (uint32_t)std::min<size_t>(S.fold_n, 0xFFFFFFFFu), 0u};
        else                    h->last.fold = K4Fold{nullptr, nullptr, 0u, 0u};
    }
    h->scan_F = S.scan ? S.F : 0;
    h->pending = true;
    return ERASOR_OK;
}

// frames [f0, f1) that fit one submission: < 2^32 points per side and at most kMaxRecords flagged-bin records
int sub_batch_end(const erasor_ctx* h, const uint64_t* map_off, const uint64_t* qry_off, int f0, int F) {
    const uint64_t lim = 0xFFFFFFF0ull;
    const int max_frames = (int)std::max<size_t>(1, kMaxRecords / (size_t)h->B);
    int f1 = f0;
    while (f1 < F && f1 - f0 < max_frames && map_off[f1 + 1] - map_off[f0] < lim && qry_off[f1 + 1] - qry_off[f0] < lim) ++f1;
    return f1;
}

int process_frames_impl(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets, const float* query_xyzi,
                        const uint64_t* query_offsets, int n_frames, uint8_t* keep_mask, int ptr_kind,
                        const uint32_t* fold_index, uint8_t* fold_global, size_t fold_n_global, bool async) {
    if (!h || !map_offsets || !query_offsets || !keep_mask) { if (h) h->err = "null argument"; return ERASOR_E_INVALID; }
    if (n_frames <= 0) { h->err = "n_frames must be positive"; return ERASOR_E_INVALID; }
    const bool qxyz = (ptr_kind & ERASOR_PTR_QUERY_XYZ) != 0;
    ptr_kind &= ~ERASOR_PTR_QUERY_XYZ;
    if (ptr_kind != ERASOR_PTR_HOST && ptr_kind != ERASOR_PTR_DEVICE) { h->err = "bad ptr_kind"; return ERASOR_E_INVALID; }
    int rc;
    if (h->pending && (rc = erasor_wait(h))) return rc;
    h->stat_F = n_frames;
    std::vector<uint64_t> mo, qo;
    for (int f0 = 0; f0 < n_frames;) {
        const int f1 = sub_batch_end(h, map_offsets, query_offsets, f0, n_frames);
        if (f1 == f0) { h->err = "a single frame exceeds 2^32 points"; return ERASOR_E_INVALID; }
        Submit S;
        S.mode = 1; S.F = f1 - f0; S.ptr_kind = ptr_kind; S.f0 = f0; S.qry_xyz = qxyz;
        const uint64_t m0 = map_offsets[f0], q0 = query_offsets[f0];
        if (f0 == 0 && f1 == n_frames) { S.map_off = map_offsets; S.qry_off = query_offsets; }
        else {
            mo.assign(map_offsets + f0, map_offsets + f1 + 1); qo.assign(query_offsets + f0, query_offsets + f1 + 1);
            for (auto& v : mo) v -= m0;
            for (auto& v : qo) v -= q0;
            S.map_off = mo.data(); S.qry_off = qo.data();
        }
        S.map_xyzi = map_xyzi ? map_xyzi + 4 * m0 : nullptr;
        S.qry_xyzi = query_xyzi ? query_xyzi + (qxyz ? 3 : 4) * q0 : nullptr;
        S.keep_mask = keep_mask + m0;
        S.fold_index = fold_index ? fold_index + m0 : nullptr; S.fold_global = fold_global; S.fold_n = fold_n_global;
        if ((rc = submit(h, S))) return rc;
        f0 = f1;
        if (f0 < n_frames && (rc = erasor_wait(h))) return rc;      // the next sub-batch reuses the handle's buffers
    }
    return async ? ERASOR_OK : erasor_wait(h);
}

// scan: erasor_process_scans -- query_xyzi holds raw scans, voxelised and moved to the body frame on the device first
int process_nodes_impl(erasor_handle_t h, const double* poses7, const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                       double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind, bool async,
                       const erasor_scan_params_t* scan = nullptr) {
    if (!h || !poses7 || !query_offsets) { if (h) h->err = "null argument"; return ERASOR_E_INVALID; }
    if (!h->map) { h->err = "erasor_process_nodes: no map attached (erasor_attach_map)"; return ERASOR_E_STATE; }
    if (n_frames <= 0) { h->err = "n_frames must be positive"; return ERASOR_E_INVALID; }
    const bool qxyz = (ptr_kind & ERASOR_PTR_QUERY_XYZ) != 0;
    ptr_kind &= ~ERASOR_PTR_QUERY_XYZ;
    if (ptr_kind != ERASOR_PTR_HOST && ptr_kind != ERASOR_PTR_DEVICE) { h->err = "bad ptr_kind"; return ERASOR_E_INVALID; }
    int rc;
    if (h->pending && (rc = erasor_wait(h))) return rc;
    const size_t N = h->map->n;
    const double range = voi_max_range > 0.0 ? voi_max_range : h->p.max_range;
    h->stat_F = n_frames;
    // scratch per (frame, map point): bin id 2 + scattered point 16 + source index 4 + class-C scratch 24 bytes
    size_t budget = (size_t)16 << 30;
    if (const char* e = std::getenv("ERASOR_B200_NODE_SCRATCH_GB")) budget = (size_t)std::max(1.0, std::atof(e)) << 30;
    const size_t by_mem = std::max<size_t>(1, budget / (46 * std::max<size_t>(N, 1)));
    const size_t by_idx = std::max<size_t>(1, (size_t)0xFFFFFFF0ull / std::max<size_t>(N, 1) - 1);
    const int max_frames = (int)std::min<size_t>({by_mem, by_idx, std::max<size_t>(1, kMaxRecords / (size_t)h->B), (size_t)n_frames});
    std::vector<uint64_t> mo, qo;
    std::vector<NodePose> poses;
    for (int f0 = 0; f0 < n_frames;) {
        int f1 = f0;
        while (f1 < n_frames && f1 - f0 < max_frames && query_offsets[f1 + 1] - query_offsets[f0] < 0xFFFFFFF0ull) ++f1;
        if (f1 == f0) { h->err = "a single query exceeds 2^32 points"; return ERASOR_E_INVALID; }
        const int F = f1 - f0;
        mo.resize((size_t)F + 1);
        for (int f = 0; f <= F; ++f) mo[f] = (uint64_t)f * N;
        const uint64_t q0 = query_offsets[f0];
        qo.assign(query_offsets + f0, query_offsets + f1 + 1);
        for (auto& v : qo) v -= q0;
        poses.resize(F);
        for (int f = 0; f < F; ++f) node_pose_of(poses7 + 7 * (size_t)(f0 + f), range, poses[f]);
        Submit S;
        S.mode = 2; S.F = F; S.ptr_kind = ptr_kind; S.f0 = f0; S.qry_xyz = scan ? false : qxyz;
        S.scan = scan; S.scan_xyz = scan ? qxyz : false;
        S.map_off = mo.data(); S.qry_off = qo.data();
        S.qry_xyzi = query_xyzi ? query_xyzi + (qxyz ? 3 : 4) * q0 : nullptr;
        S.keep_mask = frame_keep ? frame_keep + (size_t)f0 * N : nullptr;
        S.poses = poses.data();
        S.keep_out = (f1 == n_frames) ? keep_out : nullptr;
        if ((rc = submit(h, S))) return rc;
        f0 = f1;
        if (f0 < n_frames && (rc = erasor_wait(h))) return rc;
    }
    return async ? ERASOR_OK : erasor_wait(h);
}
}  // namespace

int erasor_wait(erasor_handle_t h) {
    if (!h) return ERASOR_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (h->pending) {
        h->pending = false;
        h->n_recs_host = h->words()[0];
        h->class_c_count_host = h->words()[1];
        if (h->n_recs_host > h->rec_capacity) { h->err = "internal: flagged-bin records overflowed the work queue"; return ERASOR_E_CAPACITY; }
        h->class_c_state = (int)std::min<uint32_t>(h->class_c_count_host, 0x7FFFFFFFu);
        if (!h->last.with_c && h->class_c_count_host > 0) {
            // bins beyond class B's capacity turned up in a submission that ran without class C: run that class now (R-GPF only; the
            // bins are independent, the masks only gain zeros), then repeat the output copies.  The next submissions launch it up front.
            int rc = run_compare(h, h->p.version, h->last.mode, h->last.d_keep, nullptr, h->last.fold, 4, true);
            if (rc) return rc;
            if (h->last.host && h->last.n_keep) CK(cudaMemcpyAsync(h->last.user_keep, h->last.d_keep, h->last.n_keep, cudaMemcpyDeviceToHost, h->stream));
            if (h->last.keep_out && h->last.n_map_global)
                CK(cudaMemcpyAsync(h->last.keep_out, h->map->d_keep, h->last.n_map_global, h->last.host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
            CK(cudaStreamSynchronize(h->stream));
        }
    }
    return ERASOR_OK;
}

int erasor_process_frames(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets, const float* query_xyzi,
                          const uint64_t* query_offsets, int n_frames, uint8_t* keep_mask, int ptr_kind) {
    return process_frames_impl(h, map_xyzi, map_offsets, query_xyzi, query_offsets, n_frames, keep_mask, ptr_kind, nullptr, nullptr, 0, false);
}
int erasor_process_frames_async(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets, const float* query_xyzi,
                                const uint64_t* query_offsets, int n_frames, uint8_t* keep_mask, int ptr_kind) {
    return process_frames_impl(h, map_xyzi, map_offsets, query_xyzi, query_offsets, n_frames, keep_mask, ptr_kind, nullptr, nullptr, 0, true);
}

int erasor_process_frames_fold(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets, const float* query_xyzi,
                               const uint64_t* query_offsets, int n_frames, uint8_t* keep_mask, int ptr_kind,
                               const uint32_t* voi_index, uint8_t* global_keep, size_t n_global) {
    if (!h) return ERASOR_E_INVALID;
    if (!voi_index || !global_keep) { h->err = "null fold argument"; return ERASOR_E_INVALID; }
    return process_frames_impl(h, map_xyzi, map_offsets, query_xyzi, query_offsets, n_frames, keep_mask, ptr_kind, voi_index, global_keep, n_global, false);
}
int erasor_process_frames_fold_async(erasor_handle_t h, const float* map_xyzi, const uint64_t* map_offsets, const float* query_xyzi,
                                     const uint64_t* query_offsets, int n_frames, uint8_t* keep_mask, int ptr_kind,
                                     const uint32_t* voi_index, uint8_t* global_keep, size_t n_global) {
    if (!h) return ERASOR_E_INVALID;
    if (!voi_index || !global_keep) { h->err = "null fold argument"; return ERASOR_E_INVALID; }
    return process_frames_impl(h, map_xyzi, map_offsets, query_xyzi, query_offsets, n_frames, keep_mask, ptr_kind, voi_index, global_keep, n_global, true);
}

// Multi-GPU exchange helper (DESIGN.md section 7): fold per-frame keep masks onto the global map
// (global_keep[voi_index[i]] = 0 where keep[i] == 0).  Accumulates; all pointers are DEVICE pointers; asynchronous on the
// handle's stream.  (erasor_process_frames_fold / erasor_process_nodes do this inside R-GPF's epilogue instead.)
int erasor_fold_keep_masks(erasor_handle_t h, const uint8_t* keep_mask, const uint32_t* voi_index, size_t n, uint8_t* global_keep, size_t n_global) {
    if (!h || !global_keep || (n && (!keep_mask || !voi_index))) { if (h) h->err = "null argument"; return ERASOR_E_INVALID; }
    if (n_global > 0xFFFFFFFFull) { h->err = "global map beyond 2^32 points"; return ERASOR_E_INVALID; }
    CK(cudaSetDevice(h->device));
    if (n) h->launches++;
    CK(launch_fold_keep(h->stream, keep_mask, voi_index, n, global_keep, n_global));
    return ERASOR_OK;
}

int erasor_reset_keep_mask(erasor_handle_t h, uint8_t* global_keep, size_t n_global) {
    if (!h || (n_global && !global_keep)) { if (h) h->err = "null argument"; return ERASOR_E_INVALID; }
    CK(cudaSetDevice(h->device));
    if (n_global) h->launches++;
    CK(launch_fill_u8(h->stream, global_keep, n_global, 1));
    return ERASOR_OK;
}

// ---- map-resident mode -------------------------------------------------------------------------------------------
int erasor_map_create(const float* map_xyzi, size_t n_map, int ptr_kind, int device, erasor_map_t* out) {
    if (!out || (n_map && !map_xyzi)) { g_create_error = "null argument"; return ERASOR_E_INVALID; }
    *out = nullptr;
    if (n_map >= 0xFFFFFFF0ull) { g_create_error = "map beyond 2^32 points"; return ERASOR_E_INVALID; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { g_create_error = "no CUDA device (this library has no CPU path)"; return ERASOR_E_CUDA; }
    if (device < 0 || device >= ndev) { g_create_error = "bad device index"; return ERASOR_E_INVALID; }
    erasor_map_ctx* m = new erasor_map_ctx();
    m->device = device; m->n = n_map;
    auto fail = [&](const char* what, cudaError_t ce) { g_create_error = std::string(what) + ": " + cudaGetErrorString(ce); erasor_map_destroy(m); return ERASOR_E_CUDA; };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&m->st, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaMalloc(&m->d_pts, sizeof(float4) * (n_map + kMapPad))) != cudaSuccess) return fail("cudaMalloc", e);
    if ((e = cudaMemsetAsync(m->d_pts + n_map, 0, sizeof(float4) * kMapPad, m->st)) != cudaSuccess) return fail("cudaMemset", e);
    if ((e = cudaMalloc(&m->d_keep, std::max<size_t>(n_map, 1))) != cudaSuccess) return fail("cudaMalloc", e);
    if (n_map) {
        const cudaMemcpyKind k = ptr_kind == ERASOR_PTR_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        if ((e = cudaMemcpyAsync(m->d_pts, map_xyzi, sizeof(float4) * n_map, k, m->st)) != cudaSuccess) return fail("cudaMemcpy", e);
        if ((e = cudaMemsetAsync(m->d_keep, 1, n_map, m->st)) != cudaSuccess) return fail("cudaMemset", e);
    }
    if ((e = cudaStreamSynchronize(m->st)) != cudaSuccess) return fail("cudaStreamSynchronize", e);
    *out = m;
    return ERASOR_OK;
}

void erasor_map_destroy(erasor_map_t m) {
    if (!m) return;
    cudaSetDevice(m->device);
    if (m->st) { cudaStreamSynchronize(m->st); cudaStreamDestroy(m->st); }
    if (m->d_pts) cudaFree(m->d_pts);
    if (m->d_keep) cudaFree(m->d_keep);
    delete m;
}

size_t erasor_map_size(erasor_map_t m) { return m ? m->n : 0; }
uint8_t* erasor_map_keep_device(erasor_map_t m) { return m ? m->d_keep : nullptr; }
const float* erasor_map_points_device(erasor_map_t m) { return m ? reinterpret_cast<const float*>(m->d_pts) : nullptr; }

int erasor_map_reset_keep(erasor_map_t m) {
    if (!m) return ERASOR_E_INVALID;
    if (cudaSetDevice(m->device) != cudaSuccess) return ERASOR_E_CUDA;
    if (m->n && cudaMemsetAsync(m->d_keep, 1, m->n, m->st) != cudaSuccess) return ERASOR_E_CUDA;
    return cudaStreamSynchronize(m->st) == cudaSuccess ? ERASOR_OK : ERASOR_E_CUDA;
}

int erasor_map_get_keep(erasor_map_t m, uint8_t* keep, int ptr_kind) {
    if (!m || (m->n && !keep)) return ERASOR_E_INVALID;
    if (cudaSetDevice(m->device) != cudaSuccess) return ERASOR_E_CUDA;
    const cudaMemcpyKind k = ptr_kind == ERASOR_PTR_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (m->n && cudaMemcpyAsync(keep, m->d_keep, m->n, k, m->st) != cudaSuccess) return ERASOR_E_CUDA;
    return cudaStreamSynchronize(m->st) == cudaSuccess ? ERASOR_OK : ERASOR_E_CUDA;
}

int erasor_attach_map(erasor_handle_t h, erasor_map_t m) {
    if (!h) return ERASOR_E_INVALID;
    if (m && m->device != h->device) { h->err = "map and handle live on different devices"; return ERASOR_E_INVALID; }
    int rc;
    if (h->pending && (rc = erasor_wait(h))) return rc;
    h->map = m;
    h->desc_mode = -1;
    return ERASOR_OK;
}

int erasor_process_nodes(erasor_handle_t h, const double* poses7, const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                         double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind) {
    return process_nodes_impl(h, poses7, query_xyzi, query_offsets, n_frames, voi_max_range, frame_keep, keep_out, ptr_kind, false);
}
int erasor_process_nodes_async(erasor_handle_t h, const double* poses7, const float* query_xyzi, const uint64_t* query_offsets, int n_frames,
                               double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind) {
    return process_nodes_impl(h, poses7, query_xyzi, query_offsets, n_frames, voi_max_range, frame_keep, keep_out, ptr_kind, true);
}

namespace {
int process_scans_impl(erasor_handle_t h, const erasor_scan_params_t* sp, const double* poses7, const float* scans, const uint64_t* scan_offsets,
                       int n_frames, double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind, bool async) {
    if (!h) return ERASOR_E_INVALID;
    if (!sp || !poses7 || !scan_offsets) { h->err = "null argument"; return ERASOR_E_INVALID; }
    const double leaf = sp->query_voxel_size;
    if (!(leaf > 0.0) || !std::isfinite(leaf) || !((float)leaf > 0.0f) || !std::isfinite((float)leaf)) { h->err = "query_voxel_size must be positive and finite"; return ERASOR_E_INVALID; }
    double qn = 0.0;
    for (int i = 0; i < 7; ++i) { if (!std::isfinite(sp->lidar2body[i])) { h->err = "lidar2body must be finite"; return ERASOR_E_INVALID; } }
    for (int i = 3; i < 7; ++i) qn += sp->lidar2body[i] * sp->lidar2body[i];
    if (!(qn > 0.0)) { h->err = "lidar2body: zero quaternion"; return ERASOR_E_INVALID; }
    if (n_frames > 0) {
        for (size_t i = 0; i < 7 * (size_t)n_frames; ++i) if (!std::isfinite(poses7[i])) { h->err = "poses must be finite"; return ERASOR_E_INVALID; }
        for (int f = 0; f < n_frames; ++f) if (scan_offsets[f + 1] < scan_offsets[f]) { h->err = "offsets must be non-decreasing"; return ERASOR_E_INVALID; }
        if (scan_offsets[n_frames] > scan_offsets[0] && !scans) { h->err = "null cloud"; return ERASOR_E_INVALID; }
    }
    return process_nodes_impl(h, poses7, scans, scan_offsets, n_frames, voi_max_range, frame_keep, keep_out, ptr_kind, async, sp);
}
}  // namespace

int erasor_process_scans(erasor_handle_t h, const erasor_scan_params_t* sp, const double* poses7, const float* scans, const uint64_t* scan_offsets,
                         int n_frames, double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind) {
    return process_scans_impl(h, sp, poses7, scans, scan_offsets, n_frames, voi_max_range, frame_keep, keep_out, ptr_kind, false);
}
int erasor_process_scans_async(erasor_handle_t h, const erasor_scan_params_t* sp, const double* poses7, const float* scans, const uint64_t* scan_offsets,
                               int n_frames, double voi_max_range, uint8_t* frame_keep, uint8_t* keep_out, int ptr_kind) {
    return process_scans_impl(h, sp, poses7, scans, scan_offsets, n_frames, voi_max_range, frame_keep, keep_out, ptr_kind, true);
}

int erasor_get_scan_queries(erasor_handle_t h, float* xyz, size_t cap, uint64_t* offsets) {
    if (!h) return ERASOR_E_INVALID;
    if (!offsets) { h->err = "null argument"; return ERASOR_E_INVALID; }
    if (h->scan_F <= 0) { h->err = "the last submission did not come from erasor_process_scans"; return ERASOR_E_STATE; }
    int rc;
    if ((rc = erasor_wait(h))) return rc;
    const int F = h->scan_F;
    std::vector<uint32_t> cnt((size_t)F);
    CK(cudaMemcpy(cnt.data(), h->d_scan_cnt.p, sizeof(uint32_t) * (size_t)F, cudaMemcpyDeviceToHost));
    offsets[0] = 0;
    for (int f = 0; f < F; ++f) offsets[f + 1] = offsets[f] + cnt[f];
    if (!xyz) return ERASOR_OK;
    if (cap < offsets[F]) { h->err = "output buffer too small"; return ERASOR_E_CAPACITY; }
    std::vector<float4> tmp;
    for (int f = 0; f < F; ++f) {
        tmp.resize(cnt[f]);
        if (cnt[f]) CK(cudaMemcpy(tmp.data(), h->d_scan_q.as<float4>() + h->qry_off[f], sizeof(float4) * cnt[f], cudaMemcpyDeviceToHost));
        float* o = xyz + 3 * offsets[f];
        for (uint32_t i = 0; i < cnt[f]; ++i) { o[3 * i] = tmp[i].x; o[3 * i + 1] = tmp[i].y; o[3 * i + 2] = tmp[i].z; }
    }
    return ERASOR_OK;
}

// OfflineMapUpdater::save_static_map (OfflineMapUpdater.cpp:174-196) on the attached map: keep-byte compaction, then U3 with labels
int erasor_save_static_map(erasor_handle_t h, float voxel_size, float* out_xyzi, size_t cap, size_t* n) {
    if (!h) return ERASOR_E_INVALID;
    if (!n) { h->err = "null argument"; return ERASOR_E_INVALID; }
    if (!h->map) { h->err = "erasor_save_static_map: no map attached (erasor_attach_map)"; return ERASOR_E_STATE; }
    if (!(voxel_size > 0.0f) || !std::isfinite(voxel_size)) { h->err = "voxel_size must be positive and finite"; return ERASOR_E_INVALID; }
    int rc;
    if ((rc = erasor_wait(h))) return rc;
    CK(cudaStreamSynchronize(h->map->st));
    const size_t N = h->map->n;
    CK(h->d_sv_pts.ensure(sizeof(float4) * std::max<size_t>(N, 1)));
    CK(h->d_sv_tmp.ensure(sizeof(uint32_t) * (partition_tmp_words((uint32_t)N) + 2)));
    uint32_t* d_cnt = h->d_sv_tmp.as<uint32_t>();                   // [0] kept points, [1] voxels, [2..) chunk counters
    h->launches += 3;
    CK(launch_compact_keep(h->stream, h->map->d_pts, h->map->d_keep, (uint32_t)N, h->d_sv_pts.as<float4>(), d_cnt, d_cnt + 2));
    uint32_t* w = h->h_words.as<uint32_t>();
    CK(cudaMemcpyAsync(w + 12, d_cnt, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const uint32_t nk = w[12];
    CK(h->d_sv_out.ensure(sizeof(float4) * std::max<size_t>(nk, 1)));
    CK(h->d_sv_grid.ensure(sizeof(VoxGrid)));
    CK(h->d_sv_vtmp.ensure(voxelize_tmp_bytes(nk)));
    FusedJob J{};
    J.vin = h->d_sv_pts.as<float4>(); J.vn = nk; J.leaf = voxel_size; J.grid = h->d_sv_grid.as<VoxGrid>(); J.vtmp = h->d_sv_vtmp.p;
    J.vout = h->d_sv_out.as<float4>(); J.d_n_out = d_cnt + 1; J.xform_out = 0;
    h->launches++;
    CK(launch_node_fused(h->stream, J, h->sm_count));
    CK(cudaMemcpyAsync(w + 13, d_cnt + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const uint32_t nv = w[13];
    *n = nv;
    if (!out_xyzi) return ERASOR_OK;
    if (cap < nv) { h->err = "output buffer too small"; return ERASOR_E_CAPACITY; }
    if (nv) CK(cudaMemcpy(out_xyzi, h->d_sv_out.p, sizeof(float4) * nv, cudaMemcpyDeviceToHost));
    return ERASOR_OK;
}

int erasor_get_node_stats(erasor_handle_t h, uint32_t* n_voi_points, uint32_t* n_flagged_bins, uint32_t* n_rejected_points) {
    if (!h) return ERASOR_E_INVALID;
    if (h->F <= 0 || h->desc_mode < 2) { h->err = "no node batch has run"; return ERASOR_E_STATE; }
    int rc;
    if ((rc = erasor_wait(h))) return rc;
    if (n_voi_points) {
        // |map_voi_| of every node of the LAST submission = binned + complement counts of the map cloud (K1's tables)
        const size_t row = (size_t)h->B + 1;
        std::vector<uint32_t> c((size_t)h->F * row);
        CK(cudaMemcpy(c.data(), h->d_cnt.p, sizeof(uint32_t) * c.size(), cudaMemcpyDeviceToHost));
        for (int f = 0; f < h->F; ++f) {
            uint64_t t = 0;
            for (size_t b = 0; b < row; ++b) t += c[(size_t)f * row + b];
            n_voi_points[h->f0 + f] = (uint32_t)t;
        }
    }
    if (n_flagged_bins) CK(cudaMemcpy(n_flagged_bins, h->d_nflag.p, sizeof(uint32_t) * h->stat_F, cudaMemcpyDeviceToHost));
    if (n_rejected_points) CK(cudaMemcpy(n_rejected_points, h->d_frame_rej.p, sizeof(uint32_t) * h->stat_F, cudaMemcpyDeviceToHost));
    return ERASOR_OK;
}

// ---- the path's single collective ---------------------------------------------------------------------------------
int erasor_comm_unique_id(uint8_t* id128) {
    if (!id128) return ERASOR_E_INVALID;
    NcclApi* api = nccl_api(g_create_error);
    if (!api) return ERASOR_E_UNSUPPORTED;
    static_assert(sizeof(ncclUniqueId) == ERASOR_COMM_ID_BYTES, "NCCL unique id size");
    ncclUniqueId id;
    const ncclResult_t r = api->GetUniqueId(&id);
    if (r != ncclSuccess) { g_create_error = std::string("ncclGetUniqueId: ") + api->GetErrorString(r); return ERASOR_E_CUDA; }
    std::memcpy(id128, &id, sizeof(id));
    return ERASOR_OK;
}

int erasor_comm_init(erasor_handle_t h, const uint8_t* id128, int n_ranks, int rank) {
    if (!h || !id128 || n_ranks < 1 || rank < 0 || rank >= n_ranks) { if (h) h->err = "bad communicator arguments"; return ERASOR_E_INVALID; }
    NcclApi* api = nccl_api(h->err);
    if (!api) return ERASOR_E_UNSUPPORTED;
    CK(cudaSetDevice(h->device));
    if (h->comm) { api->CommDestroy(h->comm); h->comm = nullptr; }
    ncclUniqueId id;
    std::memcpy(&id, id128, sizeof(id));
    const ncclResult_t r = api->CommInitRank(&h->comm, n_ranks, id, rank);
    if (r != ncclSuccess) { h->comm = nullptr; h->err = std::string("ncclCommInitRank: ") + api->GetErrorString(r); return ERASOR_E_CUDA; }
    h->comm_ranks = n_ranks; h->comm_rank = rank;
    return ERASOR_OK;
}

int erasor_comm_destroy(erasor_handle_t h) {
    if (!h) return ERASOR_E_INVALID;
    if (h->comm) {
        NcclApi* api = nccl_api(h->err);
        if (!api) return ERASOR_E_UNSUPPORTED;
        CK(cudaSetDevice(h->device));
        CK(cudaStreamSynchronize(h->stream));
        api->CommDestroy(h->comm);
        h->comm = nullptr; h->comm_ranks = 1; h->comm_rank = 0;
    }
    return ERASOR_OK;
}

// The local half of the exchange on its own (what runs after the all-gather): AND n_masks byte masks of n points each
// (DEVICE, contiguous [n_masks][n]) through the bit-packed form into out (DEVICE, n bytes).  Lets a single-GPU test and
// a caller with its own transport use the library's pack / AND kernels.
int erasor_and_keep_masks(erasor_handle_t h, const uint8_t* masks, int n_masks, size_t n, uint8_t* out) {
    if (!h || n_masks < 1 || (n && (!masks || !out))) { if (h) h->err = "bad argument"; return ERASOR_E_INVALID; }
    if (n == 0) return ERASOR_OK;
    CK(cudaSetDevice(h->device));
    const size_t words = (n + 31) / 32;
    CK(h->d_gather.ensure(sizeof(uint32_t) * words * (size_t)n_masks));
    for (int r = 0; r < n_masks; ++r) {
        h->launches++;
        CK(launch_pack_keep_bits(h->stream, masks + (size_t)r * n, n, h->d_gather.as<uint32_t>() + (size_t)r * words));
    }
    h->launches++;
    CK(launch_and_unpack_keep(h->stream, h->d_gather.as<uint32_t>(), n_masks, n, out));
    return ERASOR_OK;
}

int erasor_allgather_and_keep(erasor_handle_t h, uint8_t* global_keep, size_t n_global) {
    if (!h || (n_global && !global_keep)) { if (h) h->err = "null argument"; return ERASOR_E_INVALID; }
    if (!h->comm || h->comm_ranks <= 1 || n_global == 0) return ERASOR_OK;      // one rank: the folded mask is already the answer
    NcclApi* api = nccl_api(h->err);
    if (!api) return ERASOR_E_UNSUPPORTED;
    CK(cudaSetDevice(h->device));
    const size_t words = (n_global + 31) / 32;
    CK(h->d_pack.ensure(sizeof(uint32_t) * words));
    CK(h->d_gather.ensure(sizeof(uint32_t) * words * (size_t)h->comm_ranks));
    h->launches += 2;
    CK(launch_pack_keep_bits(h->stream, global_keep, n_global, h->d_pack.as<uint32_t>()));
    const ncclResult_t r = api->AllGather(h->d_pack.p, h->d_gather.p, words, ncclUint32, h->comm, h->stream);
    if (r != ncclSuccess) { h->err = std::string("ncclAllGather: ") + api->GetErrorString(r); return ERASOR_E_CUDA; }
    CK(launch_and_unpack_keep(h->stream, h->d_gather.as<uint32_t>(), h->comm_ranks, n_global, global_keep));
    return ERASOR_OK;
}

int erasor_get_frame_stats(erasor_handle_t h, uint32_t* n_flagged_bins, uint32_t* n_rejected_points) {
    if (!h) return ERASOR_E_INVALID;
    if (h->F <= 0) { h->err = "no batch has run"; return ERASOR_E_STATE; }
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    const int nf = std::max(h->stat_F, h->F);
    if (n_flagged_bins) CK(cudaMemcpy(n_flagged_bins, h->d_nflag.p, sizeof(uint32_t) * nf, cudaMemcpyDeviceToHost));
    if (n_rejected_points) CK(cudaMemcpy(n_rejected_points, h->d_frame_rej.p, sizeof(uint32_t) * nf, cudaMemcpyDeviceToHost));
    return ERASOR_OK;
}

// instrumentation: per flagged bin of the last run, n_points and the SM cycles thread 0 spent per phase
// (load + index sort, z sort, seeds, accumulate, SVD + plane, classify + compact, outputs) and the Jacobi sweep count
int erasor_get_rgpf_profile(erasor_handle_t h, uint32_t* n_points, uint32_t* prof8, size_t* n) {
    if (!h || !n) return ERASOR_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    uint32_t nr = 0;
    CK(cudaMemcpy(&nr, h->d_nrecs.p, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    nr = std::min(nr, h->rec_capacity);
    const size_t cap = *n;
    *n = nr;
    if (!n_points && !prof8) return ERASOR_OK;
    if (cap < nr) { h->err = "profile buffer too small"; return ERASOR_E_CAPACITY; }
    std::vector<FlagRec> recs(nr);
    if (nr) CK(cudaMemcpy(recs.data(), h->d_recs.p, sizeof(FlagRec) * nr, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < nr; ++i) {
        if (n_points) n_points[i] = recs[i].n_points;
        if (prof8) for (int k = 0; k < 8; ++k) prof8[i * 8 + k] = recs[i].prof[k];
    }
    return ERASOR_OK;
}

int erasor_get_srt_profile(erasor_handle_t h, uint32_t* cycles8) {
    if (!h || !cycles8) return ERASOR_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (!h->d_queue.p) { h->err = "no run yet"; return ERASOR_E_STATE; }
    CK(cudaMemcpy(cycles8, h->d_queue.as<uint32_t>() + 20, sizeof(uint32_t) * 8, cudaMemcpyDeviceToHost));
    return ERASOR_OK;
}

uint64_t erasor_kernel_launch_count(erasor_handle_t h) { return h ? h->launches : 0; }

int erasor_reset_kernel_times(erasor_handle_t h, int enable_timing) {
    if (!h) return ERASOR_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    drain_timers(h);
    for (auto& t : h->timers) { t.total_ms = 0; t.launches = 0; }
    h->timing = enable_timing != 0;
    return ERASOR_OK;
}

int erasor_get_kernel_time_ms(erasor_handle_t h, int kernel_id, double* total_ms, uint64_t* launches) {
    if (!h || kernel_id < 0 || kernel_id >= kNumTimers) return ERASOR_E_INVALID;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    drain_timers(h);
    if (total_ms) *total_ms = h->timers[kernel_id].total_ms;
    if (launches) *launches = h->timers[kernel_id].launches;
    return ERASOR_OK;
}

}  // extern "C"
