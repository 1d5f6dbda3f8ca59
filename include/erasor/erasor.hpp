// include/erasor/erasor.hpp -- ROS-free C++ host mirror of the reference's `class ERASOR`
// (reference include/erasor/erasor.h:43-147) on top of the C ABI in include/erasor_b200.h.
//
// Same public method names, argument meaning, call order and error behaviour (exceptions) as the
// reference, so that OfflineMapUpdater::callback_node (OfflineMapUpdater.cpp:266-284) compiles against it
// with two substitutions only:
//     pcl::PointCloud<pcl::PointXYZI>   ->  erasor_b200::PointCloud   (x, y, z, intensity; 16 bytes)
//     ERASOR(ros::NodeHandle*)          ->  ERASOR(const erasor_params_t&)   (the same /erasor/* keys)
// Everything the methods compute runs in the sm_100a kernels behind the C ABI; this header holds no
// arithmetic.  The rviz / debug publishers of the reference (erasor.h:67-77) are not mirrored.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../erasor_b200.h"

namespace erasor_b200 {

struct PointXYZI {          // the four floats of pcl::PointXYZI that the path uses
    float x, y, z, intensity;
};
static_assert(sizeof(PointXYZI) == 16, "PointXYZI must be one float4");
using PointCloud = std::vector<PointXYZI>;

// defaults of erasor.h:47-61 and OfflineMapUpdater.cpp:81
inline erasor_params_t default_params() {
    erasor_params_t p{};
    p.max_range = 10.0; p.num_rings = 20; p.num_sectors = 60; p.max_h = 3.0; p.min_h = 0.0; p.th_bin_max_h = 0.39;
    p.scan_ratio_threshold = 0.22; p.num_lowest_pts = 5; p.minimum_num_pts = 4; p.rejection_ratio = 0.33;
    p.gf_dist_thr = 0.05; p.gf_iter = 3; p.gf_num_lpr = 10; p.gf_th_seeds_height = 0.5; p.map_voxel_size = 0.2;
    p.version = 3; p.cov_mode = 0; p.sort_mode = 1; p.skip_voxelize = 0;
    return p;
}

class ERASOR {
public:
    // replaces ERASOR(ros::NodeHandle*): parameters are read once, R-PODs are allocated once (erasor.h:46-103)
    explicit ERASOR(const erasor_params_t& params, int device = 0) : params_(params), device_(device) {
        const int rc = erasor_create(&params_, device, &h_);
        if (rc != ERASOR_OK) throw std::runtime_error(std::string("ERASOR: ") + erasor_last_error(nullptr));
    }
    ~ERASOR() { erasor_destroy(h_); if (map_) erasor_map_destroy(map_); }
    ERASOR(const ERASOR&) = delete;
    ERASOR& operator=(const ERASOR&) = delete;

    // Inputs: transformed & cut pcs, both in the egocentric body frame (erasor.cpp:54-59)
    void set_inputs(const PointCloud& map_voi, const PointCloud& query_voi) {
        check(erasor_set_inputs(h_, reinterpret_cast<const float*>(map_voi.data()), map_voi.size(),
                                reinterpret_cast<const float*>(query_voi.data()), query_voi.size(), ERASOR_PTR_HOST));
    }
    // Version 2 algorithm (erasor.cpp:332-434)
    void compare_vois_and_revert_ground(int frame) { check(erasor_compare(h_, 2, frame)); }
    // Version 3 algorithm (erasor.cpp:438-571)
    void compare_vois_and_revert_ground_w_block(int frame) { check(erasor_compare(h_, 3, frame)); }

    void get_static_estimate(PointCloud& arranged, PointCloud& complement) {   // erasor.cpp:612-626
        size_t na = 0, nc = 0;
        check(erasor_get_output_sizes(h_, &na, &nc, nullptr, nullptr));
        arranged.resize(na); complement.resize(nc);
        check(erasor_get_static_estimate(h_, reinterpret_cast<float*>(arranged.data()), na, &na,
                                         reinterpret_cast<float*>(complement.data()), nc, &nc, ERASOR_PTR_HOST));
    }
    void get_outliers(PointCloud& map_rejected, PointCloud& curr_rejected) {   // erasor.cpp:322-327
        size_t nm = 0, nq = 0;
        check(erasor_get_output_sizes(h_, nullptr, nullptr, &nm, &nq));
        map_rejected.resize(nm); curr_rejected.resize(nq);
        check(erasor_get_outliers(h_, reinterpret_cast<float*>(map_rejected.data()), nm, &nm,
                                  reinterpret_cast<float*>(curr_rejected.data()), nq, &nq, ERASOR_PTR_HOST));
    }
    double get_max_range() { return erasor_get_max_range(h_); }               // erasor.cpp:628

    // ---- the reference's public data members (erasor.h:127, 139-145), refreshed by refresh_debug_members() ----------
    // The reference fills them as a side effect of compare_*; here they cost device -> host copies, so they are filled on
    // request: call refresh_debug_members() after compare_* (OfflineMapUpdater.cpp never reads them; rviz publishers do).
    PointCloud ground_viz;             // erasor.h:127  ground points of the flagged bins (also the tail of `arranged`)
    PointCloud debug_curr_rejected;    // erasor.h:139
    PointCloud debug_map_rejected;     // erasor.h:140
    PointCloud map_complement;         // erasor.h:141
    void refresh_debug_members() {
        size_t ng = 0;
        check(erasor_get_ground_viz(h_, nullptr, 0, &ng, ERASOR_PTR_HOST));
        ground_viz.resize(ng);
        if (ng) check(erasor_get_ground_viz(h_, reinterpret_cast<float*>(ground_viz.data()), ng, &ng, ERASOR_PTR_HOST));
        get_outliers(debug_map_rejected, debug_curr_rejected);
        PointCloud arranged_unused;
        get_static_estimate(arranged_unused, map_complement);
    }
    // r_pod_map / r_pod_curr (erasor.h:143-144) as flat tables: bin = sector * num_rings + ring.  which: ERASOR_CLOUD_MAP / _QUERY
    struct RPodTables { std::vector<int32_t> bin_of_point; std::vector<float> min_h, max_h; std::vector<uint32_t> count; };
    RPodTables r_pod(int which, size_t n_points) {
        RPodTables t;
        const size_t B = static_cast<size_t>(params_.num_rings) * params_.num_sectors;
        t.bin_of_point.resize(n_points); t.min_h.resize(B); t.max_h.resize(B); t.count.resize(B);
        check(erasor_get_bins(h_, which, t.bin_of_point.data(), t.min_h.data(), t.max_h.data(), t.count.data()));
        return t;
    }
    // ERASOR::is_dynamic_obj_close (public, erasor.h:132 / erasor.cpp:573-595) on the status of the last compare: is any of
    // the 8 neighbours of bin (r_target, theta_target) CURR_IS_HIGHER?  The theta wrap uses num_rings like the reference
    // (sic, SURVEY App. B-2); candidates that wrap out of range are skipped (the reference would index out of bounds).
    bool is_dynamic_obj_close(int r_target, int theta_target, int r_size = 1, int theta_size = 1) {
        const std::vector<float> st = get_status();
        const int R = params_.num_rings, S = params_.num_sectors;
        for (int j = theta_target - theta_size; j <= theta_target + theta_size; ++j) {
            int tj = j;
            if (j < 0) tj = j + R; else if (j >= S) tj = j - R;
            if (tj < 0 || tj >= S) continue;
            for (int r = std::max(0, r_target - r_size); r <= std::min(r_target + r_size, R - 1); ++r) {
                if (r == r_target && tj == theta_target) continue;
                if (st[static_cast<size_t>(tj) * R + r] == ERASOR_STATUS_CURR_IS_HIGHER) return true;
            }
        }
        return false;
    }

    // Frame-independent batch mode (no counterpart in the reference; BASELINE.json north_star): F independent
    // (map VoI, query VoI) pairs in one submission.  keep[f][i] == 0 where frame f rejects the i-th point of its map VoI.
    std::vector<std::vector<uint8_t>> process_frames(const std::vector<PointCloud>& map_vois, const std::vector<PointCloud>& query_vois) {
        if (map_vois.size() != query_vois.size() || map_vois.empty()) throw std::invalid_argument("ERASOR: one query VoI per map VoI");
        const size_t F = map_vois.size();
        std::vector<uint64_t> mo(F + 1, 0), qo(F + 1, 0);
        for (size_t f = 0; f < F; ++f) { mo[f + 1] = mo[f] + map_vois[f].size(); qo[f + 1] = qo[f] + query_vois[f].size(); }
        PointCloud m(mo[F]), q(qo[F]);
        for (size_t f = 0; f < F; ++f) {
            std::copy(map_vois[f].begin(), map_vois[f].end(), m.begin() + static_cast<std::ptrdiff_t>(mo[f]));
            std::copy(query_vois[f].begin(), query_vois[f].end(), q.begin() + static_cast<std::ptrdiff_t>(qo[f]));
        }
        std::vector<uint8_t> keep(mo[F] ? mo[F] : 1);
        check(erasor_process_frames(h_, reinterpret_cast<const float*>(m.data()), mo.data(), reinterpret_cast<const float*>(q.data()), qo.data(),
                                    static_cast<int>(F), keep.data(), ERASOR_PTR_HOST));
        std::vector<std::vector<uint8_t>> out(F);
        for (size_t f = 0; f < F; ++f) out[f].assign(keep.begin() + static_cast<std::ptrdiff_t>(mo[f]), keep.begin() + static_cast<std::ptrdiff_t>(mo[f + 1]));
        return out;
    }

    // ---- map-resident frame-independent mode + the single collective (north_star's multi-GPU form), C++ face ---------
    // Upload the global map once (load_global_map), then per batch only poses + body-frame queries cross PCIe.
    void load_global_map(const PointCloud& map_origin_frame) {
        if (map_) { erasor_attach_map(h_, nullptr); erasor_map_destroy(map_); map_ = nullptr; }
        int dev = 0;
        if (erasor_map_create(reinterpret_cast<const float*>(map_origin_frame.data()), map_origin_frame.size(), ERASOR_PTR_HOST, device_, &map_) != ERASOR_OK)
            throw std::runtime_error(std::string("ERASOR: ") + erasor_last_error(nullptr));
        (void)dev;
        check(erasor_attach_map(h_, map_));
    }
    // poses: x y z qx qy qz qw (body -> origin) per node; queries voxelised and in the body frame.  Returns the map's keep
    // mask after this batch (1 = static so far); it accumulates over calls (reset_static_mask() starts a job).
    std::vector<uint8_t> process_nodes(const std::vector<std::array<double, 7>>& poses, const std::vector<PointCloud>& query_vois, double voi_max_range = 0.0) {
        if (!map_) throw std::logic_error("ERASOR: load_global_map first");
        if (poses.size() != query_vois.size() || poses.empty()) throw std::invalid_argument("ERASOR: one pose per query VoI");
        const size_t F = poses.size();
        std::vector<uint64_t> qo(F + 1, 0);
        for (size_t f = 0; f < F; ++f) qo[f + 1] = qo[f] + query_vois[f].size();
        PointCloud q(qo[F]);
        for (size_t f = 0; f < F; ++f) std::copy(query_vois[f].begin(), query_vois[f].end(), q.begin() + static_cast<std::ptrdiff_t>(qo[f]));
        std::vector<uint8_t> keep(std::max<size_t>(erasor_map_size(map_), 1));
        check(erasor_process_nodes(h_, poses[0].data(), reinterpret_cast<const float*>(q.data()), qo.data(), static_cast<int>(F), voi_max_range,
                                   nullptr, keep.data(), ERASOR_PTR_HOST));
        keep.resize(erasor_map_size(map_));
        return keep;
    }
    // The same on raw scans in the LiDAR frame: every scan is voxelised at query_voxel_size and moved by lidar2body
    // (x y z qx qy qz qw) on the device first, as callback_node prepares its query (OfflineMapUpdater.cpp:237-241).
    std::vector<uint8_t> process_scans(const std::vector<std::array<double, 7>>& poses, const std::vector<PointCloud>& scans, double query_voxel_size,
                                       const std::array<double, 7>& lidar2body, double voi_max_range = 0.0) {
        if (!map_) throw std::logic_error("ERASOR: load_global_map first");
        if (poses.size() != scans.size() || poses.empty()) throw std::invalid_argument("ERASOR: one pose per scan");
        const size_t F = poses.size();
        std::vector<uint64_t> so(F + 1, 0);
        for (size_t f = 0; f < F; ++f) so[f + 1] = so[f] + scans[f].size();
        PointCloud s(so[F]);
        for (size_t f = 0; f < F; ++f) std::copy(scans[f].begin(), scans[f].end(), s.begin() + static_cast<std::ptrdiff_t>(so[f]));
        erasor_scan_params_t sp{};
        sp.query_voxel_size = query_voxel_size;
        std::copy(lidar2body.begin(), lidar2body.end(), sp.lidar2body);
        std::vector<uint8_t> keep(std::max<size_t>(erasor_map_size(map_), 1));
        check(erasor_process_scans(h_, &sp, poses[0].data(), reinterpret_cast<const float*>(s.data()), so.data(), static_cast<int>(F), voi_max_range,
                                   nullptr, keep.data(), ERASOR_PTR_HOST));
        keep.resize(erasor_map_size(map_));
        return keep;
    }
    // save_static_map of the resident map: voxelize_preserving_labels(map[keep], voxel_size) (OfflineMapUpdater.cpp:174-196)
    PointCloud save_static_map(float voxel_size) {
        if (!map_) throw std::logic_error("ERASOR: load_global_map first");
        size_t n = 0;
        check(erasor_save_static_map(h_, voxel_size, nullptr, 0, &n));
        PointCloud out(n);
        if (n) check(erasor_save_static_map(h_, voxel_size, reinterpret_cast<float*>(out.data()), n, &n));
        return out;
    }
    void reset_static_mask() { if (map_ && erasor_map_reset_keep(map_) != ERASOR_OK) throw std::runtime_error("ERASOR: erasor_map_reset_keep"); }
    // frame-sharded job: every rank processes its own nodes, then ONE all-gather (bit-packed masks over NVLink) + AND gives
    // every rank the job's static mask.  id128 from erasor_comm_unique_id() on rank 0, shipped by the host program.
    void init_communicator(const uint8_t* id128, int n_ranks, int rank) { check(erasor_comm_init(h_, id128, n_ranks, rank)); }
    std::vector<uint8_t> allgather_static_mask() {
        if (!map_) throw std::logic_error("ERASOR: load_global_map first");
        const size_t n = erasor_map_size(map_);
        check(erasor_allgather_and_keep(h_, erasor_map_keep_device(map_), n));
        check(erasor_synchronize(h_));
        std::vector<uint8_t> keep(std::max<size_t>(n, 1));
        if (erasor_map_get_keep(map_, keep.data(), ERASOR_PTR_HOST) != ERASOR_OK) throw std::runtime_error("ERASOR: erasor_map_get_keep");
        keep.resize(n);
        return keep;
    }

    // what the reference exposes as /SCDR/debug/polygons_marker likelihoods (erasor.cpp:439-441,570);
    // index = sector * num_rings + ring
    std::vector<float> get_status() {
        std::vector<float> st(static_cast<size_t>(params_.num_rings) * params_.num_sectors);
        check(erasor_get_status(h_, st.data()));
        return st;
    }
    erasor_handle_t handle() const { return h_; }
    const erasor_params_t& params() const { return params_; }

private:
    void check(int rc) const {
        if (rc == ERASOR_OK) return;
        const std::string msg = std::string("ERASOR: ") + erasor_last_error(h_);
        if (rc == ERASOR_E_INVALID) throw std::invalid_argument(msg);   // e.g. "Other version is not implemented!" (OfflineMapUpdater.cpp:274)
        throw std::runtime_error(msg);
    }
    erasor_params_t params_;
    int             device_ = 0;
    erasor_handle_t h_ = nullptr;
    erasor_map_t    map_ = nullptr;
};

}  // namespace erasor_b200

// The reference's class lives in the global namespace (`class ERASOR`, erasor.h:43).  Define ERASOR_B200_GLOBAL_NAMES before
// including this header to get that spelling, so that OfflineMapUpdater.cpp's `unique_ptr<ERASOR> erasor_` compiles unchanged.
#ifdef ERASOR_B200_GLOBAL_NAMES
using ERASOR = erasor_b200::ERASOR;
#endif
