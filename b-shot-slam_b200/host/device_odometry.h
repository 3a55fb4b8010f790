// device_odometry.h -- the body of odometry_test.cpp's per-scan loop (test/odometry_test.cpp:143-184) as one call: the
// rotation's velodyne::Laser records go to bshot_odometry_step, which runs the preprocessor, extraction, matching against
// the map, RANSAC, the gate + ICP, the map update and the reference-frame hand-over on the device and returns the pose.
// LidarOdometry and its reference-named stage methods stay available for callers that want the stages one by one.
// relocalize() finds a rotation in the whole map without a prior pose; exportMap / importMap save and restore the map.
// detectLoop() asks whether the last rotation revisits an older one; trajectory() and the loop report's T_rel are the nodes
// and edges a pose-graph back end takes; reanchor() moves the map and the pose to the trajectory the back end returns.
#ifndef BSHOT_B200_HOST_DEVICE_ODOMETRY_H
#define BSHOT_B200_HOST_DEVICE_ODOMETRY_H

#include <vector>

#include "../../include/bshot_b200.h"
#include "bshot_bits.h"
#include "bshot_headers_bits.h"
#include "preprocess.h"

namespace myslam {

class DeviceOdometry {
public:
    // a context sized for one rotation (max_points returns kept), the map of the reference driver (max_map entries)
    explicit DeviceOdometry(int device = 0, size_t max_points = 131072, size_t max_keypoints = 1024, size_t max_targets = 1u << 16,
                            size_t max_map = 1u << 16, size_t max_blocks = 4096) {
        bshot_odom_params_default(&params_);
        bshot_loop_params_default(&loop_params_);
        bshot_graph_params_default(&graph_params_);
        status_ = bshot_ctx_create(&ctx_, device, max_points, max_keypoints, max_targets);
        if (status_ == BSHOT_OK) status_ = bshot_gmap_create(ctx_, max_map, max_blocks);
    }
    ~DeviceOdometry() { if (ctx_) bshot_ctx_destroy(ctx_); }
    DeviceOdometry(const DeviceOdometry&) = delete;
    DeviceOdometry& operator=(const DeviceOdometry&) = delete;

    bshot_odom_params& params() { return params_; }

    // one rotation -> T_best (the pose poseEstimation sets); on an error the pose of the last good step is returned and
    // last_status() / bshot_last_error() say why
    Matrix4f step(const std::vector<velodyne::Laser>& lasers, const std::vector<double>& ring_deg) {
        const size_t n = lasers.size();
        az_.resize(n); vert_.resize(n); dist_.resize(n);
        for (size_t i = 0; i < n; ++i) { az_[i] = lasers[i].azimuth; vert_[i] = lasers[i].vertical; dist_[i] = lasers[i].distance; }
        if (ctx_) {
            bshot_odom_report r;
            status_ = bshot_odometry_step(ctx_, &params_, az_.data(), vert_.data(), dist_.data(), n, ring_deg.data(), ring_deg.size(), &r);
            if (status_ == BSHOT_OK) {
                report_ = r;
                for (int row = 0; row < 4; ++row) for (int col = 0; col < 4; ++col) pose_(row, col) = r.pose[4 * row + col];
            }
        }
        return pose_;
    }

    const bshot_odom_report& report() const { return report_; }
    // the pose the last step(), accepted relocalize() or reanchor() set
    const Matrix4f& pose() const { return pose_; }

    // relocalisation of one rotation against the whole map (no prior pose): true when at least min_inliers() RANSAC inliers
    // survived; then pose_ is the new pose and the next step() continues in the map frame.  Otherwise nothing changes.
    // reloc_report() holds the last report; last_status() / bshot_last_error() say why a call failed
    bool relocalize(const std::vector<velodyne::Laser>& lasers, const std::vector<double>& ring_deg) {
        const size_t n = lasers.size();
        az_.resize(n); vert_.resize(n); dist_.resize(n);
        for (size_t i = 0; i < n; ++i) { az_[i] = lasers[i].azimuth; vert_[i] = lasers[i].vertical; dist_[i] = lasers[i].distance; }
        if (!ctx_) return false;
        bshot_reloc_report r;
        status_ = bshot_relocalize(ctx_, &params_, min_inliers_, az_.data(), vert_.data(), dist_.data(), n, ring_deg.data(), ring_deg.size(), &r);
        if (status_ != BSHOT_OK) return false;
        reloc_report_ = r;
        if (!r.accepted) return false;
        for (int row = 0; row < 4; ++row) for (int col = 0; col < 4; ++col) pose_(row, col) = r.pose[4 * row + col];
        return true;
    }
    const bshot_reloc_report& reloc_report() const { return reloc_report_; }
    int& min_inliers() { return min_inliers_; }

    // the map as arrays: xyzr 4 floats {x, y, z, seg_ratio} per entry, in map order (bshot_gmap_export); importMap puts
    // such arrays back as they were (bshot_gmap_import).  Both return a BSHOT_* status
    int exportMap(std::vector<float>& xyzr, std::vector<bshot_descriptor>& desc) {
        if (!ctx_) return status_;
        size_t n = 0;
        status_ = bshot_gmap_export(ctx_, nullptr, nullptr, 0, &n);
        if (status_ != BSHOT_OK && status_ != BSHOT_E_CAPACITY) return status_;
        xyzr.resize(4 * n);
        desc.resize(n);
        status_ = bshot_gmap_export(ctx_, xyzr.data(), reinterpret_cast<uint64_t*>(desc.data()), n, &n);
        return status_;
    }
    int importMap(const std::vector<float>& xyzr, const std::vector<bshot_descriptor>& desc) {
        if (!ctx_) return status_;
        if (xyzr.size() != 4 * desc.size()) return status_ = BSHOT_E_INVALID;
        status_ = bshot_gmap_import(ctx_, xyzr.data(), reinterpret_cast<const uint64_t*>(desc.data()), desc.size());
        return status_;
    }

    // is the last rotation step() took a revisit of a rotation at least loopParams().min_gap map updates older?  true when
    // accepted; *r (may be null) receives the report either way.  Read only: the pose, the map and the next step() are
    // unaffected.  last_status() / bshot_last_error() say why a call failed
    bool detectLoop(bshot_loop_report* r = nullptr) {
        if (!ctx_) return false;
        bshot_loop_report rep;
        status_ = bshot_detect_loop(ctx_, &loop_params_, &rep);
        if (status_ != BSHOT_OK) return false;
        if (r) *r = rep;
        return rep.accepted != 0;
    }
    bshot_loop_params& loopParams() { return loop_params_; }

    // the pose each map update used, in update order (bshot_gmap_scans); empty after an error
    void trajectory(std::vector<Matrix4f>& poses) {
        poses.clear();
        if (!ctx_) return;
        size_t m = 0;   // no entry output: the map is not gathered, only the trajectory is read
        status_ = bshot_gmap_scans(ctx_, nullptr, 0, nullptr, 0, nullptr, &m);
        if (status_ != BSHOT_OK) return;
        std::vector<float> p12(12 * m);
        status_ = bshot_gmap_scans(ctx_, nullptr, 0, p12.data(), m, nullptr, &m);
        if (status_ != BSHOT_OK) return;
        poses.assign(m, Matrix4f::Identity());
        for (size_t u = 0; u < m; ++u)
            for (int row = 0; row < 3; ++row) for (int col = 0; col < 4; ++col) poses[u](row, col) = p12[12 * u + 4 * row + col];
    }

    // move the map, the trajectory and the pose to a corrected trajectory (one pose per map update, in update order, as a
    // pose-graph back end returns it from trajectory() and the loop edges; bshot_gmap_reanchor).  On success pose_ is the
    // odometry's new pose and the next step() continues from it.  Returns a BSHOT_* status; on an error nothing changes
    int reanchor(const std::vector<Matrix4f>& poses) {
        if (!ctx_) return status_;
        std::vector<float> p12(12 * poses.size());
        for (size_t u = 0; u < poses.size(); ++u)
            for (int row = 0; row < 3; ++row) for (int col = 0; col < 4; ++col) p12[12 * u + 4 * row + col] = poses[u](row, col);
        float T[16];
        status_ = bshot_gmap_reanchor(ctx_, p12.data(), poses.size(), T);
        if (status_ == BSHOT_OK)
            for (int row = 0; row < 4; ++row) for (int col = 0; col < 4; ++col) pose_(row, col) = T[4 * row + col];
        return status_;
    }

    // the trajectory's pose graph with the accepted detections as loop edges (match_scan, scan, T_rel), optimised on the
    // device (bshot_optimize_trajectory, read only): poses gets one optimised pose per map update, *rep (may be null) the
    // report.  Returns a BSHOT_* status; reanchor(poses) applies the result
    int optimizeTrajectory(const std::vector<bshot_loop_report>& loops, std::vector<Matrix4f>& poses, bshot_graph_report* rep = nullptr) {
        poses.clear();
        if (!ctx_) return status_;
        std::vector<bshot_graph_edge> edges(loops.size());
        for (size_t k = 0; k < loops.size(); ++k) {
            edges[k].from = loops[k].match_scan;
            edges[k].to = loops[k].scan;
            for (int e = 0; e < 16; ++e) edges[k].T[e] = loops[k].T_rel[e];
        }
        size_t m = 0;
        status_ = bshot_gmap_scans(ctx_, nullptr, 0, nullptr, 0, nullptr, &m);
        if (status_ != BSHOT_OK) return status_;
        std::vector<float> p12(12 * (m ? m : 1));
        bshot_graph_report r;
        status_ = bshot_optimize_trajectory(ctx_, edges.data(), edges.size(), &graph_params_, p12.data(), m, nullptr, &r);
        if (status_ != BSHOT_OK) return status_;
        if (rep) *rep = r;
        poses.assign(m, Matrix4f::Identity());
        for (size_t u = 0; u < m; ++u)
            for (int row = 0; row < 3; ++row) for (int col = 0; col < 4; ++col) poses[u](row, col) = p12[12 * u + 4 * row + col];
        return status_;
    }
    bshot_graph_params& graphParams() { return graph_params_; }

    // INITIAL status, identity pose, empty map, no reference frame
    int reset() {
        if (ctx_) status_ = bshot_odometry_reset(ctx_);
        pose_ = Matrix4f::Identity();
        report_ = bshot_odom_report();
        return status_;
    }

    int last_status() const { return status_; }
    bshot_ctx* context() { return ctx_; }

private:
    bshot_ctx* ctx_ = nullptr;
    bshot_odom_params params_;
    bshot_loop_params loop_params_;
    bshot_graph_params graph_params_;
    bshot_odom_report report_ = bshot_odom_report();
    bshot_reloc_report reloc_report_ = bshot_reloc_report();
    int min_inliers_ = 15;   // the gate's own constant (src/lidar_odometry.cpp:269-281)
    Matrix4f pose_ = Matrix4f::Identity();
    int status_ = BSHOT_OK;
    std::vector<double> az_, vert_;
    std::vector<unsigned short> dist_;
};

}  // namespace myslam
#endif
