// bshot_bits.h -- host C++ mirror of the reference's `class bshot` (include/bshot_bits.h:30-281)
// over the B200 C ABI (include/bshot_b200.h).  Same public members, same method names, same
// argument meaning, `void` methods that never throw: failures leave NaN SHOT / all-ones B-SHOT like
// PCL does and are readable through last_status()/bshot_last_error().
//
//   reference                                    here
//   minVect<T>            :6-20                   identical semantics (first minimum), header-only
//   bshot_descriptor      :23-27                  std::bitset<352> bits  (48 B, passed to the GPU as is)
//   calculate_normals(r)  :43-94                  bshot_set_cloud + bshot_set_keypoints + bshot_compute_normals
//   calculate_voxel_grid_keypoints(leaf) :97-110  bshot_voxel_grid on cloud1 and on cloud2
//   calculate_SHOT(r)     :113-135                bshot_compute_shot (fills cloud1_shot incl. rf[9])
//   compute_bshot()       :138-142                bits of the same call (already on the device)
//   compute_bshot_from_SHOT(cloud, out) :144-278  bshot_binarize
#ifndef BSHOT_B200_HOST_BSHOT_BITS_H
#define BSHOT_B200_HOST_BSHOT_BITS_H

#include <algorithm>

#include "bshot_headers_bits.h"
#include "../../include/bshot_b200.h"

template <typename T>
T minVect(const T* v, int n, int* ind = NULL) {
    assert(n > 0);
    T best = v[0];
    int arg = 0;
    for (int i = 1; i < n; ++i)
        if (v[i] < best) { best = v[i]; arg = i; }
    if (ind != NULL) *ind = arg;
    return best;
}

class bshot_descriptor {
public:
    std::bitset<352> bits;
};
static_assert(sizeof(bshot_descriptor) == 48, "bshot_descriptor must be the 48-byte device record");

class bshot {
public:
    pcl::PointCloud<pcl::PointXYZ> cloud1, cloud2;
    pcl::PointCloud<pcl::Normal> cloud1_normals, cloud2_normals;
    pcl::PointCloud<pcl::PointXYZ> cloud1_keypoints, cloud2_keypoints;
    pcl::PointCloud<pcl::SHOT352> cloud1_shot, cloud2_shot;
    std::vector<bshot_descriptor> cloud1_bshot, cloud2_bshot;

    // B200 additions (defaults reproduce the reference): normals placement mode and capacities
    int normals_mode = BSHOT_NORMALS_REFERENCE;
    int normal_max_nn = 300;  // include/bshot_bits.h:68

    explicit bshot(int device = 0, size_t max_points = 1u << 18, size_t max_keypoints = 1u << 14, size_t max_targets = 1u << 20)
        : ctx_(nullptr), status_(BSHOT_OK) {
        status_ = bshot_ctx_create(&ctx_, device, max_points, max_keypoints, max_targets);
    }
    ~bshot() { bshot_ctx_destroy(ctx_); }
    bshot(const bshot&) = delete;
    bshot& operator=(const bshot&) = delete;

    bshot_ctx* context() { return ctx_; }
    int last_status() const { return status_; }

    void calculate_normals(float radius) {
        if (!upload()) return;
        cloud1_normals.is_dense = true;
        cloud1_normals.points.resize(cloud1.size());  // keeps old entries, new ones are (0,0,0)
        std::vector<float> n4(cloud1.size() * 4);
        status_ = bshot_compute_normals(ctx_, normals_mode, radius, normal_max_nn, n4.data());
        if (status_ != BSHOT_OK) return;
        for (size_t i = 0; i < cloud1.size(); ++i) {
            pcl::Normal& n = cloud1_normals.points[i];
            n.normal_x = n4[4 * i]; n.normal_y = n4[4 * i + 1]; n.normal_z = n4[4 * i + 2]; n.curvature = n4[4 * i + 3];
            if (std::isnan(n.normal_x)) cloud1_normals.is_dense = false;
        }
        normals_uploaded_ = true;
    }

    void calculate_SHOT(float radius) {
        if (!upload()) return;
        if (!normals_uploaded_) {  // caller filled cloud1_normals itself: hand them to the device
            if (cloud1_normals.size() != cloud1.size()) { status_ = BSHOT_E_STATE; return; }
            std::vector<float> n4(cloud1.size() * 4);
            for (size_t i = 0; i < cloud1.size(); ++i) {
                const pcl::Normal& n = cloud1_normals.points[i];
                n4[4 * i] = n.normal_x; n4[4 * i + 1] = n.normal_y; n4[4 * i + 2] = n.normal_z; n4[4 * i + 3] = n.curvature;
            }
            status_ = bshot_set_normals(ctx_, n4.data(), cloud1.size());
            if (status_ != BSHOT_OK) return;
        }
        const size_t k = cloud1_keypoints.size();
        std::vector<float> shot(k * 352), rf(k * 9);
        pending_bits_.resize(k);
        status_ = bshot_compute_shot(ctx_, radius, reinterpret_cast<uint64_t*>(pending_bits_.data()), shot.data(), rf.data(),
                                     nullptr, nullptr);
        if (status_ != BSHOT_OK) return;
        cloud1_shot.points.resize(k);
        cloud1_shot.width = (uint32_t)k; cloud1_shot.height = 1; cloud1_shot.is_dense = true;
        for (size_t i = 0; i < k; ++i) {
            std::memcpy(cloud1_shot.points[i].descriptor, &shot[352 * i], sizeof(float) * 352);
            std::memcpy(cloud1_shot.points[i].rf, &rf[9 * i], sizeof(float) * 9);
            if (std::isnan(shot[352 * i])) cloud1_shot.is_dense = false;
        }
        bits_valid_ = true;
    }

    // pcl::VoxelGrid (cubic leaf) of cloud1 into cloud1_keypoints, then of cloud2 into cloud2_keypoints.  The body was
    // restated from the upstream B-SHOT header that `class bshot` comes from, not read from :97-110.  Output clouds as
    // PCL leaves them: width = count, height 1, is_dense; when the grid would overflow PCL copies the input cloud, and
    // the copy keeps the input's width, height and is_dense.  On failure status_ is set and both clouds are empty.
    // The next calculate_normals / calculate_SHOT upload the new keypoints (content fingerprint).
    void calculate_voxel_grid_keypoints(float leaf_size) {
        cloud1_keypoints.clear();
        cloud2_keypoints.clear();
        if (!ctx_) { status_ = BSHOT_E_CUDA; return; }
        if (!voxel_grid(cloud1, leaf_size, cloud1_keypoints) || !voxel_grid(cloud2, leaf_size, cloud2_keypoints)) {
            cloud1_keypoints.clear();
            cloud2_keypoints.clear();
        }
    }

    void compute_bshot() {
        if (bits_valid_ && pending_bits_.size() == cloud1_shot.size()) cloud1_bshot = pending_bits_;  // fused on the device
        else compute_bshot_from_SHOT(cloud1_shot, cloud1_bshot);
    }

    void compute_bshot_from_SHOT(pcl::PointCloud<pcl::SHOT352>& shot_descriptors_here, std::vector<bshot_descriptor>& bshot_descriptors) {
        bshot_descriptors.resize(shot_descriptors_here.size());
        if (shot_descriptors_here.size() == 0) return;
        status_ = bshot_binarize(ctx_, shot_descriptors_here.points[0].descriptor, shot_descriptors_here.size(),
                                 sizeof(pcl::SHOT352) / sizeof(float), reinterpret_cast<uint64_t*>(bshot_descriptors.data()));
    }

    // B200 addition: tells the shim that the context already holds exactly cloud1 / cloud1_keypoints (LidarOdometry's
    // extractKeypoints uploaded the cloud and left the detector's keypoints on the device): the next calculate_normals
    // / calculate_SHOT then skip the upload and the keypoint normals reuse the detector's neighbourhoods.
    void device_holds_current_inputs() {
        cloud_fp_ = fingerprint(cloud1.points.empty() ? nullptr : cloud1.points[0].data, cloud1.size());
        kp_fp_ = fingerprint(cloud1_keypoints.points.empty() ? nullptr : cloud1_keypoints.points[0].data, cloud1_keypoints.size());
        have_cloud_ = have_kp_ = true;
        normals_uploaded_ = false; bits_valid_ = false;
    }

private:
    // Content fingerprint of a point array (never its address: `cb.cloud1 = next_cloud` reuses the vector's buffer, and
    // allocators hand back the same address for a same-size cloud).  Every point is hashed up to 32 k points; above
    // that every k-th one (a new scan differs everywhere), plus the size.
    static uint64_t fingerprint(const float* xyzw, size_t n) {
        uint64_t h = 0xCBF29CE484222325ull ^ (uint64_t)n;
        if (!xyzw || n == 0) return h;
        const size_t step = n <= 32768 ? 1 : (n + 32767) / 32768;
        auto mix = [&](size_t i) {
            uint64_t a, b;
            std::memcpy(&a, xyzw + 4 * i, 8);
            std::memcpy(&b, xyzw + 4 * i + 2, 4);
            b &= 0xFFFFFFFFull;
            h = (h ^ a) * 0x100000001B3ull;
            h = (h ^ b ^ (uint64_t)i) * 0x9E3779B97F4A7C15ull;
            h ^= h >> 29;
        };
        for (size_t i = 0; i < n; i += step) mix(i);
        mix(n - 1);
        return h;
    }

    bool voxel_grid(const pcl::PointCloud<pcl::PointXYZ>& in, float leaf, pcl::PointCloud<pcl::PointXYZ>& out) {
        const size_t n = in.size();
        std::vector<float> xyz(3 * n);
        size_t count = 0;
        status_ = bshot_voxel_grid(ctx_, n ? in.points[0].data : nullptr, n, sizeof(pcl::PointXYZ), leaf, leaf, leaf, xyz.data(), n,
                                   &count);
        if (status_ != BSHOT_OK) return false;
        out.points.resize(count);
        for (size_t i = 0; i < count; ++i) out.points[i] = pcl::PointXYZ(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]);
        out.width = (uint32_t)count; out.height = 1; out.is_dense = true;
        // PCL's overflow branch is `output = *input_`: the input's layout too.  Only a result of n points can be that
        // copy; every voxel holding one point also gives n points, so the test itself decides.
        if (count == n && grid_overflows(in, leaf)) { out.width = in.width; out.height = in.height; out.is_dense = in.is_dense; }
        return true;
    }

    // PCL 1.8 VoxelGrid::applyFilter's overflow test with a cubic leaf, in the fp32 arithmetic bshot_voxel_grid uses:
    // over the finite points, (int64)((max - min) * (1 / leaf)) + 1 cells per axis, more than INT32_MAX cells in all
    static bool grid_overflows(const pcl::PointCloud<pcl::PointXYZ>& in, float leaf) {
        const float inv = 1.0f / leaf;
        float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
        bool any = false;
        for (const auto& p : in.points) {
            if (!std::isfinite(p.x) || !std::isfinite(p.y) || !std::isfinite(p.z)) continue;
            for (int a = 0; a < 3; ++a) { mn[a] = std::min(mn[a], p.data[a]); mx[a] = std::max(mx[a], p.data[a]); }
            any = true;
        }
        if (!any) return false;
        int64_t cells = 1;
        for (int a = 0; a < 3; ++a) {
            const float f = (mx[a] - mn[a]) * inv;
            if (!(f < 2147483648.0f)) return true;
            cells *= (int64_t)f + 1;
            if (cells > (int64_t)INT32_MAX) return true;
        }
        return false;
    }

    bool upload() {
        if (!ctx_) { status_ = BSHOT_E_CUDA; return false; }
        // re-upload whenever the CONTENT of the clouds changed (`cb.cloud1 = src_pcl_`, src/lidar_odometry.cpp:159-162)
        const uint64_t cfp = fingerprint(cloud1.points.empty() ? nullptr : cloud1.points[0].data, cloud1.size());
        if (!have_cloud_ || cfp != cloud_fp_) {
            status_ = bshot_set_cloud(ctx_, cloud1.points.empty() ? nullptr : cloud1.points[0].data, cloud1.size(), sizeof(pcl::PointXYZ));
            if (status_ != BSHOT_OK) return false;
            cloud_fp_ = cfp; have_cloud_ = true;
            normals_uploaded_ = false; bits_valid_ = false; have_kp_ = false;
        }
        const uint64_t kfp = fingerprint(cloud1_keypoints.points.empty() ? nullptr : cloud1_keypoints.points[0].data, cloud1_keypoints.size());
        if (!have_kp_ || kfp != kp_fp_) {
            status_ = bshot_set_keypoints(ctx_, cloud1_keypoints.points.empty() ? nullptr : cloud1_keypoints.points[0].data,
                                          cloud1_keypoints.size(), sizeof(pcl::PointXYZ));
            if (status_ != BSHOT_OK) return false;
            kp_fp_ = kfp; have_kp_ = true;
            bits_valid_ = false;
        }
        return true;
    }

    bshot_ctx* ctx_;
    int status_;
    uint64_t cloud_fp_ = 0, kp_fp_ = 0;
    bool have_cloud_ = false, have_kp_ = false;
    bool normals_uploaded_ = false, bits_valid_ = false;
    std::vector<bshot_descriptor> pending_bits_;
};

#endif
