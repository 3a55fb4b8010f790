// frame.h -- per-scan holder with the reference's public surface (include/frame.h:9-51, src/frame.cpp): id,
// timestamp, pose, point cloud, keypoints and their B-SHOT descriptors.  Nothing here computes; the front end
// (host/lidar_odometry.h) fills it.  descriptors_ is a vector of std::bitset<352>, i.e. exactly the 48-byte records
// the device produces and consumes -- descriptor_data() is what goes into bshot_match*() / bshot_map_append().
#ifndef BSHOT_B200_HOST_FRAME_H
#define BSHOT_B200_HOST_FRAME_H

#include "bshot_headers_bits.h"

namespace myslam {

class Frame {
public:
    using Ptr = std::shared_ptr<Frame>;
    using PCPtr = std::shared_ptr<std::vector<Vector3f>>;            // 12-byte points, millimetres
    using DCPPtr = std::shared_ptr<std::vector<std::bitset<352>>>;  // 48-byte records == device layout

    // ---- state (public members in the reference as well, include/frame.h:17-26) ----
    unsigned long id_ = (unsigned long)-1;
    long long timestamp_ = -1;
    Matrix4f T_c_w_ = Matrix4f::Identity();  // pose of the scan in the map frame
    PCPtr pointcloud_;                       // pre-processed scan
    PCPtr keypoints_;                        // ascending seg-ratio, as extractKeypoints leaves them
    DCPPtr descriptors_;                     // one record per keypoint
    PCPtr iss_keypoints_;                    // ISS keypoints (LidarOdometry::issKpDetection), ascending point index
    bool is_key_frame_ = false;

    Frame() = default;

    // argument order of the reference constructor (include/frame.h:30-32)
    Frame(long id, double time_stamp = 0, Matrix4f T_c_w = Matrix4f::Identity(), PCPtr pc = nullptr,
          PCPtr kps = nullptr, DCPPtr dcpts = nullptr, bool isKeyframe = false)
        : id_((unsigned long)id), timestamp_((long long)time_stamp), T_c_w_(T_c_w), pointcloud_(std::move(pc)),
          keypoints_(std::move(kps)), descriptors_(std::move(dcpts)), is_key_frame_(isKeyframe) {}

    // factory with consecutive ids (src/frame.cpp:25-29)
    static Ptr createFrame() {
        static long next = 0;
        return Ptr(new Frame(next++));
    }

    // ---- setters / getters, names as in the reference (include/frame.h:37-50) ----
    void setPose(const Matrix4f& T_c_w) { T_c_w_ = T_c_w; }
    Matrix4f getPose() { return T_c_w_; }
    void setTimestamp(const long long timestamp) { timestamp_ = timestamp; }
    long long getTimestamp() { return timestamp_; }
    void setPointCloud(PCPtr pc) { pointcloud_ = std::move(pc); }
    PCPtr getPointCloud() { return pointcloud_; }
    void setKeypoints(PCPtr kps) { keypoints_ = std::move(kps); }
    PCPtr getKeypoints() { return keypoints_; }
    void setDescriptors(DCPPtr dcpts) { descriptors_ = std::move(dcpts); }
    DCPPtr getDescriptors() { return descriptors_; }
    void setISSKeypoints(PCPtr kps) { iss_keypoints_ = std::move(kps); }
    PCPtr getISSKeypoints() { return iss_keypoints_; }
    unsigned long getID() { return id_; }
    bool isKeyframe() { return is_key_frame_; }

    // ---- device-facing views (no copies) ----
    const float* point_data() const { return pointcloud_ && !pointcloud_->empty() ? &(*pointcloud_)[0][0] : nullptr; }
    size_t point_count() const { return pointcloud_ ? pointcloud_->size() : 0; }
    const uint64_t* descriptor_data() const {
        return descriptors_ && !descriptors_->empty() ? reinterpret_cast<const uint64_t*>(descriptors_->data()) : nullptr;
    }
    size_t descriptor_count() const { return descriptors_ ? descriptors_->size() : 0; }
};

}  // namespace myslam
#endif
