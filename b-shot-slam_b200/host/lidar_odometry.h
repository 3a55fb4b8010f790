// lidar_odometry.h -- the per-frame stage methods of the reference's LidarOdometry (include/lidar_odometry.h:22-31,
// src/lidar_odometry.cpp:51-376) over the B200 C ABI: extractKeypoints, computeDescriptors, featureMatching (mutual
// Hamming matching + RANSAC rejection), evaluateEstimation (gate + ICP), poseEstimation, updateMap -- the call order of
// test/odometry_test.cpp:174-192 -- and the keypoint evaluation of the kp_test driver: issKpDetection and kpEvaluation.
// The viewer and the printing are not carried over.
#ifndef BSHOT_B200_HOST_LIDAR_ODOMETRY_H
#define BSHOT_B200_HOST_LIDAR_ODOMETRY_H

#include "bshot_bits.h"
#include "frame.h"
#include "mymap.h"

namespace myslam {

class LidarOdometry {
public:
    enum STATUS { INITIAL, RUN };
    explicit LidarOdometry(int device = 0) : cb(device), status_(INITIAL), sr_type_("CV"), top_k_(600) {}

    void setSrcFrame(Frame::Ptr src) {  // src/lidar_odometry.cpp:29-41
        src_ = src;
        Frame::PCPtr p = src_->getPointCloud();
        src_pcl_.clear();
        src_pcl_.points.resize(p->size());
        for (size_t i = 0; i < p->size(); ++i) src_pcl_.points[i] = pcl::PointXYZ((*p)[i][0], (*p)[i][1], (*p)[i][2]);
        src_pcl_.width = (uint32_t)p->size(); src_pcl_.height = 1;
    }
    void passSrc2Ref() { ref_ = src_; ref_pcl_ = src_pcl_; }
    bool isInitial() { return status_ == INITIAL; }
    void setSRType(std::string t) { sr_type_ = t; }
    void setTopK(int k) { top_k_ = k; }
    void setRun() { status_ = RUN; }

    // :51-162.  The reference also runs ISS detection from here (:164-170); that is issKpDetection() below, called
    // separately, so that the odometry path does not pay for an evaluation-only detector.
    void extractKeypoints() {
        bshot_ctx* ctx = cb.context();
        const int sr = sr_type_ == "CVS" ? BSHOT_SR_CVS : (sr_type_ == "CVSN" ? BSHOT_SR_CVSN : BSHOT_SR_CV);
        cb.cloud1 = src_pcl_;
        last_status_ = bshot_set_cloud(ctx, src_pcl_.points.empty() ? nullptr : src_pcl_.points[0].data, src_pcl_.size(), 16);
        std::vector<int> idx(top_k_);
        std::vector<float> ratio(top_k_), xyz(3 * (size_t)top_k_);
        int k = 0;
        if (last_status_ == BSHOT_OK)
            last_status_ = bshot_detect_keypoints(ctx, 3000.0f, 300, sr, top_k_, idx.data(), ratio.data(), xyz.data(), &k);
        auto kps = std::make_shared<std::vector<Vector3f>>();
        seg_ratios_.assign(ratio.begin(), ratio.begin() + k);
        for (int i = 0; i < k; ++i) kps->push_back(Vector3f(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
        src_->setKeypoints(kps);
        if (isInitial()) { passSrc2Ref(); ref_->setKeypoints(src_->getKeypoints()); }
        cb.cloud2 = ref_pcl_;
        cb.cloud1_keypoints = eigen2pcl(src_->getKeypoints());
        cb.cloud2_keypoints = eigen2pcl(ref_->getKeypoints());
        // the context already holds this cloud (voxel grid built once) and the detector's keypoints: computeDescriptors
        // does not upload them again and the keypoint normals reuse the detector's neighbourhoods
        if (last_status_ == BSHOT_OK) cb.device_holds_current_inputs();
    }

    void computeDescriptors() {  // :173-184
        cb.calculate_normals(3000);
        cb.calculate_SHOT(3000);
        cb.compute_bshot();
        auto d = std::make_shared<std::vector<std::bitset<352>>>();
        d->reserve(cb.cloud1_bshot.size());
        for (auto& it : cb.cloud1_bshot) d->push_back(it.bits);
        src_->setDescriptors(d);
    }

    void featureMatching() {  // :186-242 ; RANSAC (:251-261) is the caller's next step on `corresp`
        if (isInitial()) {
            passSrc2Ref();
            ref_->setKeypoints(src_->getKeypoints());
            cb.cloud2 = ref_pcl_;
            cb.cloud2_bshot = cb.cloud1_bshot;
            cb.cloud2_keypoints = eigen2pcl(ref_->getKeypoints());
        } else {
            Vector3f pos = ref_->getPose().translation();
            globalMap_.getKeypoints(pos, 100000, cb.cloud2_keypoints, cb.cloud2_bshot);
            Matrix4f T = ref_->getPose();
            for (auto& p : *ref_->getKeypoints()) { Vector3f w = T.apply(p); cb.cloud2_keypoints.push_back(pcl::PointXYZ(w[0], w[1], w[2])); }
            for (auto& b : *ref_->getDescriptors()) { bshot_descriptor d; d.bits = b; cb.cloud2_bshot.push_back(d); }
        }
        const size_t nq = cb.cloud1_bshot.size(), nt = cb.cloud2_bshot.size();
        std::vector<int> pairs(2 * nq + 2);
        int n = 0;
        last_status_ = bshot_match_mutual(cb.context(), reinterpret_cast<const uint64_t*>(cb.cloud1_bshot.data()), nq,
                                          reinterpret_cast<const uint64_t*>(cb.cloud2_bshot.data()), nt, pairs.data(), nullptr, &n);
        corresp.clear();
        for (int i = 0; i < n; ++i) {
            pcl::Correspondence c;
            c.index_query = pairs[2 * i];
            c.index_match = pairs[2 * i + 1];
            corresp.push_back(c);
        }
        // RANSAC based correspondence rejection (:251-261): 2000 iterations, inlier threshold 1500 mm
        corr.clear();
        if (last_status_ != BSHOT_OK) return;
        std::vector<float> s = flat(cb.cloud1_keypoints), t = flat(cb.cloud2_keypoints);
        std::vector<int> kept(2 * (size_t)n + 2);
        int n_kept = 0, iters = 0;
        float T[16];
        last_status_ = bshot_ransac(cb.context(), s.data(), cb.cloud1_keypoints.size(), t.data(), cb.cloud2_keypoints.size(), pairs.data(), (size_t)n, 2000,
                                    1500.0f, kept.data(), &n_kept, T, &iters);
        if (last_status_ != BSHOT_OK) return;
        for (int i = 0; i < n_kept; ++i) {
            pcl::Correspondence c;
            c.index_query = kept[2 * i];
            c.index_match = kept[2 * i + 1];
            corr.push_back(c);
        }
        T_ransac_ = from_row_major(T);
    }

    void evaluateEstimation() {  // :267-301 (its evaluate_corr_ statistics are prints only)
        float Tj[16], Ti[16], Tb[16];
        to_row_major(T_ransac_, Tj);
        to_row_major(ref_->getPose(), Ti);
        std::vector<float> s = flat(cb.cloud1_keypoints), t = flat(cb.cloud2_keypoints);
        int upd = 0;
        last_status_ = bshot_evaluate_estimation(cb.context(), Tj, Ti, (int)corr.size(), s.data(), cb.cloud1_keypoints.size(), t.data(),
                                                 cb.cloud2_keypoints.size(), run_icp_ ? 1 : 0, Tb, &upd, &h_diff_, &t_diff_, &icp_iterations_);
        if (last_status_ != BSHOT_OK) return;
        shouldUpdateMap = upd != 0;
        T_best_ = from_row_major(Tb);
    }

    void poseEstimation() { src_->setPose(T_best_); }  // :333-341, frame-to-localmap

    void updateMap() {  // :344-376: every keypoint of the frame, moved by T_best_
        Frame::PCPtr kps = src_->getKeypoints();
        for (size_t i = 0; i < cb.cloud1_bshot.size() && i < kps->size(); ++i) {
            // R * p + T in Eigen's order: the three products summed left to right, then the translation
            const Vector3f& p = (*kps)[i];
            Vector3f w((T_best_(0, 0) * p[0] + T_best_(0, 1) * p[1] + T_best_(0, 2) * p[2]) + T_best_(0, 3),
                       (T_best_(1, 0) * p[0] + T_best_(1, 1) * p[1] + T_best_(1, 2) * p[2]) + T_best_(1, 3),
                       (T_best_(2, 0) * p[0] + T_best_(2, 1) * p[1] + T_best_(2, 2) * p[2]) + T_best_(2, 3));
            globalMap_.addKeypoint(Keypoint::createKeypoint(w, seg_ratios_[i], cb.cloud1_bshot[i]));
        }
        status_ = RUN;
    }
    // :447-461: pcl::ISSKeypoint3D (salient radius 60, non-max radius 40, thresholds 0.975 / 0.975) on the source cloud
    // -> the source frame's ISS keypoints.  Runs on the cloud extractKeypoints() left in the context (call it after that).
    void issKpDetection() {
        bshot_ctx* ctx = cb.context();
        bshot_iss_params prm;
        bshot_iss_params_default(&prm);
        size_t n = 0;
        std::vector<int> idx(4096);
        std::vector<float> xyz(3 * idx.size());
        last_status_ = bshot_detect_iss(ctx, &prm, idx.data(), xyz.data(), idx.size(), &n, nullptr);
        if (last_status_ == BSHOT_E_CAPACITY) {
            idx.resize(n);
            xyz.resize(3 * n);
            last_status_ = bshot_detect_iss(ctx, &prm, idx.data(), xyz.data(), n, &n, nullptr);
        }
        auto kps = std::make_shared<std::vector<Vector3f>>();
        if (last_status_ == BSHOT_OK)
            for (size_t i = 0; i < n; ++i) kps->push_back(Vector3f(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
        src_->setISSKeypoints(kps);
    }

    // :392-445: repeat rates of the source frame's seg-ratio and ISS keypoints against the reference frame's, each set
    // moved by its frame's pose: the share of source keypoints whose nearest reference keypoint lies within 30 mm
    // (bshot_kp_repeatability; the port's definition, the reference prints its own "Repeat rate").  Kept, not printed.
    void kpEvaluation() {
        float Ts[16], Tr[16];
        to_row_major(src_->getPose(), Ts);
        to_row_major(ref_->getPose(), Tr);
        auto rate = [&](const Frame::PCPtr& a, const Frame::PCPtr& b, double& out) {
            out = 0.0;
            const size_t na = a ? a->size() : 0, nb = b ? b->size() : 0;
            size_t hits = 0;
            last_status_ = bshot_kp_repeatability(cb.context(), na ? &(*a)[0][0] : nullptr, na, Ts, nb ? &(*b)[0][0] : nullptr, nb, Tr, 30.0f,
                                                  nullptr, nullptr, &hits);
            if (last_status_ == BSHOT_OK && na) out = (double)hits / (double)na;
            return last_status_ == BSHOT_OK;
        };
        if (rate(src_->getKeypoints(), ref_->getKeypoints(), sr_repeat_rate_)) rate(src_->getISSKeypoints(), ref_->getISSKeypoints(), iss_repeat_rate_);
    }

    void setRunICP(bool run_icp) { run_icp_ = run_icp; }
    Matrix4f getBestTransformation() const { return T_best_; }
    Matrix4f getRansacTransformation() const { return T_ransac_; }

    static std::vector<float> flat(const pcl::PointCloud<pcl::PointXYZ>& c) {
        std::vector<float> o(3 * c.size() + 3);
        for (size_t i = 0; i < c.size(); ++i) { o[3 * i] = c.points[i].x; o[3 * i + 1] = c.points[i].y; o[3 * i + 2] = c.points[i].z; }
        return o;
    }
    static void to_row_major(const Matrix4f& M, float* o) {
        for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) o[4 * r + c] = M(r, c);
    }
    static Matrix4f from_row_major(const float* a) {
        Matrix4f M;
        for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) M(r, c) = a[4 * r + c];
        return M;
    }

    pcl::PointCloud<pcl::PointXYZ> eigen2pcl(Frame::PCPtr pc) {
        pcl::PointCloud<pcl::PointXYZ> out;
        if (pc) for (auto& p : *pc) out.push_back(pcl::PointXYZ(p[0], p[1], p[2]));
        return out;
    }
    Frame::Ptr getRefFrame() { return ref_; }
    Frame::Ptr getSrcFrame() { return src_; }
    Map& map() { return globalMap_; }
    int last_status() const { return last_status_ != BSHOT_OK ? last_status_ : cb.last_status(); }

    bshot cb;
    pcl::Correspondences corresp;   // mutual nearest neighbours (:234-242)
    pcl::Correspondences corr;      // after RANSAC rejection (:253-261)
    bool shouldUpdateMap = true;
    float h_diff_ = 0, t_diff_ = 0;
    int icp_iterations_ = 0;
    std::vector<float> seg_ratios_;
    double sr_repeat_rate_ = 0.0, iss_repeat_rate_ = 0.0;  // kpEvaluation

private:
    Frame::Ptr ref_, src_;
    pcl::PointCloud<pcl::PointXYZ> ref_pcl_, src_pcl_;
    STATUS status_;
    std::string sr_type_;
    int top_k_;
    Map globalMap_;
    int last_status_ = BSHOT_OK;
    bool run_icp_ = true;           // src/lidar_odometry.cpp:6
    Matrix4f T_ransac_ = Matrix4f::Identity(), T_best_ = Matrix4f::Identity();
};

}  // namespace myslam
#endif
