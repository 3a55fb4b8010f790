/*
 * bshot_b200.h -- C ABI of the B200-native (sm_100a) B-SHOT feature front end.
 *
 * Drop-in boundary for the per-frame front end of TingKaiChen/B-SHOT-SLAM.  The reference has no
 * FFI layer: control enters the path through C++ member calls on `class bshot`
 * (include/bshot_bits.h:30-281) made by LidarOdometry::extractKeypoints / computeDescriptors /
 * featureMatching (src/lidar_odometry.cpp:51,173,186).  Every entry point below names the
 * reference code it replaces.  The reference-named host C++ shims (headers under b-shot-slam_b200/host:
 * `bshot`, `bshot_descriptor`, `minVect`, `Frame`, `Keypoint`, `Map`) forward to this ABI; see
 * INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; all functions return 0 on success, a negative BSHOT_E_* code
 *     otherwise and never throw.  bshot_last_error() returns a thread-local message.
 *   - units are millimetres (reference: src/preprocess.cpp:46).
 *   - a descriptor record is 48 bytes = std::bitset<352> of libstdc++ (6 x u64 little endian, bit i
 *     in word i/64 at position i%64, bits 352..383 zero) == bshot_descriptor
 *     (include/bshot_bits.h:23-27), so std::vector<bshot_descriptor>::data() can be passed as is.
 *   - a context owns its device buffers (sized at creation, no per-frame allocation) and ONE
 *     CUDA stream.  It is not thread safe.  Host-buffer calls are synchronous on return.
 *     *_dev / *_resident calls take device pointers / use resident data and are asynchronous on
 *     the context stream.
 *   - there is NO CPU fallback: every call fails with BSHOT_E_CUDA when no sm_100 device is
 *     usable.
 */
#ifndef BSHOT_B200_H
#define BSHOT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSHOT_B200_VERSION 100

enum {
    BSHOT_OK = 0,
    BSHOT_E_INVALID = -1,   /* bad argument */
    BSHOT_E_CAPACITY = -2,  /* input larger than the context was created for */
    BSHOT_E_CUDA = -3,      /* CUDA runtime / launch failure, or no usable device */
    BSHOT_E_STATE = -4      /* call order violated (e.g. descriptors before a cloud) */
};

/* seg-ratio variants, LidarOdometry::sr_type_ "CV"/"CVS"/"CVSN" (src/lidar_odometry.cpp:83,98,109) */
enum { BSHOT_SR_CV = 0, BSHOT_SR_CVS = 1, BSHOT_SR_CVSN = 2 };

/* normals placement.  REFERENCE reproduces include/bshot_bits.h:58-59,79-81: the K keypoint
 * normals are stored at indices 0..K-1 of an N-sized, zero-initialised, persistent array that
 * SHOT then indexes by SURFACE point.  FULL computes a normal for every surface point (what the
 * commented-out lines include/bshot_bits.h:89-90 did). */
enum { BSHOT_NORMALS_REFERENCE = 0, BSHOT_NORMALS_FULL = 1 };

typedef struct bshot_ctx bshot_ctx;

/* one frame's parameters; bshot_params_default() fills the reference's literals */
typedef struct bshot_params {
    float kp_radius;     /* 3000  src/lidar_odometry.cpp:68 */
    int kp_max_nn;       /* 300   src/lidar_odometry.cpp:70 */
    int sr_type;         /* CV    src/lidar_odometry.cpp:6  */
    int top_k;           /* 600   src/lidar_odometry.cpp:138-142 */
    float normal_radius; /* 3000  src/lidar_odometry.cpp:174 */
    int normal_max_nn;   /* 300   include/bshot_bits.h:68 */
    int normals_mode;    /* BSHOT_NORMALS_REFERENCE */
    float shot_radius;   /* 3000  src/lidar_odometry.cpp:175 */
} bshot_params;

void bshot_params_default(bshot_params* p);

int bshot_version(void);
const char* bshot_last_error(void);

/* ---- context ------------------------------------------------------------------------------ */
/* replaces the `bshot cb` member of LidarOdometry (include/lidar_odometry.h:57) */
int bshot_ctx_create(bshot_ctx** out, int device, size_t max_points, size_t max_keypoints,
                     size_t max_targets);
void bshot_ctx_destroy(bshot_ctx* ctx);
/* the context's cudaStream_t (for CUDA-event timing by the caller) */
void* bshot_ctx_stream(bshot_ctx* ctx);
int bshot_ctx_sync(bshot_ctx* ctx);
/* forget all cross-frame state, as if `cb` were freshly constructed: the persistent normals array
 * (include/bshot_bits.h:59 resize keeps old entries), the previous frame's descriptors and the
 * map shard.  The cloud, keypoints and capacity stay. */
int bshot_ctx_reset(bshot_ctx* ctx);

/* ---- a1: cloud upload + voxel-hash build -------------------------------------------------- */
/* replaces LidarOdometry::setSrcFrame (src/lidar_odometry.cpp:29-41) + `cb.cloud1 = src_pcl_`
 * (:159) and the three pcl::KdTreeFLANN builds (:53-54, include/bshot_bits.h:52-53, PCL SHOT).
 * stride_bytes is 12 (Eigen::Vector3f) or 16 (pcl::PointXYZ). */
int bshot_set_cloud(bshot_ctx* ctx, const float* xyz, size_t n, size_t stride_bytes);

/* ---- a2+a3: seg-ratio keypoint detector ---------------------------------------------------- */
/* replaces LidarOdometry::extractKeypoints loop + sort + top-K (src/lidar_odometry.cpp:61-153).
 * Keypoints come out in ascending-ratio order (ties: descending point index), the top_k highest.
 * idx_out / ratio_out / kp_xyz_out (3 floats each) may be NULL; *count_out <= top_k.
 * The selected keypoints become the context's current keypoints (cb.cloud1_keypoints, :161). */
int bshot_detect_keypoints(bshot_ctx* ctx, float radius, int max_nn, int sr_type, int top_k,
                           int* idx_out, float* ratio_out, float* kp_xyz_out, int* count_out);
/* all N seg-ratios (NaN where the reference skips the point, :63,:121) */
int bshot_seg_ratio(bshot_ctx* ctx, float radius, int max_nn, int sr_type, float* ratio_out);
/* explicit keypoints instead of the detector: `cb.cloud1_keypoints = ...` (:161) */
int bshot_set_keypoints(bshot_ctx* ctx, const float* kp_xyz, size_t k, size_t stride_bytes);

/* ---- a4: normals ---------------------------------------------------------------------------- */
/* replaces bshot::calculate_normals (include/bshot_bits.h:43-94).  normals_out (may be NULL):
 * N x 4 floats (nx,ny,nz,curvature) indexed by surface point, i.e. cloud1_normals. */
int bshot_compute_normals(bshot_ctx* ctx, int mode, float radius, int max_nn, float* normals_out);
/* normals of arbitrary query points (Q x 4), no placement; the per-query body of :61-88 */
int bshot_query_normals(bshot_ctx* ctx, const float* q_xyz, size_t nq, float radius, int max_nn,
                        float* normals_out);
/* upload cloud1_normals verbatim (N x 4 floats) */
int bshot_set_normals(bshot_ctx* ctx, const float* normals4, size_t n);

/* ---- a5+a6+a7: SHOT LRF, SHOT352 histogram, B-SHOT bits ------------------------------------ */
/* replaces bshot::calculate_SHOT (include/bshot_bits.h:113-135) and bshot::compute_bshot (:138-142)
 * for the current keypoints and normals.  Any output may be NULL:
 *   bits_out  K x 6 u64 (bshot_descriptor)       shot_out  K x 352 f32 (pcl::SHOT352::descriptor)
 *   rf_out    K x 9 f32 (pcl::SHOT352::rf)        nn_out    K ints, neighbours within radius
 * sum_nn_out = sum of nn_out (the algorithmic-bytes unit of SURVEY 8d). */
int bshot_compute_shot(bshot_ctx* ctx, float radius, uint64_t* bits_out, float* shot_out,
                       float* rf_out, int* nn_out, long long* sum_nn_out);
/* LRF only (PCL SHOTLocalReferenceFrameEstimation behind include/bshot_bits.h:117-128) */
int bshot_compute_lrf(bshot_ctx* ctx, float radius, float* rf_out, int* valid_nn_out);
/* replaces bshot::compute_bshot_from_SHOT (include/bshot_bits.h:144-278) on caller floats.
 * shot: k records of 352 floats, stride_floats apart (361 for pcl::SHOT352). */
int bshot_binarize(bshot_ctx* ctx, const float* shot, size_t k, size_t stride_floats,
                   uint64_t* bits_out);
/* replaces LidarOdometry::computeDescriptors (src/lidar_odometry.cpp:173-184): normals + SHOT +
 * B-SHOT for the current keypoints in one call. */
int bshot_compute_descriptors(bshot_ctx* ctx, const bshot_params* p, uint64_t* bits_out);

/* ---- a10+a11: Hamming correspondence search ------------------------------------------------ */
/* replaces the two brute-force loops + minVect (src/lidar_odometry.cpp:212-232,
 * include/bshot_bits.h:6-20): left_idx[i] = argmin_k popcount(q_i ^ t_k) (first minimum wins),
 * right_idx[k] = argmin_i popcount(t_k ^ q_i).  Also returns the runner-up (second by
 * (distance, index)).  Any output may be NULL; right_idx == NULL skips the T x Q pass. */
int bshot_match(bshot_ctx* ctx, const uint64_t* q, size_t nq, const uint64_t* t, size_t nt,
                int* left_idx, int* left_dist, int* left_idx2, int* left_dist2, int* right_idx);
/* replaces the mutual-NN filter (src/lidar_odometry.cpp:234-242) fused with the search: writes
 * (index_query, index_match) pairs in ascending index_query; *count_out <= nq. Only the targets
 * that are some query's nearest neighbour get their reverse search (Q x Q instead of T x Q). */
int bshot_match_mutual(bshot_ctx* ctx, const uint64_t* q, size_t nq, const uint64_t* t, size_t nt,
                       int* pairs_out, int* dist_out, int* count_out);

/* ---- whole frame (the reference's extractKeypoints -> computeDescriptors -> featureMatching) */
/* Runs voxel build, detector, normals, SHOT, B-SHOT on `xyz` and matches the new descriptors
 * against the previous frame's descriptors kept in the context (first frame: against itself,
 * src/lidar_odometry.cpp:187-194), i.e. test/odometry_test.cpp:174-180 up to the RANSAC call.
 * One H2D copy in, one D2H copy out.  Outputs may be NULL.  kp_idx_out / bits_out hold up to
 * p->top_k records, pairs_out up to top_k (query,match) pairs. */
int bshot_process_frame(bshot_ctx* ctx, const bshot_params* p, const float* xyz, size_t n,
                        size_t stride_bytes, int* kp_idx_out, uint64_t* bits_out, int* n_kp_out,
                        int* pairs_out, int* n_pairs_out);
/* same work on a cloud that is already in device memory (d_xyz: device pointer); asynchronous on
 * the context stream, no host copies -- the HBM-resident timing leg of bench.py. */
int bshot_process_frame_dev(bshot_ctx* ctx, const bshot_params* p, const void* d_xyz, size_t n,
                            size_t stride_bytes);
/* download the results of the last bshot_process_frame_dev (synchronous).  The pairs are those of the context's last
 * matching run: a later match, step, relocalisation or loop detection replaces them */
int bshot_fetch_frame(bshot_ctx* ctx, int top_k, int* kp_idx_out, uint64_t* bits_out, int* n_kp_out,
                      int* pairs_out, int* n_pairs_out);

/* ---- GPU-resident global map + frame-to-map flow (RUN status of featureMatching) ------------------------------------
 * Replaces, on the device: Keypoint::createKeypoint's 10 mm snap (src/keypoint.cpp:23-32), Map::addKeypoint
 * (src/mymap.cpp:4-26: 10 m blocks, reject when a stored keypoint of the block within 800 mm is at least as salient, else
 * insert / overwrite at the same position), LidarOdometry::updateMap (src/lidar_odometry.cpp:343-358: every keypoint of the
 * frame in order, transformed by the pose), Map::getKeypoints (src/mymap.cpp:28-74: blocks of the +-range cube, x outermost,
 * z innermost) and the target assembly of featureMatching (src/lidar_odometry.cpp:197-206: map subset, then the reference
 * frame's keypoints transformed by its pose).  Inside a block keypoints come out in insertion order (the reference's
 * unordered_map order is implementation defined).  pose3x4 = row-major [R|T], NULL = identity.
 * Per-frame call order of a host that keeps RANSAC / ICP (src/lidar_odometry.cpp:251-301) on the CPU:
 *   bshot_extract_frame -> bshot_match_frame_to_map -> (host: pose) -> bshot_gmap_update_from_frame(pose) -> bshot_frame_commit */
int bshot_gmap_create(bshot_ctx* ctx, size_t max_entries, size_t max_blocks);
int bshot_gmap_reset(bshot_ctx* ctx);
/* entries stored so far (bshot_gmap_export returns exactly these); dropped = keypoints lost to a full block table, chunk
 * pool or entry pool (0 unless the capacities are too small).  Keypoints skipped as not storable are not dropped. */
int bshot_gmap_size(bshot_ctx* ctx, size_t* entries_out, size_t* dropped_out);
/* Map::addKeypoint for n keypoints given on the host (xyz n x 3 floats, in keypoint order), n <= max_keypoints per call.
 * A keypoint is stored only when its transformed position is storable: x, y and z finite and within +-2.1e9 mm (2100 km;
 * the 10 mm snap and the 10 m block id must fit int32).  Other keypoints (NaN, +-Inf, farther) are skipped, uncounted.
 * A pose with a non-finite element returns BSHOT_E_INVALID and changes nothing (no update is counted, the trajectory is
 * not written); so does bshot_gmap_update_from_frame. */
int bshot_gmap_add(bshot_ctx* ctx, const float* xyz, const float* seg_ratio, const uint64_t* desc, size_t n, const float* pose3x4);
/* updateMap for the frame extracted last (keypoints, seg-ratios and descriptors are still on the device); asynchronous */
int bshot_gmap_update_from_frame(bshot_ctx* ctx, const float* pose3x4);
/* Map::getKeypoints to host buffers (cap records); *n_out = keypoints in range */
int bshot_gmap_get_keypoints(bshot_ctx* ctx, const float pos[3], float range, float* xyz_out, uint64_t* desc_out, size_t cap, size_t* n_out);
/* extractKeypoints + computeDescriptors of one scan (no matching); outputs hold up to p->top_k records, any may be NULL */
int bshot_extract_frame(bshot_ctx* ctx, const bshot_params* p, const float* xyz, size_t n, size_t stride_bytes, int* kp_idx_out,
                        float* kp_xyz_out, float* seg_ratio_out, uint64_t* bits_out, int* n_kp_out);
/* featureMatching in RUN status for the frame extracted last: targets = map keypoints within `range` of ref_pos, then the
 * committed (previous) frame transformed by ref_pose3x4; mutual nearest neighbours -> pairs_out (index_query, index_match
 * into that target set).  target_xyz_out (optional, target_cap x 3 floats) = positions of the targets for the host's RANSAC. */
int bshot_match_frame_to_map(bshot_ctx* ctx, const float ref_pos[3], float range, const float* ref_pose3x4, int* pairs_out,
                             int* n_pairs_out, size_t* n_targets_out, float* target_xyz_out, size_t target_cap);
/* the frame extracted last becomes the reference frame (passSrc2Ref, src/lidar_odometry.cpp:43-47); asynchronous */
int bshot_frame_commit(bshot_ctx* ctx);
/* every map entry in map order: occupied blocks in ascending lattice coordinates (x outermost, z innermost, as
 * bshot_gmap_get_keypoints visits them), entries of a block in insertion order.  Unlike bshot_gmap_get_keypoints it is
 * not limited by a probe budget.  xyzr_out cap x 4 floats {x, y, z, seg_ratio}, desc_out cap x 6 u64 (either may be NULL);
 * *n_out = entries.  count > cap: the first cap are written and BSHOT_E_CAPACITY is returned.  Needs bshot_gmap_create
 * (BSHOT_E_STATE). */
int bshot_gmap_export(bshot_ctx* ctx, float* xyzr_out, uint64_t* desc_out, size_t cap, size_t* n_out);
/* replaces the map by these n entries (layout of bshot_gmap_export), without the admission rule: entries of one block keep
 * their relative order in the input, so a bshot_gmap_export result restores the map it came from and every later call
 * behaves as on the exporting context.  Positions are stored as given.  A position that is not storable (as
 * bshot_gmap_add defines it: non-finite, or beyond +-2.1e9 mm): BSHOT_E_INVALID;
 * n > max_entries, or more blocks / chunks than the table holds: BSHOT_E_CAPACITY.  On any error the map is empty.
 * The pose, the status and the reference frame of the odometry step are not touched. */
int bshot_gmap_import(bshot_ctx* ctx, const float* xyzr, const uint64_t* desc, size_t n);

/* ---- RANSAC correspondence rejection (the consumer of the path's output) ----------------------------------------------------
 * Replaces Ransac_based_Rejection.setMaximumIterations(2000) / setInputSource / setInputTarget / setInlierThreshold(1500) /
 * setInputCorrespondences / getCorrespondences (src/lidar_odometry.cpp:251-261), i.e. PCL 1.8's
 * CorrespondenceRejectorSampleConsensus: RandomSampleConsensus over SampleConsensusModelRegistration with PCL's deterministic
 * sample sequence (mt19937 seeded 12345), Umeyama on three pairs, adaptive stop, first best wins.  All max_iterations + 1
 * hypotheses are scored in parallel on the device; the adaptive loop is replayed over the scores.
 * pairs: n_pairs x (index_query into src, index_match into tgt).  Outputs: the surviving correspondences in their original
 * order (capacity n_pairs), their number, the best transformation (row-major 4x4, float) and the iterations PCL would have run.
 * Fewer than 3 correspondences / inliers: everything is kept and the transformation is the identity (PCL's behaviour). */
int bshot_ransac(bshot_ctx* ctx, const float* src_xyz, size_t n_src, const float* tgt_xyz, size_t n_tgt, const int* pairs,
                 size_t n_pairs, int max_iterations, float inlier_threshold, int* inlier_pairs_out, int* n_inliers_out,
                 float* transform4x4_out, int* iterations_out);

/* ---- ICP refinement and the estimation gate (SURVEY 8f next #3) ------------------------------- */
/* Replaces pcl::IterativeClosestPoint<PointXYZ, PointXYZ> with PCL's defaults as LidarOdometry::evaluateEstimation uses it
 * (src/lidar_odometry.cpp:283-291): the n_src source points are first moved by pre4x4 (row-major 4x4, NULL = identity; the
 * reference's transformPointCloud with T_est), then aligned to the n_tgt target points: nearest neighbour correspondences,
 * Umeyama without scaling, at most max_iterations (PCL default 10) rounds.  final4x4_out = icp.getFinalTransformation();
 * state_out: 0 not converged, 1 iteration limit, 2 transformation epsilon, 3 absolute MSE, 5 fewer than 3 correspondences
 * (pcl::registration::DefaultConvergenceCriteria::ConvergenceState); mse_out = mean squared correspondence distance of the
 * last round.  Any output pointer may be NULL. */
int bshot_icp(bshot_ctx* ctx, const float* src_xyz, size_t n_src, const float* tgt_xyz, size_t n_tgt, const float* pre4x4,
              int max_iterations, float* final4x4_out, int* iterations_out, int* state_out, double* mse_out);
/* LidarOdometry::evaluateEstimation (src/lidar_odometry.cpp:267-296) without its printing: T_ij = T_ref^-1 * T_ransac, heading
 * change acos(T_ij(1,1)) and translation |t_ij|; the estimate is rejected (T_est = T_ref, *should_update_map_out = 0) when the
 * heading moved more than 10 degrees, the translation more than 1200 mm or fewer than 15 correspondences survived RANSAC;
 * otherwise T_est = T_ransac.  run_icp != 0: T_best = ICP(src_kp moved by T_est -> tgt_kp) * T_est; else T_best = T_ransac. */
int bshot_evaluate_estimation(bshot_ctx* ctx, const float* T_ransac4x4, const float* T_ref4x4, int n_correspondences,
                              const float* src_kp_xyz, size_t n_src, const float* tgt_kp_xyz, size_t n_tgt, int run_icp,
                              float* T_best4x4_out, int* should_update_map_out, float* h_diff_rad_out, float* t_diff_out,
                              int* icp_iterations_out);

/* ---- scan preprocessor (SURVEY 8f next #4) ---------------------------------------------------- */
/* Replaces myslam::Preprocessor::setLasers + setVerticalAngles + run + getPointCloud (include/preprocess.h:26-33,
 * src/preprocess.cpp:213-223): one rotation of raw returns -> ground, self-car and occluded returns removed -> the cloud
 * the front end consumes, in the reference's order (azimuth-major, vertical angle ascending).
 * azimuth_deg / vertical_deg / distance: the n returns' velodyne::Laser fields (VelodyneCapture.h: azimuth and vertical in
 * degrees as double, distance in 2 mm units), sorted by azimuth as `capture.retrieve(lasers, true)` delivers them.
 * ring_deg: the sensor's nv vertical angles (setVerticalAngles).  vert_init_rad / lowpt_th: the constructor arguments
 * (the SLAM driver uses -0.6 rad and -1950 mm, test/odometry_test.cpp:32-33).  xyz_out: cap x 3 floats (mm); *n_out = number of kept points (if it
 * exceeds cap only the first cap are written and BSHOT_E_CAPACITY is returned). */
int bshot_preprocess(bshot_ctx* ctx, const double* azimuth_deg, const double* vertical_deg, const unsigned short* distance,
                     size_t n, const double* ring_deg, size_t nv, double vert_init_rad, double lowpt_th, float* xyz_out,
                     size_t cap, size_t* n_out);

/* the same with the preprocessor's point selection (setSelectedPoints / haveSelectList / saveSelectPoints,
 * include/preprocess.h:27-29): select_list holds indices into the returns; with have_select_list != 0 a return is
 * "selected" when the list names it, otherwise every return is; only returns whose selection equals save_selected != 0
 * are written (the reference's defaults: no list, save_selected = true). */
int bshot_preprocess_select(bshot_ctx* ctx, const double* azimuth_deg, const double* vertical_deg, const unsigned short* distance,
                            size_t n, const double* ring_deg, size_t nv, double vert_init_rad, double lowpt_th,
                            const int* select_list, size_t n_select, int have_select_list, int save_selected, float* xyz_out,
                            size_t cap, size_t* n_out);

/* Preprocessor::run + extractKeypoints + computeDescriptors of one rotation (test/odometry_test.cpp:143-177) in one call:
 * the preprocessed cloud stays on the device and feeds the front end directly.  cloud_xyz_out (cloud_cap x 3 floats) may be
 * NULL when the host does not need the cloud; the keypoint outputs are those of bshot_extract_frame (kp_idx indexes the
 * preprocessed cloud).  Follow with bshot_match_frame_to_map / bshot_ransac / bshot_evaluate_estimation /
 * bshot_gmap_update_from_frame / bshot_frame_commit as after bshot_extract_frame. */
int bshot_extract_scan(bshot_ctx* ctx, const bshot_params* p, const double* azimuth_deg, const double* vertical_deg,
                       const unsigned short* distance, size_t n, const double* ring_deg, size_t nv, double vert_init_rad,
                       double lowpt_th, float* cloud_xyz_out, size_t cloud_cap, size_t* n_points_out, int* kp_idx_out,
                       float* kp_xyz_out, float* seg_ratio_out, uint64_t* bits_out, int* n_kp_out);

/* ---- the per-scan odometry step on the device (test/odometry_test.cpp:143-184 in one call) ----------------------------
 * One rotation in, one pose out: Preprocessor::run -> extractKeypoints -> computeDescriptors -> featureMatching (first
 * scan: the frame against itself; later scans: map keypoints within map_range of the last pose ++ the reference frame
 * moved by that pose, mutual nearest neighbours) -> RANSAC -> evaluateEstimation (gate + ICP) -> poseEstimation ->
 * updateMap (whatever the gate says: the reference's check is commented out) -> the frame becomes the reference frame.
 * The result is bit for bit that of bshot_extract_scan, bshot_match_mutual / bshot_match_frame_to_map, bshot_ransac,
 * bshot_evaluate_estimation, bshot_gmap_update_from_frame and bshot_frame_commit called in that order, except h_diff_rad
 * (device acosf).  The context keeps the pose of the last step on the device and the INITIAL / RUN status.
 * After the preprocessor's two count read-backs nothing goes back to the host until one copy of the report at the end.
 * Needs bshot_gmap_create first (BSHOT_E_STATE).  A target set larger than max_targets returns BSHOT_E_CAPACITY; any
 * error leaves pose, status, map and reference frame as they were before the step. */
typedef struct bshot_odom_params {
    bshot_params front;          /* bshot_params_default(): the reference's extraction literals */
    double vert_init_rad;        /* -0.6    test/odometry_test.cpp:32 */
    double lowpt_th;             /* -1950   test/odometry_test.cpp:33 */
    float map_range;             /* 100000  src/lidar_odometry.cpp:198 */
    int ransac_iterations;       /* 2000    src/lidar_odometry.cpp:255 */
    float inlier_threshold;      /* 1500    src/lidar_odometry.cpp:258 */
    int run_icp;                 /* 1       src/lidar_odometry.cpp:6 */
} bshot_odom_params;
void bshot_odom_params_default(bshot_odom_params* p);

typedef struct bshot_odom_report {
    float pose[16];              /* T_best, row-major: what poseEstimation sets */
    float T_ransac[16];          /* RANSAC's transformation (identity when it kept everything) */
    size_t n_points, n_targets;  /* preprocessed points; size of the target set */
    int n_keypoints, n_pairs, n_inliers, ransac_iterations, icp_iterations, should_update_map, was_initial;
    float h_diff_rad, t_diff_mm; /* the gate's heading and translation change */
} bshot_odom_report;

/* raw returns (as bshot_extract_scan) -> pose; out may be NULL */
int bshot_odometry_step(bshot_ctx* ctx, const bshot_odom_params* p, const double* azimuth_deg, const double* vertical_deg,
                        const unsigned short* distance, size_t n, const double* ring_deg, size_t nv, bshot_odom_report* out);
/* an already-preprocessed host cloud (stride 12 or 16 bytes, as bshot_extract_frame): skips the preprocessor */
int bshot_odometry_step_cloud(bshot_ctx* ctx, const bshot_odom_params* p, const float* xyz, size_t n, size_t stride_bytes,
                              bshot_odom_report* out);
/* INITIAL status, identity pose, empty map, no reference frame, fresh persistent normals: the next step replays the
 * sequence as a new context would */
int bshot_odometry_reset(bshot_ctx* ctx);

/* ---- relocalisation: a scan against the whole map, without a prior pose ----------------------------------------------
 * The scan is extracted as by the step (p->front), then its descriptors are matched against EVERY map entry in map order
 * (bshot_gmap_export's order; the reference frame is not a target): mutual nearest neighbours, the matcher chosen by size
 * (the tensor-core pipeline above 2^21 pairs) -> RANSAC (p->ransac_iterations, p->inlier_threshold; sources the keypoints
 * in the sensor frame, targets the entries' positions) -> T_ransac, sensor to map.  p->run_icp: ICP (10 iterations,
 * pre = T_ransac) against the map keypoints within p->map_range of T_ransac's translation, T_best = ICP * T_ransac.
 * accepted = n_inliers >= min_inliers (no heading / translation gate: there is no prior pose; 15 is the gate's own
 * constant).  When accepted, the step's tail runs unchanged: the stored pose becomes T_best, the status RUN, the map is
 * updated with the frame at T_best and the frame becomes the reference frame, so the next bshot_odometry_step continues
 * in the map frame.  When not, pose, status, map and reference frame stay as they were (the extraction's cross-frame
 * front-end state, the persistent normals, moves on as after any extraction).
 * Errors: no map BSHOT_E_STATE; min_inliers < 3 BSHOT_E_INVALID; an ICP target set larger than max_targets
 * BSHOT_E_CAPACITY, with the state unchanged.  An empty map is no error: accepted = 0.  After the preprocessor's count
 * read-backs nothing goes back to the host but the report. */
typedef struct bshot_reloc_report {
    float pose[16];             /* T_best = ICP * T_ransac (T_ransac without ICP), row-major; adopted when accepted */
    float T_ransac[16];
    size_t n_points, n_map, n_icp_targets;   /* preprocessed points; map entries searched; ICP targets */
    int n_keypoints, n_pairs, n_inliers, ransac_iterations, icp_iterations, accepted;
} bshot_reloc_report;
/* raw returns (as bshot_odometry_step) / a preprocessed host cloud (as bshot_odometry_step_cloud); out may be NULL */
int bshot_relocalize(bshot_ctx* ctx, const bshot_odom_params* p, int min_inliers, const double* azimuth_deg, const double* vertical_deg,
                     const unsigned short* distance, size_t n, const double* ring_deg, size_t nv, bshot_reloc_report* out);
int bshot_relocalize_cloud(bshot_ctx* ctx, const bshot_odom_params* p, int min_inliers, const float* xyz, size_t n, size_t stride_bytes,
                           bshot_reloc_report* out);
/* ---- loop closure: revisits of older scans in the map, as constraints for a pose-graph back end ------------------------
 * Map updates are numbered 0, 1, 2, ... since bshot_gmap_create, bshot_gmap_reset or bshot_odometry_reset.  One update is
 * each: odometry step that returns BSHOT_OK, accepted relocalisation, successful bshot_gmap_update_from_frame, successful
 * bshot_gmap_add with n > 0, and successful bshot_gmap_import with n > 0 -- the imported map is update 0, with the
 * identity pose (its entries are in the map frame), and later updates count on from 1.  Failed calls and relocalisations
 * that are not accepted take no number.  Every map entry carries the number of the update that wrote it (an overwrite at
 * an equal position takes the new number: its descriptor is that scan's), and the map keeps the pose each update used
 * (the identity where it had none): the trajectory.  Neither changes what the map stores or returns.
 * bshot_gmap_scans: entry_scan_out[e] is the update of entry e of bshot_gmap_export's order, poses3x4_out (pose_cap x 12
 * floats, row-major [R|T]) the trajectory; *n_entries_out / *n_scans_out their lengths.  Either output may be NULL; an
 * output whose count is above its capacity gets the first cap records and BSHOT_E_CAPACITY is returned.  With
 * entry_scan_out and n_entries_out both NULL the map is not gathered: only the trajectory is read.  No map: BSHOT_E_STATE.  Synchronous. */
int bshot_gmap_scans(bshot_ctx* ctx, uint32_t* entry_scan_out, size_t entry_cap, float* poses3x4_out, size_t pose_cap,
                     size_t* n_entries_out, size_t* n_scans_out);

/* bshot_detect_loop: is the last scan the odometry took (scan i, the reference frame the context holds, update i) a
 * revisit of an older scan?  A read-only query; no extraction.  Candidates: the map entries written by updates
 * j <= i - min_gap, in map order.  The reference frame's descriptors are matched against them (mutual nearest neighbours,
 * the matcher chosen by size or bshot_set_matcher) -> RANSAC (sources the scan's keypoints in its sensor frame) -> T_ransac;
 * run_icp: ICP (10 iterations, pre = T_ransac) against the candidates whose block lies in the +-map_range cube around
 * T_ransac's translation, T_loop = ICP * T_ransac.  The candidates RANSAC's inliers point to vote with their update index:
 * match_scan = the most frequent (the lowest on ties), votes = its count, -1 without inliers.  T_rel = T_j^-1 * T_loop
 * (rigid inverse, T_j the trajectory's pose of match_scan; the identity when match_scan = -1) is the loop edge (j, i):
 * scan i in scan j's frame.  accepted = n_inliers >= min_inliers.  No candidates is no error: n_candidates = 0, not
 * accepted.  Pose, status, map, tags, trajectory, reference frame and the front end's state stay as they were.  The
 * matcher's pair buffer is shared with every matching call: after a detection, bshot_fetch_frame's pairs are the
 * detection's (reference frame -> candidates), as after any later matching call; the next step rewrites them.
 * Errors: BSHOT_E_STATE without a map, or when the last update was not a step or an accepted relocalisation (no step
 * yet, or an import / add / update_from_frame / reset / bshot_ctx_reset / bshot_frame_commit since); BSHOT_E_INVALID for min_gap < 1,
 * min_inliers < 3 or the bounds of bshot_odom_params; BSHOT_E_CAPACITY when the ICP targets exceed max_targets. */
typedef struct bshot_loop_params {
    int min_gap;            /* 100: entries of updates j <= i - min_gap are candidates */
    int min_inliers;        /* 15: accepted when at least this many correspondences survive RANSAC (>= 3) */
    int ransac_iterations;  /* 2000 */
    float inlier_threshold; /* 1500 mm */
    float map_range;        /* 100000 mm: ICP targets = candidates whose block lies in this cube around T_ransac */
    int run_icp;            /* 1 */
} bshot_loop_params;
void bshot_loop_params_default(bshot_loop_params* p);

typedef struct bshot_loop_report {
    float T_loop[16];       /* scan i's pose as the candidates place it: ICP * T_ransac (T_ransac without ICP), row-major */
    float T_ransac[16];
    float T_rel[16];        /* T_j^-1 * T_loop: scan i in scan j's frame, the loop edge (j, i) */
    float pose[16];         /* the odometry's own pose of scan i (T_i); T_i^-1 * T_loop is the drift */
    size_t n_candidates, n_icp_targets;
    int scan, match_scan, votes, n_keypoints, n_pairs, n_inliers, ransac_iterations, icp_iterations, accepted;
} bshot_loop_report;
int bshot_detect_loop(bshot_ctx* ctx, const bshot_loop_params* p, bshot_loop_report* out);

/* bshot_gmap_reanchor: move the map to a corrected trajectory, as a pose-graph back end computes it from the loop edges.
 * poses3x4 (n x 12 floats, row-major [R|T]) is the corrected pose of every map update, n = bshot_gmap_scans' *n_scans_out.
 * Update u's correction is C_u = T'_u * T_u^-1 (fp32, rigid inverse, as T_rel); an update whose pose equals its trajectory
 * pose bit for bit is unchanged.  Every entry of a changed update moves by its update's correction (R p + T, rounded as an
 * update transforms keypoints) and is snapped to the 10 mm lattice; its seg-ratio, descriptor and tag stay, and the entries
 * of unchanged updates stay bit for bit.  The map is then rebuilt from the entries in export order, without the admission
 * rule: two entries moved onto one position both stay, as after bshot_gmap_import.  The trajectory becomes poses3x4 bit
 * for bit.  The odometry's pose becomes T'_{n-1} when it equals T_{n-1} (as after a step), else C_{n-1} * pose; the
 * reference frame is kept in its sensor frame and moves with the pose; before the first odometry step the pose is the
 * identity, and it moves by the same rule.  pose_out (16 floats, may be NULL) gets the new pose.
 * Re-anchoring is not an update: the update count, the status and the reference frame stay, so bshot_detect_loop can run
 * again on the same scan.  Re-anchoring with the current trajectory changes nothing.  Errors (nothing changes):
 * BSHOT_E_STATE without a map; BSHOT_E_INVALID when n is not the update count, or a pose is not finite, has
 * max |R^T R - I| > 1e-3 or det R <= 0, or a moved entry is not storable (bshot_gmap_add); BSHOT_E_CAPACITY when the moved map needs more blocks or chunks than the map
 * holds.  Synchronous. */
int bshot_gmap_reanchor(bshot_ctx* ctx, const float* poses3x4, size_t n, float* pose_out);

/* bshot_optimize_trajectory: the pose graph of the map's trajectory, optimised on the device in float64.  Nodes: the n
 * trajectory poses (bshot_gmap_scans); node 0 is fixed (it defines the map frame).  Odometry edges (u, u + 1) with
 * measurement Z = T_u^-1 T_{u+1} (float64, from the fp32 trajectory); loop edges: the caller's list, e.g. {match_scan, scan,
 * T_rel} of accepted bshot_detect_loop reports.  Edge (a, b) with measurement Z = [R_z | t_z]: residuals
 * r_t = R_a^T (t_b - t_a) - t_z (mm) and r_phi = Log(R_z^T R_a^T R_b) (rad); cost F = 1/2 sum |r_t|^2 / s_t^2 + |r_phi|^2 / s_phi^2
 * with the sigmas of the edge's class.  Levenberg-Marquardt on t <- t + rho, R <- R Exp(phi): (H + lambda diag H) d = -g
 * (lambda starts at 1e-4), solved by conjugate gradients preconditioned with the block-tridiagonal part of the damped
 * matrix (block cyclic reduction along the chain).  A step that lowers F is accepted (lambda / 10), otherwise lambda * 10;
 * every solve counts as an iteration.  Stops when |g|_inf <= grad_tolerance (tested before each solve: a graph without
 * loop edges takes 0 iterations), when max |d| <= step_tolerance (that step is not taken), or after max_iterations.
 * Read only: map, tags, trajectory, pose and reference frame are unchanged; bshot_gmap_reanchor applies the result.
 * poses3x4_out (pose_cap x 12 floats): the optimised poses; node 0, and every node when no step was accepted, keep their
 * input bits.  loop_cost_out[k] (may be NULL): loop edge k's final 1/2 r^T W r.  out (may be NULL): the report.
 * Deterministic: identical inputs give identical bits.  Errors: BSHOT_E_STATE without a map; BSHOT_E_INVALID for an edge
 * index outside [0, n), from == to, a non-finite or non-rigid T (as bshot_gmap_reanchor checks), a sigma <= 0 or a negative
 * iteration count or tolerance; BSHOT_E_CAPACITY when pose_cap < n (nothing is written).  n = 1 returns the trajectory
 * after 0 iterations.  Synchronous; one copy back at the end. */
typedef struct bshot_graph_edge {
    int32_t from, to;       /* `to`'s pose in `from`'s frame is T */
    float T[16];            /* row-major */
} bshot_graph_edge;
typedef struct bshot_graph_params {
    float odom_sigma_mm, odom_sigma_deg;   /* 20 mm, 0.1 deg */
    float loop_sigma_mm, loop_sigma_deg;   /* 100 mm, 1 deg */
    int max_iterations, max_cg_iterations; /* 50, 2000 */
    double grad_tolerance, step_tolerance, cg_tolerance;   /* 1e-6, 1e-9, 1e-10 (relative residual) */
} bshot_graph_params;
void bshot_graph_params_default(bshot_graph_params* p);
typedef struct bshot_graph_report {
    int n_nodes, n_edges, iterations, cg_iterations, status;   /* status: 1 gradient, 2 step, 3 max_iterations */
    double cost_initial, cost_final, grad_inf_final;
} bshot_graph_report;
int bshot_optimize_trajectory(bshot_ctx* ctx, const bshot_graph_edge* loops, size_t n_loops, const bshot_graph_params* p, float* poses3x4_out,
                              size_t pose_cap, double* loop_cost_out, bshot_graph_report* out);

/* bshot_ransac on device buffers, asynchronous on the context stream: d_src4 / d_tgt4 float4 points (x, y, z, any),
 * d_pairs n_pairs_cap x 2 ints (index into src, index into tgt; every valid one must be in range), *d_n_pairs (int) of
 * them valid.  Outputs (device): d_inlier_pairs_out (n_pairs_cap x 2 ints), *d_n_inliers_out (int), d_transform_out
 * (16 floats, row-major), *d_iterations_out (int).  Bit for bit bshot_ransac's results, adaptive stop included
 * (device log / pow may move its count when k lies within a few ulps of an integer). */
int bshot_ransac_dev(bshot_ctx* ctx, const void* d_src4, const void* d_tgt4, const void* d_pairs, const void* d_n_pairs, size_t n_pairs_cap,
                     int max_iterations, float inlier_threshold, void* d_inlier_pairs_out, void* d_n_inliers_out, void* d_transform_out,
                     void* d_iterations_out);

/* ---- ISS keypoints and keypoint repeatability (the reference's kp_test evaluation) ------------ */
/* issKpDetection (src/lidar_odometry.cpp:447-461): pcl::ISSKeypoint3D (PCL 1.8, border radius 0) on the cloud the context
 * holds (after bshot_set_cloud / bshot_extract_frame / bshot_process_frame[_dev] / bshot_extract_scan), on its voxel table.
 * Every finite point p: neighbours = points with fp32 squared distance < salient_radius^2 (p included); with fewer than
 * min_neighbors the scatter matrix is zero, else sum (n - p)(n - p)^T in double; eigenvalues l1 >= l2 >= l3; p is salient
 * when all are finite, l3 >= 0 (PCL leaves both cases to stale memory; here they are "not salient"), l2/l1 < gamma_21 and
 * l3/l2 < gamma_32, and then third_eigen_value(p) = l3, else 0.  Keypoints: third_eigen_value > 0, at least min_neighbors
 * points within non_max_radius (p included) and none of them with a strictly larger third_eigen_value.
 * The call reads no frame state and changes none (keypoints, normals, previous frame, map stay as they were); its
 * max_points-sized buffers are allocated by the first call on a context. */
typedef struct bshot_iss_params {
    float salient_radius;   /* 60     setSalientRadius  src/lidar_odometry.cpp:447-461 */
    float non_max_radius;   /* 40     setNonMaxRadius */
    double gamma_21;        /* 0.975  setThreshold21 */
    double gamma_32;        /* 0.975  setThreshold32 */
    int min_neighbors;      /* 5      PCL's default */
} bshot_iss_params;
void bshot_iss_params_default(bshot_iss_params* p);
/* idx_out / kp_xyz_out: up to cap records, ascending point index. eig_out (N x 3 doubles, lambda1..3; zeros where
 * skipped) may be NULL. count > cap: the first cap are written and BSHOT_E_CAPACITY is returned. */
int bshot_detect_iss(bshot_ctx* ctx, const bshot_iss_params* p, int* idx_out, float* kp_xyz_out, size_t cap,
                     size_t* count_out, double* eig_out);
/* kpEvaluation (src/lidar_odometry.cpp:392-445), the port's own definition: set A (na x 3 floats) moved by a_pose3x4 and
 * set B moved by b_pose3x4 (row-major [R|T], NULL = identity, R * p + T in fp32 as updateMap does); for every point of A
 * the nearest point of B by fp32 squared distance (no FMA contraction, lowest index on ties) -> nn_idx_out[i] (-1 when B
 * is empty) and nn_dist_out[i] (Euclidean, mm); a point is a hit when its squared distance is < radius^2.  The repeat
 * rate is *hits_out / na.  Outputs may be NULL. */
int bshot_kp_repeatability(bshot_ctx* ctx, const float* a_xyz, size_t na, const float* a_pose3x4, const float* b_xyz,
                           size_t nb, const float* b_pose3x4, float radius, int* nn_idx_out, float* nn_dist_out,
                           size_t* hits_out);

/* ---- voxel-grid downsampling (the reference's bshot::calculate_voxel_grid_keypoints) --------- */
/* pcl::VoxelGrid<PointXYZ>::applyFilter of PCL 1.8 with its defaults (all fields averaged, no filter field, no minimum
 * point count) on a host cloud of n points (stride 12 or 16 bytes; not the context's cloud).  inv = 1 / leaf per axis in
 * fp32; non-finite points are skipped; bbox = fp32 min / max of the finite points.  If the grid of
 * (int64)((max - min) * inv) + 1 cells per axis has more than INT32_MAX cells, the output is the input cloud unchanged
 * (every point in order, non-finite ones included).  Otherwise min_b = (int)floor(min * inv), div_b = max_b - min_b + 1,
 * and every finite point goes to voxel idx = ijk . (1, div_b.x, div_b.x * div_b.y) modulo 2^32 with
 * ijk = (int)(floor(p * inv) - (float)min_b) (fp32 products).  One point per occupied voxel in ascending idx: the fp32
 * running sum of its points in ascending point index, divided by the (float) count.
 * xyz_out: up to cap records {x, y, z}; count > cap: the first cap are written, *count_out is the full count and
 * BSHOT_E_CAPACITY is returned.  Leaves that are not finite and > 0, or whose reciprocal is not finite: BSHOT_E_INVALID;
 * n > max_points: BSHOT_E_CAPACITY.  The call reads no frame state and changes none (cloud, voxel table, keypoints,
 * normals, previous frame, map); its max_points-sized buffers are allocated by the first call on a context. */
int bshot_voxel_grid(bshot_ctx* ctx, const float* xyz, size_t n, size_t stride_bytes, float leaf_x, float leaf_y,
                     float leaf_z, float* xyz_out, size_t cap, size_t* count_out);

/* ---- sharded map matching (north_star multi-GPU piece) -------------------------------------- */
/* The accumulated map descriptors (Map::getKeypoints output, include/mymap.h:34-38) are split
 * across ranks; each rank keeps its shard resident.  global_base = index of the shard's first
 * record in the global target array. */
int bshot_map_reset(bshot_ctx* ctx);
int bshot_map_append(bshot_ctx* ctx, const uint64_t* desc, size_t n);
/* same with descriptors that already live on the device (48-byte records) */
int bshot_map_append_dev(bshot_ctx* ctx, const void* d_desc, size_t n);
int bshot_map_size(bshot_ctx* ctx, size_t* n_out);
/* candidate record per query produced by one shard: packed keys (distance << 32 | global index),
 * 0xFFFFFFFFFFFFFFFF = none; rq = best query for target k1 among this call's queries. */
typedef struct bshot_cand {
    uint64_t k1;
    uint64_t k2;
    uint32_t rq;
    uint32_t pad;
} bshot_cand;
/* device pointers, asynchronous on the context stream: d_q (nq x 48 B) against the resident shard
 * -> d_cand_out (nq records).  with_rq != 0 also fills rq (Q x Q reverse pass). */
int bshot_match_shard_dev(bshot_ctx* ctx, const void* d_q, size_t nq, uint64_t global_base,
                          int with_rq, void* d_cand_out);
/* generic device-pointer matcher against caller-owned targets */
int bshot_match_dev(bshot_ctx* ctx, const void* d_q, size_t nq, const void* d_t, size_t nt,
                    uint64_t global_base, int with_rq, void* d_cand_out);
/* merge `nranks` candidate arrays (rank-major, nranks x nq records, e.g. an all-gather result)
 * by (distance, global index); d_out: nq merged records. mutual iff merged rq == query index. */
int bshot_merge_cands_dev(bshot_ctx* ctx, const void* d_cands, size_t nranks, size_t nq,
                          void* d_out);
/* Post-merge reverse pass, sharded: for the queries whose MERGED winner (d_merged, nq records) lies in this
 * rank's shard, find the best query of that target; d_rq_out (nq x u32) gets the query index there and
 * 0xFFFFFFFF elsewhere.  An all-reduce(MIN) of d_rq_out over the ranks followed by bshot_apply_rq_dev
 * completes the records with Q*Q/ranks pairs of work per rank (vs Q*Q for with_rq = 1 above). */
int bshot_reverse_owned_dev(bshot_ctx* ctx, const void* d_q, size_t nq, uint64_t global_base,
                            const void* d_merged, void* d_rq_out);
int bshot_apply_rq_dev(bshot_ctx* ctx, void* d_cands, const void* d_rq, size_t nq);
/* Peer-memory variant of the exchange (symmetric buffers mapped on every rank, e.g. torch symmetric memory over
 * NVLink / NVSwitch): instead of an all-gather, every rank STORES its nq records into slot `rank` of every rank's
 * gather buffer (d_peer_ptrs = device array of nranks pointers to buffers of nranks x nq records); instead of an
 * all-reduce, the owner of a winner stores rq[query] into every rank's rq array (d_peer_rq_ptrs = device array of
 * nranks pointers to nq x uint32).  The caller places one cross-rank barrier after each of the two calls. */
int bshot_push_cands_dev(bshot_ctx* ctx, const void* d_cands, size_t nq, const void* d_peer_ptrs, int nranks, int rank);
/* the barrier: d_peer_flag_ptrs = device array of nranks pointers to each rank's flag array (>= nranks uint32, zero
 * before the first barrier).  Every rank must issue the same sequence of barriers.  A rank that never arrives makes the
 * others give up after ~2 s instead of hanging; bshot_peer_barrier_timeouts then reports the epoch (0 = none). */
int bshot_peer_barrier_dev(bshot_ctx* ctx, const void* d_peer_flag_ptrs, int nranks, int rank);
/* start a new flag array: every rank calls this (collectively) right after its zeroed flag array is allocated, so the
 * barrier epoch always matches the flags -- a second matcher on the same context, or one created after a failed call,
 * starts in step.  Also clears the timeout record. */
int bshot_peer_barrier_reset(bshot_ctx* ctx);
int bshot_peer_barrier_timeouts(bshot_ctx* ctx, unsigned* epoch_out);
int bshot_reverse_owned_push_dev(bshot_ctx* ctx, const void* d_q, size_t nq, uint64_t global_base,
                                 const void* d_merged, const void* d_peer_rq_ptrs, int nranks, int rank);
/* ---- multi-rank exchange behind the C ABI (one process per GPU on one node; no Python / torch / NCCL needed) ------
 * Replaces what featureMatching (src/lidar_odometry.cpp:197-232) does against Map::getKeypoints' output when the
 * map is sharded over GPUs: every rank owns a contiguous range of the global target array (bshot_map_append) and
 * calls bshot_match_map_sharded[_dev] with the same queries; every rank receives all nq complete records (top-2 over
 * the WHOLE map with the reference's first-minimum tie-break, rq = best query of the winner).
 * Set-up, once:  bshot_comm_create on every rank -> bshot_comm_export -> exchange the 64-byte handles by any means
 * (pipe, file, MPI, torch.distributed) -> bshot_comm_import.  Ranks that live in ONE process pass device pointers
 * instead (bshot_comm_region / bshot_comm_import_ptrs; the caller enables peer access between the devices).
 * Per call (six kernel launches, stream-ordered, no host synchronisation): shard search; the merged top-2 records are
 * STORED into every rank's gather buffer over NVLink and a flag is released by the last CTA; the consumer kernel
 * acquires the flags, merges the ranks' records and selects the winners that live in its own shard; their best query
 * (Q x Q / ranks pairs) is stored into every rank's rq array behind a second flag set.  A rank that never arrives
 * makes the others give up after ~2 s: the next bshot_comm_check / bshot_match_map_sharded returns BSHOT_E_STATE. */
typedef struct bshot_ipc_handle { unsigned char bytes[64]; } bshot_ipc_handle;
int bshot_comm_create(bshot_ctx* ctx, int rank, int nranks, size_t max_queries);
int bshot_comm_export(bshot_ctx* ctx, bshot_ipc_handle* handle_out);
int bshot_comm_import(bshot_ctx* ctx, const bshot_ipc_handle* handles /* nranks entries, own entry ignored */);
int bshot_comm_region(bshot_ctx* ctx, void** d_region_out, size_t* bytes_out);
int bshot_comm_import_ptrs(bshot_ctx* ctx, void* const* d_regions /* nranks device pointers, own entry ignored */);
int bshot_comm_destroy(bshot_ctx* ctx);
int bshot_comm_check(bshot_ctx* ctx);
/* device pointers, asynchronous on the context stream: d_q (nq x 48 B) -> d_cand_out (nq bshot_cand records) */
int bshot_match_map_sharded_dev(bshot_ctx* ctx, const void* d_q, size_t nq, uint64_t global_base, void* d_cand_out);
/* host buffers, synchronous; checks the arrival of every rank */
int bshot_match_map_sharded(bshot_ctx* ctx, const uint64_t* q, size_t nq, uint64_t global_base, bshot_cand* cand_out);

/* host-buffer convenience over the three calls above for a single rank */
int bshot_match_map(bshot_ctx* ctx, const uint64_t* q, size_t nq, uint64_t global_base,
                    bshot_cand* cand_out);

/* ---- instrumentation ------------------------------------------------------------------------ */
/* number of kernels this library launched on the context since creation (bench.py gpu_launches) */
unsigned long long bshot_launch_count(bshot_ctx* ctx);
/* per-stage device times of whole-frame calls.  When enabled, CUDA events are recorded on the
 * context stream around each stage; bshot_stage_times synchronises and returns the LAST frame's
 * milliseconds: [0] voxel build, [1] seg-ratio, [2] top-K, [3] normals, [4] SHOT+B-SHOT,
 * [5] matching, [6] whole frame, [7] unused. */
int bshot_ctx_enable_timing(bshot_ctx* ctx, int on);
int bshot_stage_times(bshot_ctx* ctx, float ms_out[8]);
/* work counters of the last frame: [0] sum over points of min(#neighbours, max_nn) in the detector,
 * [1] same for the normals queries, [2] sum of SHOT neighbour counts, [3] keypoints */
int bshot_frame_counters(bshot_ctx* ctx, unsigned long long out[4]);
/* raw device counters of the last frame, for tuning the block-tiled neighbourhood kernel: [0],[1] as above,
 * [2] tiles staged, [3] tile points swept (sum over query attempts of the tile size), [4] query attempts,
 * [5] attempts whose sphere held fewer than max_nn points (retried with a larger tile), [6] queries handed to the
 * warp-per-query fallback, [7] query blocks processed (all tiled launches of the frame together) */
int bshot_debug_counters(bshot_ctx* ctx, unsigned long long out[8]);
/* Which kernel computes the Hamming distance matrix of every search on this context (all of them return the same
 * bit-exact (distance, lowest index) winners as minVect, include/bshot_bits.h:6-20):
 *   BSHOT_MATCHER_AUTO (default)  by problem size: tensor-core pipeline for searches of >= 2^21 pairs, XOR + POPC below
 *   BSHOT_MATCHER_POPC            XOR + POPC top-2 kernel, query tile in registers, targets through TMA (hamming.cu)
 *   BSHOT_MATCHER_TC              tcgen05 kind::i8, one CTA-serial tile at a time (hamming_tc.cu)
 *   BSHOT_MATCHER_TC_PIPELINED    warp-specialised tcgen05 pipeline, query tiles in tensor memory (hamming_tc2.cu)
 *   BSHOT_MATCHER_TC_PIPELINED_SMEM  the same with the query tiles in shared memory
 * The environment variable BSHOT_MATCH_TC=<kind> sets the initial value at bshot_ctx_create. */
#define BSHOT_MATCHER_AUTO (-1)
#define BSHOT_MATCHER_POPC 0
#define BSHOT_MATCHER_TC 1
#define BSHOT_MATCHER_TC_PIPELINED 2
#define BSHOT_MATCHER_TC_PIPELINED_SMEM 3
int bshot_set_matcher(bshot_ctx* ctx, int kind);
/* POPC-pipe microbenchmark: returns measured POPC32 instructions/s over the whole GPU */
int bshot_popc_peak(bshot_ctx* ctx, double* popc_per_s_out);

#ifdef __cplusplus
}
#endif
#endif
