// stages.h -- internal stage entry points (one per SURVEY 8a row); all asynchronous on ctx->stream.
#pragma once
#include "common.cuh"

namespace bshot {

// a1: caller layout in d_raw (stride 3 or 4 floats) -> d_pts, voxel grid, d_sorted   (grid.cu)
int grid_build(Ctx* c, const float* d_raw, size_t n, int stride_floats);

// a2/a3: seg-ratio for every point -> d_ratio, d_keys ; top-K -> d_kp_idx/d_kp_ratio/d_kp/d_kp_count (detect.cu)
int detect_seg_ratio(Ctx* c, float radius, int max_nn, int sr_type, int fuse = 0, int gate_top_k = 0);  // fuse: 1 FULL normals, 2 covariance sums for the keypoint normals
int detect_topk(Ctx* c, int top_k);

// block-tiled exact neighbourhoods of cloud points (tilek.cu): seg-ratio scores and / or normals; d_flags = nullptr: every
// point, else per cell-sorted position the output slot (>= 0) of the points that want a normal
int tile_neighbourhoods(Ctx* c, int sr_type, bool seg, int nrm, float radius, int max_nn, const int* d_flags, float4* d_nrm_out, int gate_top_k = 0);
bool tile_path_ok(const Ctx* c, int max_nn);
// normals of the detector's keypoints at their ordinals, from the radii the detector kept (tilek.cu)
int tile_keypoint_normals(Ctx* c, float radius, int max_nn, float4* d_nrm_out);
// normals of the queries the tiled kernel put on the fallback list (normals.cu)
int normals_fallback_list(Ctx* c, float radius, int max_nn, const int* d_flags, float4* d_out);

// a4: normals (normals.cu). normals_query: q (float4 xyz_) -> out (nx,ny,nz,curvature); in-place allowed
int normals_query(Ctx* c, const float4* d_q, size_t nq, float radius, int max_nn, float4* d_out);
int normals_compute(Ctx* c, int mode, float radius, int max_nn);

// a5/a6/a7: LRF + SHOT352 + B-SHOT for the current keypoints (shot.cu)
int shot_compute(Ctx* c, float radius, bool lrf_only, bool write_shot);
int binarize(Ctx* c, const float* d_shot, size_t k, uint64_t* d_bits);

// a10/a11 (hamming.cu)
int hamming_top2(Ctx* c, const void* d_q, size_t nq, const void* d_t, size_t nt, unsigned long long global_base,
                 bshot_cand* d_out, unsigned* d_colmin = nullptr, const unsigned* d_nq = nullptr, const unsigned* d_nt = nullptr);
int hamming_reverse_owned(Ctx* c, const void* d_q, size_t nq, const void* d_t, size_t nt, unsigned long long global_base,
                          const bshot_cand* d_merged, unsigned* d_rq_out, const void* d_peer_rq = nullptr, unsigned nranks = 1,
                          unsigned rank = 0);
int hamming_peer_barrier(Ctx* c, const void* d_peer_flags, unsigned nranks, unsigned rank);
int hamming_push_cands(Ctx* c, const bshot_cand* d_cands, size_t nq, const void* d_peer_ptrs, unsigned nranks, unsigned rank);
int hamming_apply_rq(Ctx* c, bshot_cand* d_cand, const unsigned* d_rq, size_t nq);
int hamming_match_rq(Ctx* c, const void* d_q, size_t nq, const void* d_t, size_t nt, unsigned long long global_base,
                     bshot_cand* d_out, const unsigned* d_nq = nullptr, const unsigned* d_nt = nullptr);
int hamming_reverse(Ctx* c, const void* d_q, size_t nq, const void* d_t, unsigned long long global_base,
                    bshot_cand* d_cand, const unsigned* d_nq = nullptr);
int hamming_merge_cands(Ctx* c, const void* d_cands, size_t nranks, size_t nq, void* d_out);
int hamming_unpack(Ctx* c, const bshot_cand* d_cand, size_t nq, int* idx1, int* d1, int* idx2, int* d2);
int hamming_mutual_pairs(Ctx* c, const bshot_cand* d_cand, size_t nq, int* d_pairs3, int* d_count, const unsigned* d_nq = nullptr);
int popc_peak(Ctx* c, double* out);
// sharded map match over peer memory (six launches, hamming.cu)
size_t comm_region_bytes(const Comm& m);
int comm_set_peers(Ctx* c, void* const* region_ptrs);
int hamming_preload_sharded();
int hamming_match_sharded(Ctx* c, const void* d_q, size_t nq, unsigned long long global_base, bshot_cand* d_out);

// tensor-core distance matrix (hamming_tc.cu): per-split top-2 partials in c->d_partial
int hamming_tc_partials(Ctx* c, const void* d_q, size_t nq, const void* d_t, size_t nt, unsigned long long global_base, const unsigned* d_nq,
                        const unsigned* d_nt, unsigned* nsplit_out);
int hamming_tc2_preload();
int hamming_tc2_partials(Ctx* c, const void* d_q, size_t nq, const void* d_t, size_t nt, unsigned long long global_base, const unsigned* d_nq,
                         const unsigned* d_nt, unsigned* nsplit_out, size_t live_q = 0);

// GPU-resident global map (gmap.cu)
int gmap_create(Ctx* c, size_t max_entries, size_t max_blocks);
void gmap_free(Ctx* c);
int gmap_reset(Ctx* c);
// a map update has succeeded: at most n_cap more entries, the next update number, and whether the update was a scan that is
// now the reference frame (a step or an accepted relocalisation).  Every kind of update records itself here, once
void gmap_record_update(Ctx* c, size_t n_cap, bool by_scan);
// pose_on_device: pose12 / ref_pose12 are device pointers (the odometry step); gmap_gather then takes the position from the
// translation of ref_pose12 on the device (pos unused)
int gmap_update(Ctx* c, const float4* d_kp, const float* d_ratio, const uint64_t* d_bits, const int* d_count, size_t n_cap, const float* pose12,
                bool pose_on_device = false);
int gmap_gather(Ctx* c, const float pos[3], float range, const float4* d_ref_kp, const uint64_t* d_ref_bits, const int* d_ref_count,
                size_t ref_cap, const float* ref_pose12, uint64_t* d_t_out, size_t out_cap, unsigned* d_total, bool pose_on_device = false);
// the whole map in map order (occupied blocks in ascending lattice coordinates, x outermost, entries in insertion order) ->
// gmap.d_apos / d_adesc, the count in gmap.d_actl[1]; *nt_cap_out = its host-side bound.  Asynchronous
int gmap_gather_all(Ctx* c, size_t* nt_cap_out, bool with_tags = false);
// synchronous: export copies min(count, cap) records (float4 position + seg-ratio, 48-byte descriptor); import replaces
// the map by n entries without the admission rule, keeping the input order inside each block (an empty map on any error)
int gmap_export(Ctx* c, float* xyzr_out, uint64_t* desc_out, size_t cap, size_t* n_out);
int gmap_import(Ctx* c, const float* xyzr, const uint64_t* desc, size_t n);
// the import's device core, synchronous: rebuilds the table from d_pos / d_desc (*d_n entries, n_cap without a device
// count) in their order, without the admission rule.  d_tag null: every tag 0 and the trajectory's update 0 the identity
// (an import); otherwise the tags from d_tag and the trajectory untouched.  Host state (update count, bounds) is the
// caller's; on BSHOT_E_INVALID / BSHOT_E_CAPACITY (messages prefixed by who) the table is unusable until rebuilt or reset
int gmap_import_dev(Ctx* c, const float4* d_pos, const uint64_t* d_desc, const unsigned* d_tag, size_t n_cap, const unsigned* d_n, const char* who);
// bshot_gmap_reanchor's work (synchronous), n == the update count, checked by the caller; d_pose: the odometry's pose
int gmap_reanchor(Ctx* c, const float* poses3x4, size_t n, float* d_pose, float* pose_out);
// synchronous: the entries' tags in export order and the trajectory (bshot_gmap_scans)
int gmap_scans(Ctx* c, uint32_t* entry_scan_out, size_t entry_cap, float* poses3x4_out, size_t pose_cap, size_t* n_entries_out, size_t* n_scans_out);
// loop closure, asynchronous: the whole map in map order with tags, then the entries with tag + min_gap <= scan, in map order
// -> gmap.d_lpos / d_ldesc / d_ltag, count in gmap.d_lctl[0] (*nc_cap_out = its host-side bound).  Then the candidates whose
// block lies in the +-range cube around the translation of the device pose d_T -> gmap.d_tpos, count in gmap.d_lctl[2];
// more than max_targets sets *d_err = BSHOT_E_CAPACITY
int gmap_loop_candidates(Ctx* c, unsigned scan, unsigned min_gap, size_t* nc_cap_out);
int gmap_loop_icp_targets(Ctx* c, const float* d_T, float range, size_t nc_cap, int* d_err);

// stable LSD radix sort of (u64 key, u32 value) pairs, 8 bits a pass (voxel_grid.cu): *d_m pairs (at most m_cap) in
// keys[0] / vals[0], `passes` passes from the low byte up; the result is in keys[passes & 1] / vals[passes & 1].  hist
// holds radix_hist_words(m_cap) words
size_t radix_hist_words(size_t m_cap);
int radix_sort_pairs(Ctx* c, unsigned long long* keys[2], unsigned* vals[2], unsigned* hist, const unsigned* d_m, size_t m_cap, unsigned passes);

// RANSAC correspondence rejection (ransac.cu).  ransac_run draws PCL's sample sequence on the host, ransac_run_dev on the
// device; after the sampler both run the same device tail (scoring, adaptive stop, inlier flags, ordered compaction).
// ransac_run is synchronous
int ransac_run(Ctx* c, const float* src_xyz, const float* tgt_xyz, const int* pairs, size_t n_pairs, int max_iterations, double threshold,
               int* inlier_pairs_out, int* n_inliers_out, float* transform_out, int* iterations_out);
// device inputs: d_pairs = n_cap records of pair_stride ints (query, match, ...), *d_n_pairs of them valid;
// outputs in device memory.  A set *d_skip (may be null) treats the input as empty.  Asynchronous
int ransac_run_dev(Ctx* c, const float4* d_src, const float4* d_tgt, const int* d_pairs, int pair_stride, const int* d_n_pairs, size_t n_cap,
                   int max_iterations, double threshold, int* d_pairs_out, int* d_n_out, float* d_T_out, int* d_iterations_out, const int* d_skip);

// ICP refinement (icp.cu)
struct IcpState {
    float final_T[16];
    double prev_mse, mse;
    int iterations, state, done, pad;
};
int icp_run(Ctx* c, const float* src_xyz, size_t n_src, const float* tgt_xyz, size_t n_tgt, const float* pre4x4, int max_iterations,
            float* final4x4_out, int* iterations_out, int* state_out, double* mse_out);
// icp_run uploads its inputs and runs icp_run_dev.  Points are src_stride / tgt_stride floats apart (3 or 4), the counts are
// device-side with host-known capacities (see icp.cu); the result stays in *d_st.  Asynchronous
int icp_run_dev(Ctx* c, const float* d_src, int src_stride, const int* d_ns, size_t ns_cap, const float* d_tgt, int tgt_stride, const unsigned* d_nt,
                size_t nt_cap, const float* d_pre, int max_iterations, const int* d_skip, float4* d_cur, float4* d_tgt_buf, unsigned long long* d_keys,
                IcpState* d_st);

// scan preprocessor (preprocess.cu); scratch_reserve grows one of the context's on-demand scratch buffers
int scratch_reserve(Ctx* c, int which, size_t bytes);
int preprocess_run(Ctx* c, const double* az_deg, const double* vert_deg, const unsigned short* dist, size_t n, const double* ring_deg, size_t nv,
                   double vert_init, double lowpt_th, const unsigned char* sel, int save_sel, float* xyz_out, size_t cap, size_t* n_out,
                   const float** d_xyz_out = nullptr);

// ISS keypoints on the resident cloud and keypoint repeatability (iss.cu).  iss_detect leaves the count and the first
// min(cap, n) records {index, x, y, z} in c->iss.h_rec[1..] (synchronous); the eigenvalues stay in c->iss.d_eig
int iss_detect(Ctx* c, float rs, float rnm, double g21, double g32, int min_nn, size_t cap, bool want_eig, size_t* count_out);
void iss_free(Ctx* c);
int kp_repeatability(Ctx* c, const float* a_xyz, size_t na, const float* a_pose, const float* b_xyz, size_t nb, const float* b_pose, float radius,
                     int* nn_idx_out, float* nn_dist_out, size_t* hits_out);

// voxel-grid downsampling of a host cloud (voxel_grid.cu): inv = 1 / leaf per axis.  Leaves the count and the first
// min(cap, n) records {x, y, z} in c->vg.h_out[4..] (synchronous)
int voxel_grid(Ctx* c, const float* xyz, size_t n, int stride_floats, const float inv[3], size_t cap, size_t* count_out);
void vg_free(Ctx* c);

// registration against the map (odometry.cu): the odometry step, relocalisation and loop detection run the same
// registration (match_mutual, RANSAC, optional ICP, one final kernel, one copy of the report back) on different target
// sets.  odometry_run takes the cloud already on the device and ends with one synchronisation (the report);
// odometry_reset is synchronous
int odom_ensure(Ctx* c);
void odom_free(Ctx* c);
int odometry_reset(Ctx* c);
int odometry_run(Ctx* c, const bshot_odom_params* p, const float* d_cloud, size_t n, int stride_floats, bshot_odom_report* out);
// relocalisation against the whole map; the same shape as odometry_run, and the same end when accepted
int relocalize_run(Ctx* c, const bshot_odom_params* p, int min_inliers, const float* d_cloud, size_t n, int stride_floats, bshot_reloc_report* out);
// loop detection on the reference frame against the map's older entries; reads, never changes, the odometry's state
int loop_run(Ctx* c, const bshot_loop_params* p, bshot_loop_report* out);
// re-anchoring (odometry.cu, without FMA): per update u of n, changed[u] = d_new's pose differs from d_traj's in any bit,
// and then corr[u] = T'_u * T_u^-1 (row-major 3x4); pose_new = the odometry's pose d_pose moved by update n - 1's
// correction (T'_{n-1} itself when d_pose is T_{n-1}).  Asynchronous
int reanchor_corrections(Ctx* c, const float* d_traj, const float* d_new, unsigned n, float* d_corr, unsigned* d_changed, const float* d_pose, float* d_pose_new);
// bshot_optimize_trajectory on the map's trajectory (posegraph.cu), inputs checked by the caller; synchronous
int pose_graph_run(Ctx* c, const bshot_graph_edge* loops, size_t n_loops, const bshot_graph_params* p, float* poses_out, double* loop_cost_out,
                   bshot_graph_report* out);
// bshot_gmap_reanchor on the odometry's pose (gmap_reanchor)
int reanchor_run(Ctx* c, const float* poses3x4, size_t n, float* pose_out);

// whole frame on the resident cloud (frame.cu)
int frame_extract(Ctx* c, const bshot_params* p, const float* d_raw, size_t n, int stride_floats);
// mutual nearest neighbours of k query descriptors against nt_cap targets -> c->d_pairs / c->d_pair_count.  d_nq / d_nt
// (may be null) are the device-side counts within those bounds; nt_cap == 0 only sets the pair count to 0
int match_mutual(Ctx* c, const uint64_t* d_q, size_t k, const uint64_t* d_t, size_t nt_cap, const unsigned* d_nq = nullptr,
                 const unsigned* d_nt = nullptr);
// the current frame becomes the reference frame (descriptors, keypoint positions and count stay on the device).  A set
// *d_skip (may be null) leaves the reference frame as it is; with a flag the caller sets c->n_prev once it has read it
int frame_commit(Ctx* c, size_t k, const int* d_skip = nullptr);
// featureMatching against the map (src/lidar_odometry.cpp:197-206), used by bshot_match_frame_to_map and the odometry step:
// target set = map keypoints in range ++ the reference frame moved by ref_pose12 (gmap_gather into d_t / gmap.d_tpos, the
// count in gmap.d_ctl[6]), then match_mutual of the frame's k descriptors against it (its bound *nt_cap_out)
int frame_match_map(Ctx* c, size_t k, const float pos[3], float range, const float* ref_pose12, bool pose_on_device, size_t* nt_cap_out);
// the target set overflowed max_targets: more candidates than max_targets, and the gather stopped at max_targets.  ctl is
// gmap.d_ctl after frame_match_map ([4] map keypoints in range, [6] targets assembled)
__host__ __device__ inline bool target_set_overflow(const unsigned* ctl, size_t n_prev, size_t max_targets) {
    return (size_t)ctl[4] + n_prev > max_targets && (size_t)ctl[6] == max_targets;
}
int frame_run(Ctx* c, const bshot_params* p, const float* d_raw, size_t n, int stride_floats);

}  // namespace bshot
