// odometry.cu -- the per-scan odometry step on the device (test/odometry_test.cpp:143-184 in one call).
//
// The stages are the existing ones; what changes is that their inputs stay on the device:
//   extract (frame_extract) -> first scan: the frame's descriptors against themselves, later scans: the map keypoints in
//   range of the stored pose ++ the reference frame moved by it (gmap_gather with the pose on the device) -> mutual nearest
//   neighbours (device-side counts) -> RANSAC on the device (ransac_run_dev) -> the gate of evaluateEstimation
//   (odom_math.cuh, the host's code) -> ICP on the device (icp_run_dev) -> T_best -> updateMap (gmap_update with the pose on
//   the device) -> the frame becomes the reference frame.
// The only host round trip after the preprocessor is the copy of the report at the end.  A target set larger than
// max_targets is detected on the device (the host call's test, on device counts): the flag makes RANSAC and ICP no-ops and
// keeps the pose, the map and the reference frame as they were.  Compiled with -fmad=false: the gate and the composition
// T_best = F * T_est give the host's bits.
//
// Relocalisation (relocalize_run) reuses the same stages without a prior pose: the whole map in map order is the target
// set (gmap_gather_all), RANSAC and ICP (around T_ransac) run as in the step, and the step's tail -- pose, status, map
// update, reference frame -- runs only when enough inliers survived; one device flag skips it otherwise.
//
// Loop detection (loop_run) reuses them once more on the reference frame, read only: the map's entries of updates at least
// min_gap older than the scan are the target set (gmap_loop_candidates), RANSAC, ICP against the candidates around
// T_ransac, then the candidates RANSAC kept vote for the scan they came from.  Its own device report (LoopDev); the only
// scratch it writes is the matcher's, RANSAC's and ICP's, which every step rewrites before reading.
#include <algorithm>
#include <cmath>
#include <cstddef>

#include "common.cuh"
#include "odom_math.cuh"
#include "stages.h"

namespace bshot {

struct OdomDev {
    bshot_odom_report rep;   // copied to the host at the end of a step, together with err
    int err;                 // BSHOT_E_* raised on the device during the step (0 = none)
    int eff_count;           // keypoints the map update takes: the frame's count, 0 after an error
    int reject;              // relocalisation: not accepted (or an error), skips the tail like err skips the step's
    int pad;
    bshot_reloc_report rrep; // copied to the host at the end of a relocalisation, together with err and reject
    float pose[16];          // pose of the last successful step, row-major (identity after a reset)
    float T_est[16];
    float T_ransac[16];
    int n_inliers, ransac_iterations;
};

__global__ void odom_reset_kernel(OdomDev* d) {
    if (threadIdx.x < 16) d->pose[threadIdx.x] = (threadIdx.x % 5 == 0) ? 1.0f : 0.0f;
    if (threadIdx.x == 0) { d->err = 0; d->reject = 0; }
}

// bshot_match_frame_to_map's capacity test on the device counts
__global__ void odom_check_kernel(const unsigned* __restrict__ ctl, size_t n_prev, size_t max_targets, OdomDev* d) {
    if (target_set_overflow(ctl, n_prev, max_targets)) d->err = BSHOT_E_CAPACITY;
}

// evaluateEstimation's gate (src/lidar_odometry.cpp:267-281): T_est = T_ref when rejected, else T_ransac
__global__ void odom_gate_kernel(OdomDev* d) {
    float h, t;
    const bool reject = estimation_gate(d->T_ransac, d->pose, d->n_inliers, &h, &t);
    for (int e = 0; e < 16; ++e) d->T_est[e] = reject ? d->pose[e] : d->T_ransac[e];
    d->rep.h_diff_rad = h;
    d->rep.t_diff_mm = t;
    d->rep.should_update_map = reject ? 0 : 1;
}

// T_best (:293 / :295), the report, and -- without an error -- the new pose and the map update's count
__global__ void odom_final_kernel(OdomDev* d, const IcpState* __restrict__ icp, int run_icp, const int* __restrict__ kp_count,
                                  const int* __restrict__ pair_count, const unsigned* __restrict__ d_total, int k, unsigned long long n_points,
                                  int was_initial) {
    float T_best[16];
    if (run_icp) mul4x4(icp->final_T, d->T_est, T_best);
    else for (int e = 0; e < 16; ++e) T_best[e] = d->T_ransac[e];
    bshot_odom_report& r = d->rep;
    for (int e = 0; e < 16; ++e) { r.pose[e] = T_best[e]; r.T_ransac[e] = d->T_ransac[e]; }
    const int nk = min(max(*kp_count, 0), k);
    r.n_points = (size_t)n_points;
    r.n_targets = was_initial ? (size_t)nk : (size_t)*d_total;
    r.n_keypoints = nk;
    r.n_pairs = min(max(*pair_count, 0), k);
    r.n_inliers = d->n_inliers;
    r.ransac_iterations = d->ransac_iterations;
    r.icp_iterations = run_icp ? icp->iterations : 0;
    r.was_initial = was_initial;
    if (d->err == 0) {
        for (int e = 0; e < 16; ++e) d->pose[e] = T_best[e];
        d->eff_count = *kp_count;
    } else {
        d->eff_count = 0;
    }
}

// relocalisation: T_best, the report, accepted; when accepted the new pose, the status flag and the map update's count
__global__ void reloc_final_kernel(OdomDev* d, const IcpState* __restrict__ icp, int run_icp, int min_inliers, const int* __restrict__ kp_count,
                                   const int* __restrict__ pair_count, const unsigned* __restrict__ n_map, const unsigned* __restrict__ n_icp, int k,
                                   unsigned long long n_points) {
    float T_best[16];
    if (run_icp) mul4x4(icp->final_T, d->T_ransac, T_best);
    else for (int e = 0; e < 16; ++e) T_best[e] = d->T_ransac[e];
    bshot_reloc_report& r = d->rrep;
    for (int e = 0; e < 16; ++e) { r.pose[e] = T_best[e]; r.T_ransac[e] = d->T_ransac[e]; }
    const int nk = min(max(*kp_count, 0), k);
    r.n_points = (size_t)n_points;
    r.n_map = (size_t)*n_map;
    r.n_icp_targets = run_icp ? (size_t)*n_icp : 0;
    r.n_keypoints = nk;
    r.n_pairs = min(max(*pair_count, 0), k);
    r.n_inliers = d->n_inliers;
    r.ransac_iterations = d->ransac_iterations;
    r.icp_iterations = run_icp ? icp->iterations : 0;
    const bool accepted = d->err == 0 && d->n_inliers >= min_inliers;
    r.accepted = accepted ? 1 : 0;
    d->reject = accepted ? 0 : 1;
    if (accepted) {
        for (int e = 0; e < 16; ++e) d->pose[e] = T_best[e];
        d->eff_count = *kp_count;
    } else {
        d->eff_count = 0;
    }
}

// loop detection's device report
struct LoopDev {
    bshot_loop_report rep;   // copied to the host at the end, together with err
    int err;                 // BSHOT_E_CAPACITY: more ICP targets than max_targets (ICP is skipped)
    int n_inliers, ransac_iterations, pad;
    float T_ransac[16];
};

// the vote over the candidates RANSAC kept (update index -> count; the most frequent, the lowest on ties), then T_loop,
// T_rel = T_j^-1 * T_loop and the report.  n^2 tag comparisons for n inliers (n <= the reference frame's keypoints)
__global__ void __launch_bounds__(256)
loop_final_kernel(LoopDev* d, const IcpState* __restrict__ icp, int run_icp, int min_inliers, const int* __restrict__ inl, const unsigned* __restrict__ cand_tag,
                  const float* __restrict__ traj, unsigned scan, const int* __restrict__ kp_count, const int* __restrict__ pair_count,
                  const unsigned* __restrict__ lctl, int k) {
    __shared__ unsigned long long best;   // (count << 32) | ~tag
    if (threadIdx.x == 0) best = 0ull;
    __syncthreads();
    const int n = min(max(d->n_inliers, 0), k);
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
        const unsigned tag = cand_tag[inl[2 * t + 1]];
        unsigned cnt = 0;
        for (int u = 0; u < n; ++u) cnt += cand_tag[inl[2 * u + 1]] == tag ? 1u : 0u;
        atomicMax(&best, ((unsigned long long)cnt << 32) | (unsigned long long)(0xFFFFFFFFu - tag));
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    bshot_loop_report& r = d->rep;
    float T_loop[16], Tj[16], Tj_inv[16];
    if (run_icp) mul4x4(icp->final_T, d->T_ransac, T_loop);
    else for (int e = 0; e < 16; ++e) T_loop[e] = d->T_ransac[e];
    const int match = best ? (int)(0xFFFFFFFFu - (unsigned)(best & 0xFFFFFFFFull)) : -1;
    for (int e = 0; e < 16; ++e) {
        r.T_loop[e] = T_loop[e];
        r.T_ransac[e] = d->T_ransac[e];
        r.pose[e] = e < 12 ? traj[(size_t)scan * 12 + e] : (e == 15 ? 1.0f : 0.0f);
        r.T_rel[e] = (e % 5 == 0) ? 1.0f : 0.0f;
        Tj[e] = match >= 0 && e < 12 ? traj[(size_t)match * 12 + e] : (e == 15 ? 1.0f : 0.0f);
    }
    if (match >= 0) {
        rigid_inverse4x4(Tj, Tj_inv);
        mul4x4(Tj_inv, T_loop, r.T_rel);
    }
    r.n_candidates = lctl[0];
    r.n_icp_targets = run_icp ? lctl[2] : 0;
    r.scan = (int)scan;
    r.match_scan = match;
    r.votes = best ? (int)(best >> 32) : 0;
    r.n_keypoints = min(max(*kp_count, 0), k);
    r.n_pairs = min(max(*pair_count, 0), k);
    r.n_inliers = d->n_inliers;
    r.ransac_iterations = d->ransac_iterations;
    r.icp_iterations = run_icp ? icp->iterations : 0;
    r.accepted = (d->err == 0 && d->n_inliers >= min_inliers) ? 1 : 0;
}

// re-anchoring: one thread per update.  An update whose new pose equals its old one bit for bit is unchanged (its entries
// and, for the last update, the odometry's pose stay); otherwise C_u = T'_u * T_u^-1 in fp32 (odom_math.cuh, no FMA)
__global__ void reanchor_corr_kernel(const float* __restrict__ traj, const float* __restrict__ traj_new, unsigned n, float* __restrict__ corr,
                                     unsigned* __restrict__ changed, const float* __restrict__ pose, float* __restrict__ pose_new) {
    const unsigned u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n) return;
    float T[16], Tn[16], T_inv[16], C[16];
    bool chg = false;
    for (int e = 0; e < 16; ++e) {
        T[e] = e < 12 ? traj[(size_t)u * 12 + e] : (e == 15 ? 1.0f : 0.0f);
        Tn[e] = e < 12 ? traj_new[(size_t)u * 12 + e] : T[e];
        chg = chg || __float_as_uint(T[e]) != __float_as_uint(Tn[e]);
    }
    changed[u] = chg ? 1u : 0u;
    if (chg) {
        rigid_inverse4x4(T, T_inv);
        mul4x4(Tn, T_inv, C);
        for (int e = 0; e < 12; ++e) corr[(size_t)u * 12 + e] = C[e];
    }
    if (u != n - 1) return;
    bool at_last = true;   // the pose is the last update's (the case after a step)
    for (int e = 0; e < 12; ++e) at_last = at_last && __float_as_uint(pose[e]) == __float_as_uint(T[e]);
    float P[16];
    if (!chg) for (int e = 0; e < 16; ++e) P[e] = pose[e];
    else if (at_last) for (int e = 0; e < 16; ++e) P[e] = Tn[e];
    else mul4x4(C, pose, P);
    for (int e = 0; e < 16; ++e) pose_new[e] = P[e];
}

int reanchor_corrections(Ctx* c, const float* d_traj, const float* d_new, unsigned n, float* d_corr, unsigned* d_changed, const float* d_pose, float* d_pose_new) {
    reanchor_corr_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(d_traj, d_new, n, d_corr, d_changed, d_pose, d_pose_new);
    count_launch(c);
    return check_launch("reanchor_corr_kernel");
}

int reanchor_run(Ctx* c, const float* poses3x4, size_t n, float* pose_out) {
    BSHOT_TRY(odom_ensure(c));
    return gmap_reanchor(c, poses3x4, n, c->odom.d->pose, pose_out);
}

int odom_ensure(Ctx* c) {
    Odom& o = c->odom;
    if (o.d) return BSHOT_OK;
    BSHOT_CUDA_TRY(cudaMalloc((void**)&o.d, sizeof(OdomDev)));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&o.d_inlier_pairs, sizeof(int) * 2 * c->max_kp));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&o.d_icp_cur, sizeof(float4) * c->max_kp));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&o.d_icp_keys, sizeof(unsigned long long) * c->max_kp));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&o.d_icp_tgt, sizeof(float4) * c->max_targets));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&o.d_icp_state, sizeof(IcpState)));
    BSHOT_CUDA_TRY(cudaMallocHost(&o.h_out, sizeof(OdomDev)));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&o.d_loop, sizeof(LoopDev)));
    BSHOT_CUDA_TRY(cudaMallocHost(&o.h_loop, sizeof(LoopDev)));
    BSHOT_CUDA_TRY(cudaMemsetAsync(o.d, 0, sizeof(OdomDev), c->stream));
    odom_reset_kernel<<<1, 32, 0, c->stream>>>(o.d);
    count_launch(c);
    o.run = false;
    return check_launch("odom_reset_kernel");
}

void odom_free(Ctx* c) {
    Odom& o = c->odom;
    void* ptrs[] = {o.d, o.d_inlier_pairs, o.d_icp_cur, o.d_icp_keys, o.d_icp_tgt, o.d_icp_state, o.d_loop};
    for (void* p : ptrs) if (p) cudaFree(p);
    if (o.h_out) cudaFreeHost(o.h_out);
    if (o.h_loop) cudaFreeHost(o.h_loop);
    o = Odom();
}

int odometry_reset(Ctx* c) {
    BSHOT_TRY(odom_ensure(c));
    odom_reset_kernel<<<1, 32, 0, c->stream>>>(c->odom.d);
    count_launch(c);
    BSHOT_TRY(check_launch("odom_reset_kernel"));
    c->odom.run = false;
    BSHOT_TRY(gmap_reset(c));
    c->gmap.entries_upper = 0;
    // no reference frame, and the cross-frame state of the front end as a new context has it
    BSHOT_CUDA_TRY(cudaMemsetAsync(c->d_prev_count, 0, sizeof(int), c->stream));
    BSHOT_CUDA_TRY(cudaMemsetAsync(c->d_normals, 0, sizeof(float4) * c->max_points, c->stream));
    c->n_prev = 0;
    c->normals_valid = 0;
    c->have_normals = false;
    c->gate_top_k = 0;
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return BSHOT_OK;
}

// everything after the cloud is on the device (d_cloud: n points, stride_floats 3 or 4); n_points is reported as is
int odometry_run(Ctx* c, const bshot_odom_params* p, const float* d_cloud, size_t n, int stride_floats, bshot_odom_report* out) {
    BSHOT_TRY(odom_ensure(c));
    Odom& o = c->odom;
    Gmap& g = c->gmap;
    OdomDev* d = o.d;
    BSHOT_TRY(frame_extract(c, &p->front, d_cloud, n, stride_floats));
    const size_t k = (size_t)p->front.top_k;
    const bool initial = !o.run;
    BSHOT_CUDA_TRY(cudaMemsetAsync(&d->err, 0, sizeof(int), c->stream));
    const unsigned* d_nq = reinterpret_cast<const unsigned*>(c->d_kp_count);
    const float4* tgt_pos;
    const unsigned* d_nt;
    size_t nt_cap;
    if (initial) {   // src/lidar_odometry.cpp:187-194: the target is the frame itself
        BSHOT_TRY(hamming_match_rq(c, c->d_bits, k, c->d_bits, k, 0, c->d_cand, d_nq, d_nq));
        BSHOT_TRY(hamming_mutual_pairs(c, c->d_cand, k, c->d_pairs, c->d_pair_count, d_nq));
        tgt_pos = c->d_kp;
        d_nt = d_nq;
        nt_cap = k;
    } else {         // :197-206: map keypoints in range of the last pose ++ the reference frame moved by that pose
        BSHOT_TRY(frame_match_map(c, k, nullptr, p->map_range, d->pose, /*pose_on_device=*/true, &nt_cap));
        odom_check_kernel<<<1, 1, 0, c->stream>>>(g.d_ctl, c->n_prev, c->max_targets, d);
        count_launch(c);
        tgt_pos = g.d_tpos;
        d_nt = g.d_ctl + 6;
    }
    // featureMatching's RANSAC (:251-261) on the pairs (query, match, distance) the matcher left on the device
    BSHOT_TRY(ransac_run_dev(c, c->d_kp, tgt_pos, c->d_pairs, 3, c->d_pair_count, k, p->ransac_iterations, (double)p->inlier_threshold, o.d_inlier_pairs,
                             &d->n_inliers, d->T_ransac, &d->ransac_iterations, &d->err));
    odom_gate_kernel<<<1, 1, 0, c->stream>>>(d);
    count_launch(c);
    if (p->run_icp) {   // :283-293 on the frame's keypoints and the target set
        BSHOT_TRY(icp_run_dev(c, reinterpret_cast<const float*>(c->d_kp), 4, c->d_kp_count, k, reinterpret_cast<const float*>(tgt_pos), 4, d_nt, nt_cap,
                              d->T_est, 10, &d->err, o.d_icp_cur, o.d_icp_tgt, o.d_icp_keys, o.d_icp_state));
    }
    odom_final_kernel<<<1, 1, 0, c->stream>>>(d, o.d_icp_state, p->run_icp ? 1 : 0, c->d_kp_count, c->d_pair_count, initial ? nullptr : g.d_ctl + 6, (int)k,
                                              (unsigned long long)n, initial ? 1 : 0);
    count_launch(c);
    BSHOT_TRY(check_launch("odometry step kernels"));
    // updateMap (:343-358) with T_best, whatever the gate said; after an error the count is 0 and the map stays
    BSHOT_TRY(gmap_update(c, c->d_kp, c->d_kp_ratio, c->d_bits, &d->eff_count, c->last_top_k, d->pose, /*pose_on_device=*/true));
    BSHOT_TRY(frame_commit(c, k, &d->err));   // skipped after an error: the reference frame stays
    OdomDev* h = reinterpret_cast<OdomDev*>(o.h_out);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(h, d, offsetof(OdomDev, err) + sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->n_kp = (size_t)h->rep.n_keypoints;
    if (h->err) {
        set_error("bshot_odometry_step: target set exceeds max_targets %zu", c->max_targets);
        return h->err;
    }
    g.entries_upper += c->last_top_k;
    ++g.n_updates;
    g.last_by_scan = true;
    c->n_prev = k;
    o.run = true;
    if (out) *out = h->rep;
    return BSHOT_OK;
}

// relocalisation: the step's extraction, the whole map as the target set, RANSAC, ICP against the map around T_ransac,
// acceptance by inlier count, and -- when accepted -- the step's tail.  One copy back (report + flags) at the end
int relocalize_run(Ctx* c, const bshot_odom_params* p, int min_inliers, const float* d_cloud, size_t n, int stride_floats, bshot_reloc_report* out) {
    BSHOT_TRY(odom_ensure(c));
    Odom& o = c->odom;
    Gmap& g = c->gmap;
    OdomDev* d = o.d;
    BSHOT_TRY(frame_extract(c, &p->front, d_cloud, n, stride_floats));
    const size_t k = (size_t)p->front.top_k;
    BSHOT_CUDA_TRY(cudaMemsetAsync(&d->err, 0, sizeof(int), c->stream));
    const unsigned* d_nq = reinterpret_cast<const unsigned*>(c->d_kp_count);
    // targets: every map entry in map order (no reference frame)
    size_t nm_cap;
    BSHOT_TRY(gmap_gather_all(c, &nm_cap));
    const unsigned* d_nm = g.d_actl + 1;
    if (nm_cap == 0) {
        BSHOT_CUDA_TRY(cudaMemsetAsync(c->d_pair_count, 0, sizeof(int), c->stream));
    } else {
        BSHOT_TRY(hamming_match_rq(c, c->d_bits, k, g.d_adesc, nm_cap, 0, c->d_cand, d_nq, d_nm));
        BSHOT_TRY(hamming_mutual_pairs(c, c->d_cand, k, c->d_pairs, c->d_pair_count, d_nq));
    }
    BSHOT_TRY(ransac_run_dev(c, c->d_kp, g.d_apos, c->d_pairs, 3, c->d_pair_count, k, p->ransac_iterations, (double)p->inlier_threshold, o.d_inlier_pairs,
                             &d->n_inliers, d->T_ransac, &d->ransac_iterations, nullptr));
    if (p->run_icp) {   // map keypoints within map_range of T_ransac's translation ([R|T] = its first 12 floats)
        BSHOT_TRY(gmap_gather(c, nullptr, p->map_range, nullptr, nullptr, nullptr, 0, d->T_ransac, c->d_t, c->max_targets, g.d_ctl + 6,
                              /*pose_on_device=*/true));
        odom_check_kernel<<<1, 1, 0, c->stream>>>(g.d_ctl, 0, c->max_targets, d);
        count_launch(c);
        const size_t nt_cap = std::min(c->max_targets, g.entries_upper);
        BSHOT_TRY(icp_run_dev(c, reinterpret_cast<const float*>(c->d_kp), 4, c->d_kp_count, k, reinterpret_cast<const float*>(g.d_tpos), 4, g.d_ctl + 6, nt_cap,
                              d->T_ransac, 10, &d->err, o.d_icp_cur, o.d_icp_tgt, o.d_icp_keys, o.d_icp_state));
    }
    reloc_final_kernel<<<1, 1, 0, c->stream>>>(d, o.d_icp_state, p->run_icp ? 1 : 0, min_inliers, c->d_kp_count, c->d_pair_count, d_nm, g.d_ctl + 6, (int)k,
                                               (unsigned long long)n);
    count_launch(c);
    BSHOT_TRY(check_launch("relocalisation kernels"));
    // the step's tail; not accepted: the count is 0 and the reference frame is skipped
    BSHOT_TRY(gmap_update(c, c->d_kp, c->d_kp_ratio, c->d_bits, &d->eff_count, c->last_top_k, d->pose, /*pose_on_device=*/true));
    BSHOT_TRY(frame_commit(c, k, &d->reject));
    OdomDev* h = reinterpret_cast<OdomDev*>(o.h_out);
    const size_t first = offsetof(OdomDev, err), last = offsetof(OdomDev, rrep) + sizeof(bshot_reloc_report);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(h) + first, reinterpret_cast<const char*>(d) + first, last - first, cudaMemcpyDeviceToHost,
                                   c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->n_kp = (size_t)h->rrep.n_keypoints;
    if (h->err) {
        set_error("bshot_relocalize: ICP target set exceeds max_targets %zu", c->max_targets);
        return h->err;
    }
    if (h->rrep.accepted) {
        g.entries_upper += c->last_top_k;
        ++g.n_updates;
        g.last_by_scan = true;
        c->n_prev = k;
        o.run = true;
    }
    if (out) *out = h->rrep;
    return BSHOT_OK;
}

// loop detection on the reference frame (scan i = the last update): candidates, mutual nearest neighbours, RANSAC, ICP
// around T_ransac, vote and T_rel.  Asynchronous up to one copy back (report + error) at the end
int loop_run(Ctx* c, const bshot_loop_params* p, bshot_loop_report* out) {
    Gmap& g = c->gmap;
    Odom& o = c->odom;
    if (!g.d_tab || !o.d || !g.last_by_scan || g.n_updates == 0) {
        set_error("bshot_detect_loop: the last map update was not an odometry step or an accepted relocalisation");
        return BSHOT_E_STATE;
    }
    LoopDev* d = reinterpret_cast<LoopDev*>(o.d_loop);
    const unsigned scan = g.n_updates - 1;
    const size_t k = c->n_prev;
    BSHOT_CUDA_TRY(cudaMemsetAsync(d, 0, sizeof(LoopDev), c->stream));
    size_t nc_cap;
    BSHOT_TRY(gmap_loop_candidates(c, scan, (unsigned)p->min_gap, &nc_cap));
    const unsigned* d_nq = reinterpret_cast<const unsigned*>(c->d_prev_count);
    if (nc_cap == 0) {
        BSHOT_CUDA_TRY(cudaMemsetAsync(c->d_pair_count, 0, sizeof(int), c->stream));
    } else {
        BSHOT_TRY(hamming_match_rq(c, c->d_prev_bits, k, g.d_ldesc, nc_cap, 0, c->d_cand, d_nq, g.d_lctl));
        BSHOT_TRY(hamming_mutual_pairs(c, c->d_cand, k, c->d_pairs, c->d_pair_count, d_nq));
    }
    BSHOT_TRY(ransac_run_dev(c, c->d_prev_kp, g.d_lpos, c->d_pairs, 3, c->d_pair_count, k, p->ransac_iterations, (double)p->inlier_threshold, o.d_inlier_pairs,
                             &d->n_inliers, d->T_ransac, &d->ransac_iterations, nullptr));
    if (p->run_icp) {
        BSHOT_TRY(gmap_loop_icp_targets(c, d->T_ransac, p->map_range, nc_cap, &d->err));
        const size_t nt_cap = std::min(c->max_targets, nc_cap);
        BSHOT_TRY(icp_run_dev(c, reinterpret_cast<const float*>(c->d_prev_kp), 4, c->d_prev_count, k, reinterpret_cast<const float*>(g.d_tpos), 4, g.d_lctl + 2,
                              nt_cap, d->T_ransac, 10, &d->err, o.d_icp_cur, o.d_icp_tgt, o.d_icp_keys, o.d_icp_state));
    } else {
        BSHOT_CUDA_TRY(cudaMemsetAsync(g.d_lctl + 2, 0, sizeof(unsigned) * 2, c->stream));
    }
    loop_final_kernel<<<1, 256, 0, c->stream>>>(d, o.d_icp_state, p->run_icp ? 1 : 0, p->min_inliers, o.d_inlier_pairs, g.d_ltag, g.d_traj, scan, c->d_prev_count,
                                                c->d_pair_count, g.d_lctl, (int)k);
    count_launch(c);
    BSHOT_TRY(check_launch("loop detection kernels"));
    LoopDev* h = reinterpret_cast<LoopDev*>(o.h_loop);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(h, d, offsetof(LoopDev, err) + sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (h->err) {
        set_error("bshot_detect_loop: ICP target set exceeds max_targets %zu", c->max_targets);
        return h->err;
    }
    if (out) *out = h->rep;
    return BSHOT_OK;
}

}  // namespace bshot
