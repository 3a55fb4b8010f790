// odometry.cu -- the per-scan odometry step on the device (test/odometry_test.cpp:143-184 in one call).
//
// The stages are the existing ones; what changes is that their inputs stay on the device:
//   extract (frame_extract) -> first scan: the frame's descriptors against themselves, later scans: the map keypoints in
//   range of the stored pose ++ the reference frame moved by it (gmap_gather with the pose on the device) -> mutual nearest
//   neighbours (match_mutual, device-side counts) -> RANSAC on the device (reg_ransac) -> the gate of evaluateEstimation
//   (odom_math.cuh, the host's code) -> ICP on the device (reg_icp) -> T_best -> updateMap (gmap_update with the pose on
//   the device) -> the frame becomes the reference frame (scan_enqueue).
// The only host round trip after the preprocessor is the copy of the report at the end (copy_back).  A target set larger
// than max_targets is detected on the device (the host call's test, on device counts): the flag makes RANSAC and ICP no-ops
// and keeps the pose, the map and the reference frame as they were.  Compiled with -fmad=false: the gate and the
// composition T_best = F * T_est give the host's bits.
//
// Relocalisation (relocalize_run) runs the same registration without a prior pose: the whole map in map order is the
// target set (gmap_gather_all), RANSAC and ICP (around T_ransac) run as in the step, and the step's end -- pose, status,
// map update, reference frame -- runs only when enough inliers survived; one device flag skips it otherwise.
//
// Loop detection (loop_run) runs it once more on the reference frame, read only: the map's entries of updates at least
// min_gap older than the scan are the target set (gmap_loop_candidates), RANSAC, ICP against the candidates around
// T_ransac, then the candidates RANSAC kept vote for the scan they came from.  Its own device record (LoopDev); the only
// scratch it writes is the matcher's, RANSAC's and ICP's, which every step rewrites before reading.
//
// The three share RegDev (RANSAC's outputs and the error flag), reg_ransac / reg_icp, reg_report (T_best and the counters
// of every report) and copy_back; each final kernel adds only its own fields.
#include <algorithm>
#include <cmath>
#include <cstddef>

#include "common.cuh"
#include "odom_math.cuh"
#include "stages.h"

namespace bshot {

// RANSAC's outputs and the registration's error flag: BSHOT_E_CAPACITY when the target set (the step) or the ICP targets
// (relocalisation, loop detection) exceed max_targets.  A set flag skips RANSAC and ICP
struct RegDev {
    int err;
    int n_inliers, ransac_iterations;
    float T_ransac[16];
};

// rep, reg and rrep lie next to each other: the step copies rep + reg back, relocalisation reg + rrep
struct OdomDev {
    bshot_odom_report rep;
    RegDev reg;
    bshot_reloc_report rrep;
    int eff_count;           // keypoints the map update takes: the frame's count, 0 after an error or a rejection
    int reject;              // relocalisation: not accepted (or an error), skips the reference frame as err skips the step's
    float pose[16];          // pose of the last successful step, row-major (identity after a reset)
    float T_est[16];
};

// loop detection's device record, copied back whole
struct LoopDev {
    bshot_loop_report rep;
    RegDev reg;
};

__global__ void odom_reset_kernel(OdomDev* d) {
    if (threadIdx.x < 16) d->pose[threadIdx.x] = (threadIdx.x % 5 == 0) ? 1.0f : 0.0f;
    if (threadIdx.x == 0) { d->reg.err = 0; d->reject = 0; }
}

// bshot_match_frame_to_map's capacity test on the device counts
__global__ void odom_check_kernel(const unsigned* __restrict__ ctl, size_t n_prev, size_t max_targets, OdomDev* d) {
    if (target_set_overflow(ctl, n_prev, max_targets)) d->reg.err = BSHOT_E_CAPACITY;
}

// evaluateEstimation's gate (src/lidar_odometry.cpp:267-281): T_est = T_ref when rejected, else T_ransac
__global__ void odom_gate_kernel(OdomDev* d) {
    float h, t;
    const bool reject = estimation_gate(d->reg.T_ransac, d->pose, d->reg.n_inliers, &h, &t);
    for (int e = 0; e < 16; ++e) d->T_est[e] = reject ? d->pose[e] : d->reg.T_ransac[e];
    d->rep.h_diff_rad = h;
    d->rep.t_diff_mm = t;
    d->rep.should_update_map = reject ? 0 : 1;
}

// what every registration reports: T_ransac; the keypoints and pairs, clamped to [0, k]; RANSAC's inliers and iterations;
// ICP's iterations.  T_best = ICP * T_init after ICP, else T_ransac (also in the step, whatever its gate chose)
template <class Report>
__device__ void reg_report(const RegDev& reg, const IcpState* icp, int run_icp, const float* T_init, const int* kp_count, const int* pair_count, int k,
                           Report& r, float T_best[16]) {
    if (run_icp) mul4x4(icp->final_T, T_init, T_best);
    else for (int e = 0; e < 16; ++e) T_best[e] = reg.T_ransac[e];
    for (int e = 0; e < 16; ++e) r.T_ransac[e] = reg.T_ransac[e];
    r.n_keypoints = min(max(*kp_count, 0), k);
    r.n_pairs = min(max(*pair_count, 0), k);
    r.n_inliers = reg.n_inliers;
    r.ransac_iterations = reg.ransac_iterations;
    r.icp_iterations = run_icp ? icp->iterations : 0;
}

// relocalisation and loop detection accept a registration by its inlier count
__device__ __forceinline__ bool reg_accepted(const RegDev& reg, int min_inliers) { return reg.err == 0 && reg.n_inliers >= min_inliers; }

// T_best (:293 / :295), the report, and -- without an error -- the new pose and the map update's count
__global__ void odom_final_kernel(OdomDev* d, const IcpState* __restrict__ icp, int run_icp, const int* __restrict__ kp_count,
                                  const int* __restrict__ pair_count, const unsigned* __restrict__ d_total, int k, unsigned long long n_points,
                                  int was_initial) {
    float T_best[16];
    bshot_odom_report& r = d->rep;
    reg_report(d->reg, icp, run_icp, d->T_est, kp_count, pair_count, k, r, T_best);
    for (int e = 0; e < 16; ++e) r.pose[e] = T_best[e];
    r.n_points = (size_t)n_points;
    r.n_targets = was_initial ? (size_t)r.n_keypoints : (size_t)*d_total;
    r.was_initial = was_initial;
    if (d->reg.err == 0) {
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
    bshot_reloc_report& r = d->rrep;
    reg_report(d->reg, icp, run_icp, d->reg.T_ransac, kp_count, pair_count, k, r, T_best);
    for (int e = 0; e < 16; ++e) r.pose[e] = T_best[e];
    r.n_points = (size_t)n_points;
    r.n_map = (size_t)*n_map;
    r.n_icp_targets = run_icp ? (size_t)*n_icp : 0;
    const bool accepted = reg_accepted(d->reg, min_inliers);
    r.accepted = accepted ? 1 : 0;
    d->reject = accepted ? 0 : 1;
    if (accepted) {
        for (int e = 0; e < 16; ++e) d->pose[e] = T_best[e];
        d->eff_count = *kp_count;
    } else {
        d->eff_count = 0;
    }
}

// the vote over the candidates RANSAC kept (update index -> count; the most frequent, the lowest on ties), then T_loop,
// T_rel = T_j^-1 * T_loop and the report.  n^2 tag comparisons for n inliers (n <= the reference frame's keypoints)
__global__ void __launch_bounds__(256)
loop_final_kernel(LoopDev* d, const IcpState* __restrict__ icp, int run_icp, int min_inliers, const int* __restrict__ inl, const unsigned* __restrict__ cand_tag,
                  const float* __restrict__ traj, unsigned scan, const int* __restrict__ kp_count, const int* __restrict__ pair_count,
                  const unsigned* __restrict__ lctl, int k) {
    __shared__ unsigned long long best;   // (count << 32) | ~tag
    if (threadIdx.x == 0) best = 0ull;
    __syncthreads();
    const int n = min(max(d->reg.n_inliers, 0), k);
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
    reg_report(d->reg, icp, run_icp, d->reg.T_ransac, kp_count, pair_count, k, r, T_loop);
    const int match = best ? (int)(0xFFFFFFFFu - (unsigned)(best & 0xFFFFFFFFull)) : -1;
    for (int e = 0; e < 16; ++e) {
        r.T_loop[e] = T_loop[e];
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
    r.accepted = reg_accepted(d->reg, min_inliers) ? 1 : 0;
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

// RANSAC on the matcher's pairs (queries d_src, matches d_tgt) into reg, skipped when reg->err is set
static int reg_ransac(Ctx* c, const float4* d_src, const float4* d_tgt, size_t k, int iterations, float threshold, RegDev* reg) {
    return ransac_run_dev(c, d_src, d_tgt, c->d_pairs, 3, c->d_pair_count, k, iterations, (double)threshold, c->odom.d_inlier_pairs, &reg->n_inliers,
                          reg->T_ransac, &reg->ransac_iterations, &reg->err);
}

// ICP (10 iterations from T_init) of the first *d_ns of d_src against the first *d_nt of d_tgt, skipped when reg->err is set
static int reg_icp(Ctx* c, const float4* d_src, const int* d_ns, size_t k, const float4* d_tgt, const unsigned* d_nt, size_t nt_cap, const float* T_init,
                   RegDev* reg) {
    Odom& o = c->odom;
    return icp_run_dev(c, reinterpret_cast<const float*>(d_src), 4, d_ns, k, reinterpret_cast<const float*>(d_tgt), 4, d_nt, nt_cap, T_init, 10, &reg->err,
                       o.d_icp_cur, o.d_icp_tgt, o.d_icp_keys, o.d_icp_state);
}

// the one copy back of a run: bytes [first, last) of the device record d into the pinned h, then a synchronise.  h_nk (may
// be null) is the report's keypoint count, which becomes the host-side count; a device error becomes the call's error
static int copy_back(Ctx* c, const void* d, void* h, size_t first, size_t last, const RegDev& h_reg, const int* h_nk, const char* what) {
    BSHOT_CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(h) + first, static_cast<const char*>(d) + first, last - first, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (h_nk) c->n_kp = (size_t)*h_nk;
    if (h_reg.err) {
        set_error("%s exceeds max_targets %zu", what, c->max_targets);
        return h_reg.err;
    }
    return BSHOT_OK;
}

// the end of a step or a relocalisation on the device: updateMap (:343-358) with the device pose and eff_count (0 after an
// error or a rejection: the map stays), then the frame becomes the reference frame unless *d_skip
static int scan_enqueue(Ctx* c, size_t k, const int* d_skip) {
    OdomDev* d = c->odom.d;
    BSHOT_TRY(gmap_update(c, c->d_kp, c->d_kp_ratio, c->d_bits, &d->eff_count, c->last_top_k, d->pose, /*pose_on_device=*/true));
    return frame_commit(c, k, d_skip);
}

// ... and on the host, once the report shows the scan was taken
static void scan_commit(Ctx* c, size_t k) {
    gmap_record_update(c, c->last_top_k, /*by_scan=*/true);
    c->n_prev = k;
    c->odom.run = true;
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
    BSHOT_CUDA_TRY(cudaMemsetAsync(&d->reg.err, 0, sizeof(int), c->stream));
    const unsigned* d_nq = reinterpret_cast<const unsigned*>(c->d_kp_count);
    const float4* tgt_pos;
    const unsigned* d_nt;
    size_t nt_cap;
    if (initial) {   // src/lidar_odometry.cpp:187-194: the target is the frame itself
        BSHOT_TRY(match_mutual(c, c->d_bits, k, c->d_bits, k, d_nq, d_nq));
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
    BSHOT_TRY(reg_ransac(c, c->d_kp, tgt_pos, k, p->ransac_iterations, p->inlier_threshold, &d->reg));
    odom_gate_kernel<<<1, 1, 0, c->stream>>>(d);
    count_launch(c);
    if (p->run_icp) BSHOT_TRY(reg_icp(c, c->d_kp, c->d_kp_count, k, tgt_pos, d_nt, nt_cap, d->T_est, &d->reg));   // :283-293
    odom_final_kernel<<<1, 1, 0, c->stream>>>(d, o.d_icp_state, p->run_icp ? 1 : 0, c->d_kp_count, c->d_pair_count, initial ? nullptr : g.d_ctl + 6, (int)k,
                                              (unsigned long long)n, initial ? 1 : 0);
    count_launch(c);
    BSHOT_TRY(check_launch("odometry step kernels"));
    // updateMap with T_best, whatever the gate said; after an error the reference frame stays too
    BSHOT_TRY(scan_enqueue(c, k, &d->reg.err));
    OdomDev* h = reinterpret_cast<OdomDev*>(o.h_out);
    BSHOT_TRY(copy_back(c, d, h, 0, offsetof(OdomDev, reg) + sizeof(RegDev), h->reg, &h->rep.n_keypoints, "bshot_odometry_step: target set"));
    scan_commit(c, k);
    if (out) *out = h->rep;
    return BSHOT_OK;
}

// relocalisation: the step's extraction, the whole map as the target set, RANSAC, ICP against the map around T_ransac,
// acceptance by inlier count, and -- when accepted -- the step's end.  One copy back (report + flags) at the end
int relocalize_run(Ctx* c, const bshot_odom_params* p, int min_inliers, const float* d_cloud, size_t n, int stride_floats, bshot_reloc_report* out) {
    BSHOT_TRY(odom_ensure(c));
    Odom& o = c->odom;
    Gmap& g = c->gmap;
    OdomDev* d = o.d;
    BSHOT_TRY(frame_extract(c, &p->front, d_cloud, n, stride_floats));
    const size_t k = (size_t)p->front.top_k;
    BSHOT_CUDA_TRY(cudaMemsetAsync(&d->reg.err, 0, sizeof(int), c->stream));
    // targets: every map entry in map order (no reference frame)
    size_t nm_cap;
    BSHOT_TRY(gmap_gather_all(c, &nm_cap));
    const unsigned* d_nm = g.d_actl + 1;
    BSHOT_TRY(match_mutual(c, c->d_bits, k, g.d_adesc, nm_cap, reinterpret_cast<const unsigned*>(c->d_kp_count), d_nm));
    BSHOT_TRY(reg_ransac(c, c->d_kp, g.d_apos, k, p->ransac_iterations, p->inlier_threshold, &d->reg));
    if (p->run_icp) {   // map keypoints within map_range of T_ransac's translation ([R|T] = its first 12 floats)
        BSHOT_TRY(gmap_gather(c, nullptr, p->map_range, nullptr, nullptr, nullptr, 0, d->reg.T_ransac, c->d_t, c->max_targets, g.d_ctl + 6,
                              /*pose_on_device=*/true));
        odom_check_kernel<<<1, 1, 0, c->stream>>>(g.d_ctl, 0, c->max_targets, d);
        count_launch(c);
        BSHOT_TRY(reg_icp(c, c->d_kp, c->d_kp_count, k, g.d_tpos, g.d_ctl + 6, std::min(c->max_targets, g.entries_upper), d->reg.T_ransac, &d->reg));
    }
    reloc_final_kernel<<<1, 1, 0, c->stream>>>(d, o.d_icp_state, p->run_icp ? 1 : 0, min_inliers, c->d_kp_count, c->d_pair_count, d_nm, g.d_ctl + 6, (int)k,
                                               (unsigned long long)n);
    count_launch(c);
    BSHOT_TRY(check_launch("relocalisation kernels"));
    // not accepted: the count is 0 and the reference frame is skipped
    BSHOT_TRY(scan_enqueue(c, k, &d->reject));
    OdomDev* h = reinterpret_cast<OdomDev*>(o.h_out);
    BSHOT_TRY(copy_back(c, d, h, offsetof(OdomDev, reg), offsetof(OdomDev, rrep) + sizeof(bshot_reloc_report), h->reg, &h->rrep.n_keypoints,
                        "bshot_relocalize: ICP target set"));
    if (h->rrep.accepted) scan_commit(c, k);
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
    BSHOT_TRY(match_mutual(c, c->d_prev_bits, k, g.d_ldesc, nc_cap, reinterpret_cast<const unsigned*>(c->d_prev_count), g.d_lctl));
    BSHOT_TRY(reg_ransac(c, c->d_prev_kp, g.d_lpos, k, p->ransac_iterations, p->inlier_threshold, &d->reg));
    if (p->run_icp) {
        BSHOT_TRY(gmap_loop_icp_targets(c, d->reg.T_ransac, p->map_range, nc_cap, &d->reg.err));
        BSHOT_TRY(reg_icp(c, c->d_prev_kp, c->d_prev_count, k, g.d_tpos, g.d_lctl + 2, std::min(c->max_targets, nc_cap), d->reg.T_ransac, &d->reg));
    } else {
        BSHOT_CUDA_TRY(cudaMemsetAsync(g.d_lctl + 2, 0, sizeof(unsigned) * 2, c->stream));
    }
    loop_final_kernel<<<1, 256, 0, c->stream>>>(d, o.d_icp_state, p->run_icp ? 1 : 0, p->min_inliers, o.d_inlier_pairs, g.d_ltag, g.d_traj, scan, c->d_prev_count,
                                                c->d_pair_count, g.d_lctl, (int)k);
    count_launch(c);
    BSHOT_TRY(check_launch("loop detection kernels"));
    LoopDev* h = reinterpret_cast<LoopDev*>(o.h_loop);
    BSHOT_TRY(copy_back(c, d, h, 0, sizeof(LoopDev), h->reg, nullptr, "bshot_detect_loop: ICP target set"));
    if (out) *out = h->rep;
    return BSHOT_OK;
}

}  // namespace bshot
