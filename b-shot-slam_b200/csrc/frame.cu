// frame.cu -- the reference's per-frame call order on the resident cloud, fully asynchronous:
// extractKeypoints -> computeDescriptors -> featureMatching (test/odometry_test.cpp:174-194,
// src/lidar_odometry.cpp:51-265 up to the RANSAC call).
#include <algorithm>

#include "stages.h"

namespace bshot {

__global__ void copy_prev_kernel(const uint64_t* __restrict__ bits, const float4* __restrict__ kp, const int* __restrict__ count, unsigned cap,
                                 const int* __restrict__ skip, uint64_t* __restrict__ prev, float4* __restrict__ prev_kp, int* __restrict__ prev_count) {
    if (skip && *skip) return;
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const int k = *count;
    if (i < cap * 6 && (int)(i / 6) < k) prev[i] = bits[i];
    if (i < cap && (int)i < k) prev_kp[i] = kp[i];
    if (i == 0) *prev_count = k;
}

int frame_commit(Ctx* c, size_t k, const int* d_skip) {
    copy_prev_kernel<<<(unsigned)((k * 6 + 255) / 256), 256, 0, c->stream>>>(c->d_bits, c->d_kp, c->d_kp_count, (unsigned)k, d_skip, c->d_prev_bits,
                                                                            c->d_prev_kp, c->d_prev_count);
    count_launch(c);
    if (!d_skip) {
        c->n_prev = k;
        c->gmap.last_by_scan = false;   // the reference frame is no longer the scan of the last map update
    }
    return check_launch("copy_prev_kernel");
}

int match_mutual(Ctx* c, const uint64_t* d_q, size_t k, const uint64_t* d_t, size_t nt_cap, const unsigned* d_nq, const unsigned* d_nt) {
    if (nt_cap == 0) {
        BSHOT_CUDA_TRY(cudaMemsetAsync(c->d_pair_count, 0, sizeof(int), c->stream));
        return BSHOT_OK;
    }
    BSHOT_TRY(hamming_match_rq(c, d_q, k, d_t, nt_cap, 0, c->d_cand, d_nq, d_nt));
    return hamming_mutual_pairs(c, c->d_cand, k, c->d_pairs, c->d_pair_count, d_nq);
}

int frame_match_map(Ctx* c, size_t k, const float pos[3], float range, const float* ref_pose12, bool pose_on_device, size_t* nt_cap_out) {
    unsigned* d_total = c->gmap.d_ctl + 6;
    BSHOT_TRY(gmap_gather(c, pos, range, c->d_prev_kp, c->d_prev_bits, c->d_prev_count, c->n_prev, ref_pose12, c->d_t, c->max_targets, d_total,
                          pose_on_device));
    *nt_cap_out = std::min(c->max_targets, c->gmap.entries_upper + c->n_prev);
    return match_mutual(c, c->d_bits, k, c->d_t, *nt_cap_out, reinterpret_cast<const unsigned*>(c->d_kp_count), d_total);
}

// extractKeypoints + computeDescriptors (src/lidar_odometry.cpp:51-184) on a cloud in device memory, asynchronous
int frame_extract(Ctx* c, const bshot_params* p, const float* d_raw, size_t n, int stride_floats) {
    auto mark = [&](int i) {
        if (c->timing) cudaEventRecord(c->ev[i], c->stream);
    };
    BSHOT_CUDA_TRY(cudaMemsetAsync(c->d_counters, 0, 8 * sizeof(unsigned long long), c->stream));
    mark(0);
    BSHOT_TRY(grid_build(c, d_raw, n, stride_floats));
    mark(1);
    // FULL-mode normals use the detector's own neighbourhoods when the search parameters agree: one pass for both
    const bool same = p->normal_radius == p->kp_radius && p->normal_max_nn == p->kp_max_nn;
    const int fuse = !same ? 0 : (p->normals_mode == BSHOT_NORMALS_FULL ? 1 : 2);
    // sums for the deferred keypoint normals only where the previous frame's K-th score makes a keypoint likely
    const int gate = (c->gate_top_k == p->top_k && c->gate_sr == p->sr_type && c->gate_radius == p->kp_radius && c->gate_max_nn == p->kp_max_nn) ? p->top_k : 0;
    BSHOT_TRY(detect_seg_ratio(c, p->kp_radius, p->kp_max_nn, p->sr_type, fuse, gate));
    mark(2);
    BSHOT_TRY(detect_topk(c, p->top_k));
    c->gate_top_k = p->top_k; c->gate_sr = p->sr_type; c->gate_radius = p->kp_radius; c->gate_max_nn = p->kp_max_nn;
    mark(3);
    BSHOT_TRY(normals_compute(c, p->normals_mode, p->normal_radius, p->normal_max_nn));
    mark(4);
    BSHOT_TRY(shot_compute(c, p->shot_radius, false, false));
    mark(5);
    c->last_top_k = (size_t)p->top_k;
    return BSHOT_OK;
}

int frame_run(Ctx* c, const bshot_params* p, const float* d_raw, size_t n, int stride_floats) {
    auto mark = [&](int i) {
        if (c->timing) cudaEventRecord(c->ev[i], c->stream);
    };
    BSHOT_TRY(frame_extract(c, p, d_raw, n, stride_floats));
    if (c->ev_desc) BSHOT_CUDA_TRY(cudaEventRecord(c->ev_desc, c->stream));   // descriptors complete: bshot_process_frame starts their copy here
    // featureMatching: the initial frame is matched against itself (src/lidar_odometry.cpp:187-194),
    // later frames against the previous frame's descriptors.  Host-side counts are upper bounds
    // (top_k); the kernels trim queries AND targets by the device-side keypoint counts, so a frame that
    // yields fewer than top_k keypoints (the reference's `< 600` branch, :144-151) never matches stale records.
    const size_t k = (size_t)p->top_k;
    const bool initial = (c->n_prev == 0);
    const uint64_t* tgt = initial ? c->d_bits : c->d_prev_bits;
    const size_t nt = initial ? k : c->n_prev;
    const unsigned* d_nq = reinterpret_cast<const unsigned*>(c->d_kp_count);
    const unsigned* d_nt = reinterpret_cast<const unsigned*>(initial ? c->d_kp_count : c->d_prev_count);
    BSHOT_TRY(match_mutual(c, c->d_bits, k, tgt, nt, d_nq, d_nt));
    BSHOT_TRY(frame_commit(c, k));
    mark(6);
    c->ev_valid = c->timing;
    return BSHOT_OK;
}

}  // namespace bshot
