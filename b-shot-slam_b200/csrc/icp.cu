// icp.cu -- ICP refinement of the keypoints on the device (SURVEY 8f "next" #3).
//
// Replaces the pcl::IterativeClosestPoint<PointXYZ, PointXYZ> of LidarOdometry::evaluateEstimation
// (src/lidar_odometry.cpp:285-291): the frame's keypoints, already moved by the gated estimate T_est, are aligned to the
// assembled target keypoints with PCL's defaults, i.e. PCL 1.8's loop
//   * correspondences: the nearest target of every (moved) source point, exact, squared distance in float (FLANN L2_Simple:
//     ((dx*dx) + dy*dy) + dz*dz), no distance cap (sqrt(DBL_MAX)), no rejectors; ties -> lowest target index;
//   * transformation: TransformationEstimationSVD<.., float> = Umeyama without scaling on all pairs, float sums; pcl::umeyama's
//     rank rule (float precision): rank 3 -> S(2) = sign(det Sigma), rank 2 -> right-handed completion.  Rank <= 1 (all
//     pairs on one target, sources on a line, ...) -> a deterministic proper rotation with R v0 = u0, the identity at rank 0
//     (rigid_rotation_rank01; rank 0 when sv[0] is within the fp32 rounding noise of Sigma, rigid_noise_floor).  At exact
//     rank <= 1 PCL's choice depends on Eigen's SVD internals and may be improper; for 0 < sv[1] <= 1e-5 sv[0] PCL keeps
//     the roll about the line, which this rule drops (DESIGN 3.5);
//   * the source is moved by it (float 4x4 * point, left to right), final = T * final;
//   * DefaultConvergenceCriteria as ICP configures it: 10 iterations; rotation threshold 1.0 and translation threshold 0
//     (transformation_epsilon = 0) -> only an exact identity stops it; |mse - previous mse| < 1e-12; relative mse never
//     (euclidean_fitness_epsilon = -DBL_MAX).  Fewer than 3 correspondences -> not converged.
// Two kernels an iteration and no host round trip inside the loop: a finished state turns the remaining launches into
// no-ops.  The float sums run as 256 strided partial sums + a fixed halving tree, the 3x3 SVD (one-sided Jacobi) in double;
// compiled with -fmad=false, so the CPU restatement in the test oracle (orc_icp) reproduces every bit.
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "rigid_math.cuh"
#include "stages.h"

namespace bshot {

constexpr int ICP_T = 256;        // threads of the fit kernel = number of strided partial sums
constexpr int ICP_SRC = 128;      // source points per CTA of the search kernel
constexpr int ICP_TGT = 2048;     // targets per CTA of the search kernel

enum { ICP_NOT_CONVERGED = 0, ICP_ITERATIONS = 1, ICP_TRANSFORM = 2, ICP_ABS_MSE = 3, ICP_REL_MSE = 4, ICP_NO_CORRESPONDENCES = 5 };

// nearest target of every source point: CTA = 128 sources x a slice of the targets staged through shared memory,
// the slices meet in a packed atomicMin (squared distance bits << 32 | index: lowest index wins ties)
__global__ void __launch_bounds__(ICP_SRC)
icp_nn_kernel(const float4* __restrict__ cur, unsigned ns, const float4* __restrict__ tgt, unsigned nt, unsigned long long* __restrict__ keys,
              const IcpState* __restrict__ st) {
    if (st->done) return;
    __shared__ float4 tile[256];
    const unsigned i = blockIdx.x * ICP_SRC + threadIdx.x;
    const float4 p = (i < ns) ? cur[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    const unsigned t0 = blockIdx.y * ICP_TGT, t1 = min(nt, t0 + ICP_TGT);
    unsigned long long best = ~0ull;
    for (unsigned base = t0; base < t1; base += 256) {
        __syncthreads();
        for (unsigned k = threadIdx.x; k < 256; k += ICP_SRC) tile[k] = (base + k < t1) ? tgt[base + k] : make_float4(0.f, 0.f, 0.f, 0.f);
        __syncthreads();
        const unsigned m = min(256u, t1 - base);
        for (unsigned k = 0; k < m; ++k) {
            const float4 q = tile[k];
            const float dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z;
            const float d = (dx * dx + dy * dy) + dz * dz;
            const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (base + k);
            if (d == d && key < best) best = key;   // NaN distances never match
        }
    }
    if (i < ns && best != ~0ull) atomicMin(keys + i, best);
}

template <typename T>
__device__ __forceinline__ T block_sum(T v, T* sh) {
    const int t = threadIdx.x;
    __syncthreads();
    sh[t] = v;
    __syncthreads();
    for (int s = ICP_T / 2; s > 0; s >>= 1) {
        if (t < s) sh[t] = sh[t] + sh[t + s];
        __syncthreads();
    }
    return sh[0];
}

// N sums in one pass of the halving tree: each value is reduced exactly as block_sum reduces it.  sh: N * ICP_T floats
template <int N>
__device__ __forceinline__ void block_sum_n(float (&v)[N], float* sh) {
    const int t = threadIdx.x;
    __syncthreads();
    for (int e = 0; e < N; ++e) sh[e * ICP_T + t] = v[e];
    __syncthreads();
    for (int s = ICP_T / 2; s > 0; s >>= 1) {
        if (t < s)
            for (int e = 0; e < N; ++e) sh[e * ICP_T + t] = sh[e * ICP_T + t] + sh[e * ICP_T + t + s];
        __syncthreads();
    }
    for (int e = 0; e < N; ++e) v[e] = sh[e * ICP_T];
}

// one CTA: Umeyama over the correspondences, move the source, compose, test convergence, re-arm the keys
__global__ void __launch_bounds__(ICP_T)
icp_fit_kernel(float4* __restrict__ cur, unsigned ns, const float4* __restrict__ tgt, unsigned long long* __restrict__ keys, IcpState* __restrict__ st,
               int max_iterations) {
    if (st->done) return;
    __shared__ float shf[11 * ICP_T];
    __shared__ double shd[ICP_T];
    __shared__ float Rt[16];
    __shared__ int s_stop;
    const int t = threadIdx.x;
    // correspondences: every source point with a finite nearest neighbour
    float cnt_f = 0.f;
    for (unsigned i = t; i < ns; i += ICP_T) cnt_f += (keys[i] != ~0ull) ? 1.f : 0.f;
    const unsigned n = (unsigned)block_sum(cnt_f, shf);
    if (n < 3) {  // min_number_correspondences_
        if (t == 0) { st->state = ICP_NO_CORRESPONDENCES; st->done = 1; }
        return;
    }
    const float one_over_n = 1.0f / (float)n;
    // the centroids, and sum |p|_1, sum |q|_1 for the rank-0 noise floor
    float sm[3], dm[3], abs_pq[2];
    {
        float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (unsigned i = t; i < ns; i += ICP_T) {
            const unsigned long long k = keys[i];
            if (k == ~0ull) continue;
            const float4 p = cur[i], q = tgt[(unsigned)k];
            a[0] += p.x; a[1] += p.y; a[2] += p.z; a[3] += q.x; a[4] += q.y; a[5] += q.z;
            a[6] += (fabsf(p.x) + fabsf(p.y)) + fabsf(p.z); a[7] += (fabsf(q.x) + fabsf(q.y)) + fabsf(q.z);
        }
        block_sum_n(a, shf);
        for (int c = 0; c < 3; ++c) { sm[c] = a[c] * one_over_n; dm[c] = a[3 + c] * one_over_n; }
        abs_pq[0] = a[6]; abs_pq[1] = a[7];
    }
    // the cross-covariance, and sum |s|_1, sum |d|_1 of the centred points
    float sigma[9], abs_sd[2];
    {
        float a[11] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (unsigned i = t; i < ns; i += ICP_T) {
            const unsigned long long k = keys[i];
            if (k == ~0ull) continue;
            const float4 p = cur[i], q = tgt[(unsigned)k];
            const float s[3] = {p.x - sm[0], p.y - sm[1], p.z - sm[2]}, d[3] = {q.x - dm[0], q.y - dm[1], q.z - dm[2]};
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) a[3 * r + c] += d[r] * s[c];
            a[9] += (fabsf(s[0]) + fabsf(s[1])) + fabsf(s[2]); a[10] += (fabsf(d[0]) + fabsf(d[1])) + fabsf(d[2]);
        }
        block_sum_n(a, shf);
        for (int e = 0; e < 9; ++e) sigma[e] = one_over_n * a[e];
        abs_sd[0] = a[9]; abs_sd[1] = a[10];
    }
    double mse_sum = 0.0;
    for (unsigned i = t; i < ns; i += ICP_T) {
        const unsigned long long k = keys[i];
        if (k != ~0ull) mse_sum += (double)__uint_as_float((unsigned)(k >> 32));
    }
    mse_sum = block_sum(mse_sum, shd);
    if (t == 0) {
        double sg[9], U[9], sv[3], V[9];
        for (int e = 0; e < 9; ++e) sg[e] = (double)sigma[e];
        svd3_hestenes(sg, U, sv, V);
        const double det = sg[0] * (sg[4] * sg[8] - sg[5] * sg[7]) - sg[1] * (sg[3] * sg[8] - sg[5] * sg[6]) + sg[2] * (sg[3] * sg[7] - sg[4] * sg[6]);
        // rank = number of singular values not much smaller than sv[0] (isMuchSmallerThan, float precision 1e-5); rank 0
        // when sv[0] is within the fp32 rounding noise of Sigma (rigid_noise_floor)
        const double floor0 = rigid_noise_floor((double)abs_pq[0], (double)abs_pq[1], (double)abs_sd[0], (double)abs_sd[1], (double)n,
                                                (double)((n + ICP_T - 1) / ICP_T + 8), 5.9604644775390625e-08);
        double Rd[9];
        const bool rank0 = sv[0] <= floor0;
        if (rank0 || sv[1] <= sv[0] * 1e-5) rigid_rotation_rank01(U, V, rank0, Rd);   // rank <= 1: see rigid_math.cuh (DESIGN 3.5)
        else {
            double sgn = 1.0;
            if (sv[2] <= sv[0] * 1e-5) {  // rank 2: right-handed completion, R = U V^T
                U[2] = U[3] * U[7] - U[6] * U[4]; U[5] = U[6] * U[1] - U[0] * U[7]; U[8] = U[0] * U[4] - U[3] * U[1];
                V[2] = V[3] * V[7] - V[6] * V[4]; V[5] = V[6] * V[1] - V[0] * V[7]; V[8] = V[0] * V[4] - V[3] * V[1];
            } else if (det < 0) sgn = -1.0;   // rank 3: S(2) = -1
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) Rd[3 * r + c] = (U[3 * r] * V[3 * c] + U[3 * r + 1] * V[3 * c + 1]) + sgn * (U[3 * r + 2] * V[3 * c + 2]);
        }
        float R[9];
        for (int e = 0; e < 9; ++e) R[e] = (float)Rd[e];
        for (int r = 0; r < 3; ++r) {
            Rt[4 * r] = R[3 * r]; Rt[4 * r + 1] = R[3 * r + 1]; Rt[4 * r + 2] = R[3 * r + 2];
            Rt[4 * r + 3] = dm[r] - ((R[3 * r] * sm[0] + R[3 * r + 1] * sm[1]) + R[3 * r + 2] * sm[2]);
        }
        Rt[12] = 0.f; Rt[13] = 0.f; Rt[14] = 0.f; Rt[15] = 1.f;
        // final_transformation_ = transformation_ * final_transformation_
        float F[16];
        for (int r = 0; r < 4; ++r)
            for (int c = 0; c < 4; ++c)
                F[4 * r + c] = ((Rt[4 * r] * st->final_T[c] + Rt[4 * r + 1] * st->final_T[4 + c]) + Rt[4 * r + 2] * st->final_T[8 + c]) + Rt[4 * r + 3] * st->final_T[12 + c];
        for (int e = 0; e < 16; ++e) st->final_T[e] = F[e];
        const int it = ++st->iterations;
        // DefaultConvergenceCriteria::hasConverged
        int stop = 0, state = ICP_NOT_CONVERGED;
        const double mse = mse_sum / (double)n;
        st->mse = mse;
        if (it >= max_iterations) { stop = 1; state = ICP_ITERATIONS; }
        else {
            const double cos_angle = 0.5 * (double)(((Rt[0] + Rt[5]) + Rt[10]) - 1.0f);
            const double translation_sqr = (double)((Rt[3] * Rt[3] + Rt[7] * Rt[7]) + Rt[11] * Rt[11]);
            if (cos_angle >= 1.0 && translation_sqr <= 0.0) { stop = 1; state = ICP_TRANSFORM; }
            else if (fabs(mse - st->prev_mse) < 1e-12) { stop = 1; state = ICP_ABS_MSE; }
            else st->prev_mse = mse;   // the relative test (threshold -DBL_MAX) can never fire
        }
        st->state = state;
        s_stop = stop;
    }
    __syncthreads();
    // transformCloud(*input_transformed, *input_transformed, transformation_)
    for (unsigned i = t; i < ns; i += ICP_T) {
        const float4 p = cur[i];
        float4 o;
        o.x = ((Rt[0] * p.x + Rt[1] * p.y) + Rt[2] * p.z) + Rt[3];
        o.y = ((Rt[4] * p.x + Rt[5] * p.y) + Rt[6] * p.z) + Rt[7];
        o.z = ((Rt[8] * p.x + Rt[9] * p.y) + Rt[10] * p.z) + Rt[11];
        o.w = 0.f;
        cur[i] = o;
        keys[i] = ~0ull;
    }
    if (t == 0 && s_stop) st->done = 1;
}

// host points in, host results out: the points, the pre-transform and both counts are uploaded and icp_run_dev runs on the
// true counts (no padding); one synchronisation at the end
int icp_run(Ctx* c, const float* src_xyz, size_t n_src, const float* tgt_xyz, size_t n_tgt, const float* pre4x4, int max_iterations,
            float* final4x4_out, int* iterations_out, int* state_out, double* mse_out) {
    const float ident[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    IcpState h = {};
    if (n_src && n_tgt && max_iterations > 0) {
        const size_t bytes = 12 * (n_src + n_tgt) + 16 * (n_src + n_tgt) + 8 * n_src + sizeof(IcpState) + 64 + 8 + 256 * 8;
        BSHOT_TRY(scratch_reserve(c, 2, bytes));
        char* base = (char*)c->d_pre[2];
        size_t off = 0;
        auto take = [&](size_t b) { char* r = base + off; off += (b + 255) & ~(size_t)255; return r; };
        float* d_src = (float*)take(12 * n_src); float* d_tgt3 = (float*)take(12 * n_tgt);
        float4* d_cur = (float4*)take(16 * n_src); float4* d_tgt = (float4*)take(16 * n_tgt);
        unsigned long long* d_keys = (unsigned long long*)take(8 * n_src);
        IcpState* d_st = (IcpState*)take(sizeof(IcpState)); float* d_pre = (float*)take(64);
        unsigned* d_counts = (unsigned*)take(8);
        const unsigned counts[2] = {(unsigned)n_src, (unsigned)n_tgt};
        BSHOT_CUDA_TRY(cudaMemcpyAsync(d_src, src_xyz, 12 * n_src, cudaMemcpyHostToDevice, c->stream));
        BSHOT_CUDA_TRY(cudaMemcpyAsync(d_tgt3, tgt_xyz, 12 * n_tgt, cudaMemcpyHostToDevice, c->stream));
        BSHOT_CUDA_TRY(cudaMemcpyAsync(d_pre, pre4x4 ? pre4x4 : ident, 64, cudaMemcpyHostToDevice, c->stream));
        BSHOT_CUDA_TRY(cudaMemcpyAsync(d_counts, counts, sizeof(counts), cudaMemcpyHostToDevice, c->stream));
        BSHOT_TRY(icp_run_dev(c, d_src, 3, reinterpret_cast<const int*>(d_counts), n_src, d_tgt3, 3, d_counts + 1, n_tgt, d_pre, max_iterations, nullptr, d_cur,
                              d_tgt, d_keys, d_st));
        BSHOT_CUDA_TRY(cudaMemcpyAsync(&h, d_st, sizeof(IcpState), cudaMemcpyDeviceToHost, c->stream));
        BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    } else {
        for (int e = 0; e < 16; ++e) h.final_T[e] = ident[e];
        h.state = ICP_NO_CORRESPONDENCES;
    }
    if (final4x4_out) for (int e = 0; e < 16; ++e) final4x4_out[e] = h.final_T[e];
    if (iterations_out) *iterations_out = h.iterations;
    if (state_out) *state_out = h.state;
    if (mse_out) *mse_out = h.mse;
    return BSHOT_OK;
}

// ---- device inputs (the odometry step; icp_run on its uploads) -----------------------------------------------------------------
// Sources moved by the device-side pre-transform (pcl::transformPointCloud(cb.cloud1_keypoints, icp_cloud, T_est),
// src/lidar_odometry.cpp:284) and targets are point arrays of src_stride / tgt_stride floats (3: packed xyz, 4: float4).
// Both counts stay on the device: the kernels above run on the host-known capacities, and the slots past the true counts
// hold NaN, which never becomes a correspondence (icp_nn_kernel tests d == d), so icp_fit_kernel's 256 strided partial sums
// -- and hence every bit of the result -- depend only on the true points.  A set *d_skip makes every launch a no-op.
__global__ void icp_init_dev_kernel(const float* __restrict__ src, int src_stride, const int* __restrict__ d_ns, unsigned ns_cap, const float* __restrict__ tgt,
                                    int tgt_stride, const unsigned* __restrict__ d_nt, unsigned nt_cap, const float* __restrict__ pre, const int* __restrict__ skip,
                                    float4* __restrict__ cur, float4* __restrict__ tgt_out, unsigned long long* __restrict__ keys, IcpState* __restrict__ st) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned ns = min((unsigned)max(*d_ns, 0), ns_cap), nt = min(*d_nt, nt_cap);
    const float nan = __int_as_float(0x7fc00000);
    if (i < ns_cap) {
        float4 o = make_float4(nan, nan, nan, 0.f);
        if (i < ns) {
            const float* p = src + (size_t)src_stride * i;
            const float x = p[0], y = p[1], z = p[2];
            o.x = ((pre[0] * x + pre[1] * y) + pre[2] * z) + pre[3];
            o.y = ((pre[4] * x + pre[5] * y) + pre[6] * z) + pre[7];
            o.z = ((pre[8] * x + pre[9] * y) + pre[10] * z) + pre[11];
        }
        cur[i] = o;
        keys[i] = ~0ull;
    }
    if (i < nt_cap) {
        const float* q = tgt + (size_t)tgt_stride * i;
        tgt_out[i] = (i < nt) ? make_float4(q[0], q[1], q[2], 0.f) : make_float4(nan, nan, nan, 0.f);
    }
    if (i == 0) {
        for (int e = 0; e < 16; ++e) st->final_T[e] = (e % 5 == 0) ? 1.0f : 0.0f;
        st->prev_mse = 1.7976931348623157e308;
        st->mse = 0.0; st->iterations = 0; st->state = ICP_NOT_CONVERGED; st->pad = 0;
        st->done = (skip && *skip) ? 1 : 0;
        if (ns == 0 || nt == 0) { st->state = ICP_NO_CORRESPONDENCES; st->done = 1; }
    }
}

int icp_run_dev(Ctx* c, const float* d_src, int src_stride, const int* d_ns, size_t ns_cap, const float* d_tgt, int tgt_stride, const unsigned* d_nt,
                size_t nt_cap, const float* d_pre, int max_iterations, const int* d_skip, float4* d_cur, float4* d_tgt_buf, unsigned long long* d_keys,
                IcpState* d_st) {
    const unsigned ns = (unsigned)ns_cap, nt = (unsigned)nt_cap, nmax = std::max(std::max(ns, nt), 1u);
    icp_init_dev_kernel<<<(nmax + 255) / 256, 256, 0, c->stream>>>(d_src, src_stride, d_ns, ns, d_tgt, tgt_stride, d_nt, nt, d_pre, d_skip, d_cur, d_tgt_buf,
                                                                   d_keys, d_st);
    count_launch(c);
    if (ns && nt) {
        const dim3 grid((ns + ICP_SRC - 1) / ICP_SRC, (nt + ICP_TGT - 1) / ICP_TGT);
        for (int it = 0; it < max_iterations; ++it) {
            icp_nn_kernel<<<grid, ICP_SRC, 0, c->stream>>>(d_cur, ns, d_tgt_buf, nt, d_keys, d_st);
            icp_fit_kernel<<<1, ICP_T, 0, c->stream>>>(d_cur, ns, d_tgt_buf, d_keys, d_st, max_iterations);
        }
        count_launch(c, 2 * max_iterations);
    }
    return check_launch("device ICP kernels");
}

}  // namespace bshot
