// ransac.cu -- RANSAC correspondence rejection on the device (SURVEY 8f "next" #1).
//
// Replaces the pcl::registration::CorrespondenceRejectorSampleConsensus call of LidarOdometry::featureMatching
// (src/lidar_odometry.cpp:251-261: 2000 iterations, inlier threshold 1500 mm) -- i.e. PCL 1.8's
// RandomSampleConsensus over SampleConsensusModelRegistration:
//   * sample sequence: mt19937 seeded 12345, rnd() = mt() / 2 (boost::uniform_int<>(0, INT_MAX)), drawIndexSample's
//     progressive shuffle of the index list, samples rejected while two of the three source points are closer than
//     sample_dist_thresh (mean of the square roots of the eigenvalues of the source covariance, squared) -- up to 1000 tries;
//   * model: Umeyama without scaling on the three pairs in double (SVD of the 3x3 cross-covariance, proper rotation),
//     coefficients cast to float;
//   * score: number of correspondences with |T * src - tgt|^2 < threshold^2 (float transform, float norm);
//   * adaptive stop: k = log(1 - 0.99) / log(1 - w^3) re-evaluated at every new best, first best wins ties;
//   * result: the correspondences within the threshold of the best model, in their original order, and that model.
// The sample sequence does not depend on the scores, so it is generated up front (on the host for host inputs, a few
// microseconds; on the device for device inputs), ALL hypotheses are scored in parallel (one warp each), and the adaptive
// loop is replayed over the scores exactly as PCL runs it.  Both entry points then share one tail: scoring, the adaptive
// stop (ransac_adaptive_stop, on the host for host inputs), the inlier flags and the in-order compaction.  This file is compiled with -fmad=false: the double-precision Jacobi SVD
// then uses only IEEE +, -, *, /, sqrt and is bit-identical to the oracle's restatement (orc_ransac).
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "rigid_math.cuh"
#include "stages.h"

namespace bshot {

// Umeyama without scaling for three point pairs (pcl::umeyama / Eigen::umeyama, with_scaling = false), double in, float
// 4x4 row-major out.  rank 2 (three non-collinear points): the third columns of U and V are completed as cross products,
// so both bases are right handed and R = U V^T is the proper rotation that Eq. (40)-(43) select.
__host__ __device__ inline void umeyama3(const double src[3][3], const double dst[3][3], float T[16]) {
    double sm[3], dm[3];
    for (int c = 0; c < 3; ++c) { sm[c] = (src[0][c] + src[1][c] + src[2][c]) / 3.0; dm[c] = (dst[0][c] + dst[1][c] + dst[2][c]) / 3.0; }
    double sigma[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
            double acc = 0.0;
            for (int i = 0; i < 3; ++i) acc += (dst[i][r] - dm[r]) * (src[i][c] - sm[c]);
            sigma[3 * r + c] = acc / 3.0;
        }
    double U[9], s[3], V[9];
    svd3_hestenes(sigma, U, s, V);
    // complete the last columns to right-handed bases (rank <= 2 for three points)
    U[2] = U[3] * U[7] - U[6] * U[4]; U[5] = U[6] * U[1] - U[0] * U[7]; U[8] = U[0] * U[4] - U[3] * U[1];
    V[2] = V[3] * V[7] - V[6] * V[4]; V[5] = V[6] * V[1] - V[0] * V[7]; V[8] = V[0] * V[4] - V[3] * V[1];
    double R[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[3 * r + c] = (U[3 * r] * V[3 * c] + U[3 * r + 1] * V[3 * c + 1]) + U[3 * r + 2] * V[3 * c + 2];
    for (int r = 0; r < 3; ++r) {
        const double t = dm[r] - ((R[3 * r] * sm[0] + R[3 * r + 1] * sm[1]) + R[3 * r + 2] * sm[2]);
        T[4 * r] = (float)R[3 * r]; T[4 * r + 1] = (float)R[3 * r + 1]; T[4 * r + 2] = (float)R[3 * r + 2]; T[4 * r + 3] = (float)t;
    }
    T[12] = 0.0f; T[13] = 0.0f; T[14] = 0.0f; T[15] = 1.0f;
}

// |T * src - tgt|^2 in float: Eigen's 4x4 * vec4 (columns scaled and added left to right), then squaredNorm
__host__ __device__ inline float transfer_sqd(const float T[16], float sx, float sy, float sz, float tx, float ty, float tz) {
    const float px = ((T[0] * sx + T[1] * sy) + T[2] * sz) + T[3];
    const float py = ((T[4] * sx + T[5] * sy) + T[6] * sz) + T[7];
    const float pz = ((T[8] * sx + T[9] * sy) + T[10] * sz) + T[11];
    const float dx = px - tx, dy = py - ty, dz = pz - tz;
    return (dx * dx + dy * dy) + dz * dz;
}

// ---- the tail both entry points run after their sampler -----------------------------------------------------------------
// score every hypothesis -> adaptive stop -> inlier flags of the best model -> in-order compaction.  The state lives on the
// device: n correspondences, n_valid hypotheses drawn, and the adaptive stop's best hypothesis (-1: none) and iterations.
struct RansacDevState {
    double sdt;
    int n, n_valid, best, iterations;
};

// RandomSampleConsensus::computeModel replayed over the scores: the host call runs it on the host after reading the counts
// back, the device call on one device thread
__host__ __device__ inline void ransac_adaptive_stop(RansacDevState* st, const int* counts, int max_iterations) {
    int iterations = 0, best = -1, n_best = -2147483647;
    double k = 1.0;
    const double log_probability = log(1.0 - 0.99), one_over_indices = 1.0 / (double)st->n;
    while ((double)iterations < k) {
        if (iterations >= st->n_valid) break;  // no sample could be drawn: PCL breaks out
        const int cnt = counts[iterations];
        if (cnt > n_best) {
            n_best = cnt;
            best = iterations;
            const double w = (double)n_best * one_over_indices;
            double p_no_outliers = 1.0 - pow(w, 3.0);
            p_no_outliers = fmax(2.220446049250313e-16, p_no_outliers);
            p_no_outliers = fmin(1.0 - 2.220446049250313e-16, p_no_outliers);
            k = log_probability / log(p_no_outliers);
        }
        ++iterations;
        if (iterations > max_iterations) break;
    }
    st->best = best;
    st->iterations = iterations;
}

// one warp per hypothesis: model from its three pairs, inlier count over all correspondences
__global__ void __launch_bounds__(128)
ransac_score_dev_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, const RansacDevState* __restrict__ st, const int* __restrict__ samples,
                        double thresh2, float* __restrict__ models, int* __restrict__ counts) {
    const unsigned lane = threadIdx.x & 31, h = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (st->n < 3 || h >= (unsigned)st->n_valid) return;
    const unsigned n = (unsigned)st->n;
    float T[16];
    {
        double s[3][3], d[3][3];
        for (int i = 0; i < 3; ++i) {
            const int k = samples[3 * h + i];
            const float4 a = src[k], b = tgt[k];
            s[i][0] = a.x; s[i][1] = a.y; s[i][2] = a.z;
            d[i][0] = b.x; d[i][1] = b.y; d[i][2] = b.z;
        }
        umeyama3(s, d, T);  // every lane computes the same model (no divergence, no broadcast needed)
    }
    int cnt = 0;
    for (unsigned i = lane; i < n; i += 32) {
        const float4 a = src[i], b = tgt[i];
        if ((double)transfer_sqd(T, a.x, a.y, a.z, b.x, b.y, b.z) < thresh2) ++cnt;
    }
    cnt = warp_sum(cnt);
    if (lane == 0) counts[h] = cnt;
    if (lane < 16) models[16 * h + lane] = T[lane];
}

__global__ void ransac_select_dev_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, const RansacDevState* __restrict__ st,
                                         const float* __restrict__ models, double thresh2, unsigned char* __restrict__ inlier) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (st->best < 0 || i >= (unsigned)st->n) return;
    const float* model = models + 16 * (size_t)st->best;
    float T[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) T[k] = model[k];
    const float4 a = src[i], b = tgt[i];
    inlier[i] = ((double)transfer_sqd(T, a.x, a.y, a.z, b.x, b.y, b.z) < thresh2) ? 1 : 0;
}

// one CTA: the inliers of the best model in their original order, or (fewer than 3 correspondences / no hypothesis / fewer
// than 3 inliers) every correspondence with the identity -- PCL's behaviour
__global__ void __launch_bounds__(1024)
ransac_finish_kernel(const RansacDevState* __restrict__ st, const int* __restrict__ pairs, int stride, const unsigned char* __restrict__ inlier,
                     const float* __restrict__ models, int* __restrict__ pairs_out, int* __restrict__ n_out, float* __restrict__ T_out,
                     int* __restrict__ iterations_out) {
    __shared__ unsigned ws[32];
    __shared__ unsigned carry;
    const unsigned tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned n = (unsigned)max(st->n, 0);
    const int best = st->best;
    bool keep_all = n < 3 || best < 0;
    if (tid == 0) carry = 0;
    __syncthreads();
    if (!keep_all) {
        unsigned c = 0;
        for (unsigned i = tid; i < n; i += 1024) c += inlier[i];
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0) atomicAdd(&carry, c);
        __syncthreads();
        keep_all = carry < 3;
        __syncthreads();
        if (tid == 0) carry = 0;
        __syncthreads();
    }
    for (unsigned base = 0; base < n; base += 1024) {
        const unsigned i = base + tid;
        const unsigned f = (i < n) ? (keep_all ? 1u : (unsigned)inlier[i]) : 0u;
        unsigned inc = f;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned up = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= (unsigned)o) inc += up;
        }
        if (lane == 31) ws[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            const unsigned v = ws[lane];
            unsigned winc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned up = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= (unsigned)o) winc += up;
            }
            ws[lane] = winc - v;
        }
        __syncthreads();
        const unsigned excl = carry + ws[wid] + inc - f;
        if (f) { pairs_out[2 * excl] = pairs[(size_t)stride * i]; pairs_out[2 * excl + 1] = pairs[(size_t)stride * i + 1]; }
        __syncthreads();
        if (tid == 1023) carry = excl + f;
        __syncthreads();
    }
    if (tid < 16) T_out[tid] = keep_all ? ((tid % 5 == 0) ? 1.0f : 0.0f) : models[16 * (size_t)best + tid];
    if (tid == 0) { *n_out = (int)carry; *iterations_out = keep_all ? 0 : st->iterations; }
}

// scratch of both entry points: correspondence sources | targets (cap each) in d_gather; the state, samples, models, counts
// and inlier flags in d_partial, then (16-byte aligned) `extra` bytes of the entry point's own
struct RansacScratch {
    float4 *s4, *t4;
    RansacDevState* st;
    int* samples;
    float* models;
    int* counts;
    unsigned char* inlier;
    char* extra;
};

static int ransac_scratch(Ctx* c, const char* who, int max_iterations, size_t cap, size_t extra, RansacScratch* r) {
    const size_t n_hyp = (size_t)max_iterations + 1;
    char* base = reinterpret_cast<char*>(c->d_partial);
    r->s4 = reinterpret_cast<float4*>(c->d_gather);
    r->t4 = r->s4 + cap;
    r->st = reinterpret_cast<RansacDevState*>(base);
    r->samples = reinterpret_cast<int*>(base + 64);
    r->models = reinterpret_cast<float*>(r->samples + 3 * n_hyp);
    r->counts = reinterpret_cast<int*>(r->models + 16 * n_hyp);
    r->inlier = reinterpret_cast<unsigned char*>(r->counts + n_hyp);
    r->extra = base + ((64 + (3 + 16 + 1) * n_hyp * 4 + cap + 15) & ~(size_t)15);
    if ((size_t)(r->extra - base) + extra > c->partial_cap * 8) { set_error("%s: scratch too small for %d iterations", who, max_iterations); return BSHOT_E_CAPACITY; }
    return BSHOT_OK;
}

// ---- host: PCL's sample sequence ------------------------------------------------------------------------------------------
namespace {
struct Mt19937 {  // boost::mt19937 / std::mt19937 recurrence
    uint32_t s[624];
    int idx;
    explicit Mt19937(uint32_t seed) {
        s[0] = seed;
        for (int i = 1; i < 624; ++i) s[i] = 1812433253u * (s[i - 1] ^ (s[i - 1] >> 30)) + (uint32_t)i;
        idx = 624;
    }
    uint32_t next() {
        if (idx >= 624) {
            for (int i = 0; i < 624; ++i) {
                const uint32_t y = (s[i] & 0x80000000u) | (s[(i + 1) % 624] & 0x7FFFFFFFu);
                s[i] = s[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908B0DFu : 0u);
            }
            idx = 0;
        }
        uint32_t y = s[idx++];
        y ^= y >> 11; y ^= (y << 7) & 0x9D2C5680u; y ^= (y << 15) & 0xEFC60000u; y ^= y >> 18;
        return y;
    }
};

}  // namespace

// sample_dist_thresh from the float sums {xx, xy, xz, yy, yz, zz, x, y, z} of n sources (host and device share it)
__host__ __device__ inline double sample_dist_from_sums(float a[9], size_t n) {
    const float fn = (float)n;
    for (int k = 0; k < 9; ++k) a[k] /= fn;
    const double cov[9] = {(double)(a[0] - a[6] * a[6]), (double)(a[1] - a[6] * a[7]), (double)(a[2] - a[6] * a[8]),
                           (double)(a[1] - a[6] * a[7]), (double)(a[3] - a[7] * a[7]), (double)(a[4] - a[7] * a[8]),
                           (double)(a[2] - a[6] * a[8]), (double)(a[4] - a[7] * a[8]), (double)(a[5] - a[8] * a[8])};
    double U[9], w[3], V[9];
    svd3_hestenes(cov, U, w, V);  // symmetric positive semi-definite: singular values = eigenvalues
    const float e0 = (float)w[0], e1 = (float)w[1], e2 = (float)w[2];
    double t = (double)((sqrtf(fmaxf(e0, 0.0f)) + sqrtf(fmaxf(e1, 0.0f))) + sqrtf(fmaxf(e2, 0.0f))) / 3.0;
    return t * t;
}

// sample_dist_thresh of SampleConsensusModelRegistration::computeSampleDistanceThreshold over the correspondence sources
static double sample_dist_threshold(const float* src4, size_t n) {
    // computeMeanAndCovarianceMatrix: single pass, float accumulators, index order
    float a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (size_t i = 0; i < n; ++i) {
        const float x = src4[4 * i], y = src4[4 * i + 1], z = src4[4 * i + 2];
        a[0] += x * x; a[1] += x * y; a[2] += x * z; a[3] += y * y; a[4] += y * z; a[5] += z * z; a[6] += x; a[7] += y; a[8] += z;
    }
    return sample_dist_from_sums(a, n);
}

int ransac_run(Ctx* c, const float* src_xyz, const float* tgt_xyz, const int* pairs, size_t n_pairs, int max_iterations, double threshold,
               int* inlier_pairs_out, int* n_inliers_out, float* transform_out, int* iterations_out) {
    if (n_inliers_out) *n_inliers_out = 0;
    auto keep_all = [&]() {  // PCL: computeModel failed -> all correspondences stay, identity
        if (inlier_pairs_out) memcpy(inlier_pairs_out, pairs, sizeof(int) * 2 * n_pairs);
        if (n_inliers_out) *n_inliers_out = (int)n_pairs;
        if (transform_out) for (int k = 0; k < 16; ++k) transform_out[k] = (k % 5 == 0) ? 1.0f : 0.0f;
        if (iterations_out) *iterations_out = 0;
        return BSHOT_OK;
    };
    if (n_pairs < 3) return keep_all();
    if (n_pairs > c->max_kp) { set_error("bshot_ransac: %zu correspondences > max_keypoints %zu", n_pairs, c->max_kp); return BSHOT_E_CAPACITY; }
    if (max_iterations < 1 || max_iterations > 100000) { set_error("bshot_ransac: bad max_iterations"); return BSHOT_E_INVALID; }
    const size_t n = n_pairs, n_hyp = (size_t)max_iterations + 1;
    // correspondence sources / targets in correspondence order (what indices_ / indices_tgt_ address)
    std::vector<float> s4(4 * n), t4(4 * n);
    for (size_t i = 0; i < n; ++i) {
        const int q = pairs[2 * i], m = pairs[2 * i + 1];
        for (int k = 0; k < 3; ++k) { s4[4 * i + k] = src_xyz[3 * (size_t)q + k]; t4[4 * i + k] = tgt_xyz[3 * (size_t)m + k]; }
        s4[4 * i + 3] = t4[4 * i + 3] = 1.0f;
    }
    // ---- PCL's sample sequence for iterations 0 .. max_iterations (independent of the scores) -------------------------------
    const double sdt = sample_dist_threshold(s4.data(), n);
    std::vector<int> shuffled(n), samples(3 * n_hyp);
    for (size_t i = 0; i < n; ++i) shuffled[i] = (int)i;
    Mt19937 rng(12345u);
    size_t n_valid = n_hyp;
    for (size_t h = 0; h < n_hyp; ++h) {
        bool good = false;
        for (int tries = 0; tries < 1000 && !good; ++tries) {  // max_sample_checks_
            for (size_t i = 0; i < 3; ++i) std::swap(shuffled[i], shuffled[i + ((rng.next() >> 1) % (n - i))]);
            auto d2 = [&](int a, int b) {
                const float dx = s4[4 * b] - s4[4 * a], dy = s4[4 * b + 1] - s4[4 * a + 1], dz = s4[4 * b + 2] - s4[4 * a + 2];
                return (double)(dx * dx + dy * dy + dz * dz);
            };
            good = d2(shuffled[0], shuffled[1]) > sdt && d2(shuffled[0], shuffled[2]) > sdt && d2(shuffled[1], shuffled[2]) > sdt;
        }
        if (!good) { n_valid = h; break; }  // "Could not select sample points": PCL stops the loop here
        samples[3 * h] = shuffled[0]; samples[3 * h + 1] = shuffled[1]; samples[3 * h + 2] = shuffled[2];
    }
    if (n_valid == 0) return keep_all();
    // ---- the shared tail on the uploaded correspondences and samples -----------------------------------------------------------
    // own scratch: results {n_inliers, iterations, T[16]} | input pairs (2n ints) | output pairs (2n ints)
    RansacScratch r;
    BSHOT_TRY(ransac_scratch(c, "bshot_ransac", max_iterations, n, 4 * (18 + 4 * n), &r));
    int* d_res = reinterpret_cast<int*>(r.extra);
    int* d_pairs_in = d_res + 18;
    int* d_pairs_out = d_pairs_in + 2 * n;
    RansacDevState st = {sdt, (int)n, (int)n_valid, -1, 0};
    BSHOT_CUDA_TRY(cudaMemcpyAsync(r.s4, s4.data(), 16 * n, cudaMemcpyHostToDevice, c->stream));
    BSHOT_CUDA_TRY(cudaMemcpyAsync(r.t4, t4.data(), 16 * n, cudaMemcpyHostToDevice, c->stream));
    BSHOT_CUDA_TRY(cudaMemcpyAsync(d_pairs_in, pairs, sizeof(int) * 2 * n, cudaMemcpyHostToDevice, c->stream));
    BSHOT_CUDA_TRY(cudaMemcpyAsync(r.samples, samples.data(), sizeof(int) * 3 * n_valid, cudaMemcpyHostToDevice, c->stream));
    BSHOT_CUDA_TRY(cudaMemcpyAsync(r.st, &st, sizeof(st), cudaMemcpyHostToDevice, c->stream));
    const double thresh2 = threshold * threshold;
    ransac_score_dev_kernel<<<(unsigned)((n_valid * 32 + 127) / 128), 128, 0, c->stream>>>(r.s4, r.t4, r.st, r.samples, thresh2, r.models, r.counts);
    count_launch(c);
    BSHOT_TRY(check_launch("ransac_score_dev_kernel"));
    std::vector<int> counts(n_valid);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(counts.data(), r.counts, sizeof(int) * n_valid, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    ransac_adaptive_stop(&st, counts.data(), max_iterations);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(r.st, &st, sizeof(st), cudaMemcpyHostToDevice, c->stream));
    ransac_select_dev_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(r.s4, r.t4, r.st, r.models, thresh2, r.inlier);
    ransac_finish_kernel<<<1, 1024, 0, c->stream>>>(r.st, d_pairs_in, 2, r.inlier, r.models, d_pairs_out, d_res, reinterpret_cast<float*>(d_res + 2), d_res + 1);
    count_launch(c, 2);
    BSHOT_TRY(check_launch("ransac_select_dev_kernel / ransac_finish_kernel"));
    int res[18];
    std::vector<int> kept(2 * n);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(res, d_res, sizeof(res), cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaMemcpyAsync(kept.data(), d_pairs_out, sizeof(int) * 2 * n, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (inlier_pairs_out) memcpy(inlier_pairs_out, kept.data(), sizeof(int) * 2 * (size_t)res[0]);
    if (n_inliers_out) *n_inliers_out = res[0];
    if (transform_out) memcpy(transform_out, res + 2, sizeof(float) * 16);
    if (iterations_out) *iterations_out = res[1];
    return BSHOT_OK;
}

// ---- device inputs: the whole of ransac_run without a host round trip (bshot_ransac_dev, the odometry step) ----------------
// The correspondence count stays on the device.  PCL's sample sequence is produced on the device in batches of 208 tries
// (= 624 draws, one mt19937 twist): the twist, the tempering and the moduli (mt() >> 1) % (n - j % 3) run in parallel, the
// swap chain (the only sequential part: draw j always swaps position j % 3) runs on one thread with positions 0..2 in
// registers, the distance tests of the 208 triples run in parallel, and one thread walks the test results in order, which
// makes a try a hypothesis, counts the tries of the current hypothesis and gives up after 1000 -- exactly the host loop, for
// any number of tries.  The tail after the sampler is the host call's.

constexpr int RS_TRIES = 208;           // tries per batch: 3 x 208 = 624 draws = one twist
constexpr int RS_THREADS = 256;

__global__ void ransac_gather_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, const int* __restrict__ pairs, int stride,
                                     const int* __restrict__ d_n, unsigned cap, const int* __restrict__ skip, float4* __restrict__ s_out,
                                     float4* __restrict__ t_out, RansacDevState* __restrict__ st) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned n = (skip && *skip) ? 0u : min((unsigned)max(*d_n, 0), cap);
    if (i == 0) { st->n = (int)n; st->n_valid = 0; st->best = -1; st->iterations = 0; }
    if (i >= n) return;
    const float4 a = src[pairs[(size_t)stride * i]], b = tgt[pairs[(size_t)stride * i + 1]];
    s_out[i] = make_float4(a.x, a.y, a.z, 1.0f);
    t_out[i] = make_float4(b.x, b.y, b.z, 1.0f);
}

__device__ __forceinline__ double rs_d2(const float4* __restrict__ s, int a, int b) {
    const float4 p = s[a], q = s[b];
    const float dx = q.x - p.x, dy = q.y - p.y, dz = q.z - p.z;
    return (double)(dx * dx + dy * dy + dz * dz);
}

// one CTA: sample_dist_thresh, then the sample sequence -> samples[3 * h ..], st->n_valid.  shuffled: n ints (shared memory
// when it fits, else global scratch)
__global__ void __launch_bounds__(RS_THREADS)
ransac_sample_kernel(const float4* __restrict__ s4, RansacDevState* __restrict__ st, unsigned n_hyp, int* __restrict__ samples, int* g_shuffled) {
    extern __shared__ int dyn_shuffled[];
    __shared__ uint32_t mt[624];
    __shared__ uint32_t mod[624];
    __shared__ int trip[RS_TRIES * 3];
    __shared__ unsigned char good[RS_TRIES];
    __shared__ double s_sdt;
    __shared__ int s_done;
    const int tid = threadIdx.x;
    const unsigned n = (unsigned)st->n;
    if (n < 3) return;   // everything is kept (finish kernel)
    int* sh = g_shuffled ? g_shuffled : dyn_shuffled;
    // computeMeanAndCovarianceMatrix: float sums in index order.  Warp 0 gathers 32 sources at a time and every lane replays
    // them in order, so the sequential chain never waits on a global load
    if (tid < 32) {
        float a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (unsigned base = 0; base < n; base += 32) {
            const float4 p = (base + tid < n) ? s4[base + tid] : make_float4(0.f, 0.f, 0.f, 0.f);
            const unsigned m = min(32u, n - base);
            for (unsigned j = 0; j < m; ++j) {
                const float x = __shfl_sync(0xffffffffu, p.x, j), y = __shfl_sync(0xffffffffu, p.y, j), z = __shfl_sync(0xffffffffu, p.z, j);
                a[0] += x * x; a[1] += x * y; a[2] += x * z; a[3] += y * y; a[4] += y * z; a[5] += z * z; a[6] += x; a[7] += y; a[8] += z;
            }
        }
        if (tid == 0) {
            s_sdt = sample_dist_from_sums(a, n);
            st->sdt = s_sdt;
        }
    }
    // mt19937 seeded 12345
    if (tid == 0) {
        mt[0] = 12345u;
        for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
        s_done = 0;
    }
    for (unsigned i = tid; i < n; i += RS_THREADS) sh[i] = (int)i;
    __syncthreads();
    const double sdt = s_sdt;
    int a0 = 0, a1 = 0, a2 = 0;                      // positions 0..2 of the shuffled list (thread 0)
    if (tid == 0) { a0 = sh[0]; a1 = sh[1]; a2 = sh[2]; }
    unsigned h = 0, tries = 0;                        // hypotheses found, tries of the current one (thread 0)
    while (true) {
        // twist in three dependency phases: [0, 227) reads old words only, [227, 454) reads the new [0, 227),
        // [454, 624) reads the new [227, 397) and (i = 623) the new word 0
        const int lo[3] = {0, 227, 454}, hi[3] = {227, 454, 624};
        for (int ph = 0; ph < 3; ++ph) {
            const int i = lo[ph] + tid;
            uint32_t v = 0;
            if (i < hi[ph]) {
                const uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7FFFFFFFu);
                v = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908B0DFu : 0u);
            }
            __syncthreads();
            if (i < hi[ph]) mt[i] = v;
            __syncthreads();
        }
        for (int j = tid; j < 624; j += RS_THREADS) {
            uint32_t y = mt[j];
            y ^= y >> 11; y ^= (y << 7) & 0x9D2C5680u; y ^= (y << 15) & 0xEFC60000u; y ^= y >> 18;
            mod[j] = (y >> 1) % (n - (unsigned)(j % 3));
        }
        __syncthreads();
        if (tid == 0) {   // the swap chain: std::swap(shuffled[p], shuffled[p + r]) for p = 0, 1, 2
            for (int t = 0; t < RS_TRIES; ++t) {
                const unsigned q0 = mod[3 * t], q1 = 1u + mod[3 * t + 1], q2 = 2u + mod[3 * t + 2];
                int x;
                if (q0 == 1u) { x = a0; a0 = a1; a1 = x; }
                else if (q0 == 2u) { x = a0; a0 = a2; a2 = x; }
                else if (q0 > 2u) { x = sh[q0]; sh[q0] = a0; a0 = x; }
                if (q1 == 2u) { x = a1; a1 = a2; a2 = x; }
                else if (q1 > 2u) { x = sh[q1]; sh[q1] = a1; a1 = x; }
                if (q2 > 2u) { x = sh[q2]; sh[q2] = a2; a2 = x; }
                trip[3 * t] = a0; trip[3 * t + 1] = a1; trip[3 * t + 2] = a2;
            }
        }
        __syncthreads();
        if (tid < RS_TRIES) {
            const int i0 = trip[3 * tid], i1 = trip[3 * tid + 1], i2 = trip[3 * tid + 2];
            good[tid] = (rs_d2(s4, i0, i1) > sdt && rs_d2(s4, i0, i2) > sdt && rs_d2(s4, i1, i2) > sdt) ? 1 : 0;
        }
        __syncthreads();
        if (tid == 0) {   // the host loop over the tries of this batch
            for (int t = 0; t < RS_TRIES; ++t) {
                ++tries;
                if (good[t]) {
                    samples[3 * h] = trip[3 * t]; samples[3 * h + 1] = trip[3 * t + 1]; samples[3 * h + 2] = trip[3 * t + 2];
                    ++h;
                    tries = 0;
                    if (h == n_hyp) { s_done = 1; break; }
                } else if (tries == 1000u) {   // max_sample_checks_: "Could not select sample points", PCL stops here
                    s_done = 1;
                    break;
                }
            }
            if (s_done) st->n_valid = (int)h;
        }
        __syncthreads();
        if (s_done) break;
    }
}

__global__ void ransac_replay_kernel(RansacDevState* __restrict__ st, const int* __restrict__ counts, int max_iterations) {
    if (threadIdx.x == 0 && blockIdx.x == 0) ransac_adaptive_stop(st, counts, max_iterations);
}

int ransac_run_dev(Ctx* c, const float4* d_src, const float4* d_tgt, const int* d_pairs, int pair_stride, const int* d_n_pairs, size_t n_cap,
                   int max_iterations, double threshold, int* d_pairs_out, int* d_n_out, float* d_T_out, int* d_iterations_out, const int* d_skip) {
    if (n_cap > c->max_kp) { set_error("bshot_ransac_dev: %zu correspondences > max_keypoints %zu", n_cap, c->max_kp); return BSHOT_E_CAPACITY; }
    if (max_iterations < 1 || max_iterations > 100000) { set_error("bshot_ransac_dev: bad max_iterations"); return BSHOT_E_INVALID; }
    const size_t n_hyp = (size_t)max_iterations + 1, cap = std::max<size_t>(n_cap, 1);
    // the shuffled list: n ints in shared memory when they fit, else in the scratch
    const size_t smem = 4 * cap;
    const bool in_smem = smem <= 160 * 1024;
    RansacScratch r;
    BSHOT_TRY(ransac_scratch(c, "bshot_ransac_dev", max_iterations, cap, in_smem ? 0 : 4 * cap, &r));
    const double thresh2 = threshold * threshold;
    ransac_gather_kernel<<<(unsigned)((cap + 255) / 256), 256, 0, c->stream>>>(d_src, d_tgt, d_pairs, pair_stride, d_n_pairs, (unsigned)n_cap, d_skip, r.s4, r.t4,
                                                                              r.st);
    if (in_smem && smem > 48 * 1024) BSHOT_CUDA_TRY(cudaFuncSetAttribute(ransac_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ransac_sample_kernel<<<1, RS_THREADS, in_smem ? smem : 0, c->stream>>>(r.s4, r.st, (unsigned)n_hyp, r.samples, in_smem ? nullptr : reinterpret_cast<int*>(r.extra));
    ransac_score_dev_kernel<<<(unsigned)((n_hyp * 32 + 127) / 128), 128, 0, c->stream>>>(r.s4, r.t4, r.st, r.samples, thresh2, r.models, r.counts);
    ransac_replay_kernel<<<1, 32, 0, c->stream>>>(r.st, r.counts, max_iterations);
    ransac_select_dev_kernel<<<(unsigned)((cap + 255) / 256), 256, 0, c->stream>>>(r.s4, r.t4, r.st, r.models, thresh2, r.inlier);
    ransac_finish_kernel<<<1, 1024, 0, c->stream>>>(r.st, d_pairs, pair_stride, r.inlier, r.models, d_pairs_out, d_n_out, d_T_out, d_iterations_out);
    count_launch(c, 6);
    return check_launch("device RANSAC kernels");
}

}  // namespace bshot
