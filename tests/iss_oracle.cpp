// iss_oracle.cpp -- CPU restatement of the ISS detector and of the keypoint repeatability measure, for the tests and
// tools/iss_bench.py (TEST INFRASTRUCTURE, never linked into the product).  Built on the CPU oracle's public C API
// (oracle/bshot_oracle.h): orc_radius_search for the neighbourhoods (all points with fp32 squared distance < r^2,
// ascending (distance, index)) and orc_eigh3 for the eigenvalues.  tests/iss_oracle.py compiles it into a temporary
// directory against oracle/libbshot_oracle.so.
//
// PARITY PIN: UNPINNED.  iss_ref_detect restates PCL 1.8 ISSKeypoint3D::detectKeypoints (border radius 0) as
// issKpDetection calls it (src/lidar_odometry.cpp:447-461) from the published algorithm; PCL is not available, so it is
// checked only against known answers and an independent numpy / scipy restatement (tests/test_iss.py), never against
// PCL itself.  The eigenvalues come from orc_eigh3 (Jacobi) where PCL uses Eigen::SelfAdjointEigenSolver.  Where PCL's
// `continue` leaves third_eigen_value to stale memory (non-finite eigenvalues, lambda3 < 0) the point is defined as not
// salient.  iss_ref_repeatability is the port's own definition of kpEvaluation (src/lidar_odometry.cpp:392-445): the
// source of the reference's printed "Repeat rate" is not available.
//
// Build flags: -ffp-contract=off, so the fp32 arithmetic is the plain IEEE sequence written here.
#include <algorithm>
#include <cmath>
#include <limits>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "bshot_oracle.h"

namespace {

inline bool finite3(const float* p) { return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]); }

// flann::L2_Simple in fp32
inline float sqdist(const float* a, const float* b) {
    float d = a[0] - b[0];
    float r = d * d;
    d = a[1] - b[1];
    r += d * d;
    d = a[2] - b[2];
    r += d * d;
    return r;
}

int nthreads(int threads) {
#ifdef _OPENMP
    return threads > 0 ? threads : omp_get_max_threads();
#else
    (void)threads;
    return 1;
#endif
}

}  // namespace

extern "C" {

// Salient stage per finite point p: neighbours within r_s (p included, no max_nn); fewer than min_nn -> zero scatter
// matrix, else sum (n - p)(n - p)^T in double over the neighbours in radius-search order; eigenvalues l1 >= l2 >= l3;
// salient when all finite, l3 >= 0, l2/l1 < g21 and l3/l2 < g32, third_eigen_value = l3 (else 0).  Non-max stage:
// third_eigen_value > 0, at least min_nn points within r_nm (p included), no neighbour with a strictly larger value.
// xyz: the n points the cloud c was created from (3 floats each).  Writes up to cap keypoint indices in ascending order
// and returns their count; eig_out (n x 3 doubles, l1..l3, zeros for non-finite points) may be NULL.
int iss_ref_detect(const orc_cloud* c, const float* xyz, size_t n_, float r_s, float r_nm, double g21, double g32, int min_nn,
                   int threads, int* idx_out, size_t cap, double* eig_out) {
    const int n = (int)n_;
    const int nt = nthreads(threads);
    (void)nt;
    std::vector<double> third(n, 0.0);  // third_eigen_value_, zero-initialised
    if (eig_out) std::fill(eig_out, eig_out + 3 * (size_t)n, 0.0);
#pragma omp parallel num_threads(nt)
    {
        std::vector<int> nn(std::max(n, 1));
#pragma omp for schedule(dynamic, 64)
        for (int i = 0; i < n; ++i) {
            const float* p = xyz + 3 * (size_t)i;
            if (!finite3(p)) continue;
            const int k = orc_radius_search(c, p, r_s, 0, nn.data(), nullptr, n);
            double cov[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
            if (k >= min_nn) {  // getScatterMatrix: zero below min_neighbors
                for (int m = 0; m < k; ++m) {
                    const float* q = xyz + 3 * (size_t)nn[m];
                    const double v[3] = {(double)q[0] - (double)p[0], (double)q[1] - (double)p[1], (double)q[2] - (double)p[2]};
                    for (int a = 0; a < 3; ++a)
                        for (int b = 0; b < 3; ++b) cov[3 * a + b] += v[a] * v[b];
                }
            }
            double w[3], V[9];
            orc_eigh3(cov, w, V);
            const double e1 = w[2], e2 = w[1], e3 = w[0];
            if (eig_out) { eig_out[3 * (size_t)i] = e1; eig_out[3 * (size_t)i + 1] = e2; eig_out[3 * (size_t)i + 2] = e3; }
            if (!std::isfinite(e1) || !std::isfinite(e2) || !std::isfinite(e3) || e3 < 0) continue;  // defined: not salient
            if (e2 / e1 < g21 && e3 / e2 < g32) third[i] = e3;
        }
    }
    std::vector<unsigned char> is_max(n, 0);
#pragma omp parallel num_threads(nt)
    {
        std::vector<int> nn(std::max(n, 1));
#pragma omp for schedule(dynamic, 64)
        for (int i = 0; i < n; ++i) {
            const float* p = xyz + 3 * (size_t)i;
            if (!(third[i] > 0.0) || !finite3(p)) continue;
            const int k = orc_radius_search(c, p, r_nm, 0, nn.data(), nullptr, n);
            if (k < min_nn) continue;
            bool m = true;
            for (int j = 0; j < k; ++j)
                if (third[i] < third[nn[j]]) m = false;
            is_max[i] = m ? 1 : 0;
        }
    }
    size_t k = 0;
    for (int i = 0; i < n; ++i)
        if (is_max[i]) {
            if (idx_out && k < cap) idx_out[k] = i;
            ++k;
        }
    return (int)k;
}

// A moved by pose_a, B by pose_b (row-major [R|T], NULL = identity, ((r0*x + r1*y) + r2*z) + t in fp32); per point of A
// the nearest point of B by fp32 squared distance (lowest index on ties; -1 / +inf when B is empty) -> nn_idx / nn_dist
// (Euclidean); returns the hits (squared distance < radius^2).
size_t iss_ref_repeatability(const float* a_xyz, size_t na, const float* pose_a, const float* b_xyz, size_t nb, const float* pose_b,
                             float radius, int* nn_idx_out, float* nn_dist_out) {
    auto move = [](const float* pose, const float* p, float* o) {
        if (!pose) { o[0] = p[0]; o[1] = p[1]; o[2] = p[2]; return; }
        o[0] = ((pose[0] * p[0] + pose[1] * p[1]) + pose[2] * p[2]) + pose[3];
        o[1] = ((pose[4] * p[0] + pose[5] * p[1]) + pose[6] * p[2]) + pose[7];
        o[2] = ((pose[8] * p[0] + pose[9] * p[1]) + pose[10] * p[2]) + pose[11];
    };
    std::vector<float> b(3 * nb);
    for (size_t j = 0; j < nb; ++j) move(pose_b, b_xyz + 3 * j, &b[3 * j]);
    const float r2 = (float)((double)radius * (double)radius);
    size_t hits = 0;
    for (size_t i = 0; i < na; ++i) {
        float a[3];
        move(pose_a, a_xyz + 3 * i, a);
        float best = std::numeric_limits<float>::infinity();
        int bi = -1;
        for (size_t j = 0; j < nb; ++j) {
            const float d = sqdist(a, &b[3 * j]);
            if (d < best) { best = d; bi = (int)j; }
        }
        if (nn_idx_out) nn_idx_out[i] = bi;
        if (nn_dist_out) nn_dist_out[i] = bi >= 0 ? std::sqrt(best) : std::numeric_limits<float>::infinity();
        if (best < r2) ++hits;
    }
    return hits;
}

}  // extern "C"
