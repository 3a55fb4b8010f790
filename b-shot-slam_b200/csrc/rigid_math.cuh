// rigid_math.cuh -- small dense pieces shared by the RANSAC and ICP kernels (both compiled with -fmad=false so that the
// CPU restatement in the test oracle reproduces them bit for bit).
#pragma once
#include <math.h>

namespace bshot {

// ---- 3x3 SVD by one-sided Jacobi (Hestenes), double; shared by host and device ---------------------------------------
// A = U diag(s) V^T with s[0] >= s[1] >= s[2] >= 0 and V orthonormal.  A column of U whose singular value is exactly zero
// is left zero: the callers complete the bases themselves (a cross product at rank 2, rigid_rotation_rank01 below at
// rank <= 1).  Only +, -, *, /, sqrt: reproducible bit for bit without FMA contraction.
__host__ __device__ inline void svd3_hestenes(const double a_in[9], double U[9], double s[3], double V[9]) {
    double a[3][3], v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) a[r][c] = a_in[3 * r + c];
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                double alpha = 0, beta = 0, gamma = 0;
                for (int r = 0; r < 3; ++r) { alpha += a[r][p] * a[r][p]; beta += a[r][q] * a[r][q]; gamma += a[r][p] * a[r][q]; }
                if (gamma == 0.0) continue;
                const double lim = 1e-30 * (alpha * beta);
                if (gamma * gamma <= lim) continue;
                off += gamma * gamma;
                const double zeta = (beta - alpha) / (2.0 * gamma);
                const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                const double c = 1.0 / sqrt(1.0 + t * t), sn = c * t;
                for (int r = 0; r < 3; ++r) {
                    const double x = a[r][p], y = a[r][q];
                    a[r][p] = c * x - sn * y;
                    a[r][q] = sn * x + c * y;
                    const double vx = v[r][p], vy = v[r][q];
                    v[r][p] = c * vx - sn * vy;
                    v[r][q] = sn * vx + c * vy;
                }
            }
        if (off == 0.0) break;
    }
    double n[3];
    int o[3] = {0, 1, 2};
    for (int c = 0; c < 3; ++c) n[c] = sqrt(a[0][c] * a[0][c] + a[1][c] * a[1][c] + a[2][c] * a[2][c]);
    if (n[o[0]] < n[o[1]]) { int t = o[0]; o[0] = o[1]; o[1] = t; }
    if (n[o[1]] < n[o[2]]) { int t = o[1]; o[1] = o[2]; o[2] = t; }
    if (n[o[0]] < n[o[1]]) { int t = o[0]; o[0] = o[1]; o[1] = t; }
    for (int k = 0; k < 3; ++k) {
        s[k] = n[o[k]];
        for (int r = 0; r < 3; ++r) { V[3 * r + k] = v[r][o[k]]; U[3 * r + k] = (s[k] > 0.0) ? a[r][o[k]] / s[k] : 0.0; }
    }
}

// ---- the rank-0 test of a Procrustes fit ------------------------------------------------------------------------------
// When every target (or every source) is one point, the exact Sigma is 0, but the computed one is not: the rounded
// centroid dm differs from the common target by a tiny constant, so Sigma = (T - dm) mean(s - sm)^T is rounding noise with
// s0 > 0 whenever n is not a power of two, and its singular vectors are arbitrary.  A relative test cannot see that, so
// rank 0 is decided against an absolute floor built from the data: with k roundings on every summation path and unit
// roundoff u, the centroids are off by <= gamma_{k+1} mean |p|_1 (resp. |q|_1), and when one side is a single point
// sum_rc |Sigma_rc| <= gamma_{k+3} (Ad (Ap + 2 As) + As (Aq + 2 Ad)), where Ap, Aq, As, Ad are the means of the 1-norms
// of the sources, the targets and the centred sources and targets (sums P, Q, S, D over n pairs).  s0 <= |Sigma|_F is
// at most that sum; the floor is twice the bound.  For real clouds s0 is of the order of Ad As, far above it.
__host__ __device__ inline double rigid_noise_floor(double P, double Q, double S, double D, double n, double k, double u) {
    const double ap = P / n, aq = Q / n, as = S / n, ad = D / n;
    return 2.0 * ((k + 3.0) * u) * (ad * (ap + 2.0 * as) + as * (aq + 2.0 * ad));
}

// ---- the rotation of a Procrustes fit whose cross-covariance has rank 0 or 1 (row-major R) -------------------------------
// Sigma = s0 u0 v0^T (u0 = U[:,0], v0 = V[:,0]): every proper R with R v0 = u0 maximises tr(R^T Sigma), so R is not unique.
// This one is deterministic and continuous in (u0, v0) on each side of u0.v0 = 0:
//   * u0.v0 >= 0: the minimal rotation carrying v0 onto u0, c I + [k]x + k k^T / (1 + c) with k = v0 x u0, c = v0.u0;
//   * u0.v0 < 0: a half-turn H about a fixed axis a perpendicular to v0 (a = v0 x e_j, e_j the axis of v0's smallest
//     component) carries v0 onto -v0, then the minimal rotation carrying -v0 onto u0: R = M(-v0 -> u0) H.
//     Both steps have 1 + c >= 1, so R stays orthonormal to rounding even for anti-parallel u0 and v0.
// Rank 0 (`rank0`: s0 at or below rigid_noise_floor, e.g. s0 = 0 and u0 = 0): R = I, which is what pcl::umeyama returns
// for Sigma = 0.
// pcl::umeyama returns U S V^T with Eigen's completion of the null spaces here, which may even be improper; this choice is
// a deliberate difference (DESIGN 3.5).  R is the same for (u0, v0) and (-u0, -v0).
__host__ __device__ inline void rigid_rotation_min(const double v[3], const double u[3], double R[9]) {   // v.u >= 0
    const double c = (v[0] * u[0] + v[1] * u[1]) + v[2] * u[2];
    const double k[3] = {v[1] * u[2] - v[2] * u[1], v[2] * u[0] - v[0] * u[2], v[0] * u[1] - v[1] * u[0]};
    const double f = 1.0 / (1.0 + c);
    R[0] = c + k[0] * k[0] * f; R[1] = k[0] * k[1] * f - k[2]; R[2] = k[0] * k[2] * f + k[1];
    R[3] = k[1] * k[0] * f + k[2]; R[4] = c + k[1] * k[1] * f; R[5] = k[1] * k[2] * f - k[0];
    R[6] = k[2] * k[0] * f - k[1]; R[7] = k[2] * k[1] * f + k[0]; R[8] = c + k[2] * k[2] * f;
}

__host__ __device__ inline void rigid_rotation_rank01(const double U[9], const double V[9], bool rank0, double R[9]) {
    if (rank0) {
        for (int e = 0; e < 9; ++e) R[e] = (e % 4 == 0) ? 1.0 : 0.0;
        return;
    }
    const double u[3] = {U[0], U[3], U[6]}, v[3] = {V[0], V[3], V[6]};
    if ((v[0] * u[0] + v[1] * u[1]) + v[2] * u[2] >= 0.0) { rigid_rotation_min(v, u, R); return; }
    const double ax[3] = {fabs(v[0]), fabs(v[1]), fabs(v[2])};
    const int j = (ax[0] <= ax[1] && ax[0] <= ax[2]) ? 0 : (ax[1] <= ax[2] ? 1 : 2);
    double a[3] = {0.0, 0.0, 0.0};   // v x e_j
    if (j == 0) { a[1] = v[2]; a[2] = -v[1]; }
    else if (j == 1) { a[0] = -v[2]; a[2] = v[0]; }
    else { a[0] = v[1]; a[1] = -v[0]; }
    const double na = sqrt((a[0] * a[0] + a[1] * a[1]) + a[2] * a[2]);
    for (int r = 0; r < 3; ++r) a[r] = a[r] / na;
    double H[9], M[9];
    for (int r = 0; r < 3; ++r)
        for (int q = 0; q < 3; ++q) H[3 * r + q] = 2.0 * a[r] * a[q] - (r == q ? 1.0 : 0.0);
    const double w[3] = {-v[0], -v[1], -v[2]};
    rigid_rotation_min(w, u, M);
    for (int r = 0; r < 3; ++r)
        for (int q = 0; q < 3; ++q) R[3 * r + q] = (M[3 * r] * H[q] + M[3 * r + 1] * H[3 + q]) + M[3 * r + 2] * H[6 + q];
}

}  // namespace bshot
