// posegraph.cu -- the trajectory's pose graph, optimised on the device in float64 (bshot_optimize_trajectory).
//
// One cooperative kernel runs the whole Levenberg-Marquardt solve; its control (stop tests, lambda, step acceptance, CG)
// is evaluated identically by every thread from grid-wide reductions, so the host launches once and reads back once.
// Sums are deterministic: per edge terms are gathered per node through a node -> edge incidence list the host builds (in
// a fixed order), and every reduction is a fixed CTA tree followed by a fixed-order sum of the CTA partials.  No atomics.
//
// Model (DESIGN §3.9): t <- t + rho, R <- R Exp(phi); edge (a, b), Z = [R_z | t_z]:
//   r_t = R_a^T (t_b - t_a) - t_z,  r_phi = Log(R_z^T R_a^T R_b)
//   dr_t/drho_a = -R_a^T, dr_t/drho_b = R_a^T, dr_t/dphi_a = [R_a^T (t_b - t_a)]x
//   dr_phi/dphi_b = Jr^-1(r_phi), dr_phi/dphi_a = -Jr^-1(r_phi) R_b^T R_a
// Linear solve: PCG on (H + lambda diag H) d = -g over nodes 1..n-1; the preconditioner is the block-tridiagonal part of
// that matrix (every diagonal block and the blocks between consecutive nodes), applied by block cyclic reduction: log2 n
// levels of 6x6 float64 blocks, each level one parallel pass.  The remainder is the loop edges' off-chain blocks, of rank
// <= 12 each, so in exact arithmetic CG ends within 12 L + 1 iterations.
#include <cooperative_groups.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"
#include "stages.h"

namespace cg = cooperative_groups;

namespace bshot {

constexpr int PG_THREADS = 256;

struct PgArgs {
    int n, n_edges, n_loops, n_levels;
    const float* traj;          // n x 12 (the map's trajectory)
    const float* loop_T;        // n_loops x 16
    const int* e_from;          // n_edges: odometry edges u = 0..n-2 first, then the loops
    const int* e_to;
    const int* inc_ptr;         // n + 1
    const int* inc;             // 2 n_edges: edge * 2 + side (0: the node is `from`, 1: `to`)
    const int* lvl_off;         // n_levels + 1: first entry of each reduction level
    double w_odom_t, w_odom_r, w_loop_t, w_loop_r;   // 1 / sigma^2
    int max_it, max_cg;
    double gtol, steptol, cgtol;
    // work (device)
    double* X;                  // n x 12: R row-major, t
    double* Xc;                 // n x 12: the candidate
    double* Z;                  // n_edges x 12
    double* EH;                 // n_edges x 120: H_aa, H_ab, H_bb (36 each), g_a, g_b (6 each)
    double* ecost;              // n_edges
    double* Dg;                 // n x 42: diagonal block, gradient
    double *vb, *vx, *vr, *vz, *vp, *vq;   // (n - 1) x 6 each
    double *LA, *LB, *LC, *W1, *W2;        // levels x 36
    double *LD, *LX;                       // levels x 6
    double* red;                // gridDim.x partials
    int* moved;                 // n
    float* out_poses;           // n x 12
    double* out_loop_cost;      // n_loops
    double* out_rep;            // cost_initial, cost_final, grad_inf, iterations, cg_iterations, status
};

// ---- small float64 algebra ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void skew(const double* v, double* S) {
    S[0] = 0; S[1] = -v[2]; S[2] = v[1]; S[3] = v[2]; S[4] = 0; S[5] = -v[0]; S[6] = -v[1]; S[7] = v[0]; S[8] = 0;
}
__device__ __forceinline__ void mm3(const double* A, const double* B, double* C) {   // C = A B
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
__device__ __forceinline__ void mtm3(const double* A, const double* B, double* C) {  // C = A^T B
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) C[3 * i + j] = A[i] * B[j] + A[3 + i] * B[3 + j] + A[6 + i] * B[6 + j];
}
__device__ void so3_exp(const double* w, double* R) {
    const double th2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2], th = sqrt(th2);
    double A, B;
    if (th < 1e-4) { A = 1.0 - th2 / 6.0 + th2 * th2 / 120.0; B = 0.5 - th2 / 24.0 + th2 * th2 / 720.0; }
    else { A = sin(th) / th; B = (1.0 - cos(th)) / th2; }
    double S[9], S2[9];
    skew(w, S);
    mm3(S, S, S2);
    for (int e = 0; e < 9; ++e) R[e] = (e % 4 == 0 ? 1.0 : 0.0) + A * S[e] + B * S2[e];
}
__device__ void so3_log(const double* R, double* w) {
    const double c = fmin(1.0, fmax(-1.0, 0.5 * (R[0] + R[4] + R[8] - 1.0)));
    const double v0 = R[7] - R[5], v1 = R[2] - R[6], v2 = R[3] - R[1];
    const double th = acos(c);
    if (th < 1e-4) {                       // th / (2 sin th) = 1/2 + th^2 / 12 + 7 th^4 / 720
        const double f = 0.5 + th * th / 12.0 + 7.0 * th * th * th * th / 720.0;
        w[0] = f * v0; w[1] = f * v1; w[2] = f * v2;
    } else if (th < 3.14159 - 1e-3) {
        const double f = th / (2.0 * sin(th));
        w[0] = f * v0; w[1] = f * v1; w[2] = f * v2;
    } else {                               // near pi: the axis from the symmetric part
        int k = (R[0] >= R[4] && R[0] >= R[8]) ? 0 : (R[4] >= R[8] ? 1 : 2);
        double a[3];
        a[k] = sqrt(fmax(0.0, 0.5 * (R[4 * k] + 1.0)));
        for (int j = 0; j < 3; ++j) if (j != k) a[j] = (R[3 * k + j] + R[3 * j + k]) / (4.0 * a[k]);
        const double s = (k == 0 ? v0 : (k == 1 ? v1 : v2)) < 0.0 ? -1.0 : 1.0;
        for (int j = 0; j < 3; ++j) w[j] = s * th * a[j];
    }
}
__device__ void jr_inv(const double* w, double* J) {
    const double th2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2], th = sqrt(th2);
    double C;
    if (th < 1e-4) C = 1.0 / 12.0 + th2 / 720.0 + th2 * th2 / 30240.0;
    else C = 1.0 / th2 - (1.0 + cos(th)) / (2.0 * th * sin(th));
    double S[9], S2[9];
    skew(w, S);
    mm3(S, S, S2);
    for (int e = 0; e < 9; ++e) J[e] = (e % 4 == 0 ? 1.0 : 0.0) + 0.5 * S[e] + C * S2[e];
}
// 6x6 helpers, row-major
__device__ __forceinline__ void mm6(const double* A, const double* B, double* C) {
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) { double s = 0; for (int k = 0; k < 6; ++k) s += A[6 * i + k] * B[6 * k + j]; C[6 * i + j] = s; }
}
__device__ __forceinline__ void mv6(const double* A, const double* x, double* y, bool transpose, double sign) {   // y += sign * A x (or A^T x)
    for (int i = 0; i < 6; ++i) { double s = 0; for (int k = 0; k < 6; ++k) s += (transpose ? A[6 * k + i] : A[6 * i + k]) * x[k]; y[i] += sign * s; }
}
// inverse of a symmetric positive definite 6x6 (Gauss-Jordan; the pivots of an SPD matrix are positive)
__device__ void inv6(const double* M, double* I) {
    double a[36];
    for (int e = 0; e < 36; ++e) { a[e] = M[e]; I[e] = (e % 7 == 0) ? 1.0 : 0.0; }
    for (int c = 0; c < 6; ++c) {
        const double p = 1.0 / a[6 * c + c];
        for (int j = 0; j < 6; ++j) { a[6 * c + j] *= p; I[6 * c + j] *= p; }
        for (int r = 0; r < 6; ++r) {
            if (r == c) continue;
            const double f = a[6 * r + c];
            for (int j = 0; j < 6; ++j) { a[6 * r + j] -= f * a[6 * c + j]; I[6 * r + j] -= f * I[6 * c + j]; }
        }
    }
}

// ---- grid-wide deterministic reductions ---------------------------------------------------------------------------------
// op 0 sum, 1 max.  Every thread returns the same value
__device__ double grid_reduce(cg::grid_group& grid, double v, int op, double* red, double* sh) {
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int s = PG_THREADS / 2; s > 0; s >>= 1) {
        if (threadIdx.x < (unsigned)s) sh[threadIdx.x] = op ? fmax(sh[threadIdx.x], sh[threadIdx.x + s]) : sh[threadIdx.x] + sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) red[blockIdx.x] = sh[0];
    grid.sync();
    double t = op ? 0.0 : 0.0;
    for (unsigned b = 0; b < gridDim.x; ++b) t = op ? fmax(t, red[b]) : t + red[b];
    grid.sync();   // the partials are read before the next reduction rewrites them
    return t;
}

// ---- residuals, Jacobians, linearisation --------------------------------------------------------------------------------
__device__ void edge_terms(const PgArgs& a, const double* X, int e, bool lin, double* cost_out) {
    const int ia = a.e_from[e], ib = a.e_to[e];
    const double *Ra = X + 12 * ia, *ta = Ra + 9, *Rb = X + 12 * ib, *tb = Rb + 9, *Rz = a.Z + 12 * e, *tz = Rz + 9;
    const bool loop = e >= a.n - 1;
    const double wt = loop ? a.w_loop_t : a.w_odom_t, wr = loop ? a.w_loop_r : a.w_odom_r;
    double d[3] = {tb[0] - ta[0], tb[1] - ta[1], tb[2] - ta[2]}, v[3], r[6];
    for (int i = 0; i < 3; ++i) v[i] = Ra[i] * d[0] + Ra[3 + i] * d[1] + Ra[6 + i] * d[2];   // R_a^T (t_b - t_a)
    for (int i = 0; i < 3; ++i) r[i] = v[i] - tz[i];
    double RaRb[9], E[9];
    mtm3(Ra, Rb, RaRb);
    mtm3(Rz, RaRb, E);
    so3_log(E, r + 3);
    *cost_out = 0.5 * (wt * (r[0] * r[0] + r[1] * r[1] + r[2] * r[2]) + wr * (r[3] * r[3] + r[4] * r[4] + r[5] * r[5]));
    if (!lin) return;
    double Ja[36] = {0}, Jb[36] = {0}, Jri[9], S[9], RbRa[9], M[9];
    jr_inv(r + 3, Jri);
    skew(v, S);
    mtm3(Rb, Ra, RbRa);
    mm3(Jri, RbRa, M);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            Ja[6 * i + j] = -Ra[3 * j + i];            // -R_a^T
            Jb[6 * i + j] = Ra[3 * j + i];             //  R_a^T
            Ja[6 * i + 3 + j] = S[3 * i + j];          // [R_a^T (t_b - t_a)]x
            Ja[6 * (3 + i) + 3 + j] = -M[3 * i + j];   // -Jr^-1 R_b^T R_a
            Jb[6 * (3 + i) + 3 + j] = Jri[3 * i + j];  //  Jr^-1
        }
    const double w[6] = {wt, wt, wt, wr, wr, wr};
    double* H = a.EH + (size_t)120 * e;
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) {
            double saa = 0, sab = 0, sbb = 0;
            for (int k = 0; k < 6; ++k) {
                saa += Ja[6 * k + i] * w[k] * Ja[6 * k + j];
                sab += Ja[6 * k + i] * w[k] * Jb[6 * k + j];
                sbb += Jb[6 * k + i] * w[k] * Jb[6 * k + j];
            }
            H[6 * i + j] = saa; H[36 + 6 * i + j] = sab; H[72 + 6 * i + j] = sbb;
        }
    for (int i = 0; i < 6; ++i) {
        double ga = 0, gb = 0;
        for (int k = 0; k < 6; ++k) { ga += Ja[6 * k + i] * w[k] * r[k]; gb += Jb[6 * k + i] * w[k] * r[k]; }
        H[108 + i] = ga; H[114 + i] = gb;
    }
}

// cost of X (every thread gets it); lin: also the edge blocks, the node blocks and |g|_inf (*ginf)
__device__ double evaluate(cg::grid_group& grid, const PgArgs& a, const double* X, bool lin, double* ginf, double* sh) {
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (unsigned e = tid; e < (unsigned)a.n_edges; e += nth) { double c; edge_terms(a, X, (int)e, lin, &c); a.ecost[e] = c; }
    grid.sync();
    double part = 0.0;   // the edge costs summed in edge order per thread stride, then the fixed tree
    for (unsigned e = tid; e < (unsigned)a.n_edges; e += nth) part += a.ecost[e];
    const double F = grid_reduce(grid, part, 0, a.red, sh);
    if (!lin) return F;
    double gm = 0.0;
    for (unsigned i = tid; i < (unsigned)a.n; i += nth) {
        double D[36] = {0}, g[6] = {0};
        for (int q = a.inc_ptr[i]; q < a.inc_ptr[i + 1]; ++q) {
            const int e = a.inc[q] >> 1, side = a.inc[q] & 1;
            const double* H = a.EH + (size_t)120 * e;
            for (int k = 0; k < 36; ++k) D[k] += H[side ? 72 + k : k];
            for (int k = 0; k < 6; ++k) g[k] += H[side ? 114 + k : 108 + k];
        }
        double* o = a.Dg + 42 * (size_t)i;
        for (int k = 0; k < 36; ++k) o[k] = D[k];
        for (int k = 0; k < 6; ++k) { o[36 + k] = g[k]; if (i > 0) gm = fmax(gm, fabs(g[k])); }
    }
    *ginf = grid_reduce(grid, gm, 1, a.red, sh);
    return F;
}

// the block between free nodes i and j (row i, column j) of H: the edges joining them
__device__ void off_block(const PgArgs& a, int i, int j, double* B) {
    for (int k = 0; k < 36; ++k) B[k] = 0.0;
    for (int q = a.inc_ptr[i]; q < a.inc_ptr[i + 1]; ++q) {
        const int e = a.inc[q] >> 1, side = a.inc[q] & 1;
        const int other = side ? a.e_from[e] : a.e_to[e];
        if (other != j) continue;
        const double* H = a.EH + (size_t)120 * e + 36;
        for (int r = 0; r < 6; ++r) for (int c = 0; c < 6; ++c) B[6 * r + c] += side ? H[6 * c + r] : H[6 * r + c];
    }
}

// y = (H + lambda diag H) x over the free nodes (k = node - 1)
__device__ void matvec(const PgArgs& a, double lambda, const double* x, double* y) {
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (unsigned k = tid; k < (unsigned)(a.n - 1); k += nth) {
        const int i = (int)k + 1;
        const double* D = a.Dg + 42 * (size_t)i;
        double s[6] = {0};
        mv6(D, x + 6 * k, s, false, 1.0);
        for (int r = 0; r < 6; ++r) s[r] += lambda * D[7 * r] * x[6 * k + r];
        for (int q = a.inc_ptr[i]; q < a.inc_ptr[i + 1]; ++q) {
            const int e = a.inc[q] >> 1, side = a.inc[q] & 1;
            const int j = side ? a.e_from[e] : a.e_to[e];
            if (j == 0) continue;
            mv6(a.EH + (size_t)120 * e + 36, x + 6 * (j - 1), s, side == 1, 1.0);
        }
        for (int r = 0; r < 6; ++r) y[6 * k + r] = s[r];
    }
}

// block cyclic reduction of the damped chain: level 0 holds the chain over k = 0..n-2, level l + 1 the odd entries of l
__device__ void bcr_factor(cg::grid_group& grid, const PgArgs& a, double lambda) {
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    const int m0 = a.n - 1;
    for (unsigned k = tid; k < (unsigned)m0; k += nth) {
        const int i = (int)k + 1;
        const double* D = a.Dg + 42 * (size_t)i;
        double* B = a.LB + 36 * (size_t)k;
        for (int e = 0; e < 36; ++e) B[e] = D[e];
        for (int r = 0; r < 6; ++r) B[7 * r] += lambda * D[7 * r];
        if ((int)k > 0) off_block(a, i, i - 1, a.LA + 36 * (size_t)k); else for (int e = 0; e < 36; ++e) a.LA[e] = 0.0;
        if ((int)k + 1 < m0) off_block(a, i, i + 1, a.LC + 36 * (size_t)k); else for (int e = 0; e < 36; ++e) a.LC[36 * (size_t)k + e] = 0.0;
    }
    grid.sync();
    for (int l = 0; l < a.n_levels; ++l) {
        const int off = a.lvl_off[l], m = a.lvl_off[l + 1] - off, noff = a.lvl_off[l + 1];
        for (unsigned k = tid * 2; k < (unsigned)m; k += nth * 2) inv6(a.LB + 36 * (size_t)(off + k), a.W1 + 36 * (size_t)(off + k));
        grid.sync();
        for (unsigned k = tid * 2 + 1; k < (unsigned)m; k += nth * 2) {
            const size_t p = off + k, pm = p - 1, pp = p + 1;
            const bool right = k + 1 < (unsigned)m;
            double al[36], ga[36] = {0}, T[36];
            mm6(a.LA + 36 * p, a.W1 + 36 * pm, al);
            if (right) mm6(a.LC + 36 * p, a.W1 + 36 * pp, ga);
            const size_t q = noff + (k - 1) / 2;
            double* B = a.LB + 36 * q;
            for (int e = 0; e < 36; ++e) B[e] = a.LB[36 * p + e];
            mm6(al, a.LC + 36 * pm, T);
            for (int e = 0; e < 36; ++e) B[e] -= T[e];
            mm6(al, a.LA + 36 * pm, T);
            for (int e = 0; e < 36; ++e) a.LA[36 * q + e] = -T[e];
            if (right) {
                mm6(ga, a.LA + 36 * pp, T);
                for (int e = 0; e < 36; ++e) B[e] -= T[e];
                mm6(ga, a.LC + 36 * pp, T);
                for (int e = 0; e < 36; ++e) a.LC[36 * q + e] = -T[e];
            } else {
                for (int e = 0; e < 36; ++e) a.LC[36 * q + e] = 0.0;
            }
            for (int e = 0; e < 36; ++e) { a.W1[36 * p + e] = al[e]; a.W2[36 * p + e] = ga[e]; }
        }
        grid.sync();
    }
}

// x = M^-1 d (both (n - 1) x 6)
__device__ void bcr_apply(cg::grid_group& grid, const PgArgs& a, const double* d, double* x) {
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (unsigned k = tid; k < (unsigned)(6 * (a.n - 1)); k += nth) a.LD[k] = d[k];
    grid.sync();
    for (int l = 0; l < a.n_levels; ++l) {
        const int off = a.lvl_off[l], m = a.lvl_off[l + 1] - off, noff = a.lvl_off[l + 1];
        for (unsigned k = tid * 2 + 1; k < (unsigned)m; k += nth * 2) {
            const size_t p = off + k, q = noff + (k - 1) / 2;
            double s[6];
            for (int r = 0; r < 6; ++r) s[r] = a.LD[6 * p + r];
            mv6(a.W1 + 36 * p, a.LD + 6 * (p - 1), s, false, -1.0);
            if (k + 1 < (unsigned)m) mv6(a.W2 + 36 * p, a.LD + 6 * (p + 1), s, false, -1.0);
            for (int r = 0; r < 6; ++r) a.LD[6 * q + r] = s[r];
        }
        grid.sync();
    }
    for (int l = a.n_levels - 1; l >= 0; --l) {
        const int off = a.lvl_off[l], m = a.lvl_off[l + 1] - off, noff = a.lvl_off[l + 1];
        for (unsigned k = tid; k < (unsigned)m; k += nth) {
            const size_t p = off + k;
            if (k & 1u) { for (int r = 0; r < 6; ++r) a.LX[6 * p + r] = a.LX[6 * (noff + (k - 1) / 2) + r]; continue; }
            double s[6];
            for (int r = 0; r < 6; ++r) s[r] = a.LD[6 * p + r];
            if (k > 0) mv6(a.LA + 36 * p, a.LX + 6 * (noff + (k - 1) / 2), s, false, -1.0);
            if (k + 1 < (unsigned)m) mv6(a.LC + 36 * p, a.LX + 6 * (noff + k / 2), s, false, -1.0);
            double y[6] = {0};
            mv6(a.W1 + 36 * p, s, y, false, 1.0);
            for (int r = 0; r < 6; ++r) a.LX[6 * p + r] = y[r];
        }
        grid.sync();
    }
    for (unsigned k = tid; k < (unsigned)(6 * (a.n - 1)); k += nth) x[k] = a.LX[k];
    grid.sync();
}

__device__ double dot(cg::grid_group& grid, const PgArgs& a, const double* u, const double* v, double* sh) {
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    double s = 0.0;
    for (unsigned k = tid; k < (unsigned)(6 * (a.n - 1)); k += nth) s += u[k] * v[k];
    return grid_reduce(grid, s, 0, a.red, sh);
}

__global__ void __launch_bounds__(PG_THREADS) pg_solve_kernel(PgArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double sh[PG_THREADS];
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    const int nf6 = 6 * (a.n - 1);
    // nodes and edge measurements in float64; odometry edge u: Z = T_u^-1 T_{u+1}; loop edges: the caller's T
    for (unsigned i = tid; i < (unsigned)a.n; i += nth) {
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) a.X[12 * i + 3 * r + c] = (double)a.traj[12 * i + 4 * r + c];
            a.X[12 * i + 9 + r] = (double)a.traj[12 * i + 4 * r + 3];
        }
        a.moved[i] = 0;
    }
    grid.sync();
    for (unsigned e = tid; e < (unsigned)a.n_edges; e += nth) {
        double* Z = a.Z + 12 * e;
        if ((int)e < a.n - 1) {
            const double *Ra = a.X + 12 * e, *Rb = Ra + 12;
            mtm3(Ra, Rb, Z);
            const double d[3] = {Rb[9] - Ra[9], Rb[10] - Ra[10], Rb[11] - Ra[11]};
            for (int i = 0; i < 3; ++i) Z[9 + i] = Ra[i] * d[0] + Ra[3 + i] * d[1] + Ra[6 + i] * d[2];
        } else {
            const float* T = a.loop_T + 16 * (e - (a.n - 1));
            for (int r = 0; r < 3; ++r) { for (int c = 0; c < 3; ++c) Z[3 * r + c] = (double)T[4 * r + c]; Z[9 + r] = (double)T[4 * r + 3]; }
        }
    }
    grid.sync();
    double ginf, F = evaluate(grid, a, a.X, true, &ginf, sh);
    const double F0 = F;
    double lambda = 1e-4;
    int it = 0, cg_total = 0, status = 3;
    for (;;) {
        if (ginf <= a.gtol) { status = 1; break; }
        if (it >= a.max_it) { status = 3; break; }
        ++it;
        bcr_factor(grid, a, lambda);
        // PCG from x = 0 on b = -g
        for (unsigned k = tid; k < (unsigned)nf6; k += nth) {
            const double b = -a.Dg[42 * (size_t)(k / 6 + 1) + 36 + k % 6];
            a.vb[k] = b; a.vr[k] = b; a.vx[k] = 0.0;
        }
        grid.sync();
        const double bn = sqrt(dot(grid, a, a.vb, a.vb, sh));
        bcr_apply(grid, a, a.vr, a.vz);
        for (unsigned k = tid; k < (unsigned)nf6; k += nth) a.vp[k] = a.vz[k];
        grid.sync();
        double rz = dot(grid, a, a.vr, a.vz, sh), rn = bn;
        for (int c = 0; c < a.max_cg && rn > a.cgtol * bn; ++c) {
            matvec(a, lambda, a.vp, a.vq);
            grid.sync();
            const double pq = dot(grid, a, a.vp, a.vq, sh);
            if (!(pq > 0.0)) break;
            const double al = rz / pq;
            for (unsigned k = tid; k < (unsigned)nf6; k += nth) { a.vx[k] += al * a.vp[k]; a.vr[k] -= al * a.vq[k]; }
            grid.sync();
            ++cg_total;
            rn = sqrt(dot(grid, a, a.vr, a.vr, sh));
            bcr_apply(grid, a, a.vr, a.vz);
            const double rz2 = dot(grid, a, a.vr, a.vz, sh), be = rz2 / rz;
            rz = rz2;
            for (unsigned k = tid; k < (unsigned)nf6; k += nth) a.vp[k] = a.vz[k] + be * a.vp[k];
            grid.sync();
        }
        double dm = 0.0;
        for (unsigned k = tid; k < (unsigned)nf6; k += nth) dm = fmax(dm, fabs(a.vx[k]));
        dm = grid_reduce(grid, dm, 1, a.red, sh);
        if (dm <= a.steptol) { status = 2; break; }
        // the candidate: node 0 stays; t + rho, R Exp(phi)
        for (unsigned i = tid; i < (unsigned)a.n; i += nth) {
            const double* x = a.X + 12 * i;
            double* y = a.Xc + 12 * i;
            if (i == 0) { for (int e = 0; e < 12; ++e) y[e] = x[e]; continue; }
            const double* dl = a.vx + 6 * (i - 1);
            double Ex[9];
            so3_exp(dl + 3, Ex);
            mm3(x, Ex, y);
            for (int r = 0; r < 3; ++r) y[9 + r] = x[9 + r] + dl[r];
        }
        grid.sync();
        double gdummy;
        const double Fc = evaluate(grid, a, a.Xc, false, &gdummy, sh);
        if (Fc < F) {
            for (unsigned i = tid; i < (unsigned)a.n; i += nth) {
                for (int e = 0; e < 12; ++e) a.X[12 * i + e] = a.Xc[12 * i + e];
                if (i > 0) a.moved[i] = 1;
            }
            grid.sync();
            lambda /= 10.0;
            F = evaluate(grid, a, a.X, true, &ginf, sh);
        } else {
            lambda *= 10.0;
        }
    }
    // outputs: loop costs at the final poses, the poses (input bits where nothing moved), the report
    double gdummy;
    const double Ff = evaluate(grid, a, a.X, false, &gdummy, sh);
    for (unsigned k = tid; k < (unsigned)a.n_loops; k += nth) a.out_loop_cost[k] = a.ecost[a.n - 1 + k];
    for (unsigned i = tid; i < (unsigned)a.n; i += nth)
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 4; ++c)
                a.out_poses[12 * i + 4 * r + c] = a.moved[i] ? (float)(c < 3 ? a.X[12 * i + 3 * r + c] : a.X[12 * i + 9 + r]) : a.traj[12 * i + 4 * r + c];
    if (tid == 0) {
        a.out_rep[0] = F0; a.out_rep[1] = Ff; a.out_rep[2] = ginf;
        a.out_rep[3] = it; a.out_rep[4] = cg_total; a.out_rep[5] = status;
    }
}

int pose_graph_run(Ctx* c, const bshot_graph_edge* loops, size_t n_loops, const bshot_graph_params* p, float* poses_out, double* loop_cost_out,
                   bshot_graph_report* out) {
    Gmap& g = c->gmap;
    const int n = (int)g.n_updates, L = (int)n_loops, E = n - 1 + L;
    bshot_graph_report rep = {};
    rep.n_nodes = n;
    rep.n_edges = E;
    rep.status = 1;
    if (n <= 1) {   // nothing to optimise: the trajectory as it is
        if (n == 1) BSHOT_CUDA_TRY(cudaMemcpyAsync(poses_out, g.d_traj, sizeof(float) * 12, cudaMemcpyDeviceToHost, c->stream));
        BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
        for (int k = 0; k < L; ++k) if (loop_cost_out) loop_cost_out[k] = 0.0;
        if (out) *out = rep;
        return BSHOT_OK;
    }
    // edges (odometry u = 0..n-2, then the loops) and the node -> edge incidence, in that order per node
    std::vector<int> ef(E), et(E), cnt(n + 1, 0);
    std::vector<float> lT(16 * (size_t)std::max(L, 1));
    for (int u = 0; u < n - 1; ++u) { ef[u] = u; et[u] = u + 1; }
    for (int k = 0; k < L; ++k) { ef[n - 1 + k] = loops[k].from; et[n - 1 + k] = loops[k].to; for (int e = 0; e < 16; ++e) lT[16 * k + e] = loops[k].T[e]; }
    for (int e = 0; e < E; ++e) { ++cnt[ef[e] + 1]; ++cnt[et[e] + 1]; }
    for (int i = 0; i < n; ++i) cnt[i + 1] += cnt[i];
    std::vector<int> inc(2 * (size_t)E), fill(cnt.begin(), cnt.end() - 1);
    for (int e = 0; e < E; ++e) { inc[fill[ef[e]]++] = 2 * e; inc[fill[et[e]]++] = 2 * e + 1; }
    std::vector<int> lvl(1, 0);
    for (int m = n - 1; m > 0; m /= 2) lvl.push_back(lvl.back() + m);
    const int n_levels = (int)lvl.size() - 1;
    const size_t nl = (size_t)lvl.back(), nf = (size_t)n - 1;
    int blocks_per_sm = 0;
    BSHOT_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, pg_solve_kernel, PG_THREADS, 0));
    if (blocks_per_sm < 1) { set_error("bshot_optimize_trajectory: the solver kernel does not fit on an SM"); return BSHOT_E_CUDA; }
    const size_t want = (std::max<size_t>(n, (size_t)E) + PG_THREADS - 1) / PG_THREADS;
    const int grid = (int)std::max<size_t>(1, std::min<size_t>(want, (size_t)blocks_per_sm * c->sm_count));
    // one allocation for the solve, released at the end
    const size_t ints = E * 2 + (n + 1) + 2 * E + (n_levels + 1) + n;
    const size_t dbls = 12 * (size_t)n * 2 + 12 * (size_t)E + 120 * (size_t)E + E + 42 * (size_t)n + 6 * nf * 6 + 36 * nl * 5 + 6 * nl * 2 + grid + L + 8;
    const size_t bytes = sizeof(double) * dbls + sizeof(int) * ints + sizeof(float) * (16 * lT.size() / 16 + 12 * (size_t)n) + 256;
    char* buf = nullptr;
    BSHOT_CUDA_TRY(cudaMalloc((void**)&buf, bytes));
    PgArgs a = {};
    double* dp = reinterpret_cast<double*>(buf);
    auto take = [&](size_t k) { double* r = dp; dp += k; return r; };
    a.X = take(12 * (size_t)n); a.Xc = take(12 * (size_t)n); a.Z = take(12 * (size_t)E); a.EH = take(120 * (size_t)E); a.ecost = take(E);
    a.Dg = take(42 * (size_t)n);
    a.vb = take(6 * nf); a.vx = take(6 * nf); a.vr = take(6 * nf); a.vz = take(6 * nf); a.vp = take(6 * nf); a.vq = take(6 * nf);
    a.LA = take(36 * nl); a.LB = take(36 * nl); a.LC = take(36 * nl); a.W1 = take(36 * nl); a.W2 = take(36 * nl);
    a.LD = take(6 * nl); a.LX = take(6 * nl); a.red = take(grid); a.out_loop_cost = take(std::max(L, 1)); a.out_rep = take(8);
    int* ip = reinterpret_cast<int*>(dp);
    int *d_ef = ip, *d_et = ip + E, *d_ptr = ip + 2 * E, *d_inc = d_ptr + n + 1, *d_lvl = d_inc + 2 * E;
    a.moved = d_lvl + n_levels + 1;
    float* fp = reinterpret_cast<float*>(a.moved + n);
    float* d_lT = fp;
    a.out_poses = fp + lT.size();
    int rc = BSHOT_OK;
    auto up = [&](void* dst, const void* src, size_t nb) { if (rc == BSHOT_OK && nb && cudaMemcpyAsync(dst, src, nb, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) rc = BSHOT_E_CUDA; };
    up(d_ef, ef.data(), sizeof(int) * E);
    up(d_et, et.data(), sizeof(int) * E);
    up(d_ptr, cnt.data(), sizeof(int) * (n + 1));
    up(d_inc, inc.data(), sizeof(int) * 2 * E);
    up(d_lvl, lvl.data(), sizeof(int) * (n_levels + 1));
    up(d_lT, lT.data(), sizeof(float) * lT.size());
    a.n = n; a.n_edges = E; a.n_loops = L; a.n_levels = n_levels;
    a.traj = g.d_traj; a.loop_T = d_lT; a.e_from = d_ef; a.e_to = d_et; a.inc_ptr = d_ptr; a.inc = d_inc; a.lvl_off = d_lvl;
    const double deg = 3.14159265358979323846 / 180.0;
    a.w_odom_t = 1.0 / ((double)p->odom_sigma_mm * p->odom_sigma_mm);
    a.w_odom_r = 1.0 / ((double)p->odom_sigma_deg * deg * p->odom_sigma_deg * deg);
    a.w_loop_t = 1.0 / ((double)p->loop_sigma_mm * p->loop_sigma_mm);
    a.w_loop_r = 1.0 / ((double)p->loop_sigma_deg * deg * p->loop_sigma_deg * deg);
    a.max_it = p->max_iterations; a.max_cg = p->max_cg_iterations;
    a.gtol = p->grad_tolerance; a.steptol = p->step_tolerance; a.cgtol = p->cg_tolerance;
    double h_rep[8] = {0};
    if (rc == BSHOT_OK) {
        void* args[] = {&a};
        const cudaError_t e = cudaLaunchCooperativeKernel((const void*)pg_solve_kernel, grid, PG_THREADS, args, 0, c->stream);
        count_launch(c);
        if (e != cudaSuccess) { set_error("bshot_optimize_trajectory: launch failed: %s", cudaGetErrorString(e)); rc = BSHOT_E_CUDA; }
    }
    if (rc == BSHOT_OK) {
        // the one copy back: poses, loop costs, report
        if (cudaMemcpyAsync(poses_out, a.out_poses, sizeof(float) * 12 * n, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
            (loop_cost_out && L && cudaMemcpyAsync(loop_cost_out, a.out_loop_cost, sizeof(double) * L, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) ||
            cudaMemcpyAsync(h_rep, a.out_rep, sizeof(double) * 8, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess)
            rc = BSHOT_E_CUDA;
    }
    const cudaError_t se = cudaStreamSynchronize(c->stream);
    cudaFree(buf);
    if (rc == BSHOT_OK && se != cudaSuccess) { set_error("bshot_optimize_trajectory: %s", cudaGetErrorString(se)); rc = BSHOT_E_CUDA; }
    if (rc != BSHOT_OK) return rc;
    rep.cost_initial = h_rep[0]; rep.cost_final = h_rep[1]; rep.grad_inf_final = h_rep[2];
    rep.iterations = (int)h_rep[3]; rep.cg_iterations = (int)h_rep[4]; rep.status = (int)h_rep[5];
    if (out) *out = rep;
    return BSHOT_OK;
}

}  // namespace bshot
