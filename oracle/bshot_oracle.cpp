// bshot_oracle.cpp -- CPU ORACLE (test infrastructure only; see bshot_oracle.h header comment).
//
// PARITY: reference-owned arithmetic is pinned to oracle/_ref (the reference header compiled unchanged); the
// PCL-owned arithmetic is UNPINNED (no reference golden vectors exist; PCL is not installable here) -- see bshot_oracle.h.
// Restates, function by function:
//   reference-owned code  : include/bshot_bits.h, src/lidar_odometry.cpp of /root/reference
//   PCL 1.8 algorithms     : SURVEY.md Appendix A (kd-tree radius search, centroid, normal,
//                            SHOT LRF, SHOT352)
// Build: g++ -O3 -march=native -ffp-contract=off -fopenmp (see oracle/Makefile). FP contraction
// is off so that fp32 arithmetic is the plain IEEE sequence written here.
#include "bshot_oracle.h"

#include <algorithm>
#include <cassert>
#include <cmath>
#include <cstring>
#include <limits>
#include <queue>
#include <utility>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

namespace {

struct P3 { float x, y, z; };
typedef std::pair<float, int> DistIdx;  // (squared distance, surface index); operator< = FLANN DistanceIndex

const float kNaN = std::numeric_limits<float>::quiet_NaN();

inline bool finite3(const P3& p) { return std::isfinite(p.x) && std::isfinite(p.y) && std::isfinite(p.z); }

// flann::L2_Simple<float>: result += diff*diff over x,y,z in fp32 (Appendix A.1)
inline float sqdist(const P3& a, const P3& b) {
    float d = a.x - b.x;
    float r = d * d;
    d = a.y - b.y;
    r += d * d;
    d = a.z - b.z;
    r += d * d;
    return r;
}

// Eigen 3/4-float dot as evaluated with SSE3 horizontal adds: (a0*b0 + a1*b1) + a2*b2
inline float dot3f(float ax, float ay, float az, float bx, float by, float bz) {
    return (ax * bx + ay * by) + az * bz;
}

}  // namespace

struct orc_cloud {
    std::vector<P3> pts;
    // uniform grid: points of one cell are stored in ascending surface-index order
    float ox, oy, oz, cell;
    int nx, ny, nz;
    std::vector<int> cell_start;  // ncells + 1
    std::vector<int> cell_pts;    // surface indices

    inline int cx(float v) const { return (int)std::floor((v - ox) / cell); }
    inline int cy(float v) const { return (int)std::floor((v - oy) / cell); }
    inline int cz(float v) const { return (int)std::floor((v - oz) / cell); }

    void build() {
        const size_t n = pts.size();
        float mn[3] = {0, 0, 0}, mx[3] = {0, 0, 0};
        bool first = true;
        for (size_t i = 0; i < n; ++i) {
            if (!finite3(pts[i])) continue;
            const float v[3] = {pts[i].x, pts[i].y, pts[i].z};
            for (int k = 0; k < 3; ++k) {
                if (first || v[k] < mn[k]) mn[k] = v[k];
                if (first || v[k] > mx[k]) mx[k] = v[k];
            }
            first = false;
        }
        cell = 400.0f;
        for (;;) {
            double cells = 1;
            for (int k = 0; k < 3; ++k) cells *= std::floor((mx[k] - mn[k]) / cell) + 1;
            if (cells <= 16e6) break;
            cell *= 1.5f;
        }
        ox = mn[0]; oy = mn[1]; oz = mn[2];
        nx = (int)std::floor((mx[0] - mn[0]) / cell) + 1;
        ny = (int)std::floor((mx[1] - mn[1]) / cell) + 1;
        nz = (int)std::floor((mx[2] - mn[2]) / cell) + 1;
        const size_t ncells = (size_t)nx * ny * nz;
        cell_start.assign(ncells + 1, 0);
        std::vector<int> cid(n, -1);
        for (size_t i = 0; i < n; ++i) {
            if (!finite3(pts[i])) continue;
            int ix = std::min(std::max(cx(pts[i].x), 0), nx - 1);
            int iy = std::min(std::max(cy(pts[i].y), 0), ny - 1);
            int iz = std::min(std::max(cz(pts[i].z), 0), nz - 1);
            cid[i] = (iz * ny + iy) * nx + ix;
            cell_start[cid[i] + 1]++;
        }
        for (size_t c = 0; c < ncells; ++c) cell_start[c + 1] += cell_start[c];
        cell_pts.resize(cell_start[ncells]);
        std::vector<int> cur(cell_start.begin(), cell_start.end() - 1);
        for (size_t i = 0; i < n; ++i)
            if (cid[i] >= 0) cell_pts[cur[cid[i]]++] = (int)i;
    }

    // pcl::KdTreeFLANN::radiusSearch (src/lidar_odometry.cpp:70, include/bshot_bits.h:68; A.1)
    void search(const P3& q, float radius, int max_nn, std::vector<DistIdx>& out) const {
        out.clear();
        if (!finite3(q) || pts.empty()) return;
        const float r2 = (float)((double)radius * (double)radius);  // PCL: static_cast<float>(radius*radius)
        const int qx = cx(q.x), qy = cy(q.y), qz = cz(q.z);
        const int M = (int)std::ceil(radius / cell) + 1;
        if (max_nn <= 0) {
            const int x0 = std::max(qx - M, 0), x1 = std::min(qx + M, nx - 1);
            const int y0 = std::max(qy - M, 0), y1 = std::min(qy + M, ny - 1);
            const int z0 = std::max(qz - M, 0), z1 = std::min(qz + M, nz - 1);
            for (int z = z0; z <= z1; ++z)
                for (int y = y0; y <= y1; ++y) {
                    if (x0 > x1) continue;
                    const int row = (z * ny + y) * nx;
                    for (int k = cell_start[row + x0]; k < cell_start[row + x1 + 1]; ++k) {
                        const int i = cell_pts[k];
                        const float d = sqdist(q, pts[i]);
                        if (d < r2) out.push_back(DistIdx(d, i));  // FLANN RadiusResultSet: dist < radius
                    }
                }
            std::sort(out.begin(), out.end());
            return;
        }
        // FLANN KNNRadiusResultSet: the max_nn nearest hits inside the radius. Ring expansion
        // with a bounded max-heap; exact because ring m covers every point closer than m*cell.
        std::priority_queue<DistIdx> heap;
        for (int m = 0; m <= M; ++m) {
            for (int z = qz - m; z <= qz + m; ++z) {
                if (z < 0 || z >= nz) continue;
                for (int y = qy - m; y <= qy + m; ++y) {
                    if (y < 0 || y >= ny) continue;
                    const bool shell_yz = (std::abs(z - qz) == m) || (std::abs(y - qy) == m);
                    const int row = (z * ny + y) * nx;
                    for (int pass = 0; pass < 2; ++pass) {
                        int xa, xb;
                        if (shell_yz) {
                            if (pass) break;
                            xa = qx - m; xb = qx + m;
                        } else {
                            xa = xb = pass ? qx + m : qx - m;
                            if (pass && m == 0) break;
                        }
                        xa = std::max(xa, 0); xb = std::min(xb, nx - 1);
                        if (xa > xb) continue;
                        for (int k = cell_start[row + xa]; k < cell_start[row + xb + 1]; ++k) {
                            const int i = cell_pts[k];
                            const float d = sqdist(q, pts[i]);
                            if (!(d < r2)) continue;
                            const DistIdx e(d, i);
                            if ((int)heap.size() < max_nn) heap.push(e);
                            else if (e < heap.top()) { heap.pop(); heap.push(e); }
                        }
                    }
                }
            }
            if ((int)heap.size() == max_nn) {
                const double g = (double)m * cell;  // every point closer than g has been visited
                if ((double)heap.top().first < g * g * (1.0 - 1e-5)) break;
            }
        }
        out.resize(heap.size());
        for (size_t k = heap.size(); k-- > 0;) { out[k] = heap.top(); heap.pop(); }
    }
};

namespace {

// ---------------------------------------------------------------------------------------------
// seg-ratio keypoint score, src/lidar_odometry.cpp:61-126
float seg_ratio_point(const orc_cloud& c, int i, float radius, int max_nn, int sr_type,
                      std::vector<DistIdx>& nn) {
    const P3 sp = c.pts[i];
    if (sp.x == 0 && sp.y == 0 && sp.z == 0) return kNaN;  // :63 skip the origin
    c.search(sp, radius, max_nn, nn);
    if (nn.empty()) return kNaN;  // :70 radiusSearch(...) > 0
    // pcl::computeCentroid (:76; Appendix A.2): fp32 running sum in neighbour order / count
    float sx = 0, sy = 0, sz = 0;
    for (size_t j = 0; j < nn.size(); ++j) {
        const P3& p = c.pts[nn[j].second];
        sx += p.x; sy += p.y; sz += p.z;
    }
    const float fn = (float)nn.size();
    const float ctx = sx / fn, cty = sy / fn, ctz = sz / fn;
    const float vx = sp.x - ctx, vy = sp.y - cty, vz = sp.z - ctz;  // :79 ctvec = sp - ct
    float seg;
    if (sr_type == ORC_SR_CV) {  // :83-97
        float pos = 0.0f, neg = 0.0f;
        for (size_t j = 0; j < nn.size(); ++j) {
            const P3& p = c.pts[nn[j].second];
            const float d = dot3f(vx, vy, vz, p.x - sp.x, p.y - sp.y, p.z - sp.z);
            if (d > 0) pos += 1;
            else if (d < 0) neg += 1;
        }
        seg = 1 - std::min(pos, neg) / std::max(pos, neg);
    } else {
        const float ctn = std::sqrt(dot3f(vx, vy, vz, vx, vy, vz));
        float sum = 0;
        for (size_t j = 0; j < nn.size(); ++j) {
            const P3& p = c.pts[nn[j].second];
            const float dx = p.x - sp.x, dy = p.y - sp.y, dz = p.z - sp.z;
            const float dn = std::sqrt(dot3f(dx, dy, dz, dx, dy, dz));
            if (ctn == 0 || dn == 0) continue;  // :103,:114
            const float d = dot3f(vx, vy, vz, dx, dy, dz);
            if (sr_type == ORC_SR_CVS) sum += d;       // :105
            else sum += d / (ctn * dn);                 // :116
        }
        seg = std::fabs(sum) / (float)nn.size();  // :107,:118
    }
    return seg;  // NaN => the reference skips the point (:121)
}

// ---------------------------------------------------------------------------------------------
// pcl::eigen33 / computeRoots / computeRoots2, fp32 (Appendix A.3)
void compute_roots2(float b, float c, float roots[3]) {
    roots[0] = 0.0f;
    float d = (float)(b * b - 4.0 * c);
    if (d < 0.0) d = 0.0f;
    const float sd = std::sqrt(d);
    roots[2] = 0.5f * (b + sd);
    roots[1] = 0.5f * (b - sd);
}

void compute_roots(const float m[9], float roots[3]) {
    const float m00 = m[0], m01 = m[1], m02 = m[2], m11 = m[4], m12 = m[5], m22 = m[8];
    const float c0 = m00 * m11 * m22 + 2.0f * m01 * m02 * m12 - m00 * m12 * m12 - m11 * m02 * m02 -
                     m22 * m01 * m01;
    const float c1 = m00 * m11 - m01 * m01 + m00 * m22 - m02 * m02 + m11 * m22 - m12 * m12;
    const float c2 = m00 + m11 + m22;
    if (std::fabs(c0) < std::numeric_limits<float>::epsilon()) {
        compute_roots2(c2, c1, roots);
        return;
    }
    const float s_inv3 = (float)(1.0 / 3.0);
    const float s_sqrt3 = std::sqrt(3.0f);
    const float c2_over_3 = c2 * s_inv3;
    float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
    if (a_over_3 > 0.0f) a_over_3 = 0.0f;
    const float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
    float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
    if (q > 0.0f) q = 0.0f;
    const float rho = std::sqrt(-a_over_3);
    const float theta = std::atan2(std::sqrt(-q), half_b) * s_inv3;
    const float cos_theta = std::cos(theta);
    const float sin_theta = std::sin(theta);
    roots[0] = c2_over_3 + 2.0f * rho * cos_theta;
    roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
    roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
    if (roots[0] >= roots[1]) std::swap(roots[0], roots[1]);
    if (roots[1] >= roots[2]) {
        std::swap(roots[1], roots[2]);
        if (roots[0] >= roots[1]) std::swap(roots[0], roots[1]);
    }
    if (roots[0] <= 0) compute_roots2(c2, c1, roots);
}

void eigen33_smallest(const float mat[9], float& eigenvalue, float evec[3]) {
    float scale = 0;
    for (int k = 0; k < 9; ++k) scale = std::max(scale, std::fabs(mat[k]));
    if (scale <= std::numeric_limits<float>::min()) scale = 1.0f;
    float s[9];
    for (int k = 0; k < 9; ++k) s[k] = mat[k] / scale;
    float roots[3];
    compute_roots(s, roots);
    eigenvalue = roots[0] * scale;
    s[0] -= roots[0]; s[4] -= roots[0]; s[8] -= roots[0];
    const float* r0 = s; const float* r1 = s + 3; const float* r2 = s + 6;
    float v1[3] = {r0[1] * r1[2] - r0[2] * r1[1], r0[2] * r1[0] - r0[0] * r1[2], r0[0] * r1[1] - r0[1] * r1[0]};
    float v2[3] = {r0[1] * r2[2] - r0[2] * r2[1], r0[2] * r2[0] - r0[0] * r2[2], r0[0] * r2[1] - r0[1] * r2[0]};
    float v3[3] = {r1[1] * r2[2] - r1[2] * r2[1], r1[2] * r2[0] - r1[0] * r2[2], r1[0] * r2[1] - r1[1] * r2[0]};
    const float l1 = dot3f(v1[0], v1[1], v1[2], v1[0], v1[1], v1[2]);
    const float l2 = dot3f(v2[0], v2[1], v2[2], v2[0], v2[1], v2[2]);
    const float l3 = dot3f(v3[0], v3[1], v3[2], v3[0], v3[1], v3[2]);
    const float* v; float l;
    if (l1 >= l2 && l1 >= l3) { v = v1; l = l1; }
    else if (l2 >= l1 && l2 >= l3) { v = v2; l = l2; }
    else { v = v3; l = l3; }
    const float inv = std::sqrt(l);
    for (int k = 0; k < 3; ++k) evec[k] = v[k] / inv;
}

// pcl::computePointNormal(cloud, indices, plane_parameters, curvature) (Appendix A.3): normal + curvature
// of the points `idx[0..n)` of `pts`, in index order; NaN when fewer than 3 indices.  get(i) -> P3.
template <typename Get>
void point_normal_from(Get&& get, int n, float out4[4]) {
    if (n < 3) {  // PCL >= 1.8 computePointNormal guard (version-sensitive, SURVEY 8c)
        out4[0] = out4[1] = out4[2] = out4[3] = kNaN;
        return;
    }
    // computeMeanAndCovarianceMatrix: single pass fp32, 9 accumulators, neighbour order
    float a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int j = 0; j < n; ++j) {
        const P3 p = get(j);
        a[0] += p.x * p.x; a[1] += p.x * p.y; a[2] += p.x * p.z;
        a[3] += p.y * p.y; a[4] += p.y * p.z; a[5] += p.z * p.z;
        a[6] += p.x; a[7] += p.y; a[8] += p.z;
    }
    const float fn = (float)n;
    for (int k = 0; k < 9; ++k) a[k] /= fn;
    float cov[9];
    cov[0] = a[0] - a[6] * a[6];
    cov[1] = a[1] - a[6] * a[7];
    cov[2] = a[2] - a[6] * a[8];
    cov[4] = a[3] - a[7] * a[7];
    cov[5] = a[4] - a[7] * a[8];
    cov[8] = a[5] - a[8] * a[8];
    cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
    float ev, nv[3];
    eigen33_smallest(cov, ev, nv);
    const float eig_sum = cov[0] + cov[4] + cov[8];
    out4[3] = (eig_sum != 0) ? std::fabs(ev / eig_sum) : 0.0f;
    out4[0] = nv[0]; out4[1] = nv[1]; out4[2] = nv[2];
}

// pcl::computePointNormal + flipNormalTowardsViewpoint(0,0,0)   (include/bshot_bits.h:66-87)
void normal_point(const orc_cloud& c, const P3& q, float radius, int max_nn, float out4[4],
                  std::vector<DistIdx>& nn) {
    if (finite3(q)) c.search(q, radius, max_nn, nn); else nn.clear();
    if (nn.empty()) {  // :67-74
        out4[0] = out4[1] = out4[2] = out4[3] = kNaN;
        return;
    }
    point_normal_from([&](int j) { return c.pts[nn[j].second]; }, (int)nn.size(), out4);
    if (nn.size() < 3) return;
    // flipNormalTowardsViewpoint(point, 0,0,0, ...)
    float* n = out4;
    const float vx = 0.0f - q.x, vy = 0.0f - q.y, vz = 0.0f - q.z;
    const float cos_theta = (vx * n[0] + vy * n[1] + vz * n[2]);
    if (cos_theta < 0) { n[0] *= -1; n[1] *= -1; n[2] *= -1; }
}

// ---------------------------------------------------------------------------------------------
// symmetric 3x3 eigen decomposition in double (cyclic Jacobi), ascending eigenvalues.
// Stands in for Eigen::SelfAdjointEigenSolver<Matrix3d> (Appendix A.4); checked against
// numpy.linalg.eigh in tests/test_oracle_units.py.
void eigh3(const double m[9], double w[3], double V[9]) {
    double a[3][3] = {{m[0], m[1], m[2]}, {m[1], m[4], m[5]}, {m[2], m[5], m[8]}};
    double v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int sweep = 0; sweep < 64; ++sweep) {
        const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
        const double diag = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2];
        if (off <= 1e-40 * diag || off == 0.0) break;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                if (a[p][q] == 0.0) continue;
                const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double cs = 1.0 / std::sqrt(t * t + 1.0), sn = t * cs;
                for (int k = 0; k < 3; ++k) {  // A <- A J
                    const double akp = a[k][p], akq = a[k][q];
                    a[k][p] = cs * akp - sn * akq;
                    a[k][q] = sn * akp + cs * akq;
                }
                for (int k = 0; k < 3; ++k) {  // A <- J^T A
                    const double apk = a[p][k], aqk = a[q][k];
                    a[p][k] = cs * apk - sn * aqk;
                    a[q][k] = sn * apk + cs * aqk;
                }
                for (int k = 0; k < 3; ++k) {
                    const double vkp = v[k][p], vkq = v[k][q];
                    v[k][p] = cs * vkp - sn * vkq;
                    v[k][q] = sn * vkp + cs * vkq;
                }
            }
    }
    int order[3] = {0, 1, 2};
    std::sort(order, order + 3, [&](int i, int j) { return a[i][i] < a[j][j]; });
    for (int c = 0; c < 3; ++c) {
        w[c] = a[order[c]][order[c]];
        for (int r = 0; r < 3; ++r) V[r * 3 + c] = v[r][order[c]];
    }
}

// SHOTLocalReferenceFrameEstimation::getLocalRF (Appendix A.4). nn = sorted radius search
bool lrf_point(const orc_cloud& c, const P3& central, float radius, const std::vector<DistIdx>& nn,
               float rf[9], int* valid_out) {
    for (int k = 0; k < 9; ++k) rf[k] = kNaN;
    std::vector<double> vij;
    vij.reserve(nn.size() * 3);
    double cov[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    double sum = 0.0;
    int valid = 0;
    const double R = (double)radius;
    for (size_t j = 0; j < nn.size(); ++j) {
        const P3& pt = c.pts[nn[j].second];
        if (pt.x == central.x && pt.y == central.y && pt.z == central.z) continue;
        const double vx = (double)(pt.x - central.x), vy = (double)(pt.y - central.y), vz = (double)(pt.z - central.z);
        vij.push_back(vx); vij.push_back(vy); vij.push_back(vz);
        const double w = R - std::sqrt((double)nn[j].first);
        cov[0] += w * (vx * vx); cov[1] += w * (vx * vy); cov[2] += w * (vx * vz);
        cov[4] += w * (vy * vy); cov[5] += w * (vy * vz); cov[8] += w * (vz * vz);
        sum += w;
        ++valid;
    }
    if (valid_out) *valid_out = valid;
    if (valid < 5) return false;
    cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
    for (int k = 0; k < 9; ++k) cov[k] /= sum;
    double ev[3], V[9];
    eigh3(cov, ev, V);
    if (!std::isfinite(ev[0]) || !std::isfinite(ev[1]) || !std::isfinite(ev[2])) return false;
    double v1[3] = {V[2], V[5], V[8]};  // largest eigenvalue  -> x axis
    double v3[3] = {V[0], V[3], V[6]};  // smallest eigenvalue -> z axis
    int plus_n = 0, plus_t = 0;
    for (int ne = 0; ne < valid; ++ne) {
        const double* v = &vij[3 * ne];
        if (v[0] * v1[0] + v[1] * v1[1] + v[2] * v1[2] >= 0) plus_t++;
        if (v[0] * v3[0] + v[1] * v3[1] + v[2] * v3[2] >= 0) plus_n++;
    }
    double* axes[2] = {v1, v3};
    int plus[2] = {plus_t, plus_n};
    for (int a = 0; a < 2; ++a) {
        int s = 2 * plus[a] - valid;
        double* ax = axes[a];
        if (s == 0) {  // exact tie: 5 neighbours around the median position, strictly positive votes
            const int points = 5, median = valid / 2;
            for (int i = -points / 2; i <= points / 2; ++i) {
                const double* v = &vij[3 * (median - i)];
                if (v[0] * ax[0] + v[1] * ax[1] + v[2] * ax[2] > 0) s++;
            }
            if (s < points / 2 + 1) { ax[0] = -ax[0]; ax[1] = -ax[1]; ax[2] = -ax[2]; }
        } else if (s < 0) { ax[0] = -ax[0]; ax[1] = -ax[1]; ax[2] = -ax[2]; }
    }
    const float x[3] = {(float)v1[0], (float)v1[1], (float)v1[2]};
    const float z[3] = {(float)v3[0], (float)v3[1], (float)v3[2]};
    rf[0] = x[0]; rf[1] = x[1]; rf[2] = x[2];
    rf[6] = z[0]; rf[7] = z[1]; rf[8] = z[2];
    // rf.row(1) = rf.row(2).cross(rf.row(0)) in fp32
    rf[3] = z[1] * x[2] - z[2] * x[1];
    rf[4] = z[2] * x[0] - z[0] * x[2];
    rf[5] = z[0] * x[1] - z[1] * x[0];
    return true;
}

// SHOTEstimation::computePointSHOT = createBinDistanceShape + interpolateSingleChannel +
// normalizeHistogram (Appendix A.5). normals4 indexed by surface index.
const double PST_PI = 3.1415926535897932384626433832795;
const double PST_RAD_45 = 0.78539816339744830961566084581988;
const double PST_RAD_90 = 1.5707963267948966192313216916398;
const double PST_RAD_135 = 2.3561944901923449288469825374596;
const double PST_RAD_PI_7_8 = 2.7488935718910690836548129603691;

void shot_point(const orc_cloud& c, const P3& central, float radius, const std::vector<DistIdx>& nn,
                const float* normals4, const float rf[9], float shot[352]) {
    const int nr_bins = 10;
    const int max_sectors = 32;
    if (nn.size() < 5) {
        for (int k = 0; k < 352; ++k) shot[k] = kNaN;
        return;
    }
    for (int k = 0; k < 352; ++k) shot[k] = 0.0f;
    const double radius3_4 = ((double)radius * 3) / 4;
    const double radius1_4 = (double)radius / 4;
    const double radius1_2 = (double)radius / 2;
    for (size_t j = 0; j < nn.size(); ++j) {
        const int s = nn[j].second;
        const float* nv = normals4 + 4 * (size_t)s;
        if (!std::isfinite(nv[0]) || !std::isfinite(nv[1]) || !std::isfinite(nv[2])) continue;
        double cosine = (double)dot3f(nv[0], nv[1], nv[2], rf[6], rf[7], rf[8]);
        if (cosine > 1.0) cosine = 1.0;
        if (cosine < -1.0) cosine = -1.0;
        double bin = ((1.0 + cosine) * nr_bins) / 2;

        const P3& pt = c.pts[s];
        const float dx = pt.x - central.x, dy = pt.y - central.y, dz = pt.z - central.z;
        const double distance = std::sqrt((double)nn[j].first);
        if (std::fabs(distance) < 1e-15) continue;  // areEquals(distance, 0.0)
        double xr = (double)dot3f(dx, dy, dz, rf[0], rf[1], rf[2]);
        double yr = (double)dot3f(dx, dy, dz, rf[3], rf[4], rf[5]);
        double zr = (double)dot3f(dx, dy, dz, rf[6], rf[7], rf[8]);
        if (std::fabs(yr) < 1E-30) yr = 0;
        if (std::fabs(xr) < 1E-30) xr = 0;
        if (std::fabs(zr) < 1E-30) zr = 0;
        const unsigned char bit4 = ((yr > 0) || ((yr == 0.0) && (xr < 0))) ? 1 : 0;
        const unsigned char bit3 = (unsigned char)(((xr > 0) || ((xr == 0.0) && (yr > 0))) ? !bit4 : bit4);
        int desc_index = (bit4 << 3) + (bit3 << 2);
        desc_index = desc_index << 1;
        if ((xr * yr > 0) || (xr == 0.0)) desc_index += (std::fabs(xr) >= std::fabs(yr)) ? 0 : 4;
        else desc_index += (std::fabs(xr) > std::fabs(yr)) ? 4 : 0;
        desc_index += zr > 0 ? 1 : 0;
        desc_index += (distance > radius1_2) ? 2 : 0;

        const int step_index = (int)std::floor(bin + 0.5);
        const int volume_index = desc_index * (nr_bins + 1);
        bin -= step_index;
        double w = (1 - std::fabs(bin));
        if (bin > 0) shot[volume_index + ((step_index + 1) % nr_bins)] += (float)bin;
        else shot[volume_index + ((step_index - 1 + nr_bins) % nr_bins)] += -(float)bin;

        if (distance > radius1_2) {
            const double rd = (distance - radius3_4) / radius1_2;
            if (distance > radius3_4) w += 1 - rd;
            else { w += 1 + rd; shot[(desc_index - 2) * (nr_bins + 1) + step_index] -= (float)rd; }
        } else {
            const double rd = (distance - radius1_4) / radius1_2;
            if (distance < radius1_4) w += 1 + rd;
            else { w += 1 - rd; shot[(desc_index + 2) * (nr_bins + 1) + step_index] += (float)rd; }
        }

        double inc_cos = zr / distance;
        if (inc_cos < -1.0) inc_cos = -1.0;
        if (inc_cos > 1.0) inc_cos = 1.0;
        const double inc = std::acos(inc_cos);
        if (inc > PST_RAD_90 || (std::fabs(inc - PST_RAD_90) < 1e-30 && zr <= 0)) {
            const double id = (inc - PST_RAD_135) / PST_RAD_90;
            if (inc > PST_RAD_135) w += 1 - id;
            else { w += 1 + id; shot[(desc_index + 1) * (nr_bins + 1) + step_index] -= (float)id; }
        } else {
            const double id = (inc - PST_RAD_45) / PST_RAD_90;
            if (inc < PST_RAD_45) w += 1 + id;
            else { w += 1 - id; shot[(desc_index - 1) * (nr_bins + 1) + step_index] += (float)id; }
        }

        if (yr != 0.0 || xr != 0.0) {
            const double azimuth = std::atan2(yr, xr);
            const int sel = desc_index >> 2;
            double ad = (azimuth - (-PST_RAD_PI_7_8 + PST_RAD_45 * sel)) / PST_RAD_45;
            ad = std::max(-0.5, std::min(ad, 0.5));
            if (ad > 0) {
                w += 1 - ad;
                const int ii = (desc_index + 4) % max_sectors;
                shot[ii * (nr_bins + 1) + step_index] += (float)ad;
            } else {
                const int ii = (desc_index - 4 + max_sectors) % max_sectors;
                w += 1 + ad;
                shot[ii * (nr_bins + 1) + step_index] -= (float)ad;
            }
        }
        shot[volume_index + step_index] += (float)w;
    }
    double acc = 0;
    for (int k = 0; k < 352; ++k) acc += shot[k] * shot[k];  // float product, double accumulate
    acc = std::sqrt(acc);
    const float f = (float)acc;
    for (int k = 0; k < 352; ++k) shot[k] /= f;
    (void)PST_PI;
}

// include/bshot_bits.h:144-278 : one group of 4 floats -> 4 bits (bit k = element k)
inline unsigned bshot_nibble(const float* vec) {
    const float sum = vec[0] + vec[1] + vec[2] + vec[3];  // :164 float, left to right
    const double t = 0.9 * (sum);                         // :171 double literal
    if (vec[0] == 0 && vec[1] == 0 && vec[2] == 0 && vec[3] == 0) return 0x0;
    else if (vec[0] > t) return 0x1;
    else if (vec[1] > t) return 0x2;
    else if (vec[2] > t) return 0x4;
    else if (vec[3] > t) return 0x8;
    else if ((vec[0] + vec[1]) > t) return 0x3;
    else if ((vec[1] + vec[2]) > t) return 0x6;
    else if ((vec[2] + vec[3]) > t) return 0xC;
    else if ((vec[0] + vec[3]) > t) return 0x9;
    else if ((vec[1] + vec[3]) > t) return 0xA;
    else if ((vec[0] + vec[2]) > t) return 0x5;
    else if ((vec[0] + vec[1] + vec[2]) > t) return 0x7;
    else if ((vec[1] + vec[2] + vec[3]) > t) return 0xE;
    else if ((vec[0] + vec[2] + vec[3]) > t) return 0xD;
    else if ((vec[0] + vec[1] + vec[3]) > t) return 0xB;
    return 0xF;
}

inline int hamming352(const uint64_t* a, const uint64_t* b) {
    int d = 0;
    for (int k = 0; k < 6; ++k) d += __builtin_popcountll(a[k] ^ b[k]);
    return d;
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

orc_cloud* orc_cloud_create(const float* xyz, size_t n, size_t stride_floats) {
    orc_cloud* c = new orc_cloud();
    c->pts.resize(n);
    for (size_t i = 0; i < n; ++i) {
        c->pts[i].x = xyz[i * stride_floats + 0];
        c->pts[i].y = xyz[i * stride_floats + 1];
        c->pts[i].z = xyz[i * stride_floats + 2];
    }
    c->build();
    return c;
}

void orc_cloud_destroy(orc_cloud* c) { delete c; }
size_t orc_cloud_size(const orc_cloud* c) { return c->pts.size(); }

int orc_radius_search(const orc_cloud* c, const float q[3], float radius, int max_nn, int* out_idx,
                      float* out_sqd, int cap) {
    std::vector<DistIdx> nn;
    const P3 p = {q[0], q[1], q[2]};
    c->search(p, radius, max_nn, nn);
    for (int k = 0; k < (int)nn.size() && k < cap; ++k) {
        if (out_idx) out_idx[k] = nn[k].second;
        if (out_sqd) out_sqd[k] = nn[k].first;
    }
    return (int)nn.size();
}

void orc_seg_ratio(const orc_cloud* c, float radius, int max_nn, int sr_type, float* ratio_out,
                   int threads) {
    const int n = (int)c->pts.size();
    const int nt = nthreads(threads);
    (void)nt;
#pragma omp parallel num_threads(nt)
    {
        std::vector<DistIdx> nn;
#pragma omp for schedule(dynamic, 64)
        for (int i = 0; i < n; ++i) ratio_out[i] = seg_ratio_point(*c, i, radius, max_nn, sr_type, nn);
    }
}

typedef std::pair<int, float> IdxRatioPair;
static bool comparator(const IdxRatioPair& l, const IdxRatioPair& r) { return l.second < r.second; }

int orc_select_keypoints(const float* ratio, size_t n, int top_k, int tie_mode, int* idx_out,
                         float* ratio_out) {
    std::vector<IdxRatioPair> sr;
    sr.reserve(n);
    for (size_t i = 0; i < n; ++i)
        if (!std::isnan(ratio[i])) sr.push_back(IdxRatioPair((int)i, ratio[i]));  // :121-123
    if (tie_mode == ORC_TIE_STDSORT)
        std::sort(sr.begin(), sr.end(), comparator);  // :131 (tie order = libstdc++ introsort)
    else  // deterministic: ascending ratio, ties by DESCENDING index => last K prefers low indices
        std::sort(sr.begin(), sr.end(), [](const IdxRatioPair& l, const IdxRatioPair& r) {
            return l.second < r.second || (l.second == r.second && l.first > r.first);
        });
    const size_t k = std::min((size_t)top_k, sr.size());  // :138-153
    for (size_t j = 0; j < k; ++j) {
        idx_out[j] = sr[sr.size() - k + j].first;
        if (ratio_out) ratio_out[j] = sr[sr.size() - k + j].second;
    }
    return (int)k;
}

void orc_normals(const orc_cloud* c, const float* q_xyz, size_t nq, float radius, int max_nn,
                 float* normal4_out, int threads) {
    const int nt = nthreads(threads);
    (void)nt;
#pragma omp parallel num_threads(nt)
    {
        std::vector<DistIdx> nn;
#pragma omp for schedule(dynamic, 16)
        for (long long i = 0; i < (long long)nq; ++i) {
            const P3 q = {q_xyz[3 * i], q_xyz[3 * i + 1], q_xyz[3 * i + 2]};
            normal_point(*c, q, radius, max_nn, normal4_out + 4 * i, nn);
        }
    }
}

void orc_point_normal_indices(const float* xyz, size_t n, size_t stride_floats, const int* idx, int n_idx, float out4[4]) {
    (void)n;
    point_normal_from([&](int j) {
        const float* p = xyz + (size_t)idx[j] * stride_floats;
        const P3 r = {p[0], p[1], p[2]};
        return r;
    }, n_idx, out4);
}

void orc_lrf(const orc_cloud* c, const float* kp_xyz, size_t nk, float radius, float* rf9_out,
             int* valid_nn_out, int threads) {
    const int nt = nthreads(threads);
    (void)nt;
#pragma omp parallel num_threads(nt)
    {
        std::vector<DistIdx> nn;
#pragma omp for schedule(dynamic, 4)
        for (long long i = 0; i < (long long)nk; ++i) {
            const P3 q = {kp_xyz[3 * i], kp_xyz[3 * i + 1], kp_xyz[3 * i + 2]};
            int valid = 0;
            c->search(q, radius, 0, nn);
            lrf_point(*c, q, radius, nn, rf9_out + 9 * i, &valid);
            if (valid_nn_out) valid_nn_out[i] = valid;
        }
    }
}

long long orc_shot(const orc_cloud* c, const float* kp_xyz, size_t nk, float radius,
                   const float* normals4, const float* rf9_in, float* shot352_out, float* rf9_out,
                   int* nn_out, int threads) {
    const int nt = nthreads(threads);
    (void)nt;
    long long total = 0;
#pragma omp parallel num_threads(nt) reduction(+ : total)
    {
        std::vector<DistIdx> nn;
        float shot[352];
#pragma omp for schedule(dynamic, 4)
        for (long long i = 0; i < (long long)nk; ++i) {
            const P3 q = {kp_xyz[3 * i], kp_xyz[3 * i + 1], kp_xyz[3 * i + 2]};
            float rf[9];
            c->search(q, radius, 0, nn);
            total += (long long)nn.size();
            if (nn_out) nn_out[i] = (int)nn.size();
            if (rf9_in) std::memcpy(rf, rf9_in + 9 * i, sizeof(rf));
            else lrf_point(*c, q, radius, nn, rf, nullptr);
            const bool lrf_nan = !std::isfinite(rf[0]) || !std::isfinite(rf[3]) || !std::isfinite(rf[6]);
            if (!finite3(q) || lrf_nan || nn.empty()) {  // SHOTEstimationOMP::computeFeature NaN branch
                for (int k = 0; k < 352; ++k) shot[k] = kNaN;
                for (int k = 0; k < 9; ++k) rf[k] = kNaN;
            } else {
                shot_point(*c, q, radius, nn, normals4, rf, shot);
            }
            if (shot352_out) std::memcpy(shot352_out + 352 * i, shot, sizeof(shot));
            if (rf9_out) std::memcpy(rf9_out + 9 * i, rf, sizeof(rf));
        }
    }
    return total;
}

void orc_bshot(const float* shot352, size_t nk, uint64_t* bits6_out) {
    for (size_t i = 0; i < nk; ++i) {
        uint64_t w[6] = {0, 0, 0, 0, 0, 0};
        for (int j = 0; j < 88; ++j) {
            const uint64_t nib = bshot_nibble(shot352 + 352 * i + 4 * j);
            w[(4 * j) >> 6] |= nib << ((4 * j) & 63);  // std::bitset<352>: bit b -> word b/64, bit b%64
        }
        std::memcpy(bits6_out + 6 * i, w, sizeof(w));
    }
}

void orc_match(const uint64_t* q, size_t nq, const uint64_t* t, size_t nt_, int* left_idx,
               int* left_dist, int* left_idx2, int* left_dist2, int* right_idx, int threads) {
    const int nthr = nthreads(threads);
    (void)nthr;
    const long long nQ = (long long)nq, nT = (long long)nt_;
    if (left_idx || left_dist || left_idx2 || left_dist2) {
#pragma omp parallel for schedule(static) num_threads(nthr)
        for (long long i = 0; i < nQ; ++i) {  // :217-225, minVect strict '<' => first minimum
            int b1 = -1, d1 = 1 << 30, b2 = -1, d2 = 1 << 30;
            for (long long k = 0; k < nT; ++k) {
                const int d = hamming352(q + 6 * i, t + 6 * k);
                if (d < d1) { b2 = b1; d2 = d1; b1 = (int)k; d1 = d; }
                else if (d < d2) { b2 = (int)k; d2 = d; }
            }
            if (left_idx) left_idx[i] = b1;
            if (left_dist) left_dist[i] = (b1 >= 0) ? d1 : -1;
            if (left_idx2) left_idx2[i] = b2;
            if (left_dist2) left_dist2[i] = (b2 >= 0) ? d2 : -1;
        }
    }
    if (right_idx) {
#pragma omp parallel for schedule(static) num_threads(nthr)
        for (long long i = 0; i < nT; ++i) {  // :226-232
            int b1 = -1, d1 = 1 << 30;
            for (long long k = 0; k < nQ; ++k) {
                const int d = hamming352(t + 6 * i, q + 6 * k);
                if (d < d1) { b1 = (int)k; d1 = d; }
            }
            right_idx[i] = b1;
        }
    }
}

int orc_mutual(const int* left_idx, size_t nq, const int* right_idx, int* pairs_out) {
    int n = 0;
    for (size_t i = 0; i < nq; ++i)
        if (left_idx[i] >= 0 && right_idx[left_idx[i]] == (int)i) {  // :234-242
            pairs_out[2 * n] = (int)i;
            pairs_out[2 * n + 1] = left_idx[i];
            ++n;
        }
    return n;
}

long long orc_compute_descriptors(const orc_cloud* c, const float* kp_xyz, size_t nk, float radius,
                                  int max_nn, int mode, uint64_t* bits6_out, float* shot352_out,
                                  float* rf9_out, float* normals4_out, int threads) {
    const size_t n = c->pts.size();
    std::vector<float> normals(4 * n, 0.0f);  // pcl::Normal default = (0,0,0), curvature 0
    if (mode == 0) {
        // include/bshot_bits.h:58-59,79-81: normal of keypoint ordinal idx lands at index idx
        std::vector<float> kn(4 * nk);
        orc_normals(c, kp_xyz, nk, radius, max_nn, kn.data(), threads);
        std::memcpy(normals.data(), kn.data(), sizeof(float) * 4 * std::min(nk, n));
    } else {
        std::vector<float> q(3 * n);
        for (size_t i = 0; i < n; ++i) { q[3 * i] = c->pts[i].x; q[3 * i + 1] = c->pts[i].y; q[3 * i + 2] = c->pts[i].z; }
        orc_normals(c, q.data(), n, radius, max_nn, normals.data(), threads);
    }
    if (normals4_out) std::memcpy(normals4_out, normals.data(), sizeof(float) * 4 * n);
    std::vector<float> shot(352 * nk);
    const long long total = orc_shot(c, kp_xyz, nk, radius, normals.data(), nullptr, shot.data(), rf9_out, nullptr, threads);
    if (shot352_out) std::memcpy(shot352_out, shot.data(), sizeof(float) * 352 * nk);
    if (bits6_out) orc_bshot(shot.data(), nk, bits6_out);
    return total;
}

// ---------------------------------------------------------------------------------------------
// global keypoint map: src/keypoint.cpp:23-32 (10 mm snap), src/mymap.cpp:4-26 (addKeypoint), :28-74 (getKeypoints),
// :103-112 (getBlockID), src/lidar_odometry.cpp:343-358 (updateMap: every keypoint of the frame in order, R * p + T).
// Order inside a block: insertion order (the reference iterates an unordered_map: implementation defined).
struct orc_map_entry { float x, y, z, ratio; uint64_t d[6]; };
struct orc_map {
    std::vector<std::pair<uint64_t, std::vector<orc_map_entry>>> blocks;  // creation order; lookups are linear (test sizes)
    std::vector<orc_map_entry>* find(uint64_t id) {
        for (auto& b : blocks) if (b.first == id) return &b.second;
        return nullptr;
    }
};
static uint64_t map_block_id(float x, float y, float z) {
    const int prec = 10000;
    const float v[3] = {x, y, z};
    uint64_t key = 0;
    for (int a = 0; a < 3; ++a) {
        const int g = int(std::round(v[a] / prec)) * prec;
        key = (key << 21) | ((uint64_t)(int64_t)g & 0x1FFFFFull);
    }
    return key;
}

orc_map* orc_map_create() { return new orc_map(); }
void orc_map_destroy(orc_map* m) { delete m; }
size_t orc_map_size(const orc_map* m) {
    size_t n = 0;
    for (auto& b : m->blocks) n += b.second.size();
    return n;
}

void orc_map_add(orc_map* m, const float* xyz, const float* ratio, const uint64_t* desc, size_t n, const float* pose12) {
    for (size_t i = 0; i < n; ++i) {
        float x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
        if (pose12) {  // kp_pos = R * kp_pos + T (src/lidar_odometry.cpp:351)
            const float px = x, py = y, pz = z;
            x = ((pose12[0] * px + pose12[1] * py) + pose12[2] * pz) + pose12[3];
            y = ((pose12[4] * px + pose12[5] * py) + pose12[6] * pz) + pose12[7];
            z = ((pose12[8] * px + pose12[9] * py) + pose12[10] * pz) + pose12[11];
        }
        orc_map_entry e;  // Keypoint::createKeypoint: int(trunc(pos / prec)) * prec, prec = 10
        e.x = (float)(int(std::trunc(x / 10)) * 10);
        e.y = (float)(int(std::trunc(y / 10)) * 10);
        e.z = (float)(int(std::trunc(z / 10)) * 10);
        e.ratio = ratio[i];
        std::memcpy(e.d, desc + 6 * i, 48);
        const uint64_t id = map_block_id(e.x, e.y, e.z);
        std::vector<orc_map_entry>* blk = m->find(id);
        if (!blk) {  // :7-11 new block
            m->blocks.push_back(std::make_pair(id, std::vector<orc_map_entry>(1, e)));
            continue;
        }
        bool candidate = true;  // :15-21
        for (auto& k : *blk) {
            const float dx = e.x - k.x, dy = e.y - k.y, dz = e.z - k.z;
            if (std::sqrt(dot3f(dx, dy, dz, dx, dy, dz)) < 800 && e.ratio <= k.ratio) candidate = false;
        }
        if (!candidate) continue;
        bool over = false;      // :23 keypoints_[block][position] = keypoint
        for (auto& k : *blk)
            if (k.x == e.x && k.y == e.y && k.z == e.z) { k = e; over = true; break; }
        if (!over) blk->push_back(e);
    }
}

size_t orc_map_get(orc_map* m, const float pos[3], float range, float* xyz_out, uint64_t* desc_out, size_t cap) {
    const int prec = 10000;
    int lo[3], hi[3];
    for (int a = 0; a < 3; ++a) {
        lo[a] = int(std::round((pos[a] - range) / prec)) * prec;
        hi[a] = int(std::round((pos[a] + range) / prec)) * prec;
    }
    size_t n = 0;
    for (int x = lo[0]; x <= hi[0]; x += prec)
        for (int y = lo[1]; y <= hi[1]; y += prec)
            for (int z = lo[2]; z <= hi[2]; z += prec) {
                std::vector<orc_map_entry>* blk = m->find(map_block_id((float)x, (float)y, (float)z));
                if (!blk) continue;
                for (auto& k : *blk) {
                    if (n < cap) {
                        if (xyz_out) { xyz_out[3 * n] = k.x; xyz_out[3 * n + 1] = k.y; xyz_out[3 * n + 2] = k.z; }
                        if (desc_out) std::memcpy(desc_out + 6 * n, k.d, 48);
                    }
                    ++n;
                }
            }
    return n;
}

// ---------------------------------------------------------------------------------------------
// RANSAC correspondence rejection: src/lidar_odometry.cpp:251-261 -> PCL 1.8 CorrespondenceRejectorSampleConsensus =
// RandomSampleConsensus::computeModel over SampleConsensusModelRegistration (restated from the published PCL 1.8 sources;
// PCL is not installable here: UNPINNED like the rest of the PCL arithmetic).  Sequential, exactly as PCL runs it.
namespace {
struct OrcMt19937 {
    uint32_t s[624]; int idx;
    explicit OrcMt19937(uint32_t seed) { s[0] = seed; for (int i = 1; i < 624; ++i) s[i] = 1812433253u * (s[i - 1] ^ (s[i - 1] >> 30)) + (uint32_t)i; idx = 624; }
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

// Eigen::JacobiSVD stand-in: one-sided Jacobi (Hestenes) in double, singular values descending; a column of U whose
// singular value is exactly zero is left zero (the callers complete the bases)
void orc_svd3(const double a_in[9], double U[9], double sv[3], double V[9]) {
    double a[3][3], v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) a[r][c] = a_in[3 * r + c];
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                double alpha = 0, beta = 0, gamma = 0;
                for (int r = 0; r < 3; ++r) { alpha += a[r][p] * a[r][p]; beta += a[r][q] * a[r][q]; gamma += a[r][p] * a[r][q]; }
                if (gamma == 0.0) continue;
                if (gamma * gamma <= 1e-30 * (alpha * beta)) continue;
                off += gamma * gamma;
                const double zeta = (beta - alpha) / (2.0 * gamma);
                const double t = (zeta >= 0 ? 1.0 : -1.0) / (std::fabs(zeta) + std::sqrt(1.0 + zeta * zeta));
                const double c = 1.0 / std::sqrt(1.0 + t * t), sn = c * t;
                for (int r = 0; r < 3; ++r) {
                    const double x = a[r][p], y = a[r][q];
                    a[r][p] = c * x - sn * y; a[r][q] = sn * x + c * y;
                    const double vx = v[r][p], vy = v[r][q];
                    v[r][p] = c * vx - sn * vy; v[r][q] = sn * vx + c * vy;
                }
            }
        if (off == 0.0) break;
    }
    double n[3]; int o[3] = {0, 1, 2};
    for (int c = 0; c < 3; ++c) n[c] = std::sqrt(a[0][c] * a[0][c] + a[1][c] * a[1][c] + a[2][c] * a[2][c]);
    if (n[o[0]] < n[o[1]]) std::swap(o[0], o[1]);
    if (n[o[1]] < n[o[2]]) std::swap(o[1], o[2]);
    if (n[o[0]] < n[o[1]]) std::swap(o[0], o[1]);
    for (int k = 0; k < 3; ++k) {
        sv[k] = n[o[k]];
        for (int r = 0; r < 3; ++r) { V[3 * r + k] = v[r][o[k]]; U[3 * r + k] = (sv[k] > 0.0) ? a[r][o[k]] / sv[k] : 0.0; }
    }
}

// R for a cross-covariance of rank 0 or 1, Sigma = s0 u0 v0^T: a deterministic proper rotation with R v0 = u0 (any such R
// is optimal).  u0.v0 >= 0: the minimal rotation; u0.v0 < 0: a half-turn about a = v0 x e_j (e_j: the axis of v0's smallest
// component), then the minimal rotation from -v0 to u0.  Rank 0: the identity, as pcl::umeyama gives for Sigma = 0.
// pcl::umeyama's own rank <= 1 result depends on Eigen's SVD internals (and can be improper): a deliberate difference.
// Rank 0 is s0 at or below orc_noise_floor: the rounding noise of Sigma when one side is a single point (the rounded
// centroid does not return that point, so Sigma is tiny but not zero), twice gamma_{k+3} (Ad (Ap + 2 As) + As (Aq + 2 Ad))
// with A* the means of the 1-norms of the sources, targets, centred sources and centred targets.
double orc_noise_floor(double P, double Q, double S, double D, double n, double k, double u) {
    const double ap = P / n, aq = Q / n, as = S / n, ad = D / n;
    return 2.0 * ((k + 3.0) * u) * (ad * (ap + 2.0 * as) + as * (aq + 2.0 * ad));
}

void orc_rotation_min(const double v[3], const double u[3], double R[9]) {
    const double c = (v[0] * u[0] + v[1] * u[1]) + v[2] * u[2];
    const double k[3] = {v[1] * u[2] - v[2] * u[1], v[2] * u[0] - v[0] * u[2], v[0] * u[1] - v[1] * u[0]};
    const double f = 1.0 / (1.0 + c);
    R[0] = c + k[0] * k[0] * f; R[1] = k[0] * k[1] * f - k[2]; R[2] = k[0] * k[2] * f + k[1];
    R[3] = k[1] * k[0] * f + k[2]; R[4] = c + k[1] * k[1] * f; R[5] = k[1] * k[2] * f - k[0];
    R[6] = k[2] * k[0] * f - k[1]; R[7] = k[2] * k[1] * f + k[0]; R[8] = c + k[2] * k[2] * f;
}

void orc_rotation_rank01(const double U[9], const double V[9], bool rank0, double R[9]) {
    if (rank0) {
        for (int e = 0; e < 9; ++e) R[e] = (e % 4 == 0) ? 1.0 : 0.0;
        return;
    }
    const double u[3] = {U[0], U[3], U[6]}, v[3] = {V[0], V[3], V[6]};
    if ((v[0] * u[0] + v[1] * u[1]) + v[2] * u[2] >= 0.0) { orc_rotation_min(v, u, R); return; }
    const double ax[3] = {std::fabs(v[0]), std::fabs(v[1]), std::fabs(v[2])};
    const int j = (ax[0] <= ax[1] && ax[0] <= ax[2]) ? 0 : (ax[1] <= ax[2] ? 1 : 2);
    double a[3] = {0.0, 0.0, 0.0};
    if (j == 0) { a[1] = v[2]; a[2] = -v[1]; }
    else if (j == 1) { a[0] = -v[2]; a[2] = v[0]; }
    else { a[0] = v[1]; a[1] = -v[0]; }
    const double na = std::sqrt((a[0] * a[0] + a[1] * a[1]) + a[2] * a[2]);
    for (int r = 0; r < 3; ++r) a[r] = a[r] / na;
    double H[9], M[9];
    for (int r = 0; r < 3; ++r)
        for (int q = 0; q < 3; ++q) H[3 * r + q] = 2.0 * a[r] * a[q] - (r == q ? 1.0 : 0.0);
    const double w[3] = {-v[0], -v[1], -v[2]};
    orc_rotation_min(w, u, M);
    for (int r = 0; r < 3; ++r)
        for (int q = 0; q < 3; ++q) R[3 * r + q] = (M[3 * r] * H[q] + M[3 * r + 1] * H[3 + q]) + M[3 * r + 2] * H[6 + q];
}

// pcl::umeyama (with_scaling = false) on three pairs; float row-major 4x4 (estimateRigidTransformationSVD's cast)
void orc_umeyama3(const double src[3][3], const double dst[3][3], float T[16]) {
    double sm[3], dm[3];
    for (int c = 0; c < 3; ++c) { sm[c] = (src[0][c] + src[1][c] + src[2][c]) / 3.0; dm[c] = (dst[0][c] + dst[1][c] + dst[2][c]) / 3.0; }
    double sigma[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
            double acc = 0.0;
            for (int i = 0; i < 3; ++i) acc += (dst[i][r] - dm[r]) * (src[i][c] - sm[c]);
            sigma[3 * r + c] = acc / 3.0;
        }
    double U[9], sv[3], V[9];
    orc_svd3(sigma, U, sv, V);
    double R[9];
    double abs_s = 0.0, abs_d = 0.0, abs_p = 0.0, abs_q = 0.0;
    for (int i = 0; i < 3; ++i)
        for (int c = 0; c < 3; ++c) {
            abs_p += std::fabs(src[i][c]); abs_q += std::fabs(dst[i][c]); abs_s += std::fabs(src[i][c] - sm[c]); abs_d += std::fabs(dst[i][c] - dm[c]);
        }
    const bool rank0 = sv[0] <= orc_noise_floor(abs_p, abs_q, abs_s, abs_d, 3.0, 3.0, 1.1102230246251565e-16);
    if (rank0 || sv[1] <= sv[0] * 1e-12) orc_rotation_rank01(U, V, rank0, R);   // rank <= 1 (double precision)
    else {
        // rank 2: right-handed completion of both bases -> R = U V^T is the proper rotation of Eq. (40)-(43)
        U[2] = U[3] * U[7] - U[6] * U[4]; U[5] = U[6] * U[1] - U[0] * U[7]; U[8] = U[0] * U[4] - U[3] * U[1];
        V[2] = V[3] * V[7] - V[6] * V[4]; V[5] = V[6] * V[1] - V[0] * V[7]; V[8] = V[0] * V[4] - V[3] * V[1];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) R[3 * r + c] = (U[3 * r] * V[3 * c] + U[3 * r + 1] * V[3 * c + 1]) + U[3 * r + 2] * V[3 * c + 2];
    }
    for (int r = 0; r < 3; ++r) {
        const double t = dm[r] - ((R[3 * r] * sm[0] + R[3 * r + 1] * sm[1]) + R[3 * r + 2] * sm[2]);
        T[4 * r] = (float)R[3 * r]; T[4 * r + 1] = (float)R[3 * r + 1]; T[4 * r + 2] = (float)R[3 * r + 2]; T[4 * r + 3] = (float)t;
    }
    T[12] = T[13] = T[14] = 0.0f; T[15] = 1.0f;
}

inline float orc_transfer_sqd(const float T[16], const float* s, const float* t) {
    const float px = ((T[0] * s[0] + T[1] * s[1]) + T[2] * s[2]) + T[3];
    const float py = ((T[4] * s[0] + T[5] * s[1]) + T[6] * s[2]) + T[7];
    const float pz = ((T[8] * s[0] + T[9] * s[1]) + T[10] * s[2]) + T[11];
    const float dx = px - t[0], dy = py - t[1], dz = pz - t[2];
    return (dx * dx + dy * dy) + dz * dz;
}
}  // namespace

int orc_ransac(const float* src_xyz, const float* tgt_xyz, const int* pairs, size_t n_pairs, int max_iterations, double threshold,
               int* inlier_pairs_out, float transform_out[16], int* iterations_out) {
    const size_t n = n_pairs;
    auto keep_all = [&]() {
        if (inlier_pairs_out) std::memcpy(inlier_pairs_out, pairs, sizeof(int) * 2 * n);
        if (transform_out) for (int k = 0; k < 16; ++k) transform_out[k] = (k % 5 == 0) ? 1.0f : 0.0f;
        if (iterations_out) *iterations_out = 0;
        return (int)n;
    };
    if (n < 3) return keep_all();
    std::vector<float> s(3 * n), t(3 * n);
    for (size_t i = 0; i < n; ++i)
        for (int k = 0; k < 3; ++k) { s[3 * i + k] = src_xyz[3 * (size_t)pairs[2 * i] + k]; t[3 * i + k] = tgt_xyz[3 * (size_t)pairs[2 * i + 1] + k]; }
    // computeSampleDistanceThreshold: covariance of the sources (single pass, float), eigenvalues, (mean of sqrt)^2
    double sdt;
    {
        float a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (size_t i = 0; i < n; ++i) {
            const float x = s[3 * i], y = s[3 * i + 1], z = s[3 * i + 2];
            a[0] += x * x; a[1] += x * y; a[2] += x * z; a[3] += y * y; a[4] += y * z; a[5] += z * z; a[6] += x; a[7] += y; a[8] += z;
        }
        const float fn = (float)n;
        for (int k = 0; k < 9; ++k) a[k] /= fn;
        const double cov[9] = {(double)(a[0] - a[6] * a[6]), (double)(a[1] - a[6] * a[7]), (double)(a[2] - a[6] * a[8]),
                               (double)(a[1] - a[6] * a[7]), (double)(a[3] - a[7] * a[7]), (double)(a[4] - a[7] * a[8]),
                               (double)(a[2] - a[6] * a[8]), (double)(a[4] - a[7] * a[8]), (double)(a[5] - a[8] * a[8])};
        double U[9], w[3], V[9];
        orc_svd3(cov, U, w, V);
        const float e0 = (float)w[0], e1 = (float)w[1], e2 = (float)w[2];
        const double m = (double)((std::sqrt(std::max(e0, 0.0f)) + std::sqrt(std::max(e1, 0.0f))) + std::sqrt(std::max(e2, 0.0f))) / 3.0;
        sdt = m * m;
    }
    std::vector<int> shuffled(n);
    for (size_t i = 0; i < n; ++i) shuffled[i] = (int)i;
    OrcMt19937 rng(12345u);
    const double thresh2 = threshold * threshold;
    int iterations = 0, n_best = -2147483647;
    double k = 1.0;
    const double log_probability = std::log(1.0 - 0.99), one_over_indices = 1.0 / (double)n;
    float best_T[16];
    bool have = false;
    while ((double)iterations < k) {
        bool good = false;  // getSamples: drawIndexSample until isSampleGood, at most 1000 tries
        for (int tries = 0; tries < 1000 && !good; ++tries) {
            for (size_t i = 0; i < 3; ++i) std::swap(shuffled[i], shuffled[i + ((rng.next() >> 1) % (n - i))]);
            auto d2 = [&](int a, int b) {
                const float dx = s[3 * b] - s[3 * a], dy = s[3 * b + 1] - s[3 * a + 1], dz = s[3 * b + 2] - s[3 * a + 2];
                return (double)(dx * dx + dy * dy + dz * dz);
            };
            good = d2(shuffled[0], shuffled[1]) > sdt && d2(shuffled[0], shuffled[2]) > sdt && d2(shuffled[1], shuffled[2]) > sdt;
        }
        if (!good) break;
        double sp[3][3], dp[3][3];
        for (int i = 0; i < 3; ++i)
            for (int c = 0; c < 3; ++c) { sp[i][c] = s[3 * (size_t)shuffled[i] + c]; dp[i][c] = t[3 * (size_t)shuffled[i] + c]; }
        float T[16];
        orc_umeyama3(sp, dp, T);
        int cnt = 0;  // countWithinDistance
        for (size_t i = 0; i < n; ++i)
            if ((double)orc_transfer_sqd(T, &s[3 * i], &t[3 * i]) < thresh2) ++cnt;
        if (cnt > n_best) {
            n_best = cnt;
            std::memcpy(best_T, T, sizeof(T));
            have = true;
            const double w = (double)n_best * one_over_indices;
            double p_no_outliers = 1.0 - std::pow(w, 3.0);
            p_no_outliers = std::max(std::numeric_limits<double>::epsilon(), p_no_outliers);
            p_no_outliers = std::min(1.0 - std::numeric_limits<double>::epsilon(), p_no_outliers);
            k = log_probability / std::log(p_no_outliers);
        }
        ++iterations;
        if (iterations > max_iterations) break;
    }
    if (!have) return keep_all();
    std::vector<int> keep;  // selectWithinDistance, original order
    for (size_t i = 0; i < n; ++i)
        if ((double)orc_transfer_sqd(best_T, &s[3 * i], &t[3 * i]) < thresh2) keep.push_back((int)i);
    if (keep.size() < 3) return keep_all();
    for (size_t j = 0; j < keep.size(); ++j)
        if (inlier_pairs_out) { inlier_pairs_out[2 * j] = pairs[2 * keep[j]]; inlier_pairs_out[2 * j + 1] = pairs[2 * keep[j] + 1]; }
    if (transform_out) std::memcpy(transform_out, best_T, sizeof(best_T));
    if (iterations_out) *iterations_out = iterations;
    return (int)keep.size();
}

// ---- ICP (src/lidar_odometry.cpp:283-291: pcl::IterativeClosestPoint with PCL's defaults) ----------------------------
// PCL 1.8 restated (UNPINNED: PCL is not installable here): IterativeClosestPoint::computeTransformation,
// CorrespondenceEstimation::determineCorrespondences (nearest target, squared float distance, no cap),
// TransformationEstimationSVD<.., float> -> pcl::umeyama without scaling, DefaultConvergenceCriteria::hasConverged with
// ICP's settings (10 iterations, rotation threshold 1 - 0 and translation threshold 0, absolute mse 1e-12, relative mse
// -DBL_MAX).  Eigen's vectorised float sums have no defined order: they are taken as 256 strided partial sums and a
// halving tree -- the order the device uses; the 3x3 SVD runs in double (orc_svd3) on the float cross-covariance.
}  // extern "C"
namespace {
template <typename T, typename F>
T orc_strided_sum(size_t n, F term) {
    T part[256];
    for (int t = 0; t < 256; ++t) {
        T a = 0;
        for (size_t i = (size_t)t; i < n; i += 256) a += term(i);
        part[t] = a;
    }
    for (int s = 128; s > 0; s >>= 1)
        for (int t = 0; t < s; ++t) part[t] = part[t] + part[t + s];
    return part[0];
}
inline void orc_apply(const float T[16], const float* p, float* o) {
    const float x = p[0], y = p[1], z = p[2];
    o[0] = ((T[0] * x + T[1] * y) + T[2] * z) + T[3];
    o[1] = ((T[4] * x + T[5] * y) + T[6] * z) + T[7];
    o[2] = ((T[8] * x + T[9] * y) + T[10] * z) + T[11];
}
inline void orc_mul4(const float* a, const float* b, float* o) {
    float r[16];
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) r[4 * i + j] = ((a[4 * i] * b[j] + a[4 * i + 1] * b[4 + j]) + a[4 * i + 2] * b[8 + j]) + a[4 * i + 3] * b[12 + j];
    std::memcpy(o, r, sizeof(r));
}
}  // namespace
extern "C" {

int orc_icp(const float* src_xyz, size_t n_src, const float* tgt_xyz, size_t n_tgt, const float* pre4x4, int max_iterations, float final_out[16],
            int* iterations_out, double* mse_out) {
    const float ident[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    float F[16];
    std::memcpy(F, ident, sizeof(F));
    int iterations = 0, state = 0;
    double prev_mse = std::numeric_limits<double>::max(), mse = 0.0;
    std::vector<float> cur(3 * n_src);
    for (size_t i = 0; i < n_src; ++i) orc_apply(pre4x4 ? pre4x4 : ident, &src_xyz[3 * i], &cur[3 * i]);   // transformPointCloud(.., T_est)
    std::vector<long long> nn(n_src);
    std::vector<float> nd(n_src);
    if (n_src == 0 || n_tgt == 0 || max_iterations <= 0) state = 5;
    while (state == 0) {
#pragma omp parallel for schedule(static)
        for (long long i = 0; i < (long long)n_src; ++i) {   // nearestKSearch(.., 1, ..): first minimum = lowest index
            float best = 0.f; long long bi = -1;
            for (size_t k = 0; k < n_tgt; ++k) {
                const float dx = cur[3 * i] - tgt_xyz[3 * k], dy = cur[3 * i + 1] - tgt_xyz[3 * k + 1], dz = cur[3 * i + 2] - tgt_xyz[3 * k + 2];
                const float d = (dx * dx + dy * dy) + dz * dz;
                if (d == d && (bi < 0 || d < best)) { best = d; bi = (long long)k; }
            }
            nn[i] = bi; nd[i] = best;
        }
        const float cnt = orc_strided_sum<float>(n_src, [&](size_t i) { return nn[i] >= 0 ? 1.f : 0.f; });
        const unsigned n = (unsigned)cnt;
        if (n < 3) { state = 5; break; }
        const float one_over_n = 1.0f / (float)n;
        float sm[3], dm[3];
        for (int c = 0; c < 3; ++c) {
            sm[c] = orc_strided_sum<float>(n_src, [&](size_t i) { return nn[i] >= 0 ? cur[3 * i + c] : 0.f; }) * one_over_n;
            dm[c] = orc_strided_sum<float>(n_src, [&](size_t i) { return nn[i] >= 0 ? tgt_xyz[3 * nn[i] + c] : 0.f; }) * one_over_n;
        }
        double sg[9];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c)
                sg[3 * r + c] = (double)(one_over_n * orc_strided_sum<float>(n_src, [&](size_t i) {
                                             return nn[i] >= 0 ? (tgt_xyz[3 * nn[i] + r] - dm[r]) * (cur[3 * i + c] - sm[c]) : 0.f; }));
        const double mse_sum = orc_strided_sum<double>(n_src, [&](size_t i) { return nn[i] >= 0 ? (double)nd[i] : 0.0; });
        double U[9], sv[3], V[9];
        orc_svd3(sg, U, sv, V);
        const double det = sg[0] * (sg[4] * sg[8] - sg[5] * sg[7]) - sg[1] * (sg[3] * sg[8] - sg[5] * sg[6]) + sg[2] * (sg[3] * sg[7] - sg[4] * sg[6]);
        double Rd[9];
        // sums of the 1-norms of the sources, targets, centred sources and centred targets: the rank-0 noise floor
        const float abs_p = orc_strided_sum<float>(n_src, [&](size_t i) {
            return nn[i] >= 0 ? (std::fabs(cur[3 * i]) + std::fabs(cur[3 * i + 1])) + std::fabs(cur[3 * i + 2]) : 0.f; });
        const float abs_q = orc_strided_sum<float>(n_src, [&](size_t i) {
            if (nn[i] < 0) return 0.f;
            const float* q = &tgt_xyz[3 * nn[i]];
            return (std::fabs(q[0]) + std::fabs(q[1])) + std::fabs(q[2]); });
        const float abs_s = orc_strided_sum<float>(n_src, [&](size_t i) {
            return nn[i] >= 0 ? (std::fabs(cur[3 * i] - sm[0]) + std::fabs(cur[3 * i + 1] - sm[1])) + std::fabs(cur[3 * i + 2] - sm[2]) : 0.f; });
        const float abs_d = orc_strided_sum<float>(n_src, [&](size_t i) {
            if (nn[i] < 0) return 0.f;
            const float* q = &tgt_xyz[3 * nn[i]];
            return (std::fabs(q[0] - dm[0]) + std::fabs(q[1] - dm[1])) + std::fabs(q[2] - dm[2]); });
        const bool rank0 = sv[0] <= orc_noise_floor((double)abs_p, (double)abs_q, (double)abs_s, (double)abs_d, (double)n,
                                                    (double)((n + 255) / 256 + 8), 5.9604644775390625e-08);
        if (rank0 || sv[1] <= sv[0] * 1e-5) orc_rotation_rank01(U, V, rank0, Rd);   // rank <= 1 (float precision)
        else {
            double sgn = 1.0;
            if (sv[2] <= sv[0] * 1e-5) {   // rank 2
                U[2] = U[3] * U[7] - U[6] * U[4]; U[5] = U[6] * U[1] - U[0] * U[7]; U[8] = U[0] * U[4] - U[3] * U[1];
                V[2] = V[3] * V[7] - V[6] * V[4]; V[5] = V[6] * V[1] - V[0] * V[7]; V[8] = V[0] * V[4] - V[3] * V[1];
            } else if (det < 0) sgn = -1.0;
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) Rd[3 * r + c] = (U[3 * r] * V[3 * c] + U[3 * r + 1] * V[3 * c + 1]) + sgn * (U[3 * r + 2] * V[3 * c + 2]);
        }
        float Rt[16];
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) Rt[4 * r + c] = (float)Rd[3 * r + c];
            Rt[4 * r + 3] = dm[r] - ((Rt[4 * r] * sm[0] + Rt[4 * r + 1] * sm[1]) + Rt[4 * r + 2] * sm[2]);
        }
        Rt[12] = Rt[13] = Rt[14] = 0.f; Rt[15] = 1.f;
        for (size_t i = 0; i < n_src; ++i) { float o[3]; orc_apply(Rt, &cur[3 * i], o); cur[3 * i] = o[0]; cur[3 * i + 1] = o[1]; cur[3 * i + 2] = o[2]; }
        orc_mul4(Rt, F, F);
        ++iterations;
        mse = mse_sum / (double)n;
        if (iterations >= max_iterations) state = 1;
        else {
            const double cos_angle = 0.5 * (double)(((Rt[0] + Rt[5]) + Rt[10]) - 1.0f);
            const double translation_sqr = (double)((Rt[3] * Rt[3] + Rt[7] * Rt[7]) + Rt[11] * Rt[11]);
            if (cos_angle >= 1.0 && translation_sqr <= 0.0) state = 2;
            else if (std::fabs(mse - prev_mse) < 1e-12) state = 3;
            else prev_mse = mse;
        }
    }
    if (final_out) std::memcpy(final_out, F, sizeof(F));
    if (iterations_out) *iterations_out = iterations;
    if (mse_out) *mse_out = mse;
    return state;
}

// LidarOdometry::evaluateEstimation (src/lidar_odometry.cpp:267-296)
int orc_evaluate_estimation(const float* T_j, const float* T_i, int n_corr, const float* src_kp, size_t n_src, const float* tgt_kp, size_t n_tgt,
                            int run_icp, float T_best[16], float* h_diff_out, float* t_diff_out) {
    // rigid T_i: inverse = [R^T | -R^T t] would do; the reference inverts the general 4x4 (Matrix4f::inverse) -- by cofactors here
    double m[16], inv[16];
    for (int e = 0; e < 16; ++e) m[e] = T_i[e];
    // Gauss-Jordan in double, cast to float: an independent route to the same inverse (agreement with the device's float
    // cofactor expansion is to rounding, which is what the gate needs)
    double a[4][8];
    for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) { a[r][c] = m[4 * r + c]; a[r][4 + c] = r == c ? 1.0 : 0.0; }
    for (int col = 0; col < 4; ++col) {
        int piv = col;
        for (int r = col + 1; r < 4; ++r) if (std::fabs(a[r][col]) > std::fabs(a[piv][col])) piv = r;
        for (int c = 0; c < 8; ++c) std::swap(a[col][c], a[piv][c]);
        const double d = a[col][col];
        for (int c = 0; c < 8; ++c) a[col][c] /= d;
        for (int r = 0; r < 4; ++r) if (r != col) { const double f = a[r][col]; for (int c = 0; c < 8; ++c) a[r][c] -= f * a[col][c]; }
    }
    for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) inv[4 * r + c] = a[r][4 + c];
    float Ti_inv[16], Tij[16];
    for (int e = 0; e < 16; ++e) Ti_inv[e] = (float)inv[e];
    orc_mul4(Ti_inv, T_j, Tij);
    const float h_diff = std::acos(Tij[5]);
    const float t_diff = std::sqrt((Tij[3] * Tij[3] + Tij[7] * Tij[7]) + Tij[11] * Tij[11]);
    const bool reject = (double)(h_diff * 180) / M_PI > 10 || t_diff > 1200 || n_corr < 15;
    const float* T_est = reject ? T_i : T_j;
    if (h_diff_out) *h_diff_out = h_diff;
    if (t_diff_out) *t_diff_out = t_diff;
    if (run_icp) {
        float F[16];
        orc_icp(src_kp, n_src, tgt_kp, n_tgt, T_est, 10, F, nullptr, nullptr);
        orc_mul4(F, T_est, T_best);
    } else std::memcpy(T_best, T_j, 16 * sizeof(float));
    return reject ? 0 : 1;
}

void orc_eigh3(const double m[9], double evals[3], double evecs_cols[9]) { eigh3(m, evals, evecs_cols); }
void orc_eigen33_smallest(const float m[9], float* eval, float evec[3]) { eigen33_smallest(m, *eval, evec); }

}  // extern "C"
