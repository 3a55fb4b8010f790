// voxel_grid_oracle.cpp -- CPU restatement of pcl::VoxelGrid<PointXYZ>::applyFilter (PCL 1.8, filters/impl/voxel_grid.hpp)
// with PCL's defaults: downsample_all_data_ true, no filter field, min_points_per_voxel_ 0.  Test infrastructure for
// bshot_voxel_grid (tests/test_voxel_grid.py); built by tests/voxel_grid_oracle.py into a temporary directory.
//
// Parity pin: this restates PCL's published algorithm step by step and is never checked against PCL itself.
//   1. inv = 1.0f / leaf per axis (fp32).
//   2. bbox = fp32 min / max over the finite points (PCL's !is_dense branch); no finite point (or n = 0): empty output.
//   3. d_a = (int64)((max_a - min_a) * inv_a) + 1; dx * dy * dz > INT32_MAX: the output is the input cloud unchanged
//      (PCL 1.8; 1.7.2 has no such test).
//   4. min_b = (int)floor(min * inv), max_b = (int)floor(max * inv), div_b = max_b - min_b + 1,
//      multipliers (1, div_b.x, div_b.x * div_b.y).
//   5. per finite point ijk_a = (int)(floor(p_a * inv_a) - (float)min_b_a) (one fp32 multiply), idx = ijk . mul
//      modulo 2^32 (what PCL's int arithmetic yields on two's-complement machines; done here in unsigned arithmetic).
//   6. one point per occupied voxel, ascending idx: fp32 running sum from zero, then sum / (float)count.
//   7. order inside a voxel: "index" (order 0) = std::stable_sort of the (idx, point) pairs on idx, i.e. ascending point
//      index, the port's definition; "pcl" (order 1) = std::sort with PCL's idx-only comparator, the order a g++-built
//      PCL leaves (introsort is unstable).  Membership, count and output order are the same under both.
// Out of int's range (coordinates beyond 2^31 leaves from the origin) PCL's float -> int conversions are undefined;
// here they saturate, as the device's conversion does.
// Compiled with -ffp-contract=off: every operation is the fp32 operation written.
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <vector>

namespace {

struct Pair {
    unsigned idx;
    unsigned cloud_point_index;
    bool operator<(const Pair& p) const { return idx < p.idx; }  // PCL's cloud_point_index_idx::operator<
};

int to_int(float f) {  // (int) of an integral float, saturating
    if (f >= 2147483648.0f) return INT32_MAX;
    if (f < -2147483648.0f) return INT32_MIN;
    return (int)f;
}

bool finite3(const float* p) { return std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]); }

}  // namespace

extern "C" size_t vg_ref_filter(const float* xyz, size_t n, size_t stride_floats, float leaf_x, float leaf_y, float leaf_z,
                                int order, float* out) {
    const float leaf[3] = {leaf_x, leaf_y, leaf_z};
    float inv[3];
    for (int a = 0; a < 3; ++a) inv[a] = 1.0f / leaf[a];
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    size_t nfin = 0;
    for (size_t i = 0; i < n; ++i) {
        const float* p = xyz + i * stride_floats;
        if (!finite3(p)) continue;
        for (int a = 0; a < 3; ++a) { mn[a] = std::min(mn[a], p[a]); mx[a] = std::max(mx[a], p[a]); }
        ++nfin;
    }
    if (nfin == 0) return 0;
    int64_t prod = 1;
    bool ovf = false;
    for (int a = 0; a < 3 && !ovf; ++a) {
        const float f = (mx[a] - mn[a]) * inv[a];
        if (!(f < 2147483648.0f)) { ovf = true; break; }  // d_a > INT32_MAX on its own (PCL's int64 product could overflow)
        prod *= (int64_t)f + 1;
        ovf = prod > (int64_t)INT32_MAX;
    }
    if (ovf) {
        for (size_t i = 0; i < n; ++i)
            for (int a = 0; a < 3; ++a) out[3 * i + a] = xyz[i * stride_floats + a];
        return n;
    }
    int min_b[3], max_b[3];
    for (int a = 0; a < 3; ++a) {
        min_b[a] = to_int(std::floor(mn[a] * inv[a]));
        max_b[a] = to_int(std::floor(mx[a] * inv[a]));
    }
    const unsigned div0 = (unsigned)max_b[0] - (unsigned)min_b[0] + 1u, div1 = (unsigned)max_b[1] - (unsigned)min_b[1] + 1u;
    const unsigned mul[3] = {1u, div0, div0 * div1};
    std::vector<Pair> pairs;
    pairs.reserve(nfin);
    for (size_t i = 0; i < n; ++i) {
        const float* p = xyz + i * stride_floats;
        if (!finite3(p)) continue;
        unsigned idx = 0;
        for (int a = 0; a < 3; ++a) idx += (unsigned)to_int(std::floor(p[a] * inv[a]) - (float)min_b[a]) * mul[a];
        pairs.push_back(Pair{idx, (unsigned)i});
    }
    if (order == 0) std::stable_sort(pairs.begin(), pairs.end());
    else std::sort(pairs.begin(), pairs.end());
    size_t count = 0;
    for (size_t s = 0; s < pairs.size();) {
        size_t e = s + 1;
        while (e < pairs.size() && pairs[e].idx == pairs[s].idx) ++e;
        float sum[3] = {0.0f, 0.0f, 0.0f};
        for (size_t k = s; k < e; ++k)
            for (int a = 0; a < 3; ++a) sum[a] += xyz[(size_t)pairs[k].cloud_point_index * stride_floats + a];
        for (int a = 0; a < 3; ++a) out[3 * count + a] = sum[a] / (float)(e - s);
        ++count;
        s = e;
    }
    return count;
}
