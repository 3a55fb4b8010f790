// shot.cu -- SHOT local reference frame, SHOT352 histogram and B-SHOT bits (SURVEY 8a rows a5-a7).
//
// Replaces bshot::calculate_SHOT (include/bshot_bits.h:113-135; PCL SHOTEstimationOMP +
// SHOTLocalReferenceFrameEstimation, SURVEY Appendix A.4/A.5) and bshot::compute_bshot_from_SHOT
// (include/bshot_bits.h:144-278).  One CTA per keypoint:
//   phase A  weighted covariance about the keypoint in fp64 (weight R - d), CTA reduce,
//            3x3 symmetric eigen-solve (cyclic Jacobi, fp64)
//   phase B  sign disambiguation votes (exact-tie median rule via a CTA-wide radix select)
//   phase C  quadrilinear interpolation into a 352-float shared-memory histogram (<= 5 atomics
//            per neighbour), fp64 intermediates like PCL
//   phase D  L2 normalisation, optional float output, 88 nibbles -> packed 352-bit record
// The float histogram never has to touch HBM when only the bits are wanted.
#include <math.h>
#include <stdlib.h>

#include "eigh3.cuh"
#include "nbr.cuh"
#include "stages.h"

namespace bshot {

constexpr int SH_MAX_THREADS = 256;
constexpr int SH_WARPS = SH_MAX_THREADS / 32;  // smem reduction slots (upper bound)
constexpr int SH_MAXSEG = 1024;
constexpr int SH_MAXB = 2048;  // batch table covers 65536 candidates per keypoint
constexpr int SH_TIE_CAP = 512;

struct ShotSmem {
    SegList<SH_MAXSEG, SH_MAXB> sl;
    float hist[352];
    unsigned int acc[352];  // fixed-point accumulators (native 32-bit shared atomics)
    unsigned int tie_hist[256];
    unsigned long long tie_list[SH_TIE_CAP];
    unsigned tie_n, tie_below, tie_blo, tie_bhi;
    double red[SH_WARPS][8];
    int redi[SH_WARPS][4];
    double v1[3], v3[3];
    float rf[9];
    unsigned words[12];
    int valid, count_all;
    int tie1, tie3;
    int ok;
    unsigned cnt;
    double norm;
};

// include/bshot_bits.h:160-260 : 4 floats -> nibble (bit k = element k)
__device__ __forceinline__ unsigned bshot_nibble(float v0, float v1, float v2, float v3) {
    const float sum = __fadd_rn(__fadd_rn(__fadd_rn(v0, v1), v2), v3);
    const double t = 0.9 * (double)sum;
    if (v0 == 0.0f && v1 == 0.0f && v2 == 0.0f && v3 == 0.0f) return 0x0u;
    if ((double)v0 > t) return 0x1u;
    if ((double)v1 > t) return 0x2u;
    if ((double)v2 > t) return 0x4u;
    if ((double)v3 > t) return 0x8u;
    if ((double)__fadd_rn(v0, v1) > t) return 0x3u;
    if ((double)__fadd_rn(v1, v2) > t) return 0x6u;
    if ((double)__fadd_rn(v2, v3) > t) return 0xCu;
    if ((double)__fadd_rn(v0, v3) > t) return 0x9u;
    if ((double)__fadd_rn(v1, v3) > t) return 0xAu;
    if ((double)__fadd_rn(v0, v2) > t) return 0x5u;
    if ((double)__fadd_rn(__fadd_rn(v0, v1), v2) > t) return 0x7u;
    if ((double)__fadd_rn(__fadd_rn(v1, v2), v3) > t) return 0xEu;
    if ((double)__fadd_rn(__fadd_rn(v0, v2), v3) > t) return 0xDu;
    if ((double)__fadd_rn(__fadd_rn(v0, v1), v3) > t) return 0xBu;
    return 0xFu;
}

// hist (352 floats in smem) -> 12 u32 words (smem) ; threads 0..87 active, all threads sync
template <int NT>
__device__ __forceinline__ void pack_bits_block(const float* hist, unsigned* words, unsigned tid) {
    if (tid < 12) words[tid] = 0u;
    __syncthreads();
    for (unsigned j = tid; j < 88; j += NT) {
        const unsigned nib = bshot_nibble(hist[4 * j], hist[4 * j + 1], hist[4 * j + 2], hist[4 * j + 3]);
        if (nib) atomicOr(&words[j >> 3], nib << ((j & 7) * 4));
    }
    __syncthreads();
}

// acos(x), x in [-1, 1]: sqrt(1 - |x|) * P7(|x|) (Abramowitz & Stegun 4.4.46), |error| < 2.5e-7 rad in fp32 -- the
// elevation angle only enters the descriptor linearly, as an interpolation weight on a ~4e-6 fixed-point grid
__device__ __forceinline__ float acos_poly(float x) {
    const float a = fabsf(x);
    float p = -0.0012624911f;
    p = fmaf(p, a, 0.0066700901f);
    p = fmaf(p, a, -0.0170881256f);
    p = fmaf(p, a, 0.0308918810f);
    p = fmaf(p, a, -0.0501743046f);
    p = fmaf(p, a, 0.0889789874f);
    p = fmaf(p, a, -0.2145988016f);
    p = fmaf(p, a, 1.5707963050f);
    const float r = __fsqrt_rn(1.0f - a) * p;
    return x < 0.0f ? 3.14159265358979f - r : r;
}

// atan(t) for |t| <= 0.47 (an angle inside one 45-degree azimuth sector, measured from the sector centre):
// odd polynomial, |error| < 4e-8 rad in fp32
__device__ __forceinline__ float atan_sector(float t) {
    const float u = t * t;
    float p = -0.05407935f;
    p = fmaf(p, u, 0.10297535f);
    p = fmaf(p, u, -0.1419787f);
    p = fmaf(p, u, 0.19995609f);
    p = fmaf(p, u, -0.33333252f);
    p = fmaf(p, u, 1.0f);
    return p * t;
}

#ifndef BSHOT_SHOT_FP64_INTERP
#define BSHOT_SHOT_FP64_INTERP 0  // 1: PCL's double-precision interpolation arithmetic (slower; same bits to >= 99.9 %)
#endif
#ifndef BSHOT_SH_MINBLOCKS
#define BSHOT_SH_MINBLOCKS 9
#endif
template <int SH_THREADS>
__global__ void __launch_bounds__(SH_THREADS, (SH_THREADS == 128) ? BSHOT_SH_MINBLOCKS : 1)
shot_kernel(const GridParams* __restrict__ gp, const unsigned* __restrict__ cell_start,
            const float4* __restrict__ sorted, const float4* __restrict__ kp, const int* __restrict__ kp_count,
            const float4* __restrict__ normals, unsigned normals_limit, float radius, float r2_4, int lrf_only,
            float* __restrict__ rf_out, int* __restrict__ nn_out, float* __restrict__ shot_out,
            uint64_t* __restrict__ bits_out, unsigned long long* __restrict__ sum_nn, const unsigned* __restrict__ order) {
    __shared__ ShotSmem sm;
    const unsigned tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if ((int)blockIdx.x >= *kp_count) return;
    const int k = order ? (int)order[blockIdx.x] : (int)blockIdx.x;
    const GridParams g = *gp;
    const float4 q = kp[k];
    const float R = radius;
    const float R2 = (float)((double)R * (double)R);
    const bool q_finite = isfinite(q.x) && isfinite(q.y) && isfinite(q.z);
    const float nanf_ = __int_as_float(0x7FC00000);

    RowRange rr = row_range(g, q.y, q.z, R);
    if (!q_finite) rr.nrows = 0;
    bool cached = false;
    auto sync = [] { __syncthreads(); };
    auto for_each = [&](auto&& f) {
        for (int row0 = 0; row0 < rr.nrows; row0 += SH_MAXSEG) {
            if (!(cached && rr.nrows <= SH_MAXSEG)) {
                build_segments<SH_THREADS, SH_MAXSEG, SH_MAXB>(g, cell_start, q.x, q.y, q.z, R, rr, row0, sm.sl, tid, sync);
                cached = true;
            }
            const unsigned total = sm.sl.total;
            for (unsigned j = tid; j < total; j += SH_THREADS * 2) {  // 2 candidate loads in flight per thread
                const unsigned j1 = j + SH_THREADS;
                const float4 p0 = __ldg(sorted + seg_lookup(sm.sl, j));
                const float4 p1 = __ldg(sorted + seg_lookup(sm.sl, j1 < total ? j1 : j));
                f(p0);
                if (j1 < total) f(p1);
            }
            if (rr.nrows > SH_MAXSEG) __syncthreads();
        }
    };

    // ---- phase A: weighted covariance about the keypoint (Appendix A.4) -------------------------
    double acc[7] = {0, 0, 0, 0, 0, 0, 0};
    int valid = 0, count_all = 0;
    for_each([&](const float4 p) {
        const float sqd = sqdist_rn(q.x, q.y, q.z, p.x, p.y, p.z);
        if (!(sqd < R2)) return;
        ++count_all;
        if (p.x == q.x && p.y == q.y && p.z == q.z) return;
        const double vx = (double)__fsub_rn(p.x, q.x), vy = (double)__fsub_rn(p.y, q.y), vz = (double)__fsub_rn(p.z, q.z);
        const double w = (double)R - sqrt((double)sqd);
        acc[0] += w * (vx * vx); acc[1] += w * (vx * vy); acc[2] += w * (vx * vz);
        acc[3] += w * (vy * vy); acc[4] += w * (vy * vz); acc[5] += w * (vz * vz);
        acc[6] += w;
        ++valid;
    });
#pragma unroll
    for (int i = 0; i < 7; ++i) acc[i] = warp_sum(acc[i]);
    valid = warp_sum(valid);
    count_all = warp_sum(count_all);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 7; ++i) sm.red[wid][i] = acc[i];
        sm.redi[wid][0] = valid;
        sm.redi[wid][1] = count_all;
    }
    __syncthreads();
    if (tid == 0) {
        double m[7];
        int nv = 0, na = 0;
        for (int i = 0; i < 7; ++i) { m[i] = 0; for (int w = 0; w < SH_THREADS / 32; ++w) m[i] += sm.red[w][i]; }
        for (int w = 0; w < SH_THREADS / 32; ++w) { nv += sm.redi[w][0]; na += sm.redi[w][1]; }
        sm.valid = nv;
        sm.count_all = na;
        int ok = (nv >= 5) ? 1 : 0;
        if (ok) {
            double c[6];
            for (int i = 0; i < 6; ++i) c[i] = m[i] / m[6];
            double w[3], V[3][3];
            eigh3_jacobi(c, w, V);
            if (!isfinite(w[0]) || !isfinite(w[1]) || !isfinite(w[2])) ok = 0;
            for (int r = 0; r < 3; ++r) { sm.v1[r] = V[r][2]; sm.v3[r] = V[r][0]; }
        }
        sm.ok = ok;
    }
    __syncthreads();
    const int ok = sm.ok;
    const int n_valid = sm.valid, n_all = sm.count_all;

    // ---- phase B: sign disambiguation ---------------------------------------------------------
    if (ok) {
        const double v1x = sm.v1[0], v1y = sm.v1[1], v1z = sm.v1[2];
        const double v3x = sm.v3[0], v3y = sm.v3[1], v3z = sm.v3[2];
        int plus_t = 0, plus_n = 0;
        for_each([&](const float4 p) {
            const float sqd = sqdist_rn(q.x, q.y, q.z, p.x, p.y, p.z);
            if (!(sqd < R2)) return;
            if (p.x == q.x && p.y == q.y && p.z == q.z) return;
            const double vx = (double)__fsub_rn(p.x, q.x), vy = (double)__fsub_rn(p.y, q.y), vz = (double)__fsub_rn(p.z, q.z);
            if (vx * v1x + vy * v1y + vz * v1z >= 0) ++plus_t;
            if (vx * v3x + vy * v3y + vz * v3z >= 0) ++plus_n;
        });
        plus_t = warp_sum(plus_t);
        plus_n = warp_sum(plus_n);
        __syncthreads();
        if (lane == 0) { sm.redi[wid][0] = plus_t; sm.redi[wid][1] = plus_n; }
        __syncthreads();
        if (tid == 0) {
            int pt = 0, pn = 0;
            for (int w = 0; w < SH_THREADS / 32; ++w) { pt += sm.redi[w][0]; pn += sm.redi[w][1]; }
            const int st = 2 * pt - n_valid, sn = 2 * pn - n_valid;
            sm.tie1 = (st == 0);
            sm.tie3 = (sn == 0);
            if (st < 0) { sm.v1[0] = -sm.v1[0]; sm.v1[1] = -sm.v1[1]; sm.v1[2] = -sm.v1[2]; }
            if (sn < 0) { sm.v3[0] = -sm.v3[0]; sm.v3[1] = -sm.v3[1]; sm.v3[2] = -sm.v3[2]; }
        }
        __syncthreads();
        if (sm.tie1 || sm.tie3) {
            // exact tie: votes of the 5 neighbours at sorted positions median-2..median+2 of the valid
            // list ordered by (sqd, index).  CTA-wide MSB-first radix select of the two bounding keys.
            const int median = n_valid / 2;
            unsigned long long bound[2];
            // Fast path: 256-bin histogram of sqd over the valid neighbours, collect the bins that hold ranks
            // median-2 .. median+2, rank that short list exactly by (sqd, index).
            for (unsigned i = tid; i < 256; i += SH_THREADS) sm.tie_hist[i] = 0u;
            if (tid == 0) sm.tie_n = 0;
            __syncthreads();
            const float tscale = 256.0f / R2;
            for_each([&](const float4 p) {
                const float sqd = sqdist_rn(q.x, q.y, q.z, p.x, p.y, p.z);
                if (!(sqd < R2)) return;
                if (p.x == q.x && p.y == q.y && p.z == q.z) return;
                atomicAdd(&sm.tie_hist[min(255, (int)(sqd * tscale))], 1u);
            });
            __syncthreads();
            if (tid == 0) {
                unsigned cum = 0, blo = 255, bhi = 255, below = 0;
                bool flo = false, fhi = false;
                for (unsigned bn = 0; bn < 256; ++bn) {
                    const unsigned h = sm.tie_hist[bn];
                    if (!flo && cum + h > (unsigned)(median - 2)) { blo = bn; below = cum; flo = true; }
                    if (!fhi && cum + h > (unsigned)(median + 2)) { bhi = bn; fhi = true; }
                    cum += h;
                }
                sm.tie_blo = blo; sm.tie_bhi = bhi; sm.tie_below = below;
            }
            __syncthreads();
            const int blo = (int)sm.tie_blo, bhi = (int)sm.tie_bhi;
            for_each([&](const float4 p) {
                const float sqd = sqdist_rn(q.x, q.y, q.z, p.x, p.y, p.z);
                if (!(sqd < R2)) return;
                if (p.x == q.x && p.y == q.y && p.z == q.z) return;
                const int bn = min(255, (int)(sqd * tscale));
                if (bn < blo || bn > bhi) return;
                const unsigned slot = atomicAdd(&sm.tie_n, 1u);
                if (slot < (unsigned)SH_TIE_CAP) sm.tie_list[slot] = ((unsigned long long)__float_as_uint(sqd) << 32) | __float_as_uint(p.w);
            });
            __syncthreads();
            const unsigned tn = sm.tie_n;
            if (tn <= (unsigned)SH_TIE_CAP) {
                // local ranks median-2-below and median+2-below bound the five keys
                const unsigned r_lo = (unsigned)(median - 2) - sm.tie_below, r_hi = (unsigned)(median + 2) - sm.tie_below;
                for (unsigned e = tid; e < tn; e += SH_THREADS) {
                    const unsigned long long ke = sm.tie_list[e];
                    unsigned rank = 0;
                    for (unsigned o = 0; o < tn; ++o) rank += (sm.tie_list[o] < ke) ? 1u : 0u;
                    if (rank == r_lo) sm.red[0][0] = __longlong_as_double((long long)ke);
                    if (rank == r_hi) sm.red[0][1] = __longlong_as_double((long long)ke);
                }
                __syncthreads();
                bound[0] = (unsigned long long)__double_as_longlong(sm.red[0][0]);
                bound[1] = (unsigned long long)__double_as_longlong(sm.red[0][1]);
                __syncthreads();
            } else
            // Slow path (more than SH_TIE_CAP neighbours in the median bins): CTA-wide MSB-first radix select.
            for (int which = 0; which < 2; ++which) {
                unsigned rank = (unsigned)(median + (which ? 2 : -2));
                unsigned long long prefix = 0;
                for (int bit = 62; bit >= 0; --bit) {
                    unsigned c0 = 0;
                    for_each([&](const float4 p) {
                        const float sqd = sqdist_rn(q.x, q.y, q.z, p.x, p.y, p.z);
                        if (!(sqd < R2)) return;
                        if (p.x == q.x && p.y == q.y && p.z == q.z) return;
                        const unsigned long long key = ((unsigned long long)__float_as_uint(sqd) << 32) | __float_as_uint(p.w);
                        if ((key >> (bit + 1)) == (prefix >> (bit + 1)) && !((key >> bit) & 1ull)) ++c0;
                    });
                    c0 = (unsigned)warp_sum((int)c0);
                    __syncthreads();
                    if (tid == 0) sm.cnt = 0;
                    __syncthreads();
                    if (lane == 0) atomicAdd(&sm.cnt, c0);
                    __syncthreads();
                    const unsigned tot0 = sm.cnt;
                    if (rank >= tot0) { rank -= tot0; prefix |= (1ull << bit); }
                }
                bound[which] = prefix;
            }
            const double a1x = sm.v1[0], a1y = sm.v1[1], a1z = sm.v1[2];
            const double a3x = sm.v3[0], a3y = sm.v3[1], a3z = sm.v3[2];
            int p1 = 0, p3 = 0;
            for_each([&](const float4 p) {
                const float sqd = sqdist_rn(q.x, q.y, q.z, p.x, p.y, p.z);
                if (!(sqd < R2)) return;
                if (p.x == q.x && p.y == q.y && p.z == q.z) return;
                const unsigned long long key = ((unsigned long long)__float_as_uint(sqd) << 32) | __float_as_uint(p.w);
                if (key < bound[0] || key > bound[1]) return;
                const double vx = (double)__fsub_rn(p.x, q.x), vy = (double)__fsub_rn(p.y, q.y), vz = (double)__fsub_rn(p.z, q.z);
                if (vx * a1x + vy * a1y + vz * a1z > 0) ++p1;
                if (vx * a3x + vy * a3y + vz * a3z > 0) ++p3;
            });
            p1 = warp_sum(p1);
            p3 = warp_sum(p3);
            __syncthreads();
            if (lane == 0) { sm.redi[wid][0] = p1; sm.redi[wid][1] = p3; }
            __syncthreads();
            if (tid == 0) {
                int c1 = 0, c3 = 0;
                for (int w = 0; w < SH_THREADS / 32; ++w) { c1 += sm.redi[w][0]; c3 += sm.redi[w][1]; }
                if (sm.tie1 && c1 < 3) { sm.v1[0] = -sm.v1[0]; sm.v1[1] = -sm.v1[1]; sm.v1[2] = -sm.v1[2]; }
                if (sm.tie3 && c3 < 3) { sm.v3[0] = -sm.v3[0]; sm.v3[1] = -sm.v3[1]; sm.v3[2] = -sm.v3[2]; }
            }
            __syncthreads();
        }
    }
    if (tid == 0) {
        if (ok) {
            const float x0 = (float)sm.v1[0], x1 = (float)sm.v1[1], x2 = (float)sm.v1[2];
            const float z0 = (float)sm.v3[0], z1 = (float)sm.v3[1], z2 = (float)sm.v3[2];
            sm.rf[0] = x0; sm.rf[1] = x1; sm.rf[2] = x2;
            sm.rf[6] = z0; sm.rf[7] = z1; sm.rf[8] = z2;
            sm.rf[3] = __fsub_rn(__fmul_rn(z1, x2), __fmul_rn(z2, x1));  // y = z x x in fp32
            sm.rf[4] = __fsub_rn(__fmul_rn(z2, x0), __fmul_rn(z0, x2));
            sm.rf[5] = __fsub_rn(__fmul_rn(z0, x1), __fmul_rn(z1, x0));
        } else {
            for (int i = 0; i < 9; ++i) sm.rf[i] = nanf_;
        }
    }
    __syncthreads();
    if (tid < 9) rf_out[(size_t)k * 9 + tid] = sm.rf[tid];
    if (tid == 0) {
        nn_out[k] = lrf_only ? n_valid : n_all;
        if (!lrf_only) atomicAdd(sum_nn, (unsigned long long)n_all);
    }
    if (lrf_only) return;

    // ---- phase C: SHOT352 quadrilinear histogram (Appendix A.5) ---------------------------------
    for (unsigned i = tid; i < 352; i += SH_THREADS) sm.acc[i] = 0u;
    __syncthreads();
    const bool describe = ok && n_all >= 5;
    // Votes are accumulated in 32-bit fixed point: float atomicAdd on shared memory is a CAS spin loop
    // (SASS ATOMS.CAST.SPIN), integer add is native (ATOMS.ADD).  A bin receives at most 4 per
    // neighbour, so 2^fx_bits * 4.1 * n_all < 2^32 cannot overflow; the sum is order independent.
    // = largest b <= 28 with 2^b <= room (room >= 2 for any neighbour count below 5e8)
    const int fx_bits = min(28, max(0, ilogb(4294967295.0 / (4.1 * (double)max(n_all, 1)))));
    const float fx_scale = (float)(1u << fx_bits);
    const float fx_inv = 1.0f / fx_scale;
    if (describe) {
        const float fx0 = sm.rf[0], fx1 = sm.rf[1], fx2 = sm.rf[2];
        const float fy0 = sm.rf[3], fy1 = sm.rf[4], fy2 = sm.rf[5];
        const float fz0 = sm.rf[6], fz1 = sm.rf[7], fz2 = sm.rf[8];
        const double radius3_4 = ((double)R * 3) / 4, radius1_4 = (double)R / 4, radius1_2 = (double)R / 2;
        const double RAD_45 = 0.78539816339744830961566084581988, RAD_90 = 1.5707963267948966192313216916398;
        const double RAD_135 = 2.3561944901923449288469825374596, RAD_PI_7_8 = 2.7488935718910690836548129603691;
        unsigned int* hist = sm.acc;
        auto vote = [&](int idx, float v) { atomicAdd(&hist[idx], __float2uint_rn(v * fx_scale)); };
#if BSHOT_SHOT_FP64_INTERP
        for_each([&](const float4 p) {
            const float sqd = sqdist_rn(q.x, q.y, q.z, p.x, p.y, p.z);
            if (!(sqd < R2)) return;
            const unsigned sidx = __float_as_uint(p.w);
            float4 nv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (sidx < normals_limit) nv = __ldg(normals + sidx);
            if (!isfinite(nv.x) || !isfinite(nv.y) || !isfinite(nv.z)) return;
            double cosine = (double)dot3_rn(nv.x, nv.y, nv.z, fz0, fz1, fz2);
            if (cosine > 1.0) cosine = 1.0;
            if (cosine < -1.0) cosine = -1.0;
            double bin = ((1.0 + cosine) * 10) / 2;
            const double distance = sqrt((double)sqd);
            if (fabs(distance) < 1e-15) return;
            const float dx = __fsub_rn(p.x, q.x), dy = __fsub_rn(p.y, q.y), dz = __fsub_rn(p.z, q.z);
            double xr = (double)dot3_rn(dx, dy, dz, fx0, fx1, fx2);
            double yr = (double)dot3_rn(dx, dy, dz, fy0, fy1, fy2);
            double zr = (double)dot3_rn(dx, dy, dz, fz0, fz1, fz2);
            if (fabs(yr) < 1E-30) yr = 0;
            if (fabs(xr) < 1E-30) xr = 0;
            if (fabs(zr) < 1E-30) zr = 0;
            const int bit4 = ((yr > 0) || ((yr == 0.0) && (xr < 0))) ? 1 : 0;
            const int bit3 = ((xr > 0) || ((xr == 0.0) && (yr > 0))) ? !bit4 : bit4;
            int desc_index = ((bit4 << 3) + (bit3 << 2)) << 1;
            if ((xr * yr > 0) || (xr == 0.0)) desc_index += (fabs(xr) >= fabs(yr)) ? 0 : 4;
            else desc_index += (fabs(xr) > fabs(yr)) ? 4 : 0;
            desc_index += zr > 0 ? 1 : 0;
            desc_index += (distance > radius1_2) ? 2 : 0;
            const int step_index = (int)floor(bin + 0.5);
            const int volume_index = desc_index * 11;
            bin -= step_index;
            double w = 1 - fabs(bin);
            {   // cosine interpolation: |bin| to the next / previous shape bin
                const float fb = (float)fabs(bin);
                const int nb_step = (bin > 0) ? (step_index + 1) % 10 : (step_index + 9) % 10;
                if (fb != 0.0f) vote(volume_index + nb_step, fb);
            }
            {   // radial interpolation (branches of PCL folded: every case adds 1 - |rd| to the own bin and,
                // towards the neighbouring husk, |rd|)
                const bool outer = distance > radius1_2;
                const double rd = (distance - (outer ? radius3_4 : radius1_4)) / radius1_2;
                w += 1 - fabs(rd);
                const bool to_nb = outer ? (rd < 0) : (rd > 0);
                if (to_nb) vote((desc_index + (outer ? -2 : 2)) * 11 + step_index, (float)fabs(rd));
            }
            {   // elevation interpolation. PCL tests `inc > 90deg || (|inc - 90deg| < 1e-30 && z <= 0)`, which for a
                // monotone acos is exactly z <= 0; the angle itself only enters linearly -> fp32 acos suffices
                double inc_cos = zr / distance;
                inc_cos = fmin(1.0, fmax(-1.0, inc_cos));
                const double inc = (double)acosf((float)inc_cos);
                const bool lower = !(zr > 0);
                const double id = (inc - (lower ? RAD_135 : RAD_45)) / RAD_90;
                w += 1 - fabs(id);
                const bool to_nb = lower ? !(id > 0) : !(id < 0);
                const float fv = (float)fabs(id);
                if (to_nb && fv != 0.0f) vote((desc_index + (lower ? 1 : -1)) * 11 + step_index, fv);
            }
            if (yr != 0.0 || xr != 0.0) {  // azimuth interpolation
                const double azimuth = (double)atan2f((float)yr, (float)xr);
                const int sel = desc_index >> 2;
                double ad = (azimuth - (-RAD_PI_7_8 + RAD_45 * sel)) / RAD_45;
                ad = fmax(-0.5, fmin(ad, 0.5));
                w += 1 - fabs(ad);
                const int nbv = (ad > 0) ? ((desc_index + 4) & 31) : ((desc_index + 28) & 31);
                const float fv = (float)fabs(ad);
                if (fv != 0.0f) vote(nbv * 11 + step_index, fv);
            }
            vote(volume_index + step_index, (float)w);
        });
#else
        // Interpolation weights in fp32: every DECISION below (volume index, shape bin, which neighbour bin
        // receives the second vote) is taken on exactly the values PCL compares -- fp32 dot products, the
        // fp32 squared distance against (R/2)^2, the double shape bin -- only the weights themselves, which
        // are rounded to a 2^-fx_bits fixed-point grid anyway, are computed in single precision (relative
        // error 1e-7 against a grid of ~4e-6).  Saves the fp64 sqrt and five fp64 divisions per neighbour.
        const float r12 = (float)radius1_2, r34 = (float)radius3_4, r14 = (float)radius1_4;
        const float inv_r12 = 1.0f / r12;
        // distance > R/2  <=>  sqd > r2_4, exact for an fp32 sqd: r2_4 is R^2/4 rounded DOWN (shell_threshold)
        const float F_45 = (float)RAD_45, F_135 = (float)RAD_135, F_78 = (float)RAD_PI_7_8;
        const float INV_90 = (float)(1.0 / RAD_90), INV_45 = (float)(1.0 / RAD_45);
        for_each([&](const float4 p) {
            const float sqd = sqdist_rn(q.x, q.y, q.z, p.x, p.y, p.z);
            if (!(sqd < R2)) return;
            const unsigned sidx = __float_as_uint(p.w);
            float4 nv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (sidx < normals_limit) nv = __ldg(normals + sidx);
            if (!isfinite(nv.x) || !isfinite(nv.y) || !isfinite(nv.z)) return;
            double cosine = (double)dot3_rn(nv.x, nv.y, nv.z, fz0, fz1, fz2);
            if (cosine > 1.0) cosine = 1.0;
            if (cosine < -1.0) cosine = -1.0;
            const double bin = ((1.0 + cosine) * 10) / 2;
            if (sqd < 1e-30f) return;  // |distance| < 1e-15
            const float dist = __fsqrt_rn(sqd);
            const float dx = __fsub_rn(p.x, q.x), dy = __fsub_rn(p.y, q.y), dz = __fsub_rn(p.z, q.z);
            float xr = dot3_rn(dx, dy, dz, fx0, fx1, fx2);
            float yr = dot3_rn(dx, dy, dz, fy0, fy1, fy2);
            float zr = dot3_rn(dx, dy, dz, fz0, fz1, fz2);
            if (fabsf(yr) < 1E-30f) yr = 0.0f;
            if (fabsf(xr) < 1E-30f) xr = 0.0f;
            if (fabsf(zr) < 1E-30f) zr = 0.0f;
            const int bit4 = ((yr > 0.0f) || ((yr == 0.0f) && (xr < 0.0f))) ? 1 : 0;
            const int bit3 = ((xr > 0.0f) || ((xr == 0.0f) && (yr > 0.0f))) ? !bit4 : bit4;
            int desc_index = ((bit4 << 3) + (bit3 << 2)) << 1;
            const bool same_sign = (xr > 0.0f && yr > 0.0f) || (xr < 0.0f && yr < 0.0f);  // xr * yr > 0 without underflow
            if (same_sign || (xr == 0.0f)) desc_index += (fabsf(xr) >= fabsf(yr)) ? 0 : 4;
            else desc_index += (fabsf(xr) > fabsf(yr)) ? 4 : 0;
            desc_index += zr > 0.0f ? 1 : 0;
            const bool outer = sqd > r2_4;
            desc_index += outer ? 2 : 0;
            const int step_index = (int)floor(bin + 0.5);
            const int volume_index = desc_index * 11;
            const float fbin = (float)(bin - (double)step_index);
            float w = 1.0f - fabsf(fbin);
            {   // cosine interpolation: |bin| to the next / previous shape bin
                const float fb = fabsf(fbin);
                const int nb_step = (fbin > 0.0f) ? (step_index + 1) % 10 : (step_index + 9) % 10;
                if (fb != 0.0f) vote(volume_index + nb_step, fb);
            }
            {   // radial interpolation
                const float rd = (dist - (outer ? r34 : r14)) * inv_r12;
                w += 1.0f - fabsf(rd);
                const bool to_nb = outer ? (rd < 0.0f) : (rd > 0.0f);
                if (to_nb) vote((desc_index + (outer ? -2 : 2)) * 11 + step_index, fabsf(rd));
            }
            {   // elevation interpolation (z <= 0 is PCL's `inclination > 90 deg` test, see above)
                const float inc_cos = fminf(1.0f, fmaxf(-1.0f, zr / dist));
                const float inc = acos_poly(inc_cos);
                const bool lower = !(zr > 0.0f);
                const float id = (inc - (lower ? F_135 : F_45)) * INV_90;
                w += 1.0f - fabsf(id);
                const bool to_nb = lower ? !(id > 0.0f) : !(id < 0.0f);
                const float fv = fabsf(id);
                if (to_nb && fv != 0.0f) vote((desc_index + (lower ? 1 : -1)) * 11 + step_index, fv);
            }
            if (yr != 0.0f || xr != 0.0f) {  // azimuth interpolation
                // angle from the centre of the point's 45-degree sector: rotate (xr, yr) by minus the sector's reference
                // angle and take the arctangent of a ratio that stays below tan(22.5 deg) -- no full-range atan2
                const int sel = desc_index >> 2;
                const float cr = ((sel + 2) & 4) ? 0.92387953f : -0.92387953f, cq = ((sel + 2) & 4) ? 0.38268343f : -0.38268343f;
                const bool steep = ((sel + 1) & 2) != 0;  // sectors 1, 2, 5, 6: |sin| = 0.9239
                const float cs = steep ? cq : cr;                                          // cos(ref)
                const float sn = (sel < 4 ? -1.0f : 1.0f) * (steep ? 0.92387953f : 0.38268343f);  // sin(ref)
                const float xq = fmaf(xr, cs, yr * sn), yq = fmaf(yr, cs, -(xr * sn));
                float delta;
                if (xq > 0.0f && fabsf(yq) <= 0.47f * xq) delta = atan_sector(yq / xq);
                else delta = atan2f(yr, xr) - (F_45 * (float)sel - F_78);                // (never on consistent sector bits)
                float ad = delta * INV_45;
                ad = fmaxf(-0.5f, fminf(ad, 0.5f));
                w += 1.0f - fabsf(ad);
                const int nbv = (ad > 0.0f) ? ((desc_index + 4) & 31) : ((desc_index + 28) & 31);
                const float fv = fabsf(ad);
                if (fv != 0.0f) vote(nbv * 11 + step_index, fv);
            }
            vote(volume_index + step_index, w);
        });
#endif
    }
    __syncthreads();

    // ---- phase D: normalise, emit, binarise ----------------------------------------------------
    {
        for (unsigned i = tid; i < 352; i += SH_THREADS) sm.hist[i] = (float)sm.acc[i] * fx_inv;
        __syncthreads();
        double part = 0.0;
        for (unsigned i = tid; i < 352; i += SH_THREADS) part += (double)__fmul_rn(sm.hist[i], sm.hist[i]);
        part = warp_sum(part);
        if (lane == 0) sm.red[wid][0] = part;
        __syncthreads();
        if (tid == 0) {
            double s = 0;
            for (int w = 0; w < SH_THREADS / 32; ++w) s += sm.red[w][0];
            sm.norm = sqrt(s);
        }
        __syncthreads();
        const float f = (float)sm.norm;
        for (unsigned i = tid; i < 352; i += SH_THREADS) {
            float v = describe ? (sm.hist[i] / f) : nanf_;
            sm.hist[i] = v;
            if (shot_out) shot_out[(size_t)k * 352 + i] = v;
        }
        __syncthreads();
        pack_bits_block<SH_THREADS>(sm.hist, sm.words, tid);
        if (tid < 6) bits_out[(size_t)k * 6 + tid] = ((uint64_t)sm.words[2 * tid + 1] << 32) | sm.words[2 * tid];
    }
}

// standalone binarisation of caller-provided SHOT floats: one warp per descriptor
__global__ void __launch_bounds__(128)
binarize_kernel(const float* __restrict__ shot, unsigned k, uint64_t* __restrict__ bits) {
    const unsigned warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= k) return;
    const float4* s4 = reinterpret_cast<const float4*>(shot + (size_t)warp * 352);
    unsigned nib[3] = {0, 0, 0};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const unsigned j = r * 32 + lane;
        if (j < 88) {
            const float4 v = __ldg(s4 + j);
            nib[r] = bshot_nibble(v.x, v.y, v.z, v.w);
        }
    }
    // word w (8 nibbles) = nibbles 8w..8w+7 ; lanes 8a..8a+7 of round r hold word 4r + a
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        unsigned v = nib[r] << ((lane & 7) * 4);
        v |= __shfl_xor_sync(0xffffffffu, v, 1);
        v |= __shfl_xor_sync(0xffffffffu, v, 2);
        v |= __shfl_xor_sync(0xffffffffu, v, 4);
        nib[r] = v;  // every lane of an 8-group holds the group's word
    }
    // words 0..10 (+ word 11 = 0): lane l < 6 assembles u64 l from words 2l, 2l+1
    unsigned lo = 0, hi = 0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        // word index 4r + a lives in lanes 8a..8a+7
        for (int a = 0; a < 4; ++a) {
            const unsigned wv = __shfl_sync(0xffffffffu, nib[r], 8 * a);
            const int widx = 4 * r + a;
            if (widx == 2 * (int)lane) lo = wv;
            if (widx == 2 * (int)lane + 1) hi = wv;
        }
    }
    if (lane < 6) bits[(size_t)warp * 6 + lane] = ((uint64_t)hi << 32) | lo;
}

// Keypoints differ ten-fold in cost (126 .. 2800 neighbours) and a CTA per keypoint in index order leaves the SMs idle for
// ~11 % of the launch while the last heavy ones finish.  Longest-processing-time-first: the keypoints are taken in the
// order of the radius that held max_nn neighbours in the detector pass (small radius = dense = expensive).  One CTA,
// 256-bin counting sort; the order only decides WHEN a keypoint is processed, never what is computed.
constexpr int SO_PER = 16;  // keypoints per thread held in registers (1024 threads: 16 384 keypoints in one sweep)
__global__ void __launch_bounds__(1024)
shot_order_kernel(const float4* __restrict__ kp, const int* __restrict__ kp_count, unsigned kcap, const float* __restrict__ rho_hint, unsigned n_points,
                  float R, unsigned* __restrict__ order) {
    __shared__ unsigned hist[256];
    const unsigned tid = threadIdx.x;
    const unsigned K = min(kcap, (unsigned)max(*kp_count, 0));
    if (tid < 256) hist[tid] = 0u;
    __syncthreads();
    const float scale = 255.0f / R;
    for (unsigned k0 = 0; k0 < K; k0 += 1024 * SO_PER) {   // one round unless K > 16 384
        // all loads of a thread are independent: the two dependent round trips (keypoint -> its radius) overlap 16-fold
        unsigned idx[SO_PER], bin[SO_PER];
#pragma unroll
        for (int j = 0; j < SO_PER; ++j) {
            const unsigned k = k0 + tid + 1024u * j;
            idx[j] = k < K ? __float_as_uint(kp[k].w) : 0xFFFFFFFFu;
        }
#pragma unroll
        for (int j = 0; j < SO_PER; ++j) {
            const float rho = idx[j] < n_points ? rho_hint[idx[j]] : R;
            bin[j] = (rho > 0.0f) ? min(255u, (unsigned)(rho * scale)) : 255u;
        }
        if (k0 == 0 && K <= 1024 * SO_PER) {   // the common case: histogram, scan and scatter from registers
#pragma unroll
            for (int j = 0; j < SO_PER; ++j)
                if (k0 + tid + 1024u * j < K) atomicAdd(&hist[bin[j]], 1u);
            __syncthreads();
            if (tid < 32) {   // exclusive scan of 256 bins by one warp: 8 bins per lane
                unsigned h[8], sum = 0;
#pragma unroll
                for (int i = 0; i < 8; ++i) { h[i] = hist[tid * 8 + i]; sum += h[i]; }
                unsigned inc = sum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned up = __shfl_up_sync(0xffffffffu, inc, o);
                    if (tid >= (unsigned)o) inc += up;
                }
                unsigned run = inc - sum;
#pragma unroll
                for (int i = 0; i < 8; ++i) { hist[tid * 8 + i] = run; run += h[i]; }
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < SO_PER; ++j) {
                const unsigned k = k0 + tid + 1024u * j;
                if (k < K) order[atomicAdd(&hist[bin[j]], 1u)] = k;
            }
            return;
        }
        // more keypoints than one sweep holds: plain index order for this launch (correct, only the schedule differs)
#pragma unroll
        for (int j = 0; j < SO_PER; ++j) {
            const unsigned k = k0 + tid + 1024u * j;
            if (k < K) order[k] = k;
        }
    }
}

// The half-radius shell test, distance > R/2, as a test on the fp32 squared distance: sqd > R^2/4.  R^2/4 is exact in
// double; the largest float not above it makes `sqd > threshold` exact for every fp32 sqd.  Rounding to nearest instead
// can round up, and a neighbour with sqd equal to that value would land in the inner shell where PCL puts it in the outer.
// Passed as a kernel parameter: the comparison reads it from the constant bank and holds no register in the vote loop.
static float shell_threshold(float radius) {
    const double q = ((double)radius * (double)radius) / 4.0;
    float t = (float)q;
    if ((double)t > q) t = nextafterf(t, 0.0f);
    return t;
}

int shot_compute(Ctx* c, float radius, bool lrf_only, bool write_shot) {
    const size_t k = c->n_kp;
    if (k == 0) return BSHOT_OK;
    if (!lrf_only) BSHOT_CUDA_TRY(cudaMemsetAsync(c->d_sum_nn, 0, sizeof(unsigned long long), c->stream));
    const unsigned limit = (unsigned)std::min(c->normals_valid, c->n_points);
    // processing order: only when the keypoints are the detector's (d_kp[i].w = surface index) and its radii are at hand
    static const bool lpt = [] { const char* e = getenv("BSHOT_SHOT_LPT"); return !e || atoi(e) != 0; }();
    const unsigned* order = nullptr;
    if (lpt && c->kp_from_detector && c->sel_valid && k >= 512) {
        shot_order_kernel<<<1, 1024, 0, c->stream>>>(c->d_kp, c->d_kp_count, (unsigned)k, c->d_rho_hint, (unsigned)c->n_points, c->sel_radius, c->d_shot_order);
        count_launch(c);
        order = c->d_shot_order;
    }
    const float r2_4 = shell_threshold(radius);
    static const int nthreads = [] { const char* e = getenv("BSHOT_SHOT_THREADS"); const int v = e ? atoi(e) : 128; return (v == 64 || v == 128 || v == 256) ? v : 128; }();
#define BSHOT_LAUNCH_SHOT(NT)                                                                                              \
    shot_kernel<NT><<<(unsigned)k, NT, 0, c->stream>>>(c->d_grid, c->d_cell_start, c->d_sorted, c->d_kp, c->d_kp_count,   \
                                                      c->d_normals, limit, radius, r2_4, lrf_only ? 1 : 0, c->d_rf, c->d_nn, \
                                                      write_shot ? c->d_shot : nullptr, c->d_bits, c->d_sum_nn, order)
    if (nthreads == 64) BSHOT_LAUNCH_SHOT(64);
    else if (nthreads == 256) BSHOT_LAUNCH_SHOT(256);
    else BSHOT_LAUNCH_SHOT(128);
#undef BSHOT_LAUNCH_SHOT
    count_launch(c);
    return check_launch("shot_kernel");
}

int binarize(Ctx* c, const float* d_shot, size_t k, uint64_t* d_bits) {
    if (k == 0) return BSHOT_OK;
    const unsigned blocks = (unsigned)((k * 32 + 127) / 128);
    binarize_kernel<<<blocks, 128, 0, c->stream>>>(d_shot, (unsigned)k, d_bits);
    count_launch(c);
    return check_launch("binarize_kernel");
}

}  // namespace bshot
