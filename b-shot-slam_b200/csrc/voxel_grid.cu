// voxel_grid.cu -- voxel-grid downsampling: pcl::VoxelGrid<PointXYZ>::applyFilter of PCL 1.8 with its default settings
// (all fields averaged, no filter field, no minimum point count), as the reference's
// bshot::calculate_voxel_grid_keypoints calls it (SURVEY row 1).
//
// The cloud comes from the host (it is not the context's cloud); nothing of the context's frame state is read or
// written.  Launches, all sized from n on the host, everything else decided on the device:
//   bbox      tiles of 1024 points: bbox of the finite points + finite count per tile; the last CTA derives inv-leaf
//             bins, multipliers, PCL's overflow test and the number of significant key bits (-> radix passes)
//   key       finite points -> (voxel index, point index), compacted in index order
//   4 x (rx_hist, rx_scatter)  stable LSD radix sort of the voxel indices, 8 bits a pass; passes beyond the significant bits
//             return at once, so the pass count costs no host round trip
//   heads, seg  first sorted position of every voxel (voxel count on the device)
//   centroid  one warp per voxel: the warp gathers 256 points at a time in parallel, then replays the fp32 sums in
//             ascending point index (shuffles), so a voxel that holds the whole cloud is no dependent chain of gathers;
//             sum / count as an IEEE division.  On overflow it writes the input cloud unchanged instead.
// Output: one buffer {count, 3 unused words, x y z records}, so one device-to-host copy returns everything.
// The arithmetic is written with explicit round-to-nearest intrinsics (and the file is compiled without FMA
// contraction): every product, difference and sum is the fp32 operation PCL performs.
#include <algorithm>

#include "stages.h"

namespace bshot {

constexpr int VG_THREADS = 256;
constexpr int VG_TILE = VG_THREADS * 4;   // points per bbox / key / head tile (4 per thread)
constexpr int RX_ITEMS = 8;               // keys per thread and radix pass
constexpr int RX_TILE = VG_THREADS * RX_ITEMS;
constexpr int RX_WARPS = VG_THREADS / 32;
constexpr int RX_PASSES = 4;              // 8-bit digits of a 32-bit key

enum VgMode : unsigned { VG_VOXELS = 0, VG_COPY = 1, VG_EMPTY = 2 };

struct VgKey {
    int min_b[3];
    unsigned mul1, mul2;    // voxel index multipliers of y and z (x: 1), modulo 2^32 as PCL's int arithmetic
};

struct VgParams {
    float bbox[6];          // min xyz, max xyz of the finite points; +-inf between calls (re-armed by the last CTA)
    unsigned ticket;        // CTAs of the bbox pass done; 0 between calls
    unsigned m;             // keyed points: the finite points in VG_VOXELS mode, else 0
    VgKey key;
    unsigned npasses;       // radix passes over the significant key bits
    unsigned mode;          // VgMode
    unsigned nvox;          // occupied voxels (seg pass)
};

// (int) of an integral float; out of int's range it saturates (PCL's conversion is undefined there)
__device__ __forceinline__ int vg_int(float f) { return __float2int_rz(f); }

__device__ __forceinline__ unsigned vg_key(float x, float y, float z, float3 inv, const VgKey& P) {
    const int i = vg_int(__fsub_rn(floorf(__fmul_rn(x, inv.x)), __int2float_rn(P.min_b[0])));
    const int j = vg_int(__fsub_rn(floorf(__fmul_rn(y, inv.y)), __int2float_rn(P.min_b[1])));
    const int k = vg_int(__fsub_rn(floorf(__fmul_rn(z, inv.z)), __int2float_rn(P.min_b[2])));
    return (unsigned)i + (unsigned)j * P.mul1 + (unsigned)k * P.mul2;
}

__device__ __forceinline__ bool load_point(const float* __restrict__ in, int stride, unsigned i, float& x, float& y, float& z) {
    const float* q = in + (size_t)i * stride;
    x = q[0]; y = q[1]; z = q[2];
    return isfinite(x) && isfinite(y) && isfinite(z);
}

// exclusive prefix of v over the block (VG_THREADS threads) in block order; *total = the sum
__device__ __forceinline__ unsigned block_excl_scan(unsigned v, unsigned* s_warp, unsigned* total) {
    const unsigned lane = lane_id(), wid = threadIdx.x >> 5;
    unsigned inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += up;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    unsigned run = inc - v, tot = 0;
    for (int w = 0; w < VG_THREADS / 32; ++w) {
        const unsigned t = s_warp[w];
        if (w < (int)wid) run += t;
        tot += t;
    }
    __syncthreads();
    if (total) *total = tot;
    return run;
}

// sum of tile_sums[0 .. blockIdx.x) by warp 0 -> *s_base
__device__ __forceinline__ void tiles_before(const unsigned* __restrict__ tile_sums, unsigned* s_base) {
    if (threadIdx.x < 32) {
        unsigned part = 0;
        for (unsigned t = threadIdx.x; t < blockIdx.x; t += 32) part += tile_sums[t];
        part = (unsigned)warp_sum((int)part);
        if (threadIdx.x == 0) *s_base = part;
    }
}

// the last CTA of the bbox pass: PCL's parameters from the box (voxel_grid.hpp, applyFilter)
__device__ void vg_params(VgParams* P, unsigned nfin, float3 inv) {
    volatile float* vb = P->bbox;
    const float mn[3] = {vb[0], vb[1], vb[2]}, mx[3] = {vb[3], vb[4], vb[5]};
    const float iv[3] = {inv.x, inv.y, inv.z};
    vb[0] = vb[1] = vb[2] = __int_as_float(0x7F800000);
    vb[3] = vb[4] = vb[5] = __int_as_float(0xFF800000);
    P->ticket = 0u;
    P->nvox = 0u;
    if (nfin == 0) { P->mode = VG_EMPTY; P->m = 0; P->npasses = 0; return; }
    // d_a = (int64)((max - min) * inv) + 1; dx * dy * dz > INT32_MAX: the output is the input cloud
    unsigned long long prod = 1;
    bool ovf = false;
    for (int a = 0; a < 3 && !ovf; ++a) {
        const float f = __fmul_rn(__fsub_rn(mx[a], mn[a]), iv[a]);
        if (!(f < 2147483648.0f)) { ovf = true; break; }
        prod *= (unsigned long long)__float2ll_rz(f) + 1ull;
        ovf = prod > 0x7FFFFFFFull;
    }
    if (ovf) { P->mode = VG_COPY; P->m = 0; P->npasses = 0; return; }
    bool in_range = true;
    int min_b[3], max_b[3];
    for (int a = 0; a < 3; ++a) {
        const float lo = floorf(__fmul_rn(mn[a], iv[a])), hi = floorf(__fmul_rn(mx[a], iv[a]));
        in_range = in_range && lo >= -2147483648.0f && hi < 2147483648.0f;
        min_b[a] = vg_int(lo);
        max_b[a] = vg_int(hi);
        P->key.min_b[a] = min_b[a];
    }
    const unsigned div0 = (unsigned)max_b[0] - (unsigned)min_b[0] + 1u, div1 = (unsigned)max_b[1] - (unsigned)min_b[1] + 1u;
    P->key.mul1 = div0;
    P->key.mul2 = div0 * div1;
    // significant key bits: every point's ijk lies in [0, ijk(max)] per axis (floor, the fp32 difference and the
    // conversion are monotone), so the key is at most B = ijk(max) . (1, div0, div0 * div1) unless that reaches 2^32
    // (then the key wraps like PCL's int and all 32 bits are sorted)
    int bits = 32;
    if (in_range) {
        double B = 0.0, mul = 1.0;
        unsigned long long Bi = 0, muli = 1;
        for (int a = 0; a < 3; ++a) {
            const int ijk = vg_int(__fsub_rn(floorf(__fmul_rn(mx[a], iv[a])), __int2float_rn(min_b[a])));
            B += (double)ijk * mul;
            if (B < 4294967296.0) Bi += (unsigned long long)ijk * muli;
            const unsigned long long dv = (unsigned long long)((unsigned)max_b[a] - (unsigned)min_b[a]) + 1ull;
            mul *= (double)dv;
            muli = mul < 4294967296.0 ? muli * dv : 0ull;
        }
        if (B < 4294967296.0) bits = Bi ? 64 - __clzll((long long)Bi) : 0;
    }
    P->npasses = (unsigned)(bits + 7) / 8u;
    P->mode = VG_VOXELS;
    P->m = nfin;
}

__global__ void __launch_bounds__(VG_THREADS)
vg_bbox_kernel(const float* __restrict__ in, unsigned n, int stride, float3 inv, VgParams* __restrict__ P, unsigned* __restrict__ tile_fin) {
    const float inf = __int_as_float(0x7F800000);
    float mn[3] = {inf, inf, inf}, mx[3] = {-inf, -inf, -inf};
    unsigned c = 0;
    const unsigned i0 = blockIdx.x * VG_TILE + threadIdx.x * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float x, y, z;
        if (i0 + k < n && load_point(in, stride, i0 + k, x, y, z)) {
            mn[0] = fminf(mn[0], x); mn[1] = fminf(mn[1], y); mn[2] = fminf(mn[2], z);
            mx[0] = fmaxf(mx[0], x); mx[1] = fmaxf(mx[1], y); mx[2] = fmaxf(mx[2], z);
            ++c;
        }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
            mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
        }
    }
    c = (unsigned)warp_sum((int)c);
    __shared__ float smn[VG_THREADS / 32][3], smx[VG_THREADS / 32][3];
    __shared__ unsigned sc[VG_THREADS / 32], s_last;
    const unsigned lane = lane_id(), wid = threadIdx.x >> 5;
    if (lane == 0) {
        for (int k = 0; k < 3; ++k) { smn[wid][k] = mn[k]; smx[wid][k] = mx[k]; }
        sc[wid] = c;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        const int k = threadIdx.x;
        float a = inf, b = -inf;
        for (int w = 0; w < VG_THREADS / 32; ++w) { a = fminf(a, smn[w][k]); b = fmaxf(b, smx[w][k]); }
        if (a <= b) { atomic_min_float(&P->bbox[k], a); atomic_max_float(&P->bbox[3 + k], b); }
    } else if (threadIdx.x == 32) {
        unsigned t = 0;
        for (int w = 0; w < VG_THREADS / 32; ++w) t += sc[w];
        tile_fin[blockIdx.x] = t;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(&P->ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        const volatile unsigned* tf = tile_fin;
        unsigned nfin = 0;
        for (unsigned t = 0; t < gridDim.x; ++t) nfin += tf[t];
        vg_params(P, nfin, inv);
    }
}

// finite points -> keys (voxel index) and values (point index) at their rank among the finite points
__global__ void __launch_bounds__(VG_THREADS)
vg_key_kernel(const float* __restrict__ in, unsigned n, int stride, float3 inv, const VgParams* __restrict__ Pg,
              const unsigned* __restrict__ tile_fin, unsigned* __restrict__ keys, unsigned* __restrict__ vals) {
    if (Pg->mode != VG_VOXELS) return;
    const VgKey P = Pg->key;
    __shared__ unsigned s_warp[VG_THREADS / 32], s_base;
    tiles_before(tile_fin, &s_base);
    const unsigned i0 = blockIdx.x * VG_TILE + threadIdx.x * 4;
    unsigned key[4], fin = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float x, y, z;
        const bool f = i0 + k < n && load_point(in, stride, i0 + k, x, y, z);
        key[k] = f ? vg_key(x, y, z, inv, P) : 0u;
        fin |= (unsigned)f << k;
    }
    unsigned run = block_excl_scan(__popc(fin), s_warp, nullptr) + s_base;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (!(fin >> k & 1u)) continue;
        keys[run] = key[k];
        vals[run] = i0 + k;
        ++run;
    }
}

// ---- stable LSD radix sort of (key, value) pairs, 8 bits a pass (also the map's sorts, gmap.cu) -----------------------
// *d_m pairs; a pass at or past *d_npasses (null: never) returns at once, so a pass count decided on the device costs no
// host round trip.  Pass p reads buffer p & 1 and writes the other.

// radix pass `pass`: 256 digit counts of each RX_TILE tile, hist[tile * 256 + digit]
template <typename K>
__global__ void __launch_bounds__(VG_THREADS)
rx_hist_kernel(const unsigned* __restrict__ d_m, const unsigned* __restrict__ d_npasses, unsigned pass, const K* __restrict__ keys0,
               const K* __restrict__ keys1, unsigned* __restrict__ hist) {
    if (d_npasses && pass >= *d_npasses) return;
    const unsigned m = *d_m, sh = 8u * pass;
    const K* __restrict__ keys = (pass & 1) ? keys1 : keys0;
    __shared__ unsigned s[256];
    s[threadIdx.x] = 0;
    __syncthreads();
    const unsigned t0 = blockIdx.x * RX_TILE;
#pragma unroll
    for (int k = 0; k < RX_ITEMS; ++k) {
        const unsigned i = t0 + k * VG_THREADS + threadIdx.x;
        if (i < m) atomicAdd(&s[(unsigned)(keys[i] >> sh) & 255u], 1u);
    }
    __syncthreads();
    hist[blockIdx.x * 256 + threadIdx.x] = s[threadIdx.x];
}

// radix pass `pass`: stable scatter.  Warp w of a tile owns its items [w * 256, (w + 1) * 256) and takes them 32 at a
// time in index order; within 32, lanes with the same digit are ranked by lane.  Position = digits before + this
// digit in earlier tiles + in earlier warps of this tile + earlier in this warp.
template <typename K>
__global__ void __launch_bounds__(VG_THREADS)
rx_scatter_kernel(const unsigned* __restrict__ d_m, const unsigned* __restrict__ d_npasses, unsigned pass, K* __restrict__ keys0,
                  unsigned* __restrict__ vals0, K* __restrict__ keys1, unsigned* __restrict__ vals1, const unsigned* __restrict__ hist) {
    if (d_npasses && pass >= *d_npasses) return;
    const unsigned m = *d_m, sh = 8u * pass;
    const K* __restrict__ kin = (pass & 1) ? keys1 : keys0;
    const unsigned* __restrict__ vin = (pass & 1) ? vals1 : vals0;
    K* __restrict__ kout = (pass & 1) ? keys0 : keys1;
    unsigned* __restrict__ vout = (pass & 1) ? vals0 : vals1;
    __shared__ unsigned s_cnt[RX_WARPS][256];
    __shared__ unsigned s_base[256], s_warp[VG_THREADS / 32];
    const unsigned lane = lane_id(), wid = threadIdx.x >> 5, d0 = threadIdx.x;
#pragma unroll
    for (int w = 0; w < RX_WARPS; ++w) s_cnt[w][d0] = 0;
    unsigned tot = 0, pre = 0;
    for (unsigned b = 0; b < gridDim.x; ++b) {
        const unsigned h = hist[b * 256 + d0];
        tot += h;
        if (b < blockIdx.x) pre += h;
    }
    s_base[d0] = block_excl_scan(tot, s_warp, nullptr) + pre;  // its __syncthreads also orders the zeroing above
    const unsigned lt = (1u << lane) - 1u;
    K key[RX_ITEMS];
    unsigned val[RX_ITEMS], dig[RX_ITEMS], loc[RX_ITEMS];
    const unsigned w0 = blockIdx.x * RX_TILE + wid * (32 * RX_ITEMS);
#pragma unroll
    for (int r = 0; r < RX_ITEMS; ++r) {
        const unsigned i = w0 + r * 32 + lane;
        key[r] = i < m ? kin[i] : (K)0;
        val[r] = i < m ? vin[i] : 0u;
        dig[r] = i < m ? (unsigned)(key[r] >> sh) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, dig[r]);
        const unsigned old = dig[r] < 256u ? s_cnt[wid][dig[r]] : 0u;
        __syncwarp();
        if (dig[r] < 256u && (peers & lt) == 0u) s_cnt[wid][dig[r]] = old + __popc(peers);
        __syncwarp();
        loc[r] = old + __popc(peers & lt);
    }
    __syncthreads();
    unsigned run = 0;
#pragma unroll
    for (int w = 0; w < RX_WARPS; ++w) {
        const unsigned c = s_cnt[w][d0];
        s_cnt[w][d0] = run;
        run += c;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RX_ITEMS; ++r) {
        if (dig[r] >= 256u) continue;
        const unsigned pos = s_base[dig[r]] + s_cnt[wid][dig[r]] + loc[r];
        kout[pos] = key[r];
        vout[pos] = val[r];
    }
}

template <typename K>
static int radix_sort_launch(Ctx* c, K* keys[2], unsigned* vals[2], unsigned* hist, const unsigned* d_m, const unsigned* d_npasses, size_t m_cap,
                             unsigned passes) {
    const unsigned rtiles = (unsigned)std::max<size_t>((m_cap + RX_TILE - 1) / RX_TILE, 1);
    for (unsigned pass = 0; pass < passes; ++pass) {
        rx_hist_kernel<K><<<rtiles, VG_THREADS, 0, c->stream>>>(d_m, d_npasses, pass, keys[0], keys[1], hist);
        rx_scatter_kernel<K><<<rtiles, VG_THREADS, 0, c->stream>>>(d_m, d_npasses, pass, keys[0], vals[0], keys[1], vals[1], hist);
    }
    count_launch(c, 2 * passes);
    return check_launch("radix sort");
}

size_t radix_hist_words(size_t m_cap) { return 256 * std::max<size_t>((m_cap + RX_TILE - 1) / RX_TILE, 1); }

int radix_sort_pairs(Ctx* c, unsigned long long* keys[2], unsigned* vals[2], unsigned* hist, const unsigned* d_m, size_t m_cap, unsigned passes) {
    return radix_sort_launch<unsigned long long>(c, keys, vals, hist, d_m, nullptr, m_cap, passes);
}

__device__ __forceinline__ unsigned vg_heads(const unsigned* __restrict__ K, unsigned m, unsigned i0, bool h[4]) {
    unsigned c = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const unsigned i = i0 + k;
        h[k] = i < m && (i == 0 || K[i] != K[i - 1]);
        c += h[k];
    }
    return c;
}

// voxel heads (first sorted position of every distinct key) per tile
__global__ void __launch_bounds__(VG_THREADS)
vg_head_count_kernel(const VgParams* __restrict__ P, const unsigned* __restrict__ keys0, const unsigned* __restrict__ keys1,
                     unsigned* __restrict__ tile_sums) {
    const unsigned m = P->m;
    const unsigned* __restrict__ K = (P->npasses & 1) ? keys1 : keys0;
    bool h[4];
    unsigned c = vg_heads(K, m, blockIdx.x * VG_TILE + threadIdx.x * 4, h);
    __shared__ unsigned s_warp[VG_THREADS / 32];
    c = (unsigned)warp_sum((int)c);
    if (lane_id() == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
        for (int w = 0; w < VG_THREADS / 32; ++w) t += s_warp[w];
        tile_sums[blockIdx.x] = t;
    }
}

// seg[v] = first sorted position of voxel v; the last thread writes seg[nvox] = m and the voxel count
__global__ void __launch_bounds__(VG_THREADS)
vg_seg_kernel(VgParams* __restrict__ P, const unsigned* __restrict__ keys0, const unsigned* __restrict__ keys1,
              const unsigned* __restrict__ tile_sums, unsigned* __restrict__ seg) {
    const unsigned m = P->m;
    const unsigned* __restrict__ K = (P->npasses & 1) ? keys1 : keys0;
    __shared__ unsigned s_warp[VG_THREADS / 32], s_base;
    tiles_before(tile_sums, &s_base);
    const unsigned i0 = blockIdx.x * VG_TILE + threadIdx.x * 4;
    bool h[4];
    const unsigned c = vg_heads(K, m, i0, h);
    unsigned run = block_excl_scan(c, s_warp, nullptr) + s_base;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (h[k]) seg[run++] = i0 + k;
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == VG_THREADS - 1) {
        seg[run] = m;
        P->nvox = run;
    }
}

// one warp per voxel: centroid = fp32 running sum in ascending point index (from +0), / (float)count
__global__ void __launch_bounds__(VG_THREADS)
vg_centroid_kernel(const VgParams* __restrict__ Pg, const unsigned* __restrict__ vals0, const unsigned* __restrict__ vals1,
                   const unsigned* __restrict__ seg, const float* __restrict__ in, unsigned n, int stride, float* __restrict__ out) {
    const VgParams P = *Pg;
    const unsigned gtid = blockIdx.x * VG_THREADS + threadIdx.x;
    if (gtid == 0) reinterpret_cast<unsigned*>(out)[0] = P.mode == VG_COPY ? n : P.nvox;
    float* rec = out + 4;
    if (P.mode == VG_COPY) {  // PCL: output = *input_ (every point, non-finite ones included)
        for (unsigned i = gtid; i < n; i += gridDim.x * VG_THREADS) {
            const float* q = in + (size_t)i * stride;
            rec[3 * (size_t)i] = q[0]; rec[3 * (size_t)i + 1] = q[1]; rec[3 * (size_t)i + 2] = q[2];
        }
        return;
    }
    const unsigned* __restrict__ V = (P.npasses & 1) ? vals1 : vals0;
    const unsigned lane = lane_id(), nwarps = gridDim.x * (VG_THREADS / 32);
    for (unsigned v = gtid / 32; v < P.nvox; v += nwarps) {
        const unsigned s = seg[v], cnt = seg[v + 1] - s;
        float sx = 0.0f, sy = 0.0f, sz = 0.0f;
        for (unsigned base = 0; base < cnt; base += 32 * RX_ITEMS) {
            float x[RX_ITEMS], y[RX_ITEMS], z[RX_ITEMS];
#pragma unroll
            for (int k = 0; k < RX_ITEMS; ++k) {
                const unsigned j = base + 32 * k + lane;
                x[k] = y[k] = z[k] = 0.0f;
                if (j < cnt) {
                    const float* q = in + (size_t)__ldg(V + s + j) * stride;
                    x[k] = q[0]; y[k] = q[1]; z[k] = q[2];
                }
            }
            const unsigned rem = min(32u * RX_ITEMS, cnt - base);
#pragma unroll
            for (int k = 0; k < RX_ITEMS; ++k) {
                if (32u * k >= rem) break;
                const unsigned lim = min(32u, rem - 32u * k);
                if (lim == 32u) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        sx = __fadd_rn(sx, __shfl_sync(0xffffffffu, x[k], j));
                        sy = __fadd_rn(sy, __shfl_sync(0xffffffffu, y[k], j));
                        sz = __fadd_rn(sz, __shfl_sync(0xffffffffu, z[k], j));
                    }
                } else {
                    for (unsigned j = 0; j < lim; ++j) {
                        sx = __fadd_rn(sx, __shfl_sync(0xffffffffu, x[k], j));
                        sy = __fadd_rn(sy, __shfl_sync(0xffffffffu, y[k], j));
                        sz = __fadd_rn(sz, __shfl_sync(0xffffffffu, z[k], j));
                    }
                }
            }
        }
        if (lane == 0) {
            const float fc = __uint2float_rn(cnt);
            rec[3 * (size_t)v] = __fdiv_rn(sx, fc);
            rec[3 * (size_t)v + 1] = __fdiv_rn(sy, fc);
            rec[3 * (size_t)v + 2] = __fdiv_rn(sz, fc);
        }
    }
}

static int vg_alloc(Ctx* c) {
    Vg& g = c->vg;
    if (g.d_in) return BSHOT_OK;
    const size_t N = std::max<size_t>(c->max_points, 1), tiles = (N + VG_TILE - 1) / VG_TILE, rtiles = (N + RX_TILE - 1) / RX_TILE;
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_in, sizeof(float) * 4 * N));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_ctl, sizeof(VgParams)));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_tile, sizeof(unsigned) * tiles));
    for (int k = 0; k < 2; ++k) {
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_keys[k], sizeof(unsigned) * N));
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_vals[k], sizeof(unsigned) * N));
    }
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_hist, sizeof(unsigned) * 256 * rtiles));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_seg, sizeof(unsigned) * (N + 1)));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_out, sizeof(float) * (4 + 3 * N)));
    BSHOT_CUDA_TRY(cudaMallocHost((void**)&g.h_out, sizeof(float) * (4 + 3 * N)));
    VgParams p{};
    p.bbox[0] = p.bbox[1] = p.bbox[2] = __builtin_huge_valf();
    p.bbox[3] = p.bbox[4] = p.bbox[5] = -__builtin_huge_valf();
    BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_ctl, &p, sizeof(p), cudaMemcpyHostToDevice, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return BSHOT_OK;
}

void vg_free(Ctx* c) {
    Vg& g = c->vg;
    void* ptrs[] = {g.d_in, g.d_ctl, g.d_tile, g.d_keys[0], g.d_keys[1], g.d_vals[0], g.d_vals[1], g.d_hist, g.d_seg, g.d_out};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (g.h_out) cudaFreeHost(g.h_out);
    g = Vg();
}

int voxel_grid(Ctx* c, const float* xyz, size_t n, int stride_floats, const float inv[3], size_t cap, size_t* count_out) {
    BSHOT_TRY(vg_alloc(c));
    Vg& g = c->vg;
    if (n == 0) { *count_out = 0; return BSHOT_OK; }
    const unsigned nn = (unsigned)n;
    const float3 iv = make_float3(inv[0], inv[1], inv[2]);
    const unsigned tiles = (nn + VG_TILE - 1) / VG_TILE;
    const unsigned cblocks = std::min<unsigned>((nn + RX_WARPS - 1) / RX_WARPS, (unsigned)c->sm_count * 16u);
    VgParams* P = reinterpret_cast<VgParams*>(g.d_ctl);
    cudaStream_t s = c->stream;
    BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_in, xyz, sizeof(float) * stride_floats * n, cudaMemcpyHostToDevice, s));
    vg_bbox_kernel<<<tiles, VG_THREADS, 0, s>>>(g.d_in, nn, stride_floats, iv, P, g.d_tile);
    vg_key_kernel<<<tiles, VG_THREADS, 0, s>>>(g.d_in, nn, stride_floats, iv, P, g.d_tile, g.d_keys[0], g.d_vals[0]);
    BSHOT_TRY(radix_sort_launch<unsigned>(c, g.d_keys, g.d_vals, g.d_hist, &P->m, &P->npasses, n, RX_PASSES));
    vg_head_count_kernel<<<tiles, VG_THREADS, 0, s>>>(P, g.d_keys[0], g.d_keys[1], g.d_tile);
    vg_seg_kernel<<<tiles, VG_THREADS, 0, s>>>(P, g.d_keys[0], g.d_keys[1], g.d_tile, g.d_seg);
    vg_centroid_kernel<<<cblocks, VG_THREADS, 0, s>>>(P, g.d_vals[0], g.d_vals[1], g.d_seg, g.d_in, nn, stride_floats, g.d_out);
    count_launch(c, 5);
    BSHOT_TRY(check_launch("voxel_grid"));
    BSHOT_CUDA_TRY(cudaMemcpyAsync(g.h_out, g.d_out, sizeof(float) * (4 + 3 * std::min(cap, n)), cudaMemcpyDeviceToHost, s));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(s));
    *count_out = (size_t)reinterpret_cast<const unsigned*>(g.h_out)[0];
    return BSHOT_OK;
}

}  // namespace bshot
