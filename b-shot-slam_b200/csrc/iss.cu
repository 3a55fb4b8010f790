// iss.cu -- ISS keypoints (PCL 1.8 ISSKeypoint3D::detectKeypoints, border radius 0) and the keypoint repeatability
// measure of the reference's kp_test driver (src/lidar_odometry.cpp:392-461, SURVEY rows 10-11).
//
// Runs on the cloud the context holds, over the cell-sorted points and the voxel table of grid_build; nothing of the
// frame path (keypoints, normals, fused sums, previous frame, map) is read or written.  Four launches:
//   saliency  one warp per 32 consecutive cell-sorted points: for each point in turn the warp sweeps the row segments
//             of its r_s ball (fp32 distance test, fp64 scatter sums about the point, warp reduction in a fixed order);
//             lane t keeps the sums of point t and then solves its own 3x3 (eigh3_jacobi), so the eigen-solves run
//             32 wide.  Writes third_eigen_value per sorted position (0 = not salient) and optionally lambda1..3 per
//             original index.
//   non-max   the same warp layout over the r_nm ball: points with third_eigen_value > 0, at least min_neighbors
//             neighbours and no neighbour with a strictly larger value are flagged (by original index).
//   count + compact  flags -> keypoint records {index, x, y, z} in ascending index, the count in record 0, so one
//             device-to-host copy returns everything.
// Neighbourhoods are unbounded: every loop walks the row segments of the ball, any radius is exact.
#include <algorithm>

#include "eigh3.cuh"
#include "nbr.cuh"
#include "stages.h"

namespace bshot {

constexpr int ISS_THREADS = 256;
constexpr int ISS_PPW = 32;                          // points per warp (one per lane for the eigen-solve)
constexpr int ISS_PPB = ISS_PPW * ISS_THREADS / 32;  // points per block
constexpr int CMP_THREADS = 256;
constexpr int CMP_TILE = CMP_THREADS * 4;            // flags per compaction block (4 per thread)

// calls f(j, q) for every cell-sorted point q = sorted[j] of the row segments that may lie within R of p, lanes striding
// over each segment; the caller applies the exact distance test
template <typename F>
__device__ __forceinline__ void for_each_candidate(const GridParams& g, const unsigned* __restrict__ cell_start,
                                                   const float4* __restrict__ sorted, const float4 p, float R, unsigned lane,
                                                   F&& f) {
    const RowRange rr = row_range(g, p.y, p.z, R);
    for (int r = 0; r < rr.nrows; ++r) {
        int iy, iz;
        row_coords(rr, r, iy, iz);
        unsigned s, e;
        if (!row_segment(g, cell_start, p.x, p.y, p.z, R, iy, iz, s, e)) continue;
        for (unsigned j = s + lane; j < e; j += 32) f(j, __ldg(sorted + j));
    }
}

__global__ void __launch_bounds__(ISS_THREADS)
iss_saliency_kernel(const GridParams* __restrict__ gp, const unsigned* __restrict__ cell_start, const float4* __restrict__ sorted,
                    float rs, int min_nn, double g21, double g32, double* __restrict__ l3_sorted, double* __restrict__ eig_out) {
    const GridParams g = *gp;
    const unsigned nb = __ldg(cell_start + g.ncells);  // binned (finite) points
    const unsigned lane = lane_id();
    const unsigned base = (blockIdx.x * ISS_THREADS + threadIdx.x) / 32 * ISS_PPW;
    if (base >= nb) return;
    const float R2 = (float)((double)rs * (double)rs);  // PCL: static_cast<float>(radius * radius)
    double mine[6] = {0, 0, 0, 0, 0, 0};
    int mine_n = 0;
    const unsigned npts = min((unsigned)ISS_PPW, nb - base);
    for (unsigned t = 0; t < npts; ++t) {
        const float4 p = __ldg(sorted + base + t);
        const double px = (double)p.x, py = (double)p.y, pz = (double)p.z;
        double s[6] = {0, 0, 0, 0, 0, 0};
        int n = 0;
        for_each_candidate(g, cell_start, sorted, p, rs, lane, [&](unsigned, const float4 q) {
            if (!(sqdist_rn(p.x, p.y, p.z, q.x, q.y, q.z) < R2)) return;
            const double dx = (double)q.x - px, dy = (double)q.y - py, dz = (double)q.z - pz;
            s[0] += dx * dx; s[1] += dx * dy; s[2] += dx * dz;
            s[3] += dy * dy; s[4] += dy * dz; s[5] += dz * dz;
            ++n;
        });
#pragma unroll
        for (int k = 0; k < 6; ++k) s[k] = warp_sum(s[k]);
        n = warp_sum(n);
        if (lane == t) {
#pragma unroll
            for (int k = 0; k < 6; ++k) mine[k] = s[k];
            mine_n = n;
        }
    }
    if (lane >= npts) return;
    double lam1 = 0.0, lam2 = 0.0, lam3 = 0.0;
    if (mine_n >= min_nn) {  // fewer neighbours: PCL leaves the scatter matrix zero
        double w[3], V[3][3];
        eigh3_jacobi(mine, w, V);
        lam1 = w[2]; lam2 = w[1]; lam3 = w[0];
    }
    // non-finite eigenvalues or lambda3 < 0: PCL `continue`s and leaves third_eigen_value to whatever the buffer held;
    // defined here as "not salient"
    const bool ok = isfinite(lam1) && isfinite(lam2) && isfinite(lam3) && lam3 >= 0.0;
    const bool salient = ok && (lam2 / lam1 < g21) && (lam3 / lam2 < g32);
    l3_sorted[base + lane] = salient ? lam3 : 0.0;
    if (eig_out) {
        const unsigned orig = __float_as_uint(__ldg(sorted + base + lane).w);
        eig_out[3 * (size_t)orig] = lam1;
        eig_out[3 * (size_t)orig + 1] = lam2;
        eig_out[3 * (size_t)orig + 2] = lam3;
    }
}

__global__ void __launch_bounds__(ISS_THREADS)
iss_nonmax_kernel(const GridParams* __restrict__ gp, const unsigned* __restrict__ cell_start, const float4* __restrict__ sorted,
                  float rnm, int min_nn, const double* __restrict__ l3_sorted, unsigned char* __restrict__ flag) {
    const GridParams g = *gp;
    const unsigned nb = __ldg(cell_start + g.ncells);
    const unsigned lane = lane_id();
    const unsigned base = (blockIdx.x * ISS_THREADS + threadIdx.x) / 32 * ISS_PPW;
    if (base >= nb) return;
    const float R2 = (float)((double)rnm * (double)rnm);
    const unsigned npts = min((unsigned)ISS_PPW, nb - base);
    for (unsigned t = 0; t < npts; ++t) {
        const double own = __ldg(l3_sorted + base + t);
        if (!(own > 0.0)) continue;
        const float4 p = __ldg(sorted + base + t);
        int n = 0;
        bool larger = false;
        for_each_candidate(g, cell_start, sorted, p, rnm, lane, [&](unsigned j, const float4 q) {
            if (!(sqdist_rn(p.x, p.y, p.z, q.x, q.y, q.z) < R2)) return;
            ++n;
            if (own < __ldg(l3_sorted + j)) larger = true;
        });
        n = warp_sum(n);
        larger = __any_sync(0xffffffffu, larger);
        if (lane == 0 && n >= min_nn && !larger) flag[__float_as_uint(p.w)] = 1;
    }
}

// keypoints per tile of CMP_TILE flags
__global__ void __launch_bounds__(CMP_THREADS)
iss_count_kernel(const unsigned char* __restrict__ flag, unsigned n, unsigned* __restrict__ tile_sums) {
    __shared__ unsigned warp_tot[CMP_THREADS / 32];
    const unsigned i0 = blockIdx.x * CMP_TILE + threadIdx.x * 4;
    unsigned c = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) c += (i0 + k < n) ? flag[i0 + k] : 0u;
    c = (unsigned)warp_sum((int)c);
    if (lane_id() == 0) warp_tot[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
        for (int w = 0; w < CMP_THREADS / 32; ++w) t += warp_tot[w];
        tile_sums[blockIdx.x] = t;
    }
}

// flags -> records {index, x, y, z} at 1 + rank (ascending index); record 0 .x = keypoint count
__global__ void __launch_bounds__(CMP_THREADS)
iss_compact_kernel(const unsigned char* __restrict__ flag, unsigned n, const unsigned* __restrict__ tile_sums,
                   const float4* __restrict__ pts, int4* __restrict__ rec) {
    __shared__ unsigned warp_tot[CMP_THREADS / 32];
    __shared__ unsigned tile_base;
    const unsigned lane = lane_id(), wid = threadIdx.x >> 5;
    if (wid == 0) {  // keypoints of the tiles before this one
        unsigned part = 0;
        for (unsigned t = lane; t < blockIdx.x; t += 32) part += tile_sums[t];
        part = (unsigned)warp_sum((int)part);
        if (lane == 0) tile_base = part;
    }
    const unsigned i0 = blockIdx.x * CMP_TILE + threadIdx.x * 4;
    unsigned f[4], c = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) { f[k] = (i0 + k < n) ? flag[i0 + k] : 0u; c += f[k]; }
    unsigned inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += up;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    unsigned run = tile_base + inc - c;
    for (unsigned w = 0; w < wid; ++w) run += warp_tot[w];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (!f[k]) continue;
        const float4 p = pts[i0 + k];
        rec[1 + run] = make_int4((int)(i0 + k), __float_as_int(p.x), __float_as_int(p.y), __float_as_int(p.z));
        ++run;
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == CMP_THREADS - 1) rec[0] = make_int4((int)run, 0, 0, 0);
}

static int iss_alloc(Ctx* c) {
    Iss& s = c->iss;
    if (s.d_l3) return BSHOT_OK;
    const size_t N = c->max_points, tiles = (N + CMP_TILE - 1) / CMP_TILE;
    BSHOT_CUDA_TRY(cudaMalloc((void**)&s.d_l3, sizeof(double) * N));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&s.d_eig, sizeof(double) * 3 * N));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&s.d_flag, N));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&s.d_tile_sums, sizeof(unsigned) * tiles));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&s.d_rec, sizeof(int4) * (N + 1)));
    BSHOT_CUDA_TRY(cudaMallocHost((void**)&s.h_rec, sizeof(int4) * (N + 1)));
    return BSHOT_OK;
}

void iss_free(Ctx* c) {
    Iss& s = c->iss;
    void* ptrs[] = {s.d_l3, s.d_eig, s.d_flag, s.d_tile_sums, s.d_rec};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (s.h_rec) cudaFreeHost(s.h_rec);
    s = Iss();
}

int iss_detect(Ctx* c, float rs, float rnm, double g21, double g32, int min_nn, size_t cap, bool want_eig, size_t* count_out) {
    BSHOT_TRY(iss_alloc(c));
    Iss& s = c->iss;
    const size_t n = c->n_points;
    if (n == 0) { *count_out = 0; return BSHOT_OK; }
    const unsigned nn = (unsigned)n;
    if (want_eig) BSHOT_CUDA_TRY(cudaMemsetAsync(s.d_eig, 0, sizeof(double) * 3 * n, c->stream));  // points that are not binned
    BSHOT_CUDA_TRY(cudaMemsetAsync(s.d_flag, 0, n, c->stream));
    const unsigned blocks = (nn + ISS_PPB - 1) / ISS_PPB, tiles = (nn + CMP_TILE - 1) / CMP_TILE;
    iss_saliency_kernel<<<blocks, ISS_THREADS, 0, c->stream>>>(c->d_grid, c->d_cell_start, c->d_sorted, rs, min_nn, g21, g32, s.d_l3,
                                                               want_eig ? s.d_eig : nullptr);
    iss_nonmax_kernel<<<blocks, ISS_THREADS, 0, c->stream>>>(c->d_grid, c->d_cell_start, c->d_sorted, rnm, min_nn, s.d_l3, s.d_flag);
    iss_count_kernel<<<tiles, CMP_THREADS, 0, c->stream>>>(s.d_flag, nn, s.d_tile_sums);
    iss_compact_kernel<<<tiles, CMP_THREADS, 0, c->stream>>>(s.d_flag, nn, s.d_tile_sums, c->d_pts, s.d_rec);
    count_launch(c, 4);
    BSHOT_TRY(check_launch("iss_detect"));
    BSHOT_CUDA_TRY(cudaMemcpyAsync(s.h_rec, s.d_rec, sizeof(int4) * (1 + std::min(cap, n)), cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    *count_out = (size_t)s.h_rec[0].x;
    return BSHOT_OK;
}

// ---- keypoint repeatability (kp_test, src/lidar_odometry.cpp:392-445) -----------------------------------------------
struct Pose12 {
    float m[12];
};

// the points moved by the pose as updateMap moves keypoints (pose_apply_rn), w = 0
__global__ void rep_pose_kernel(const float* __restrict__ xyz, unsigned n, Pose12 P, int has, float4* __restrict__ out) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = xyz[3 * (size_t)i], y = xyz[3 * (size_t)i + 1], z = xyz[3 * (size_t)i + 2];
    const float3 q = has ? pose_apply_rn(P.m, x, y, z) : make_float3(x, y, z);
    out[i] = make_float4(q.x, q.y, q.z, 0.0f);
}

// one warp per point of A: nearest point of B by fp32 squared distance, lowest index on ties
__global__ void __launch_bounds__(256)
rep_nn_kernel(const float4* __restrict__ a, unsigned na, const float4* __restrict__ b, unsigned nb, float r2, int* __restrict__ nn_idx,
              float* __restrict__ nn_dist, unsigned* __restrict__ hits) {
    const unsigned w = (blockIdx.x * blockDim.x + threadIdx.x) / 32, lane = lane_id();
    if (w >= na) return;
    const float4 p = a[w];
    float best = __int_as_float(0x7F800000);
    int bi = -1;
    for (unsigned j = lane; j < nb; j += 32) {
        const float4 q = b[j];
        const float d = sqdist_rn(p.x, p.y, p.z, q.x, q.y, q.z);
        if (d < best) { best = d; bi = (int)j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ob < best || (ob == best && (unsigned)oi < (unsigned)bi)) { best = ob; bi = oi; }
    }
    if (lane == 0) {
        nn_idx[w] = bi;
        nn_dist[w] = bi >= 0 ? __fsqrt_rn(best) : __int_as_float(0x7F800000);
        if (best < r2) atomicAdd(hits, 1u);
    }
}

int kp_repeatability(Ctx* c, const float* a_xyz, size_t na, const float* a_pose, const float* b_xyz, size_t nb, const float* b_pose, float radius,
                     int* nn_idx_out, float* nn_dist_out, size_t* hits_out) {
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t bytes = up(12 * na) + up(12 * nb) + up(16 * na) + up(16 * nb) + up(4 * na) + up(4 * na) + up(4);
    BSHOT_TRY(scratch_reserve(c, 2, bytes));
    char* base = (char*)c->d_pre[2];
    size_t off = 0;
    auto take = [&](size_t b) { char* r = base + off; off += up(b); return r; };
    float* d_a = (float*)take(12 * na);
    float* d_b = (float*)take(12 * nb);
    float4* d_ta = (float4*)take(16 * na);
    float4* d_tb = (float4*)take(16 * nb);
    int* d_idx = (int*)take(4 * na);
    float* d_dist = (float*)take(4 * na);
    unsigned* d_hits = (unsigned*)take(4);
    if (na) BSHOT_CUDA_TRY(cudaMemcpyAsync(d_a, a_xyz, 12 * na, cudaMemcpyHostToDevice, c->stream));
    if (nb) BSHOT_CUDA_TRY(cudaMemcpyAsync(d_b, b_xyz, 12 * nb, cudaMemcpyHostToDevice, c->stream));
    BSHOT_CUDA_TRY(cudaMemsetAsync(d_hits, 0, sizeof(unsigned), c->stream));
    Pose12 pa{}, pb{};
    if (a_pose) for (int k = 0; k < 12; ++k) pa.m[k] = a_pose[k];
    if (b_pose) for (int k = 0; k < 12; ++k) pb.m[k] = b_pose[k];
    const float r2 = (float)((double)radius * (double)radius);
    unsigned launches = 0;
    if (nb) { rep_pose_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, c->stream>>>(d_b, (unsigned)nb, pb, b_pose != nullptr, d_tb); ++launches; }
    if (na) {
        rep_pose_kernel<<<(unsigned)((na + 255) / 256), 256, 0, c->stream>>>(d_a, (unsigned)na, pa, a_pose != nullptr, d_ta);
        rep_nn_kernel<<<(unsigned)((na * 32 + 255) / 256), 256, 0, c->stream>>>(d_ta, (unsigned)na, d_tb, (unsigned)nb, r2, d_idx, d_dist, d_hits);
        launches += 2;
    }
    count_launch(c, launches);
    BSHOT_TRY(check_launch("kp_repeatability"));
    unsigned* h_hits = reinterpret_cast<unsigned*>(&c->h_scratch[48]);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(h_hits, d_hits, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    if (nn_idx_out && na) BSHOT_CUDA_TRY(cudaMemcpyAsync(nn_idx_out, d_idx, 4 * na, cudaMemcpyDeviceToHost, c->stream));
    if (nn_dist_out && na) BSHOT_CUDA_TRY(cudaMemcpyAsync(nn_dist_out, d_dist, 4 * na, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (hits_out) *hits_out = *h_hits;
    return BSHOT_OK;
}

}  // namespace bshot
