// grid.cu -- cloud ingest + voxel table build (SURVEY 8a row a1 + the kd-tree builds it replaces).
//
// Replaces LidarOdometry::setSrcFrame (src/lidar_odometry.cpp:29-41: Vector3f -> PointXYZ copy) and
// the three pcl::KdTreeFLANN builds per frame (src/lidar_odometry.cpp:53-54,
// include/bshot_bits.h:52-53, PCL-internal in SHOT).  The search structure is a perfect spatial
// hash: cell (ix,iy,iz) of edge `cell` over the cloud's bounding box, linearised x-fastest, so that
// the cells of one (iy,iz) row that a radius query needs are ONE contiguous range of the
// cell-sorted point array (float4, w = original index) -> coalesced float4 row-segment gathers.
// Everything is sized on the device (no host round trip), six launches: convert + bbox (the last CTA to finish turns
// the box into the grid parameters and re-arms the box for the next frame) -> zero tables -> count -> tile sums ->
// exclusive scan (every tile adds up the sums of the tiles before it) -> scatter.  The count pass also fills point counts of the 2^3 / 4^3 / 8^3-cell cubes
// and the scatter pass cuts the grid into the query BLOCKS of the tiled neighbourhood kernels (tile.cuh): the
// coarsest cube around a point that holds at most TL_QCAP points (denser single cells are sliced).
#include "common.cuh"
#include "nbr.cuh"
#include "tile.cuh"

namespace bshot {

constexpr int GB_THREADS = 256;
constexpr int SCAN_THREADS = 1024;
constexpr int SCAN_ITEMS = 8;                        // cells per thread
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS; // 8192 cells per block

__device__ void grid_params_from_bbox(float* bbox, unsigned n, float cell0, float yz_mul, unsigned max_cells, GridParams* g) {
    GridParams p;
    float mn[3] = {bbox[0], bbox[1], bbox[2]}, mx[3] = {bbox[3], bbox[4], bbox[5]};
    if (!(mn[0] <= mx[0])) { mn[0] = mn[1] = mn[2] = 0.0f; mx[0] = mx[1] = mx[2] = 0.0f; }  // empty cloud
    float cell = cell0;
    for (;;) {
        const double cyz = (double)cell * (double)yz_mul;
        const double cells = (floor((double)(mx[0] - mn[0]) / cell) + 1.0) * (floor((double)(mx[1] - mn[1]) / cyz) + 1.0) *
                             (floor((double)(mx[2] - mn[2]) / cyz) + 1.0);
        if (cells <= (double)max_cells) break;
        cell *= 1.125f;
    }
    p.ox = mn[0]; p.oy = mn[1]; p.oz = mn[2];
    p.cell = cell;
    p.inv_cell = 1.0f / cell;
    p.cell_yz = cell * yz_mul;
    p.inv_cell_yz = 1.0f / p.cell_yz;
    p.nx = cell_coord(mx[0], p.ox, p.inv_cell) + 1;
    p.ny = cell_coord(mx[1], p.oy, p.inv_cell_yz) + 1;
    p.nz = cell_coord(mx[2], p.oz, p.inv_cell_yz) + 1;
    // cell_coord rounds in fp32; shrink until the table fits (never triggers in practice)
    while ((double)p.nx * p.ny * p.nz > (double)max_cells) {
        if (p.nx >= p.ny && p.nx >= p.nz) p.nx--; else if (p.ny >= p.nz) p.ny--; else p.nz--;
    }
    p.ncells = (unsigned)p.nx * (unsigned)p.ny * (unsigned)p.nz;
    p.npoints = n;
    *g = p;
    // re-arm the box for the next frame (it starts armed: bshot_ctx_create)
    bbox[0] = bbox[1] = bbox[2] = __int_as_float(0x7F800000);
    bbox[3] = bbox[4] = bbox[5] = __int_as_float(0xFF800000);
}

// raw caller layout -> float4 (x,y,z,1) + bounding box of the finite points; the last CTA to finish (ticket) derives the
// grid parameters from the box.  bbox[6] is the ticket counter (as unsigned), kept at zero between frames.
__global__ void __launch_bounds__(GB_THREADS)
convert_bbox_kernel(const float* __restrict__ raw, unsigned n, int stride, float4* __restrict__ pts,
                    float* __restrict__ bbox, float cell0, float yz_mul, unsigned max_cells, GridParams* __restrict__ g) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const float inf = __int_as_float(0x7F800000);
    float mn[3] = {inf, inf, inf}, mx[3] = {-inf, -inf, -inf};
    if (i < n) {
        float x, y, z;
        if (stride == 4) {
            const float4 v = reinterpret_cast<const float4*>(raw)[i];
            x = v.x; y = v.y; z = v.z;
        } else {
            x = raw[(size_t)i * 3]; y = raw[(size_t)i * 3 + 1]; z = raw[(size_t)i * 3 + 2];
        }
        pts[i] = make_float4(x, y, z, 1.0f);
        if (isfinite(x) && isfinite(y) && isfinite(z)) {
            mn[0] = mx[0] = x; mn[1] = mx[1] = y; mn[2] = mx[2] = z;
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
    __shared__ float smn[GB_THREADS / 32][3], smx[GB_THREADS / 32][3];
    __shared__ unsigned s_last;
    const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0)
        for (int k = 0; k < 3; ++k) { smn[wid][k] = mn[k]; smx[wid][k] = mx[k]; }
    __syncthreads();
    if (threadIdx.x < 3) {
        const int k = threadIdx.x;
        float a = inf, b = -inf;
        for (int w = 0; w < GB_THREADS / 32; ++w) { a = fminf(a, smn[w][k]); b = fmaxf(b, smx[w][k]); }
        if (a <= b) { atomic_min_float(&bbox[k], a); atomic_max_float(&bbox[3 + k], b); }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(reinterpret_cast<unsigned*>(bbox) + 6, 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        volatile float* vb = bbox;
        float box[6] = {vb[0], vb[1], vb[2], vb[3], vb[4], vb[5]};
        grid_params_from_bbox(box, n, cell0, yz_mul, max_cells, g);
#pragma unroll
        for (int k = 0; k < 6; ++k) vb[k] = box[k];
        reinterpret_cast<unsigned*>(bbox)[6] = 0u;
    }
}

// empty cloud: no convert launch, the parameters of an empty grid
__global__ void grid_params_empty_kernel(float* bbox, float cell0, float yz_mul, unsigned max_cells, GridParams* g) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        float box[6] = {__int_as_float(0x7F800000), __int_as_float(0x7F800000), __int_as_float(0x7F800000),
                        __int_as_float(0xFF800000), __int_as_float(0xFF800000), __int_as_float(0xFF800000)};
        grid_params_from_bbox(box, 0u, cell0, yz_mul, max_cells, g);
    }
}

__global__ void zero_cells_kernel(const GridParams* __restrict__ g, unsigned* __restrict__ cursor, unsigned* __restrict__ lvl,
                                  unsigned* __restrict__ nblocks) {
    const unsigned n = g->ncells;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) cursor[i] = 0;
    const unsigned nl = lvl_total(*g);
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < nl; i += gridDim.x * blockDim.x) lvl[i] = 0;
    if (blockIdx.x == 0 && threadIdx.x < (unsigned)kBlockClasses) nblocks[16 + threadIdx.x] = 0;
}

// one atomicAdd per RUN of equal keys inside a warp: lidar points arrive in firing order, neighbouring lanes mostly
// fall into the same cell / cube, and thousands of points share one 8^3-cell cube (a hot address otherwise)
__device__ __forceinline__ void run_add(unsigned* __restrict__ table, unsigned key, bool valid, unsigned lane) {
    const unsigned prev = __shfl_up_sync(0xffffffffu, key, 1);
    const bool head = (lane == 0) || (key != prev);
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    if (head && valid) {
        const unsigned next = heads & ~((2u << lane) - 1u);  // heads above this lane (lane 31: 2u << 31 == 0 -> mask 0xFFFFFFFF -> none)
        const unsigned end = (lane == 31 || next == 0u) ? 32u : (unsigned)(__ffs(next) - 1);
        atomicAdd(&table[key], end - lane);
    }
}

__global__ void __launch_bounds__(GB_THREADS)
count_kernel(const float4* __restrict__ pts, unsigned n, const GridParams* __restrict__ gp,
             unsigned* __restrict__ cell_of, unsigned* __restrict__ cursor, unsigned* __restrict__ lvl) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
    const GridParams g = *gp;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < n) p = pts[i];
    const bool valid = i < n && isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
    unsigned cid = 0xFFFFFFFFu, k1 = 0xFFFFFFFFu, k2 = 0xFFFFFFFFu, k3 = 0xFFFFFFFFu;
    if (valid) {
        const int ix = min(max(cell_coord(p.x, g.ox, g.inv_cell), 0), g.nx - 1);
        const int iy = min(max(cell_coord(p.y, g.oy, g.inv_cell_yz), 0), g.ny - 1);
        const int iz = min(max(cell_coord(p.z, g.oz, g.inv_cell_yz), 0), g.nz - 1);
        cid = ((unsigned)iz * g.ny + iy) * g.nx + ix;
        k1 = lvl_index(g, 1, ix, iy, iz);
        k2 = lvl_index(g, 2, ix, iy, iz);
        k3 = lvl_index(g, 3, ix, iy, iz);
    }
    run_add(cursor, cid, valid, lane);
    run_add(lvl, k1, valid, lane);
    run_add(lvl, k2, valid, lane);
    run_add(lvl, k3, valid, lane);
    if (i < n) cell_of[i] = cid;
}

// exclusive scan of cursor[0..ncells) -> cell_start[0..ncells], three kernels
__global__ void __launch_bounds__(SCAN_THREADS)
scan_reduce_kernel(const GridParams* __restrict__ gp, const unsigned* __restrict__ cnt, unsigned* __restrict__ block_sums) {
    const unsigned n = gp->ncells;
    const unsigned base = blockIdx.x * SCAN_TILE;
    if (base >= n) return;
    unsigned s = 0;
    const unsigned i0 = base + threadIdx.x * SCAN_ITEMS;
    if (i0 + SCAN_ITEMS <= n) {  // 8 consecutive cells = two 16-byte loads (the table is 16-byte aligned)
        const uint4 a = reinterpret_cast<const uint4*>(cnt + i0)[0], b = reinterpret_cast<const uint4*>(cnt + i0)[1];
        s = a.x + a.y + a.z + a.w + b.x + b.y + b.z + b.w;
    } else {
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; ++k)
            if (i0 + k < n) s += cnt[i0 + k];
    }
    s = (unsigned)warp_sum((int)s);
    __shared__ unsigned ws[32];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned v = ws[threadIdx.x];
        v = (unsigned)warp_sum((int)v);
        if (threadIdx.x == 0) block_sums[blockIdx.x] = v;
    }
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_final_kernel(const GridParams* __restrict__ gp, unsigned* __restrict__ cursor, const unsigned* __restrict__ block_sums,
                  unsigned* __restrict__ cell_start) {
    const unsigned n = gp->ncells;
    const unsigned base = blockIdx.x * SCAN_TILE;
    if (base >= n) return;
    unsigned v[SCAN_ITEMS];
    unsigned s = 0;
    const unsigned i0 = base + threadIdx.x * SCAN_ITEMS;
    const bool full = i0 + SCAN_ITEMS <= n;
    if (full) {
        const uint4 a = reinterpret_cast<const uint4*>(cursor + i0)[0], b = reinterpret_cast<const uint4*>(cursor + i0)[1];
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; ++k) v[k] = (i0 + k < n) ? cursor[i0 + k] : 0u;
    }
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) s += v[k];
    // block-exclusive prefix of the per-thread sums
    const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += up;
    }
    __shared__ unsigned ws[32];
    if (lane == 31) ws[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        unsigned w = ws[lane];
        unsigned winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned up = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= (unsigned)o) winc += up;
        }
        ws[lane] = winc - w;
    }
    __syncthreads();
    // exclusive prefix of this tile = sum of the sums of the tiles before it (at most 1024 values: one pass of the CTA)
    __shared__ unsigned tile_base;
    {
        unsigned part = 0;
        for (unsigned t = threadIdx.x; t < blockIdx.x; t += SCAN_THREADS) part += block_sums[t];
        part = (unsigned)warp_sum((int)part);
        __shared__ unsigned wb[32];
        if (lane == 0) wb[wid] = part;
        __syncthreads();
        if (wid == 0) {
            unsigned v2 = wb[lane];
            v2 = (unsigned)warp_sum((int)v2);
            if (lane == 0) tile_base = v2;
        }
        __syncthreads();
    }
    if (threadIdx.x == SCAN_THREADS - 1 && base + SCAN_TILE >= n) cell_start[n] = tile_base + ws[wid] + inc;  // grand total (last tile)
    unsigned run = tile_base + ws[wid] + (inc - s);
    unsigned o[SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) { o[k] = run; run += v[k]; }
    if (full) {  // scatter cursor starts at the cell's first slot
        const uint4 a = make_uint4(o[0], o[1], o[2], o[3]), b = make_uint4(o[4], o[5], o[6], o[7]);
        reinterpret_cast<uint4*>(cell_start + i0)[0] = a; reinterpret_cast<uint4*>(cell_start + i0)[1] = b;
        reinterpret_cast<uint4*>(cursor + i0)[0] = a; reinterpret_cast<uint4*>(cursor + i0)[1] = b;
    } else {
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; ++k)
            if (i0 + k < n) { cell_start[i0 + k] = o[k]; cursor[i0 + k] = o[k]; }
    }
}

// Scatter into cell order + block emission.  Leaf level of a point = coarsest cube (8^3, 4^3, 2^3 cells, 1 cell) around
// it with at most TL_QCAP points; all points of a cube take the same decision, one of them (claim bit 31 of the
// cube's counter; the first point of a single cell) emits the block(s).  blk_area = surface area per point (mm^2) seen
// one level up, from which the kernels predict the radius that holds max_nn neighbours.
__global__ void __launch_bounds__(GB_THREADS)
scatter_kernel(const float4* __restrict__ pts, unsigned n, const unsigned* __restrict__ cell_of, const GridParams* __restrict__ gp,
               const unsigned* __restrict__ cell_start, unsigned* __restrict__ cursor, float4* __restrict__ sorted,
               unsigned* __restrict__ sorted_pos, unsigned* __restrict__ lvl, uint4* __restrict__ blocks,
               float* __restrict__ blk_area, unsigned* __restrict__ nblocks, unsigned block_cap) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned cid = cell_of[i];
    if (cid == 0xFFFFFFFFu) { sorted_pos[i] = 0xFFFFFFFFu; return; }
    const unsigned pos = atomicAdd(&cursor[cid], 1u);
    float4 p = pts[i];
    p.w = __uint_as_float(i);
    sorted[pos] = p;
    sorted_pos[i] = pos;
    const GridParams g = *gp;
    const int ix = (int)(cid % (unsigned)g.nx), iy = (int)((cid / (unsigned)g.nx) % (unsigned)g.ny), iz = (int)(cid / ((unsigned)g.nx * (unsigned)g.ny));
    const unsigned c0 = __ldg(cell_start + cid + 1) - __ldg(cell_start + cid);
    unsigned cnt[4];
    cnt[0] = c0;
#pragma unroll
    for (int l = 1; l <= 3; ++l) cnt[l] = lvl[lvl_index(g, l, ix, iy, iz)] & 0x7FFFFFFFu;
    int leaf = 0;
#pragma unroll
    for (int l = 1; l <= 3; ++l)
        if (cnt[l] <= (unsigned)TL_QCAP) leaf = l;
    bool emit;
    if (leaf == 0) emit = (pos == __ldg(cell_start + cid));
    else emit = ((atomicOr(&lvl[lvl_index(g, leaf, ix, iy, iz)], 0x80000000u) >> 31) == 0u);
    if (!emit) return;
    const float side = fmaxf(g.cell, g.cell_yz);
    float area;
    if (leaf == 3) area = (8.0f * side) * (8.0f * side) / (float)max(cnt[3], 1u);
    else if (leaf == 0 && c0 > (unsigned)TL_QCAP) area = side * side / (float)c0;
    else { const float s2 = side * (float)(2 << leaf); area = s2 * s2 / (float)cnt[leaf + 1]; }
    const unsigned nb = (leaf == 0) ? (c0 + TL_QCAP - 1) / TL_QCAP : 1u;
    const int L = 1 << leaf;
    // blocks are listed by weight class (class 0: the most queries); the kernels walk class after class, so the expensive
    // blocks start first and the launch ends on blocks of a few queries (longest-processing-time-first: a 64-query block takes
    // a third of the whole launch, with two classes the last block pulled could still hold 31 queries)
    for (unsigned sidx = 0; sidx < nb; ++sidx) {
        const unsigned weight = (leaf == 0) ? min(c0 - sidx * TL_QCAP, (unsigned)TL_QCAP) : cnt[leaf];
        const unsigned cls = ((unsigned)TL_QCAP - min(max(weight, 1u), (unsigned)TL_QCAP)) * (unsigned)kBlockClasses / (unsigned)TL_QCAP;
        const unsigned slot = cls * block_cap + atomicAdd(nblocks + 16 + cls, 1u);
        blocks[slot] = make_uint4((unsigned)(ix & ~(L - 1)), (unsigned)(iy & ~(L - 1)), (unsigned)(iz & ~(L - 1)), (unsigned)L | (sidx << 4));
        blk_area[slot] = area;
    }
}

int grid_build(Ctx* c, const float* d_raw, size_t n, int stride_floats) {
    const unsigned nn = (unsigned)n;
    const unsigned pb = (nn + GB_THREADS - 1) / GB_THREADS;
    const unsigned scan_blocks = (c->max_cells + SCAN_TILE - 1) / SCAN_TILE;
    if (pb) convert_bbox_kernel<<<pb, GB_THREADS, 0, c->stream>>>(d_raw, nn, stride_floats, c->d_pts, c->d_bbox, kDefaultCell, c->yz_mul, c->max_cells, c->d_grid);
    else grid_params_empty_kernel<<<1, 32, 0, c->stream>>>(c->d_bbox, kDefaultCell, c->yz_mul, c->max_cells, c->d_grid);
    zero_cells_kernel<<<c->sm_count * 4, 1024, 0, c->stream>>>(c->d_grid, c->d_cell_cursor, c->d_lvl, c->d_nblocks);
    if (pb) count_kernel<<<pb, GB_THREADS, 0, c->stream>>>(c->d_pts, nn, c->d_grid, c->d_cell_of, c->d_cell_cursor, c->d_lvl);
    scan_reduce_kernel<<<scan_blocks, SCAN_THREADS, 0, c->stream>>>(c->d_grid, c->d_cell_cursor, c->d_block_sums);
    scan_final_kernel<<<scan_blocks, SCAN_THREADS, 0, c->stream>>>(c->d_grid, c->d_cell_cursor, c->d_block_sums, c->d_cell_start);
    if (pb) scatter_kernel<<<pb, GB_THREADS, 0, c->stream>>>(c->d_pts, nn, c->d_cell_of, c->d_grid, c->d_cell_start, c->d_cell_cursor, c->d_sorted,
                                                             c->d_sorted_pos, c->d_lvl, c->d_blocks, c->d_blk_area, c->d_nblocks, (unsigned)c->max_points);
    count_launch(c, pb ? 6 : 4);
    BSHOT_TRY(check_launch("grid_build"));
    // vector::resize semantics of cloud1_normals (include/bshot_bits.h:59): entries beyond the new
    // size are dropped, so stale keypoint normals above n must not survive a smaller cloud
    if (c->normals_valid > n) {
        BSHOT_CUDA_TRY(cudaMemsetAsync(c->d_normals + n, 0, sizeof(float4) * (c->normals_valid - n), c->stream));
        c->normals_valid = n;
    }
    c->n_points = n;
    c->have_cloud = true;
    c->have_kp = false;
    c->kp_from_detector = false;
    c->sel_valid = false;
    c->fused_sums = false;
    c->have_normals = c->normals_valid > 0;
    return BSHOT_OK;
}

}  // namespace bshot
