// common.cuh -- context, error plumbing and small device helpers shared by all kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "../../include/bshot_b200.h"

namespace bshot {

void set_error(const char* fmt, ...);

#define BSHOT_CUDA_TRY(expr)                                                                   \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            ::bshot::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                               __LINE__);                                                      \
            return BSHOT_E_CUDA;                                                               \
        }                                                                                      \
    } while (0)

#define BSHOT_TRY(expr)          \
    do {                         \
        int _r = (expr);         \
        if (_r != BSHOT_OK) return _r; \
    } while (0)

// voxel grid parameters, computed on the device (no host round trip)
struct GridParams {
    float ox, oy, oz;   // origin = bbox min
    float cell;         // cell edge along x (mm)
    float inv_cell;
    float cell_yz;      // cell edge along y and z: rows (runs of x cells) are the unit of every gather, so they
    float inv_cell_yz;  // are made thicker than a cell is long -- fewer, longer row segments per query sphere
    int nx, ny, nz;
    unsigned int ncells;
    unsigned int npoints;  // finite points that were binned
};

constexpr unsigned int kMaxCells = 1u << 23;       // cell_start capacity (32 MB of u32)

// point counts of the 2^l-cell cubes (l = 1, 2, 3), three dense tables back to back (grid.cu, tile.cuh)
__host__ __device__ __forceinline__ unsigned lvl_dim(int n, int l) { return (unsigned)((n + (1 << l) - 1) >> l); }
__host__ __device__ __forceinline__ unsigned lvl_size(const GridParams& g, int l) { return lvl_dim(g.nx, l) * lvl_dim(g.ny, l) * lvl_dim(g.nz, l); }
__host__ __device__ __forceinline__ unsigned lvl_total(const GridParams& g) { return lvl_size(g, 1) + lvl_size(g, 2) + lvl_size(g, 3); }
__host__ __device__ __forceinline__ unsigned lvl_index(const GridParams& g, int l, int ix, int iy, int iz) {
    unsigned off = 0;
    for (int k = 1; k < l; ++k) off += lvl_size(g, k);
    return off + ((unsigned)(iz >> l) * lvl_dim(g.ny, l) + (unsigned)(iy >> l)) * lvl_dim(g.nx, l) + (unsigned)(ix >> l);
}
constexpr int kDescWords = 12;                      // 48-byte record as u32 words (11 used)
constexpr float kDefaultCell = 375.0f;              // R/8 for the reference radius 3000 mm

// peer-memory exchange of the sharded map match (hamming.cu, capi.cu): one region per rank, mapped on every rank
struct Comm {
    int rank = -1, nranks = 0;
    size_t max_q = 0;
    unsigned char* d_region = nullptr;        // own region: [gather nranks x max_q records][rq max_q u32][flags 64 u32]
    void* opened[32] = {nullptr};             // regions of the other ranks opened through CUDA IPC (closed on destroy)
    bshot_cand** d_peer_gather = nullptr;     // device arrays of nranks pointers into every rank's region
    unsigned** d_peer_rq = nullptr;
    unsigned** d_peer_flags = nullptr;
    unsigned* d_ticket = nullptr;             // 2 "last CTA" tickets
    unsigned epoch = 0;                       // calls issued so far (the flags carry it)
    bool connected = false;
};

// which points get their covariance sums stored by the detector (deferred keypoint normals): the ones whose score reaches
// the K-th score of the previous frame less a margin.  top_k == 0: every point.  A keypoint that was not predicted simply
// has no sums and is searched on its own (exactness never depends on the prediction).
struct SumGate {
    const float* kth_ratio;  // d_kp_ratio: keypoints in ascending score order, [0] = the K-th best of the previous frame
    const int* kth_count;    // d_kp_count
    int top_k;
};

struct IcpState;   // icp.cu / stages.h

// GPU-resident global keypoint map (gmap.cu)
struct Gmap {
    void* d_tab = nullptr;              // block hash table (GmapBlock[tab_cap])
    float4* d_epos = nullptr;           // entries: snapped position + seg-ratio
    uint64_t* d_edesc = nullptr;        // entries: 48-byte descriptors
    unsigned* d_chunks = nullptr;       // 33-word chunks: 32 entry indices + next chunk
    float4* d_world = nullptr;          // per update: snapped world positions of the frame's keypoints
    unsigned* d_blk_of = nullptr;       // per update: block slot of every keypoint
    unsigned* d_touched = nullptr;      // per update: distinct blocks
    unsigned* d_probe_slot = nullptr;   // per gather: slot / offset of every probed block
    unsigned* d_probe_off = nullptr;
    unsigned* d_ctl = nullptr;          // [0] entries [1] touched [2] chunks [3] dropped [4] gathered [5] probes [6] total targets
    float* d_pose = nullptr;            // 2 x 12 floats
    float4* d_tpos = nullptr;           // positions of the assembled target set (max_targets)
    unsigned tab_cap = 0, max_entries = 0, max_chunks = 0, max_probe = 0, epoch = 0;
    size_t n_gathered = 0;
    size_t entries_upper = 0;           // host-side upper bound of the number of entries (sizes the match grid without a sync);
                                        // it and n_updates are written only by gmap_reset and gmap_record_update
    // the whole map in map order (gmap_gather_all, export, relocalisation) and the import's rebuild: allocated by the first
    // call that needs them
    float4* d_apos = nullptr;           // max_entries: positions + seg-ratio in map order
    uint64_t* d_adesc = nullptr;        // max_entries: descriptors in map order
    unsigned long long* d_skeys[2] = {nullptr, nullptr};  // max(tab_cap, max_entries): radix ping-pong (block order keys / slots)
    unsigned* d_svals[2] = {nullptr, nullptr};            // max(tab_cap, max_entries): slots / entry indices
    unsigned* d_shist = nullptr;        // radix histograms
    unsigned* d_boff = nullptr;         // tab_cap: entry offset of each listed block / first sorted entry of each slot (import)
    unsigned* d_actl = nullptr;         // [0] listed blocks [1] entries gathered [2] import error bits [3] import entries
    unsigned* d_atag = nullptr;         // max_entries: tags in map order (gmap_gather_all with tags)
    // loop closure (gmap_scans, bshot_detect_loop).  Updates are numbered 0, 1, ... since create / reset / import (update
    // 0) / odometry reset; gmap_record_update advances n_updates with entries_upper, once the update has succeeded
    unsigned* d_etag = nullptr;         // max_entries: index of the update that wrote each entry
    float* d_traj = nullptr;            // traj_cap x 12: row-major [R|T] each update used (identity without a pose)
    size_t traj_cap = 0;
    unsigned n_updates = 0;
    bool last_by_scan = false;          // the last update was a step or an accepted relocalisation, and its scan is still the reference frame
    // loop-closure selections, allocated by the first detection: candidates in map order, tile counts / offsets, counts
    float4* d_lpos = nullptr;           // max_entries
    uint64_t* d_ldesc = nullptr;        // max_entries x 6
    unsigned* d_ltag = nullptr;         // max_entries
    unsigned* d_ltile = nullptr;        // 2 x ltile_cap
    size_t ltile_cap = 0;
    unsigned* d_lctl = nullptr;         // [0] candidates [1] candidates (uncapped) [2] ICP targets (<= max_targets) [3] ICP targets (uncapped)
    // re-anchoring (bshot_gmap_reanchor), allocated by the first call
    float* d_rtraj = nullptr;           // rcap x 12: the new trajectory
    float* d_rcorr = nullptr;           // rcap x 12 corrections C_u, then the odometry's new pose (16)
    unsigned* d_rchg = nullptr;         // rcap flags: update u changed; then the count of entries to rebuild
    size_t rcap = 0;
};

// ISS keypoints (iss.cu): max_points-sized buffers, allocated by the first bshot_detect_iss of the context
struct Iss {
    double* d_l3 = nullptr;             // per cell-sorted position: third_eigen_value (0 = not salient)
    double* d_eig = nullptr;            // per original index: lambda1..3
    unsigned char* d_flag = nullptr;    // per original index: keypoint
    unsigned* d_tile_sums = nullptr;    // keypoints per compaction tile
    int4* d_rec = nullptr;              // [0].x = count, then {index, x, y, z} records in ascending index
    int4* h_rec = nullptr;              // pinned staging of d_rec
};

// voxel-grid downsampling (voxel_grid.cu): max_points-sized buffers, allocated by the first bshot_voxel_grid of the context
struct Vg {
    float* d_in = nullptr;              // staging of the caller's cloud (stride 12 or 16)
    unsigned* d_ctl = nullptr;          // VgParams + bbox + ticket (voxel_grid.cu)
    unsigned* d_tile = nullptr;         // per compaction tile: finite points, then voxel heads
    unsigned* d_keys[2] = {nullptr, nullptr};  // voxel index per finite point, radix ping-pong
    unsigned* d_vals[2] = {nullptr, nullptr};  // point index per finite point, radix ping-pong
    unsigned* d_hist = nullptr;         // per radix tile: 256 digit counts
    unsigned* d_seg = nullptr;          // first sorted position of every voxel, then the finite count
    float* d_out = nullptr;             // [0] = count (as unsigned), [1..3] unused, then {x, y, z} records
    float* h_out = nullptr;             // pinned staging of d_out
};

// per-scan odometry step (odometry.cu): allocated by the first bshot_odometry_step / bshot_ransac_dev of the context
struct OdomDev;
struct Odom {
    OdomDev* d = nullptr;               // report, error flag, pose, gate matrices, RANSAC outputs (odometry.cu)
    int* d_inlier_pairs = nullptr;      // max_kp x 2: the pairs RANSAC keeps
    float4* d_icp_cur = nullptr;        // max_kp: ICP sources (moved)
    unsigned long long* d_icp_keys = nullptr;  // max_kp
    float4* d_icp_tgt = nullptr;        // max_targets: ICP targets, NaN past the true count
    IcpState* d_icp_state = nullptr;
    void* h_out = nullptr;              // pinned staging of the report
    void* d_loop = nullptr;             // loop detection's report, error flag and RANSAC outputs (LoopDev, odometry.cu)
    void* h_loop = nullptr;             // pinned staging of its report
    bool run = false;                   // RUN status: a step has succeeded since creation / bshot_odometry_reset
};

// query blocks are listed by weight class (class c: kBlockClasses regions of max_points entries in d_blocks / d_blk_area)
constexpr int kBlockClasses = 8;

struct Ctx {
    int device = 0;
    int sm_count = 148;
    int match_tc = -1;                 // bshot_set_matcher / BSHOT_MATCH_TC: -1 by problem size, 0 XOR + POPC (hamming.cu), 1 tensor cores (hamming_tc.cu), 2 / 3 pipelined tensor-core kernel (hamming_tc2.cu)
    bool no_deferred_normals = false;  // BSHOT_DEFERRED_NORMALS=0: keypoint normals by a second search (tile_keypoint_normals) instead of the detector's sums (tests)
    bool force_warp_path = false;  // BSHOT_WARP_PATH=1: skip the block-tiled kernels (tile.cuh), warp-per-query kernels everywhere (tests)
    unsigned max_cells = 1u << 22;  // voxel table size actually used (<= kMaxCells; BSHOT_MAX_CELLS_LOG2): zeroed and scanned every frame
    float yz_mul = 1.0f;  // cell_yz / cell (tuning knob BSHOT_YZ_MUL; 2 helps SHOT by ~3 %, costs the detector ~6 %)
    cudaStream_t stream = nullptr;
    unsigned long long launches = 0;
    size_t max_points = 0, max_kp = 0, max_targets = 0;

    // cloud + voxel grid
    size_t n_points = 0;
    bool have_cloud = false;
    float* d_raw = nullptr;            // staging of caller layout (stride 12 or 16)
    float4* d_pts = nullptr;           // original order, w = 1
    float4* d_sorted = nullptr;        // cell order, w = bit pattern of the original index
    unsigned int* d_cell_of = nullptr; // cell id per point (0xFFFFFFFF = not binned)
    unsigned int* d_cell_start = nullptr;  // kMaxCells + 1
    unsigned int* d_cell_cursor = nullptr; // kMaxCells
    unsigned int* d_block_sums = nullptr;
    GridParams* d_grid = nullptr;
    float* d_bbox = nullptr;           // 6 floats as ordered ints
    unsigned* d_lvl = nullptr;         // kMaxCells + 16: point counts of the 2^3 / 4^3 / 8^3-cell cubes (bit 31 = block emitted)
    unsigned* d_sorted_pos = nullptr;  // N: original index -> position in d_sorted (0xFFFFFFFF = not binned)
    int* d_kp_flag = nullptr;          // N: per sorted position, keypoint ordinal or -1 (reset by the grid build)
    uint4* d_blocks = nullptr;         // N: query blocks {ix0, iy0, iz0, cells per edge | slice << 4} (tile.cuh)
    float* d_blk_area = nullptr;       // N: surface area per point around the block (radius prediction)
    unsigned* d_nblocks = nullptr;     // [1] fallback-list length, [2],[3] work counters, [4] overflow queries, [6] wide overflow queries, [16 + c] blocks of weight class c
    float* d_qsums = nullptr;          // N x 10: covariance sums + count of the detector's neighbourhood of every point (deferred normals)
    float* d_rho_hint = nullptr;       // N: radius of the detector's neighbourhood of every point (distance of its last member)
    unsigned* d_shot_order = nullptr;  // K: order in which shot_kernel takes the keypoints (densest neighbourhoods first)
    uint2* d_ovf = nullptr;            // N: queries whose block tile overflowed {position in d_sorted, radius bits} (tilek.cu)
    unsigned* d_fb_list = nullptr;     // N: sorted positions of the queries the tiled kernels hand to the fallback

    // detector
    float* d_ratio = nullptr;                // N
    unsigned long long* d_keys = nullptr;    // N sortable keys
    int* d_kp_idx = nullptr;                 // K surface indices (-1 = not a surface point)
    float* d_kp_ratio = nullptr;             // K
    float4* d_kp = nullptr;                  // K keypoint positions (w = index bits)
    int* d_kp_count = nullptr;               // device-side keypoint count
    bool sel_valid = false;                  // the detector ran on the current cloud with (sel_radius, sel_max_nn)
    float sel_radius = 0.0f;
    int sel_max_nn = 0;
    int gate_top_k = 0;                      // the previous frame_extract ran with these detector parameters and left its K-th ratio in d_kp_ratio[0]
    int gate_sr = -1;
    float gate_radius = 0.0f;
    int gate_max_nn = 0;
    bool fused_sums = false;                 // d_qsums is valid for (fused_radius, fused_max_nn)
    bool fused_normals = false;              // d_normals already holds the FULL-mode normals for (fused_radius, fused_max_nn)
    float fused_radius = 0.0f;
    int fused_max_nn = 0;
    bool kp_from_detector = false;           // d_kp[i].w is the surface index of keypoint i
    unsigned* d_tk_hist = nullptr;           // top-K: 4096-bin ratio histogram (kept zeroed between frames)
    unsigned* d_tk_state = nullptr;          // top-K: 16 words of device-side state
    unsigned long long* d_tk_sure = nullptr; // top-K: keys above the threshold bin (< K)
    unsigned long long* d_tk_tie = nullptr;  // top-K: keys inside the threshold bin (<= N)
    size_t n_kp = 0;                         // host-side count (upper bound when detector ran async)
    bool have_kp = false;

    // normals
    float4* d_normals = nullptr;   // N, persistent across frames (reference quirk)
    float4* d_qnormals = nullptr;  // max(N) query normals scratch
    size_t normals_valid = 0;      // entries of d_normals that have ever been written
    bool have_normals = false;

    // SHOT / B-SHOT
    float* d_shot = nullptr;            // K x 352
    float* d_rf = nullptr;              // K x 9
    int* d_nn = nullptr;                // K
    unsigned long long* d_sum_nn = nullptr;
    uint64_t* d_bits = nullptr;         // K x 6
    uint64_t* d_prev_bits = nullptr;    // K x 6 (previous frame)
    size_t n_prev = 0;                  // host-side upper bound (top_k of the previous frame); d_prev_count is the real count
    int* d_prev_count = nullptr;
    size_t last_top_k = 0;              // top_k of the last frame_run (what bshot_fetch_frame may copy out)

    // matching
    uint64_t* d_q = nullptr;            // max_kp x 6
    uint64_t* d_t = nullptr;            // max_targets x 6 (host-API staging)
    uint64_t* d_map = nullptr;          // max_targets x 6 resident shard
    size_t n_map = 0;
    unsigned long long* d_partial = nullptr;  // [nsplit][nq][2]
    size_t partial_cap = 0;                   // in u64
    bshot_cand* d_cand = nullptr;       // max(max_kp, ...) records
    bshot_cand* d_cand2 = nullptr;
    uint64_t* d_gather = nullptr;       // max_kp x 6 gathered targets for the reverse pass
    int* d_left = nullptr;              // 4 x max_kp ints (idx, dist, idx2, dist2)
    int* d_right = nullptr;             // max_targets ints
    int* d_pairs = nullptr;             // 3 x max_kp (q, m, dist)
    int* d_pair_count = nullptr;        // [0] mutual pairs, [1] owned winners, [3] peer-barrier timeout flag
    unsigned peer_epoch = 0;            // barriers issued on the symmetric flag array so far

    Comm comm;
    Gmap gmap;
    Iss iss;
    Vg vg;
    Odom odom;
    float4* d_prev_kp = nullptr;        // K: keypoint positions of the previous frame (reference frame of the map match)
    void* d_pre[3] = {nullptr, nullptr, nullptr};  // scratch grown on demand: preprocessor per-return / per-column, ICP
    size_t pre_bytes[3] = {0, 0, 0};

    // pinned host scratch
    int* h_scratch = nullptr;           // 64 ints
    int* h_pairs = nullptr;             // 3 x max_kp ints: (query, match, distance) staging for the D2H copy

    // instrumentation
    unsigned long long* d_counters = nullptr;  // 8 work counters (see bshot_frame_counters)
    bool timing = false;
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;   // bshot_process_frame: keypoints + descriptors travel to the host while the frame is still being matched
    cudaEvent_t ev_desc = nullptr;        // recorded when the descriptors of the frame are complete
    bool ev_valid = false;
};

inline void count_launch(Ctx* c, unsigned n = 1) { c->launches += n; }

int check_launch(const char* what);

}  // namespace bshot

struct bshot_ctx : public bshot::Ctx {};

// ---- device helpers --------------------------------------------------------------------------
// -DBSHOT_DEBUG_BOUNDS: device-side asserts on every shared-memory / list index the kernels compute (the pool has no
// compute-sanitizer); a violated bound traps the kernel and the next API call reports the CUDA error.
#ifdef BSHOT_DEBUG_BOUNDS
#include <assert.h>
#define BSHOT_ASSERT(cond) assert(cond)
#else
#define BSHOT_ASSERT(cond) ((void)0)
#endif

namespace bshot {

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// float min / max through the integer atomics, for non-NaN values.  v >= 0 takes the signed path, where the order of the
// bit patterns is the order of the floats; v < 0 takes the unsigned path, where it is the reverse.  -0.0 compares
// >= 0 but its bit pattern is INT_MIN, so it is first turned into +0.0 (-0 + +0 = +0; every other v is unchanged); the
// stored extreme is then +0.0 where the floats' extreme is a zero of either sign.
__device__ __forceinline__ void atomic_min_float(float* a, float v) {
    v = __fadd_rn(v, 0.0f);
    if (v >= 0.0f) atomicMin(reinterpret_cast<int*>(a), __float_as_int(v));
    else atomicMax(reinterpret_cast<unsigned*>(a), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_float(float* a, float v) {
    v = __fadd_rn(v, 0.0f);
    if (v >= 0.0f) atomicMax(reinterpret_cast<int*>(a), __float_as_int(v));
    else atomicMin(reinterpret_cast<unsigned*>(a), __float_as_uint(v));
}

// FLANN L2_Simple in fp32 without FMA contraction (SURVEY Appendix A.1)
__device__ __forceinline__ float sqdist_rn(float ax, float ay, float az, float bx, float by, float bz) {
    float d = __fsub_rn(ax, bx);
    float r = __fmul_rn(d, d);
    d = __fsub_rn(ay, by);
    r = __fadd_rn(r, __fmul_rn(d, d));
    d = __fsub_rn(az, bz);
    r = __fadd_rn(r, __fmul_rn(d, d));
    return r;
}

// (a0*b0 + a1*b1) + a2*b2 in fp32 without contraction
__device__ __forceinline__ float dot3_rn(float ax, float ay, float az, float bx, float by, float bz) {
    return __fadd_rn(__fadd_rn(__fmul_rn(ax, bx), __fmul_rn(ay, by)), __fmul_rn(az, bz));
}

// R * p + T on a row-major 3x4 [R|T] in fp32 without contraction: the products summed left to right, then the translation
// (updateMap's kp_pos = R * kp_pos + T, src/lidar_odometry.cpp:351).  The map and the keypoint repeatability move points
// with it, so the same pose puts a point at the same bits in both
__device__ __forceinline__ float3 pose_apply_rn(const float* m, float x, float y, float z) {
    return make_float3(__fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], x), __fmul_rn(m[1], y)), __fmul_rn(m[2], z)), m[3]),
                       __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[4], x), __fmul_rn(m[5], y)), __fmul_rn(m[6], z)), m[7]),
                       __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[8], x), __fmul_rn(m[9], y)), __fmul_rn(m[10], z)), m[11]));
}

}  // namespace bshot
