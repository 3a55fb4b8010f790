// capi.cu -- the extern "C" boundary declared in include/bshot_b200.h.
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <new>
#include <vector>

#include "common.cuh"
#include <stdlib.h>

#include "odom_math.cuh"
#include "stages.h"

namespace bshot {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
        return BSHOT_E_CUDA;
    }
    return BSHOT_OK;
}

template <typename T>
static int dmalloc(T** p, size_t count) {
    BSHOT_CUDA_TRY(cudaMalloc((void**)p, sizeof(T) * (count ? count : 1)));
    return BSHOT_OK;
}

static int sync(Ctx* c) {
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return BSHOT_OK;
}

static int h2d(Ctx* c, void* dst, const void* src, size_t bytes) {
    if (bytes == 0) return BSHOT_OK;
    BSHOT_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return BSHOT_OK;
}
static int d2h(Ctx* c, void* dst, const void* src, size_t bytes) {
    if (bytes == 0 || dst == nullptr) return BSHOT_OK;
    BSHOT_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    return BSHOT_OK;
}

}  // namespace bshot

using namespace bshot;

#define CHECK_CTX(ctx)                          \
    do {                                        \
        if ((ctx) == nullptr) {                 \
            set_error("null context");          \
            return BSHOT_E_INVALID;             \
        }                                       \
        cudaError_t _e = cudaSetDevice((ctx)->device); \
        if (_e != cudaSuccess) {                \
            set_error("cudaSetDevice failed: %s", cudaGetErrorString(_e)); \
            return BSHOT_E_CUDA;                \
        }                                       \
    } while (0)

extern "C" {

void bshot_params_default(bshot_params* p) {
    if (!p) return;
    p->kp_radius = 3000.0f;
    p->kp_max_nn = 300;
    p->sr_type = BSHOT_SR_CV;
    p->top_k = 600;
    p->normal_radius = 3000.0f;
    p->normal_max_nn = 300;
    p->normals_mode = BSHOT_NORMALS_REFERENCE;
    p->shot_radius = 3000.0f;
}

int bshot_version(void) { return BSHOT_B200_VERSION; }
const char* bshot_last_error(void) { return g_err; }

int bshot_ctx_create(bshot_ctx** out, int device, size_t max_points, size_t max_keypoints, size_t max_targets) {
    if (!out || max_points == 0 || max_keypoints == 0) {
        set_error("bshot_ctx_create: bad arguments");
        return BSHOT_E_INVALID;
    }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available: this library has no CPU fallback");
        return BSHOT_E_CUDA;
    }
    if (device < 0 || device >= ndev) {
        set_error("device %d out of range (%d devices)", device, ndev);
        return BSHOT_E_INVALID;
    }
    BSHOT_CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    BSHOT_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major, prop.minor);
        return BSHOT_E_CUDA;
    }
    bshot_ctx* c = new (std::nothrow) bshot_ctx();
    if (!c) {
        set_error("out of host memory");
        return BSHOT_E_INVALID;
    }
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    if (const char* e = getenv("BSHOT_WARP_PATH")) c->force_warp_path = (atoi(e) != 0);
    if (const char* e = getenv("BSHOT_MATCH_TC")) c->match_tc = atoi(e);
    if (const char* e = getenv("BSHOT_DEFERRED_NORMALS")) c->no_deferred_normals = (atoi(e) == 0);
    if (const char* e = getenv("BSHOT_MAX_CELLS_LOG2")) {  // tuning knob: voxel table size (default 2^22 cells)
        const int v = atoi(e);
        if (v >= 10 && v <= 23) c->max_cells = 1u << v;
    }
    if (const char* e = getenv("BSHOT_YZ_MUL")) {  // tuning knob: row thickness relative to the cell length
        const float v = (float)atof(e);
        if (v >= 1.0f && v <= 8.0f) c->yz_mul = v;
    }
    if (max_targets < max_keypoints) max_targets = max_keypoints;
    c->max_points = max_points;
    c->max_kp = max_keypoints;
    c->max_targets = max_targets;
    const size_t N = max_points, K = max_keypoints, T = max_targets;
    const size_t QN = std::max(N, K);
    int r = BSHOT_OK;
    auto A = [&](int rr) { if (r == BSHOT_OK) r = rr; };
    cudaError_t se = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (se != cudaSuccess) { set_error("cudaStreamCreate failed: %s", cudaGetErrorString(se)); delete c; return BSHOT_E_CUDA; }
    A(dmalloc(&c->d_raw, N * 4));
    A(dmalloc(&c->d_pts, N));
    A(dmalloc(&c->d_sorted, N));
    A(dmalloc(&c->d_cell_of, N));
    A(dmalloc(&c->d_cell_start, (size_t)kMaxCells + 1));
    A(dmalloc(&c->d_cell_cursor, (size_t)kMaxCells));
    A(dmalloc(&c->d_block_sums, 4096));
    A(dmalloc(&c->d_grid, 1));
    A(dmalloc(&c->d_bbox, 8));
    A(dmalloc(&c->d_lvl, (size_t)kMaxCells + 16));
    A(dmalloc(&c->d_sorted_pos, N));
    A(dmalloc(&c->d_kp_flag, N));
    A(dmalloc(&c->d_blocks, (size_t)kBlockClasses * N));
    A(dmalloc(&c->d_blk_area, (size_t)kBlockClasses * N));
    A(dmalloc(&c->d_nblocks, 32));
    A(dmalloc(&c->d_ovf, N));
    A(dmalloc(&c->d_rho_hint, N));
    A(dmalloc(&c->d_shot_order, K));
    A(dmalloc(&c->d_qsums, 10 * N));
    A(dmalloc(&c->d_fb_list, N));
    A(dmalloc(&c->d_ratio, N));
    A(dmalloc(&c->d_keys, N));
    A(dmalloc(&c->d_kp_idx, K));
    A(dmalloc(&c->d_kp_ratio, K));
    A(dmalloc(&c->d_kp, K));
    A(dmalloc(&c->d_kp_count, 4));
    A(dmalloc(&c->d_tk_hist, 4096));
    A(dmalloc(&c->d_tk_state, 16));
    A(dmalloc(&c->d_tk_sure, K));
    A(dmalloc(&c->d_tk_tie, N));
    A(dmalloc(&c->d_normals, N));
    A(dmalloc(&c->d_qnormals, QN));
    A(dmalloc(&c->d_shot, K * 352));
    A(dmalloc(&c->d_rf, K * 9));
    A(dmalloc(&c->d_nn, K));
    A(dmalloc(&c->d_sum_nn, 2));
    A(dmalloc(&c->d_bits, K * 6));
    A(dmalloc(&c->d_prev_bits, K * 6));
    A(dmalloc(&c->d_prev_kp, K));
    A(dmalloc(&c->d_prev_count, 4));
    A(dmalloc(&c->d_q, K * 6));
    A(dmalloc(&c->d_t, T * 6));
    A(dmalloc(&c->d_map, T * 6));
    c->partial_cap = std::max(K * 2 * 256, T * 2 + 1024);
    A(dmalloc(&c->d_partial, c->partial_cap));
    A(dmalloc(&c->d_cand, std::max(K, T)));
    A(dmalloc(&c->d_cand2, std::max(K, T)));
    A(dmalloc(&c->d_gather, K * 6));
    A(dmalloc(&c->d_left, K * 4));
    A(dmalloc(&c->d_right, T));
    A(dmalloc(&c->d_pairs, K * 3));
    A(dmalloc(&c->d_pair_count, 4));
    A(dmalloc(&c->d_counters, 8));
    if (r == BSHOT_OK && (cudaMallocHost((void**)&c->h_scratch, 64 * sizeof(int)) != cudaSuccess ||
                          cudaMallocHost((void**)&c->h_pairs, 3 * K * sizeof(int)) != cudaSuccess)) {
        set_error("cudaMallocHost failed");
        r = BSHOT_E_CUDA;
    }
    if (r == BSHOT_OK) {
        // pcl::Normal default-constructs to (0,0,0): the persistent normals array starts zeroed
        cudaError_t e = cudaMemsetAsync(c->d_normals, 0, sizeof(float4) * N, c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_prev_count, 0, 4 * sizeof(int), c->stream);
        if (e == cudaSuccess) {  // bounding box armed (+inf / -inf), ticket zero: the grid build re-arms it after every frame
            const float inf = __builtin_inff();
            const float box[8] = {inf, inf, inf, -inf, -inf, -inf, 0.0f, 0.0f};
            e = cudaMemcpyAsync(c->d_bbox, box, sizeof(box), cudaMemcpyHostToDevice, c->stream);
        }
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_kp_count, 0, 4 * sizeof(int), c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_pair_count, 0, 4 * sizeof(int), c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_tk_hist, 0, 4096 * sizeof(unsigned), c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_tk_state, 0, 16 * sizeof(unsigned), c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_counters, 0, 8 * sizeof(unsigned long long), c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_sum_nn, 0, 2 * sizeof(unsigned long long), c->stream);
        for (int i = 0; i < 8 && e == cudaSuccess; ++i) e = cudaEventCreate(&c->ev[i]);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_desc, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { set_error("context init failed: %s", cudaGetErrorString(e)); r = BSHOT_E_CUDA; }
    }
    if (r != BSHOT_OK) {
        bshot_ctx_destroy(c);
        return r;
    }
    *out = c;
    return BSHOT_OK;
}

static void comm_free(bshot_ctx* c);

void bshot_ctx_destroy(bshot_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    comm_free(c);
    gmap_free(c);
    iss_free(c);
    vg_free(c);
    odom_free(c);
    void* ptrs[] = {c->d_raw, c->d_pts, c->d_sorted, c->d_cell_of, c->d_cell_start, c->d_cell_cursor, c->d_block_sums,
                    c->d_grid, c->d_bbox, c->d_lvl, c->d_sorted_pos, c->d_kp_flag, c->d_blocks, c->d_blk_area, c->d_nblocks, c->d_ovf, c->d_rho_hint, c->d_shot_order, c->d_qsums, c->d_fb_list, c->d_ratio, c->d_keys, c->d_kp_idx, c->d_kp_ratio, c->d_kp, c->d_kp_count,
                    c->d_tk_hist, c->d_tk_state, c->d_tk_sure, c->d_tk_tie, c->d_normals, c->d_qnormals, c->d_shot, c->d_rf, c->d_nn, c->d_sum_nn, c->d_bits, c->d_prev_bits, c->d_prev_kp,
                    c->d_prev_count, c->d_q, c->d_t, c->d_map, c->d_partial, c->d_cand, c->d_cand2, c->d_gather,
                    c->d_left, c->d_right, c->d_pairs, c->d_pair_count, c->d_counters, c->d_pre[0], c->d_pre[1], c->d_pre[2]};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (c->h_scratch) cudaFreeHost(c->h_scratch);
    if (c->h_pairs) cudaFreeHost(c->h_pairs);
    for (int i = 0; i < 8; ++i)
        if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    if (c->ev_desc) cudaEventDestroy(c->ev_desc);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

void* bshot_ctx_stream(bshot_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int bshot_ctx_sync(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    return sync(ctx);
}

int bshot_ctx_reset(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    BSHOT_CUDA_TRY(cudaMemsetAsync(ctx->d_normals, 0, sizeof(float4) * ctx->max_points, ctx->stream));
    BSHOT_CUDA_TRY(cudaMemsetAsync(ctx->d_prev_count, 0, sizeof(int), ctx->stream));
    ctx->normals_valid = 0;
    ctx->have_normals = false;
    ctx->n_prev = 0;
    ctx->gmap.last_by_scan = false;   // no reference frame: nothing for bshot_detect_loop to query
    ctx->n_map = 0;
    ctx->gate_top_k = 0;
    return sync(ctx);
}

unsigned long long bshot_launch_count(bshot_ctx* ctx) { return ctx ? ctx->launches : 0ull; }

int bshot_set_matcher(bshot_ctx* ctx, int kind) {
    CHECK_CTX(ctx);
    if (kind < -1 || kind > 3) { set_error("bshot_set_matcher: kind %d (expected -1 .. 3)", kind); return BSHOT_E_INVALID; }
    ctx->match_tc = kind;
    return BSHOT_OK;
}

int bshot_popc_peak(bshot_ctx* ctx, double* out) {
    CHECK_CTX(ctx);
    if (!out) { set_error("null output"); return BSHOT_E_INVALID; }
    return popc_peak(ctx, out);
}

// ---- a1 ---------------------------------------------------------------------------------------
int bshot_set_cloud(bshot_ctx* ctx, const float* xyz, size_t n, size_t stride_bytes) {
    CHECK_CTX(ctx);
    if (!xyz && n) { set_error("bshot_set_cloud: null cloud"); return BSHOT_E_INVALID; }
    if (stride_bytes != 12 && stride_bytes != 16) { set_error("bshot_set_cloud: stride must be 12 or 16 bytes"); return BSHOT_E_INVALID; }
    if (n > ctx->max_points) { set_error("bshot_set_cloud: %zu points > capacity %zu", n, ctx->max_points); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(h2d(ctx, ctx->d_raw, xyz, n * stride_bytes));
    BSHOT_TRY(grid_build(ctx, ctx->d_raw, n, (int)(stride_bytes / 4)));
    return sync(ctx);
}

// ---- a2 + a3 ----------------------------------------------------------------------------------
int bshot_seg_ratio(bshot_ctx* ctx, float radius, int max_nn, int sr_type, float* ratio_out) {
    CHECK_CTX(ctx);
    if (!ctx->have_cloud) { set_error("bshot_seg_ratio: no cloud"); return BSHOT_E_STATE; }
    BSHOT_TRY(detect_seg_ratio(ctx, radius, max_nn, sr_type));
    BSHOT_TRY(d2h(ctx, ratio_out, ctx->d_ratio, sizeof(float) * ctx->n_points));
    return sync(ctx);
}

int bshot_detect_keypoints(bshot_ctx* ctx, float radius, int max_nn, int sr_type, int top_k, int* idx_out,
                           float* ratio_out, float* kp_xyz_out, int* count_out) {
    CHECK_CTX(ctx);
    if (!ctx->have_cloud) { set_error("bshot_detect_keypoints: no cloud"); return BSHOT_E_STATE; }
    if (top_k <= 0 || (size_t)top_k > ctx->max_kp) { set_error("bshot_detect_keypoints: top_k %d outside (0, %zu]", top_k, ctx->max_kp); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(detect_seg_ratio(ctx, radius, max_nn, sr_type));
    BSHOT_TRY(detect_topk(ctx, top_k));
    BSHOT_TRY(d2h(ctx, ctx->h_scratch, ctx->d_kp_count, sizeof(int)));
    BSHOT_TRY(sync(ctx));
    const int k = ctx->h_scratch[0];
    ctx->n_kp = (size_t)k;
    ctx->have_kp = true;
    if (count_out) *count_out = k;
    BSHOT_TRY(d2h(ctx, idx_out, ctx->d_kp_idx, sizeof(int) * k));
    BSHOT_TRY(d2h(ctx, ratio_out, ctx->d_kp_ratio, sizeof(float) * k));
    if (kp_xyz_out && k) {
        BSHOT_CUDA_TRY(cudaMemcpy2DAsync(kp_xyz_out, 12, ctx->d_kp, 16, 12, k, cudaMemcpyDeviceToHost, ctx->stream));
    }
    return sync(ctx);
}

int bshot_set_keypoints(bshot_ctx* ctx, const float* kp_xyz, size_t k, size_t stride_bytes) {
    CHECK_CTX(ctx);
    if (!kp_xyz && k) { set_error("bshot_set_keypoints: null keypoints"); return BSHOT_E_INVALID; }
    if (stride_bytes != 12 && stride_bytes != 16) { set_error("bshot_set_keypoints: stride must be 12 or 16 bytes"); return BSHOT_E_INVALID; }
    if (k > ctx->max_kp) { set_error("bshot_set_keypoints: %zu keypoints > capacity %zu", k, ctx->max_kp); return BSHOT_E_CAPACITY; }
    if (k) {
        BSHOT_CUDA_TRY(cudaMemsetAsync(ctx->d_kp, 0, sizeof(float4) * k, ctx->stream));
        BSHOT_CUDA_TRY(cudaMemcpy2DAsync(ctx->d_kp, 16, kp_xyz, stride_bytes, 12, k, cudaMemcpyHostToDevice, ctx->stream));
    }
    ctx->h_scratch[8] = (int)k;
    BSHOT_TRY(h2d(ctx, ctx->d_kp_count, &ctx->h_scratch[8], sizeof(int)));
    ctx->n_kp = k;
    ctx->have_kp = true;
    ctx->kp_from_detector = false;
    ctx->gate_top_k = 0;
    return sync(ctx);
}

// ---- a4 ---------------------------------------------------------------------------------------
int bshot_compute_normals(bshot_ctx* ctx, int mode, float radius, int max_nn, float* normals_out) {
    CHECK_CTX(ctx);
    if (!ctx->have_cloud) { set_error("bshot_compute_normals: no cloud"); return BSHOT_E_STATE; }
    if (mode == BSHOT_NORMALS_REFERENCE && !ctx->have_kp) { set_error("bshot_compute_normals: REFERENCE mode needs keypoints"); return BSHOT_E_STATE; }
    if (mode != BSHOT_NORMALS_REFERENCE && mode != BSHOT_NORMALS_FULL) { set_error("bshot_compute_normals: bad mode"); return BSHOT_E_INVALID; }
    BSHOT_TRY(normals_compute(ctx, mode, radius, max_nn));
    BSHOT_TRY(d2h(ctx, normals_out, ctx->d_normals, sizeof(float4) * ctx->n_points));
    return sync(ctx);
}

int bshot_query_normals(bshot_ctx* ctx, const float* q_xyz, size_t nq, float radius, int max_nn, float* normals_out) {
    CHECK_CTX(ctx);
    if (!ctx->have_cloud) { set_error("bshot_query_normals: no cloud"); return BSHOT_E_STATE; }
    if (nq > std::max(ctx->max_points, ctx->max_kp)) { set_error("bshot_query_normals: too many queries"); return BSHOT_E_CAPACITY; }
    if (nq == 0) return BSHOT_OK;
    // stage the queries in d_qnormals (float4) then overwrite in place
    BSHOT_CUDA_TRY(cudaMemsetAsync(ctx->d_qnormals, 0, sizeof(float4) * nq, ctx->stream));
    BSHOT_CUDA_TRY(cudaMemcpy2DAsync(ctx->d_qnormals, 16, q_xyz, 12, 12, nq, cudaMemcpyHostToDevice, ctx->stream));
    BSHOT_TRY(normals_query(ctx, ctx->d_qnormals, nq, radius, max_nn, ctx->d_qnormals));
    BSHOT_TRY(d2h(ctx, normals_out, ctx->d_qnormals, sizeof(float4) * nq));
    return sync(ctx);
}

int bshot_set_normals(bshot_ctx* ctx, const float* normals4, size_t n) {
    CHECK_CTX(ctx);
    if (!ctx->have_cloud || n != ctx->n_points) { set_error("bshot_set_normals: need a cloud with exactly n points"); return BSHOT_E_STATE; }
    BSHOT_TRY(h2d(ctx, ctx->d_normals, normals4, sizeof(float4) * n));
    ctx->have_normals = true;
    ctx->normals_valid = std::max(ctx->normals_valid, n);
    return sync(ctx);
}

// ---- a5 + a6 + a7 -----------------------------------------------------------------------------
int bshot_compute_lrf(bshot_ctx* ctx, float radius, float* rf_out, int* valid_nn_out) {
    CHECK_CTX(ctx);
    if (!ctx->have_cloud || !ctx->have_kp) { set_error("bshot_compute_lrf: need cloud and keypoints"); return BSHOT_E_STATE; }
    BSHOT_TRY(shot_compute(ctx, radius, /*lrf_only=*/true, /*write_shot=*/false));
    BSHOT_TRY(d2h(ctx, rf_out, ctx->d_rf, sizeof(float) * 9 * ctx->n_kp));
    BSHOT_TRY(d2h(ctx, valid_nn_out, ctx->d_nn, sizeof(int) * ctx->n_kp));
    return sync(ctx);
}

int bshot_compute_shot(bshot_ctx* ctx, float radius, uint64_t* bits_out, float* shot_out, float* rf_out, int* nn_out,
                       long long* sum_nn_out) {
    CHECK_CTX(ctx);
    if (!ctx->have_cloud || !ctx->have_kp) { set_error("bshot_compute_shot: need cloud and keypoints"); return BSHOT_E_STATE; }
    if (!ctx->have_normals) { set_error("bshot_compute_shot: no normals (call bshot_compute_normals / bshot_set_normals)"); return BSHOT_E_STATE; }
    BSHOT_TRY(shot_compute(ctx, radius, /*lrf_only=*/false, /*write_shot=*/shot_out != nullptr));
    const size_t k = ctx->n_kp;
    BSHOT_TRY(d2h(ctx, bits_out, ctx->d_bits, sizeof(uint64_t) * 6 * k));
    BSHOT_TRY(d2h(ctx, shot_out, ctx->d_shot, sizeof(float) * 352 * k));
    BSHOT_TRY(d2h(ctx, rf_out, ctx->d_rf, sizeof(float) * 9 * k));
    BSHOT_TRY(d2h(ctx, nn_out, ctx->d_nn, sizeof(int) * k));
    unsigned long long* h_sum = reinterpret_cast<unsigned long long*>(&ctx->h_scratch[16]);
    BSHOT_TRY(d2h(ctx, h_sum, ctx->d_sum_nn, sizeof(unsigned long long)));
    BSHOT_TRY(sync(ctx));
    if (sum_nn_out) *sum_nn_out = (long long)*h_sum;
    return BSHOT_OK;
}

int bshot_binarize(bshot_ctx* ctx, const float* shot, size_t k, size_t stride_floats, uint64_t* bits_out) {
    CHECK_CTX(ctx);
    if ((!shot || !bits_out) && k) { set_error("bshot_binarize: null buffer"); return BSHOT_E_INVALID; }
    if (stride_floats < 352) { set_error("bshot_binarize: stride < 352 floats"); return BSHOT_E_INVALID; }
    if (k > ctx->max_kp) { set_error("bshot_binarize: %zu descriptors > capacity %zu", k, ctx->max_kp); return BSHOT_E_CAPACITY; }
    if (k == 0) return BSHOT_OK;
    BSHOT_CUDA_TRY(cudaMemcpy2DAsync(ctx->d_shot, 352 * sizeof(float), shot, stride_floats * sizeof(float),
                                     352 * sizeof(float), k, cudaMemcpyHostToDevice, ctx->stream));
    BSHOT_TRY(binarize(ctx, ctx->d_shot, k, ctx->d_bits));
    BSHOT_TRY(d2h(ctx, bits_out, ctx->d_bits, sizeof(uint64_t) * 6 * k));
    return sync(ctx);
}

int bshot_compute_descriptors(bshot_ctx* ctx, const bshot_params* p, uint64_t* bits_out) {
    CHECK_CTX(ctx);
    bshot_params dp;
    if (!p) { bshot_params_default(&dp); p = &dp; }
    if (!ctx->have_cloud || !ctx->have_kp) { set_error("bshot_compute_descriptors: need cloud and keypoints"); return BSHOT_E_STATE; }
    BSHOT_TRY(normals_compute(ctx, p->normals_mode, p->normal_radius, p->normal_max_nn));
    BSHOT_TRY(shot_compute(ctx, p->shot_radius, false, false));
    BSHOT_TRY(d2h(ctx, bits_out, ctx->d_bits, sizeof(uint64_t) * 6 * ctx->n_kp));
    return sync(ctx);
}

// ---- a10 + a11 --------------------------------------------------------------------------------
static int upload_qt(bshot_ctx* ctx, const uint64_t* q, size_t nq, const uint64_t* t, size_t nt, const char* who) {
    if ((!q && nq) || (!t && nt)) { set_error("%s: null descriptors", who); return BSHOT_E_INVALID; }
    if (nq > ctx->max_kp) { set_error("%s: %zu queries > capacity %zu", who, nq, ctx->max_kp); return BSHOT_E_CAPACITY; }
    if (nt > ctx->max_targets) { set_error("%s: %zu targets > capacity %zu", who, nt, ctx->max_targets); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(h2d(ctx, ctx->d_q, q, nq * 48));
    BSHOT_TRY(h2d(ctx, ctx->d_t, t, nt * 48));
    return BSHOT_OK;
}

int bshot_match(bshot_ctx* ctx, const uint64_t* q, size_t nq, const uint64_t* t, size_t nt, int* left_idx,
                int* left_dist, int* left_idx2, int* left_dist2, int* right_idx) {
    CHECK_CTX(ctx);
    BSHOT_TRY(upload_qt(ctx, q, nq, t, nt, "bshot_match"));
    if (nq && (left_idx || left_dist || left_idx2 || left_dist2)) {
        if (nt == 0) {
            for (size_t i = 0; i < nq; ++i) {
                if (left_idx) left_idx[i] = -1;
                if (left_dist) left_dist[i] = -1;
                if (left_idx2) left_idx2[i] = -1;
                if (left_dist2) left_dist2[i] = -1;
            }
        } else {
            BSHOT_TRY(hamming_top2(ctx, ctx->d_q, nq, ctx->d_t, nt, 0, ctx->d_cand));
            int* L = ctx->d_left;
            BSHOT_TRY(hamming_unpack(ctx, ctx->d_cand, nq, L, L + nq, L + 2 * nq, L + 3 * nq));
            BSHOT_TRY(d2h(ctx, left_idx, L, sizeof(int) * nq));
            BSHOT_TRY(d2h(ctx, left_dist, L + nq, sizeof(int) * nq));
            BSHOT_TRY(d2h(ctx, left_idx2, L + 2 * nq, sizeof(int) * nq));
            BSHOT_TRY(d2h(ctx, left_dist2, L + 3 * nq, sizeof(int) * nq));
        }
    }
    if (right_idx && nt) {
        if (nq == 0) {
            for (size_t i = 0; i < nt; ++i) right_idx[i] = -1;
        } else {
            // the reference's second loop (src/lidar_odometry.cpp:226-232): roles swapped
            BSHOT_TRY(hamming_top2(ctx, ctx->d_t, nt, ctx->d_q, nq, 0, ctx->d_cand2));
            BSHOT_TRY(hamming_unpack(ctx, ctx->d_cand2, nt, ctx->d_right, nullptr, nullptr, nullptr));
            BSHOT_TRY(d2h(ctx, right_idx, ctx->d_right, sizeof(int) * nt));
        }
    }
    return sync(ctx);
}

int bshot_match_mutual(bshot_ctx* ctx, const uint64_t* q, size_t nq, const uint64_t* t, size_t nt, int* pairs_out,
                       int* dist_out, int* count_out) {
    CHECK_CTX(ctx);
    BSHOT_TRY(upload_qt(ctx, q, nq, t, nt, "bshot_match_mutual"));
    if (count_out) *count_out = 0;
    if (nq == 0 || nt == 0) return sync(ctx);
    BSHOT_TRY(match_mutual(ctx, ctx->d_q, nq, ctx->d_t, nt));
    BSHOT_TRY(d2h(ctx, ctx->h_scratch, ctx->d_pair_count, sizeof(int)));
    BSHOT_TRY(sync(ctx));
    const int n = ctx->h_scratch[0];
    if (count_out) *count_out = n;
    if (n > 0 && (pairs_out || dist_out)) {
        int* tmp = ctx->h_pairs;  // pinned, max_keypoints x 3
        BSHOT_CUDA_TRY(cudaMemcpyAsync(tmp, ctx->d_pairs, sizeof(int) * 3 * n, cudaMemcpyDeviceToHost, ctx->stream));
        BSHOT_TRY(sync(ctx));
        for (int i = 0; i < n; ++i) {
            if (pairs_out) { pairs_out[2 * i] = tmp[3 * i]; pairs_out[2 * i + 1] = tmp[3 * i + 1]; }
            if (dist_out) dist_out[i] = tmp[3 * i + 2];
        }
    }
    return BSHOT_OK;
}

// ---- whole frame --------------------------------------------------------------------------------
static int frame_args_ok(bshot_ctx* ctx, const bshot_params* p, size_t n, size_t stride_bytes, const char* who) {
    if (stride_bytes != 12 && stride_bytes != 16) { set_error("%s: stride must be 12 or 16 bytes", who); return BSHOT_E_INVALID; }
    if (n > ctx->max_points) { set_error("%s: %zu points > capacity %zu", who, n, ctx->max_points); return BSHOT_E_CAPACITY; }
    if (p->top_k <= 0 || (size_t)p->top_k > ctx->max_kp) { set_error("%s: top_k %d outside (0, %zu]", who, p->top_k, ctx->max_kp); return BSHOT_E_CAPACITY; }
    return BSHOT_OK;
}

int bshot_process_frame_dev(bshot_ctx* ctx, const bshot_params* p, const void* d_xyz, size_t n, size_t stride_bytes) {
    CHECK_CTX(ctx);
    bshot_params dp;
    if (!p) { bshot_params_default(&dp); p = &dp; }
    if (!d_xyz && n) { set_error("bshot_process_frame_dev: null cloud"); return BSHOT_E_INVALID; }
    BSHOT_TRY(frame_args_ok(ctx, p, n, stride_bytes, "bshot_process_frame_dev"));
    return frame_run(ctx, p, reinterpret_cast<const float*>(d_xyz), n, (int)(stride_bytes / 4));
}

static int fetch_frame_impl(bshot_ctx* ctx, int top_k, int* kp_idx_out, uint64_t* bits_out, int* n_kp_out, int* pairs_out,
                            int* n_pairs_out, bool payload_early);

int bshot_fetch_frame(bshot_ctx* ctx, int top_k, int* kp_idx_out, uint64_t* bits_out, int* n_kp_out, int* pairs_out,
                      int* n_pairs_out) {
    return fetch_frame_impl(ctx, top_k, kp_idx_out, bits_out, n_kp_out, pairs_out, n_pairs_out, false);
}

// payload_early: keypoint indices and descriptors go over the copy stream as soon as the descriptors are complete (event
// recorded by frame_run), i.e. while the match stage still runs; only the counts and the pairs wait for the end of the frame
static int fetch_frame_impl(bshot_ctx* ctx, int top_k, int* kp_idx_out, uint64_t* bits_out, int* n_kp_out, int* pairs_out,
                            int* n_pairs_out, bool payload_early) {
    CHECK_CTX(ctx);
    if (top_k <= 0 || (size_t)top_k > ctx->max_kp) { set_error("bshot_fetch_frame: bad top_k"); return BSHOT_E_INVALID; }
    if (ctx->last_top_k == 0) { set_error("bshot_fetch_frame: no frame has been processed"); return BSHOT_E_STATE; }
    if ((size_t)top_k < ctx->last_top_k) { set_error("bshot_fetch_frame: top_k %d smaller than the %zu the frame was processed with", top_k, ctx->last_top_k); return BSHOT_E_INVALID; }
    const size_t kmax = ctx->last_top_k;
    // counts + payload in one stream-ordered batch, a single synchronisation
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[0], ctx->d_kp_count, sizeof(int)));
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[1], ctx->d_pair_count, sizeof(int)));
    cudaStream_t ps = payload_early ? ctx->copy_stream : ctx->stream;
    if (payload_early) BSHOT_CUDA_TRY(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_desc, 0));
    if (kp_idx_out) BSHOT_CUDA_TRY(cudaMemcpyAsync(kp_idx_out, ctx->d_kp_idx, sizeof(int) * kmax, cudaMemcpyDeviceToHost, ps));
    if (bits_out) BSHOT_CUDA_TRY(cudaMemcpyAsync(bits_out, ctx->d_bits, sizeof(uint64_t) * 6 * kmax, cudaMemcpyDeviceToHost, ps));
    int* tmp = ctx->h_pairs;  // pinned, max_keypoints x 3: no per-frame host allocation, a true async copy
    if (pairs_out) BSHOT_CUDA_TRY(cudaMemcpyAsync(tmp, ctx->d_pairs, sizeof(int) * 3 * kmax, cudaMemcpyDeviceToHost, ctx->stream));
    BSHOT_TRY(sync(ctx));
    if (payload_early) BSHOT_CUDA_TRY(cudaStreamSynchronize(ctx->copy_stream));
    const int k = std::min(ctx->h_scratch[0], (int)kmax), np = std::min(ctx->h_scratch[1], k);
    ctx->n_kp = (size_t)k;
    if (n_kp_out) *n_kp_out = k;
    if (n_pairs_out) *n_pairs_out = np;
    if (pairs_out)
        for (int i = 0; i < np; ++i) { pairs_out[2 * i] = tmp[3 * i]; pairs_out[2 * i + 1] = tmp[3 * i + 1]; }
    return BSHOT_OK;
}

int bshot_process_frame(bshot_ctx* ctx, const bshot_params* p, const float* xyz, size_t n, size_t stride_bytes,
                        int* kp_idx_out, uint64_t* bits_out, int* n_kp_out, int* pairs_out, int* n_pairs_out) {
    CHECK_CTX(ctx);
    bshot_params dp;
    if (!p) { bshot_params_default(&dp); p = &dp; }
    if (!xyz && n) { set_error("bshot_process_frame: null cloud"); return BSHOT_E_INVALID; }
    BSHOT_TRY(frame_args_ok(ctx, p, n, stride_bytes, "bshot_process_frame"));
    BSHOT_TRY(h2d(ctx, ctx->d_raw, xyz, n * stride_bytes));
    BSHOT_TRY(frame_run(ctx, p, ctx->d_raw, n, (int)(stride_bytes / 4)));
    return fetch_frame_impl(ctx, p->top_k, kp_idx_out, bits_out, n_kp_out, pairs_out, n_pairs_out, true);
}

int bshot_ctx_enable_timing(bshot_ctx* ctx, int on) {
    CHECK_CTX(ctx);
    ctx->timing = on != 0;
    ctx->ev_valid = false;
    return BSHOT_OK;
}

int bshot_stage_times(bshot_ctx* ctx, float ms_out[8]) {
    CHECK_CTX(ctx);
    if (!ms_out) { set_error("bshot_stage_times: null output"); return BSHOT_E_INVALID; }
    if (!ctx->ev_valid) { set_error("bshot_stage_times: no timed frame (call bshot_ctx_enable_timing first)"); return BSHOT_E_STATE; }
    BSHOT_TRY(sync(ctx));
    for (int i = 0; i < 6; ++i) BSHOT_CUDA_TRY(cudaEventElapsedTime(&ms_out[i], ctx->ev[i], ctx->ev[i + 1]));
    BSHOT_CUDA_TRY(cudaEventElapsedTime(&ms_out[6], ctx->ev[0], ctx->ev[6]));
    ms_out[7] = 0.0f;
    return BSHOT_OK;
}

int bshot_frame_counters(bshot_ctx* ctx, unsigned long long out[4]) {
    CHECK_CTX(ctx);
    if (!out) { set_error("bshot_frame_counters: null output"); return BSHOT_E_INVALID; }
    unsigned long long* h = reinterpret_cast<unsigned long long*>(&ctx->h_scratch[32]);
    BSHOT_TRY(d2h(ctx, h, ctx->d_counters, 2 * sizeof(unsigned long long)));
    BSHOT_TRY(d2h(ctx, h + 2, ctx->d_sum_nn, sizeof(unsigned long long)));
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[0], ctx->d_kp_count, sizeof(int)));
    BSHOT_TRY(sync(ctx));
    out[0] = h[0]; out[1] = h[1]; out[2] = h[2]; out[3] = (unsigned long long)ctx->h_scratch[0];
    return BSHOT_OK;
}

int bshot_debug_counters(bshot_ctx* ctx, unsigned long long out[8]) {
    CHECK_CTX(ctx);
    if (!out) { set_error("bshot_debug_counters: null output"); return BSHOT_E_INVALID; }
    BSHOT_CUDA_TRY(cudaMemcpyAsync(out, ctx->d_counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    return sync(ctx);
}

// ---- sharded map --------------------------------------------------------------------------------
int bshot_map_reset(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    ctx->n_map = 0;
    return BSHOT_OK;
}

int bshot_map_append(bshot_ctx* ctx, const uint64_t* desc, size_t n) {
    CHECK_CTX(ctx);
    if (!desc && n) { set_error("bshot_map_append: null descriptors"); return BSHOT_E_INVALID; }
    if (ctx->n_map + n > ctx->max_targets) { set_error("bshot_map_append: shard would hold %zu > capacity %zu", ctx->n_map + n, ctx->max_targets); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(h2d(ctx, ctx->d_map + ctx->n_map * 6, desc, n * 48));
    ctx->n_map += n;
    return sync(ctx);
}

int bshot_map_append_dev(bshot_ctx* ctx, const void* d_desc, size_t n) {
    CHECK_CTX(ctx);
    if (!d_desc && n) { set_error("bshot_map_append_dev: null descriptors"); return BSHOT_E_INVALID; }
    if (ctx->n_map + n > ctx->max_targets) { set_error("bshot_map_append_dev: shard would hold %zu > capacity %zu", ctx->n_map + n, ctx->max_targets); return BSHOT_E_CAPACITY; }
    if (n) BSHOT_CUDA_TRY(cudaMemcpyAsync(ctx->d_map + ctx->n_map * 6, d_desc, n * 48, cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->n_map += n;
    return sync(ctx);
}

int bshot_map_size(bshot_ctx* ctx, size_t* n_out) {
    if (!ctx || !n_out) { set_error("bshot_map_size: null argument"); return BSHOT_E_INVALID; }
    *n_out = ctx->n_map;
    return BSHOT_OK;
}

int bshot_match_dev(bshot_ctx* ctx, const void* d_q, size_t nq, const void* d_t, size_t nt, uint64_t global_base,
                    int with_rq, void* d_cand_out) {
    CHECK_CTX(ctx);
    if (!d_q || !d_cand_out || (!d_t && nt)) { set_error("bshot_match_dev: null device pointer"); return BSHOT_E_INVALID; }
    if (nq > std::max(ctx->max_kp, ctx->max_targets)) { set_error("bshot_match_dev: %zu queries > capacity", nq); return BSHOT_E_CAPACITY; }
    bshot_cand* out = reinterpret_cast<bshot_cand*>(d_cand_out);
    if (nt == 0) {
        BSHOT_CUDA_TRY(cudaMemsetAsync(out, 0xFF, sizeof(bshot_cand) * nq, ctx->stream));
        return BSHOT_OK;
    }
    if (with_rq) {
        if (nq > ctx->max_kp) { set_error("bshot_match_dev: reverse pass needs nq <= max_keypoints"); return BSHOT_E_CAPACITY; }
        return hamming_match_rq(ctx, d_q, nq, d_t, nt, global_base, out);
    }
    return hamming_top2(ctx, d_q, nq, d_t, nt, global_base, out);
}

int bshot_match_shard_dev(bshot_ctx* ctx, const void* d_q, size_t nq, uint64_t global_base, int with_rq, void* d_cand_out) {
    if (!ctx) { set_error("null context"); return BSHOT_E_INVALID; }
    return bshot_match_dev(ctx, d_q, nq, ctx->d_map, ctx->n_map, global_base, with_rq, d_cand_out);
}

int bshot_merge_cands_dev(bshot_ctx* ctx, const void* d_cands, size_t nranks, size_t nq, void* d_out) {
    CHECK_CTX(ctx);
    if (!d_cands || !d_out || nranks == 0) { set_error("bshot_merge_cands_dev: bad arguments"); return BSHOT_E_INVALID; }
    return hamming_merge_cands(ctx, d_cands, nranks, nq, d_out);
}

int bshot_reverse_owned_dev(bshot_ctx* ctx, const void* d_q, size_t nq, uint64_t global_base, const void* d_merged,
                            void* d_rq_out) {
    CHECK_CTX(ctx);
    if (!d_q || !d_merged || !d_rq_out) { set_error("bshot_reverse_owned_dev: null device pointer"); return BSHOT_E_INVALID; }
    return hamming_reverse_owned(ctx, d_q, nq, ctx->d_map, ctx->n_map, global_base, reinterpret_cast<const bshot_cand*>(d_merged),
                                 reinterpret_cast<unsigned*>(d_rq_out));
}

int bshot_peer_barrier_dev(bshot_ctx* ctx, const void* d_peer_flag_ptrs, int nranks, int rank) {
    CHECK_CTX(ctx);
    if (!d_peer_flag_ptrs || nranks <= 0 || rank < 0 || rank >= nranks) { set_error("bshot_peer_barrier_dev: bad arguments"); return BSHOT_E_INVALID; }
    return hamming_peer_barrier(ctx, d_peer_flag_ptrs, (unsigned)nranks, (unsigned)rank);
}

int bshot_peer_barrier_reset(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    BSHOT_TRY(sync(ctx));
    ctx->peer_epoch = 0;   // the epoch belongs to the (freshly zeroed) flag array the caller is about to use
    BSHOT_CUDA_TRY(cudaMemsetAsync(ctx->d_pair_count + 3, 0, sizeof(int), ctx->stream));
    return sync(ctx);
}

int bshot_peer_barrier_timeouts(bshot_ctx* ctx, unsigned* epoch_out) {
    CHECK_CTX(ctx);
    if (!epoch_out) { set_error("bshot_peer_barrier_timeouts: null output"); return BSHOT_E_INVALID; }
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[16], ctx->d_pair_count + 3, sizeof(int)));
    BSHOT_TRY(sync(ctx));
    *epoch_out = (unsigned)ctx->h_scratch[16];
    return BSHOT_OK;
}

int bshot_push_cands_dev(bshot_ctx* ctx, const void* d_cands, size_t nq, const void* d_peer_ptrs, int nranks, int rank) {
    CHECK_CTX(ctx);
    if (!d_cands || !d_peer_ptrs || nranks <= 0 || rank < 0 || rank >= nranks) { set_error("bshot_push_cands_dev: bad arguments"); return BSHOT_E_INVALID; }
    return hamming_push_cands(ctx, reinterpret_cast<const bshot_cand*>(d_cands), nq, d_peer_ptrs, (unsigned)nranks, (unsigned)rank);
}

int bshot_reverse_owned_push_dev(bshot_ctx* ctx, const void* d_q, size_t nq, uint64_t global_base, const void* d_merged,
                                 const void* d_peer_rq_ptrs, int nranks, int rank) {
    CHECK_CTX(ctx);
    if (!d_q || !d_merged || !d_peer_rq_ptrs || nranks <= 0 || rank < 0 || rank >= nranks) { set_error("bshot_reverse_owned_push_dev: bad arguments"); return BSHOT_E_INVALID; }
    return hamming_reverse_owned(ctx, d_q, nq, ctx->d_map, ctx->n_map, global_base, reinterpret_cast<const bshot_cand*>(d_merged),
                                 nullptr, d_peer_rq_ptrs, (unsigned)nranks, (unsigned)rank);
}

int bshot_apply_rq_dev(bshot_ctx* ctx, void* d_cands, const void* d_rq, size_t nq) {
    CHECK_CTX(ctx);
    if (!d_cands || !d_rq) { set_error("bshot_apply_rq_dev: null device pointer"); return BSHOT_E_INVALID; }
    return hamming_apply_rq(ctx, reinterpret_cast<bshot_cand*>(d_cands), reinterpret_cast<const unsigned*>(d_rq), nq);
}

// ---- GPU-resident global map + frame-to-map flow (SURVEY 8a row a9, 8f #2) --------------------------------------------
int bshot_gmap_create(bshot_ctx* ctx, size_t max_entries, size_t max_blocks) {
    CHECK_CTX(ctx);
    if (max_entries == 0 || max_blocks == 0 || max_entries > 0x7FFFFFFFull) { set_error("bshot_gmap_create: bad capacities"); return BSHOT_E_INVALID; }
    if (ctx->gmap.d_tab) { set_error("bshot_gmap_create: the context already has a map"); return BSHOT_E_STATE; }
    BSHOT_TRY(gmap_create(ctx, max_entries, max_blocks));
    return sync(ctx);
}

int bshot_gmap_reset(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    BSHOT_TRY(gmap_reset(ctx));
    return sync(ctx);
}

int bshot_gmap_size(bshot_ctx* ctx, size_t* entries_out, size_t* dropped_out) {
    CHECK_CTX(ctx);
    if (!ctx->gmap.d_tab) { set_error("bshot_gmap_size: no map"); return BSHOT_E_STATE; }
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[40], ctx->gmap.d_ctl, 8 * sizeof(unsigned)));
    BSHOT_TRY(sync(ctx));
    if (entries_out) *entries_out = (size_t)(unsigned)ctx->h_scratch[40];
    if (dropped_out) *dropped_out = (size_t)(unsigned)ctx->h_scratch[43];
    return BSHOT_OK;
}

// a map update's pose (NULL = identity) must be finite: a NaN or an infinity would make every keypoint unstorable, and the
// update would still count and write its pose into the trajectory
static bool pose_finite(const float* pose3x4, const char* who) {
    if (pose3x4)
        for (int k = 0; k < 12; ++k)
            if (!std::isfinite(pose3x4[k])) { set_error("%s: the pose is not finite", who); return false; }
    return true;
}

int bshot_gmap_add(bshot_ctx* ctx, const float* xyz, const float* seg_ratio, const uint64_t* desc, size_t n, const float* pose3x4) {
    CHECK_CTX(ctx);
    if (!pose_finite(pose3x4, "bshot_gmap_add")) return BSHOT_E_INVALID;
    if (n == 0) return BSHOT_OK;
    if (!xyz || !seg_ratio || !desc) { set_error("bshot_gmap_add: null input"); return BSHOT_E_INVALID; }
    if (n > ctx->max_kp) { set_error("bshot_gmap_add: %zu keypoints > max_keypoints %zu per call", n, ctx->max_kp); return BSHOT_E_CAPACITY; }
    // staged in the scratch buffers of the matcher (d_gather as float4 positions, d_left as ratios, d_q as descriptors)
    float4* d_pos = reinterpret_cast<float4*>(ctx->d_gather);
    float* d_ratio = reinterpret_cast<float*>(ctx->d_left);
    BSHOT_CUDA_TRY(cudaMemsetAsync(d_pos, 0, sizeof(float4) * n, ctx->stream));
    BSHOT_CUDA_TRY(cudaMemcpy2DAsync(d_pos, 16, xyz, 12, 12, n, cudaMemcpyHostToDevice, ctx->stream));
    BSHOT_TRY(h2d(ctx, d_ratio, seg_ratio, sizeof(float) * n));
    BSHOT_TRY(h2d(ctx, ctx->d_q, desc, 48 * n));
    BSHOT_TRY(gmap_update(ctx, d_pos, d_ratio, ctx->d_q, nullptr, n, pose3x4));
    gmap_record_update(ctx, n, /*by_scan=*/false);
    return sync(ctx);
}

int bshot_gmap_update_from_frame(bshot_ctx* ctx, const float* pose3x4) {
    CHECK_CTX(ctx);
    if (!ctx->have_kp || ctx->last_top_k == 0) { set_error("bshot_gmap_update_from_frame: no extracted frame"); return BSHOT_E_STATE; }
    if (!pose_finite(pose3x4, "bshot_gmap_update_from_frame")) return BSHOT_E_INVALID;
    BSHOT_TRY(gmap_update(ctx, ctx->d_kp, ctx->d_kp_ratio, ctx->d_bits, ctx->d_kp_count, ctx->last_top_k, pose3x4));
    gmap_record_update(ctx, ctx->last_top_k, /*by_scan=*/false);
    return BSHOT_OK;  // asynchronous
}

int bshot_gmap_get_keypoints(bshot_ctx* ctx, const float pos[3], float range, float* xyz_out, uint64_t* desc_out, size_t cap, size_t* n_out) {
    CHECK_CTX(ctx);
    if (!pos) { set_error("bshot_gmap_get_keypoints: null position"); return BSHOT_E_INVALID; }
    unsigned* d_total = ctx->gmap.d_ctl ? ctx->gmap.d_ctl + 6 : nullptr;
    BSHOT_TRY(gmap_gather(ctx, pos, range, nullptr, nullptr, nullptr, 0, nullptr, ctx->d_t, ctx->max_targets, d_total));
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[40], ctx->gmap.d_ctl, 8 * sizeof(unsigned)));
    BSHOT_TRY(sync(ctx));
    const size_t n = (size_t)(unsigned)ctx->h_scratch[44];
    if (n_out) *n_out = n;
    if (n > ctx->max_targets) { set_error("bshot_gmap_get_keypoints: %zu keypoints in range > max_targets %zu", n, ctx->max_targets); return BSHOT_E_CAPACITY; }
    const size_t m = std::min(n, cap);
    if (xyz_out && m) BSHOT_CUDA_TRY(cudaMemcpy2DAsync(xyz_out, 12, ctx->gmap.d_tpos, 16, 12, m, cudaMemcpyDeviceToHost, ctx->stream));
    if (desc_out && m) BSHOT_TRY(d2h(ctx, desc_out, ctx->d_t, 48 * m));
    return sync(ctx);
}

int bshot_gmap_export(bshot_ctx* ctx, float* xyzr_out, uint64_t* desc_out, size_t cap, size_t* n_out) {
    CHECK_CTX(ctx);
    if (!ctx->gmap.d_tab) { set_error("bshot_gmap_export: no map (bshot_gmap_create)"); return BSHOT_E_STATE; }
    return gmap_export(ctx, xyzr_out, desc_out, cap, n_out);
}

int bshot_gmap_import(bshot_ctx* ctx, const float* xyzr, const uint64_t* desc, size_t n) {
    CHECK_CTX(ctx);
    if (!ctx->gmap.d_tab) { set_error("bshot_gmap_import: no map (bshot_gmap_create)"); return BSHOT_E_STATE; }
    if (n && (!xyzr || !desc)) { set_error("bshot_gmap_import: null input"); return BSHOT_E_INVALID; }
    return gmap_import(ctx, xyzr, desc, n);
}

int bshot_gmap_scans(bshot_ctx* ctx, uint32_t* entry_scan_out, size_t entry_cap, float* poses3x4_out, size_t pose_cap, size_t* n_entries_out,
                     size_t* n_scans_out) {
    CHECK_CTX(ctx);
    if (!ctx->gmap.d_tab) { set_error("bshot_gmap_scans: no map (bshot_gmap_create)"); return BSHOT_E_STATE; }
    return gmap_scans(ctx, entry_scan_out, entry_cap, poses3x4_out, pose_cap, n_entries_out, n_scans_out);
}

// a finite rigid [R|T] (row-major, rows 4 floats apart): max |R^T R - I| <= 1e-3 and det R > 0
static bool rigid_ok(const float* T, const char* who, const char* what, size_t index) {
    for (int r = 0; r < 3; ++r)
        for (int e = 0; e < 4; ++e)
            if (!std::isfinite(T[4 * r + e])) { set_error("%s: %s %zu is not finite", who, what, index); return false; }
    double R[3][3], dev = 0.0;
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) R[i][j] = T[4 * i + j];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            const double d = R[0][i] * R[0][j] + R[1][i] * R[1][j] + R[2][i] * R[2][j] - (i == j ? 1.0 : 0.0);
            dev = std::max(dev, std::fabs(d));
        }
    const double det = R[0][0] * (R[1][1] * R[2][2] - R[1][2] * R[2][1]) - R[0][1] * (R[1][0] * R[2][2] - R[1][2] * R[2][0]) +
                       R[0][2] * (R[1][0] * R[2][1] - R[1][1] * R[2][0]);
    if (dev > 1e-3 || !(det > 0.0)) { set_error("%s: %s %zu is not a rotation (|R^T R - I| %.3g, det %.3g)", who, what, index, dev, det); return false; }
    return true;
}

int bshot_gmap_reanchor(bshot_ctx* ctx, const float* poses3x4, size_t n, float* pose_out) {
    CHECK_CTX(ctx);
    if (!ctx->gmap.d_tab) { set_error("bshot_gmap_reanchor: no map (bshot_gmap_create)"); return BSHOT_E_STATE; }
    if (n != ctx->gmap.n_updates) { set_error("bshot_gmap_reanchor: %zu poses for %u map updates", n, ctx->gmap.n_updates); return BSHOT_E_INVALID; }
    if (n && !poses3x4) { set_error("bshot_gmap_reanchor: null poses"); return BSHOT_E_INVALID; }
    for (size_t u = 0; u < n; ++u)
        if (!rigid_ok(poses3x4 + 12 * u, "bshot_gmap_reanchor", "pose", u)) return BSHOT_E_INVALID;
    return reanchor_run(ctx, poses3x4, n, pose_out);
}

void bshot_graph_params_default(bshot_graph_params* p) {
    if (!p) return;
    p->odom_sigma_mm = 20.0f;
    p->odom_sigma_deg = 0.1f;
    p->loop_sigma_mm = 100.0f;
    p->loop_sigma_deg = 1.0f;
    p->max_iterations = 50;
    p->max_cg_iterations = 2000;
    p->grad_tolerance = 1e-6;
    p->step_tolerance = 1e-9;
    p->cg_tolerance = 1e-10;
}

int bshot_optimize_trajectory(bshot_ctx* ctx, const bshot_graph_edge* loops, size_t n_loops, const bshot_graph_params* p, float* poses3x4_out,
                              size_t pose_cap, double* loop_cost_out, bshot_graph_report* out) {
    CHECK_CTX(ctx);
    const char* who = "bshot_optimize_trajectory";
    bshot_graph_params dp;
    if (!p) { bshot_graph_params_default(&dp); p = &dp; }
    if (!ctx->gmap.d_tab) { set_error("%s: no map (bshot_gmap_create)", who); return BSHOT_E_STATE; }
    const float sig[4] = {p->odom_sigma_mm, p->odom_sigma_deg, p->loop_sigma_mm, p->loop_sigma_deg};
    for (float s : sig) if (!(s > 0.0f) || !std::isfinite(s)) { set_error("%s: every sigma must be finite and > 0", who); return BSHOT_E_INVALID; }
    if (p->max_iterations < 0 || p->max_cg_iterations < 0) { set_error("%s: negative iteration count", who); return BSHOT_E_INVALID; }
    if (!(p->grad_tolerance >= 0.0) || !(p->step_tolerance >= 0.0) || !(p->cg_tolerance >= 0.0)) { set_error("%s: negative tolerance", who); return BSHOT_E_INVALID; }
    if (n_loops && !loops) { set_error("%s: null loop edges", who); return BSHOT_E_INVALID; }
    if (n_loops > 0x7FFFFFFFull) { set_error("%s: too many loop edges", who); return BSHOT_E_INVALID; }
    const size_t n = ctx->gmap.n_updates;
    for (size_t k = 0; k < n_loops; ++k) {
        const bshot_graph_edge& e = loops[k];
        if (e.from < 0 || e.to < 0 || (size_t)e.from >= n || (size_t)e.to >= n || e.from == e.to) {
            set_error("%s: loop edge %zu (%d, %d) outside [0, %zu) or a self-loop", who, k, e.from, e.to, n);
            return BSHOT_E_INVALID;
        }
        if (!rigid_ok(e.T, who, "loop edge", k)) return BSHOT_E_INVALID;
    }
    if (pose_cap < n || (n && !poses3x4_out)) { set_error("%s: %zu nodes > pose capacity %zu", who, n, pose_cap); return BSHOT_E_CAPACITY; }
    return pose_graph_run(ctx, loops, n_loops, p, poses3x4_out, loop_cost_out, out);
}

int bshot_extract_frame(bshot_ctx* ctx, const bshot_params* p, const float* xyz, size_t n, size_t stride_bytes, int* kp_idx_out, float* kp_xyz_out,
                        float* seg_ratio_out, uint64_t* bits_out, int* n_kp_out) {
    CHECK_CTX(ctx);
    bshot_params dp;
    if (!p) { bshot_params_default(&dp); p = &dp; }
    if (!xyz && n) { set_error("bshot_extract_frame: null cloud"); return BSHOT_E_INVALID; }
    BSHOT_TRY(frame_args_ok(ctx, p, n, stride_bytes, "bshot_extract_frame"));
    BSHOT_TRY(h2d(ctx, ctx->d_raw, xyz, n * stride_bytes));
    BSHOT_TRY(frame_extract(ctx, p, ctx->d_raw, n, (int)(stride_bytes / 4)));
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[0], ctx->d_kp_count, sizeof(int)));
    BSHOT_TRY(sync(ctx));
    const int k = std::min(ctx->h_scratch[0], p->top_k);
    ctx->n_kp = (size_t)k;
    if (n_kp_out) *n_kp_out = k;
    BSHOT_TRY(d2h(ctx, kp_idx_out, ctx->d_kp_idx, sizeof(int) * k));
    BSHOT_TRY(d2h(ctx, seg_ratio_out, ctx->d_kp_ratio, sizeof(float) * k));
    BSHOT_TRY(d2h(ctx, bits_out, ctx->d_bits, 48 * (size_t)k));
    if (kp_xyz_out && k) BSHOT_CUDA_TRY(cudaMemcpy2DAsync(kp_xyz_out, 12, ctx->d_kp, 16, 12, k, cudaMemcpyDeviceToHost, ctx->stream));
    return sync(ctx);
}

int bshot_extract_scan(bshot_ctx* ctx, const bshot_params* p, const double* azimuth_deg, const double* vertical_deg, const unsigned short* distance, size_t n,
                       const double* ring_deg, size_t nv, double vert_init_rad, double lowpt_th, float* cloud_xyz_out, size_t cloud_cap,
                       size_t* n_points_out, int* kp_idx_out, float* kp_xyz_out, float* seg_ratio_out, uint64_t* bits_out, int* n_kp_out) {
    CHECK_CTX(ctx);
    bshot_params dp;
    if (!p) { bshot_params_default(&dp); p = &dp; }
    if (n && (!azimuth_deg || !vertical_deg || !distance)) { set_error("bshot_extract_scan: null input"); return BSHOT_E_INVALID; }
    if (nv && !ring_deg) { set_error("bshot_extract_scan: null ring table"); return BSHOT_E_INVALID; }
    if (n > 0xFFFFFFFFull) { set_error("bshot_extract_scan: too many returns"); return BSHOT_E_CAPACITY; }
    // Preprocessor::run; the cloud stays on the device and goes straight into the front end (no host round trip)
    size_t kept = 0;
    const float* d_cloud = nullptr;
    BSHOT_TRY(preprocess_run(ctx, azimuth_deg, vertical_deg, distance, n, ring_deg, nv, vert_init_rad, lowpt_th, nullptr, 1, cloud_xyz_out,
                             cloud_xyz_out ? cloud_cap : std::max<size_t>(n, 1), &kept, &d_cloud));
    if (n_points_out) *n_points_out = kept;
    if (cloud_xyz_out && kept > cloud_cap) { set_error("bshot_extract_scan: %zu points kept > capacity %zu", kept, cloud_cap); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(frame_args_ok(ctx, p, kept, 12, "bshot_extract_scan"));
    BSHOT_TRY(frame_extract(ctx, p, d_cloud, kept, 3));
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[0], ctx->d_kp_count, sizeof(int)));
    BSHOT_TRY(sync(ctx));
    const int k = std::min(ctx->h_scratch[0], p->top_k);
    ctx->n_kp = (size_t)k;
    if (n_kp_out) *n_kp_out = k;
    if (kp_idx_out) BSHOT_TRY(d2h(ctx, kp_idx_out, ctx->d_kp_idx, sizeof(int) * k));
    if (seg_ratio_out) BSHOT_TRY(d2h(ctx, seg_ratio_out, ctx->d_kp_ratio, sizeof(float) * k));
    if (bits_out) BSHOT_TRY(d2h(ctx, bits_out, ctx->d_bits, 48 * (size_t)k));
    if (kp_xyz_out && k) BSHOT_CUDA_TRY(cudaMemcpy2DAsync(kp_xyz_out, 12, ctx->d_kp, 16, 12, k, cudaMemcpyDeviceToHost, ctx->stream));
    return sync(ctx);
}

int bshot_frame_commit(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    if (ctx->last_top_k == 0) { set_error("bshot_frame_commit: no extracted frame"); return BSHOT_E_STATE; }
    return frame_commit(ctx, ctx->last_top_k);
}

int bshot_match_frame_to_map(bshot_ctx* ctx, const float ref_pos[3], float range, const float* ref_pose3x4, int* pairs_out, int* n_pairs_out,
                             size_t* n_targets_out, float* target_xyz_out, size_t target_cap) {
    CHECK_CTX(ctx);
    if (!ref_pos) { set_error("bshot_match_frame_to_map: null position"); return BSHOT_E_INVALID; }
    if (!ctx->gmap.d_tab || ctx->last_top_k == 0) { set_error("bshot_match_frame_to_map: needs a map and an extracted frame"); return BSHOT_E_STATE; }
    const size_t k = ctx->last_top_k;
    size_t nt_cap;
    BSHOT_TRY(frame_match_map(ctx, k, ref_pos, range, ref_pose3x4, /*pose_on_device=*/false, &nt_cap));
    if (nt_cap == 0) { if (n_pairs_out) *n_pairs_out = 0; if (n_targets_out) *n_targets_out = 0; return sync(ctx); }
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[1], ctx->d_pair_count, sizeof(int)));
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[40], ctx->gmap.d_ctl, 8 * sizeof(unsigned)));
    if (pairs_out) BSHOT_CUDA_TRY(cudaMemcpyAsync(ctx->h_pairs, ctx->d_pairs, sizeof(int) * 3 * k, cudaMemcpyDeviceToHost, ctx->stream));
    BSHOT_TRY(sync(ctx));
    const unsigned* ctl = reinterpret_cast<const unsigned*>(&ctx->h_scratch[40]);
    const size_t total = ctl[6];
    if (target_set_overflow(ctl, ctx->n_prev, ctx->max_targets)) { set_error("bshot_match_frame_to_map: target set exceeds max_targets %zu", ctx->max_targets); return BSHOT_E_CAPACITY; }
    const int np = std::min(ctx->h_scratch[1], (int)k);
    if (n_pairs_out) *n_pairs_out = np;
    if (n_targets_out) *n_targets_out = total;
    if (pairs_out) for (int i = 0; i < np; ++i) { pairs_out[2 * i] = ctx->h_pairs[3 * i]; pairs_out[2 * i + 1] = ctx->h_pairs[3 * i + 1]; }
    if (target_xyz_out && total) {
        BSHOT_CUDA_TRY(cudaMemcpy2DAsync(target_xyz_out, 12, ctx->gmap.d_tpos, 16, 12, std::min(total, target_cap), cudaMemcpyDeviceToHost, ctx->stream));
        BSHOT_TRY(sync(ctx));
    }
    return BSHOT_OK;
}

// ---- RANSAC correspondence rejection (SURVEY 8f #1) -----------------------------------------------------------------------
int bshot_ransac(bshot_ctx* ctx, const float* src_xyz, size_t n_src, const float* tgt_xyz, size_t n_tgt, const int* pairs, size_t n_pairs,
                 int max_iterations, float inlier_threshold, int* inlier_pairs_out, int* n_inliers_out, float* transform4x4_out, int* iterations_out) {
    CHECK_CTX(ctx);
    if ((!src_xyz || !tgt_xyz || !pairs) && n_pairs) { set_error("bshot_ransac: null input"); return BSHOT_E_INVALID; }
    for (size_t i = 0; i < n_pairs; ++i)
        if (pairs[2 * i] < 0 || (size_t)pairs[2 * i] >= n_src || pairs[2 * i + 1] < 0 || (size_t)pairs[2 * i + 1] >= n_tgt) {
            set_error("bshot_ransac: correspondence %zu out of range", i);
            return BSHOT_E_INVALID;
        }
    return ransac_run(ctx, src_xyz, tgt_xyz, pairs, n_pairs, max_iterations, (double)inlier_threshold, inlier_pairs_out, n_inliers_out, transform4x4_out,
                      iterations_out);
}

int bshot_icp(bshot_ctx* ctx, const float* src_xyz, size_t n_src, const float* tgt_xyz, size_t n_tgt, const float* pre4x4, int max_iterations,
              float* final4x4_out, int* iterations_out, int* state_out, double* mse_out) {
    CHECK_CTX(ctx);
    if ((n_src && !src_xyz) || (n_tgt && !tgt_xyz)) { set_error("bshot_icp: null input"); return BSHOT_E_INVALID; }
    if (max_iterations < 0 || max_iterations > 1000) { set_error("bshot_icp: max_iterations out of range"); return BSHOT_E_INVALID; }
    if (n_src > 0x7FFFFFFFull || n_tgt > 0x7FFFFFFFull) { set_error("bshot_icp: too many points"); return BSHOT_E_CAPACITY; }
    return icp_run(ctx, src_xyz, n_src, tgt_xyz, n_tgt, pre4x4, max_iterations, final4x4_out, iterations_out, state_out, mse_out);
}

int bshot_evaluate_estimation(bshot_ctx* ctx, const float* T_ransac, const float* T_ref, int n_correspondences, const float* src_kp, size_t n_src,
                              const float* tgt_kp, size_t n_tgt, int run_icp, float* T_best_out, int* should_update_map_out, float* h_diff_out,
                              float* t_diff_out, int* icp_iterations_out) {
    CHECK_CTX(ctx);
    if (!T_ransac || !T_ref || !T_best_out) { set_error("bshot_evaluate_estimation: null matrix"); return BSHOT_E_INVALID; }
    float h_diff, t_diff;
    const bool reject = estimation_gate(T_ransac, T_ref, n_correspondences, &h_diff, &t_diff);   // :269-281 (odom_math.cuh)
    const float* T_est = reject ? T_ref : T_ransac;
    if (should_update_map_out) *should_update_map_out = reject ? 0 : 1;
    if (h_diff_out) *h_diff_out = h_diff;
    if (t_diff_out) *t_diff_out = t_diff;
    if (icp_iterations_out) *icp_iterations_out = 0;
    if (run_icp) {
        float F[16];
        BSHOT_TRY(bshot_icp(ctx, src_kp, n_src, tgt_kp, n_tgt, T_est, 10, F, icp_iterations_out, nullptr, nullptr));
        mul4x4(F, T_est, T_best_out);                                // T_best_ = icp.getFinalTransformation() * T_est (:293)
    } else {
        for (int e = 0; e < 16; ++e) T_best_out[e] = T_ransac[e];    // :295
    }
    return BSHOT_OK;
}

int bshot_preprocess_select(bshot_ctx* ctx, const double* azimuth_deg, const double* vertical_deg, const unsigned short* distance, size_t n,
                            const double* ring_deg, size_t nv, double vert_init_rad, double lowpt_th, const int* select_list, size_t n_select,
                            int have_select_list, int save_selected, float* xyz_out, size_t cap, size_t* n_out) {
    CHECK_CTX(ctx);
    if (n && (!azimuth_deg || !vertical_deg || !distance)) { set_error("bshot_preprocess: null input"); return BSHOT_E_INVALID; }
    if (nv && !ring_deg) { set_error("bshot_preprocess: null ring table"); return BSHOT_E_INVALID; }
    if (n_select && !select_list) { set_error("bshot_preprocess: null select list"); return BSHOT_E_INVALID; }
    if (n > 0xFFFFFFFFull) { set_error("bshot_preprocess: too many returns"); return BSHOT_E_CAPACITY; }
    // selmap of readFrame (src/preprocess.cpp:58-67): the sorted list (setSelectedPoints sorts it, :25-28) is walked with one
    // cursor that only advances on a hit -- restated as is, including what a duplicated entry does to the rest of the list
    std::vector<unsigned char> sel;
    if (have_select_list) {
        std::vector<int> list(select_list, select_list + n_select);
        std::sort(list.begin(), list.end());
        sel.assign(n, 0);
        size_t cursor = 0;
        for (size_t i = 0; i < n; ++i)
            if (cursor < list.size() && list[cursor] == (int)i) { sel[i] = 1; ++cursor; }
    }
    size_t kept = 0;
    BSHOT_TRY(preprocess_run(ctx, azimuth_deg, vertical_deg, distance, n, ring_deg, nv, vert_init_rad, lowpt_th, have_select_list ? sel.data() : nullptr,
                             save_selected, xyz_out, cap, &kept));
    if (n_out) *n_out = kept;
    if (kept > cap && xyz_out) { set_error("bshot_preprocess: %zu points kept > capacity %zu", kept, cap); return BSHOT_E_CAPACITY; }
    return BSHOT_OK;
}

int bshot_preprocess(bshot_ctx* ctx, const double* azimuth_deg, const double* vertical_deg, const unsigned short* distance, size_t n, const double* ring_deg,
                     size_t nv, double vert_init_rad, double lowpt_th, float* xyz_out, size_t cap, size_t* n_out) {
    return bshot_preprocess_select(ctx, azimuth_deg, vertical_deg, distance, n, ring_deg, nv, vert_init_rad, lowpt_th, nullptr, 0, 0, 1, xyz_out, cap, n_out);
}

// ---- the per-scan odometry step (test/odometry_test.cpp:143-184, odometry.cu) ---------------------------------------
void bshot_odom_params_default(bshot_odom_params* p) {
    if (!p) return;
    bshot_params_default(&p->front);
    p->vert_init_rad = -0.6;
    p->lowpt_th = -1950.0;
    p->map_range = 100000.0f;
    p->ransac_iterations = 2000;
    p->inlier_threshold = 1500.0f;
    p->run_icp = 1;
}

// the registration parameters of the step, relocalisation (min_inliers) and loop detection (min_inliers), and the map
static int reg_args_ok(bshot_ctx* ctx, const int* min_inliers, int ransac_iterations, float inlier_threshold, float map_range, const char* who) {
    if (min_inliers && *min_inliers < 3) { set_error("%s: min_inliers %d < 3", who, *min_inliers); return BSHOT_E_INVALID; }
    if (ransac_iterations < 1 || ransac_iterations > 100000) { set_error("%s: ransac_iterations %d outside [1, 100000]", who, ransac_iterations); return BSHOT_E_INVALID; }
    if (!(inlier_threshold > 0.0f) || !std::isfinite(inlier_threshold)) { set_error("%s: inlier_threshold must be finite and > 0", who); return BSHOT_E_INVALID; }
    if (!(map_range >= 0.0f) || !std::isfinite(map_range)) { set_error("%s: map_range must be finite and >= 0", who); return BSHOT_E_INVALID; }
    if (!ctx->gmap.d_tab) { set_error("%s: needs a map (bshot_gmap_create)", who); return BSHOT_E_STATE; }
    return BSHOT_OK;
}

// raw returns of the step or a relocalisation: the returns' and the parameters' checks, then Preprocessor::run, whose two
// count read-backs size the front end's grids; the cloud (*kept points, 3 floats each) stays on the device in *d_cloud
static int scan_to_device(bshot_ctx* ctx, const bshot_odom_params* p, const int* min_inliers, const double* azimuth_deg, const double* vertical_deg,
                          const unsigned short* distance, size_t n, const double* ring_deg, size_t nv, const char* who, const float** d_cloud, size_t* kept) {
    if (n && (!azimuth_deg || !vertical_deg || !distance)) { set_error("%s: null input", who); return BSHOT_E_INVALID; }
    if (nv && !ring_deg) { set_error("%s: null ring table", who); return BSHOT_E_INVALID; }
    if (n > 0xFFFFFFFFull) { set_error("%s: too many returns", who); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(reg_args_ok(ctx, min_inliers, p->ransac_iterations, p->inlier_threshold, p->map_range, who));
    BSHOT_TRY(preprocess_run(ctx, azimuth_deg, vertical_deg, distance, n, ring_deg, nv, p->vert_init_rad, p->lowpt_th, nullptr, 1, nullptr, std::max<size_t>(n, 1),
                             kept, d_cloud));
    return frame_args_ok(ctx, &p->front, *kept, 12, who);
}

// a preprocessed host cloud of the step or a relocalisation: the checks, then the upload into ctx->d_raw
static int cloud_to_device(bshot_ctx* ctx, const bshot_odom_params* p, const int* min_inliers, const float* xyz, size_t n, size_t stride_bytes, const char* who) {
    if (!xyz && n) { set_error("%s: null cloud", who); return BSHOT_E_INVALID; }
    BSHOT_TRY(reg_args_ok(ctx, min_inliers, p->ransac_iterations, p->inlier_threshold, p->map_range, who));
    BSHOT_TRY(frame_args_ok(ctx, &p->front, n, stride_bytes, who));
    return h2d(ctx, ctx->d_raw, xyz, n * stride_bytes);
}

int bshot_odometry_step(bshot_ctx* ctx, const bshot_odom_params* p, const double* azimuth_deg, const double* vertical_deg, const unsigned short* distance,
                        size_t n, const double* ring_deg, size_t nv, bshot_odom_report* out) {
    CHECK_CTX(ctx);
    bshot_odom_params dp;
    if (!p) { bshot_odom_params_default(&dp); p = &dp; }
    size_t kept = 0;
    const float* d_cloud = nullptr;
    BSHOT_TRY(scan_to_device(ctx, p, nullptr, azimuth_deg, vertical_deg, distance, n, ring_deg, nv, "bshot_odometry_step", &d_cloud, &kept));
    return odometry_run(ctx, p, d_cloud, kept, 3, out);
}

int bshot_odometry_step_cloud(bshot_ctx* ctx, const bshot_odom_params* p, const float* xyz, size_t n, size_t stride_bytes, bshot_odom_report* out) {
    CHECK_CTX(ctx);
    bshot_odom_params dp;
    if (!p) { bshot_odom_params_default(&dp); p = &dp; }
    BSHOT_TRY(cloud_to_device(ctx, p, nullptr, xyz, n, stride_bytes, "bshot_odometry_step_cloud"));
    return odometry_run(ctx, p, ctx->d_raw, n, (int)(stride_bytes / 4), out);
}

int bshot_relocalize(bshot_ctx* ctx, const bshot_odom_params* p, int min_inliers, const double* azimuth_deg, const double* vertical_deg,
                     const unsigned short* distance, size_t n, const double* ring_deg, size_t nv, bshot_reloc_report* out) {
    CHECK_CTX(ctx);
    bshot_odom_params dp;
    if (!p) { bshot_odom_params_default(&dp); p = &dp; }
    size_t kept = 0;
    const float* d_cloud = nullptr;
    BSHOT_TRY(scan_to_device(ctx, p, &min_inliers, azimuth_deg, vertical_deg, distance, n, ring_deg, nv, "bshot_relocalize", &d_cloud, &kept));
    return relocalize_run(ctx, p, min_inliers, d_cloud, kept, 3, out);
}

int bshot_relocalize_cloud(bshot_ctx* ctx, const bshot_odom_params* p, int min_inliers, const float* xyz, size_t n, size_t stride_bytes,
                           bshot_reloc_report* out) {
    CHECK_CTX(ctx);
    bshot_odom_params dp;
    if (!p) { bshot_odom_params_default(&dp); p = &dp; }
    BSHOT_TRY(cloud_to_device(ctx, p, &min_inliers, xyz, n, stride_bytes, "bshot_relocalize_cloud"));
    return relocalize_run(ctx, p, min_inliers, ctx->d_raw, n, (int)(stride_bytes / 4), out);
}

void bshot_loop_params_default(bshot_loop_params* p) {
    if (!p) return;
    p->min_gap = 100;
    p->min_inliers = 15;
    p->ransac_iterations = 2000;
    p->inlier_threshold = 1500.0f;
    p->map_range = 100000.0f;
    p->run_icp = 1;
}

int bshot_detect_loop(bshot_ctx* ctx, const bshot_loop_params* p, bshot_loop_report* out) {
    CHECK_CTX(ctx);
    bshot_loop_params dp;
    if (!p) { bshot_loop_params_default(&dp); p = &dp; }
    if (p->min_gap < 1) { set_error("bshot_detect_loop: min_gap %d < 1", p->min_gap); return BSHOT_E_INVALID; }
    BSHOT_TRY(reg_args_ok(ctx, &p->min_inliers, p->ransac_iterations, p->inlier_threshold, p->map_range, "bshot_detect_loop"));
    return loop_run(ctx, p, out);
}

int bshot_odometry_reset(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    if (!ctx->gmap.d_tab) { set_error("bshot_odometry_reset: needs a map (bshot_gmap_create)"); return BSHOT_E_STATE; }
    return odometry_reset(ctx);
}

int bshot_ransac_dev(bshot_ctx* ctx, const void* d_src4, const void* d_tgt4, const void* d_pairs, const void* d_n_pairs, size_t n_pairs_cap,
                     int max_iterations, float inlier_threshold, void* d_inlier_pairs_out, void* d_n_inliers_out, void* d_transform_out,
                     void* d_iterations_out) {
    CHECK_CTX(ctx);
    if (!d_n_pairs || !d_n_inliers_out || !d_transform_out || !d_iterations_out || (n_pairs_cap && (!d_src4 || !d_tgt4 || !d_pairs || !d_inlier_pairs_out))) {
        set_error("bshot_ransac_dev: null device pointer");
        return BSHOT_E_INVALID;
    }
    return ransac_run_dev(ctx, reinterpret_cast<const float4*>(d_src4), reinterpret_cast<const float4*>(d_tgt4), reinterpret_cast<const int*>(d_pairs), 2,
                          reinterpret_cast<const int*>(d_n_pairs), n_pairs_cap, max_iterations, (double)inlier_threshold, reinterpret_cast<int*>(d_inlier_pairs_out),
                          reinterpret_cast<int*>(d_n_inliers_out), reinterpret_cast<float*>(d_transform_out), reinterpret_cast<int*>(d_iterations_out), nullptr);
}

// ---- ISS keypoints + keypoint repeatability (kp_test evaluation, src/lidar_odometry.cpp:392-461) -----------------------
void bshot_iss_params_default(bshot_iss_params* p) {
    if (!p) return;
    p->salient_radius = 60.0f;
    p->non_max_radius = 40.0f;
    p->gamma_21 = 0.975;
    p->gamma_32 = 0.975;
    p->min_neighbors = 5;
}

int bshot_detect_iss(bshot_ctx* ctx, const bshot_iss_params* p, int* idx_out, float* kp_xyz_out, size_t cap, size_t* count_out,
                     double* eig_out) {
    CHECK_CTX(ctx);
    bshot_iss_params dp;
    if (!p) { bshot_iss_params_default(&dp); p = &dp; }
    if (!(p->salient_radius > 0.0f) || !(p->non_max_radius > 0.0f) || !std::isfinite(p->salient_radius) || !std::isfinite(p->non_max_radius) ||
        p->min_neighbors < 1 || !std::isfinite(p->gamma_21) || !std::isfinite(p->gamma_32)) {
        set_error("bshot_detect_iss: radii must be finite and > 0, min_neighbors >= 1, thresholds finite");
        return BSHOT_E_INVALID;
    }
    if (!ctx->have_cloud) { set_error("bshot_detect_iss: no cloud"); return BSHOT_E_STATE; }
    size_t count = 0;
    BSHOT_TRY(iss_detect(ctx, p->salient_radius, p->non_max_radius, p->gamma_21, p->gamma_32, p->min_neighbors, cap, eig_out != nullptr, &count));
    if (count_out) *count_out = count;
    const size_t m = std::min(count, cap);
    const int4* rec = ctx->iss.h_rec + 1;
    for (size_t i = 0; i < m; ++i) {
        if (idx_out) idx_out[i] = rec[i].x;
        if (kp_xyz_out) {
            memcpy(&kp_xyz_out[3 * i], &rec[i].y, sizeof(float));
            memcpy(&kp_xyz_out[3 * i + 1], &rec[i].z, sizeof(float));
            memcpy(&kp_xyz_out[3 * i + 2], &rec[i].w, sizeof(float));
        }
    }
    if (eig_out) {
        BSHOT_TRY(d2h(ctx, eig_out, ctx->iss.d_eig, sizeof(double) * 3 * ctx->n_points));
        BSHOT_TRY(sync(ctx));
    }
    if (count > cap) { set_error("bshot_detect_iss: %zu keypoints > capacity %zu", count, cap); return BSHOT_E_CAPACITY; }
    return BSHOT_OK;
}

int bshot_kp_repeatability(bshot_ctx* ctx, const float* a_xyz, size_t na, const float* a_pose3x4, const float* b_xyz, size_t nb,
                           const float* b_pose3x4, float radius, int* nn_idx_out, float* nn_dist_out, size_t* hits_out) {
    CHECK_CTX(ctx);
    if ((!a_xyz && na) || (!b_xyz && nb)) { set_error("bshot_kp_repeatability: null point set"); return BSHOT_E_INVALID; }
    if (!(radius > 0.0f) || !std::isfinite(radius)) { set_error("bshot_kp_repeatability: radius must be finite and > 0"); return BSHOT_E_INVALID; }
    if (na > 0x7FFFFFFull || nb > 0x7FFFFFFull) { set_error("bshot_kp_repeatability: too many points"); return BSHOT_E_CAPACITY; }
    return kp_repeatability(ctx, a_xyz, na, a_pose3x4, b_xyz, nb, b_pose3x4, radius, nn_idx_out, nn_dist_out, hits_out);
}

// ---- voxel-grid downsampling (bshot::calculate_voxel_grid_keypoints, pcl::VoxelGrid) ------------------------------------
int bshot_voxel_grid(bshot_ctx* ctx, const float* xyz, size_t n, size_t stride_bytes, float leaf_x, float leaf_y, float leaf_z,
                     float* xyz_out, size_t cap, size_t* count_out) {
    CHECK_CTX(ctx);
    if (!xyz && n) { set_error("bshot_voxel_grid: null cloud"); return BSHOT_E_INVALID; }
    if (stride_bytes != 12 && stride_bytes != 16) { set_error("bshot_voxel_grid: stride must be 12 or 16 bytes"); return BSHOT_E_INVALID; }
    const float leaf[3] = {leaf_x, leaf_y, leaf_z};
    float inv[3];
    for (int a = 0; a < 3; ++a) {
        inv[a] = 1.0f / leaf[a];  // PCL: inverse_leaf_size_ = Array4f::Ones () / leaf_size_
        if (!(leaf[a] > 0.0f) || !std::isfinite(leaf[a]) || !std::isfinite(inv[a])) {
            set_error("bshot_voxel_grid: leaf sizes must be finite and > 0 with a finite reciprocal");
            return BSHOT_E_INVALID;
        }
    }
    if (n > ctx->max_points) { set_error("bshot_voxel_grid: %zu points > capacity %zu", n, ctx->max_points); return BSHOT_E_CAPACITY; }
    size_t count = 0;
    BSHOT_TRY(voxel_grid(ctx, xyz, n, (int)(stride_bytes / 4), inv, cap, &count));
    if (count_out) *count_out = count;
    if (xyz_out) memcpy(xyz_out, ctx->vg.h_out + 4, sizeof(float) * 3 * std::min(count, cap));
    if (count > cap) { set_error("bshot_voxel_grid: %zu voxels > capacity %zu", count, cap); return BSHOT_E_CAPACITY; }
    return BSHOT_OK;
}

// ---- multi-rank exchange behind the C ABI (no Python / torch needed) -------------------------------------------
static void comm_free(bshot_ctx* c) {
    Comm& m = c->comm;
    for (int p = 0; p < 32; ++p)
        if (m.opened[p]) { cudaIpcCloseMemHandle(m.opened[p]); m.opened[p] = nullptr; }
    if (m.d_region) cudaFree(m.d_region);
    if (m.d_peer_gather) cudaFree(m.d_peer_gather);
    if (m.d_peer_rq) cudaFree(m.d_peer_rq);
    if (m.d_peer_flags) cudaFree(m.d_peer_flags);
    if (m.d_ticket) cudaFree(m.d_ticket);
    m = Comm();
}

int bshot_comm_create(bshot_ctx* ctx, int rank, int nranks, size_t max_queries) {
    CHECK_CTX(ctx);
    if (nranks < 1 || nranks > 32 || rank < 0 || rank >= nranks || max_queries == 0) { set_error("bshot_comm_create: bad arguments"); return BSHOT_E_INVALID; }
    if (max_queries > ctx->max_kp) { set_error("bshot_comm_create: max_queries %zu > max_keypoints %zu", max_queries, ctx->max_kp); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(sync(ctx));
    comm_free(ctx);
    BSHOT_TRY(hamming_preload_sharded());
    Comm& m = ctx->comm;
    m.rank = rank; m.nranks = nranks; m.max_q = max_queries;
    const size_t bytes = comm_region_bytes(m);
    BSHOT_CUDA_TRY(cudaMalloc((void**)&m.d_region, bytes));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&m.d_peer_gather, sizeof(void*) * 32));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&m.d_peer_rq, sizeof(void*) * 32));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&m.d_peer_flags, sizeof(void*) * 32));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&m.d_ticket, sizeof(unsigned) * 4));
    BSHOT_CUDA_TRY(cudaMemsetAsync(m.d_region, 0, bytes, ctx->stream));          // flags start at epoch 0
    BSHOT_CUDA_TRY(cudaMemsetAsync(m.d_ticket, 0, sizeof(unsigned) * 4, ctx->stream));
    BSHOT_CUDA_TRY(cudaMemsetAsync(ctx->d_pair_count + 3, 0, sizeof(int), ctx->stream));
    BSHOT_TRY(sync(ctx));
    if (nranks == 1) {
        void* none[1] = {nullptr};
        return comm_set_peers(ctx, none);
    }
    return BSHOT_OK;
}

int bshot_comm_destroy(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    BSHOT_TRY(sync(ctx));
    comm_free(ctx);
    return BSHOT_OK;
}

int bshot_comm_region(bshot_ctx* ctx, void** d_region_out, size_t* bytes_out) {
    CHECK_CTX(ctx);
    if (!ctx->comm.d_region) { set_error("bshot_comm_region: no communicator"); return BSHOT_E_STATE; }
    if (d_region_out) *d_region_out = ctx->comm.d_region;
    if (bytes_out) *bytes_out = comm_region_bytes(ctx->comm);
    return BSHOT_OK;
}

int bshot_comm_export(bshot_ctx* ctx, bshot_ipc_handle* handle_out) {
    CHECK_CTX(ctx);
    if (!ctx->comm.d_region || !handle_out) { set_error("bshot_comm_export: no communicator / null output"); return BSHOT_E_STATE; }
    static_assert(sizeof(cudaIpcMemHandle_t) <= sizeof(bshot_ipc_handle), "handle size");
    cudaIpcMemHandle_t h;
    BSHOT_CUDA_TRY(cudaIpcGetMemHandle(&h, ctx->comm.d_region));
    memset(handle_out, 0, sizeof(*handle_out));
    memcpy(handle_out, &h, sizeof(h));
    return BSHOT_OK;
}

int bshot_comm_import(bshot_ctx* ctx, const bshot_ipc_handle* handles) {
    CHECK_CTX(ctx);
    Comm& m = ctx->comm;
    if (!m.d_region || !handles) { set_error("bshot_comm_import: no communicator / null handles"); return BSHOT_E_STATE; }
    void* ptrs[32] = {nullptr};
    for (int p = 0; p < m.nranks; ++p) {
        if (p == m.rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, &handles[p], sizeof(h));
        BSHOT_CUDA_TRY(cudaIpcOpenMemHandle(&m.opened[p], h, cudaIpcMemLazyEnablePeerAccess));
        ptrs[p] = m.opened[p];
    }
    return comm_set_peers(ctx, ptrs);
}

int bshot_comm_import_ptrs(bshot_ctx* ctx, void* const* d_regions) {
    CHECK_CTX(ctx);
    if (!ctx->comm.d_region || !d_regions) { set_error("bshot_comm_import_ptrs: no communicator / null pointers"); return BSHOT_E_STATE; }
    return comm_set_peers(ctx, d_regions);
}

int bshot_comm_check(bshot_ctx* ctx) {
    CHECK_CTX(ctx);
    BSHOT_TRY(d2h(ctx, &ctx->h_scratch[16], ctx->d_pair_count + 3, sizeof(int)));
    BSHOT_TRY(sync(ctx));
    if (ctx->h_scratch[16] != 0) {
        set_error("sharded match: a rank did not arrive within the time limit (call #%u); the records of that call are incomplete", (unsigned)ctx->h_scratch[16]);
        return BSHOT_E_STATE;
    }
    return BSHOT_OK;
}

int bshot_match_map_sharded_dev(bshot_ctx* ctx, const void* d_q, size_t nq, uint64_t global_base, void* d_cand_out) {
    CHECK_CTX(ctx);
    if (!d_q || !d_cand_out) { set_error("bshot_match_map_sharded_dev: null device pointer"); return BSHOT_E_INVALID; }
    return hamming_match_sharded(ctx, d_q, nq, global_base, reinterpret_cast<bshot_cand*>(d_cand_out));
}

int bshot_match_map_sharded(bshot_ctx* ctx, const uint64_t* q, size_t nq, uint64_t global_base, bshot_cand* cand_out) {
    CHECK_CTX(ctx);
    if ((!q || !cand_out) && nq) { set_error("bshot_match_map_sharded: null buffer"); return BSHOT_E_INVALID; }
    if (nq > ctx->max_kp) { set_error("bshot_match_map_sharded: %zu queries > capacity %zu", nq, ctx->max_kp); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(h2d(ctx, ctx->d_q, q, nq * 48));
    BSHOT_TRY(hamming_match_sharded(ctx, ctx->d_q, nq, global_base, ctx->d_cand2));
    BSHOT_TRY(d2h(ctx, cand_out, ctx->d_cand2, sizeof(bshot_cand) * nq));
    return bshot_comm_check(ctx);
}

int bshot_match_map(bshot_ctx* ctx, const uint64_t* q, size_t nq, uint64_t global_base, bshot_cand* cand_out) {
    CHECK_CTX(ctx);
    if ((!q || !cand_out) && nq) { set_error("bshot_match_map: null buffer"); return BSHOT_E_INVALID; }
    if (nq > ctx->max_kp) { set_error("bshot_match_map: %zu queries > capacity %zu", nq, ctx->max_kp); return BSHOT_E_CAPACITY; }
    BSHOT_TRY(h2d(ctx, ctx->d_q, q, nq * 48));
    BSHOT_TRY(bshot_match_shard_dev(ctx, ctx->d_q, nq, global_base, 1, ctx->d_cand));
    BSHOT_TRY(d2h(ctx, cand_out, ctx->d_cand, sizeof(bshot_cand) * nq));
    return sync(ctx);
}

}  // extern "C"
