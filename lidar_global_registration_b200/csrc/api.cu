// api.cu -- the C-ABI of libb200match.so (see include/b200match.h): context, descriptor
// upload, the kNN driver (tensor-core candidates -> exact re-rank -> exact fallback) and the
// whole-matcher call.  Host-side C++ only; every kernel lives in its own translation unit.
//
// Reference seams replaced (paths relative to the reference root):
//   b200m_upload   pcl2cv<FeatureT>                      include/matching.h:553-560
//   b200m_knn      matchBF / matchFLANN / matchLocal(inf) include/matching.h:594-634, :562-592, :637-678
//   b200m_match    OneSided/LeftToRight(/Ratio)Matcher::match_impl + printDebugInfo's average
//                  include/matching.h:395-411, :428-453, :470-473; src/matching.cpp:3-19
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <thread>
#include <vector>

#include "internal.cuh"

static thread_local std::string g_create_err;
extern "C" {
static void stage_release(b200m_ctx *ctx);
}

cudaError_t DevBuf::reserve(size_t bytes) {
    if (bytes <= cap && p) return cudaSuccess;
    if (p) {
        cudaError_t e = cudaFree(p);
        p = nullptr;
        cap = 0;
        if (e != cudaSuccess) return e;
    }
    size_t want = bytes < 256 ? 256 : bytes;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) { p = nullptr; return e; }
    cap = want;
    return cudaSuccess;
}

void DevBuf::release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
}

int b200m_fail(b200m_ctx *ctx, const char *what, cudaError_t e, const char *file, int line) {
    std::string m = std::string(what) + ": " + cudaGetErrorString(e) + " (" + file + ":" + std::to_string(line) + ")";
    if (ctx) ctx->err = m; else g_create_err = m;
    return 1;
}

int b200m_fail_msg(b200m_ctx *ctx, const std::string &msg) {
    if (ctx) ctx->err = msg; else g_create_err = msg;
    return 1;
}

// ---- event-pool timing ----------------------------------------------------------------------
void b200m_resolve_events(b200m_ctx *ctx) {
    EventPool *pl = ctx->pool;
    if (!pl || pl->used == 0) return;
    cudaEventSynchronize(pl->ev[2 * (pl->used - 1) + 1]);
    for (int i = 0; i < pl->used; ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, pl->ev[2 * i], pl->ev[2 * i + 1]) == cudaSuccess) *pl->slot[i] += ms;
    }
    pl->used = 0;
}

StatTimer::StatTimer(b200m_ctx *c, double *s) : ctx(c) {
    if (!ctx->profiling) return;
    if (!ctx->pool) ctx->pool = new EventPool();
    EventPool *pl = ctx->pool;
    if (!pl->created) {
        for (int i = 0; i < 2 * EventPool::kPairs; ++i) cudaEventCreate(&pl->ev[i]);
        pl->created = true;
    }
    if (pl->used == EventPool::kPairs) b200m_resolve_events(ctx);
    pair = pl->used++;
    pl->slot[pair] = s;
    cudaEventRecord(pl->ev[2 * pair], ctx->stream);
}

void StatTimer::stop() {
    if (pair >= 0) cudaEventRecord(ctx->pool->ev[2 * pair + 1], ctx->stream);
}

#define REQUIRE_CTX()                                          \
    do {                                                       \
        if (!ctx) return b200m_fail_msg(nullptr, "null context"); \
        CK(cudaSetDevice(ctx->device));                        \
    } while (0)

extern "C" {

int b200m_version(void) { return 200; }

int b200m_create(b200m_ctx **out, int device) {
    b200m_ctx *ctx = nullptr;
    if (!out) return b200m_fail_msg(nullptr, "b200m_create: null output pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return b200m_fail_msg(nullptr, std::string("b200m_create: no CUDA device (there is no CPU fallback): ") +
                                           cudaGetErrorString(e));
    if (device < 0 || device >= n) return b200m_fail_msg(nullptr, "b200m_create: device index out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return b200m_fail_msg(nullptr, std::string("b200m_create: this library is built for sm_100a (B200) only; device is ") +
                                           prop.name + " (sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + ")");
    ctx = new b200m_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev[0])) != cudaSuccess || (e = cudaEventCreate(&ctx->ev[1])) != cudaSuccess) {
        b200m_fail(nullptr, "b200m_create", e, __FILE__, __LINE__);
        delete ctx;
        return 1;
    }
    ctx->stream = ctx->own_stream;
    if (const char *e = getenv("B200M_TC_CLUSTER")) {
        int c = atoi(e);
        if (c == 1 || c == 2 || c == 4) { ctx->tc_cluster = c; ctx->tc_pair = 0; }
    }
    if (const char *e = getenv("B200M_TC_DEBUG")) ctx->tc_debug = atoi(e);
    if (const char *e = getenv("B200M_TC_SPLITS")) ctx->tc_splits = atoi(e);
    if (const char *e = getenv("B200M_TC_LEAN")) ctx->tc_lean = atoi(e);
    if (const char *e = getenv("B200M_TC_SPLITN")) ctx->tc_splitn = atoi(e);
    if (const char *e = getenv("B200M_TC_ALT")) ctx->tc_alt = atoi(e);
    if (const char *e = getenv("B200M_TC_SWEEP_LAG")) ctx->tc_sweep_lag = atoi(e);
    if (const char *e = getenv("B200M_LOCAL_MIN_ROWS")) ctx->local_min_rows = atoi(e);
    if (const char *e = getenv("B200M_MASKED_MIN_PAIRS")) ctx->masked_min_pairs = atof(e);
    if (const char *e = getenv("B200M_TC_MODE")) {
        if (!strcmp(e, "mcast")) ctx->tc_pair = 0;
        if (!strcmp(e, "pair")) ctx->tc_pair = 1;
    }
    *out = ctx;
    return 0;
}

void b200m_destroy(b200m_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (int s = 0; s < 2; ++s) {
        Side &sd = ctx->side[s];
        sd.staging.release(); sd.f32.release(); sd.valid.release(); sd.stats.release();
        sd.op_query.release(); sd.op_train.release(); sd.norm16.release();
        ctx->ws_thr[s].release();
    }
    ctx->prep.mean.release(); ctx->prep.red.release();
    DevBuf *ws[] = {&ctx->ws_cand_idx, &ctx->ws_cand_cnt, &ctx->ws_flag_rows, &ctx->ws_counters, &ctx->ws_scan,
                    &ctx->ws_out, &ctx->ws_misc, &ctx->ws_fidx, &ctx->ws_fdist, &ctx->ws_fcnt, &ctx->ws_ridx,
                    &ctx->ws_rdist, &ctx->ws_rcnt, &ctx->ws_corr, &ctx->ws_totals, &ctx->ws_part_i, &ctx->ws_part_d,
                    &ctx->ws_done, &ctx->ws_cand_val, &ctx->ws_cand_thr, &ctx->ws_row_list, &ctx->ws_row_flags,
                    &ctx->ws_sel_ops, &ctx->ws_sel_norm, &ctx->ws_sweep_hint, &ctx->ws_batch};
    for (DevBuf *b : ws) b->release();
    tc_release(ctx);
    multiscale_release(ctx);
    cluster_release(ctx);
    wide_release(ctx);
    wide_batch_release(ctx);
    comm_release(ctx);
    local_release(ctx);
    stage_release(ctx);
    if (ctx->pool) {
        if (ctx->pool->created)
            for (int i = 0; i < 2 * EventPool::kPairs; ++i) cudaEventDestroy(ctx->pool->ev[i]);
        delete ctx->pool;
    }
    if (ctx->ev[0]) cudaEventDestroy(ctx->ev[0]);
    if (ctx->ev[1]) cudaEventDestroy(ctx->ev[1]);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

const char *b200m_last_error(const b200m_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int b200m_set_stream(b200m_ctx *ctx, void *cuda_stream) {
    REQUIRE_CTX();
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? (cudaStream_t) cuda_stream : ctx->own_stream;
    return 0;
}

int b200m_sync(b200m_ctx *ctx) {
    REQUIRE_CTX();
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int b200m_set_profiling(b200m_ctx *ctx, int on) {
    REQUIRE_CTX();
    ctx->profiling = on != 0;
    return 0;
}

int b200m_get_stats(b200m_ctx *ctx, b200m_stats *out) {
    REQUIRE_CTX();
    if (!out) return b200m_fail_msg(ctx, "b200m_get_stats: null output");
    CK(cudaStreamSynchronize(ctx->stream));
    b200m_resolve_events(ctx);
    if (ctx->totals_init) {
        unsigned long long h[2] = {0, 0};
        CK(cudaMemcpy(h, ctx->ws_totals.p, sizeof(h), cudaMemcpyDeviceToHost));
        ctx->stats.rows_flagged = (int64_t) h[0];
        ctx->stats.candidates = (int64_t) h[1];
    }
    *out = ctx->stats;
    return 0;
}

int b200m_reset_stats(b200m_ctx *ctx) {
    REQUIRE_CTX();
    b200m_resolve_events(ctx);
    ctx->stats = b200m_stats{};
    if (ctx->totals_init) CK(cudaMemsetAsync(ctx->ws_totals.p, 0, 64, ctx->stream));
    return 0;
}

// ---- uploads from pageable host memory ------------------------------------------------------------------
// The reference hands the matcher pcl::PointCloud buffers: ordinary (pageable) memory, which cudaMemcpyAsync moves through
// the driver's own single-threaded staging at ~11 GB/s (C3: 1.44 GB of descriptors = 130 ms of a 337 ms call).  Here the
// bytes go through four 16 MB pinned bounce buffers: a few host threads copy chunk c+1 into one while the DMA engine
// drains chunk c from another.
struct StagePool {
    static const int kBufs = 4;
    static const size_t kChunk = (size_t) 16 << 20;
    void *buf[kBufs] = {};
    cudaEvent_t free_ev[kBufs] = {};
    bool ready = false;
};

static void stage_release(b200m_ctx *ctx) {
    StagePool *sp = static_cast<StagePool *>(ctx->stage);
    if (!sp) return;
    for (int i = 0; i < StagePool::kBufs; ++i) {
        if (sp->buf[i]) cudaFreeHost(sp->buf[i]);
        if (sp->free_ev[i]) cudaEventDestroy(sp->free_ev[i]);
    }
    delete sp;
    ctx->stage = nullptr;
}

bool is_pageable(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

int staged_h2d(b200m_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (!ctx->stage) ctx->stage = new StagePool();
    StagePool *sp = static_cast<StagePool *>(ctx->stage);
    if (!sp->ready) {
        for (int i = 0; i < StagePool::kBufs; ++i) {
            CK(cudaHostAlloc(&sp->buf[i], StagePool::kChunk, cudaHostAllocDefault));
            CK(cudaEventCreateWithFlags(&sp->free_ev[i], cudaEventDisableTiming));
        }
        sp->ready = true;
    }
    unsigned hw = std::thread::hardware_concurrency();
    const int n_thr = hw >= 8 ? 4 : hw >= 4 ? 2 : 1;
    size_t off = 0;
    for (int c = 0; off < bytes; ++c) {
        const int b = c % StagePool::kBufs;
        const size_t len = bytes - off < StagePool::kChunk ? bytes - off : StagePool::kChunk;
        // the DMA out of this buffer has finished (also the one queued by the previous call: a batch stages many sets in a row)
        CK(cudaEventSynchronize(sp->free_ev[b]));
        const char *s = static_cast<const char *>(src) + off;
        char *d = static_cast<char *>(sp->buf[b]);
        const size_t part = (len / n_thr + 4095) & ~(size_t) 4095;
        std::vector<std::thread> th;
        for (int t = 1; t < n_thr; ++t) {
            const size_t lo = (size_t) t * part;
            if (lo >= len) break;
            const size_t n = lo + part < len ? part : len - lo;
            th.emplace_back([=] { memcpy(d + lo, s + lo, n); });
        }
        memcpy(d, s, part < len ? part : len);
        for (std::thread &t : th) t.join();
        CK(cudaMemcpyAsync(static_cast<char *>(dst) + off, d, len, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaEventRecord(sp->free_ev[b], ctx->stream));
        off += len;
    }
    return 0;
}

// ---- upload -----------------------------------------------------------------------------
int upload_common(b200m_ctx *ctx, int side, const float *device_aos, size_t n, size_t stride_bytes, int dim,
                         int64_t index_offset, const int32_t *seg_blk, const SetRef *sets) {
    Side &sd = ctx->side[side];
    sd.n = n;
    sd.n_pad = (n + B200M_TILE_N - 1) / B200M_TILE_N * B200M_TILE_N;
    sd.dim = dim;
    sd.dp = (dim + 3) / 4 * 4;
    sd.kp = (dim + B200M_AUG_COLS + 63) / 64 * 64;
    sd.index_offset = index_offset;
    sd.version++;
    ctx->prep.ready = false;
    if (n == 0) return 0;
    CK(sd.f32.reserve(sizeof(float) * n * (size_t) sd.dp));
    CK(sd.valid.reserve(n));
    CK(sd.stats.reserve(pack_stats_bytes(ctx->sm_count, sd.dp)));
    StatTimer t(ctx, &ctx->stats.ms_pack);
    CK(launch_pack_f32(device_aos, n, stride_bytes, dim, sd.dp, sd.f32.as<float>(), sd.valid.as<uint8_t>(),
                       sd.stats.as<float>(), ctx->sm_count, ctx->stream, seg_blk, sets));
    ctx->stats.launches += 1;
    t.stop();
    return 0;
}

int check_upload_args(b200m_ctx *ctx, int side, const float *base, size_t n, size_t stride_bytes, int dim) {
    if (side != 0 && side != 1) return b200m_fail_msg(ctx, "b200m_upload: side must be 0 (source) or 1 (target)");
    if (dim < 1 || dim > B200M_MAX_DIM) return b200m_fail_msg(ctx, "b200m_upload: dim out of range [1, 2048]");
    if (stride_bytes % 4 != 0 || stride_bytes < (size_t) dim * 4)
        return b200m_fail_msg(ctx, "b200m_upload: stride_bytes must be a multiple of 4 and >= 4*dim");
    if (n > 0 && !base) return b200m_fail_msg(ctx, "b200m_upload: null descriptor pointer");
    if (n >= (size_t) 1 << 31) return b200m_fail_msg(ctx, "b200m_upload: more than 2^31-1 rows (indices are int32, as pcl::index_t)");
    return 0;
}

int b200m_upload(b200m_ctx *ctx, int side, const float *host_base, size_t n, size_t stride_bytes, int dim,
                 int64_t index_offset) {
    REQUIRE_CTX();
    if (check_upload_args(ctx, side, host_base, n, stride_bytes, dim)) return 1;
    Side &sd = ctx->side[side];
    if (n) {
        // last row may be shorter than the stride (the caller owns only dim floats of it)
        size_t bytes = (n - 1) * stride_bytes + (size_t) dim * 4;
        CK(sd.staging.reserve(n * stride_bytes));
        if (bytes >= ((size_t) 32 << 20) && is_pageable(host_base)) {
            if (staged_h2d(ctx, sd.staging.p, host_base, bytes)) return 1;
        } else {
            CK(cudaMemcpyAsync(sd.staging.p, host_base, bytes, cudaMemcpyHostToDevice, ctx->stream));
        }
    }
    return upload_common(ctx, side, sd.staging.as<float>(), n, stride_bytes, dim, index_offset);
}

int b200m_upload_device(b200m_ctx *ctx, int side, const float *device_base, size_t n, size_t stride_bytes, int dim,
                        int64_t index_offset) {
    REQUIRE_CTX();
    if (check_upload_args(ctx, side, device_base, n, stride_bytes, dim)) return 1;
    return upload_common(ctx, side, device_base, n, stride_bytes, dim, index_offset);
}

// ---- kNN --------------------------------------------------------------------------------
__global__ void accumulate_counters_kernel(const int32_t *counters, unsigned long long *totals) {
    totals[0] += (unsigned long long) counters[0];
    totals[1] += *reinterpret_cast<const unsigned long long *>(counters + 2);
}

__global__ void fill_empty_kernel(size_t n_rows, int k, int32_t *idx, float *dist, int32_t *count) {
    size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_rows * (size_t) k) { idx[i] = -1; dist[i] = 0.f; }
    if (i < n_rows) count[i] = 0;
}

int check_params(b200m_ctx *ctx, const b200m_params *p) {
    if (!p) return b200m_fail_msg(ctx, "null params");
    if (p->k < 1 || p->k > B200M_MAX_K) return b200m_fail_msg(ctx, "params.k must be in [1, 32]");
    if (p->mode < B200M_MODE_KNN_ONLY || p->mode > B200M_MODE_CLUSTER) return b200m_fail_msg(ctx, "params.mode unknown");
    if (p->precision != B200M_PREC_TC_F16 && p->precision != B200M_PREC_F32_EXACT)
        return b200m_fail_msg(ctx, "params.precision unknown");
    if ((p->mode == B200M_MODE_RATIO || p->mode == B200M_MODE_RATIO_MUTUAL) && p->k < 2)
        return b200m_fail_msg(ctx, "ratio modes need k >= 2 (MATCHING_RATIO_K, reference include/common.h:51)");
    return 0;
}

// ---- row selection (masked kNN) ---------------------------------------------------------------------
// The mutual filter only ever looks at the reverse lists of target rows that some forward list names
// (LeftToRightMatcher::match_impl, reference include/matching.h:433-449: rev[j] is read for j in fwd[i] only), so
// the reverse pass can skip every other target row -- 30 % of them in the benchmark's data.
__global__ void mark_referenced_kernel(const int32_t *__restrict__ fidx, const int32_t *__restrict__ fcount, size_t n_rows,
                                       int k, long long index_offset, uint8_t *__restrict__ flags, size_t n_flags) {
    const size_t e = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_rows * (size_t) k) return;
    if ((int) (e % k) >= fcount[e / k]) return;
    const long long j = (long long) fidx[e] - index_offset;
    if (j >= 0 && (size_t) j < n_flags) flags[j] = 1;
}

// rows of [row_begin, row_begin + n_rows) that are flagged AND valid -> row_list (unordered; warp-aggregated append)
__global__ void select_rows_kernel(const uint8_t *__restrict__ flags, const uint8_t *__restrict__ valid, size_t row_begin,
                                   size_t n_rows, int32_t *__restrict__ row_list, int32_t *__restrict__ n_selected) {
    const size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    const bool take = i < n_rows && flags[row_begin + i] && valid[row_begin + i];
    const unsigned m = __ballot_sync(0xffffffffu, take);
    if (!m) return;
    const int lane = threadIdx.x & 31, leader = __ffs((int) m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(n_selected, __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (take) row_list[base + __popc(m & ((1u << lane) - 1u))] = (int32_t) (row_begin + i);
}

// compact copy of the selected rows' query-form operands and norms (zero rows behind the last one, up to n_pad)
__global__ void gather_query_rows_kernel(const int32_t *__restrict__ row_list, size_t n_sel, size_t n_pad, int kp,
                                         const uint4 *__restrict__ op_query, const float *__restrict__ norm16,
                                         uint4 *__restrict__ op_out, float *__restrict__ norm_out) {
    const int lane = threadIdx.x & 31;
    const size_t r = (size_t) blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= n_pad) return;
    const int per_row = kp / 8;   // uint4 = 8 halves
    if (r < n_sel) {
        const size_t src = (size_t) row_list[r];
        for (int c = lane; c < per_row; c += 32) op_out[r * per_row + c] = __ldg(op_query + src * per_row + c);
        if (lane == 0) norm_out[r] = norm16[src];
    } else {
        for (int c = lane; c < per_row; c += 32) op_out[r * per_row + c] = make_uint4(0u, 0u, 0u, 0u);
        if (lane == 0) norm_out[r] = 0.f;
    }
}

// kNN of query rows [row_begin, row_begin + n_rows) of `direction`; with d_flags, only of the flagged (and valid) rows --
// every other row gets an empty list.  Outputs are indexed by (row - row_begin).
int b200m_knn_rows(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin, size_t n_rows,
                   const uint8_t *d_flags, int32_t *d_idx, float *d_dist, int32_t *d_count, const SegTable *seg) {
    Side &q = ctx->side[direction], &t = ctx->side[1 - direction];
    const int k = p->k;
    cudaStream_t st = ctx->stream;
    ctx->stats.rows_total += (int64_t) n_rows;
    if (t.n == 0) {   // nothing to match against: every list is empty
        size_t ne = n_rows * (size_t) k;
        fill_empty_kernel<<<(unsigned) ((ne + 255) / 256), 256, 0, st>>>(n_rows, k, d_idx, d_dist, d_count);
        ctx->stats.launches += 1;
        CK(cudaGetLastError());
        return 0;
    }
    bool use_tc = p->precision == B200M_PREC_TC_F16 && tc_supported(ctx, q.dim, k);
    if (use_tc) {
        if (!ctx->prep.ready || ctx->prep.ver[0] != ctx->side[0].version || ctx->prep.ver[1] != ctx->side[1].version) {
            StatTimer tp(ctx, &ctx->stats.ms_prepare);
            CK(launch_tc_prepare(ctx));
            tp.stop();
        }
        // device prepare (batch plans): the candidate kernel routes data outside the window to the exact fallback itself
        use_tc = ctx->device_prepare || ctx->prep.usable;
    }
    // row selection: compact list of the rows to answer (the one host round trip of this path: the launch geometry
    // of the candidate kernel depends on how many there are)
    const int32_t *row_map = nullptr;
    size_t n_work = n_rows;
    if (d_flags) {
        size_t ne = n_rows * (size_t) k;
        fill_empty_kernel<<<(unsigned) ((ne + 255) / 256), 256, 0, st>>>(n_rows, k, d_idx, d_dist, d_count);
        CK(ctx->ws_row_list.reserve(sizeof(int32_t) * n_rows + 64));
        int32_t *d_nsel = ctx->ws_row_list.as<int32_t>();          // [0] = number selected, list from [16]
        int32_t *d_list = d_nsel + 16;
        CK(cudaMemsetAsync(d_nsel, 0, sizeof(int32_t), st));
        select_rows_kernel<<<(unsigned) ((n_rows + 255) / 256), 256, 0, st>>>(d_flags, q.valid.as<uint8_t>(), row_begin, n_rows,
                                                                              d_list, d_nsel);
        CK(cudaGetLastError());
        ctx->stats.launches += 2;
        int32_t n_sel = 0;
        CK(cudaMemcpyAsync(&n_sel, d_nsel, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (n_sel == 0) return 0;
        row_map = d_list;
        n_work = (size_t) n_sel;
    }
    if (!use_tc) {
        StatTimer tf(ctx, &ctx->stats.ms_fallback);
        CK(launch_exact_rows(q.f32.as<float>(), q.valid.as<uint8_t>(), q.dp, q.dim, t.f32.as<float>(),
                             t.valid.as<uint8_t>(), t.n, t.index_offset, row_begin, n_work, nullptr, nullptr, k, d_idx,
                             d_dist, d_count, 1 << 30, 0, nullptr, nullptr, nullptr, row_map, st, seg ? seg->range : nullptr));
        ctx->stats.launches += 1;
        tf.stop();
        return 0;
    }
    // 1. tensor-core candidate pass: per row a certified superset of the exact top-k
    int n_lists = 0, cap = 0, has_values = 0;
    ctx->stats.rows_answered += (int64_t) n_work;
    ctx->stats.pairs_scored += (int64_t) n_work * (int64_t) t.n;
    {
        const void *q_ops = nullptr;
        const float *q_norm = nullptr;
        size_t q_pad = 0;
        if (row_map) {   // the candidate kernel reads whole 128-row operand tiles: give it the selected rows back to back
            q_pad = (n_work + B200M_TILE_N - 1) / B200M_TILE_N * B200M_TILE_N;
            CK(ctx->ws_sel_ops.reserve(sizeof(__half) * q_pad * (size_t) q.kp));
            CK(ctx->ws_sel_norm.reserve(sizeof(float) * q_pad));
            StatTimer tg(ctx, &ctx->stats.ms_prepare);
            gather_query_rows_kernel<<<(unsigned) ((q_pad + 7) / 8), 256, 0, st>>>(
                row_map, n_work, q_pad, q.kp, q.op_query.as<uint4>(), q.norm16.as<float>(), ctx->ws_sel_ops.as<uint4>(),
                ctx->ws_sel_norm.as<float>());
            CK(cudaGetLastError());
            ctx->stats.launches += 1;
            tg.stop();
            q_ops = ctx->ws_sel_ops.p;
            q_norm = ctx->ws_sel_norm.as<float>();
        }
        StatTimer tc(ctx, &ctx->stats.ms_candidates);
        if (tc_candidates(ctx, direction, row_map ? 0 : row_begin, n_work, k, p->cand_cap, &n_lists, &cap, &has_values, nullptr, 0,
                          q_ops, q_norm, q_pad, seg))
            return 1;
        tc.stop();
    }
    // 2. exact FP32 re-rank of the candidates (bit-identical arithmetic to the reference)
    CK(ctx->ws_flag_rows.reserve(sizeof(int32_t) * n_work));
    CK(ctx->ws_counters.reserve(64));
    CK(cudaMemsetAsync(ctx->ws_counters.p, 0, 64, st));
    {
        StatTimer tr(ctx, &ctx->stats.ms_rerank);
        CK(launch_rerank(q.f32.as<float>(), q.valid.as<uint8_t>(), q.dp, q.dim, t.f32.as<float>(), t.valid.as<uint8_t>(),
                         t.n, t.index_offset, row_begin, n_work, k, ctx->ws_cand_idx.as<int32_t>(),
                         ctx->ws_cand_cnt.as<int32_t>(), n_lists, cap,
                         has_values ? ctx->ws_cand_val.as<float>() : nullptr,
                         has_values ? ctx->ws_cand_thr.as<float>() : nullptr, d_idx, d_dist, d_count,
                         ctx->ws_flag_rows.as<int32_t>(), ctx->ws_counters.as<int32_t>(), ctx->sm_count, row_map,
                         has_values == 2 ? 1 : 0, st));
        ctx->stats.launches += 1;
        tr.stop();
    }
    // 3. rows whose candidate list overflowed: exact row kernel (row list and its length stay on the device)
    {
        StatTimer tf(ctx, &ctx->stats.ms_fallback);
        size_t max_blocks = (size_t) ctx->sm_count * 8;
        const int split_blocks = ctx->sm_count * 2;
        const size_t part = exact_split_ws_entries(split_blocks, k);
        CK(ctx->ws_part_i.reserve(sizeof(int32_t) * part));
        CK(ctx->ws_part_d.reserve(sizeof(float) * part));
        CK(ctx->ws_done.reserve(sizeof(unsigned int) * (size_t) exact_split_max_rows()));
        if (!ctx->done_init) {   // the merging CTA leaves every counter at zero again
            CK(cudaMemsetAsync(ctx->ws_done.p, 0, sizeof(unsigned int) * (size_t) exact_split_max_rows(), st));
            ctx->done_init = true;
        }
        CK(launch_exact_rows(q.f32.as<float>(), q.valid.as<uint8_t>(), q.dp, q.dim, t.f32.as<float>(),
                             t.valid.as<uint8_t>(), t.n, t.index_offset, row_begin, n_work,
                             ctx->ws_flag_rows.as<int32_t>(), ctx->ws_counters.as<int32_t>(), k, d_idx, d_dist, d_count,
                             (int) (n_work < max_blocks ? n_work : max_blocks), split_blocks, ctx->ws_part_i.as<int32_t>(),
                             ctx->ws_part_d.as<float>(), ctx->ws_done.as<unsigned int>(), row_map, st,
                             seg ? seg->range : nullptr));
        ctx->stats.launches += 2;
        tf.stop();
    }
    if (ctx->profiling) {   // fold this call's counters into the running totals on the device (read at get_stats)
        CK(ctx->ws_totals.reserve(64));
        if (!ctx->totals_init) {
            CK(cudaMemsetAsync(ctx->ws_totals.p, 0, 64, st));
            ctx->totals_init = true;
        }
        accumulate_counters_kernel<<<1, 1, 0, st>>>(ctx->ws_counters.as<int32_t>(),
                                                    ctx->ws_totals.as<unsigned long long>());
        CK(cudaGetLastError());
    }
    return 0;
}

static int check_knn_args(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin, size_t *row_end,
                          const void *d_idx, const void *d_dist, const void *d_count) {
    if (check_params(ctx, p)) return 1;
    if (direction != 0 && direction != 1) return b200m_fail_msg(ctx, "b200m_knn: direction must be 0 or 1");
    Side &q = ctx->side[direction], &t = ctx->side[1 - direction];
    if (*row_end == 0) *row_end = q.n;
    if (row_begin > *row_end || *row_end > q.n) return b200m_fail_msg(ctx, "b200m_knn: query row range out of bounds");
    if (*row_end > row_begin && (!d_idx || !d_dist || !d_count)) return b200m_fail_msg(ctx, "b200m_knn: null output pointer");
    if (t.n && q.dim != t.dim) return b200m_fail_msg(ctx, "b200m_knn: source and target descriptor lengths differ");
    return 0;
}

int b200m_knn_device(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin, size_t row_end,
                     int32_t *d_idx, float *d_dist, int32_t *d_count) {
    REQUIRE_CTX();
    if (check_knn_args(ctx, p, direction, row_begin, &row_end, d_idx, d_dist, d_count)) return 1;
    if (row_end == row_begin) return 0;
    return b200m_knn_rows(ctx, p, direction, row_begin, row_end - row_begin, nullptr, d_idx, d_dist, d_count);
}

int b200m_knn_masked_device(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin, size_t row_end,
                            const uint8_t *d_row_flags, int32_t *d_idx, float *d_dist, int32_t *d_count) {
    REQUIRE_CTX();
    if (check_knn_args(ctx, p, direction, row_begin, &row_end, d_idx, d_dist, d_count)) return 1;
    if (row_end == row_begin) return 0;
    if (!d_row_flags) return b200m_fail_msg(ctx, "b200m_knn_masked: null row flags");
    return b200m_knn_rows(ctx, p, direction, row_begin, row_end - row_begin, d_row_flags, d_idx, d_dist, d_count);
}

int b200m_mark_referenced_device(b200m_ctx *ctx, int k, const int32_t *d_fidx, const int32_t *d_fcount, size_t n_rows,
                                 int64_t index_offset, uint8_t *d_flags, size_t n_flags) {
    REQUIRE_CTX();
    if (k < 1 || k > B200M_MAX_K) return b200m_fail_msg(ctx, "b200m_mark_referenced: k must be in [1, 32]");
    if (n_rows == 0) return 0;
    if (!d_fidx || !d_fcount || !d_flags) return b200m_fail_msg(ctx, "b200m_mark_referenced: null pointer");
    const size_t ne = n_rows * (size_t) k;
    mark_referenced_kernel<<<(unsigned) ((ne + 255) / 256), 256, 0, ctx->stream>>>(d_fidx, d_fcount, n_rows, k,
                                                                                   (long long) index_offset, d_flags, n_flags);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

int b200m_knn(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin, size_t row_end, int32_t *idx,
              float *dist, int32_t *count) {
    REQUIRE_CTX();
    if (direction != 0 && direction != 1) return b200m_fail_msg(ctx, "b200m_knn: direction must be 0 or 1");
    if (check_params(ctx, p)) return 1;
    Side &q = ctx->side[direction];
    size_t re = row_end == 0 ? q.n : row_end;
    if (row_begin > re || re > q.n) return b200m_fail_msg(ctx, "b200m_knn: query row range out of bounds");
    size_t n_rows = re - row_begin;
    if (n_rows == 0) return 0;
    if (!idx || !dist || !count) return b200m_fail_msg(ctx, "b200m_knn: null output pointer");
    const int k = p->k;
    CK(ctx->ws_fidx.reserve(sizeof(int32_t) * n_rows * k));
    CK(ctx->ws_fdist.reserve(sizeof(float) * n_rows * k));
    CK(ctx->ws_fcnt.reserve(sizeof(int32_t) * n_rows));
    if (b200m_knn_device(ctx, p, direction, row_begin, re, ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(),
                         ctx->ws_fcnt.as<int32_t>()))
        return 1;
    CK(cudaMemcpyAsync(idx, ctx->ws_fidx.p, sizeof(int32_t) * n_rows * k, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(dist, ctx->ws_fdist.p, sizeof(float) * n_rows * k, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(count, ctx->ws_fcnt.p, sizeof(int32_t) * n_rows, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ---- matchLocal with a finite radius ------------------------------------------------------------------
int b200m_knn_local_device(b200m_ctx *ctx, const b200m_params *p, int direction, const float *d_query_xyz,
                           const float *d_train_xyz, size_t xyz_stride_bytes, float radius, int32_t *d_idx, float *d_dist,
                           int32_t *d_count) {
    REQUIRE_CTX();
    if (check_params(ctx, p)) return 1;
    if (direction != 0 && direction != 1) return b200m_fail_msg(ctx, "b200m_knn_local: direction must be 0 or 1");
    if (xyz_stride_bytes % 4 != 0 || xyz_stride_bytes < 12) return b200m_fail_msg(ctx, "b200m_knn_local: xyz stride must be a multiple of 4 and >= 12 bytes");
    Side &q = ctx->side[direction], &t = ctx->side[1 - direction];
    if (q.n == 0) return 0;
    if (!d_idx || !d_dist || !d_count) return b200m_fail_msg(ctx, "b200m_knn_local: null output pointer");
    if (t.n && q.dim != t.dim) return b200m_fail_msg(ctx, "b200m_knn_local: source and target descriptor lengths differ");
    ctx->stats.rows_total += (int64_t) q.n;
    if (t.n == 0) {
        size_t ne = q.n * (size_t) p->k;
        fill_empty_kernel<<<(unsigned) ((ne + 255) / 256), 256, 0, ctx->stream>>>(q.n, p->k, d_idx, d_dist, d_count);
        ctx->stats.launches += 1;
        CK(cudaGetLastError());
        return 0;
    }
    if (!d_query_xyz || !d_train_xyz) return b200m_fail_msg(ctx, "b200m_knn_local: null keypoint coordinates");
    StatTimer tf(ctx, &ctx->stats.ms_fallback);
    {   // a radius that is small against the cloud: cell list of the train keypoints (local.cu)
        const int rc = launch_local_cells(ctx, direction, d_query_xyz, d_train_xyz, xyz_stride_bytes, radius, p->k, d_idx, d_dist, d_count);
        if (rc == 1) return 1;
        if (rc == 0) {
            tf.stop();
            return 0;
        }
    }
    CK(launch_local_rows(q.f32.as<float>(), q.valid.as<uint8_t>(), q.dp, t.f32.as<float>(), t.valid.as<uint8_t>(), t.n,
                         t.index_offset, q.n, d_query_xyz, d_train_xyz, xyz_stride_bytes, radius, p->k, d_idx, d_dist, d_count,
                         1 << 30, ctx->stream));
    ctx->stats.launches += 1;
    tf.stop();
    return 0;
}

int b200m_knn_local(b200m_ctx *ctx, const b200m_params *p, int direction, const float *query_xyz, const float *train_xyz,
                    size_t xyz_stride_bytes, float radius, int32_t *idx, float *dist, int32_t *count) {
    REQUIRE_CTX();
    if (check_params(ctx, p)) return 1;
    if (direction != 0 && direction != 1) return b200m_fail_msg(ctx, "b200m_knn_local: direction must be 0 or 1");
    if (xyz_stride_bytes % 4 != 0 || xyz_stride_bytes < 12) return b200m_fail_msg(ctx, "b200m_knn_local: xyz stride must be a multiple of 4 and >= 12 bytes");
    Side &q = ctx->side[direction], &t = ctx->side[1 - direction];
    const size_t nq = q.n, nt = t.n;
    if (nq == 0) return 0;
    if (!idx || !dist || !count) return b200m_fail_msg(ctx, "b200m_knn_local: null output pointer");
    if (!query_xyz || (nt && !train_xyz)) return b200m_fail_msg(ctx, "b200m_knn_local: null keypoint coordinates");
    const int k = p->k;
    CK(ctx->ws_fidx.reserve(sizeof(int32_t) * nq * k));
    CK(ctx->ws_fdist.reserve(sizeof(float) * nq * k));
    CK(ctx->ws_fcnt.reserve(sizeof(int32_t) * nq));
    CK(ctx->ws_thr[0].reserve(nq * xyz_stride_bytes + 16));
    CK(ctx->ws_thr[1].reserve(nt * xyz_stride_bytes + 16));
    CK(cudaMemcpyAsync(ctx->ws_thr[0].p, query_xyz, (nq - 1) * xyz_stride_bytes + 12, cudaMemcpyHostToDevice, ctx->stream));
    if (nt) CK(cudaMemcpyAsync(ctx->ws_thr[1].p, train_xyz, (nt - 1) * xyz_stride_bytes + 12, cudaMemcpyHostToDevice, ctx->stream));
    if (b200m_knn_local_device(ctx, p, direction, ctx->ws_thr[0].as<float>(), ctx->ws_thr[1].as<float>(), xyz_stride_bytes, radius,
                               ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>()))
        return 1;
    CK(cudaMemcpyAsync(idx, ctx->ws_fidx.p, sizeof(int32_t) * nq * k, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(dist, ctx->ws_fdist.p, sizeof(float) * nq * k, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(count, ctx->ws_fcnt.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ---- filters ----------------------------------------------------------------------------
int b200m_filter_device(b200m_ctx *ctx, const b200m_params *p, size_t row_begin, size_t row_end,
                        const int32_t *d_fidx, const float *d_fdist, const int32_t *d_fcount,
                        const int32_t *d_ridx, const float *d_rdist, const int32_t *d_rcount, size_t n_rev_rows,
                        const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                        unsigned long long *d_n_out, float *d_avg) {
    REQUIRE_CTX();
    if (check_params(ctx, p)) return 1;
    if (p->mode == B200M_MODE_KNN_ONLY) return b200m_fail_msg(ctx, "b200m_filter: mode KNN_ONLY has no filter");
    if (p->mode == B200M_MODE_CLUSTER) return b200m_fail_msg(ctx, "b200m_filter: the cluster filter needs keypoint coordinates, use b200m_cluster_filter_device");
    if (row_end < row_begin) return b200m_fail_msg(ctx, "b200m_filter: bad row range");
    const size_t n_rows = row_end - row_begin;
    const bool mutual = p->mode == B200M_MODE_MUTUAL || p->mode == B200M_MODE_RATIO_MUTUAL;
    if (mutual && n_rev_rows && (!d_ridx || !d_rdist || !d_rcount))
        return b200m_fail_msg(ctx, "b200m_filter: mutual modes need the reverse table");
    if (!d_n_out || (n_rows && (!d_fidx || !d_fdist || !d_fcount)) || (cap && !d_out))
        return b200m_fail_msg(ctx, "b200m_filter: null pointer");
    size_t ws = filter_scan_ws_bytes(n_rows, p->k);
    CK(ctx->ws_scan.reserve(ws));
    int launches = 0;
    StatTimer t(ctx, &ctx->stats.ms_filter);
    CK(launch_filter(p->mode, p->k, p->ratio_thr, p->distance_thr, row_begin, n_rows, d_fidx, d_fdist, d_fcount, d_ridx,
                     d_rdist, d_rcount, n_rev_rows, d_thr_src, d_thr_tgt, ctx->side[0].index_offset, ctx->side[1].index_offset, d_out, cap,
                     d_n_out,
                     d_avg, ctx->ws_scan.p, ctx->ws_scan.cap, ctx->stream, &launches));
    ctx->stats.launches += launches;
    t.stop();
    return 0;
}

int b200m_merge_device(b200m_ctx *ctx, int k, int n_lists, size_t nq, const int32_t *d_idx_in, const float *d_dist_in,
                       const int32_t *d_count_in, int32_t *d_idx, float *d_dist, int32_t *d_count) {
    REQUIRE_CTX();
    if (k < 1 || k > B200M_MAX_K || n_lists < 1 || n_lists > 8)
        return b200m_fail_msg(ctx, "b200m_merge: k in [1,32], n_lists in [1,8]");
    CK(launch_merge(k, n_lists, nq, d_idx_in, d_dist_in, d_count_in, d_idx, d_dist, d_count, ctx->stream));
    ctx->stats.launches += nq ? 1 : 0;
    return 0;
}

int b200m_match(b200m_ctx *ctx, const b200m_params *p, const float *thr_src, const float *thr_tgt, b200m_corr *out,
                size_t cap, size_t *n_out, float *avg_first_dist) {
    REQUIRE_CTX();
    if (check_params(ctx, p)) return 1;
    if (p->mode == B200M_MODE_KNN_ONLY) return b200m_fail_msg(ctx, "b200m_match: use b200m_knn for raw k-lists");
    if (p->mode == B200M_MODE_CLUSTER) return b200m_fail_msg(ctx, "b200m_match: the cluster filter needs keypoint coordinates, use b200m_match_cluster");
    if (!n_out) return b200m_fail_msg(ctx, "b200m_match: null n_out");
    *n_out = 0;
    Side &src = ctx->side[0], &tgt = ctx->side[1];
    if ((thr_src == nullptr) != (thr_tgt == nullptr))
        return b200m_fail_msg(ctx, "b200m_match: give both threshold arrays or neither");
    const int k = p->k;
    const bool mutual = p->mode == B200M_MODE_MUTUAL || p->mode == B200M_MODE_RATIO_MUTUAL;
    const size_t nq = src.n, nt = tgt.n;
    cudaStream_t st = ctx->stream;
    CK(ctx->ws_misc.reserve(64));
    float *d_avg = ctx->ws_misc.as<float>();
    unsigned long long *d_n = reinterpret_cast<unsigned long long *>(ctx->ws_misc.as<char>() + 16);
    if (nq == 0) {
        if (avg_first_dist) *avg_first_dist = 3.402823466e+38F;   // FLT_MAX, reference include/matching.h:41
        return 0;
    }
    CK(ctx->ws_fidx.reserve(sizeof(int32_t) * nq * k));
    CK(ctx->ws_fdist.reserve(sizeof(float) * nq * k));
    CK(ctx->ws_fcnt.reserve(sizeof(int32_t) * nq));
    if (b200m_knn_device(ctx, p, 0, 0, nq, ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>()))
        return 1;
    if (mutual && nt) {
        CK(ctx->ws_ridx.reserve(sizeof(int32_t) * nt * k));
        CK(ctx->ws_rdist.reserve(sizeof(float) * nt * k));
        CK(ctx->ws_rcnt.reserve(sizeof(int32_t) * nt));
        // reverse lists are only ever read for target rows that a forward list names: skip the rest when the pass is big
        // enough to pay for the extra host round trip (row selection)
        const uint8_t *d_flags = nullptr;
        if ((double) nq * (double) nt >= ctx->masked_min_pairs) {
            CK(ctx->ws_row_flags.reserve(nt));
            CK(cudaMemsetAsync(ctx->ws_row_flags.p, 0, nt, st));
            if (b200m_mark_referenced_device(ctx, k, ctx->ws_fidx.as<int32_t>(), ctx->ws_fcnt.as<int32_t>(), nq, tgt.index_offset,
                                             ctx->ws_row_flags.as<uint8_t>(), nt))
                return 1;
            d_flags = ctx->ws_row_flags.as<uint8_t>();
        }
        if (b200m_knn_rows(ctx, p, 1, 0, nt, d_flags, ctx->ws_ridx.as<int32_t>(), ctx->ws_rdist.as<float>(), ctx->ws_rcnt.as<int32_t>()))
            return 1;
    }
    const float *d_thr_s = nullptr, *d_thr_t = nullptr;
    if (thr_src && nt) {
        CK(ctx->ws_thr[0].reserve(sizeof(float) * nq));
        CK(ctx->ws_thr[1].reserve(sizeof(float) * nt));
        CK(cudaMemcpyAsync(ctx->ws_thr[0].p, thr_src, sizeof(float) * nq, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->ws_thr[1].p, thr_tgt, sizeof(float) * nt, cudaMemcpyHostToDevice, st));
        d_thr_s = ctx->ws_thr[0].as<float>();
        d_thr_t = ctx->ws_thr[1].as<float>();
    }
    const size_t kk = (p->mode == B200M_MODE_MUTUAL) ? (size_t) k : 1;
    const size_t max_out = nq * kk;
    CK(ctx->ws_corr.reserve(sizeof(b200m_corr) * max_out));
    if (b200m_filter_device(ctx, p, 0, nq, ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>(),
                            ctx->ws_ridx.as<int32_t>(), ctx->ws_rdist.as<float>(), ctx->ws_rcnt.as<int32_t>(),
                            mutual ? nt : 0, d_thr_s, d_thr_t, ctx->ws_corr.as<b200m_corr>(), max_out, d_n,
                            avg_first_dist ? d_avg : nullptr))
        return 1;
    struct { float avg; float pad[3]; unsigned long long n; } h;
    CK(cudaMemcpyAsync(&h, ctx->ws_misc.p, sizeof(h), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (avg_first_dist) *avg_first_dist = h.avg;
    *n_out = (size_t) h.n;
    if (h.n > cap) return b200m_fail_msg(ctx, "b200m_match: output capacity too small (" + std::to_string(h.n) + " correspondences)");
    if (h.n) {
        if (!out) return b200m_fail_msg(ctx, "b200m_match: null output buffer");
        CK(cudaMemcpyAsync(out, ctx->ws_corr.p, sizeof(b200m_corr) * h.n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return 0;
}

// ---- test hooks -------------------------------------------------------------------------
int b200m_debug_operands(b200m_ctx *ctx, int side, int as_query, uint16_t *host_out, size_t out_halves, float *norm16,
                         float *scale, int32_t *kp, int64_t *n_pad) {
    REQUIRE_CTX();
    if (side != 0 && side != 1) return b200m_fail_msg(ctx, "debug_operands: bad side");
    if (!ctx->side[0].n || !ctx->side[1].n) return b200m_fail_msg(ctx, "debug_operands: upload both sides first");
    if (!tc_supported(ctx, ctx->side[side].dim, 1)) return b200m_fail_msg(ctx, "debug_operands: dim not supported by the tensor-core pass");
    if (!ctx->prep.ready || ctx->prep.ver[0] != ctx->side[0].version || ctx->prep.ver[1] != ctx->side[1].version)
        CK(launch_tc_prepare(ctx));
    Side &sd = ctx->side[side];
    size_t halves = sd.n_pad * (size_t) sd.kp;
    if (kp) *kp = sd.kp;
    if (n_pad) *n_pad = (int64_t) sd.n_pad;
    if (scale) *scale = ctx->prep.scale;
    if (host_out) {
        if (out_halves < halves) return b200m_fail_msg(ctx, "debug_operands: output buffer too small");
        CK(cudaMemcpyAsync(host_out, as_query ? sd.op_query.p : sd.op_train.p, halves * 2, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (norm16) CK(cudaMemcpyAsync(norm16, sd.norm16.p, sizeof(float) * sd.n_pad, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int b200m_debug_tc_tile(b200m_ctx *ctx, int direction, size_t q_row0, size_t t_tile, float *host_out) {
    REQUIRE_CTX();
    if (direction != 0 && direction != 1) return b200m_fail_msg(ctx, "debug_tc_tile: bad direction");
    Side &q = ctx->side[direction], &t = ctx->side[1 - direction];
    if (!q.n || !t.n || !host_out) return b200m_fail_msg(ctx, "debug_tc_tile: upload both sides first");
    if (!tc_supported(ctx, q.dim, 1)) return b200m_fail_msg(ctx, "debug_tc_tile: dim not supported by the tensor-core pass");
    if (q_row0 >= q.n || t_tile * B200M_TILE_N >= t.n_pad) return b200m_fail_msg(ctx, "debug_tc_tile: tile out of range");
    if (!ctx->prep.ready || ctx->prep.ver[0] != ctx->side[0].version || ctx->prep.ver[1] != ctx->side[1].version)
        CK(launch_tc_prepare(ctx));
    CK(ctx->ws_out.reserve(sizeof(float) * 2 * B200M_TILE_M * B200M_TILE_N));   // pair mode dumps two query tiles
    CK(cudaMemsetAsync(ctx->ws_out.p, 0xff, sizeof(float) * 2 * B200M_TILE_M * B200M_TILE_N, ctx->stream));
    int n_lists = 0, cap = 0, has_values = 0;
    size_t n_rows = q.n - q_row0 < (size_t) B200M_TILE_M ? q.n - q_row0 : (size_t) B200M_TILE_M;
    if (tc_candidates(ctx, direction, q_row0, n_rows, 1, 0, &n_lists, &cap, &has_values, ctx->ws_out.as<float>(), t_tile)) return 1;
    CK(cudaMemcpyAsync(host_out, ctx->ws_out.p, sizeof(float) * B200M_TILE_M * B200M_TILE_N, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

}  // extern "C"
