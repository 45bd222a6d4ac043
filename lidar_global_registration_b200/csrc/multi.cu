// multi.cu -- multi-GPU partitioning of the matcher INSIDE the library (SURVEY 8e; north star item 5): source queries
// sharded / target replicated with ONE exchange step (the reverse table of the mutual test), or the target sharded with a
// per-query top-k merge -- NCCL over NVLink, queued on each rank's stream next to the kernels.
//
// Two ways to form the ranks, one code path underneath:
//   * b200m_comm_attach      one process per GPU (torchrun, MPI, ...): every process attaches a communicator to its own
//                            context (ncclCommInitRank with an id from b200m_comm_unique_id) and calls the *_sharded entry
//                            points collectively;
//   * b200m_create_multi     ONE process -- the reference's shape: FeatureBasedMatcher::match() is a single call in a single
//                            address space (src/correspondence_search.cpp:14-15, include/matching.h:148-161) -- a group of
//                            contexts, one per device, each driven by its own host thread inside the library
//                            (ncclCommInitAll); b200m_group_upload / _match / _knn take and return whole host arrays.
//
// Row partition: rank r owns rows [r*R, min(n, (r+1)*R)) with R = ceil(n / ranks), so that the all-gathered tables are
// directly the row-major tables of ALL rows (slot r starts at row r*R) and every collective is an in-place
// ncclAllGather of equal counts -- no packing kernels, no copies.  NCCL is bound at run time (dlopen of libnccl.so.2: the
// copy torch already loaded when the library runs inside a torch process, the system one otherwise), so single-GPU users
// need no NCCL at all.
#include <dlfcn.h>
#include <nccl.h>
#include <float.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "internal.cuh"

namespace {

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    std::string error;
};

NcclApi *nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names) {
            api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) {
            api.error = std::string("NCCL is not available (dlopen libnccl.so.2: ") + dlerror() + ")";
            return;
        }
        auto sym = [&](const char *name) {
            void *p = dlsym(api.handle, name);
            if (!p && api.error.empty()) api.error = std::string("libnccl lacks ") + name;
            return p;
        };
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
        api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
        api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
        api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
        api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
        api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    });
    return &api;
}

struct Comm {
    ncclComm_t comm = nullptr;
    int rank = 0, n_ranks = 1;
    DevBuf favg_d, favg_c;   // gathered first-NN distances / counts (the average over ALL source rows)
};

#define NCK(expr)                                                                                        \
    do {                                                                                                 \
        ncclResult_t _r = (expr);                                                                        \
        if (_r != ncclSuccess)                                                                           \
            return b200m_fail_msg(ctx, std::string(#expr) + ": " + nccl_api()->GetErrorString(_r));      \
    } while (0)

Comm *comm_of(b200m_ctx *ctx) { return static_cast<Comm *>(ctx->comm); }

inline size_t rows_per_rank(size_t n, int ranks) { return (n + (size_t) ranks - 1) / (size_t) ranks; }
inline void rank_rows(size_t n, int ranks, int rank, size_t *lo, size_t *hi) {
    const size_t R = rows_per_rank(n, ranks);
    *lo = (size_t) rank * R < n ? (size_t) rank * R : n;
    *hi = *lo + R < n ? *lo + R : n;
}

__global__ void first_entries_kernel(const float *__restrict__ fdist, const int32_t *__restrict__ fcount, size_t n_rows, int k,
                                     float *__restrict__ d0, int32_t *__restrict__ c0) {
    const size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    d0[i] = fdist[i * k];
    c0[i] = fcount[i] > 0 ? 1 : 0;
}

// ---- the per-rank bodies (collective: every rank of the communicator runs them with the same arguments) ------------------

// Query-sharded matcher call (SURVEY 8e): forward kNN of this rank's source rows, reverse kNN of this rank's target rows
// (only the rows a forward list of ANY rank names, when the problem is big enough), all-gather of the reverse table, filter
// of this rank's rows.  Records -> d_out (this rank's slice, ascending index_query), count -> d_n_out, average -> d_avg.
int match_sharded_core(b200m_ctx *ctx, const b200m_params *p, const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out,
                       size_t cap, unsigned long long *d_n_out, float *d_avg) {
    Comm *cm = comm_of(ctx);
    NcclApi *nc = nccl_api();
    const int W = cm->n_ranks, r = cm->rank, k = p->k;
    Side &src = ctx->side[0], &tgt = ctx->side[1];
    const size_t nq = src.n, nt = tgt.n;
    const size_t Rq = rows_per_rank(nq, W), Rt = rows_per_rank(nt, W);
    size_t q0, q1, t0, t1;
    rank_rows(nq, W, r, &q0, &q1);
    rank_rows(nt, W, r, &t0, &t1);
    cudaStream_t st = ctx->stream;
    const bool mutual = p->mode == B200M_MODE_MUTUAL || p->mode == B200M_MODE_RATIO_MUTUAL;
    b200m_params pk = *p;
    pk.mode = B200M_MODE_KNN_ONLY;
    CK(ctx->ws_fidx.reserve(sizeof(int32_t) * (Rq * k + 1)));
    CK(ctx->ws_fdist.reserve(sizeof(float) * (Rq * k + 1)));
    CK(ctx->ws_fcnt.reserve(sizeof(int32_t) * (Rq + 1)));
    int32_t *fidx = ctx->ws_fidx.as<int32_t>(), *fcnt = ctx->ws_fcnt.as<int32_t>();
    float *fdist = ctx->ws_fdist.as<float>();
    if (q1 > q0 && b200m_knn_rows(ctx, &pk, 0, q0, q1 - q0, nullptr, fidx, fdist, fcnt)) return 1;
    int32_t *ridx = nullptr, *rcnt = nullptr;
    float *rdist = nullptr;
    if (mutual && nt) {
        CK(ctx->ws_ridx.reserve(sizeof(int32_t) * Rt * W * k));
        CK(ctx->ws_rdist.reserve(sizeof(float) * Rt * W * k));
        CK(ctx->ws_rcnt.reserve(sizeof(int32_t) * Rt * W));
        ridx = ctx->ws_ridx.as<int32_t>();
        rdist = ctx->ws_rdist.as<float>();
        rcnt = ctx->ws_rcnt.as<int32_t>();
        const uint8_t *d_flags = nullptr;
        if ((double) nq * (double) nt >= ctx->masked_min_pairs) {
            // the mutual test reads rev[j] only for targets j some forward list names: every rank marks the ones its own
            // source rows name, the flags are max-reduced (nt bytes), the reverse pass answers the flagged rows only
            CK(ctx->ws_row_flags.reserve(nt));
            CK(cudaMemsetAsync(ctx->ws_row_flags.p, 0, nt, st));
            if (q1 > q0 && b200m_mark_referenced_device(ctx, k, fidx, fcnt, q1 - q0, tgt.index_offset, ctx->ws_row_flags.as<uint8_t>(), nt))
                return 1;
            NCK(nc->AllReduce(ctx->ws_row_flags.p, ctx->ws_row_flags.p, nt, ncclUint8, ncclMax, cm->comm, st));
            d_flags = ctx->ws_row_flags.as<uint8_t>();
        }
        int32_t *my_idx = ridx + (size_t) r * Rt * k, *my_cnt = rcnt + (size_t) r * Rt;
        float *my_dist = rdist + (size_t) r * Rt * k;
        if (t1 > t0 && b200m_knn_rows(ctx, &pk, 1, t0, t1 - t0, d_flags, my_idx, my_dist, my_cnt)) return 1;
        // the path's one exchange step: three in-place all-gathers fused into one NCCL group (one launch)
        NCK(nc->GroupStart());
        NCK(nc->AllGather(my_idx, ridx, Rt * k, ncclInt32, cm->comm, st));
        NCK(nc->AllGather(my_dist, rdist, Rt * k, ncclFloat32, cm->comm, st));
        NCK(nc->AllGather(my_cnt, rcnt, Rt, ncclInt32, cm->comm, st));
        NCK(nc->GroupEnd());
    }
    if (d_avg) {
        // printDebugInfo's average runs over ALL source rows in order (sequential FP32 sum, src/matching.cpp:6-11): gather
        // the first-NN distances, then the same kernel as the single-GPU call
        CK(cm->favg_d.reserve(sizeof(float) * Rq * W + 16));
        CK(cm->favg_c.reserve(sizeof(int32_t) * Rq * W + 16));
        float *gd = cm->favg_d.as<float>();
        int32_t *gc = cm->favg_c.as<int32_t>();
        if (q1 > q0)
            first_entries_kernel<<<(unsigned) ((q1 - q0 + 255) / 256), 256, 0, st>>>(fdist, fcnt, q1 - q0, k, gd + (size_t) r * Rq,
                                                                                   gc + (size_t) r * Rq);
        CK(cudaGetLastError());
        NCK(nc->GroupStart());
        NCK(nc->AllGather(gd + (size_t) r * Rq, gd, Rq, ncclFloat32, cm->comm, st));
        NCK(nc->AllGather(gc + (size_t) r * Rq, gc, Rq, ncclInt32, cm->comm, st));
        NCK(nc->GroupEnd());
        if (nq) CK(launch_average(gd, gc, nq, 1, d_avg, st));
        ctx->stats.launches += 2;
    }
    b200m_params pf = *p;
    if (b200m_filter_device(ctx, &pf, q0, q1, fidx, fdist, fcnt, ridx, rdist, rcnt, mutual ? nt : 0, d_thr_src, d_thr_tgt, d_out, cap,
                            d_n_out, nullptr))
        return 1;
    return 0;
}

// Target-sharded kNN (SURVEY 8e, BASELINE configs[4]): side 1 of every rank holds ITS shard of the target set (uploaded
// with index_offset = first global row of the shard), side 0 all queries.  Exact local top-k with global indices ->
// all-gather -> merge kernel (canonical tie rule); every rank ends up with the full result.
int knn_target_sharded_core(b200m_ctx *ctx, const b200m_params *p, int32_t *d_idx, float *d_dist, int32_t *d_count) {
    Comm *cm = comm_of(ctx);
    NcclApi *nc = nccl_api();
    const int W = cm->n_ranks, r = cm->rank, k = p->k;
    const size_t nq = ctx->side[0].n;
    if (nq == 0) return 0;
    cudaStream_t st = ctx->stream;
    b200m_params pk = *p;
    pk.mode = B200M_MODE_KNN_ONLY;
    CK(ctx->ws_ridx.reserve(sizeof(int32_t) * nq * W * k));
    CK(ctx->ws_rdist.reserve(sizeof(float) * nq * W * k));
    CK(ctx->ws_rcnt.reserve(sizeof(int32_t) * nq * W));
    int32_t *gi = ctx->ws_ridx.as<int32_t>(), *gc = ctx->ws_rcnt.as<int32_t>();
    float *gd = ctx->ws_rdist.as<float>();
    if (b200m_knn_rows(ctx, &pk, 0, 0, nq, nullptr, gi + (size_t) r * nq * k, gd + (size_t) r * nq * k, gc + (size_t) r * nq)) return 1;
    NCK(nc->GroupStart());
    NCK(nc->AllGather(gi + (size_t) r * nq * k, gi, nq * k, ncclInt32, cm->comm, st));
    NCK(nc->AllGather(gd + (size_t) r * nq * k, gd, nq * k, ncclFloat32, cm->comm, st));
    NCK(nc->AllGather(gc + (size_t) r * nq, gc, nq, ncclInt32, cm->comm, st));
    NCK(nc->GroupEnd());
    return b200m_merge_device(ctx, k, W, nq, gi, gd, gc, d_idx, d_dist, d_count);
}

// Replicate a HOST descriptor set on every rank: rank r copies only its 1/ranks slice over PCIe, the slices are
// all-gathered over NVLink (ranks pulling the whole set through the host's memory system at once is what limits a
// replicated upload), then the pack kernel runs on the full set.
int upload_replicated_core(b200m_ctx *ctx, int side, const float *host_base, size_t n, size_t stride_bytes, int dim) {
    Comm *cm = comm_of(ctx);
    NcclApi *nc = nccl_api();
    const int W = cm->n_ranks, r = cm->rank;
    Side &sd = ctx->side[side];
    const size_t R = rows_per_rank(n, W);
    size_t lo, hi;
    rank_rows(n, W, r, &lo, &hi);
    CK(sd.staging.reserve(R * W * stride_bytes + 16));
    char *base = sd.staging.as<char>();
    if (hi > lo) {
        size_t bytes = (hi - lo) * stride_bytes;
        if (hi == n) bytes = (hi - lo - 1) * stride_bytes + (size_t) dim * 4;   // the caller owns only dim floats of the last row
        CK(cudaMemcpyAsync(base + lo * stride_bytes, reinterpret_cast<const char *>(host_base) + lo * stride_bytes, bytes,
                           cudaMemcpyHostToDevice, ctx->stream));
    }
    if (n) NCK(nc->AllGather(base + (size_t) r * R * stride_bytes, base, R * stride_bytes, ncclUint8, cm->comm, ctx->stream));
    return b200m_upload_device(ctx, side, sd.staging.as<float>(), n, stride_bytes, dim, 0);
}

int require_comm(b200m_ctx *ctx, const char *what) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    if (!ctx->comm) return b200m_fail_msg(ctx, std::string(what) + ": no communicator attached (b200m_comm_attach / b200m_create_multi)");
    return 0;
}

}  // namespace

void comm_release(b200m_ctx *ctx) {
    Comm *cm = comm_of(ctx);
    if (!cm) return;
    if (cm->comm) nccl_api()->CommDestroy(cm->comm);
    cm->favg_d.release();
    cm->favg_c.release();
    delete cm;
    ctx->comm = nullptr;
}

// ---- single-process group: one worker thread per device -------------------------------------------------------------
struct b200m_group {
    std::vector<b200m_ctx *> ctx;
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::function<int(int)> job;
    uint64_t generation = 0;
    int pending = 0;
    bool stop = false;
    std::vector<int> rc;
    std::string err;
    // host-side gather of the per-rank record slices
    std::vector<unsigned long long> counts;
    int ranges_per_device = 1;   // group batch calls (B200M_GROUP_RANGES)

    int run(std::function<int(int)> f) {
        {
            std::unique_lock<std::mutex> lk(mu);
            job = std::move(f);
            pending = (int) ctx.size();
            ++generation;
        }
        cv_work.notify_all();
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return pending == 0; });
        for (size_t i = 0; i < ctx.size(); ++i)
            if (rc[i]) {
                err = "device " + std::to_string(ctx[i]->device) + ": " + ctx[i]->err;
                return 1;
            }
        return 0;
    }
    void worker(int i) {
        uint64_t seen = 0;
        cudaSetDevice(ctx[i]->device);
        for (;;) {
            std::function<int(int)> f;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_work.wait(lk, [&] { return stop || generation != seen; });
                if (stop) return;
                seen = generation;
                f = job;
            }
            const int r = f(i);
            {
                std::unique_lock<std::mutex> lk(mu);
                rc[i] = r;
                if (--pending == 0) cv_done.notify_all();
            }
        }
    }
};

static thread_local std::string g_group_err;

// ---- group batch calls: a batch's pairs split into contiguous ranges, one host batch form per device -------------------
namespace {

// Estimated cost of one kNN pass of nq x nt descriptor rows: the tensor-core pass's K extent is dim + 3 norm columns,
// padded to 64.  Shapes only; a guessed (gated) pass sweeps at most this much.
double desc_cost(size_t nq, size_t nt, int dim) {
    const int d = std::min(std::max(dim, 1), B200M_MAX_DIM);
    return (double) nq * (double) nt * (double) ((d + 3 + 63) / 64 * 64);
}

// ClusterMatcher's 3-D neighbourhoods (knn3d, brute force inside each pair) cost kC3d * (n_src_kps^2 + n_tgt_kps^2) in
// desc_cost units.  Measured on one B200 with the FPFH-33 20k x 20k one-scale ClusterMatcher batch against the same
// LeftToRight batch (tools/bench_group_batch.py, DESIGN.md section 3.19).
constexpr double kC3d = 211.0;

double wide_cost(const b200m_params *p, const b200m_wide_pair &w, int dim) {
    if (!w.n_src_kps || w.n_scales < 1 || w.n_scales > 32 || !w.scales) return 0.0;   // no scale takes part
    double c = 0.0;
    for (int s = 0; s < w.n_scales; ++s) c += desc_cost(w.scales[s].n_src, w.scales[s].n_tgt, dim);
    if (p->mode != B200M_MODE_ONE_SIDED) c *= 2.0;   // the reverse pass
    if (p->mode == B200M_MODE_CLUSTER) c += kC3d * ((double) w.n_src_kps * (double) w.n_src_kps + (double) w.n_tgt_kps * (double) w.n_tgt_kps);
    return c;
}

// Runs f(device, range index, first pair, end pair, range) on every non-empty range of the cost partition: ranges i, i + W,
// i + 2W, ... on device i, the devices concurrently.  W * g->ranges_per_device ranges (B200M_GROUP_RANGES, a diagnostic
// switch: several ranges per device exercise the split on a box with one GPU).  whole: the arguments cannot be split (no
// pairs, or params the single form rejects before it reads a pair): device 0 runs the whole call as given, f(0, 0, 0,
// n_pairs).  On failure g->err is the text the single form gives on the whole batch: the error of the lowest range that
// failed its checks; else the smallest bad-map key; else the lowest range's error.
int run_ranges(b200m_group *g, int n_pairs, bool whole, const std::vector<double> &cost,
               const std::function<int(int, int, int, int, BatchRange *)> &f, std::vector<int> *first) {
    const int W = (int) g->ctx.size(), P = W * g->ranges_per_device;
    first->assign((size_t) P + 1, whole ? n_pairs : 0);
    (*first)[0] = 0;
    if (!whole && b200m_batch_partition(cost.data(), n_pairs, P, first->data())) {
        g->err = "group batch: bad cost estimate";
        return 1;
    }
    std::vector<BatchRange> r((size_t) P);
    std::vector<int> rc((size_t) P, 0);
    std::vector<std::string> err((size_t) P);   // taken at once: a later range on the device overwrites the context's text
    g->run([&](int i) {
        for (int j = i; j < P; j += W) {
            const int p0 = (*first)[(size_t) j], p1 = (*first)[(size_t) j + 1];
            if (whole ? j != 0 : p0 == p1) continue;
            r[(size_t) j].pair_base = p0;
            rc[(size_t) j] = f(i, j, p0, p1, &r[(size_t) j]);
            if (rc[(size_t) j]) err[(size_t) j] = g->ctx[(size_t) i]->err;
        }
        return 0;
    });
    int pick = -1;
    for (int j = 0; j < P && pick < 0; ++j)
        if (rc[(size_t) j] && !r[(size_t) j].validated) pick = j;
    unsigned long long key = ~0ull;
    for (int j = 0; j < P && pick < 0; ++j)
        if (rc[(size_t) j] && r[(size_t) j].bad_key < key) key = r[(size_t) j].bad_key;
    for (int j = 0; j < P && pick < 0; ++j)
        if (rc[(size_t) j] && (key == ~0ull || r[(size_t) j].bad_key == key)) pick = j;
    if (pick < 0) return 0;
    g->err = err[(size_t) pick];
    return 1;
}

// The host staging of one range's records, offsets and averages, and the merge into the caller's arrays in pair order.
struct RangeOutputs {
    std::vector<std::unique_ptr<b200m_corr[]>> rec;   // not zero-filled: the records found are written, nothing else is read
    std::vector<size_t> cap;
    std::vector<std::vector<size_t>> off;
    std::vector<std::vector<float>> avg;
    explicit RangeOutputs(size_t P) : rec(P), cap(P, 0), off(P), avg(P) {}
    void size(int j, int n, size_t max_records) {
        cap[(size_t) j] = std::max<size_t>(max_records, 1);
        rec[(size_t) j].reset(new b200m_corr[cap[(size_t) j]]);
        off[(size_t) j].assign((size_t) n + 1, ~(size_t) 0);   // the single form zeroes them once its arguments pass
        avg[(size_t) j].resize((size_t) std::max(n, 1));
    }
    // after an error: the caller's offsets as the single form leaves them -- zeroed when its argument checks had passed
    // (every range runs the same ones), untouched otherwise
    void failed(size_t *offsets, int n_pairs) {
        for (const std::vector<size_t> &o : off)
            if (!o.empty() && o[0] == 0) {
                for (int j = 0; j <= n_pairs; ++j) offsets[j] = 0;
                return;
            }
    }
    // offsets concatenated and rebased, averages copied, then the capacity check on the total (offsets and averages are
    // written also when it fails, as the single forms write them) and the records
    int merge(b200m_group *g, const char *name, const std::vector<int> &first, b200m_corr *out, size_t cap, size_t *offsets, float *avg_out) {
        const int P = (int) first.size() - 1;
        offsets[0] = 0;
        for (int r = 0; r < P; ++r)
            for (int j = first[(size_t) r]; j < first[(size_t) r + 1]; ++j) {
                offsets[j + 1] = offsets[first[(size_t) r]] + off[(size_t) r][(size_t) (j - first[(size_t) r] + 1)];
                if (avg_out) avg_out[j] = avg[(size_t) r][(size_t) (j - first[(size_t) r])];
            }
        const size_t total = offsets[first[(size_t) P]];
        if (total > cap) {
            g->err = std::string(name) + ": output capacity too small (" + std::to_string(total) + " correspondences)";
            return 1;
        }
        if (total && !out) {
            g->err = std::string(name) + ": null output buffer";
            return 1;
        }
        for (int r = 0; r < P; ++r) {
            const size_t o = offsets[first[(size_t) r]], n = offsets[first[(size_t) r + 1]] - o;
            if (n) memcpy(out + o, rec[(size_t) r].get(), sizeof(b200m_corr) * n);
        }
        return 0;
    }
};

}  // namespace

extern "C" {

int b200m_comm_unique_id(void *id_out, size_t bytes) {
    NcclApi *nc = nccl_api();
    if (!nc->error.empty()) return b200m_fail_msg(nullptr, nc->error);
    if (!id_out || bytes < sizeof(ncclUniqueId)) return b200m_fail_msg(nullptr, "b200m_comm_unique_id: buffer of B200M_UNIQUE_ID_BYTES needed");
    ncclUniqueId id;
    ncclResult_t r = nc->GetUniqueId(&id);
    if (r != ncclSuccess) return b200m_fail_msg(nullptr, std::string("ncclGetUniqueId: ") + nc->GetErrorString(r));
    memcpy(id_out, &id, sizeof(id));
    return 0;
}

int b200m_comm_attach(b200m_ctx *ctx, int n_ranks, int rank, const void *unique_id) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    NcclApi *nc = nccl_api();
    if (!nc->error.empty()) return b200m_fail_msg(ctx, nc->error);
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks || !unique_id) return b200m_fail_msg(ctx, "b200m_comm_attach: bad rank / id");
    comm_release(ctx);
    Comm *cm = new Comm();
    cm->rank = rank;
    cm->n_ranks = n_ranks;
    ncclUniqueId id;
    memcpy(&id, unique_id, sizeof(id));
    ncclResult_t r = nc->CommInitRank(&cm->comm, n_ranks, id, rank);
    if (r != ncclSuccess) {
        delete cm;
        return b200m_fail_msg(ctx, std::string("ncclCommInitRank: ") + nc->GetErrorString(r));
    }
    ctx->comm = cm;
    return 0;
}

int b200m_comm_rank(const b200m_ctx *ctx, int *rank, int *n_ranks) {
    const Comm *cm = ctx ? static_cast<const Comm *>(ctx->comm) : nullptr;
    if (rank) *rank = cm ? cm->rank : 0;
    if (n_ranks) *n_ranks = cm ? cm->n_ranks : 1;
    return 0;
}

int b200m_shard_rows(size_t n, int n_ranks, int rank, size_t *row_begin, size_t *row_end) {
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks || !row_begin || !row_end) return 1;
    rank_rows(n, n_ranks, rank, row_begin, row_end);
    return 0;
}

int b200m_upload_replicated(b200m_ctx *ctx, int side, const float *host_base, size_t n, size_t stride_bytes, int dim) {
    if (require_comm(ctx, "b200m_upload_replicated")) return 1;
    CK(cudaSetDevice(ctx->device));
    if (side != 0 && side != 1) return b200m_fail_msg(ctx, "b200m_upload_replicated: side must be 0 or 1");
    if (n && !host_base) return b200m_fail_msg(ctx, "b200m_upload_replicated: null descriptor pointer");
    if (dim < 1 || dim > B200M_MAX_DIM || stride_bytes % 4 != 0 || stride_bytes < (size_t) dim * 4)
        return b200m_fail_msg(ctx, "b200m_upload_replicated: bad dim / stride");
    return upload_replicated_core(ctx, side, host_base, n, stride_bytes, dim);
}

int b200m_match_sharded_device(b200m_ctx *ctx, const b200m_params *p, const float *d_thr_src, const float *d_thr_tgt,
                               b200m_corr *d_out, size_t cap, unsigned long long *d_n_out, float *d_avg) {
    if (require_comm(ctx, "b200m_match_sharded")) return 1;
    CK(cudaSetDevice(ctx->device));
    if (!p || p->k < 1 || p->k > B200M_MAX_K) return b200m_fail_msg(ctx, "b200m_match_sharded: params.k must be in [1, 32]");
    if (p->mode < B200M_MODE_ONE_SIDED || p->mode > B200M_MODE_RATIO_MUTUAL)
        return b200m_fail_msg(ctx, "b200m_match_sharded: mode must be ONE_SIDED, MUTUAL, RATIO or RATIO_MUTUAL");
    if (!d_n_out) return b200m_fail_msg(ctx, "b200m_match_sharded: null n_out");
    return match_sharded_core(ctx, p, d_thr_src, d_thr_tgt, d_out, cap, d_n_out, d_avg);
}

int b200m_match_sharded(b200m_ctx *ctx, const b200m_params *p, const float *thr_src, const float *thr_tgt, b200m_corr *out,
                        size_t cap, size_t *n_out, float *avg_first_dist) {
    if (require_comm(ctx, "b200m_match_sharded")) return 1;
    CK(cudaSetDevice(ctx->device));
    if (!p || !n_out) return b200m_fail_msg(ctx, "b200m_match_sharded: null params / n_out");
    *n_out = 0;
    if ((thr_src == nullptr) != (thr_tgt == nullptr)) return b200m_fail_msg(ctx, "b200m_match_sharded: give both threshold arrays or neither");
    const size_t nq = ctx->side[0].n, nt = ctx->side[1].n;
    cudaStream_t st = ctx->stream;
    const float *d_ts = nullptr, *d_tt = nullptr;
    if (thr_src && nq && nt) {
        CK(ctx->ws_thr[0].reserve(sizeof(float) * nq));
        CK(ctx->ws_thr[1].reserve(sizeof(float) * nt));
        CK(cudaMemcpyAsync(ctx->ws_thr[0].p, thr_src, sizeof(float) * nq, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->ws_thr[1].p, thr_tgt, sizeof(float) * nt, cudaMemcpyHostToDevice, st));
        d_ts = ctx->ws_thr[0].as<float>();
        d_tt = ctx->ws_thr[1].as<float>();
    }
    Comm *cm = comm_of(ctx);
    const size_t Rq = rows_per_rank(nq, cm->n_ranks);
    const size_t kk = p->mode == B200M_MODE_MUTUAL ? (size_t) p->k : 1, max_out = Rq * kk;
    CK(ctx->ws_corr.reserve(sizeof(b200m_corr) * (max_out + 1)));
    CK(ctx->ws_misc.reserve(64));
    float *d_avg = ctx->ws_misc.as<float>();
    unsigned long long *d_n = reinterpret_cast<unsigned long long *>(ctx->ws_misc.as<char>() + 16);
    if (b200m_match_sharded_device(ctx, p, d_ts, d_tt, ctx->ws_corr.as<b200m_corr>(), max_out, d_n, avg_first_dist ? d_avg : nullptr))
        return 1;
    struct { float avg; float pad[3]; unsigned long long n; } h;
    CK(cudaMemcpyAsync(&h, ctx->ws_misc.p, sizeof(h), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (avg_first_dist) *avg_first_dist = nq ? h.avg : 3.402823466e+38F;
    *n_out = (size_t) h.n;
    if (h.n > cap) return b200m_fail_msg(ctx, "b200m_match_sharded: output capacity too small (" + std::to_string(h.n) + " correspondences)");
    if (h.n) {
        if (!out) return b200m_fail_msg(ctx, "b200m_match_sharded: null output buffer");
        CK(cudaMemcpyAsync(out, ctx->ws_corr.p, sizeof(b200m_corr) * h.n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return 0;
}

int b200m_knn_target_sharded_device(b200m_ctx *ctx, const b200m_params *p, int32_t *d_idx, float *d_dist, int32_t *d_count) {
    if (require_comm(ctx, "b200m_knn_target_sharded")) return 1;
    CK(cudaSetDevice(ctx->device));
    if (!p || p->k < 1 || p->k > B200M_MAX_K) return b200m_fail_msg(ctx, "b200m_knn_target_sharded: params.k must be in [1, 32]");
    if (comm_of(ctx)->n_ranks > 8) return b200m_fail_msg(ctx, "b200m_knn_target_sharded: at most 8 ranks (merge kernel)");
    if (ctx->side[0].n && (!d_idx || !d_dist || !d_count)) return b200m_fail_msg(ctx, "b200m_knn_target_sharded: null output pointer");
    return knn_target_sharded_core(ctx, p, d_idx, d_dist, d_count);
}

// ---- the single-process group -------------------------------------------------------------------------------------------
const char *b200m_group_last_error(const b200m_group *g) { return g ? g->err.c_str() : g_group_err.c_str(); }

int b200m_create_multi(b200m_group **out, const int *device_ids, int n) {
    if (!out) { g_group_err = "b200m_create_multi: null output pointer"; return 1; }
    *out = nullptr;
    if (n < 1 || n > 64 || !device_ids) { g_group_err = "b200m_create_multi: need 1..64 device ids"; return 1; }
    NcclApi *nc = nccl_api();
    if (n > 1 && !nc->error.empty()) { g_group_err = nc->error; return 1; }
    b200m_group *g = new b200m_group();
    for (int i = 0; i < n; ++i) {
        b200m_ctx *c = nullptr;
        if (b200m_create(&c, device_ids[i])) {
            g_group_err = b200m_last_error(nullptr);
            for (b200m_ctx *x : g->ctx) b200m_destroy(x);
            delete g;
            return 1;
        }
        g->ctx.push_back(c);
    }
    std::vector<ncclComm_t> comms((size_t) n);
    if (n > 1 || nc->error.empty()) {
        ncclResult_t r = nc->CommInitAll(comms.data(), n, device_ids);
        if (r != ncclSuccess) {
            g_group_err = std::string("ncclCommInitAll: ") + nc->GetErrorString(r);
            for (b200m_ctx *x : g->ctx) b200m_destroy(x);
            delete g;
            return 1;
        }
        for (int i = 0; i < n; ++i) {
            Comm *cm = new Comm();
            cm->comm = comms[(size_t) i];
            cm->rank = i;
            cm->n_ranks = n;
            g->ctx[(size_t) i]->comm = cm;
        }
    } else {
        g_group_err = nc->error;
        for (b200m_ctx *x : g->ctx) b200m_destroy(x);
        delete g;
        return 1;
    }
    if (const char *e = getenv("B200M_GROUP_RANGES")) g->ranges_per_device = std::min(std::max(atoi(e), 1), 64);
    g->rc.assign((size_t) n, 0);
    g->counts.assign((size_t) n, 0);
    for (int i = 0; i < n; ++i) g->workers.emplace_back([g, i] { g->worker(i); });
    *out = g;
    return 0;
}

void b200m_destroy_multi(b200m_group *g) {
    if (!g) return;
    {
        std::unique_lock<std::mutex> lk(g->mu);
        g->stop = true;
    }
    g->cv_work.notify_all();
    for (std::thread &t : g->workers) t.join();
    for (b200m_ctx *c : g->ctx) b200m_destroy(c);
    delete g;
}

int b200m_group_size(const b200m_group *g) { return g ? (int) g->ctx.size() : 0; }
b200m_ctx *b200m_group_ctx(b200m_group *g, int i) { return g && i >= 0 && i < (int) g->ctx.size() ? g->ctx[(size_t) i] : nullptr; }

int b200m_group_upload(b200m_group *g, int side, const float *host_base, size_t n, size_t stride_bytes, int dim) {
    if (!g) { g_group_err = "null group"; return 1; }
    return g->run([=](int i) { return b200m_upload_replicated(g->ctx[(size_t) i], side, host_base, n, stride_bytes, dim); });
}

int b200m_group_upload_sharded(b200m_group *g, int side, const float *host_base, size_t n, size_t stride_bytes, int dim) {
    if (!g) { g_group_err = "null group"; return 1; }
    const int W = (int) g->ctx.size();
    return g->run([=](int i) {
        size_t lo, hi;
        rank_rows(n, W, i, &lo, &hi);
        return b200m_upload(g->ctx[(size_t) i], side, reinterpret_cast<const float *>(reinterpret_cast<const char *>(host_base) + lo * stride_bytes),
                            hi - lo, stride_bytes, dim, (int64_t) lo);
    });
}

int b200m_group_match(b200m_group *g, const b200m_params *p, const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap,
                      size_t *n_out, float *avg_first_dist) {
    if (!g) { g_group_err = "null group"; return 1; }
    if (!p || !n_out) { g->err = "b200m_group_match: null params / n_out"; return 1; }
    *n_out = 0;
    const int W = (int) g->ctx.size();
    const size_t nq = g->ctx[0]->side[0].n;
    const size_t Rq = rows_per_rank(nq, W);
    const size_t kk = p->mode == B200M_MODE_MUTUAL ? (size_t) p->k : 1;
    // every rank's slice lands in a staging area of the caller's buffer size class, then is packed in rank order
    std::vector<std::vector<b200m_corr>> slices((size_t) W);
    std::vector<float> avgs((size_t) W, 0.f);
    int rc = g->run([&](int i) {
        slices[(size_t) i].resize(Rq * kk + 1);
        size_t n = 0;
        int r = b200m_match_sharded(g->ctx[(size_t) i], p, thr_src, thr_tgt, slices[(size_t) i].data(), slices[(size_t) i].size(), &n,
                                    avg_first_dist ? &avgs[(size_t) i] : nullptr);
        g->counts[(size_t) i] = n;
        return r;
    });
    if (rc) return 1;
    size_t total = 0;
    for (int i = 0; i < W; ++i) total += (size_t) g->counts[(size_t) i];
    *n_out = total;
    if (avg_first_dist) *avg_first_dist = avgs[0];
    if (total > cap) { g->err = "b200m_group_match: output capacity too small (" + std::to_string(total) + " correspondences)"; return 1; }
    size_t off = 0;
    for (int i = 0; i < W; ++i) {   // rank order == ascending index_query
        if (g->counts[(size_t) i]) memcpy(out + off, slices[(size_t) i].data(), sizeof(b200m_corr) * (size_t) g->counts[(size_t) i]);
        off += (size_t) g->counts[(size_t) i];
    }
    return 0;
}

int b200m_group_knn(b200m_group *g, const b200m_params *p, int32_t *idx, float *dist, int32_t *count) {
    if (!g) { g_group_err = "null group"; return 1; }
    if (!p) { g->err = "b200m_group_knn: null params"; return 1; }
    const int W = (int) g->ctx.size(), k = p->k;
    const size_t nq = g->ctx[0]->side[0].n;
    if (nq == 0) return 0;
    if (!idx || !dist || !count) { g->err = "b200m_group_knn: null output pointer"; return 1; }
    if (p->shard == B200M_SHARD_TARGET) {
        // every rank ends with the merged lists; rank i copies rows of its own slice to the host (PCIe in parallel)
        return g->run([=](int i) {
            b200m_ctx *ctx = g->ctx[(size_t) i];
            CK(cudaSetDevice(ctx->device));
            CK(ctx->ws_fidx.reserve(sizeof(int32_t) * nq * k));
            CK(ctx->ws_fdist.reserve(sizeof(float) * nq * k));
            CK(ctx->ws_fcnt.reserve(sizeof(int32_t) * nq));
            if (b200m_knn_target_sharded_device(ctx, p, ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>()))
                return 1;
            size_t lo, hi;
            rank_rows(nq, W, i, &lo, &hi);
            if (hi > lo) {
                CK(cudaMemcpyAsync(idx + lo * k, ctx->ws_fidx.as<int32_t>() + lo * k, sizeof(int32_t) * (hi - lo) * k, cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaMemcpyAsync(dist + lo * k, ctx->ws_fdist.as<float>() + lo * k, sizeof(float) * (hi - lo) * k, cudaMemcpyDeviceToHost, ctx->stream));
                CK(cudaMemcpyAsync(count + lo, ctx->ws_fcnt.as<int32_t>() + lo, sizeof(int32_t) * (hi - lo), cudaMemcpyDeviceToHost, ctx->stream));
            }
            CK(cudaStreamSynchronize(ctx->stream));
            return 0;
        });
    }
    // query-sharded: rank i answers its own rows against the full (replicated) target
    return g->run([=](int i) {
        size_t lo, hi;
        rank_rows(nq, W, i, &lo, &hi);
        if (hi == lo) return 0;
        return b200m_knn(g->ctx[(size_t) i], p, 0, lo, hi, idx + lo * k, dist + lo * k, count + lo);
    });
}

int b200m_batch_partition(const double *cost, int n_pairs, int n_parts, int *first) {
    if (n_pairs < 0 || n_parts < 1 || !first || (n_pairs && !cost)) return 1;
    std::vector<double> pre((size_t) n_pairs + 1, 0.0);
    for (int i = 0; i < n_pairs; ++i) {
        if (!(cost[i] >= 0.0) || cost[i] > DBL_MAX) return 1;   // NaN, negative or infinite
        pre[(size_t) i + 1] = pre[(size_t) i] + cost[i];
    }
    // A range [a, b) costs pre[b] - pre[a], which grows as the range grows, so the greedy cut (each range as long as the
    // bound allows) needs the fewest ranges for a bound, and the least feasible bound is the optimum.  The bound is searched
    // over the bit patterns of the non-negative doubles, which order as the values do: the result is exactly one of the
    // range costs.
    // A range also stops growing once no more pairs are left than parts after it, so that every part gets a pair when there
    // are enough (the rest of the pairs then go one per part, which any feasible bound allows).
    auto cut = [&](double bound, int *f) {   // ranges the greedy cut needs (n_parts + 1: infeasible)
        int parts = 0;
        for (int a = 0; a < n_pairs;) {
            int b = a;
            while (b < n_pairs && pre[(size_t) b + 1] - pre[(size_t) a] <= bound && (b == a || n_pairs - b > n_parts - parts - 1)) ++b;
            if (b == a || parts == n_parts) return n_parts + 1;
            if (f) f[parts] = a;
            ++parts;
            a = b;
        }
        return parts;
    };
    const double all = pre[(size_t) n_pairs];
    if (all > DBL_MAX) return 1;
    uint64_t lo = 0, hi;
    memcpy(&hi, &all, sizeof(hi));
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        double bound;
        memcpy(&bound, &mid, sizeof(bound));
        if (cut(bound, nullptr) <= n_parts) hi = mid; else lo = mid + 1;
    }
    double bound;
    memcpy(&bound, &lo, sizeof(bound));
    const int used = cut(bound, first);
    for (int i = used; i <= n_parts; ++i) first[i] = n_pairs;   // unused parts: empty ranges at the end
    return 0;
}

int b200m_group_knn_batch(b200m_group *g, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes, int dim,
                          int32_t *idx, float *dist, int32_t *count) {
    if (!g) {
        knn_batch_host(nullptr, p, pairs, n_pairs, stride_bytes, dim, idx, dist, count, nullptr);
        g_group_err = b200m_last_error(nullptr);
        return 1;
    }
    const bool whole = !p || !pairs || n_pairs <= 0 || p->k < 1 || p->k > B200M_MAX_K;
    std::vector<double> cost(whole ? 0 : (size_t) n_pairs);
    std::vector<size_t> rows_before(whole ? 1 : (size_t) n_pairs + 1, 0);
    for (size_t i = 0; i < cost.size(); ++i) {
        cost[i] = desc_cost(pairs[i].n_src, pairs[i].n_tgt, dim);
        rows_before[i + 1] = rows_before[i] + pairs[i].n_src;
    }
    std::vector<int> first;
    return run_ranges(g, n_pairs, whole, cost, [&](int i, int, int p0, int p1, BatchRange *r) {
        if (whole) return knn_batch_host(g->ctx[0], p, pairs, n_pairs, stride_bytes, dim, idx, dist, count, r);
        // the k-lists go straight to the caller's arrays at the range's first row
        const size_t o = rows_before[(size_t) p0], k = (size_t) p->k;
        return knn_batch_host(g->ctx[(size_t) i], p, pairs + p0, p1 - p0, stride_bytes, dim, idx ? idx + o * k : nullptr,
                              dist ? dist + o * k : nullptr, count ? count + o : nullptr, r);
    }, &first);
}

int b200m_group_match_batch(b200m_group *g, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes, int dim,
                            const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap, size_t *offsets, float *avg) {
    if (!g) {
        match_batch_host(nullptr, p, pairs, n_pairs, stride_bytes, dim, thr_src, thr_tgt, out, cap, offsets, avg, nullptr);
        g_group_err = b200m_last_error(nullptr);
        return 1;
    }
    const bool whole = !p || !pairs || n_pairs <= 0 || p->k < 1 || p->k > B200M_MAX_K;
    const bool mutual = p && (p->mode == B200M_MODE_MUTUAL || p->mode == B200M_MODE_RATIO_MUTUAL);
    std::vector<double> cost(whole ? 0 : (size_t) n_pairs);
    std::vector<size_t> before[2] = {std::vector<size_t>(cost.size() + 1, 0), std::vector<size_t>(cost.size() + 1, 0)};
    for (size_t i = 0; i < cost.size(); ++i) {
        cost[i] = desc_cost(pairs[i].n_src, pairs[i].n_tgt, dim) * (mutual ? 2.0 : 1.0);
        before[0][i + 1] = before[0][i] + pairs[i].n_src;
        before[1][i + 1] = before[1][i] + pairs[i].n_tgt;
    }
    RangeOutputs ro(g->ctx.size() * (size_t) g->ranges_per_device);
    std::vector<int> first;
    if (run_ranges(g, n_pairs, whole, cost, [&](int i, int j, int p0, int p1, BatchRange *r) {
            if (whole)
                return match_batch_host(g->ctx[0], p, pairs, n_pairs, stride_bytes, dim, thr_src, thr_tgt, out, cap, offsets, avg, r);
            const size_t kk = p->mode == B200M_MODE_MUTUAL ? (size_t) p->k : 1;
            ro.size(j, p1 - p0, (before[0][(size_t) p1] - before[0][(size_t) p0]) * kk);
            return match_batch_host(g->ctx[(size_t) i], p, pairs + p0, p1 - p0, stride_bytes, dim,
                                    thr_src ? thr_src + before[0][(size_t) p0] : nullptr,
                                    thr_tgt ? thr_tgt + before[1][(size_t) p0] : nullptr, ro.rec[(size_t) j].get(),
                                    ro.cap[(size_t) j], offsets ? ro.off[(size_t) j].data() : nullptr,
                                    avg ? ro.avg[(size_t) j].data() : nullptr, r);
        }, &first)) {
        if (!whole && offsets) ro.failed(offsets, n_pairs);
        return 1;
    }
    return whole ? 0 : ro.merge(g, "b200m_match_batch", first, out, cap, offsets, avg);
}

namespace {

int group_wide_batch(b200m_group *g, const b200m_params *p, const b200m_wide_pair *pairs, bool gated, const b200m_local_pair *locals,
                     int n_pairs, size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k, float radius,
                     const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap, size_t *offsets, float *avg) {
    if (!g) {
        match_multiscale_batch_host(nullptr, p, pairs, gated, locals, n_pairs, stride_bytes, dim, xyz_stride_bytes, cluster_k, radius,
                                    thr_src, thr_tgt, out, cap, offsets, avg, nullptr);
        g_group_err = b200m_last_error(nullptr);
        return 1;
    }
    const bool whole = !p || !pairs || (gated && !locals) || n_pairs <= 0 || p->k < 1 || p->k > B200M_MAX_K;
    std::vector<double> cost(whole ? 0 : (size_t) n_pairs);
    std::vector<size_t> before[2] = {std::vector<size_t>(cost.size() + 1, 0), std::vector<size_t>(cost.size() + 1, 0)};
    for (size_t i = 0; i < cost.size(); ++i) {
        cost[i] = wide_cost(p, pairs[i], dim);
        before[0][i + 1] = before[0][i] + pairs[i].n_src_kps;
        before[1][i + 1] = before[1][i] + pairs[i].n_tgt_kps;
    }
    RangeOutputs ro(g->ctx.size() * (size_t) g->ranges_per_device);
    std::vector<int> first;
    if (run_ranges(g, n_pairs, whole, cost, [&](int i, int j, int p0, int p1, BatchRange *r) {
            if (whole)
                return match_multiscale_batch_host(g->ctx[0], p, pairs, gated, locals, n_pairs, stride_bytes, dim, xyz_stride_bytes,
                                                   cluster_k, radius, thr_src, thr_tgt, out, cap, offsets, avg, r);
            ro.size(j, p1 - p0, before[0][(size_t) p1] - before[0][(size_t) p0]);
            return match_multiscale_batch_host(g->ctx[(size_t) i], p, pairs + p0, gated, gated ? locals + p0 : nullptr, p1 - p0,
                                               stride_bytes, dim, xyz_stride_bytes, cluster_k, radius,
                                               thr_src ? thr_src + before[0][(size_t) p0] : nullptr,
                                               thr_tgt ? thr_tgt + before[1][(size_t) p0] : nullptr, ro.rec[(size_t) j].get(),
                                               ro.cap[(size_t) j], offsets ? ro.off[(size_t) j].data() : nullptr,
                                               avg ? ro.avg[(size_t) j].data() : nullptr, r);
        }, &first)) {
        if (!whole && offsets) ro.failed(offsets, n_pairs);
        return 1;
    }
    return whole ? 0 : ro.merge(g, gated ? "b200m_match_multiscale_local_batch" : "b200m_match_multiscale_batch", first, out, cap, offsets, avg);
}

}  // namespace

int b200m_group_match_multiscale_batch(b200m_group *g, const b200m_params *p, const b200m_wide_pair *pairs, int n_pairs,
                                       size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k, const float *thr_src,
                                       const float *thr_tgt, b200m_corr *out, size_t cap, size_t *offsets, float *avg) {
    return group_wide_batch(g, p, pairs, false, nullptr, n_pairs, stride_bytes, dim, xyz_stride_bytes, cluster_k, 0.f, thr_src, thr_tgt,
                            out, cap, offsets, avg);
}

int b200m_group_match_multiscale_local_batch(b200m_group *g, const b200m_params *p, const b200m_wide_pair *pairs,
                                             const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim,
                                             size_t xyz_stride_bytes, int cluster_k, float match_search_radius, const float *thr_src,
                                             const float *thr_tgt, b200m_corr *out, size_t cap, size_t *offsets, float *avg) {
    return group_wide_batch(g, p, pairs, true, locals, n_pairs, stride_bytes, dim, xyz_stride_bytes, cluster_k, match_search_radius,
                            thr_src, thr_tgt, out, cap, offsets, avg);
}

}  // extern "C"
