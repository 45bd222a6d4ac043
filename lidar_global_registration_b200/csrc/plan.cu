// plan.cu -- batch plans: b200m_knn_batch_device / b200m_match_batch_device and the matcher-class batches
// b200m_match_multiscale(_local)_batch_device bound once, then enqueued without the host.
//
// A device batch call stops the host twice: the prepare step reads its statistics back (the certificate's window decides
// tensor cores or exact path, and the norm bound is a kernel parameter), and the match form reads the result area back
// (per-pair counts -> offsets, averages, the capacity check, then a copy of a host-known number of records).  It also
// builds and uploads its tables, queries every pointer and grows its workspaces on every call.  None of that is legal
// while a stream is being captured into a CUDA graph, and each sync stalls the thread that feeds the GPU.
//
// A plan does all the host work once, at creation, and b200m_plan_run only enqueues kernels and memsets:
//
//   tables      stage_batch_tables at creation, in the plan's own context; run enqueues stage_batch_pack (the segmented pack)
//   prepare     the plan's context has device_prepare set: launch_tc_prepare ends in prep_decide_kernel, which writes the
//               window decision and the norm bounds into PrepDev, and the candidate kernel's DP form reads them there.
//               Data outside the window leaves every candidate list overflowed, so the exact fallback that runs on every
//               call answers each row -- the same exact kernels the host decision would have picked.
//   results     plan_finish_kernel turns the per-pair counts into offsets, copies averages and the record count, and
//               copies min(n_out, cap) records: capacity is reported (n_out > cap), not enforced.
//   wide        the matcher-class plans keep the driver of wide_batch.cu in its parts: wide_batch_tables at creation (every
//               scale's batch tables in a buffer of its own), wide_batch_enqueue on every run.  The run resets the result
//               area on the device; the finish step also copies the bad-map key to the caller's status word, which
//               b200m_plan_status_error turns into the device form's text.
//   ownership   the plan's buffers live in a private b200m_ctx (created with the caller's device and environment), so no
//               later call on the caller's context can move memory a captured graph points to.  Every workspace size
//               follows from shapes only; the run at creation grows them all, and later runs allocate nothing.
//
// Profiling (b200m_set_profiling) and its StatTimer regions do not apply to plans: their context never profiles.
#include <string>
#include <vector>

#include "internal.cuh"

struct b200m_plan {
    b200m_ctx *ctx = nullptr;   // private: owns every buffer the plan's kernels touch
    bool match = false;
    b200m_params p{};
    std::vector<b200m_pair> pairs;
    size_t stride_bytes = 0;
    int dim = 0;
    BatchLayout L;
    const float *thr_src = nullptr, *thr_tgt = nullptr;
    // knn plans
    int32_t *idx = nullptr;
    float *dist = nullptr;
    int32_t *count = nullptr;
    // match plans
    b200m_corr *out = nullptr;
    size_t cap = 0;
    uint64_t *offsets = nullptr;
    float *avg = nullptr;
    uint64_t *n_out = nullptr;
    // matcher-class plans
    struct WidePlan *wide = nullptr;
    uint64_t *status = nullptr;
    mutable std::string status_text;   // b200m_plan_status_error's last answer
};

// A matcher-class plan's own copies of the call's host arrays (the caller's may go away after creation).
struct WidePlan {
    WideCall call;
    std::vector<b200m_wide_pair> pairs;
    std::vector<std::vector<b200m_scale>> scales;
    std::vector<b200m_local_pair> locals;
    WideLayout layout;
};

namespace {

constexpr int kFinishThreads = 256;

// Block 0: offsets = exclusive scan of the per-pair counts (a thread per contiguous chunk of pairs), the averages and the
// record count.  Every block: records [0, min(n_out, cap)) from the work buffer.  empty: the batch has no source rows
// (no kernel before this one ran): zero offsets and count, FLT_MAX averages, as b200m_match_batch_device gives them.
__global__ void __launch_bounds__(kFinishThreads)
plan_finish_kernel(const unsigned long long *__restrict__ n_found, const unsigned *__restrict__ counts,
                   const float *__restrict__ avgs, int n_pairs, int empty, const b200m_corr *__restrict__ rec, size_t cap,
                   uint64_t *__restrict__ offsets, float *__restrict__ avg, uint64_t *__restrict__ n_out,
                   b200m_corr *__restrict__ out, const unsigned long long *__restrict__ bad, uint64_t *__restrict__ status) {
    const unsigned long long n = empty ? 0ull : *n_found;
    if (blockIdx.x == 0) {
        __shared__ unsigned long long part[kFinishThreads];
        const int per = (n_pairs + kFinishThreads - 1) / kFinishThreads;
        const int i0 = min(n_pairs, (int) threadIdx.x * per), i1 = min(n_pairs, i0 + per);
        unsigned long long s = 0;
        for (int i = i0; i < i1; ++i) s += empty ? 0u : counts[i];
        part[threadIdx.x] = s;
        __syncthreads();
        for (int o = 1; o < kFinishThreads; o <<= 1) {   // inclusive scan of the chunk sums
            const unsigned long long v = threadIdx.x >= (unsigned) o ? part[threadIdx.x - o] : 0ull;
            __syncthreads();
            part[threadIdx.x] += v;
            __syncthreads();
        }
        unsigned long long run = part[threadIdx.x] - s;
        for (int i = i0; i < i1; ++i) {
            run += empty ? 0u : counts[i];
            offsets[i + 1] = run;
        }
        if (threadIdx.x == 0) {
            offsets[0] = 0;
            *n_out = n;
            if (status) *status = empty ? ~0ull : *bad;   // matcher-class plans: the bad-map key, ~0 = clean
        }
        if (avg)
            for (int i = threadIdx.x; i < n_pairs; i += kFinishThreads) avg[i] = empty ? 3.402823466e+38F : avgs[i];
    }
    const size_t m = n < cap ? (size_t) n : cap;
    for (size_t i = (size_t) blockIdx.x * kFinishThreads + threadIdx.x; i < m; i += (size_t) gridDim.x * kFinishThreads)
        out[i] = rec[i];
}

int enqueue(b200m_plan *pl) {
    b200m_ctx *ctx = pl->ctx;
    const unsigned long long *found, *bad = nullptr;
    const unsigned *counts;
    const float *avgs;
    int n_pairs, empty;
    if (pl->wide) {
        const WideLayout &W = pl->wide->layout;
        if (wide_batch_enqueue(ctx, pl->wide->call, W)) return 1;
        found = W.n_out;
        bad = W.bad;
        counts = W.counts;
        avgs = W.avgs;
        n_pairs = pl->wide->call.n_pairs;
        empty = W.n_scales == 0;
    } else {
        const BatchLayout &L = pl->L;
        n_pairs = (int) pl->pairs.size();
        const bool rows = L.real_src > 0;
        if (rows && stage_batch_pack(ctx, pl->pairs.data(), n_pairs, pl->stride_bytes, pl->dim, L, true)) return 1;
        if (!pl->match) return rows ? knn_batch_lists(ctx, &pl->p, L, pl->idx, pl->dist, pl->count) : 0;
        if (rows && match_batch_records(ctx, &pl->p, L, pl->pairs.data(), n_pairs, true, pl->thr_src, pl->thr_tgt, pl->avg != nullptr))
            return 1;
        found = L.n_out;
        counts = L.counts;
        avgs = L.avgs;
        empty = rows ? 0 : 1;
    }
    const unsigned blocks = (unsigned) ctx->sm_count * 2;
    plan_finish_kernel<<<blocks, kFinishThreads, 0, ctx->stream>>>(found, counts, avgs, n_pairs, empty, ctx->ws_corr.as<b200m_corr>(),
                                                                   pl->cap, pl->offsets, pl->avg, pl->n_out, pl->out, bad,
                                                                   pl->status);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

// The checks of the device form (same texts), then the plan's context, its tables and one synchronised run.
int plan_create(b200m_ctx *ctx, const char *fn, b200m_plan *pl, b200m_plan **out) {
    const std::string f(fn);
    const b200m_params *p = &pl->p;
    const int n_pairs = (int) pl->pairs.size();
    if (pl->wide) {   // the matcher-class checks that concern the call's tables come with wide_batch_tables below
        if (!pl->n_out) return b200m_fail_msg(ctx, f + ": null n_out");
        if (!pl->status) return b200m_fail_msg(ctx, f + ": null status");
        if (pl->cap && !pl->out) return b200m_fail_msg(ctx, f + ": null output buffer");
        if (check_device_ptr(ctx, f + ": offsets", pl->offsets) || check_device_ptr(ctx, f + ": avg", pl->avg) ||
            check_device_ptr(ctx, f + ": n_out", pl->n_out) || check_device_ptr(ctx, f + ": status", pl->status))
            return 1;
    } else if (pl->match) {
        if (p->mode == B200M_MODE_KNN_ONLY) return b200m_fail_msg(ctx, f + ": use b200m_knn_batch for raw k-lists");
        if (p->mode == B200M_MODE_CLUSTER)
            return b200m_fail_msg(ctx, f + ": the cluster filter needs keypoint coordinates, use b200m_match_cluster");
        if (!pl->offsets) return b200m_fail_msg(ctx, f + ": null offsets");
        if (!pl->n_out) return b200m_fail_msg(ctx, f + ": null n_out");
        if ((pl->thr_src == nullptr) != (pl->thr_tgt == nullptr))
            return b200m_fail_msg(ctx, f + ": give both threshold arrays or neither");
        if (pl->cap && !pl->out) return b200m_fail_msg(ctx, f + ": null output buffer");
        if (check_device_ptr(ctx, f + ": thr_src", pl->thr_src) || check_device_ptr(ctx, f + ": thr_tgt", pl->thr_tgt) ||
            check_device_ptr(ctx, f + ": out", pl->out) || check_device_ptr(ctx, f + ": offsets", pl->offsets) ||
            check_device_ptr(ctx, f + ": avg", pl->avg) || check_device_ptr(ctx, f + ": n_out", pl->n_out))
            return 1;
    } else if (check_device_ptr(ctx, f + ": idx", pl->idx) || check_device_ptr(ctx, f + ": dist", pl->dist) ||
               check_device_ptr(ctx, f + ": count", pl->count)) {
        return 1;
    }
    b200m_ctx *own = nullptr;
    if (b200m_create(&own, ctx->device)) return b200m_fail_msg(ctx, f + ": " + b200m_last_error(nullptr));
    pl->ctx = own;
    own->device_prepare = true;
    own->stream = ctx->stream;   // creation runs on the caller's stream; every run names its own
    if (pl->wide) {
        if (wide_batch_tables(own, pl->wide->call, &pl->wide->layout, true)) return b200m_fail_msg(ctx, own->err);
    } else if (stage_batch_tables(own, fn, p, pl->pairs.data(), n_pairs, pl->stride_bytes, pl->dim, &pl->L, true, pl->thr_src,
                                  pl->thr_tgt)) {
        return b200m_fail_msg(ctx, own->err);
    }
    if (!pl->match && pl->L.real_src && (!pl->idx || !pl->dist || !pl->count))
        return b200m_fail_msg(ctx, f + ": null output pointer");
    // every workspace grows to its shape-determined size here, and every kernel module is loaded before any capture
    if (enqueue(pl)) return b200m_fail_msg(ctx, own->err);
    const cudaError_t e = cudaStreamSynchronize(own->stream);
    if (e != cudaSuccess) return b200m_fail(ctx, "cudaStreamSynchronize(plan run)", e, __FILE__, __LINE__);
    if (pl->wide) {   // the creation run is synchronised anyway: a bad map entry fails it, as it fails the device form
        uint64_t status = ~0ull;
        const cudaError_t ec = cudaMemcpy(&status, pl->status, sizeof(status), cudaMemcpyDeviceToHost);
        if (ec != cudaSuccess) return b200m_fail(ctx, "cudaMemcpy(plan status)", ec, __FILE__, __LINE__);
        if (status != ~0ull) return b200m_fail_msg(ctx, f + ": " + map_status_text(status));
    }
    own->stream = own->own_stream;
    *out = pl;
    return 0;
}

// Takes ownership of pl (destroyed unless the plan is made).
int make_plan(b200m_ctx *ctx, const char *fn, b200m_plan *pl, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
              size_t stride_bytes, int dim, b200m_plan **out) {
    const std::string f(fn);
    int rc = 0;
    if (!ctx) rc = b200m_fail_msg(nullptr, "null context");
    else if (!out) rc = b200m_fail_msg(ctx, f + ": null plan pointer");
    else if (cudaSetDevice(ctx->device) != cudaSuccess) rc = b200m_fail_msg(ctx, f + ": cudaSetDevice failed");
    else if (check_params(ctx, p)) rc = 1;
    else if (n_pairs < 0) rc = b200m_fail_msg(ctx, f + ": n_pairs < 0");
    else if (n_pairs > 0 && !pairs) rc = b200m_fail_msg(ctx, f + ": null pairs");
    if (out) *out = nullptr;
    if (rc) {
        delete pl;
        return rc;
    }
    pl->p = *p;
    pl->pairs.assign(pairs, pairs + n_pairs);
    pl->stride_bytes = stride_bytes;
    pl->dim = dim;
    if (plan_create(ctx, fn, pl, out)) {
        b200m_plan_destroy(pl);
        return 1;
    }
    return 0;
}

// The matcher-class plans: the device form's arguments.  The plan copies the host arrays they point to (malformed ones are
// left as given, for wide_batch_tables to refuse with the device form's texts).
int wide_plan(b200m_ctx *ctx, const char *name, bool gated, const b200m_params *p, const b200m_wide_pair *pairs,
              const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k,
              float radius, const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap, uint64_t *d_offsets,
              float *d_avg, uint64_t *d_n_out, uint64_t *d_status, b200m_plan **out) {
    const std::string f(name);
    if (out) *out = nullptr;
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    if (!out) return b200m_fail_msg(ctx, f + ": null plan pointer");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return b200m_fail_msg(ctx, f + ": cudaSetDevice failed");
    if (!p || !d_offsets) return b200m_fail_msg(ctx, f + ": null params / offsets");
    b200m_plan *pl = new b200m_plan();
    pl->match = true;
    pl->out = d_out;
    pl->cap = cap;
    pl->offsets = d_offsets;
    pl->avg = d_avg;
    pl->n_out = d_n_out;
    pl->status = d_status;
    WidePlan *w = pl->wide = new WidePlan();
    WideCall &c = w->call;
    c.name = name;
    c.dev = true;
    c.gated = gated;
    c.p = *p;
    c.n_pairs = n_pairs;
    c.stride_bytes = stride_bytes;
    c.dim = dim;
    c.xyz_stride_bytes = xyz_stride_bytes;
    c.cluster_k = cluster_k;
    c.radius = radius;
    c.thr_src = d_thr_src;
    c.thr_tgt = d_thr_tgt;
    c.out = d_out;
    c.want_avg = d_avg != nullptr;
    c.pairs = pairs;
    c.locals = locals;
    if (pairs && n_pairs > 0) {
        w->pairs.assign(pairs, pairs + n_pairs);
        w->scales.resize(n_pairs);
        for (int i = 0; i < n_pairs; ++i) {
            b200m_wide_pair &wp = w->pairs[i];
            if (wp.scales && wp.n_scales > 0 && wp.n_scales <= 32) {
                w->scales[i].assign(wp.scales, wp.scales + wp.n_scales);
                wp.scales = w->scales[i].data();
            }
        }
        c.pairs = w->pairs.data();
    }
    if (locals && n_pairs > 0) {
        w->locals.assign(locals, locals + n_pairs);
        c.locals = w->locals.data();
    }
    if (plan_create(ctx, name, pl, out)) {
        b200m_plan_destroy(pl);
        return 1;
    }
    return 0;
}

}  // namespace

extern "C" {

int b200m_plan_knn_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes,
                         int dim, int32_t *d_idx, float *d_dist, int32_t *d_count, b200m_plan **plan) {
    b200m_plan *pl = new b200m_plan();
    pl->idx = d_idx;
    pl->dist = d_dist;
    pl->count = d_count;
    return make_plan(ctx, "b200m_plan_knn_batch", pl, p, pairs, n_pairs, stride_bytes, dim, plan);
}

int b200m_plan_match_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes,
                           int dim, const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                           uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out, b200m_plan **plan) {
    b200m_plan *pl = new b200m_plan();
    pl->match = true;
    pl->thr_src = d_thr_src;
    pl->thr_tgt = d_thr_tgt;
    pl->out = d_out;
    pl->cap = cap;
    pl->offsets = d_offsets;
    pl->avg = d_avg;
    pl->n_out = d_n_out;
    return make_plan(ctx, "b200m_plan_match_batch", pl, p, pairs, n_pairs, stride_bytes, dim, plan);
}

int b200m_plan_match_multiscale_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs, int n_pairs,
                                      size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k, const float *d_thr_src,
                                      const float *d_thr_tgt, b200m_corr *d_out, size_t cap, uint64_t *d_offsets, float *d_avg,
                                      uint64_t *d_n_out, uint64_t *d_status, b200m_plan **plan) {
    return wide_plan(ctx, "b200m_plan_match_multiscale_batch", false, p, pairs, nullptr, n_pairs, stride_bytes, dim,
                     xyz_stride_bytes, cluster_k, 0.f, d_thr_src, d_thr_tgt, d_out, cap, d_offsets, d_avg, d_n_out, d_status, plan);
}

int b200m_plan_match_multiscale_local_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                            const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim,
                                            size_t xyz_stride_bytes, int cluster_k, float match_search_radius,
                                            const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                            uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out, uint64_t *d_status,
                                            b200m_plan **plan) {
    return wide_plan(ctx, "b200m_plan_match_multiscale_local_batch", true, p, pairs, locals, n_pairs, stride_bytes, dim,
                     xyz_stride_bytes, cluster_k, match_search_radius, d_thr_src, d_thr_tgt, d_out, cap, d_offsets, d_avg, d_n_out,
                     d_status, plan);
}

int b200m_plan_run(b200m_plan *plan, void *cuda_stream) {
    if (!plan) return b200m_fail_msg(nullptr, "b200m_plan_run: null plan");
    b200m_ctx *ctx = plan->ctx;
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t) cuda_stream;
    return enqueue(plan);
}

void b200m_plan_destroy(b200m_plan *plan) {
    if (!plan) return;
    if (plan->ctx) {
        plan->ctx->stream = plan->ctx->own_stream;
        b200m_destroy(plan->ctx);
    }
    delete plan->wide;
    delete plan;
}

const char *b200m_plan_last_error(const b200m_plan *plan) {
    return plan && plan->ctx ? plan->ctx->err.c_str() : b200m_last_error(nullptr);
}

const char *b200m_plan_status_error(const b200m_plan *plan, uint64_t status) {
    static thread_local std::string without_plan;
    if (status == ~0ull) return nullptr;
    std::string &s = plan ? plan->status_text : without_plan;
    s = map_status_text(status);
    return s.c_str();
}

}  // extern "C"
