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
//   live rows   the *_rows k-list / match plans bind capacities: stage_batch_tables lays every pair out in a slot of
//               pad_rows(capacity) rows per side, so the block -> pair tables and pair_info are static.  Every run starts
//               with plan_rows_kernel, which rewrites the tables that depend on the live counts (segment ranges, the
//               segmented pack's and the thresholds' row counts, the averages' segments) from the caller's device array.
//               The rest of a slot packs as gap rows -- invalid, never returned -- so the answers are the device form's on
//               the live prefixes (DESIGN.md section 3.18).  No existing kernel changed.
//   ownership   the plan's buffers live in a private b200m_ctx (created with the caller's device and environment), so no
//               later call on the caller's context can move memory a captured graph points to.  Every workspace size
//               follows from shapes only; the run at creation grows them all, and later runs allocate nothing.
//
// Profiling (b200m_set_profiling) and its StatTimer regions do not apply to plans: their context never profiles.
#include <string.h>

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
    // k-list / match plans with live counts (the *_rows creators): the pairs' sizes are capacities
    const uint32_t *rows = nullptr;   // [n_pairs][2] live (source, target) rows, the caller's device memory; matcher-class
                                      // plans: [sum of the pairs' scales][2], pair-then-scale order
    const uint32_t *kps = nullptr;    // matcher-class plans with live counts: [n_pairs][2] live (source, target) keypoints
    DevBuf slots;                     // [n_pairs] int4 {first source row, source capacity, first target row, target capacity};
                                      // matcher-class plans: the static tables and scratch of plan_wide_rows_kernel
    struct WideRowsArgs *wr = nullptr;
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

constexpr int kRowsThreads = 128;

// One CTA per pair: pair p's live counts -> the tables stage_batch_tables built for its capacities, rewritten in place.
// The set and threshold tables get the live rows (the pack writes the rest of the pair's slot as gap rows), the average its
// live segment, and every 256-row query block of the slot the pair's live train range -- empty for a block that holds no
// live row, so its candidate CTAs take the empty-range exit and the exact kernels scan nothing.  The block -> pair tables
// and pair_info (whose row count is the whole slot: the k-list rows past the live count come out of the kNN as gap rows,
// i.e. as the empty list) stay as built.  A count above its capacity empties the pair and is keyed into *status.
__global__ void __launch_bounds__(kRowsThreads)
plan_rows_kernel(const uint2 *__restrict__ live, const int4 *__restrict__ slots, SetRef *__restrict__ sets0,
                 SetRef *__restrict__ sets1, GatherSet *__restrict__ thr0, GatherSet *__restrict__ thr1,
                 int2 *__restrict__ avg_segs, int2 *__restrict__ range0, int2 *__restrict__ range1,
                 unsigned long long *__restrict__ status) {
    const int p = blockIdx.x;
    const int4 sl = slots[p];   // {s0, cap_s, t0, cap_t}
    const uint2 n = live[p];
    const bool over_s = n.x > (unsigned) sl.y, over_t = n.y > (unsigned) sl.w;
    const int ns = over_s || over_t ? 0 : (int) n.x, nt = over_s || over_t ? 0 : (int) n.y;
    if (threadIdx.x == 0) {
        if ((over_s || over_t) && status) atomicMin(status, ((unsigned long long) p << 16) | (over_s ? 2ull : 3ull));
        sets0[p].rows = ns;
        sets1[p].rows = nt;
        if (thr0) {
            thr0[p].rows = ns;
            thr1[p].rows = nt;
        }
        avg_segs[p] = make_int2(sl.x, ns);
    }
    const int nb0 = (sl.y + B200M_TILE_N - 1) / B200M_TILE_N, nb1 = (sl.w + B200M_TILE_N - 1) / B200M_TILE_N;
    for (int b = threadIdx.x; b < nb0; b += kRowsThreads)
        range0[sl.x / B200M_TILE_N + b] = make_int2(sl.z, b * B200M_TILE_N < ns ? sl.z + nt : sl.z);
    for (int b = threadIdx.x; b < nb1; b += kRowsThreads)
        range1[sl.z / B200M_TILE_N + b] = make_int2(sl.x, b * B200M_TILE_N < nt ? sl.x + ns : sl.x);
}

}  // namespace

// A matcher-class plan with live counts: the device image of wide_batch_tables' host loop, from the live counts.
struct WideRowsArgs {
    const uint2 *kps, *rows;       // the caller's live counts
    const int4 *pinfo;             // [n_pairs] {source keypoint capacity, target keypoint capacity, scales, first entry of rows}
    const uint2 *rcap;             // [sum of scales] the bound sets' row capacities
    const int4 *slots;             // [n_scales][n_pairs] plan_rows_kernel's slot of every pair in every scale
    uint2 *eff;                    // [n_scales][n_pairs] the rows each scale's tables take (0 past the pair's live scales)
    uint2 *live_kps;               // [n_pairs] the keypoints the pair takes (0, 0 for a pair with a count above its capacity)
    int32_t *off0, *off1;          // [n_pairs + 1] the dense keypoint tables' offsets
    int2 *segs;                    // [n_pairs] the averages' segments
    GatherSet *gxyz, *gmap, *thr;  // [4][n_pairs] coordinates, [n_gmap] maps, [2][n_pairs] thresholds (or null)
    const int32_t *gmap_keys;      // [n_gmap][3] (side, scale, pair)
    char *d;                       // the layout's tables; per scale the int4 row table at d + o_rows[s]
    const long long *o_rows;
    unsigned long long *key;       // the first count above its capacity (~0: none)
    int n_pairs, n_scales, n_gmap;
};

namespace {

constexpr int kWideRowsThreads = 1024;

// One CTA.  Per pair: the capacity rule (a keypoint count above its capacity is keyed with scale 0xFFFF; a scale's row count
// with its scale), the live keypoints, and the rule of wide_batch_tables that a pair without source keypoints takes part in
// no scale.  Then the keypoint offsets as an exclusive scan, and every table that depends on them or on the live rows: the
// per-scale row tables, the averages' segments, and the row counts and destinations of the coordinate, map and threshold
// gathers.  The scale tables of batch.cu (packs, segment ranges) follow in plan_rows_kernel, once per scale.
__global__ void __launch_bounds__(kWideRowsThreads) plan_wide_rows_kernel(WideRowsArgs a) {
    __shared__ long long part[2][kWideRowsThreads];
    const int n = a.n_pairs, t = threadIdx.x;
    const int per = (n + kWideRowsThreads - 1) / kWideRowsThreads;
    const int i0 = min(n, t * per), i1 = min(n, i0 + per);
    long long sum[2] = {0, 0};
    for (int i = i0; i < i1; ++i) {
        const int4 pi = a.pinfo[i];
        const uint2 k = a.kps[i];
        unsigned long long key = ~0ull;
        if (k.x > (unsigned) pi.x || k.y > (unsigned) pi.y)
            key = (0xFFFFull << 48) | ((unsigned long long) i << 16) | (k.x > (unsigned) pi.x ? 2ull : 3ull);
        for (int s = 0; s < pi.z; ++s) {
            const uint2 r = a.rows[pi.w + s], c = a.rcap[pi.w + s];
            if (r.x > c.x || r.y > c.y)
                key = min(key, ((unsigned long long) s << 48) | ((unsigned long long) i << 16) | (r.x > c.x ? 2ull : 3ull));
        }
        if (key != ~0ull) atomicMin(a.key, key);
        const unsigned ns = key == ~0ull ? k.x : 0u, nt = key == ~0ull ? k.y : 0u;
        a.live_kps[i] = make_uint2(ns, nt);
        const int eff = ns ? pi.z : 0;
        for (int s = 0; s < a.n_scales; ++s) a.eff[(size_t) s * n + i] = s < eff ? a.rows[pi.w + s] : make_uint2(0u, 0u);
        sum[0] += ns;
        sum[1] += nt;
    }
    if (!a.d) return;   // no pair has source keypoint capacity and a scale: nothing is queued
    for (int side = 0; side < 2; ++side) part[side][t] = sum[side];
    __syncthreads();
    for (int o = 1; o < kWideRowsThreads; o <<= 1) {   // inclusive scan of the chunk sums
        long long v[2];
        for (int side = 0; side < 2; ++side) v[side] = t >= o ? part[side][t - o] : 0ll;
        __syncthreads();
        for (int side = 0; side < 2; ++side) part[side][t] += v[side];
        __syncthreads();
    }
    long long run[2] = {part[0][t] - sum[0], part[1][t] - sum[1]};
    for (int i = i0; i < i1; ++i) {
        const uint2 lk = a.live_kps[i];
        const int o0 = (int) run[0], o1 = (int) run[1];
        a.off0[i] = o0;
        a.off1[i] = o1;
        run[0] += lk.x;
        run[1] += lk.y;
        a.segs[i] = make_int2(o0, (int) lk.x);
        // coordinates of the pairs that take part: xyz_t, xyz_s, mov_s, mov_t (entries of unused tables are never launched)
        const int nt = lk.x ? (int) lk.y : 0;
        const int dst[4] = {o1, o0, o0, o1}, rows[4] = {nt, (int) lk.x, (int) lk.x, nt};
        for (int q = 0; q < 4; ++q) {
            a.gxyz[(size_t) q * n + i].dst_row = dst[q];
            a.gxyz[(size_t) q * n + i].rows = rows[q];
        }
        if (a.thr) {
            a.thr[i].dst_row = o0;
            a.thr[i].rows = (int) lk.x;
            a.thr[n + i].dst_row = o1;
            a.thr[n + i].rows = (int) lk.y;
        }
        for (int s = 0; s < a.n_scales; ++s) {
            int4 *rt = reinterpret_cast<int4 *>(a.d + a.o_rows[s]) + i;
            const uint2 e = a.eff[(size_t) s * n + i];
            rt->y = (int) e.x;
            rt->w = (int) e.y;
        }
    }
    if (t == kWideRowsThreads - 1) {
        a.off0[n] = (int) part[0][t];
        a.off1[n] = (int) part[1][t];
    }
    __syncthreads();   // eff[] of every pair is written
    for (int e = t; e < a.n_gmap; e += kWideRowsThreads) {
        const int side = a.gmap_keys[3 * e], s = a.gmap_keys[3 * e + 1], p = a.gmap_keys[3 * e + 2];
        const uint2 r = a.eff[(size_t) s * n + p];
        a.gmap[e].rows = (int) (side ? r.y : r.x);
    }
}

// *status = min(*status, *key): the finish step copied the bad-map key, this adds the first count above its capacity
__global__ void plan_status_merge_kernel(uint64_t *status, const unsigned long long *key) {
    if (*key < *status) *status = *key;
}

// A *_rows plan's run starts here, on the run's stream: the status word's reset, then the live-count tables.
int enqueue_rows(b200m_plan *pl) {
    b200m_ctx *ctx = pl->ctx;
    const BatchLayout &L = pl->L;
    if (pl->wide) {
        const WideLayout &W = pl->wide->layout;
        const WideRowsArgs &a = *pl->wr;
        CK(cudaMemsetAsync(a.key, 0xFF, sizeof(unsigned long long), ctx->stream));
        if (!a.n_pairs) return 0;
        plan_wide_rows_kernel<<<1, kWideRowsThreads, 0, ctx->stream>>>(a);
        CK(cudaGetLastError());
        ctx->stats.launches += 1;
        for (int s = 0; s < W.n_scales; ++s) {   // the scale tables are the plan's own (one buffer per scale)
            const BatchLayout &Ls = W.scale_tables[s];
            plan_rows_kernel<<<(unsigned) a.n_pairs, kRowsThreads, 0, ctx->stream>>>(
                a.eff + (size_t) s * a.n_pairs, a.slots + (size_t) s * a.n_pairs, const_cast<SetRef *>(Ls.sets[0]),
                const_cast<SetRef *>(Ls.sets[1]), nullptr, nullptr, const_cast<int2 *>(Ls.avg_segs),
                const_cast<int2 *>(Ls.seg[0].range), const_cast<int2 *>(Ls.seg[1].range), nullptr);
            CK(cudaGetLastError());
            ctx->stats.launches += 1;
        }
        return 0;
    }
    CK(cudaMemsetAsync(pl->status, 0xFF, sizeof(uint64_t), ctx->stream));
    const int n_pairs = (int) pl->pairs.size();
    if (!n_pairs) return 0;
    // the plan's own tables (stage_batch_tables put them in its context's ws_batch): writable here
    plan_rows_kernel<<<(unsigned) n_pairs, kRowsThreads, 0, ctx->stream>>>(
        reinterpret_cast<const uint2 *>(pl->rows), pl->slots.as<int4>(), const_cast<SetRef *>(L.sets[0]),
        const_cast<SetRef *>(L.sets[1]), const_cast<GatherSet *>(L.thr_sets[0]), const_cast<GatherSet *>(L.thr_sets[1]),
        const_cast<int2 *>(L.avg_segs), const_cast<int2 *>(L.seg[0].range), const_cast<int2 *>(L.seg[1].range),
        reinterpret_cast<unsigned long long *>(pl->status));
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

int enqueue(b200m_plan *pl) {
    b200m_ctx *ctx = pl->ctx;
    const unsigned long long *found, *bad = nullptr;
    const unsigned *counts;
    const float *avgs;
    int n_pairs, empty;
    if (pl->rows && enqueue_rows(pl)) return 1;
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
                                                                   pl->wide ? pl->status : nullptr);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    if (pl->wide && pl->wr) {
        plan_status_merge_kernel<<<1, 1, 0, ctx->stream>>>(pl->status, pl->wr->key);
        CK(cudaGetLastError());
        ctx->stats.launches += 1;
    }
    return 0;
}

// A matcher-class plan with live counts, after wide_batch_tables: the static tables of plan_wide_rows_kernel (per pair its
// capacities and scales, the bound row capacities, per scale every pair's slot) and its scratch, in one upload.
int wide_rows_tables(b200m_ctx *ctx, b200m_plan *pl) {
    const WideCall &c = pl->wide->call;
    WideLayout &W = pl->wide->layout;
    const int n = c.n_pairs, S = W.n_scales;
    std::vector<int4> pinfo(n);
    std::vector<uint2> rcap;
    std::vector<int4> slots((size_t) S * n);
    std::vector<GatherSet> thr(c.thr_src ? 2 * (size_t) n : 0);
    size_t start[2][32] = {};
    long long cs = 0, ct = 0;
    for (int i = 0; i < n; ++i) {
        const b200m_wide_pair &w = c.pairs[i];
        pinfo[i] = make_int4((int) w.n_src_kps, (int) w.n_tgt_kps, w.n_scales, (int) rcap.size());
        for (int s = 0; s < w.n_scales; ++s) rcap.push_back(make_uint2((unsigned) w.scales[s].n_src, (unsigned) w.scales[s].n_tgt));
        for (int s = 0; s < S; ++s) {   // wide_batch_tables' layout: a pair without source keypoint capacity takes no rows
            const bool has = w.n_src_kps && s < w.n_scales;
            const size_t ns = has ? w.scales[s].n_src : 0, nt = has ? w.scales[s].n_tgt : 0;
            slots[(size_t) s * n + i] = make_int4((int) start[0][s], (int) ns, (int) start[1][s], (int) nt);
            start[0][s] += pad_rows(ns);
            start[1][s] += pad_rows(nt);
        }
        if (c.thr_src) {
            thr[i] = GatherSet{c.thr_src + cs, 1, 0, 0, 0};
            thr[n + i] = GatherSet{c.thr_tgt + ct, 1, 0, 0, 0};
        }
        cs += (long long) w.n_src_kps;
        ct += (long long) w.n_tgt_kps;
    }
    std::vector<long long> o_rows(W.o_rows.begin(), W.o_rows.end());
    const size_t o_pinfo = 0, o_slots = align16(sizeof(int4) * n), o_thr = align16(o_slots + sizeof(int4) * slots.size());
    const size_t o_rcap = align16(o_thr + sizeof(GatherSet) * thr.size()), o_keys = align16(o_rcap + sizeof(uint2) * rcap.size());
    const size_t o_orows = align16(o_keys + sizeof(int32_t) * W.gmap_keys.size());
    const size_t o_eff = align16(o_orows + sizeof(long long) * o_rows.size()), o_live = align16(o_eff + sizeof(uint2) * S * n);
    const size_t o_key = align16(o_live + sizeof(uint2) * n), bytes = o_key + 16;
    std::vector<char> h(bytes, 0);
    auto put = [&](size_t o, const void *src, size_t b) { if (b) memcpy(h.data() + o, src, b); };
    put(o_pinfo, pinfo.data(), sizeof(int4) * n);
    put(o_slots, slots.data(), sizeof(int4) * slots.size());
    put(o_thr, thr.data(), sizeof(GatherSet) * thr.size());
    put(o_rcap, rcap.data(), sizeof(uint2) * rcap.size());
    put(o_keys, W.gmap_keys.data(), sizeof(int32_t) * W.gmap_keys.size());
    put(o_orows, o_rows.data(), sizeof(long long) * o_rows.size());
    CK(pl->slots.reserve(bytes));
    CK(cudaMemcpy(pl->slots.p, h.data(), bytes, cudaMemcpyHostToDevice));
    char *d = pl->slots.as<char>();
    WideRowsArgs &a = *(pl->wr = new WideRowsArgs());
    a.kps = reinterpret_cast<const uint2 *>(pl->kps);
    a.rows = reinterpret_cast<const uint2 *>(pl->rows);
    a.pinfo = reinterpret_cast<const int4 *>(d + o_pinfo);
    a.rcap = reinterpret_cast<const uint2 *>(d + o_rcap);
    a.slots = reinterpret_cast<const int4 *>(d + o_slots);
    a.eff = reinterpret_cast<uint2 *>(d + o_eff);
    a.live_kps = reinterpret_cast<uint2 *>(d + o_live);
    a.key = reinterpret_cast<unsigned long long *>(d + o_key);
    a.n_pairs = n;
    a.n_scales = S;
    if (S) {   // wide_batch_tables uploaded the layout's tables (W.d)
        a.d = W.d;
        a.off0 = reinterpret_cast<int32_t *>(W.d + W.o_off[0]);
        a.off1 = reinterpret_cast<int32_t *>(W.d + W.o_off[1]);
        a.segs = reinterpret_cast<int2 *>(W.d + W.o_segs);
        a.gxyz = reinterpret_cast<GatherSet *>(W.d + W.o_gxyz);
        a.gmap = reinterpret_cast<GatherSet *>(W.d + W.o_gmap);
        a.thr = c.thr_src ? reinterpret_cast<GatherSet *>(d + o_thr) : nullptr;
        a.gmap_keys = reinterpret_cast<const int32_t *>(d + o_keys);
        a.o_rows = reinterpret_cast<const long long *>(d + o_orows);
        a.n_gmap = (int) W.n_gmap;
        W.thr_sets = a.thr;
    }
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
    if (pl->wide && (pl->kps || pl->rows)) {   // the matcher-class *_rows creators
        if (pl->wide->call.n_pairs > 0 && (!pl->kps || !pl->rows)) return b200m_fail_msg(ctx, f + ": null kps / rows");
        if (check_device_ptr(ctx, f + ": kps", pl->kps) || check_device_ptr(ctx, f + ": rows", pl->rows)) return 1;
    } else if (!pl->wide && (pl->rows || pl->status)) {   // the k-list / match *_rows creators: both device words are required
        if (n_pairs > 0 && !pl->rows) return b200m_fail_msg(ctx, f + ": null rows");
        if (!pl->status) return b200m_fail_msg(ctx, f + ": null status");
        if (check_device_ptr(ctx, f + ": rows", pl->rows) || check_device_ptr(ctx, f + ": status", pl->status)) return 1;
    }
    b200m_ctx *own = nullptr;
    if (b200m_create(&own, ctx->device)) return b200m_fail_msg(ctx, f + ": " + b200m_last_error(nullptr));
    pl->ctx = own;
    own->device_prepare = true;
    own->stream = ctx->stream;   // creation runs on the caller's stream; every run names its own
    if (pl->wide) {
        if (wide_batch_tables(own, pl->wide->call, &pl->wide->layout, true)) return b200m_fail_msg(ctx, own->err);
        if (pl->rows && wide_rows_tables(own, pl)) return b200m_fail_msg(ctx, own->err);
    } else if (stage_batch_tables(own, fn, p, pl->pairs.data(), n_pairs, pl->stride_bytes, pl->dim, &pl->L, true, pl->thr_src,
                                  pl->thr_tgt)) {
        return b200m_fail_msg(ctx, own->err);
    }
    if (!pl->match && pl->L.real_src && (!pl->idx || !pl->dist || !pl->count))
        return b200m_fail_msg(ctx, f + ": null output pointer");
    if (pl->rows && n_pairs) {   // every pair's slot: where its rows start on both sides and how many it may have
        std::vector<int4> slots(n_pairs);
        int s0 = 0, t0 = 0;
        for (int i = 0; i < n_pairs; ++i) {
            const b200m_pair &q = pl->pairs[i];
            slots[i] = make_int4(s0, (int) q.n_src, t0, (int) q.n_tgt);
            s0 += (int) pad_rows(q.n_src);
            t0 += (int) pad_rows(q.n_tgt);
        }
        cudaError_t ce = pl->slots.reserve(sizeof(int4) * n_pairs);
        if (ce == cudaSuccess) ce = cudaMemcpy(pl->slots.p, slots.data(), sizeof(int4) * n_pairs, cudaMemcpyHostToDevice);
        if (ce != cudaSuccess) return b200m_fail(ctx, "cudaMemcpy(plan slots)", ce, __FILE__, __LINE__);
    }
    // every workspace grows to its shape-determined size here, and every kernel module is loaded before any capture
    if (enqueue(pl)) return b200m_fail_msg(ctx, own->err);
    const cudaError_t e = cudaStreamSynchronize(own->stream);
    if (e != cudaSuccess) return b200m_fail(ctx, "cudaStreamSynchronize(plan run)", e, __FILE__, __LINE__);
    // the creation run is synchronised anyway: a bad map entry or a live count above its capacity fails it, as a bad map
    // entry fails the device form
    if (pl->status) {
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
              float *d_avg, uint64_t *d_n_out, uint64_t *d_status, const uint32_t *d_kps, const uint32_t *d_rows,
              b200m_plan **out) {
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
    pl->kps = d_kps;
    pl->rows = d_rows;
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

int b200m_plan_knn_batch_rows(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes,
                              int dim, int32_t *d_idx, float *d_dist, int32_t *d_count, const uint32_t *d_rows,
                              uint64_t *d_status, b200m_plan **plan) {
    b200m_plan *pl = new b200m_plan();
    pl->idx = d_idx;
    pl->dist = d_dist;
    pl->count = d_count;
    pl->rows = d_rows;
    pl->status = d_status;
    return make_plan(ctx, "b200m_plan_knn_batch_rows", pl, p, pairs, n_pairs, stride_bytes, dim, plan);
}

int b200m_plan_match_batch_rows(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes,
                                int dim, const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out, const uint32_t *d_rows, uint64_t *d_status,
                                b200m_plan **plan) {
    b200m_plan *pl = new b200m_plan();
    pl->match = true;
    pl->thr_src = d_thr_src;
    pl->thr_tgt = d_thr_tgt;
    pl->out = d_out;
    pl->cap = cap;
    pl->offsets = d_offsets;
    pl->avg = d_avg;
    pl->n_out = d_n_out;
    pl->rows = d_rows;
    pl->status = d_status;
    return make_plan(ctx, "b200m_plan_match_batch_rows", pl, p, pairs, n_pairs, stride_bytes, dim, plan);
}

int b200m_plan_match_multiscale_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs, int n_pairs,
                                      size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k, const float *d_thr_src,
                                      const float *d_thr_tgt, b200m_corr *d_out, size_t cap, uint64_t *d_offsets, float *d_avg,
                                      uint64_t *d_n_out, uint64_t *d_status, b200m_plan **plan) {
    return wide_plan(ctx, "b200m_plan_match_multiscale_batch", false, p, pairs, nullptr, n_pairs, stride_bytes, dim,
                     xyz_stride_bytes, cluster_k, 0.f, d_thr_src, d_thr_tgt, d_out, cap, d_offsets, d_avg, d_n_out, d_status, nullptr,
                     nullptr, plan);
}

int b200m_plan_match_multiscale_local_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                            const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim,
                                            size_t xyz_stride_bytes, int cluster_k, float match_search_radius,
                                            const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                            uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out, uint64_t *d_status,
                                            b200m_plan **plan) {
    return wide_plan(ctx, "b200m_plan_match_multiscale_local_batch", true, p, pairs, locals, n_pairs, stride_bytes, dim,
                     xyz_stride_bytes, cluster_k, match_search_radius, d_thr_src, d_thr_tgt, d_out, cap, d_offsets, d_avg, d_n_out,
                     d_status, nullptr, nullptr, plan);
}

int b200m_plan_match_multiscale_batch_rows(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs, int n_pairs,
                                           size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k,
                                           const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                           uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out, uint64_t *d_status,
                                           const uint32_t *d_kps, const uint32_t *d_rows, b200m_plan **plan) {
    return wide_plan(ctx, "b200m_plan_match_multiscale_batch_rows", false, p, pairs, nullptr, n_pairs, stride_bytes, dim,
                     xyz_stride_bytes, cluster_k, 0.f, d_thr_src, d_thr_tgt, d_out, cap, d_offsets, d_avg, d_n_out, d_status, d_kps,
                     d_rows, plan);
}

int b200m_plan_match_multiscale_local_batch_rows(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                 const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim,
                                                 size_t xyz_stride_bytes, int cluster_k, float match_search_radius,
                                                 const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                                 uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out, uint64_t *d_status,
                                                 const uint32_t *d_kps, const uint32_t *d_rows, b200m_plan **plan) {
    return wide_plan(ctx, "b200m_plan_match_multiscale_local_batch_rows", true, p, pairs, locals, n_pairs, stride_bytes, dim,
                     xyz_stride_bytes, cluster_k, match_search_radius, d_thr_src, d_thr_tgt, d_out, cap, d_offsets, d_avg, d_n_out,
                     d_status, d_kps, d_rows, plan);
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
        cudaSetDevice(plan->ctx->device);
        plan->slots.release();
        plan->ctx->stream = plan->ctx->own_stream;
        b200m_destroy(plan->ctx);
    }
    delete plan->wide;
    delete plan->wr;
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
