// batch.cu -- many independent (source, target) pairs in one call: b200m_knn_batch and b200m_match_batch.
//
// The reference answers one pair per FeatureBasedMatcher::match() call; at keypoint-set sizes (20k rows) a single pair
// is about one wave of the candidate kernel and the fixed cost of a call (16 launches, 3 host round trips) dominates.
// Here every pair's rows go into ONE padded concatenation per side and the ordinary kNN driver runs once per direction:
//
//   layout      pair p's rows start at a multiple of B200M_TILE_N (256 = a train tile = the query rows of one CTA pair)
//               on both sides; the rows in between are 0xFF bytes -- NaN floats, so the pack marks them invalid: the pack
//               statistics skip them, pack_operands gives them the sentinel norm, and the re-rank drops their non-finite
//               distances against valid[] -- they can never be returned.
//   segments    seg_range[query row / 256] = {first, end} train row of that query block's pair (one table per
//               direction).  The candidate kernel sweeps only those train tiles, the exact kernels only those rows.
//   filter      runs on the padded global row numbers (forward lists carry global target rows, the reverse table is
//               indexed by them), so the mutual test is the single-pair one; gap rows have empty lists.
//   output      records ascend in global source row, i.e. they are already in pair order; one kernel makes their
//               indices pair-local and counts them per pair, the host turns the counts into offsets.  The average is
//               average_kernel's sequential FP32 chain over each pair's own rows (one CTA per pair).
//
// Pair p's output is, byte for byte, what b200m_upload(0, src_p) + b200m_upload(1, tgt_p) + b200m_match / b200m_knn give:
// one centre, scale and norm bound serve the whole batch, which DESIGN.md section 4 admits (any centre and scale that fit
// FP16, any upper bound on |b16|); only the candidate counts can differ, never the exact re-rank's answer.
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "internal.cuh"

#define REQUIRE_CTX()                                             \
    do {                                                          \
        if (!ctx) return b200m_fail_msg(nullptr, "null context"); \
        CK(cudaSetDevice(ctx->device));                           \
    } while (0)

namespace {

__global__ void localize_lists_kernel(const int32_t *__restrict__ idx, const float *__restrict__ dist,
                                      const int32_t *__restrict__ cnt, size_t n_rows, int k,
                                      const int32_t *__restrict__ block_pair, const int4 *__restrict__ pair_info,
                                      int32_t *__restrict__ o_idx, float *__restrict__ o_dist, int32_t *__restrict__ o_cnt) {
    const size_t r = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int4 pi = pair_info[block_pair[r / B200M_TILE_N]];
    const size_t local = r - (size_t) pi.x;
    if (local >= (size_t) pi.z) return;   // gap row
    const size_t dense = (size_t) pi.w + local;
    for (int m = 0; m < k; ++m) {
        const int32_t j = idx[r * k + m];
        o_idx[dense * k + m] = j >= 0 ? j - pi.y : -1;
        o_dist[dense * k + m] = dist[r * k + m];
    }
    o_cnt[dense] = cnt[r];
}

__global__ void localize_records_kernel(b200m_corr *__restrict__ rec, const unsigned long long *__restrict__ n_out, size_t cap,
                                        const int32_t *__restrict__ block_pair, const int4 *__restrict__ pair_info,
                                        unsigned *__restrict__ counts) {
    const size_t n = *n_out < cap ? (size_t) *n_out : cap;
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        b200m_corr c = rec[i];
        const int p = block_pair[c.index_query / B200M_TILE_N];
        const int4 pi = pair_info[p];
        c.index_query -= pi.x;
        c.index_match -= pi.y;
        rec[i] = c;
        // records are sorted by pair: neighbouring lanes mostly share one, one atomic per run
        const unsigned peers = __match_any_sync(__activemask(), p);
        if ((int) (threadIdx.x & 31) == __ffs((int) peers) - 1) atomicAdd(counts + p, (unsigned) __popc(peers));
    }
}

// One CTA column per set (blockIdx.x), its rows spread over blockIdx.y and the threads: w words of every row.
__global__ void gather_sets_kernel(const GatherSet *__restrict__ sets, int w, size_t dst_stride, uint32_t *__restrict__ dst) {
    const GatherSet g = sets[blockIdx.x];
    const uint32_t *src = static_cast<const uint32_t *>(g.src);
    for (long long r = (long long) blockIdx.y * blockDim.x + threadIdx.x; r < g.rows; r += (long long) gridDim.y * blockDim.x) {
        uint32_t *d = dst + (size_t) (g.dst_row + r) * dst_stride;
        if (!src) {
            d[0] = (uint32_t) r;
            continue;
        }
        for (int c = 0; c < w; ++c) d[c] = __ldg(src + r * g.src_stride + c);
    }
}

}  // namespace

cudaError_t launch_gather_sets(const GatherSet *d_sets, int n_sets, size_t max_rows, int w, size_t dst_stride_words, void *dst,
                               cudaStream_t st) {
    if (n_sets == 0 || max_rows == 0) return cudaSuccess;
    const unsigned chunks = (unsigned) std::min<size_t>((max_rows + 255) / 256, 32);
    gather_sets_kernel<<<dim3((unsigned) n_sets, chunks), 256, 0, st>>>(d_sets, w, dst_stride_words, static_cast<uint32_t *>(dst));
    return cudaGetLastError();
}

int check_device_ptr(b200m_ctx *ctx, const std::string &where, const void *ptr) {
    if (!ptr) return 0;
    cudaPointerAttributes a;
    const cudaError_t e = cudaPointerGetAttributes(&a, ptr);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return b200m_fail_msg(ctx, where + " is not device memory (" + cudaGetErrorString(e) + ")");
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged)
        return b200m_fail_msg(ctx, where + " is not device memory (" +
                                       (a.type == cudaMemoryTypeHost ? "page-locked host memory" : "host memory") + ")");
    if (a.device != ctx->device)
        return b200m_fail_msg(ctx, where + " is memory of device " + std::to_string(a.device) + ", the context's device is " +
                                       std::to_string(ctx->device));
    return 0;
}

// Validates the batch and uploads the segment tables.  dev: the descriptor pointers are device pointers, checked here and
// read in place by the segmented pack (the per-pair SetRef tables and side 1's block table go up with the other tables).
int stage_batch_tables(b200m_ctx *ctx, const char *fn, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                       size_t stride_bytes, int dim, BatchLayout *L, bool dev, const float *d_thr_src, const float *d_thr_tgt,
                       DevBuf *dst) {
    const std::string f(fn);
    if (n_pairs < 0) return b200m_fail_msg(ctx, f + ": n_pairs < 0");
    if (n_pairs > 0 && !pairs) return b200m_fail_msg(ctx, f + ": null pairs");
    if (dim < 1 || dim > B200M_MAX_DIM) return b200m_fail_msg(ctx, f + ": dim out of range [1, 2048]");
    if (stride_bytes % 4 != 0 || stride_bytes < (size_t) dim * 4)
        return b200m_fail_msg(ctx, f + ": stride_bytes must be a multiple of 4 and >= 4*dim");
    if (p->precision == B200M_PREC_TC_F16 && !ctx->tc_pair && ctx->tc_cluster == 4)
        return b200m_fail_msg(ctx, f + ": B200M_TC_MODE=mcast with B200M_TC_CLUSTER=4 is not supported by batch calls (a cluster "
                                       "of four CTAs would span two pairs)");
    std::vector<size_t> start[2];
    start[0].resize(n_pairs);
    start[1].resize(n_pairs);
    size_t max_rows[2] = {0, 0};
    for (int i = 0; i < n_pairs; ++i) {
        const size_t n[2] = {pairs[i].n_src, pairs[i].n_tgt};
        const float *base[2] = {pairs[i].src, pairs[i].tgt};
        for (int s = 0; s < 2; ++s) {
            if (n[s] && !base[s])
                return b200m_fail_msg(ctx, f + ": null descriptor pointer in pair " + std::to_string(i + L->pair_base));
            if (dev && n[s] && check_device_ptr(ctx, f + ": pair " + std::to_string(i) + ": " + (s ? "tgt" : "src"), base[s]))
                return 1;
            start[s][i] = L->n_rows[s];
            L->n_rows[s] += pad_rows(n[s]);
            if (n[s] > max_rows[s]) max_rows[s] = n[s];
        }
        L->real_src += n[0];
    }
    if (L->n_rows[0] >= (size_t) 1 << 31 || L->n_rows[1] >= (size_t) 1 << 31)
        return b200m_fail_msg(ctx, f + ": more than 2^31-1 rows per side after padding (indices are int32, as pcl::index_t)");
    // segment tables, pair bookkeeping and the result area in one device buffer, the tables in one upload
    const size_t nb[2] = {L->n_rows[0] / B200M_TILE_N, L->n_rows[1] / B200M_TILE_N};
    const size_t o_range0 = 0, o_range1 = align16(o_range0 + sizeof(int2) * nb[0]);
    const size_t o_bpair = align16(o_range1 + sizeof(int2) * nb[1]);
    const size_t o_info = align16(o_bpair + sizeof(int32_t) * nb[0]);
    const size_t o_avgs = align16(o_info + sizeof(int4) * n_pairs);
    // device calls only: side 1's block -> pair table and both sides' SetRef tables
    const size_t o_bpair1 = align16(o_avgs + sizeof(int2) * n_pairs);
    const size_t o_sets0 = align16(o_bpair1 + (dev ? sizeof(int32_t) * nb[1] : 0));
    const size_t o_sets1 = o_sets0 + (dev ? sizeof(SetRef) * n_pairs : 0);
    // ... and the gather tables of b200m_match_batch_device's thresholds
    const bool thr = dev && d_thr_src;
    const size_t o_thr0 = align16(o_sets1 + (dev ? sizeof(SetRef) * n_pairs : 0));
    const size_t o_thr1 = o_thr0 + (thr ? sizeof(GatherSet) * n_pairs : 0);
    const size_t o_res = align16(o_thr1 + (thr ? sizeof(GatherSet) * n_pairs : 0));
    L->result_bytes = 16 + align16(sizeof(unsigned) * n_pairs) + sizeof(float) * n_pairs;
    std::vector<char> h(o_res);
    int2 *range0 = reinterpret_cast<int2 *>(h.data() + o_range0), *range1 = reinterpret_cast<int2 *>(h.data() + o_range1);
    int32_t *bpair = reinterpret_cast<int32_t *>(h.data() + o_bpair);
    int4 *info = reinterpret_cast<int4 *>(h.data() + o_info);
    int2 *avg_segs = reinterpret_cast<int2 *>(h.data() + o_avgs);
    int32_t *bpair1 = reinterpret_cast<int32_t *>(h.data() + o_bpair1);
    SetRef *sets[2] = {reinterpret_cast<SetRef *>(h.data() + o_sets0), reinterpret_cast<SetRef *>(h.data() + o_sets1)};
    GatherSet *thr_sets[2] = {reinterpret_cast<GatherSet *>(h.data() + o_thr0), reinterpret_cast<GatherSet *>(h.data() + o_thr1)};
    size_t dense = 0, dense_t = 0;
    for (int i = 0; i < n_pairs; ++i) {
        const int s0 = (int) start[0][i], t0 = (int) start[1][i], ns = (int) pairs[i].n_src, nt = (int) pairs[i].n_tgt;
        if (thr) {   // the thresholds are concatenated in pair order, dense
            thr_sets[0][i] = GatherSet{d_thr_src + dense, 1, s0, ns, 0};
            thr_sets[1][i] = GatherSet{d_thr_tgt + dense_t, 1, t0, nt, 0};
            dense_t += (size_t) nt;
        }
        for (size_t b = s0 / B200M_TILE_N; b < (s0 + pad_rows(ns)) / B200M_TILE_N; ++b) {
            range0[b] = make_int2(t0, t0 + nt);
            bpair[b] = i;
        }
        for (size_t b = t0 / B200M_TILE_N; b < (t0 + pad_rows(nt)) / B200M_TILE_N; ++b) {
            range1[b] = make_int2(s0, s0 + ns);
            if (dev) bpair1[b] = i;
        }
        if (dev) {
            sets[0][i] = SetRef{pairs[i].src, s0, ns};
            sets[1][i] = SetRef{pairs[i].tgt, t0, nt};
        }
        info[i] = make_int4(s0, t0, ns, (int) dense);
        avg_segs[i] = make_int2(s0, ns);
        dense += (size_t) ns;
    }
    if (!dst) dst = &ctx->ws_batch;
    CK(dst->reserve(o_res + L->result_bytes));
    char *d = dst->as<char>();
    cudaStream_t st = ctx->stream;
    CK(cudaMemcpyAsync(d, h.data(), o_res, cudaMemcpyHostToDevice, st));
    L->seg[0] = SegTable{reinterpret_cast<const int2 *>(d + o_range0), (int) (pad_rows(max_rows[1]) / B200M_TILE_N)};
    L->seg[1] = SegTable{reinterpret_cast<const int2 *>(d + o_range1), (int) (pad_rows(max_rows[0]) / B200M_TILE_N)};
    L->block_pair = reinterpret_cast<const int32_t *>(d + o_bpair);
    L->pair_info = reinterpret_cast<const int4 *>(d + o_info);
    L->avg_segs = reinterpret_cast<const int2 *>(d + o_avgs);
    L->n_out = reinterpret_cast<unsigned long long *>(d + o_res);
    L->counts = reinterpret_cast<unsigned *>(d + o_res + 16);
    L->avgs = reinterpret_cast<float *>(d + o_res + 16 + align16(sizeof(unsigned) * n_pairs));
    if (thr) {
        L->thr_sets[0] = reinterpret_cast<const GatherSet *>(d + o_thr0);
        L->thr_sets[1] = reinterpret_cast<const GatherSet *>(d + o_thr1);
    }
    L->max_rows[0] = max_rows[0];
    L->max_rows[1] = max_rows[1];
    if (dev) {
        L->seg_blk[0] = L->block_pair;
        L->seg_blk[1] = reinterpret_cast<const int32_t *>(d + o_bpair1);
        L->sets[0] = reinterpret_cast<const SetRef *>(d + o_sets0);
        L->sets[1] = reinterpret_cast<const SetRef *>(d + o_sets1);
    }
    return 0;
}

int stage_batch_pack(b200m_ctx *ctx, const b200m_pair *pairs, int n_pairs, size_t stride_bytes, int dim, const BatchLayout &L,
                     bool dev) {
    if (dev) {   // the segmented pack reads every pair's rows where they are and writes the gap rows itself
        for (int s = 0; s < 2; ++s)
            if (upload_common(ctx, s, nullptr, L.n_rows[s], stride_bytes, dim, 0, L.seg_blk[s], L.sets[s])) return 1;
        return 0;
    }
    // descriptors: gap bytes 0xFF (NaN rows), then every pair's rows at its offset -- (n - 1) * stride + dim floats, as
    // b200m_upload copies: the caller owns only `dim` floats of a set's last row
    cudaStream_t st = ctx->stream;
    for (int s = 0; s < 2; ++s) {
        Side &sd = ctx->side[s];
        if (L.n_rows[s]) {
            CK(sd.staging.reserve(L.n_rows[s] * stride_bytes));
            CK(cudaMemsetAsync(sd.staging.p, 0xFF, L.n_rows[s] * stride_bytes, st));
            size_t start = 0;   // pair i's first padded row
            for (int i = 0; i < n_pairs; ++i) {
                const size_t n = s ? pairs[i].n_tgt : pairs[i].n_src;
                const size_t first = start;
                start += pad_rows(n);
                if (!n) continue;
                const float *src = s ? pairs[i].tgt : pairs[i].src;
                const size_t bytes = (n - 1) * stride_bytes + (size_t) dim * 4;
                char *dst = sd.staging.as<char>() + first * stride_bytes;
                if (bytes >= ((size_t) 32 << 20) && is_pageable(src)) {
                    if (staged_h2d(ctx, dst, src, bytes)) return 1;
                } else {
                    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
                }
            }
        }
        if (upload_common(ctx, s, sd.staging.as<float>(), L.n_rows[s], stride_bytes, dim, 0)) return 1;
    }
    return 0;
}

int stage_batch(b200m_ctx *ctx, const char *fn, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                size_t stride_bytes, int dim, BatchLayout *L, bool dev, const float *d_thr_src, const float *d_thr_tgt) {
    if (stage_batch_tables(ctx, fn, p, pairs, n_pairs, stride_bytes, dim, L, dev, d_thr_src, d_thr_tgt)) return 1;
    return stage_batch_pack(ctx, pairs, n_pairs, stride_bytes, dim, *L, dev);
}

int knn_batch_lists(b200m_ctx *ctx, const b200m_params *p, const BatchLayout &L, int32_t *o_idx, float *o_dist, int32_t *o_cnt) {
    const int k = p->k;
    const size_t S = L.n_rows[0];
    CK(ctx->ws_fidx.reserve(sizeof(int32_t) * S * k));
    CK(ctx->ws_fdist.reserve(sizeof(float) * S * k));
    CK(ctx->ws_fcnt.reserve(sizeof(int32_t) * S));
    if (b200m_knn_rows(ctx, p, 0, 0, S, nullptr, ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>(),
                       &L.seg[0]))
        return 1;
    localize_lists_kernel<<<(unsigned) ((S + 255) / 256), 256, 0, ctx->stream>>>(
        ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>(), S, k, L.block_pair, L.pair_info, o_idx,
        o_dist, o_cnt);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

int match_batch_records(b200m_ctx *ctx, const b200m_params *p, const BatchLayout &L, const b200m_pair *pairs, int n_pairs,
                        bool dev, const float *thr_src, const float *thr_tgt, bool want_avg) {
    const int k = p->k;
    const bool mutual = p->mode == B200M_MODE_MUTUAL || p->mode == B200M_MODE_RATIO_MUTUAL;
    const size_t S = L.n_rows[0], T = L.n_rows[1];
    cudaStream_t st = ctx->stream;
    CK(ctx->ws_fidx.reserve(sizeof(int32_t) * S * k));
    CK(ctx->ws_fdist.reserve(sizeof(float) * S * k));
    CK(ctx->ws_fcnt.reserve(sizeof(int32_t) * S));
    if (b200m_knn_rows(ctx, p, 0, 0, S, nullptr, ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>(),
                       &L.seg[0]))
        return 1;
    if (mutual && T) {   // every target row: the masked reverse pass's compact row list would mix pairs inside a tile
        CK(ctx->ws_ridx.reserve(sizeof(int32_t) * T * k));
        CK(ctx->ws_rdist.reserve(sizeof(float) * T * k));
        CK(ctx->ws_rcnt.reserve(sizeof(int32_t) * T));
        if (b200m_knn_rows(ctx, p, 1, 0, T, nullptr, ctx->ws_ridx.as<int32_t>(), ctx->ws_rdist.as<float>(), ctx->ws_rcnt.as<int32_t>(),
                           &L.seg[1]))
            return 1;
    }
    const float *d_thr_s = nullptr, *d_thr_t = nullptr;
    if (thr_src && T && dev) {   // the gather kernel files the device thresholds in the padded layout
        CK(ctx->ws_thr[0].reserve(sizeof(float) * S));
        CK(ctx->ws_thr[1].reserve(sizeof(float) * T));
        for (int s = 0; s < 2; ++s) {
            CK(launch_gather_sets(L.thr_sets[s], n_pairs, L.max_rows[s], 1, 1, ctx->ws_thr[s].p, st));
            ctx->stats.launches += 1;
        }
        d_thr_s = ctx->ws_thr[0].as<float>();
        d_thr_t = ctx->ws_thr[1].as<float>();
    } else if (thr_src && T) {   // the pairs' thresholds in the padded layout (gap rows never produce a record)
        std::vector<float> hs(S, 0.f), ht(T, 0.f);
        size_t cs = 0, ct = 0, os = 0, ot = 0;
        for (int i = 0; i < n_pairs; ++i) {
            const size_t ns = pairs[i].n_src, nt = pairs[i].n_tgt;
            if (ns) memcpy(hs.data() + os, thr_src + cs, sizeof(float) * ns);
            if (nt) memcpy(ht.data() + ot, thr_tgt + ct, sizeof(float) * nt);
            cs += ns;
            ct += nt;
            os += pad_rows(ns);
            ot += pad_rows(nt);
        }
        CK(ctx->ws_thr[0].reserve(sizeof(float) * S));
        CK(ctx->ws_thr[1].reserve(sizeof(float) * T));
        CK(cudaMemcpyAsync(ctx->ws_thr[0].p, hs.data(), sizeof(float) * S, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->ws_thr[1].p, ht.data(), sizeof(float) * T, cudaMemcpyHostToDevice, st));
        d_thr_s = ctx->ws_thr[0].as<float>();
        d_thr_t = ctx->ws_thr[1].as<float>();
    }
    const size_t kk = (p->mode == B200M_MODE_MUTUAL) ? (size_t) k : 1;
    const size_t max_out = S * kk;
    CK(ctx->ws_corr.reserve(sizeof(b200m_corr) * max_out));
    if (b200m_filter_device(ctx, p, 0, S, ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>(),
                            ctx->ws_ridx.as<int32_t>(), ctx->ws_rdist.as<float>(), ctx->ws_rcnt.as<int32_t>(), mutual ? T : 0,
                            d_thr_s, d_thr_t, ctx->ws_corr.as<b200m_corr>(), max_out, L.n_out, nullptr))
        return 1;
    CK(cudaMemsetAsync(L.counts, 0, sizeof(unsigned) * n_pairs, st));
    if (want_avg) {
        CK(launch_average_segments(ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>(), L.avg_segs, n_pairs, k, L.avgs, st));
        ctx->stats.launches += 1;
    }
    localize_records_kernel<<<(unsigned) ctx->sm_count * 4, 256, 0, st>>>(ctx->ws_corr.as<b200m_corr>(), L.n_out, max_out,
                                                                          L.block_pair, L.pair_info, L.counts);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

namespace {

// dev: b200m_knn_batch_device (device descriptors, the k-lists are written to the caller's device arrays in place)
// r: a range of a group call (multi.cu), or NULL
int knn_batch(b200m_ctx *ctx, const char *fn, bool dev, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
              size_t stride_bytes, int dim, int32_t *idx, float *dist, int32_t *count, BatchRange *r = nullptr) {
    REQUIRE_CTX();
    if (check_params(ctx, p)) return 1;
    const std::string f(fn);
    if (dev && (check_device_ptr(ctx, f + ": idx", idx) || check_device_ptr(ctx, f + ": dist", dist) ||
                check_device_ptr(ctx, f + ": count", count)))
        return 1;
    BatchLayout L;
    if (r) L.pair_base = r->pair_base;
    if (stage_batch(ctx, fn, p, pairs, n_pairs, stride_bytes, dim, &L, dev)) return 1;
    if (r) r->validated = true;
    if (L.real_src == 0) return 0;
    if (!idx || !dist || !count) return b200m_fail_msg(ctx, f + ": null output pointer");
    // the pairs' real rows back to back, with pair-local train indices (a device call writes the caller's arrays directly,
    // a host call the reverse-table buffers, which are free here)
    if (dev) return knn_batch_lists(ctx, p, L, idx, dist, count);
    const int k = p->k;
    const size_t R = L.real_src;
    cudaStream_t st = ctx->stream;
    CK(ctx->ws_ridx.reserve(sizeof(int32_t) * R * k));
    CK(ctx->ws_rdist.reserve(sizeof(float) * R * k));
    CK(ctx->ws_rcnt.reserve(sizeof(int32_t) * R));
    if (knn_batch_lists(ctx, p, L, ctx->ws_ridx.as<int32_t>(), ctx->ws_rdist.as<float>(), ctx->ws_rcnt.as<int32_t>())) return 1;
    CK(cudaMemcpyAsync(idx, ctx->ws_ridx.p, sizeof(int32_t) * R * k, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(dist, ctx->ws_rdist.p, sizeof(float) * R * k, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(count, ctx->ws_rcnt.p, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

// dev: b200m_match_batch_device (device descriptors and thresholds, records to the caller's device buffer)
int match_batch(b200m_ctx *ctx, const char *fn, bool dev, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                size_t stride_bytes, int dim, const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap,
                size_t *offsets, float *avg, BatchRange *r = nullptr) {
    REQUIRE_CTX();
    if (check_params(ctx, p)) return 1;
    const std::string f(fn);
    if (p->mode == B200M_MODE_KNN_ONLY) return b200m_fail_msg(ctx, f + ": use b200m_knn_batch for raw k-lists");
    if (p->mode == B200M_MODE_CLUSTER)
        return b200m_fail_msg(ctx, f + ": the cluster filter needs keypoint coordinates, use b200m_match_cluster");
    if (!offsets) return b200m_fail_msg(ctx, f + ": null offsets");
    if ((thr_src == nullptr) != (thr_tgt == nullptr))
        return b200m_fail_msg(ctx, f + ": give both threshold arrays or neither");
    if (dev && (check_device_ptr(ctx, f + ": thr_src", thr_src) || check_device_ptr(ctx, f + ": thr_tgt", thr_tgt) ||
                check_device_ptr(ctx, f + ": out", out)))
        return 1;
    for (int i = 0; i <= n_pairs; ++i) offsets[i] = 0;
    BatchLayout L;
    if (r) L.pair_base = r->pair_base;
    if (stage_batch(ctx, fn, p, pairs, n_pairs, stride_bytes, dim, &L, dev, thr_src, thr_tgt)) return 1;
    if (r) r->validated = true;
    if (L.real_src == 0) {
        if (avg)
            for (int i = 0; i < n_pairs; ++i) avg[i] = 3.402823466e+38F;   // FLT_MAX, reference include/matching.h:41
        return 0;
    }
    if (match_batch_records(ctx, p, L, pairs, n_pairs, dev, thr_src, thr_tgt, avg != nullptr)) return 1;
    cudaStream_t st = ctx->stream;
    std::vector<char> res(L.result_bytes);
    CK(cudaMemcpyAsync(res.data(), L.n_out, L.result_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    unsigned long long n;
    memcpy(&n, res.data(), sizeof(n));
    const unsigned *cnt = reinterpret_cast<const unsigned *>(res.data() + 16);
    for (int i = 0; i < n_pairs; ++i) offsets[i + 1] = offsets[i] + cnt[i];
    if (avg) memcpy(avg, res.data() + 16 + align16(sizeof(unsigned) * n_pairs), sizeof(float) * n_pairs);
    if (n > cap) return b200m_fail_msg(ctx, f + ": output capacity too small (" + std::to_string(n) + " correspondences)");
    if (n) {
        if (!out) return b200m_fail_msg(ctx, f + ": null output buffer");
        if (dev) {   // stream-ordered: the caller's next work on the stream sees the records
            CK(cudaMemcpyAsync(out, ctx->ws_corr.p, sizeof(b200m_corr) * n, cudaMemcpyDeviceToDevice, st));
            return 0;
        }
        CK(cudaMemcpyAsync(out, ctx->ws_corr.p, sizeof(b200m_corr) * n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return 0;
}

}  // namespace

int knn_batch_host(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes, int dim,
                   int32_t *idx, float *dist, int32_t *count, BatchRange *r) {
    return knn_batch(ctx, "b200m_knn_batch", false, p, pairs, n_pairs, stride_bytes, dim, idx, dist, count, r);
}

int match_batch_host(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes, int dim,
                     const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap, size_t *offsets, float *avg,
                     BatchRange *r) {
    return match_batch(ctx, "b200m_match_batch", false, p, pairs, n_pairs, stride_bytes, dim, thr_src, thr_tgt, out, cap, offsets,
                       avg, r);
}

extern "C" {

int b200m_knn_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes, int dim,
                    int32_t *idx, float *dist, int32_t *count) {
    return knn_batch_host(ctx, p, pairs, n_pairs, stride_bytes, dim, idx, dist, count, nullptr);
}

int b200m_knn_batch_device(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes,
                           int dim, int32_t *d_idx, float *d_dist, int32_t *d_count) {
    return knn_batch(ctx, "b200m_knn_batch_device", true, p, pairs, n_pairs, stride_bytes, dim, d_idx, d_dist, d_count);
}

int b200m_match_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes, int dim,
                      const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap, size_t *offsets, float *avg) {
    return match_batch_host(ctx, p, pairs, n_pairs, stride_bytes, dim, thr_src, thr_tgt, out, cap, offsets, avg, nullptr);
}

int b200m_match_batch_device(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs, size_t stride_bytes,
                             int dim, const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap, size_t *offsets,
                             float *avg) {
    return match_batch(ctx, "b200m_match_batch_device", true, p, pairs, n_pairs, stride_bytes, dim, d_thr_src, d_thr_tgt, d_out, cap,
                       offsets, avg);
}

}  // extern "C"
