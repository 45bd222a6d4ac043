// wide_batch.cu -- b200m_match_multiscale_batch: the matcher classes at the WIDE seam (wide.cu) for many independent
// (source, target) cloud pairs in one call.  Pair p's records and average equal, byte for byte, what
// b200m_match_multiscale returns for that pair alone, with pair-local keypoint ids.
//
//   per scale s     every pair's scale-s descriptor sets go into the padded layout of batch.cu (stage_batch; a pair with
//                   fewer scales gives empty sets), and the kNN driver runs once per direction over all pairs with the
//                   per-direction segment table -- forward, and for the two-way matchers the whole reverse pass (a masked
//                   one would mix pairs inside a tile, as b200m_match_batch explains).
//   scatter         ms_scatter_batch_kernel files the k-lists under GLOBAL keypoint ids: the keypoint tables are the pairs'
//                   keypoints back to back with no padding (they never reach the candidate kernel); a query row finds its
//                   pair in the 256-row block table, a train row goes global row -> pair-local row -> that pair's map ->
//                   + the pair's first train keypoint.  The maps of a side are concatenated per scale in the padded row
//                   layout (identity for a NULL map) and uploaded once with every other table.
//   vote            ms_vote_kernel<SEG = true> over the concatenated coordinates, each query keypoint with its own pair's
//                   radius (iss_radius_tgt forward, iss_radius_src reverse).
//   filter          one-sided / mutual: b200m_filter_device with k = 1 on the global voted lists (ids of different pairs
//                   never meet); cluster: knn3d_kernel<SEG = true> keeps every 3-D neighbourhood inside its pair, then the
//                   single-pair cluster distance and compaction.
//   output          records ascend in global source keypoint, i.e. in pair order; one kernel makes them pair-local and
//                   counts them per pair; the average is average_kernel's chain over each pair's voted forward lists.
//
// b200m_match_multiscale_local_batch is the same driver with a guess: per scale and direction the kNN pass is the gated
// kNN of local.cu's batch form (launch_local_cells_batch) over the caller's moved query keypoints; everything after it is
// unchanged (DESIGN.md section 3.13).
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "internal.cuh"

namespace {

struct WideBatchState {
    MultiscaleState fwd, rev;
    DevBuf tables, xyz_s, xyz_t, kidx, kdist, kcnt, vfi, vfd, vfc, vri, vrd, vrc;
    DevBuf mov_s, mov_t;   // guessed calls: the moved source / target keypoints
    DevBuf scale_tables[32];   // batch plans: every scale's batch tables (batch.cu), staged once
};

WideBatchState *wb_state(b200m_ctx *ctx) {
    if (!ctx->wide_batch) ctx->wide_batch = new WideBatchState();
    return static_cast<WideBatchState *>(ctx->wide_batch);
}

// ms_scatter_kernel over the padded global rows of one scale and direction (q_side 0: queries = source rows).
// rows[p] = {first source row, source rows, first target row, target rows} of pair p at this scale.
__global__ void ms_scatter_batch_kernel(size_t n_rows, int k, int scale, int n_scales, int q_side, const int32_t *__restrict__ idx,
                                        const float *__restrict__ dist, const int32_t *__restrict__ count,
                                        const int32_t *__restrict__ block_pair, const int4 *__restrict__ rows,
                                        const int32_t *__restrict__ q_map, const int32_t *__restrict__ t_map,
                                        const int32_t *__restrict__ q_kp_off, const int32_t *__restrict__ t_kp_off,
                                        int32_t *__restrict__ s_idx, float *__restrict__ s_dist, int32_t *__restrict__ s_cnt,
                                        unsigned long long *__restrict__ bad) {
    const size_t row = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const int p = block_pair[row / B200M_TILE_N];
    const int4 r = rows[p];
    const long long q0 = q_side ? r.z : r.x, qn = q_side ? r.w : r.y, t0 = q_side ? r.x : r.z, tn = q_side ? r.y : r.w;
    if ((long long) row - q0 >= qn) return;   // gap row
    const long long qk0 = q_kp_off[p], n_qk = q_kp_off[p + 1] - qk0;
    const long long tk0 = t_kp_off[p], n_tk = t_kp_off[p + 1] - tk0;
    const long long kp = q_map[row];
    if (kp < 0 || kp >= n_qk) { flag_bad(bad, scale, p, q_side); return; }
    const size_t g = (size_t) (qk0 + kp);
    const int c = count[row];
    const size_t slot = (g * n_scales + scale) * k;
    for (int m = 0; m < c && m < k; ++m) {
        const long long j = (long long) idx[row * k + m] - t0;   // pair-local row of the train side of this scale
        long long tj = -1;
        if (j >= 0 && j < tn) tj = t_map[t0 + j];
        if (tj < 0 || tj >= n_tk) {
            flag_bad(bad, scale, p, 1 - q_side);
            tj = -1;
        } else {
            tj += tk0;
        }
        s_idx[slot + m] = (int32_t) tj;
        s_dist[slot + m] = dist[row * k + m];
    }
    s_cnt[g * n_scales + scale] = c < k ? c : k;
}

__global__ void localize_kp_records_kernel(b200m_corr *__restrict__ rec, const unsigned long long *__restrict__ n_out, size_t cap,
                                           const int32_t *__restrict__ src_off, const int32_t *__restrict__ tgt_off, int n_pairs,
                                           unsigned *__restrict__ counts) {
    const size_t n = *n_out < cap ? (size_t) *n_out : cap;
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        b200m_corr c = rec[i];
        const int p = pair_of(src_off, n_pairs, c.index_query);
        c.index_query -= src_off[p];
        c.index_match -= tgt_off[p];
        rec[i] = c;
        // records are sorted by pair: neighbouring lanes mostly share one, one atomic per run
        const unsigned peers = __match_any_sync(__activemask(), p);
        if ((int) (threadIdx.x & 31) == __ffs((int) peers) - 1) atomicAdd(counts + p, (unsigned) __popc(peers));
    }
}

int copy_xyz(b200m_ctx *ctx, char *dst, const float *host, size_t n, size_t stride_bytes) {
    if (n) CK(cudaMemcpyAsync(dst, host, (n - 1) * stride_bytes + 12, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

}  // namespace

void wide_batch_release(b200m_ctx *ctx) {
    WideBatchState *ws = static_cast<WideBatchState *>(ctx->wide_batch);
    if (!ws) return;
    for (MultiscaleState *ms : {&ws->fwd, &ws->rev}) {
        DevBuf *b[] = {&ms->idx, &ms->dist, &ms->cnt, &ms->bad, &ms->qmap, &ms->tmap, &ms->xyz, &ms->oidx, &ms->odist, &ms->ocnt,
                       &ms->kidx, &ms->kdist, &ms->kcnt};
        for (DevBuf *x : b) x->release();
    }
    DevBuf *b[] = {&ws->tables, &ws->xyz_s, &ws->xyz_t, &ws->kidx, &ws->kdist, &ws->kcnt, &ws->vfi, &ws->vfd, &ws->vfc,
                   &ws->vri, &ws->vrd, &ws->vrc, &ws->mov_s, &ws->mov_t};
    for (DevBuf *x : b) x->release();
    for (DevBuf &x : ws->scale_tables) x.release();
    delete ws;
    ctx->wide_batch = nullptr;
}

std::string map_status_text(unsigned long long key) {
    const std::string head = "pair " + std::to_string((key >> 16) & 0xffffffffull) + ", scale " + std::to_string(key >> 48);
    if ((key & 0xffff) >= 2 && (key >> 48) == 0xffff)   // a batch plan's live keypoint count (plan.cu)
        return "pair " + std::to_string((key >> 16) & 0xffffffffull) + ": the live " + ((key & 1) ? "target" : "source") +
               " keypoint count is above its capacity";
    if ((key & 0xffff) >= 2)   // a batch plan's live row count (plan.cu)
        return head + ": the live " + ((key & 1) ? "target" : "source") + " row count is above its capacity";
    return head + ": an index map entry of the " + ((key & 1) ? "target" : "source") + " cloud is outside its keypoint range";
}

// gated = false: b200m_match_multiscale_batch; true: the guessed form, whose kNN passes are gated by `radius`.
// dev: the *_device forms -- every data pointer of the pairs, the thresholds and `out` are device pointers (checked before
// anything is queued); descriptors are packed in place, maps and coordinates are filed by gather_sets_kernel, thresholds
// are read in place and the records stay on the device.
// Part 1: the checks, then one host image of every table, uploaded at once (and the host forms' coordinates).
int wide_batch_tables(b200m_ctx *ctx, const WideCall &c, WideLayout *W, bool keep_scales) {
    const std::string fn = std::string(c.name) + ": ";
    const b200m_params *p = &c.p;
    const b200m_wide_pair *pairs = c.pairs;
    const b200m_local_pair *locals = c.locals;
    const int n_pairs = c.n_pairs;
    const bool dev = c.dev, gated = c.gated;
    const int base = c.range ? c.range->pair_base : 0;
    if (n_pairs < 0) return b200m_fail_msg(ctx, fn + "n_pairs < 0");
    if (n_pairs > 0 && !pairs) return b200m_fail_msg(ctx, fn + "null pairs");
    if (gated && n_pairs > 0 && !locals) return b200m_fail_msg(ctx, fn + "null local pairs");
    const int mode = p->mode;
    if (mode != B200M_MODE_ONE_SIDED && mode != B200M_MODE_MUTUAL && mode != B200M_MODE_CLUSTER)
        return b200m_fail_msg(ctx, fn + "mode must be ONE_SIDED, MUTUAL or CLUSTER (the reference's implemented matchers)");
    if (p->k < 1 || p->k > B200M_MAX_K) return b200m_fail_msg(ctx, fn + "params.k must be in [1, 32]");
    if (mode == B200M_MODE_CLUSTER && (c.cluster_k < 1 || c.cluster_k > 64))
        return b200m_fail_msg(ctx, fn + "cluster_k must be in [1, 64]");
    if ((c.thr_src == nullptr) != (c.thr_tgt == nullptr)) return b200m_fail_msg(ctx, fn + "give both threshold arrays or neither");
    const size_t xyz_stride_bytes = c.xyz_stride_bytes;
    if (xyz_stride_bytes % 4 != 0 || xyz_stride_bytes < 12)
        return b200m_fail_msg(ctx, fn + "xyz stride must be a multiple of 4 and >= 12 bytes");
    const bool two_way = mode != B200M_MODE_ONE_SIDED;
    const int k = p->k;
    // per pair: scales that take part (none when the pair has no source keypoints: b200m_match_multiscale returns at once)
    std::vector<int> eff(n_pairs);
    std::vector<int32_t> kp_off[2] = {std::vector<int32_t>(n_pairs + 1, 0), std::vector<int32_t>(n_pairs + 1, 0)};
    size_t tot[2] = {0, 0};
    int n_scales = 0;
    for (int i = 0; i < n_pairs; ++i) {
        const b200m_wide_pair &w = pairs[i];
        const std::string pi = fn + "pair " + std::to_string(i + base) + ": ";
        if (w.n_scales < 0 || w.n_scales > 32) return b200m_fail_msg(ctx, pi + "n_scales must be in [0, 32]");
        if (w.n_scales && !w.scales) return b200m_fail_msg(ctx, pi + "null scales");
        if (w.n_scales * k > 128) return b200m_fail_msg(ctx, pi + "n_scales * k > 128");
        kp_off[0][i] = (int32_t) tot[0];
        kp_off[1][i] = (int32_t) tot[1];
        tot[0] += w.n_src_kps;
        tot[1] += w.n_tgt_kps;
        if (w.n_src_kps >= ((size_t) 1 << 31) || w.n_tgt_kps >= ((size_t) 1 << 31) || tot[0] >= ((size_t) 1 << 31) ||
            tot[1] >= ((size_t) 1 << 31))
            return b200m_fail_msg(ctx, pi + "more than 2^31-1 keypoints per side in the batch");
        eff[i] = w.n_src_kps ? w.n_scales : 0;
        if (dev) {
            if (check_device_ptr(ctx, pi + "src_kps_xyz", w.src_kps_xyz) || check_device_ptr(ctx, pi + "tgt_kps_xyz", w.tgt_kps_xyz))
                return 1;
            if (gated && (check_device_ptr(ctx, pi + "src_kps_moved", locals[i].src_kps_moved) ||
                          check_device_ptr(ctx, pi + "tgt_kps_moved", locals[i].tgt_kps_moved)))
                return 1;
            for (int s = 0; s < w.n_scales; ++s) {
                const b200m_scale &sc = w.scales[s];
                const std::string ps = pi + "scale " + std::to_string(s) + ": ";
                if (check_device_ptr(ctx, ps + "src_desc", sc.src_desc) || check_device_ptr(ctx, ps + "tgt_desc", sc.tgt_desc) ||
                    check_device_ptr(ctx, ps + "src_map", sc.src_map) || check_device_ptr(ctx, ps + "tgt_map", sc.tgt_map))
                    return 1;
            }
        }
        if (!w.n_src_kps) continue;
        if ((w.n_tgt_kps && !w.tgt_kps_xyz) || (two_way && !w.src_kps_xyz))
            return b200m_fail_msg(ctx, pi + "null keypoint coordinates");
        if (gated && (!locals[i].src_kps_moved || (two_way && w.n_tgt_kps && !locals[i].tgt_kps_moved)))
            return b200m_fail_msg(ctx, pi + "null moved keypoint coordinates");
        for (int s = 0; s < w.n_scales; ++s) {
            const b200m_scale &sc = w.scales[s];
            if ((sc.n_src && !sc.src_desc) || (sc.n_tgt && !sc.tgt_desc))
                return b200m_fail_msg(ctx, pi + "null descriptor pointer in scale " + std::to_string(s));
        }
        n_scales = std::max(n_scales, w.n_scales);
    }
    if (dev && (check_device_ptr(ctx, fn + "thr_src", c.thr_src) || check_device_ptr(ctx, fn + "thr_tgt", c.thr_tgt) ||
                check_device_ptr(ctx, fn + "out", c.out)))
        return 1;
    kp_off[0][n_pairs] = (int32_t) tot[0];
    kp_off[1][n_pairs] = (int32_t) tot[1];
    *W = WideLayout();
    W->n_scales = n_scales;
    W->two_way = two_way;
    W->NS = tot[0];
    W->NT = tot[1];
    if (n_scales == 0) return 0;   // no pair has source keypoints and a scale
    auto n_rows = [&](int i, int s, int side) -> size_t {
        if (s >= eff[i]) return 0;
        return side ? pairs[i].scales[s].n_tgt : pairs[i].scales[s].n_src;
    };
    // one host image of every table, uploaded at once: result area (initial values), keypoint offsets, radii, average
    // segments, then per scale the row table and the two block -> pair tables, then per side and scale the maps over the
    // padded rows
    std::vector<size_t> rows_pad[2];   // padded rows per scale and side
    for (int side = 0; side < 2; ++side) {
        rows_pad[side].assign(n_scales, 0);
        for (int s = 0; s < n_scales; ++s) {
            for (int i = 0; i < n_pairs; ++i) rows_pad[side][s] += pad_rows(n_rows(i, s, side));
            if (rows_pad[side][s] >= ((size_t) 1 << 31))
                return b200m_fail_msg(ctx, fn + "more than 2^31-1 descriptor rows per side in scale " + std::to_string(s) + " after padding");
        }
    }
    const size_t o_n = 0, o_bad = 8, o_counts = 16, o_avgs = align16(o_counts + sizeof(unsigned) * n_pairs);
    const size_t result_bytes = align16(o_avgs + sizeof(float) * n_pairs);
    const size_t o_off0 = result_bytes, o_off1 = align16(o_off0 + sizeof(int32_t) * (n_pairs + 1));
    const size_t o_rad0 = align16(o_off1 + sizeof(int32_t) * (n_pairs + 1)), o_rad1 = align16(o_rad0 + sizeof(float) * n_pairs);
    const size_t o_segs = align16(o_rad1 + sizeof(float) * n_pairs);
    size_t o = align16(o_segs + sizeof(int2) * n_pairs);
    W->o_rows.resize(n_scales);
    for (int s = 0; s < n_scales; ++s) {
        W->o_rows[s] = o;
        o = align16(o + sizeof(int4) * n_pairs);
        for (int side = 0; side < 2; ++side) {
            W->o_blk[side].push_back(o);
            o = align16(o + sizeof(int32_t) * (rows_pad[side][s] / B200M_TILE_N));
        }
    }
    // device calls: the gather tables of the maps (every side, scale and pair) and of the four coordinate tables; the maps
    // come last and are not uploaded (gather_sets_kernel fills their real rows, gap rows are never read)
    size_t o_gmap = 0, o_gxyz = 0, n_gmap = 0;
    if (dev) {
        for (int side = 0; side < 2; ++side)
            for (int s = 0; s < n_scales; ++s)
                for (int i = 0; i < n_pairs; ++i) n_gmap += n_rows(i, s, side) ? 1 : 0;
        o_gmap = o;
        o = align16(o + sizeof(GatherSet) * n_gmap);
        o_gxyz = o;   // [4][n_pairs]: xyz_t, xyz_s, mov_s, mov_t
        o = align16(o + sizeof(GatherSet) * 4 * n_pairs);
    }
    const size_t maps_begin = o;
    for (int side = 0; side < 2; ++side)
        for (int s = 0; s < n_scales; ++s) {
            W->o_map[side].push_back(o);
            o = align16(o + sizeof(int32_t) * rows_pad[side][s]);
        }
    const size_t table_bytes = o;
    // the result area stays zero here: every enqueue resets it on the device
    std::vector<char> h(dev ? maps_begin : table_bytes, 0);
    memcpy(h.data() + o_off0, kp_off[0].data(), sizeof(int32_t) * (n_pairs + 1));
    memcpy(h.data() + o_off1, kp_off[1].data(), sizeof(int32_t) * (n_pairs + 1));
    for (int i = 0; i < n_pairs; ++i) {
        reinterpret_cast<float *>(h.data() + o_rad0)[i] = pairs[i].iss_radius_src;
        reinterpret_cast<float *>(h.data() + o_rad1)[i] = pairs[i].iss_radius_tgt;
        reinterpret_cast<int2 *>(h.data() + o_segs)[i] = make_int2(kp_off[0][i], (int) pairs[i].n_src_kps);
    }
    GatherSet *gmap = dev ? reinterpret_cast<GatherSet *>(h.data() + o_gmap) : nullptr;
    size_t max_map_rows = 0;
    n_gmap = 0;
    for (int s = 0; s < n_scales; ++s) {
        size_t start[2] = {0, 0};
        int4 *rows = reinterpret_cast<int4 *>(h.data() + W->o_rows[s]);
        for (int i = 0; i < n_pairs; ++i) {
            const size_t n[2] = {n_rows(i, s, 0), n_rows(i, s, 1)};
            rows[i] = make_int4((int) start[0], (int) n[0], (int) start[1], (int) n[1]);
            for (int side = 0; side < 2; ++side) {
                int32_t *blk = reinterpret_cast<int32_t *>(h.data() + W->o_blk[side][s]);
                for (size_t b = start[side] / B200M_TILE_N; b < (start[side] + pad_rows(n[side])) / B200M_TILE_N; ++b) blk[b] = i;
                const int32_t *given = n[side] ? (side ? pairs[i].scales[s].tgt_map : pairs[i].scales[s].src_map) : nullptr;
                if (dev) {   // filed on the device, after the table upload (a NULL map: identity)
                    if (n[side]) {
                        gmap[n_gmap++] = GatherSet{given, 1, (int) (W->o_map[side][s] / 4 + start[side]), (int) n[side], 0};
                        W->gmap_keys.insert(W->gmap_keys.end(), {side, s, i});
                        max_map_rows = std::max(max_map_rows, n[side]);
                    }
                } else {
                    int32_t *map = reinterpret_cast<int32_t *>(h.data() + W->o_map[side][s]) + start[side];
                    if (given)
                        memcpy(map, given, sizeof(int32_t) * n[side]);
                    else
                        for (size_t r = 0; r < n[side]; ++r) map[r] = (int32_t) r;
                }
                start[side] += pad_rows(n[side]);
            }
        }
    }
    // coordinates of the pairs that take part (the host copy's rule): the first three floats of a row, which is all the
    // gather of local.cu, the vote and knn3d read
    GatherSet *gxyz = dev ? reinterpret_cast<GatherSet *>(h.data() + o_gxyz) : nullptr;
    if (dev) {
        const long long xs = (long long) (xyz_stride_bytes / 4);
        for (int i = 0; i < n_pairs; ++i) {
            const b200m_wide_pair &w = pairs[i];
            if (!w.n_src_kps) continue;
            gxyz[i] = GatherSet{w.tgt_kps_xyz, xs, kp_off[1][i], (int) w.n_tgt_kps, 0};
            if (two_way) gxyz[n_pairs + i] = GatherSet{w.src_kps_xyz, xs, kp_off[0][i], (int) w.n_src_kps, 0};
            if (gated) gxyz[2 * n_pairs + i] = GatherSet{locals[i].src_kps_moved, xs, kp_off[0][i], (int) w.n_src_kps, 0};
            if (gated && two_way) gxyz[3 * n_pairs + i] = GatherSet{locals[i].tgt_kps_moved, xs, kp_off[1][i], (int) w.n_tgt_kps, 0};
            W->max_kps[0] = std::max(W->max_kps[0], w.n_src_kps);
            W->max_kps[1] = std::max(W->max_kps[1], w.n_tgt_kps);
        }
    }
    // every scale's descriptor sets of every pair, as one batch per scale (a pair with fewer scales gives empty sets)
    W->pk = *p;
    W->pk.mode = B200M_MODE_KNN_ONLY;
    if (gated) W->pk.precision = B200M_PREC_F32_EXACT;   // the gated kNN is exact CUDA-core arithmetic: no tensor-core set-up
    W->sets.assign(n_scales, std::vector<b200m_pair>(n_pairs));
    for (int s = 0; s < n_scales; ++s)
        for (int i = 0; i < n_pairs; ++i) {
            const bool has = s < eff[i];
            W->sets[s][i] = b200m_pair{has ? pairs[i].scales[s].src_desc : nullptr, n_rows(i, s, 0),
                                       has ? pairs[i].scales[s].tgt_desc : nullptr, n_rows(i, s, 1)};
        }
    W->result_bytes = result_bytes;
    W->o_avgs = o_avgs;
    W->o_off[0] = o_off0;
    W->o_off[1] = o_off1;
    W->o_rad[0] = o_rad0;
    W->o_rad[1] = o_rad1;
    W->o_segs = o_segs;
    W->o_gmap = o_gmap;
    W->o_gxyz = o_gxyz;
    W->n_gmap = n_gmap;
    W->max_map_rows = max_map_rows;
    cudaStream_t st = ctx->stream;
    WideBatchState *ws = wb_state(ctx);
    if (keep_scales) {   // a plan: every scale's batch tables at once, each in its own buffer (the runs only pack)
        W->scale_tables.resize(n_scales);
        for (int s = 0; s < n_scales; ++s)
            if (stage_batch_tables(ctx, c.name, &W->pk, W->sets[s].data(), n_pairs, c.stride_bytes, c.dim, &W->scale_tables[s], dev,
                                   nullptr, nullptr, &ws->scale_tables[s]))
                return 1;
    }
    CK(ws->tables.reserve(table_bytes));
    char *d = ws->tables.as<char>();
    W->d = d;
    W->n_out = reinterpret_cast<unsigned long long *>(d + o_n);
    W->bad = reinterpret_cast<unsigned long long *>(d + o_bad);
    W->counts = reinterpret_cast<unsigned *>(d + o_counts);
    W->avgs = reinterpret_cast<float *>(d + o_avgs);
    CK(cudaMemcpyAsync(d, h.data(), h.size(), cudaMemcpyHostToDevice, st));
    // keypoint coordinates of all pairs back to back, `xyz_stride_bytes` apart
    const size_t NS = tot[0], NT = tot[1];
    CK(ws->xyz_t.reserve(NT * xyz_stride_bytes + 16));
    if (two_way) CK(ws->xyz_s.reserve(NS * xyz_stride_bytes + 16));
    if (gated) CK(ws->mov_s.reserve(NS * xyz_stride_bytes + 16));
    if (gated && two_way) CK(ws->mov_t.reserve(NT * xyz_stride_bytes + 16));
    for (int i = 0; i < n_pairs && !dev; ++i) {
        if (!pairs[i].n_src_kps) continue;
        if (copy_xyz(ctx, ws->xyz_t.as<char>() + (size_t) kp_off[1][i] * xyz_stride_bytes, pairs[i].tgt_kps_xyz, pairs[i].n_tgt_kps,
                     xyz_stride_bytes))
            return 1;
        if (two_way && copy_xyz(ctx, ws->xyz_s.as<char>() + (size_t) kp_off[0][i] * xyz_stride_bytes, pairs[i].src_kps_xyz,
                                pairs[i].n_src_kps, xyz_stride_bytes))
            return 1;
        if (gated) {
            if (copy_xyz(ctx, ws->mov_s.as<char>() + (size_t) kp_off[0][i] * xyz_stride_bytes, locals[i].src_kps_moved,
                         pairs[i].n_src_kps, xyz_stride_bytes))
                return 1;
            if (two_way && copy_xyz(ctx, ws->mov_t.as<char>() + (size_t) kp_off[1][i] * xyz_stride_bytes, locals[i].tgt_kps_moved,
                                    pairs[i].n_tgt_kps, xyz_stride_bytes))
                return 1;
        }
    }
    return 0;
}

// Part 2: kernels and memsets only.  Every workspace is sized from the call's shapes, so once a run has grown them, later
// runs of the same layout allocate nothing.
int wide_batch_enqueue(b200m_ctx *ctx, const WideCall &c, const WideLayout &W) {
    if (W.n_scales == 0) return 0;
    const int n_pairs = c.n_pairs, n_scales = W.n_scales, k = c.p.k, mode = c.p.mode;
    const bool dev = c.dev, gated = c.gated, two_way = W.two_way;
    const size_t NS = W.NS, NT = W.NT, xyz_stride_bytes = c.xyz_stride_bytes;
    cudaStream_t st = ctx->stream;
    WideBatchState *ws = wb_state(ctx);
    char *d = W.d;
    // the result area: no records, no bad map entry (~0), zero per-pair counts
    CK(cudaMemsetAsync(d, 0, W.o_avgs, st));
    CK(cudaMemsetAsync(W.bad, 0xFF, sizeof(unsigned long long), st));
    if (dev) {
        CK(launch_gather_sets(reinterpret_cast<const GatherSet *>(d + W.o_gmap), (int) W.n_gmap, W.max_map_rows, 1, 1, d, st));
        ctx->stats.launches += W.n_gmap ? 1 : 0;
        const size_t xs = xyz_stride_bytes / 4;
        const GatherSet *g = reinterpret_cast<const GatherSet *>(d + W.o_gxyz);
        DevBuf *dst[4] = {&ws->xyz_t, &ws->xyz_s, &ws->mov_s, &ws->mov_t};
        const bool used[4] = {true, two_way, gated, gated && two_way};
        const size_t mx[4] = {W.max_kps[1], W.max_kps[0], W.max_kps[0], W.max_kps[1]};
        for (int t = 0; t < 4; ++t) {
            if (!used[t] || !mx[t]) continue;
            CK(launch_gather_sets(g + (size_t) t * n_pairs, n_pairs, mx[t], 3, xs, dst[t]->p, st));
            ctx->stats.launches += 1;
        }
    }
    unsigned long long *d_n = W.n_out, *d_bad = W.bad;
    const int32_t *d_off0 = reinterpret_cast<const int32_t *>(d + W.o_off[0]), *d_off1 = reinterpret_cast<const int32_t *>(d + W.o_off[1]);
    const float *d_rad0 = reinterpret_cast<const float *>(d + W.o_rad[0]), *d_rad1 = reinterpret_cast<const float *>(d + W.o_rad[1]);
    if (ms_begin(ctx, &ws->fwd, NS, n_scales, k)) return 1;
    if (two_way && ms_begin(ctx, &ws->rev, NT, n_scales, k)) return 1;
    CK(ws->vfi.reserve(sizeof(int32_t) * NS));
    CK(ws->vfd.reserve(sizeof(float) * NS));
    CK(ws->vfc.reserve(sizeof(int32_t) * NS));
    if (two_way) {
        CK(ws->vri.reserve(sizeof(int32_t) * (NT + 1)));
        CK(ws->vrd.reserve(sizeof(float) * (NT + 1)));
        CK(ws->vrc.reserve(sizeof(int32_t) * (NT + 1)));
    }
    const b200m_params &pk = W.pk;
    for (int s = 0; s < n_scales; ++s) {
        BatchLayout L;
        if (!W.scale_tables.empty()) {
            L = W.scale_tables[s];
            if (stage_batch_pack(ctx, W.sets[s].data(), n_pairs, c.stride_bytes, c.dim, L, dev)) return 1;
        } else if (stage_batch(ctx, c.name, &pk, W.sets[s].data(), n_pairs, c.stride_bytes, c.dim, &L, dev)) {
            return 1;
        }
        const size_t S = L.n_rows[0], T = L.n_rows[1], n_max = std::max(S, T);
        CK(ws->kidx.reserve(sizeof(int32_t) * (n_max * k + 1)));
        CK(ws->kdist.reserve(sizeof(float) * (n_max * k + 1)));
        CK(ws->kcnt.reserve(sizeof(int32_t) * (n_max + 1)));
        const int4 *d_rows = reinterpret_cast<const int4 *>(d + W.o_rows[s]);
        const int32_t *d_map0 = reinterpret_cast<const int32_t *>(d + W.o_map[0][s]), *d_map1 = reinterpret_cast<const int32_t *>(d + W.o_map[1][s]);
        for (int dir = 0; dir < (two_way ? 2 : 1); ++dir) {
            const size_t nq = dir ? T : S;
            if (!nq) continue;
            MultiscaleState &ms = dir ? ws->rev : ws->fwd;
            if (gated) {
                LocalBatch lb;
                lb.direction = dir;
                lb.scale = s;
                lb.n_pairs = n_pairs;
                lb.k = k;
                lb.rows = d_rows;
                for (int side = 0; side < 2; ++side) {
                    lb.blk[side] = reinterpret_cast<const int32_t *>(d + W.o_blk[side][s]);
                    lb.map[side] = side ? d_map1 : d_map0;
                    lb.kp_off[side] = side ? d_off1 : d_off0;
                }
                lb.q_xyz = dir ? ws->mov_t.as<float>() : ws->mov_s.as<float>();
                lb.t_xyz = dir ? ws->xyz_s.as<float>() : ws->xyz_t.as<float>();
                lb.xyz_stride_bytes = xyz_stride_bytes;
                lb.radius = c.radius;
                lb.bad = d_bad;
                StatTimer tf(ctx, &ctx->stats.ms_fallback);
                if (launch_local_cells_batch(ctx, lb, ws->kidx.as<int32_t>(), ws->kdist.as<float>(), ws->kcnt.as<int32_t>())) return 1;
                tf.stop();
            } else if (b200m_knn_rows(ctx, &pk, dir, 0, nq, nullptr, ws->kidx.as<int32_t>(), ws->kdist.as<float>(),
                                      ws->kcnt.as<int32_t>(), &L.seg[dir])) {
                return 1;
            }
            ms_scatter_batch_kernel<<<(unsigned) ((nq + 255) / 256), 256, 0, st>>>(
                nq, k, s, n_scales, dir, ws->kidx.as<int32_t>(), ws->kdist.as<float>(), ws->kcnt.as<int32_t>(),
                reinterpret_cast<const int32_t *>(d + W.o_blk[dir][s]), d_rows, dir ? d_map1 : d_map0, dir ? d_map0 : d_map1,
                dir ? d_off1 : d_off0, dir ? d_off0 : d_off1, ms.idx.as<int32_t>(), ms.dist.as<float>(), ms.cnt.as<int32_t>(), d_bad);
            CK(cudaGetLastError());
            ctx->stats.launches += 1;
        }
    }
    // the two votes: train keypoints = the OTHER cloud's, radius = the train side's of the query keypoint's pair
    if (ms_vote_batch_device(ctx, &ws->fwd, ws->xyz_t.as<float>(), xyz_stride_bytes, d_off0, n_pairs, d_rad1, ws->vfi.as<int32_t>(),
                             ws->vfd.as<float>(), ws->vfc.as<int32_t>()))
        return 1;
    if (two_way && ms_vote_batch_device(ctx, &ws->rev, ws->xyz_s.as<float>(), xyz_stride_bytes, d_off1, n_pairs, d_rad0,
                                        ws->vri.as<int32_t>(), ws->vrd.as<float>(), ws->vrc.as<int32_t>()))
        return 1;
    const float *d_thr_s = nullptr, *d_thr_t = nullptr;
    if (c.thr_src && NT && W.thr_sets) {   // a plan with live counts: capacity-layout thresholds gathered into the dense layout
        for (int side = 0; side < 2; ++side) {
            CK(ctx->ws_thr[side].reserve(sizeof(float) * (side ? NT : NS)));
            CK(launch_gather_sets(W.thr_sets + (size_t) side * n_pairs, n_pairs, W.max_kps[side], 1, 1, ctx->ws_thr[side].p, st));
            ctx->stats.launches += 1;
        }
        d_thr_s = ctx->ws_thr[0].as<float>();
        d_thr_t = ctx->ws_thr[1].as<float>();
    } else if (c.thr_src && NT && dev) {   // the device thresholds are the dense keypoint-table layout already
        d_thr_s = c.thr_src;
        d_thr_t = c.thr_tgt;
    } else if (c.thr_src && NT) {   // keypoint tables are dense: the concatenated thresholds are indexed by the global ids as they are
        CK(ctx->ws_thr[0].reserve(sizeof(float) * NS));
        CK(ctx->ws_thr[1].reserve(sizeof(float) * NT));
        CK(cudaMemcpyAsync(ctx->ws_thr[0].p, c.thr_src, sizeof(float) * NS, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->ws_thr[1].p, c.thr_tgt, sizeof(float) * NT, cudaMemcpyHostToDevice, st));
        d_thr_s = ctx->ws_thr[0].as<float>();
        d_thr_t = ctx->ws_thr[1].as<float>();
    }
    CK(ctx->ws_corr.reserve(sizeof(b200m_corr) * NS));
    b200m_params p1 = c.p;
    p1.k = 1;   // the voted lists hold at most one match
    if (mode == B200M_MODE_CLUSTER) {
        if (cluster_filter_batch_device(ctx, &p1, c.cluster_k, 0.95f /* MATCHING_CLUSTER_THRESHOLD, include/common.h:52 */, NS, NT,
                                        ws->vfi.as<int32_t>(), ws->vfd.as<float>(), ws->vfc.as<int32_t>(), ws->vri.as<int32_t>(),
                                        ws->vrc.as<int32_t>(), ws->xyz_s.as<float>(), ws->xyz_t.as<float>(), xyz_stride_bytes, d_off0,
                                        d_off1, n_pairs, d_thr_s, d_thr_t, ctx->ws_corr.as<b200m_corr>(), NS, d_n))
            return 1;
    } else if (b200m_filter_device(ctx, &p1, 0, NS, ws->vfi.as<int32_t>(), ws->vfd.as<float>(), ws->vfc.as<int32_t>(),
                                   ws->vri.as<int32_t>(), ws->vrd.as<float>(), ws->vrc.as<int32_t>(), mode == B200M_MODE_MUTUAL ? NT : 0,
                                   d_thr_s, d_thr_t, ctx->ws_corr.as<b200m_corr>(), NS, d_n, nullptr)) {
        return 1;
    }
    if (c.want_avg) {
        CK(launch_average_segments(ws->vfd.as<float>(), ws->vfc.as<int32_t>(), reinterpret_cast<const int2 *>(d + W.o_segs), n_pairs, 1,
                                   W.avgs, st));
        ctx->stats.launches += 1;
    }
    localize_kp_records_kernel<<<(unsigned) ctx->sm_count * 4, 256, 0, st>>>(ctx->ws_corr.as<b200m_corr>(), d_n, NS, d_off0, d_off1,
                                                                             n_pairs, W.counts);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

// Part 3 (host and device forms): the result area back, then the bad-map check, offsets, averages, capacity and records.
int wide_batch_results(b200m_ctx *ctx, const WideCall &c, const WideLayout &W, b200m_corr *out, size_t cap, size_t *offsets,
                       float *avg) {
    const std::string fn = std::string(c.name) + ": ";
    const int n_pairs = c.n_pairs;
    if (W.n_scales == 0) {
        if (avg)
            for (int i = 0; i < n_pairs; ++i) avg[i] = 3.402823466e+38F;   // FLT_MAX, reference include/matching.h:41
        return 0;
    }
    cudaStream_t st = ctx->stream;
    std::vector<char> res(W.result_bytes);
    CK(cudaMemcpyAsync(res.data(), W.d, W.result_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    unsigned long long n, bad;
    memcpy(&n, res.data(), sizeof(n));
    memcpy(&bad, res.data() + 8, sizeof(bad));
    if (bad != ~0ull) {
        if (c.range) {   // the key with the group call's pair number: (scale, pair, side) order is kept
            bad += (unsigned long long) c.range->pair_base << 16;
            c.range->bad_key = bad;
        }
        return b200m_fail_msg(ctx, fn + map_status_text(bad));
    }
    const unsigned *cnt = reinterpret_cast<const unsigned *>(res.data() + 16);
    for (int i = 0; i < n_pairs; ++i) offsets[i + 1] = offsets[i] + cnt[i];
    if (avg) memcpy(avg, res.data() + W.o_avgs, sizeof(float) * n_pairs);
    if (n > cap) return b200m_fail_msg(ctx, fn + "output capacity too small (" + std::to_string(n) + " correspondences)");
    if (n) {
        if (!out) return b200m_fail_msg(ctx, fn + "null output buffer");
        if (c.dev) {   // stream-ordered: the caller's next work on the stream sees the records
            CK(cudaMemcpyAsync(out, ctx->ws_corr.p, sizeof(b200m_corr) * n, cudaMemcpyDeviceToDevice, st));
            return 0;
        }
        CK(cudaMemcpyAsync(out, ctx->ws_corr.p, sizeof(b200m_corr) * n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return 0;
}

namespace {

// r: a range of a group call (multi.cu), or NULL
int match_multiscale_batch(b200m_ctx *ctx, const char *name, bool dev, const b200m_params *p, const b200m_wide_pair *pairs,
                           bool gated, const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim,
                           size_t xyz_stride_bytes, int cluster_k, float radius, const float *thr_src, const float *thr_tgt,
                           b200m_corr *out, size_t cap, size_t *offsets, float *avg, BatchRange *r = nullptr) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    if (!p || !offsets) return b200m_fail_msg(ctx, std::string(name) + ": null params / offsets");
    for (int i = 0; i <= n_pairs; ++i) offsets[i] = 0;
    WideCall c;
    c.name = name;
    c.dev = dev;
    c.gated = gated;
    c.p = *p;
    c.pairs = pairs;
    c.locals = locals;
    c.n_pairs = n_pairs;
    c.stride_bytes = stride_bytes;
    c.xyz_stride_bytes = xyz_stride_bytes;
    c.dim = dim;
    c.cluster_k = cluster_k;
    c.radius = radius;
    c.thr_src = thr_src;
    c.thr_tgt = thr_tgt;
    c.out = out;
    c.want_avg = avg != nullptr;
    c.range = r;
    WideLayout W;
    if (wide_batch_tables(ctx, c, &W, false)) return 1;
    if (r) r->validated = true;
    if (wide_batch_enqueue(ctx, c, W)) return 1;
    return wide_batch_results(ctx, c, W, out, cap, offsets, avg);
}

}  // namespace

int match_multiscale_batch_host(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs, bool gated,
                                const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim, size_t xyz_stride_bytes,
                                int cluster_k, float radius, const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap,
                                size_t *offsets, float *avg, BatchRange *r) {
    return match_multiscale_batch(ctx, gated ? "b200m_match_multiscale_local_batch" : "b200m_match_multiscale_batch", false, p, pairs,
                                  gated, locals, n_pairs, stride_bytes, dim, xyz_stride_bytes, cluster_k, radius, thr_src, thr_tgt, out,
                                  cap, offsets, avg, r);
}

extern "C" int b200m_match_multiscale_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs, int n_pairs,
                                            size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k,
                                            const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap,
                                            size_t *offsets, float *avg) {
    return match_multiscale_batch(ctx, "b200m_match_multiscale_batch", false, p, pairs, false, nullptr, n_pairs, stride_bytes, dim,
                                  xyz_stride_bytes, cluster_k, 0.f, thr_src, thr_tgt, out, cap, offsets, avg);
}

extern "C" int b200m_match_multiscale_batch_device(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs, int n_pairs,
                                                   size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k,
                                                   const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                                   size_t *offsets, float *avg) {
    return match_multiscale_batch(ctx, "b200m_match_multiscale_batch_device", true, p, pairs, false, nullptr, n_pairs, stride_bytes,
                                  dim, xyz_stride_bytes, cluster_k, 0.f, d_thr_src, d_thr_tgt, d_out, cap, offsets, avg);
}

extern "C" int b200m_match_multiscale_local_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                  const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim,
                                                  size_t xyz_stride_bytes, int cluster_k, float match_search_radius,
                                                  const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap,
                                                  size_t *offsets, float *avg) {
    return match_multiscale_batch(ctx, "b200m_match_multiscale_local_batch", false, p, pairs, true, locals, n_pairs, stride_bytes,
                                  dim, xyz_stride_bytes, cluster_k, match_search_radius, thr_src, thr_tgt, out, cap, offsets, avg);
}

extern "C" int b200m_match_multiscale_local_batch_device(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                         const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim,
                                                         size_t xyz_stride_bytes, int cluster_k, float match_search_radius,
                                                         const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out,
                                                         size_t cap, size_t *offsets, float *avg) {
    return match_multiscale_batch(ctx, "b200m_match_multiscale_local_batch_device", true, p, pairs, true, locals, n_pairs,
                                  stride_bytes, dim, xyz_stride_bytes, cluster_k, match_search_radius, d_thr_src, d_thr_tgt, d_out,
                                  cap, offsets, avg);
}
