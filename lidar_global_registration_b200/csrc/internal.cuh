// internal.cuh -- shared declarations of libb200match (not part of the C-ABI).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/b200match.h"

#define B200M_MAX_K 32
#define B200M_MAX_DIM 2048
#define B200M_TILE_N 256     // train rows per candidate-kernel tile; operand row counts are padded to this
#define B200M_TILE_M 128     // query rows per CTA
#define B200M_AUG_COLS 3     // extra K columns carrying |b|^2 as an FP16 triple
#define B200M_SENTINEL 60000.0f  // |b|^2 stand-in for invalid/padding train rows (FP16-representable)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes);   // grow-only
    void release();
    template <typename T> T *as() const { return (T *) p; }
};

struct Side {
    size_t n = 0;          // rows
    size_t n_pad = 0;      // rows rounded up to B200M_TILE_N
    int dim = 0;           // descriptor length
    int dp = 0;            // f32 row pitch in floats (dim rounded up to 4)
    int kp = 0;            // fp16 operand row pitch in halves (multiple of 64)
    int64_t index_offset = 0;
    uint64_t version = 0;  // bumped on every upload
    DevBuf staging;        // raw AoS as uploaded from the host
    DevBuf f32;            // [n][dp] dense FP32, zero padded columns
    DevBuf valid;          // [n] uint8
    DevBuf stats;          // per-CTA column statistics of the pack kernel (see pack.cu)
    DevBuf op_query;       // [n_pad][kp] fp16: -2*x16, 1,1,1, 0...
    DevBuf op_train;       // [n_pad][kp] fp16:  x16, nb_hi, nb_mid, nb_lo, 0...
    DevBuf norm16;         // [n_pad] float: |x16|^2 in scaled units
};

// Device-resident results of the prepare step (pack.cu), in TcPrep::red: written by prep_finalize / pack_operands, read by
// the operand pack, copied to the host once afterwards -- or, in a context with device_prepare, turned into the routing
// decision by prep_decide_kernel and read by the candidate kernel (DP form) instead.
struct PrepDev {
    int maxabs_bits;        // max |x - mean| over the valid rows of both sides, as the bits of a non-negative float
    int max_norm_bits[2];   // max |x16| per side, likewise (atomicMax)
    int usable;             // device_prepare: 1 when the data lies inside the certificate's window (tc_window, pack.cu)
    float bmax[2];          // device_prepare: max |b16| per side, the candidate kernel's norm bound of that side as train side
};

struct TcPrep {            // state shared by both sides' FP16 operands
    uint64_t ver[2] = {0, 0};
    bool ready = false;
    DevBuf mean;           // [dp] float centre
    DevBuf red;            // reduction scratch
    float scale = 1.f;     // power of two applied after centring
    float max_norm[2] = {0.f, 0.f};   // max |x16| per side (scaled units)
    bool usable = false;   // false when the data cannot be scaled into FP16 range (non-finite spread)
};

struct b200m_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    std::string err;
    Side side[2];
    TcPrep prep;
    DevBuf ws_cand_idx, ws_cand_cnt, ws_flag_rows, ws_counters, ws_scan, ws_out, ws_misc;
    DevBuf ws_part_i, ws_part_d, ws_done, ws_cand_val, ws_cand_thr;
    DevBuf ws_sweep_hint;   // [<= 64 train splits] int: where the candidate kernel's CTA pairs currently are in their sweep
    DevBuf ws_row_list, ws_row_flags, ws_sel_ops, ws_sel_norm;   // row selection (masked kNN)
    bool done_init = false;
    DevBuf ws_fidx, ws_fdist, ws_fcnt, ws_ridx, ws_rdist, ws_rcnt, ws_thr[2], ws_corr, ws_totals;
    DevBuf ws_batch;       // batch calls (batch.cu): segment tables, per-pair bookkeeping and per-pair results
    bool totals_init = false;
    void *tmap_cache = nullptr;
    void *multiscale = nullptr;   // MultiscaleState (multiscale.cu)
    void *cluster = nullptr;      // ClusterState (cluster.cu)
    void *wide = nullptr;         // WideState (wide.cu)
    void *wide_batch = nullptr;   // WideBatchState (wide_batch.cu)
    void *comm = nullptr;         // Comm (multi.cu): this context's rank in an NCCL communicator
    void *local = nullptr;        // LocalState (local.cu): the cell list of the gated kNN
    void *stage = nullptr;        // StagePool (api.cu): pinned bounce buffers for uploads from pageable host memory
    int local_min_rows = 4096;    // B200M_LOCAL_MIN_ROWS: train sets below this use the brute-force gate kernel
    int tc_cluster = 0;    // 0 = default; test/tuning override of the multicast cluster size (B200M_TC_CLUSTER)
    double masked_min_pairs = 1e9;   // B200M_MASKED_MIN_PAIRS: b200m_match skips unreferenced target rows in the reverse pass
                                     // from this many (source, target) pairs on (below, the row selection's host round trip
                                     // costs more than it saves)
    int tc_splits = 0;     // B200M_TC_SPLITS: 0 = chosen per launch (wave balance); > 0 forces the number of train splits
    int tc_splitn = 1;     // split-N candidate kernel for one-atom descriptors (B200M_TC_SPLITN=0: one N = 256 MMA per tile)
    int tc_alt = -1;       // B200M_TC_ALT: epilogue layout of the split-N kernel (4 / 5 chunk entries drained by 32- / 16-column
                           // TMEM loads; column entries: 1 alternating tiles, 2 quarter columns, 0 eight warps);
                           // -1 = by measurement: 5 up to k = 2, 4 beyond
    int tc_sweep_lag = -1; // B200M_TC_SWEEP_LAG: tiles between followers of the chunk-entry kernels' rotated sweep (0 = off, -1 = by size)
    int tc_lean = 1;       // B200M_TC_LEAN=0: general MMA issue loop also for one-atom descriptors (comparison)
    int tc_debug = 0;      // B200M_TC_DEBUG: timing experiments (results are NOT valid when set)
    int tc_pair = 1;       // 1 = CTA-pair (cta_group::2) candidate kernel; 0 = cta_group::1 + multicast (B200M_TC_MODE=mcast)
    // Batch plans (plan.cu): the tensor-core / exact routing and the norm bounds stay on the device (prep_decide_kernel and
    // the candidate kernel's DP form), so the kNN driver enqueues without a host round trip.  Only a plan's private
    // context sets it.
    bool device_prepare = false;
    bool profiling = false;
    b200m_stats stats{};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    struct EventPool *pool = nullptr;
};

int b200m_fail(b200m_ctx *ctx, const char *what, cudaError_t e, const char *file, int line);
int b200m_fail_msg(b200m_ctx *ctx, const std::string &msg);

#define CK(expr)                                                                   \
    do {                                                                           \
        cudaError_t _e = (expr);                                                   \
        if (_e != cudaSuccess) return b200m_fail(ctx, #expr, _e, __FILE__, __LINE__); \
    } while (0)

// Per-region device timing without host synchronisation: when profiling is on, a region records a pair of
// events from the context's pool on the stream; pairs are resolved (cudaEventElapsedTime) when the stats are
// read or the pool fills up, so the timed program runs exactly as it does unprofiled.
struct EventPool {
    static const int kPairs = 128;
    cudaEvent_t ev[2 * kPairs] = {};
    double *slot[kPairs] = {};
    int used = 0;
    bool created = false;
};
void b200m_resolve_events(b200m_ctx *ctx);

struct StatTimer {
    b200m_ctx *ctx;
    int pair = -1;
    StatTimer(b200m_ctx *c, double *s);
    void stop();
};

// A batch call's layout (batch.cu), per query direction: every pair's rows start at a multiple of B200M_TILE_N on both
// sides, and range[query row / B200M_TILE_N] = {first, end} train row of that block's pair.  max_tiles: train tiles of the
// largest segment.
struct SegTable {
    const int2 *range = nullptr;
    int max_tiles = 0;
};

// A device batch call's descriptor set in the padded layout: `rows` rows at `base` (the caller's device memory, the
// call's stride apart) fill padded rows [first, first + rows) of their side.
struct alignas(16) SetRef {
    const float *base;
    int first, rows;
};

inline size_t pad_rows(size_t n) { return (n + B200M_TILE_N - 1) / B200M_TILE_N * B200M_TILE_N; }
inline size_t align16(size_t b) { return (b + 15) & ~(size_t) 15; }

// batch.cu: what stage_batch leaves on the device.  Pair p's rows start at the sum of pad_rows() of the pairs before it.
// A batch plan with live counts (plan.cu) rewrites sets, thr_sets, avg_segs and seg[].range in place on every run: they
// live in a buffer of the plan's own context and are never shared with another layout.
// pair_info[p] = {first source row, first target row, source rows, first row of the pair in the dense k-list output}
struct BatchLayout {
    size_t n_rows[2] = {0, 0};   // padded rows per side
    size_t real_src = 0;         // sum of the pairs' source rows
    SegTable seg[2];             // per query direction
    const int32_t *block_pair = nullptr;   // [source rows / 256] pair of that source block
    const int4 *pair_info = nullptr;       // [n_pairs]
    const int2 *avg_segs = nullptr;        // [n_pairs] {first source row, source rows}
    unsigned long long *n_out = nullptr;   // result area: record count, then per-pair counts and averages
    unsigned *counts = nullptr;
    float *avgs = nullptr;
    size_t result_bytes = 0;
    size_t max_rows[2] = {0, 0};                   // largest set per side
    const struct GatherSet *thr_sets[2] = {nullptr, nullptr};   // device calls with thresholds: [n_pairs] per side
    const int32_t *seg_blk[2] = {nullptr, nullptr};   // device calls: per side block -> pair table of the segmented pack
    const SetRef *sets[2] = {nullptr, nullptr};       // device calls: per side [n_pairs] sets of the segmented pack
};
// Validates the pairs, packs both sides in the padded layout (replacing what b200m_upload put in the context) and uploads
// the segment tables into ctx->ws_batch.  dev: every descriptor pointer is a device pointer of the context's device
// (checked; the segmented pack reads the sets in place); d_thr_src / d_thr_tgt (dev only): the concatenated device
// thresholds, for which gather tables into the padded layout go up with the segment tables.
// = stage_batch_tables, then stage_batch_pack.
int stage_batch(b200m_ctx *ctx, const char *fn, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                size_t stride_bytes, int dim, BatchLayout *L, bool dev = false, const float *d_thr_src = nullptr,
                const float *d_thr_tgt = nullptr);
// The validation and the tables (one upload into *dst, ctx->ws_batch when null, reserved here); nothing is packed.
int stage_batch_tables(b200m_ctx *ctx, const char *fn, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                       size_t stride_bytes, int dim, BatchLayout *L, bool dev, const float *d_thr_src, const float *d_thr_tgt,
                       DevBuf *dst = nullptr);
// The pack of both sides into the layout the tables describe.  dev: kernels only (no copy, no allocation once the sides'
// buffers have grown to the layout), which is what a batch plan's run enqueues.
int stage_batch_pack(b200m_ctx *ctx, const b200m_pair *pairs, int n_pairs, size_t stride_bytes, int dim, const BatchLayout &L,
                     bool dev);
// After stage_batch: the k-lists of every pair, pair-local, rows back to back, into the device arrays o_idx / o_dist / o_cnt.
int knn_batch_lists(b200m_ctx *ctx, const b200m_params *p, const BatchLayout &L, int32_t *o_idx, float *o_dist, int32_t *o_cnt);
// After stage_batch (real_src > 0): kNN, thresholds, filter, averages (want_avg: into L.avgs) and the records made pair-local
// in ctx->ws_corr, their number in *L.n_out and the per-pair counts in L.counts.  dev: thresholds are device pointers (filed
// by the gather tables), else host arrays.
int match_batch_records(b200m_ctx *ctx, const b200m_params *p, const BatchLayout &L, const b200m_pair *pairs, int n_pairs,
                        bool dev, const float *thr_src, const float *thr_tgt, bool want_avg);

// Device batch calls: `rows` rows of `w` 4-byte words, src_stride words apart at `src`, go to rows dst_row.. of a
// destination (dst_stride words apart).  src = null writes the identity (row r -> r, w = 1): a NULL index map.
struct alignas(16) GatherSet {
    const void *src;
    long long src_stride;
    int dst_row, rows;
    int pad;
};
// batch.cu: one launch for n_sets sets (max_rows: the largest)
cudaError_t launch_gather_sets(const GatherSet *d_sets, int n_sets, size_t max_rows, int w, size_t dst_stride_words, void *dst,
                               cudaStream_t st);
// 0 when ptr is null or device / managed memory of the context's device; else fails with "<where> is not device memory ..."
int check_device_ptr(b200m_ctx *ctx, const std::string &where, const void *ptr);

// ---- kernel launchers (one translation unit each) ---------------------------
// pack.cu
// dense FP32 copy + validity + per-CTA column statistics (sum, min, max over valid rows) into `stats`
// (pack_stats_bytes() bytes), which launch_tc_prepare turns into the common centre and FP16 scale
// With `sets` (device batch calls) the rows come from the caller's sets instead of `aos`: padded row r is row
// r - sets[b].first of set b = seg_blk[r / 256] (a gap row past the set's end packs as NaN, see pack.cu)
cudaError_t launch_pack_f32(const float *aos, size_t n, size_t stride_bytes, int dim, int dp,
                            float *f32, uint8_t *valid, float *stats, int sm_count, cudaStream_t st,
                            const int32_t *seg_blk = nullptr, const SetRef *sets = nullptr);
size_t pack_stats_bytes(int sm_count, int dp);
// centre/scale + FP16 operand tiles for both sides; with ctx->device_prepare the routing decision and the norm bounds stay
// in PrepDev (prep_decide_kernel) and nothing is read back
cudaError_t launch_tc_prepare(b200m_ctx *ctx);

// exact.cu
cudaError_t launch_exact_rows(const float *q_f32, const uint8_t *q_valid, int dp, int dim,
                              const float *t_f32, const uint8_t *t_valid, size_t nt, int64_t t_index_offset,
                              size_t row_begin, size_t n_rows, const int32_t *row_list, const int32_t *row_list_count,
                              int k, int32_t *idx, float *dist, int32_t *count, int max_blocks,
                              // few flagged rows (row_list given): split_blocks CTAs share every row; workspace of
                              // exact_split_ws_entries() int32 + float entries and exact_split_max_rows() zeroed counters
                              int split_blocks, int32_t *part_i, float *part_d, unsigned int *done,
                              // row_map (or null): the call's rows are row_map[0..n_rows) instead of row_begin + 0..n_rows;
                              // results are always stored at (row - row_begin)
                              const int32_t *row_map, cudaStream_t st,
                              // seg_range (or null): query row qi only looks at train rows [seg_range[qi / 256].x, .y)
                              const int2 *seg_range = nullptr);
cudaError_t launch_local_rows(const float *q_f32, const uint8_t *q_valid, int dp, const float *t_f32,
                              const uint8_t *t_valid, size_t nt, int64_t t_index_offset, size_t n_rows,
                              const float *q_xyz, const float *t_xyz, size_t xyz_stride_bytes, float radius, int k,
                              int32_t *idx, float *dist, int32_t *count, int max_blocks, cudaStream_t st);
size_t exact_split_ws_entries(int split_blocks, int k);
int exact_split_max_rows();
cudaError_t launch_rerank(const float *q_f32, const uint8_t *q_valid, int dp, int dim,
                          const float *t_f32, const uint8_t *t_valid, size_t nt, int64_t t_index_offset,
                          size_t row_begin, size_t n_rows, int k,
                          const int32_t *cand_idx, const int32_t *cand_cnt, int n_lists, int cap,
                          const float *cand_val, const float *cand_thr /* both null: no pruning */,
                          int32_t *idx, float *dist, int32_t *count,
                          int32_t *flag_rows, int32_t *counters /*[0]=flagged rows, [1..2]=candidate pairs (u64)*/,
                          int sm_count, const int32_t *row_map,
                          int chunk_entries /* 1: an entry is the first of 32 consecutive train rows + the chunk's minimum */,
                          cudaStream_t st);

// filter.cu
cudaError_t launch_filter(int mode, int k, float ratio_thr, float distance_thr, size_t row_begin, size_t n_rows,
                          const int32_t *fidx, const float *fdist, const int32_t *fcount,
                          const int32_t *ridx, const float *rdist, const int32_t *rcount, size_t n_rev_rows,
                          const float *thr_src, const float *thr_tgt, int64_t src_offset, int64_t tgt_offset,
                          b200m_corr *out, size_t cap, unsigned long long *n_out, float *avg,
                          void *scan_ws, size_t scan_ws_bytes, cudaStream_t st, int *n_launches,
                          const float *cdist = nullptr /* B200M_MODE_CLUSTER: [n_rows][k] from cluster.cu */);
size_t filter_scan_ws_bytes(size_t n_rows, int k);
cudaError_t launch_average(const float *fdist, const int32_t *fcount, size_t n_rows, int k, float *avg,
                           cudaStream_t st);
// one average per segment: avg[s] over rows [segs[s].x, segs[s].x + segs[s].y) (one CTA per segment)
cudaError_t launch_average_segments(const float *fdist, const int32_t *fcount, const int2 *segs, int n_segs, int k, float *avg,
                                    cudaStream_t st);
cudaError_t launch_merge(int k, int n_lists, size_t nq, const int32_t *idx_in, const float *dist_in,
                         const int32_t *count_in, int32_t *idx, float *dist, int32_t *count, cudaStream_t st);

// candidates_tc.cu
// Fills ws_cand_idx [n_lists][n_rows][cap] and ws_cand_cnt [n_lists][n_rows] (entries appended per list; a
// count above cap marks an overflowed list).  dump != nullptr: single tile, raw accumulators to dump[128][256].
// *has_values_out = 1: ws_cand_val [n_lists][n_rows][cap] and ws_cand_thr [n_lists][n_rows] are filled too;
// = 2: the same, and every entry is a 32-row CHUNK (first train row, smallest accumulator of the chunk).
// q_ops != null: the query rows are rows 0..n_rows of this compact [q_pad][kp] operand array (norms in q_norm) instead of
// rows row_begin.. of the query side's own array.
int tc_candidates(b200m_ctx *ctx, int direction, size_t row_begin, size_t n_rows, int k, int cap_request,
                  int *n_lists_out, int *cap_out, int *has_values_out, float *dump, size_t dump_t_tile,
                  const void *q_ops = nullptr, const float *q_norm = nullptr, size_t q_pad = 0,
                  const SegTable *seg = nullptr /* batch: every query block sweeps its own pair's train tiles only */);
bool tc_supported(const b200m_ctx *ctx, int dim, int k);
void tc_release(b200m_ctx *ctx);

// multiscale.cu: one table of per-scale k-lists filed under the query keypoints (match_multiscale's concatenation)
struct MultiscaleState {
    size_t n_query_kps = 0;
    int n_scales = 0, k = 0;
    DevBuf idx, dist, cnt, bad, qmap, tmap, xyz, oidx, odist, ocnt, kidx, kdist, kcnt;
};
void multiscale_release(b200m_ctx *ctx);
void ms_free(MultiscaleState *ms);
int ms_begin(b200m_ctx *ctx, MultiscaleState *ms, size_t n_query_kps, int n_scales, int k);
int ms_add_device(b200m_ctx *ctx, MultiscaleState *ms, int scale, size_t n_rows, const int32_t *d_idx, const float *d_dist,
                  const int32_t *d_count, const int32_t *d_query_map, const int32_t *d_train_map, size_t n_train_rows,
                  int64_t train_index_offset, size_t n_train_kps);
int ms_vote_device(b200m_ctx *ctx, MultiscaleState *ms, const float *d_train_xyz, size_t xyz_stride_bytes, float iss_radius,
                   int32_t *d_idx, float *d_dist, int32_t *d_count);

// Batch form of ms_vote_device (used by wide_batch.cu): the query keypoints of all pairs back to back, train ids global over the
// concatenated train keypoints; query keypoint i belongs to pair p with kp_off[p] <= i < kp_off[p + 1] and votes with
// radii[p].
int ms_vote_batch_device(b200m_ctx *ctx, MultiscaleState *ms, const float *d_train_xyz, size_t xyz_stride_bytes,
                         const int32_t *d_kp_off, int n_pairs, const float *d_radii, int32_t *d_idx, float *d_dist,
                         int32_t *d_count);

// wide.cu
void wide_release(b200m_ctx *ctx);
void wide_batch_release(b200m_ctx *ctx);

// wide_batch.cu: b200m_match_multiscale(_local)_batch(_device) in three parts.  wide_batch_tables validates the call and
// uploads every table once; wide_batch_enqueue queues the batch with kernels and memsets only (no copy, no read-back, and
// no allocation once the workspaces have grown to the call's shapes); wide_batch_results reads the result area back (host
// and device forms).  A batch plan (plan.cu) calls the first at creation and the second on every run.
struct WideCall {
    const char *name = "";
    bool dev = false, gated = false;
    b200m_params p{};
    const b200m_wide_pair *pairs = nullptr;
    const b200m_local_pair *locals = nullptr;   // gated calls
    int n_pairs = 0;
    size_t stride_bytes = 0, xyz_stride_bytes = 0;
    int dim = 0, cluster_k = 0;
    float radius = 0.f;                          // gated calls: match_search_radius
    const float *thr_src = nullptr, *thr_tgt = nullptr;
    const b200m_corr *out = nullptr;             // dev: checked with the other pointers
    bool want_avg = false;
};
struct WideLayout {
    int n_scales = 0;   // 0: no pair has source keypoints and a scale -- nothing is queued
    bool two_way = false;
    size_t NS = 0, NT = 0;   // keypoints per side, all pairs
    b200m_params pk{};       // the kNN passes' params
    std::vector<std::vector<b200m_pair>> sets;   // [scale][pair] descriptor sets (empty past a pair's scales)
    std::vector<BatchLayout> scale_tables;       // keep_scales: every scale's batch tables, staged once
    char *d = nullptr;                           // the uploaded tables, the result area first
    size_t result_bytes = 0, o_avgs = 0, o_off[2] = {0, 0}, o_rad[2] = {0, 0}, o_segs = 0, o_gmap = 0, o_gxyz = 0;
    std::vector<size_t> o_rows, o_blk[2], o_map[2];
    size_t n_gmap = 0, max_map_rows = 0, max_kps[2] = {0, 0};
    // the result area: record count, bad-map key (~0 = clean), per-pair counts and averages
    unsigned long long *n_out = nullptr, *bad = nullptr;
    std::vector<int32_t> gmap_keys;   // dev: (side, scale, pair) of every map gather entry, in table order
    const GatherSet *thr_sets = nullptr;   // plans with live counts: [2][n_pairs] gathers of the thresholds into the dense keypoint
                                            // layout (else device thresholds are read in place)
    unsigned *counts = nullptr;
    float *avgs = nullptr;
};
// keep_scales (plans): also stage every scale's batch tables, each into a buffer of its own
int wide_batch_tables(b200m_ctx *ctx, const WideCall &c, WideLayout *W, bool keep_scales);
int wide_batch_enqueue(b200m_ctx *ctx, const WideCall &c, const WideLayout &W);
int wide_batch_results(b200m_ctx *ctx, const WideCall &c, const WideLayout &W, b200m_corr *out, size_t cap, size_t *offsets,
                       float *avg);
// The text of a bad-map key (flag_bad): "pair P, scale S: an index map entry of the source|target cloud is outside its
// keypoint range"; of an over-capacity key of a plan with live counts (side 2 / 3): "... the live source|target row count is
// above its capacity"
std::string map_status_text(unsigned long long key);

// multi.cu
void comm_release(b200m_ctx *ctx);

// local.cu: matchLocal with a finite radius over a cell list of the train keypoints; 0 = done, 1 = error, 2 = not worth a
// grid (the caller runs launch_local_rows)
void local_release(b200m_ctx *ctx);
int launch_local_cells(b200m_ctx *ctx, int direction, const float *d_query_xyz, const float *d_train_xyz, size_t xyz_stride_bytes,
                       float radius, int k, int32_t *d_idx, float *d_dist, int32_t *d_count);
// The batch form for b200m_match_multiscale_local_batch (wide_batch.cu): one scale and direction of every pair at once over
// the padded layout stage_batch left in the context; train indices come out as global padded rows.  Per side (0 = source,
// 1 = target) the scale's block -> pair table, row -> keypoint map over the padded rows and keypoint offsets ([n_pairs + 1]).
struct LocalBatch {
    int direction = 0, scale = 0, n_pairs = 0, k = 1;
    const int4 *rows = nullptr;   // [n_pairs] {first source row, source rows, first target row, target rows} of this scale
    const int32_t *blk[2] = {nullptr, nullptr}, *map[2] = {nullptr, nullptr}, *kp_off[2] = {nullptr, nullptr};
    const float *q_xyz = nullptr;   // the query side's keypoints MOVED by the guess (forward) / its inverse (reverse)
    const float *t_xyz = nullptr;   // the train side's keypoints, unmoved
    size_t xyz_stride_bytes = 16;
    float radius = 0.f;
    unsigned long long *bad = nullptr;   // flag_bad() key of the first out-of-range map entry
};
int launch_local_cells_batch(b200m_ctx *ctx, const LocalBatch &a, int32_t *d_idx, float *d_dist, int32_t *d_count);

// first out-of-range map entry of a batch call, smallest (scale, pair, side) wins; side 0 = a source map, 1 = a target map
__device__ __forceinline__ void flag_bad(unsigned long long *bad, int scale, int pair, int side) {
    atomicMin(bad, ((unsigned long long) scale << 48) | ((unsigned long long) pair << 16) | (unsigned long long) side);
}

// api.cu: kNN of query rows [row_begin, row_begin + n_rows) of `direction` on device buffers; with d_flags only the flagged
// (and valid) rows are answered, the others get empty lists.  Outputs are indexed by (row - row_begin).
// With seg (batch calls, no flags) every query row is answered from its own pair's train rows only.
extern "C" int b200m_knn_rows(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin, size_t n_rows, const uint8_t *d_flags,
                   int32_t *d_idx, float *d_dist, int32_t *d_count, const SegTable *seg = nullptr);
extern "C" {
int check_params(b200m_ctx *ctx, const b200m_params *p);
int check_upload_args(b200m_ctx *ctx, int side, const float *base, size_t n, size_t stride_bytes, int dim);
bool is_pageable(const void *p);
int staged_h2d(b200m_ctx *ctx, void *dst, const void *src, size_t bytes);   // pageable host -> device through pinned buffers
// pack `n` rows of device AoS data into side `side` (b200m_upload's device half)
// with `sets` the segmented pack of a device batch call (see launch_pack_f32)
int upload_common(b200m_ctx *ctx, int side, const float *device_aos, size_t n, size_t stride_bytes, int dim, int64_t index_offset,
                  const int32_t *seg_blk = nullptr, const SetRef *sets = nullptr);
}

// cluster.cu
void cluster_release(b200m_ctx *ctx);
// b200m_cluster_filter_device over many pairs' keypoints back to back (used by wide_batch.cu): the 3-D neighbourhoods stay inside a
// keypoint's own pair (src_off / tgt_off: [n_pairs + 1] first keypoint of every pair and the total), every id is global.
int cluster_filter_batch_device(b200m_ctx *ctx, const b200m_params *p, int cluster_k, float cluster_thr, size_t n_src, size_t n_tgt,
                                const int32_t *d_fidx, const float *d_fdist, const int32_t *d_fcount, const int32_t *d_ridx,
                                const int32_t *d_rcount, const float *d_src_xyz, const float *d_tgt_xyz, size_t xyz_stride_bytes,
                                const int32_t *d_src_off, const int32_t *d_tgt_off, int n_pairs, const float *d_thr_src,
                                const float *d_thr_tgt, b200m_corr *d_out, size_t cap, unsigned long long *d_n_out);
__device__ __forceinline__ int pair_of(const int32_t *__restrict__ off, int n_pairs, long long i) {
    // the last pair p with off[p] <= i (empty pairs share their offset with the next one)
    int lo = 0, hi = n_pairs;   // off[lo] <= i < off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}
