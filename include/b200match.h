/*
 * b200match.h -- C-ABI of libb200match.so: the B200 (sm_100a) descriptor-space
 * kNN correspondence search that replaces the reference's CPU matchers.
 *
 * The reference (aleksandrina-streltsova/lidar-global-registration) has no FFI
 * layer; its seams are C++ templates in include/matching.h.  Every entry point
 * below names the reference interface it stands in for (paths relative to the
 * reference root).  The C++ shim include/b200match_shim.hpp puts the reference's
 * own signatures (matchBF<FeatureT>, OneSided/LeftToRight/Ratio matchers) back
 * on top of these calls; INTEGRATION.md shows the binding a maintainer adds.
 *
 * Conventions: plain pointers and sizes only; return 0 = ok, non-zero = error
 * (message via b200m_last_error); the caller owns every host buffer, the
 * library owns device memory it allocates; one context per host thread, calls on
 * one context are serialised.  There is NO CPU fallback: without a CUDA device
 * b200m_create fails.
 */
#ifndef B200MATCH_H
#define B200MATCH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200M_API __attribute__((visibility("default")))

typedef struct b200m_ctx b200m_ctx;

/* == reference `Correspondence` (include/common.h:120-131): pcl::Correspondence
 * {int index_query; int index_match; float distance;} + float threshold -- 16 B. */
typedef struct {
    int32_t index_query;
    int32_t index_match;
    float distance;
    float threshold;
} b200m_corr;

/* filter policy == which reference matcher class the call stands in for */
enum {
    B200M_MODE_KNN_ONLY = 0,     /* raw k-lists: matchBF / matchFLANN / matchLocal(inf) seam, include/matching.h:368-383 */
    B200M_MODE_ONE_SIDED = 1,    /* OneSidedMatcher::match_impl, include/matching.h:395-411 */
    B200M_MODE_MUTUAL = 2,       /* LeftToRightMatcher::match_impl (k-list form), include/matching.h:428-453 */
    B200M_MODE_RATIO = 3,        /* RatioMatcher (reference stub :470-473; semantics from include/common.h:50-51) */
    B200M_MODE_RATIO_MUTUAL = 4, /* ratio test on the forward lists, then the mutual test */
    B200M_MODE_CLUSTER = 5       /* ClusterMatcher::match_impl, include/matching.h:492-517 (b200m_match_cluster only) */
};

/* how candidates are produced; the result is the same exact FP32 answer either way */
enum {
    B200M_PREC_TC_F16 = 0,   /* tcgen05 FP16-operand candidate pass (certified superset) + exact FP32 re-rank (default) */
    B200M_PREC_F32_EXACT = 2 /* CUDA-core exact FP32 brute force only (no tensor cores) */
};

/* The hot-path subset of the reference's AlignmentParameters (include/common.h:135-163):
 * k = randomness (:147), ratio_thr = MATCHING_RATIO_THRESHOLD (:50), distance_thr (:139). */
typedef struct {
    int32_t k;            /* neighbours per query, 1..32 */
    int32_t mode;         /* B200M_MODE_* */
    float ratio_thr;      /* 1.1f in the reference's constants */
    float distance_thr;   /* AlignmentParameters::distance_thr; caps the per-correspondence threshold */
    int32_t precision;    /* B200M_PREC_* */
    int32_t cand_cap;     /* candidate slots per query row and train split in the tensor-core pass
                             (0 = default chosen from k; rows that overflow go through the exact row kernel) */
    int32_t n_gpus;       /* multi-GPU calls: 0 = every rank of the communicator / group (the only value accepted besides
                             the communicator's size; kept for the reference-side config, SURVEY 8b) */
    int32_t shard;        /* multi-GPU calls: B200M_SHARD_QUERY (source rows split, target replicated) or
                             B200M_SHARD_TARGET (target rows split, per-query top-k merge) */
} b200m_params;

enum { B200M_SHARD_QUERY = 0, B200M_SHARD_TARGET = 1 };

/* per-call device timings and counters, filled by the *_device calls when
 * profiling is on (b200m_set_profiling); times are CUDA-event milliseconds on the
 * context's stream, accumulated since the last b200m_reset_stats. */
typedef struct {
    double ms_pack;        /* AoS -> f32 tiles + validity */
    double ms_prepare;     /* centring/scaling + FP16 operand tiles */
    double ms_candidates;  /* tcgen05 candidate kernel */
    double ms_rerank;      /* exact FP32 re-rank of the candidates */
    double ms_fallback;    /* exact row kernel over overflowed rows (or the whole F32_EXACT pass) */
    double ms_filter;      /* filter + compaction (+ average distance) */
    int64_t launches;      /* kernels launched by this library */
    int64_t candidate_launches;
    int64_t rows_total;    /* query rows processed by knn */
    int64_t rows_flagged;  /* rows whose candidate list overflowed and went through the exact row kernel */
    int64_t candidates;    /* candidate (query, train) pairs re-ranked exactly */
    int64_t rows_answered; /* query rows actually searched (masked kNN: the selected rows only) */
    int64_t pairs_scored;  /* (query, train) pairs whose distance the candidate kernel evaluated: sum of
                              rows_answered x train rows over the tensor-core launches */
} b200m_stats;

/* ---- context -------------------------------------------------------------- */
B200M_API int b200m_create(b200m_ctx **ctx, int device);
B200M_API void b200m_destroy(b200m_ctx *ctx);
B200M_API const char *b200m_last_error(const b200m_ctx *ctx); /* ctx may be NULL: last create error */
/* run on the caller's CUDA stream (a cudaStream_t passed as void*), e.g. torch's current stream; NULL = the
 * context's own non-blocking stream.  To name the legacy default stream pass cudaStreamLegacy ((void*)0x1). */
B200M_API int b200m_set_stream(b200m_ctx *ctx, void *cuda_stream);
B200M_API int b200m_sync(b200m_ctx *ctx);
B200M_API int b200m_set_profiling(b200m_ctx *ctx, int on);
B200M_API int b200m_get_stats(b200m_ctx *ctx, b200m_stats *out); /* synchronises the stream */
B200M_API int b200m_reset_stats(b200m_ctx *ctx);

/* ---- descriptor upload: replaces pcl2cv<FeatureT> (include/matching.h:553-560) --
 * side 0 = source (query of the forward pass), side 1 = target (train of the forward
 * pass).  `base` points at the first descriptor value of row 0, rows are
 * `stride_bytes` apart (sizeof(FeatureT): 132 FPFH33, 540 Histogram<135>, 1444 SHOT352),
 * `dim` leading floats of each row are the descriptor
 * (DefaultPointRepresentation<FeatureT>::getNumberOfDimensions()).
 * index_offset is added to every index reported for rows of this side (target
 * shards of a multi-GPU run report global row numbers). */
B200M_API int b200m_upload(b200m_ctx *ctx, int side, const float *host_base, size_t n,
                           size_t stride_bytes, int dim, int64_t index_offset);
B200M_API int b200m_upload_device(b200m_ctx *ctx, int side, const float *device_base, size_t n,
                                  size_t stride_bytes, int dim, int64_t index_offset);

/* ---- raw k-lists: replaces matchBF / matchFLANN / matchLocal(radius=inf) ---------
 * (include/matching.h:594-634, :562-592, :637-678).  direction 0: queries = side 0,
 * train = side 1; direction 1: roles swapped (the reverse pass of the mutual filter,
 * include/matching.h:432).  Query rows [row_begin,row_end) of the query side are
 * processed (row_end = 0 means "all"); outputs are (row_end-row_begin) x k, row-major:
 * idx (-1 padded), dist (L2, sqrt'ed, ascending; ties -> lower index), count.
 * Entry i is empty (count 0) for a non-finite query; non-finite train rows are never
 * returned. */
B200M_API int b200m_knn(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin,
                        size_t row_end, int32_t *idx, float *dist, int32_t *count);
B200M_API int b200m_knn_device(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin,
                               size_t row_end, int32_t *d_idx, float *d_dist, int32_t *d_count);

/* ---- masked kNN: only the flagged query rows are answered (the rest get empty lists) --------------
 * The mutual filter reads the reverse list of target row j only if some forward list names j
 * (LeftToRightMatcher::match_impl, include/matching.h:433-449), so the reverse pass may skip every other target row
 * (b200m_match does this by itself for large problems).  b200m_mark_referenced_device sets flags[j - index_offset] = 1
 * for every entry j of the given k-lists (flags must be zeroed by the caller; sharded runs OR / max-reduce the flags of
 * all ranks); b200m_knn_masked_device is b200m_knn_device restricted to rows with flags[row] != 0 (flags cover ALL rows of
 * the query side).  Device pointers, queued on the context's stream; one host round trip (the number of selected rows). */
B200M_API int b200m_mark_referenced_device(b200m_ctx *ctx, int k, const int32_t *d_fidx, const int32_t *d_fcount,
                                           size_t n_rows, int64_t index_offset, uint8_t *d_flags, size_t n_flags);
B200M_API int b200m_knn_masked_device(b200m_ctx *ctx, const b200m_params *p, int direction, size_t row_begin,
                                      size_t row_end, const uint8_t *d_row_flags, int32_t *d_idx, float *d_dist,
                                      int32_t *d_count);

/* ---- matchLocal with a finite match_search_radius (include/matching.h:637-678): the guess-conditioned kNN
 * match_multiscale uses when AlignmentParameters::guess is set (:297-304).  query_xyz: the query side's keypoints
 * AFTER the guess transform (pcl::transformPointCloudWithNormals, :644 -- done by the caller, so its arithmetic stays
 * PCL's), train_xyz: the train side's keypoints; one row per descriptor row, `xyz_stride_bytes` apart.  A train row
 * is considered iff its squared 3-D distance (FLANN L2_Simple) is < radius*radius; among equal descriptor distances the
 * spatially nearer row comes first (radiusSearch's sorted order + KNNResult), then the lower index.  Exact CUDA-core
 * path (one CTA per query row); outputs as b200m_knn's. */
B200M_API int b200m_knn_local(b200m_ctx *ctx, const b200m_params *p, int direction, const float *query_xyz,
                              const float *train_xyz, size_t xyz_stride_bytes, float radius, int32_t *idx,
                              float *dist, int32_t *count);
B200M_API int b200m_knn_local_device(b200m_ctx *ctx, const b200m_params *p, int direction, const float *d_query_xyz,
                                     const float *d_train_xyz, size_t xyz_stride_bytes, float radius,
                                     int32_t *d_idx, float *d_dist, int32_t *d_count);

/* ---- whole matcher call: replaces FeatureBasedMatcher::match()'s match_impl ------
 * (include/matching.h:395-411, :428-453) at the k-list seam, single GPU, host buffers.
 * thr_src / thr_tgt: optional per-point thresholds (calculateSmoothedDensities,
 * src/common.cpp:531-547) or NULL; emitted threshold = min(max(thr_src[i], thr_tgt[j]),
 * distance_thr).  out: capacity `cap` records, ascending index_query; *n_out = number
 * produced (error if cap is too small; nq*k always suffices).  avg_first_dist (may be
 * NULL) = FeatureBasedMatcher::getAverageDistance() (src/matching.cpp:3-19). */
B200M_API int b200m_match(b200m_ctx *ctx, const b200m_params *p, const float *thr_src,
                          const float *thr_tgt, b200m_corr *out, size_t cap, size_t *n_out,
                          float *avg_first_dist);

/* ---- batches: many independent (source, target) pairs in one call -----------------------------
 * Multi-view registration (all pairs of N scans), one scan against many submaps, or a whole table of evaluation
 * pairs: one call per direction fills the GPU instead of one small call per pair.  All pairs share the descriptor
 * type (stride_bytes, dim) and the params.  Pair p's output equals, byte for byte, what b200m_upload(0, src_p),
 * b200m_upload(1, tgt_p) and then b200m_knn (direction 0, all rows) / b200m_match on that pair alone return, with
 * pair-local indices.  Empty sets are allowed on either side (empty lists, no records).  A batch call REPLACES the
 * descriptor sets b200m_upload put in the context (upload again before the next single-pair call).  Host pointers. */
typedef struct {
    const float *src;   /* first descriptor value of source row 0 (rows stride_bytes apart) */
    size_t n_src;
    const float *tgt;
    size_t n_tgt;
} b200m_pair;
/* raw k-lists of every pair, direction 0: rows concatenated in pair order ([sum n_src][k], [sum n_src]), pair-local train
 * indices, -1 padded as b200m_knn's */
B200M_API int b200m_knn_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                              size_t stride_bytes, int dim, int32_t *idx, float *dist, int32_t *count);
/* b200m_match of every pair (modes as b200m_match accepts; CLUSTER is an error): records of pair p are
 * out[offsets[p] .. offsets[p+1]), ascending index_query, pair-local indices; offsets has n_pairs + 1 entries and is
 * filled also when cap is too small (error; sum n_src * k always suffices); avg (may be NULL) gets n_pairs averages;
 * thr_src / thr_tgt are the pairs' thresholds concatenated in pair order (sum n_src / sum n_tgt floats) or both NULL. */
B200M_API int b200m_match_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                                size_t stride_bytes, int dim, const float *thr_src, const float *thr_tgt,
                                b200m_corr *out, size_t cap, size_t *offsets, float *avg);

/* ---- device-side building blocks for sharded (multi-GPU) runs ----------------
 * All pointers are device pointers on the context's device; work is queued on the
 * context's stream.  Forward tables cover query rows [row_begin,row_end) of side 0;
 * the reverse table (mutual modes) covers ALL rows of side 1 and carries side-0 row
 * numbers.  d_n_out: one device size_t-sized (uint64) counter; d_avg may be NULL. */
B200M_API int b200m_filter_device(b200m_ctx *ctx, const b200m_params *p, size_t row_begin, size_t row_end,
                                  const int32_t *d_fidx, const float *d_fdist, const int32_t *d_fcount,
                                  const int32_t *d_ridx, const float *d_rdist, const int32_t *d_rcount,
                                  size_t n_rev_rows, const float *d_thr_src, const float *d_thr_tgt,
                                  b200m_corr *d_out, size_t cap, unsigned long long *d_n_out, float *d_avg);
/* per-query merge of `n_lists` k-lists (target-sharded run after the all-gather):
 * tables are [n_lists][nq][k] / [n_lists][nq]; keeps the k best by (dist, idx) --
 * the cross-block role of updateMultivaluedCorrespondence (src/common.cpp:517-529)
 * under the canonical tie rule. */
B200M_API int b200m_merge_device(b200m_ctx *ctx, int k, int n_lists, size_t nq,
                                 const int32_t *d_idx_in, const float *d_dist_in, const int32_t *d_count_in,
                                 int32_t *d_idx, float *d_dist, int32_t *d_count);

/* ---- multi-scale merge + spatial vote: the tail of match_multiscale -------------
 * (include/matching.h:264-354).  The reference runs one kNN per scale over that scale's
 * keypoint subset and descriptors (:297-311), remaps per-scale row numbers to keypoint ids
 * (:313-321, kps_indices_multiscale), concatenates the candidates per query keypoint in scale
 * order and lets a spatial vote keep at most ONE match per keypoint (:327-352).  Here:
 *   b200m_multiscale_begin(n_query_kps, n_scales, k)
 *   per scale:  b200m_upload(query side, ...); b200m_upload(train side, ...);
 *               b200m_multiscale_add(params, direction, scale, query_map, train_map, n_train_kps)
 *                   -- runs the scale's kNN (as b200m_knn would) and files the lists under
 *                      query_map[row] with train rows renamed train_map[row] (NULL = identity)
 *   b200m_multiscale_vote(train_xyz, n_train_kps, stride, iss_radius, idx, dist, count)
 *                   -- outputs are [n_query_kps]: the chosen train keypoint id (or -1), its
 *                      descriptor distance, count 0/1 -- the one-entry MultivaluedCorrespondence
 *                      match_multiscale returns; xyz rows are `stride` bytes apart (pcl::PointXYZ: 16).
 * The *_device forms take device pointers (k-lists from b200m_knn_device) and queue on the stream. */
B200M_API int b200m_multiscale_begin(b200m_ctx *ctx, size_t n_query_kps, int n_scales, int k);
B200M_API int b200m_multiscale_add(b200m_ctx *ctx, const b200m_params *p, int direction, int scale,
                                   const int32_t *query_map, const int32_t *train_map, size_t n_train_kps);
B200M_API int b200m_multiscale_vote(b200m_ctx *ctx, const float *train_xyz, size_t n_train_kps,
                                    size_t xyz_stride_bytes, float iss_radius, int32_t *idx, float *dist,
                                    int32_t *count);
B200M_API int b200m_multiscale_add_device(b200m_ctx *ctx, int scale, size_t n_rows, const int32_t *d_idx,
                                          const float *d_dist, const int32_t *d_count,
                                          const int32_t *d_query_map, const int32_t *d_train_map,
                                          size_t n_train_rows, int64_t train_index_offset, size_t n_train_kps);
B200M_API int b200m_multiscale_vote_device(b200m_ctx *ctx, const float *d_train_xyz, size_t xyz_stride_bytes,
                                           float iss_radius, int32_t *d_idx, float *d_dist, int32_t *d_count);

/* ---- ClusterMatcher<FeatureT>::match_impl (include/matching.h:492-517), the reference's default matching_id --
 * A forward pair (i, j) survives when, of the matches of i's cluster_k nearest keypoints (3-D,
 * pcl KdTree nearestKSearch on the keypoint cloud, i itself included), fewer than
 * MATCHING_CLUSTER_THRESHOLD (0.95) fail to land among j's cluster_k nearest keypoints -- and the same with the
 * roles swapped over the reverse k-lists (calculateCorrespondenceDistance, :519-550).  Emitted distance =
 * max(d_i, d_j), threshold as in b200m_match, ascending index_query then list order.
 * b200m_match_cluster: whole call on host buffers over the uploaded sides (forward and reverse kNN, k = p->k, the
 *   reference's two match_multiscale calls); src/tgt_kps_xyz are the keypoint coordinates of side 0 / side 1, one row
 *   per descriptor row, `xyz_stride_bytes` apart (pcl::PointXYZ: 16).  cluster_k = AlignmentParameters::cluster_k
 *   (MATCHING_CLUSTER_K = 40, include/common.h:53), at most 64.
 * b200m_cluster_filter_device: the filter alone on device k-lists (e.g. b200m_multiscale_vote_device outputs with
 *   p->k = 1); b200m_knn3d_device: the 3-D neighbourhoods alone ([n][k] int32, -1 padded when n < k; neighbours are
 *   chosen by (squared distance, lower index)). */
B200M_API int b200m_match_cluster(b200m_ctx *ctx, const b200m_params *p, int cluster_k, const float *src_kps_xyz,
                                  const float *tgt_kps_xyz, size_t xyz_stride_bytes, const float *thr_src,
                                  const float *thr_tgt, b200m_corr *out, size_t cap, size_t *n_out,
                                  float *avg_first_dist);
B200M_API int b200m_cluster_filter_device(b200m_ctx *ctx, const b200m_params *p, int cluster_k, float cluster_thr,
                                          size_t n_src, size_t n_tgt, const int32_t *d_fidx, const float *d_fdist,
                                          const int32_t *d_fcount, const int32_t *d_ridx, const int32_t *d_rcount,
                                          const float *d_src_xyz, const float *d_tgt_xyz, size_t xyz_stride_bytes,
                                          const float *d_thr_src, const float *d_thr_tgt, b200m_corr *d_out,
                                          size_t cap, unsigned long long *d_n_out, float *d_avg);
B200M_API int b200m_knn3d_device(b200m_ctx *ctx, const float *d_xyz, size_t n, size_t xyz_stride_bytes, int k,
                                 int32_t *d_nbr);

/* ---- multi-GPU: the partitioning of SURVEY 8e inside the library (NCCL over NVLink, bound at run time) ----------------
 * Rank r of W owns rows [r*R, min(n, (r+1)*R)), R = ceil(n / W) (b200m_shard_rows).
 *
 * (1) One process per GPU: create a context per process, exchange a B200M_UNIQUE_ID_BYTES id made by
 *     b200m_comm_unique_id on one rank (any transport: MPI, torch.distributed, a file), b200m_comm_attach on every rank,
 *     then call the *_sharded entry points COLLECTIVELY (every rank, same arguments, same order):
 *       b200m_upload_replicated      every rank holds the whole HOST set: rank r copies 1/W of it over PCIe, the slices are
 *                                    all-gathered over NVLink, the pack kernel runs on the full set (or use
 *                                    b200m_upload[_device] per rank when the set is already resident)
 *       b200m_match_sharded[_device] the whole matcher call, query-sharded / target-replicated: forward kNN of this rank's
 *                                    source rows, reverse kNN of this rank's (referenced) target rows, ONE all-gather of the
 *                                    reverse table, filter of this rank's rows.  Output = this rank's slice, ascending
 *                                    index_query; the slices in rank order are the single-GPU output.  The average is the
 *                                    one over ALL source rows on every rank.
 *       b200m_knn_target_sharded_device   side 1 = this rank's target shard (uploaded with index_offset = its first
 *                                    global row), side 0 all queries: exact local top-k, all-gather, merge -> every rank
 *                                    holds the full k-lists (BASELINE configs[4]; at most 8 ranks).
 * (2) One process, several GPUs -- the reference's shape (one FeatureBasedMatcher::match() call in one address space,
 *     src/correspondence_search.cpp:14-15): b200m_create_multi makes one context per device plus one host thread per
 *     device inside the library; the b200m_group_* calls take and return WHOLE host arrays. */
#define B200M_UNIQUE_ID_BYTES 128
B200M_API int b200m_comm_unique_id(void *id_out, size_t bytes);
B200M_API int b200m_comm_attach(b200m_ctx *ctx, int n_ranks, int rank, const void *unique_id);
B200M_API int b200m_comm_rank(const b200m_ctx *ctx, int *rank, int *n_ranks);
B200M_API int b200m_shard_rows(size_t n, int n_ranks, int rank, size_t *row_begin, size_t *row_end);
B200M_API int b200m_upload_replicated(b200m_ctx *ctx, int side, const float *host_base, size_t n, size_t stride_bytes,
                                      int dim);
B200M_API int b200m_match_sharded(b200m_ctx *ctx, const b200m_params *p, const float *thr_src, const float *thr_tgt,
                                  b200m_corr *out, size_t cap, size_t *n_out, float *avg_first_dist);
B200M_API int b200m_match_sharded_device(b200m_ctx *ctx, const b200m_params *p, const float *d_thr_src,
                                         const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                         unsigned long long *d_n_out, float *d_avg);
B200M_API int b200m_knn_target_sharded_device(b200m_ctx *ctx, const b200m_params *p, int32_t *d_idx, float *d_dist,
                                              int32_t *d_count);

typedef struct b200m_group b200m_group;
B200M_API int b200m_create_multi(b200m_group **group, const int *device_ids, int n);
B200M_API void b200m_destroy_multi(b200m_group *group);
B200M_API const char *b200m_group_last_error(const b200m_group *group); /* group may be NULL: last create error */
B200M_API int b200m_group_size(const b200m_group *group);
B200M_API b200m_ctx *b200m_group_ctx(b200m_group *group, int i);        /* e.g. for b200m_get_stats */
/* replicated upload (query-sharded runs) / row-sharded upload with global index offsets (target-sharded runs) */
B200M_API int b200m_group_upload(b200m_group *group, int side, const float *host_base, size_t n, size_t stride_bytes,
                                 int dim);
B200M_API int b200m_group_upload_sharded(b200m_group *group, int side, const float *host_base, size_t n,
                                         size_t stride_bytes, int dim);
/* == b200m_match / b200m_knn(direction 0, all rows) on the whole problem; p->shard picks the partition for the kNN
 * (B200M_SHARD_TARGET needs the target uploaded with b200m_group_upload_sharded) */
B200M_API int b200m_group_match(b200m_group *group, const b200m_params *p, const float *thr_src, const float *thr_tgt,
                                b200m_corr *out, size_t cap, size_t *n_out, float *avg_first_dist);
B200M_API int b200m_group_knn(b200m_group *group, const b200m_params *p, int32_t *idx, float *dist, int32_t *count);

/* ---- the matcher classes at the WIDE seam: FeatureBasedMatcherImpl<FeatureT>::match_impl -------------------------
 * (include/matching.h:395-411 OneSidedMatcher, :428-453 LeftToRightMatcher, :492-517 ClusterMatcher), composed as
 * the reference composes it: match_multiscale in both directions (per-scale kNN with k = p->k = randomness, remap
 * to keypoint ids, concatenation, spatial vote -> at most ONE match per keypoint, :264-354; the reverse direction is
 * the reference's inverse_tn call), printDebugInfo's average over the VOTED forward lists, then the matcher's filter
 * loop over the voted lists.  p->mode: ONE_SIDED, MUTUAL or CLUSTER.
 * scales[s] (ascending log2 radius, the scales common to both clouds): the two clouds' descriptor rows of that scale
 * (kps_features_multiscale[s]: host pointers, rows `stride_bytes` apart, `dim` leading floats) and the row -> keypoint
 * id maps (kps_indices_multiscale[s]; NULL = identity).  src/tgt_kps_xyz: st_src_.kps / st_tgt_.kps coordinates, one
 * row per keypoint, `xyz_stride_bytes` apart; iss_radius_src/tgt: Storage::iss_radius of the two clouds (the vote over
 * the forward lists uses the TARGET keypoints and iss_radius_tgt).  cluster_k: AlignmentParameters::cluster_k (CLUSTER
 * mode only).  Outputs as b200m_match's: records in ascending index_query (keypoint ids; finalize's map to cloud
 * indices stays with the caller), at most n_src_kps of them. */
typedef struct {
    const float *src_desc;   /* source cloud, this scale: first descriptor value of row 0 */
    size_t n_src;
    const int32_t *src_map;  /* [n_src] row -> source keypoint id, or NULL */
    const float *tgt_desc;
    size_t n_tgt;
    const int32_t *tgt_map;  /* [n_tgt] row -> target keypoint id, or NULL */
} b200m_scale;
B200M_API int b200m_match_multiscale(b200m_ctx *ctx, const b200m_params *p, const b200m_scale *scales, int n_scales,
                                     size_t stride_bytes, int dim, const float *src_kps_xyz, size_t n_src_kps,
                                     const float *tgt_kps_xyz, size_t n_tgt_kps, size_t xyz_stride_bytes,
                                     float iss_radius_src, float iss_radius_tgt, int cluster_k, const float *thr_src,
                                     const float *thr_tgt, b200m_corr *out, size_t cap, size_t *n_out,
                                     float *avg_first_dist);

/* ---- the matcher classes at the WIDE seam, many (source, target) cloud pairs in one call ------------------------------
 * b200m_match_multiscale of every pair: multi-view registration, one scan against many submaps or an evaluation table
 * run their OneSided / LeftToRight / ClusterMatcher calls as one batch.  Pair p's records and average equal, byte for
 * byte, what b200m_match_multiscale returns for pair p alone (with pair-local keypoint ids), the masked reverse pass
 * included (its output is the same).  All pairs share the descriptor type (stride_bytes, dim), the keypoint row stride,
 * the params and cluster_k; each pair has its own scales (its common scales, ascending; 0..32 of them, n_scales * k <=
 * 128), keypoint coordinates and radii.  The validation rules per pair are b200m_match_multiscale's; an error names the
 * pair (and the scale).  A pair without source keypoints or without scales gives no records and the average FLT_MAX.
 * Per scale the pairs' descriptor sets are packed as b200m_match_batch packs them and answered by one kNN pass per
 * direction; the votes, the filter and the 3-D neighbourhoods of the cluster filter run once over all pairs, each pair's
 * neighbourhoods inside its own keypoints.
 * Outputs as b200m_match_batch's: records of pair p are out[offsets[p] .. offsets[p+1]) (at most n_src_kps each;
 * offsets has n_pairs + 1 entries and is filled also when cap is too small), avg (may be NULL) gets n_pairs averages,
 * thr_src / thr_tgt are the pairs' per-keypoint thresholds concatenated in pair order (sum n_src_kps / sum n_tgt_kps
 * floats) or both NULL.  Like the other batch calls, this call REPLACES the descriptor sets b200m_upload put in the
 * context.  Host pointers. */
typedef struct {
    const b200m_scale *scales;   /* this pair's common scales, ascending; n_scales in [0, 32] */
    int n_scales;
    const float *src_kps_xyz;    /* n_src_kps rows, xyz_stride_bytes apart (may be NULL in ONE_SIDED mode) */
    size_t n_src_kps;
    const float *tgt_kps_xyz;
    size_t n_tgt_kps;
    float iss_radius_src, iss_radius_tgt;
} b200m_wide_pair;
B200M_API int b200m_match_multiscale_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs, int n_pairs,
                                           size_t stride_bytes, int dim, size_t xyz_stride_bytes, int cluster_k,
                                           const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap,
                                           size_t *offsets, float *avg);

/* ---- the matcher classes at the WIDE seam with AlignmentParameters::guess set, many cloud pairs in one call ----------
 * With a guess, match_multiscale answers every scale with matchLocal (include/matching.h:297-311, :637-678): the query
 * keypoints are moved by the guess (the reverse call, inverse_tn, by its inverse) and only train keypoints within
 * match_search_radius compete.  This is b200m_match_multiscale_batch with that kNN: for pair p and scale s, source row r
 * is gated at src_kps_moved[src_map[r]] against the target keypoints tgt_kps_xyz (unmoved); in the reverse pass target
 * row c is gated at tgt_kps_moved[tgt_map[c]] against the source keypoints (unmoved).  The gate and the order are
 * b200m_knn_local's: FP32 L2_Simple squared distance < radius*radius (radius 0 or NaN: nothing passes; FLT_MAX or inf:
 * every finite row), entries ordered by (descriptor distance, spatial distance, index), a non-finite query keypoint or
 * descriptor gets an empty list, a non-finite train row is never returned.  The moved coordinates come from the caller
 * (pcl::transformPointCloudWithNormals in a PCL build), so the transform's arithmetic stays the caller's; the library never
 * inverts a matrix.  Everything after the kNN -- remap, votes over the unmoved keypoints, average, filter, outputs and
 * errors -- is b200m_match_multiscale_batch's.  p->precision does not apply (exact CUDA-core path).  A single pair is a
 * batch of one.  Host pointers; this call REPLACES the descriptor sets b200m_upload put in the context. */
typedef struct {
    const float *src_kps_moved;   /* n_src_kps rows, xyz_stride_bytes apart: the source keypoints moved by this pair's guess */
    const float *tgt_kps_moved;   /* n_tgt_kps rows: the target keypoints moved by the guess's inverse (may be NULL in
                                     ONE_SIDED mode) */
} b200m_local_pair;
B200M_API int b200m_match_multiscale_local_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                 const b200m_local_pair *locals, int n_pairs, size_t stride_bytes, int dim,
                                                 size_t xyz_stride_bytes, int cluster_k, float match_search_radius,
                                                 const float *thr_src, const float *thr_tgt, b200m_corr *out, size_t cap,
                                                 size_t *offsets, float *avg);

/* ---- device-resident batch calls: the four batch calls on descriptors, maps, keypoints and records in HBM -------------
 * For a caller whose sets already live on the GPU (a GPU feature stage, a torch pipeline, sets reused across calls).
 * Each takes its host form's arguments: the arrays of b200m_pair / b200m_wide_pair / b200m_scale / b200m_local_pair and
 * every size and radius in them stay HOST memory, but every data pointer inside them (descriptors, index maps, keypoint
 * coordinates, moved keypoints) and the threshold arrays are DEVICE pointers on the context's device.  Different pairs may
 * point at the same memory (one scan against many submaps).  Pair p's records, offsets, average and k-lists are byte for
 * byte what the host form returns on the same data; validation, errors (under the new name), "replaces the uploaded sets"
 * and the capacity rule are the host form's.
 * Outputs: b200m_knn_batch_device writes d_idx [sum n_src][k], d_dist and d_count (device); the match calls write the
 * records to d_out (device, `cap` records) and offsets [n_pairs + 1] / avg [n_pairs] to HOST arrays (the call reads its
 * result area back once anyway, and the caller needs host integers to split the records).  Work is queued on the
 * context's stream; on return the records and k-lists are ordered on that stream, not yet complete.
 * Every non-null data pointer is checked with cudaPointerGetAttributes before anything is queued: it must be device or
 * managed memory of the context's device, otherwise the call fails with an error naming the pair, scale and field.
 * Only the call's own tables go host -> device (segment, row and block tables, offsets, radii); the descriptors are
 * packed where they are and maps, coordinates and thresholds are filed by one gather kernel per table, so the number of
 * launches and copies does not depend on n_pairs (DESIGN.md section 3.14). */
B200M_API int b200m_knn_batch_device(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                                     size_t stride_bytes, int dim, int32_t *d_idx, float *d_dist, int32_t *d_count);
B200M_API int b200m_match_batch_device(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                                       size_t stride_bytes, int dim, const float *d_thr_src, const float *d_thr_tgt,
                                       b200m_corr *d_out, size_t cap, size_t *offsets, float *avg);
B200M_API int b200m_match_multiscale_batch_device(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                  int n_pairs, size_t stride_bytes, int dim, size_t xyz_stride_bytes,
                                                  int cluster_k, const float *d_thr_src, const float *d_thr_tgt,
                                                  b200m_corr *d_out, size_t cap, size_t *offsets, float *avg);
B200M_API int b200m_match_multiscale_local_batch_device(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                        const b200m_local_pair *locals, int n_pairs, size_t stride_bytes,
                                                        int dim, size_t xyz_stride_bytes, int cluster_k,
                                                        float match_search_radius, const float *d_thr_src,
                                                        const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                                        size_t *offsets, float *avg);

/* ---- batch plans: device batch calls bound once, enqueued without the host --------------------------------------------
 * A plan binds b200m_knn_batch_device's / b200m_match_batch_device's arguments: *p, the pairs (their device pointers and
 * sizes), the stride, dim, the threshold and output pointers.  Creation does every check of the device form (same error
 * texts, in ctx's last error), builds and uploads the batch tables, allocates every workspace in a context of the plan's
 * own (on ctx's device, with the same environment settings; later calls on ctx cannot move the plan's memory) and runs the
 * batch once on ctx's stream, synchronised (the outputs are written), so that every kernel module is loaded.
 * b200m_plan_run then only enqueues kernels and memsets on `cuda_stream` (NULL: the legacy default stream): no host round
 * trip, allocation, host <-> device copy or pointer query, so it may be captured into a CUDA graph (global capture mode),
 * and a run (or a replay) after the inputs were rewritten in place gives what the device form gives on the new data.  The
 * routing between tensor cores and the exact path is decided on the device.  Profiling (b200m_set_profiling) does not
 * apply to plans.  Destroy a plan only when no work or graph that uses it is left.
 * Match plans: records of pair p are d_out[d_offsets[p] .. d_offsets[p+1]) as b200m_match_batch_device's; d_n_out gets the
 * number of records found and only the first min(*d_n_out, cap) are written (*d_n_out > cap: truncated, nothing past cap
 * is touched); d_offsets are always the full offsets; d_avg (may be NULL) gets the averages (FLT_MAX for a batch without
 * source rows).  d_offsets [n_pairs + 1], d_n_out [1]. */
typedef struct b200m_plan b200m_plan;
B200M_API int b200m_plan_knn_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                                   size_t stride_bytes, int dim, int32_t *d_idx, float *d_dist, int32_t *d_count,
                                   b200m_plan **plan);
B200M_API int b200m_plan_match_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                                     size_t stride_bytes, int dim, const float *d_thr_src, const float *d_thr_tgt,
                                     b200m_corr *d_out, size_t cap, uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out,
                                     b200m_plan **plan);
/* Plans with live counts: the same plans for sets whose sizes change from run to run (a stream of scans with a different
 * number of keypoints each).  Every n_src / n_tgt of the pairs is a CAPACITY: the most rows the plan will ever answer for
 * that set (the pointers must hold that many rows).  d_rows [n_pairs][2] (device) holds the live (source rows, target
 * rows) of every pair; every run reads it at its start, so the caller rewrites counts and rows in place between runs or
 * graph replays.  Pair p's outputs are, byte for byte, what the device form gives on the live prefixes: the first n rows
 * of each set and the first n thresholds of the pair's slice.  Rows past a live count are never read (they may hold
 * anything).  Layouts:
 *   thresholds   capacity layout: pair p's slice starts at the sum of the earlier pairs' capacities (one tensor per side);
 *   records      dense, with d_offsets, as the match plan writes them;
 *   k-lists      capacity layout: pair p's rows start at the sum of the earlier pairs' source capacities (d_idx / d_dist
 *                [sum n_src][k], d_count [sum n_src]); rows from the live count up to the capacity hold the empty list
 *                (index -1, distance 0, count 0), so a consumer sees fixed addresses.
 * A count above its capacity makes its pair answer as empty (no records, empty lists, the average FLT_MAX of a pair without
 * source rows; nothing past the capacity is read or written; the other pairs are unaffected), and d_status (device, one
 * word) gets the key of the first such pair, in the layout of the matcher-class plans' status word: (pair << 16) | side
 * with side 2 = source rows, 3 = target rows and scale 0; ~0 when every count fits.  Every run starts from a clean key.
 * Creation runs once, synchronised, on the live counts d_rows holds then, and fails with the status text when a count is
 * above its capacity. */
B200M_API int b200m_plan_knn_batch_rows(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                                        size_t stride_bytes, int dim, int32_t *d_idx, float *d_dist, int32_t *d_count,
                                        const uint32_t *d_rows, uint64_t *d_status, b200m_plan **plan);
B200M_API int b200m_plan_match_batch_rows(b200m_ctx *ctx, const b200m_params *p, const b200m_pair *pairs, int n_pairs,
                                          size_t stride_bytes, int dim, const float *d_thr_src, const float *d_thr_tgt,
                                          b200m_corr *d_out, size_t cap, uint64_t *d_offsets, float *d_avg,
                                          uint64_t *d_n_out, const uint32_t *d_rows, uint64_t *d_status, b200m_plan **plan);
/* Matcher-class plans: b200m_match_multiscale_batch_device's / b200m_match_multiscale_local_batch_device's arguments, with
 * the offsets and averages on the device and two more device words, d_n_out and d_status.  Creation copies the host arrays
 * (pairs, their scales, locals) and binds the device pointers inside them; every scale's tables are built once.  A run
 * re-gathers every map and coordinate table, packs and matches every scale, votes, filters, averages and localises, then
 * writes d_offsets [n_pairs + 1], d_avg [n_pairs] (may be NULL; FLT_MAX for a pair without voted forward lists and for
 * every pair of a batch without source keypoints), d_n_out and the first min(*d_n_out, cap) records, as match plans do
 * (cap = the total source keypoints is always enough: the voted lists hold at most one match per source keypoint).
 * d_status gets the bad-map key, a public layout: ~0 when every map entry was in range, otherwise the first bad entry by
 * (scale, pair, side) as (scale << 48) | (pair << 16) | side, side 0 = a source map, 1 = a target map.  Every run starts
 * from a clean key, so a replay after the map was fixed reports ~0 again.  Creation fails, with the device form's text,
 * when its own run finds a bad entry. */
B200M_API int b200m_plan_match_multiscale_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                int n_pairs, size_t stride_bytes, int dim, size_t xyz_stride_bytes,
                                                int cluster_k, const float *d_thr_src, const float *d_thr_tgt,
                                                b200m_corr *d_out, size_t cap, uint64_t *d_offsets, float *d_avg,
                                                uint64_t *d_n_out, uint64_t *d_status, b200m_plan **plan);
B200M_API int b200m_plan_match_multiscale_local_batch(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                      const b200m_local_pair *locals, int n_pairs, size_t stride_bytes,
                                                      int dim, size_t xyz_stride_bytes, int cluster_k,
                                                      float match_search_radius, const float *d_thr_src,
                                                      const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                                      uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out,
                                                      uint64_t *d_status, b200m_plan **plan);
/* Matcher-class plans with live counts: the same plans for keypoint clouds whose sizes change from run to run.  Every
 * n_src_kps / n_tgt_kps and every scale's n_src / n_tgt is a CAPACITY (the bound keypoints, maps, descriptors, moved
 * keypoints and thresholds hold that many rows).  d_kps [n_pairs][2] (device) holds the live (source, target) keypoints of
 * every pair and d_rows [sum of the pairs' n_scales][2] (device, pair-then-scale order) the live (source, target) rows of
 * every scale; every run reads both at its start.  The number of pairs and each pair's number of scales stay as created.
 * Pair p's records, offsets and average are byte for byte the device form's on the live prefixes: the first n keypoints,
 * moved keypoints and thresholds, the first n rows of each scale's descriptors and index maps.  Rows past a live count are
 * never read (out-of-range map entries there are not reported).  Thresholds use the capacity layout: pair p's slice starts
 * at the sum of the earlier pairs' keypoint capacities.  A count above its capacity makes its pair answer as empty (no
 * records, average FLT_MAX), and d_status gets the key of the first such count with side 2 = source, 3 = target and
 * scale = the scale of a row count or 0xFFFF for a keypoint count; a bad map entry in the live rows keys as before, and
 * the smaller key wins.  Creation fails with the status text when its own run finds either. */
B200M_API int b200m_plan_match_multiscale_batch_rows(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                     int n_pairs, size_t stride_bytes, int dim, size_t xyz_stride_bytes,
                                                     int cluster_k, const float *d_thr_src, const float *d_thr_tgt,
                                                     b200m_corr *d_out, size_t cap, uint64_t *d_offsets, float *d_avg,
                                                     uint64_t *d_n_out, uint64_t *d_status, const uint32_t *d_kps,
                                                     const uint32_t *d_rows, b200m_plan **plan);
B200M_API int b200m_plan_match_multiscale_local_batch_rows(b200m_ctx *ctx, const b200m_params *p, const b200m_wide_pair *pairs,
                                                           const b200m_local_pair *locals, int n_pairs, size_t stride_bytes,
                                                           int dim, size_t xyz_stride_bytes, int cluster_k,
                                                           float match_search_radius, const float *d_thr_src,
                                                           const float *d_thr_tgt, b200m_corr *d_out, size_t cap,
                                                           uint64_t *d_offsets, float *d_avg, uint64_t *d_n_out,
                                                           uint64_t *d_status, const uint32_t *d_kps, const uint32_t *d_rows,
                                                           b200m_plan **plan);
B200M_API int b200m_plan_run(b200m_plan *plan, void *cuda_stream); /* enqueue only */
B200M_API void b200m_plan_destroy(b200m_plan *plan);
B200M_API const char *b200m_plan_last_error(const b200m_plan *plan); /* plan may be NULL: errors without a plan */
/* The text of a status word: NULL for ~0, else "pair P, scale S: an index map entry of the source|target cloud is outside
 * its keypoint range" (side 0 / 1) -- the device forms fail with this text after their name -- or "pair P, scale S: the
 * live source|target row count is above its capacity" (side 2 / 3, the plans with live counts) or, for scale 0xFFFF, "pair
 * P: the live source|target keypoint count is above its capacity".  Valid until the next call
 * with the same plan (plan may be NULL). */
B200M_API const char *b200m_plan_status_error(const b200m_plan *plan, uint64_t status);

B200M_API int b200m_version(void);

/* ---- test hooks (used by tests/ only; not part of the reference-facing surface) ----
 * b200m_debug_operands: copy the FP16 operand tiles the tensor-core pass reads to the host:
 *   as_query=1 -> [n_pad][kp] rows (-2*x16, 1,1,1, 0..), else the train form (x16, |x16|^2 hi/mid/lo, 0..);
 *   norm16 (may be NULL) receives |x16|^2 per row [n_pad]; scale/kp/n_pad are returned through the pointers.
 * b200m_debug_tc_tile: raw tensor-core accumulators (|b16|^2 - 2 a16.b16) of query rows
 *   [q_row0, q_row0+128) x train rows [t_tile*256, +256) of `direction`, row-major [128][256]. */
B200M_API int b200m_debug_operands(b200m_ctx *ctx, int side, int as_query, uint16_t *host_out, size_t out_halves,
                                   float *norm16, float *scale, int32_t *kp, int64_t *n_pad);
B200M_API int b200m_debug_tc_tile(b200m_ctx *ctx, int direction, size_t q_row0, size_t t_tile, float *host_out);

#ifdef __cplusplus
}
#endif
#endif /* B200MATCH_H */
