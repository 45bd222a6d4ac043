// b200match_shim.hpp -- header-only C++ host mirror of the reference's matcher interface on top of
// the C-ABI in b200match.h.  It puts the reference's own names and signatures back:
//
//   matchBF<FeatureT> / matchFLANN<FeatureT> / matchLocal<FeatureT>(radius = inf)
//                                  reference include/matching.h:368-383, :562-678
//   knnBatch<FeatureT> / matchBatch<FeatureT>
//                                  many (source, target) cloud pairs in one call: matchBF / the k-list filter per pair
//   MultivaluedCorrespondence      reference include/common.h:192-195
//   Correspondence                 reference include/common.h:120-127
//   FeatureBasedMatcher, FeatureBasedMatcherImpl<FeatureT>::Storage, OneSidedMatcher / LeftToRightMatcher /
//   RatioMatcher / ClusterMatcher  (match(), getAverageDistance(), getClassName())
//                                  reference include/matching.h:25-42, :96-161, :385-551
//   matchMany<FeatureT>            match() of many OneSided / LeftToRight / ClusterMatchers (cloud pairs) in one call
// With AlignmentParameters::guess set, the matcher classes and matchMany run match_multiscale's matchLocal form
// (b200m_match_multiscale_local_batch): each scale's kNN gated at match_search_radius around the moved keypoints.
// The matcher classes run match_impl as the reference composes it -- match_multiscale (per-scale kNN, spatial vote ->
// at most one match per keypoint) in one or both directions, then the filter over the voted lists -- in ONE library
// call (b200m_match_multiscale); the narrow-seam functions share one context per host thread and device, so calling
// them per scale and per direction does not pay for streams and device allocations again.
//
// With -DB200MATCH_WITH_PCL the feature types are PCL's (pcl::FPFHSignature33, pcl::SHOT352,
// pcl::Histogram<135>, pcl::UniqueShapeContext1960) and clouds are pcl::PointCloud<FeatureT>::ConstPtr exactly as in the reference; without
// it (this repository's tests: PCL is not installed) layout-identical mirror structs are used and a "cloud"
// is a std::vector<FeatureT>.  Errors surface as std::runtime_error -- the convention of the reference's
// rassert (include/utils.h:9).  There is no CPU fallback anywhere below.
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <limits>
#include <map>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "b200match.h"

#ifdef B200MATCH_WITH_PCL
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#include <pcl/point_representation.h>
#endif

namespace b200match {

#ifndef B200MATCH_WITH_PCL
// Layout mirrors of the PCL point structs the reference matches on (sizeof must equal PCL's).
struct FPFHSignature33 { float histogram[33]; static constexpr int descriptorSize() { return 33; } };
struct SHOT352 { float descriptor[352]; float rf[9]; static constexpr int descriptorSize() { return 352; } };
struct Histogram135 { float histogram[135]; static constexpr int descriptorSize() { return 135; } };
struct UniqueShapeContext1960 { float descriptor[1960]; float rf[9]; static constexpr int descriptorSize() { return 1960; } };
static_assert(sizeof(FPFHSignature33) == 132, "pcl::FPFHSignature33 is 132 bytes");
static_assert(sizeof(SHOT352) == 1444, "pcl::SHOT352 is 1444 bytes");
static_assert(sizeof(Histogram135) == 540, "pcl::Histogram<135> is 540 bytes");
static_assert(sizeof(UniqueShapeContext1960) == 7876, "pcl::UniqueShapeContext1960 is 7876 bytes");
template <typename FeatureT> using FeatureCloud = std::vector<FeatureT>;
template <typename FeatureT> inline const FeatureT *cloud_data(const FeatureCloud<FeatureT> &c) { return c.data(); }
template <typename FeatureT> inline size_t cloud_size(const FeatureCloud<FeatureT> &c) { return c.size(); }
template <typename FeatureT> inline int feature_dim() { return FeatureT::descriptorSize(); }
#else
template <typename FeatureT> using FeatureCloud = typename pcl::PointCloud<FeatureT>::ConstPtr;
template <typename FeatureT> inline const FeatureT *cloud_data(const FeatureCloud<FeatureT> &c) { return c->points.data(); }
template <typename FeatureT> inline size_t cloud_size(const FeatureCloud<FeatureT> &c) { return c->size(); }
template <typename FeatureT> inline int feature_dim() {
    return pcl::DefaultPointRepresentation<FeatureT>().getNumberOfDimensions();   // as include/matching.h:598-599
}
#endif

// reference include/common.h:192-195 (pcl::Indices == std::vector<int>)
struct MultivaluedCorrespondence {
    std::vector<int> match_indices;
    std::vector<float> distances;
};

// reference include/common.h:120-127; binary-identical to b200m_corr
struct Correspondence {
    int index_query = -1, index_match = -1;
    float distance = std::numeric_limits<float>::max();
    float threshold = 0.f;
};
static_assert(sizeof(Correspondence) == sizeof(b200m_corr), "Correspondence must stay 16 bytes");
typedef std::vector<Correspondence> Correspondences;
typedef std::shared_ptr<Correspondences> CorrespondencesPtr;

// The fields of AlignmentParameters (reference include/common.h:135-163) read on this path.
struct AlignmentParameters {
    bool use_bfmatcher = true;      // :144  either backend maps to the same exact GPU search
    int bf_block_size = 10000;      // :145  accepted, unused
    int ratio_k = 2;                // :146  MATCHING_RATIO_K
    int cluster_k = 40;             // :146  MATCHING_CLUSTER_K (include/common.h:53)
    int randomness = 1;             // :147  k
    float distance_thr = std::numeric_limits<float>::max();   // :139
    std::string matching_id = "lr"; // :149  one_sided | lr | ratio | cluster
    float ratio_thr = 1.1f;         // MATCHING_RATIO_THRESHOLD, include/common.h:50
    float match_search_radius = std::numeric_limits<float>::max();   // :160  matchLocal's 3-D gate
    std::optional<std::array<float, 16>> guess;   // :161  prior pose, row-major (Eigen::Matrix4f): match_multiscale then uses
                                                  // matchLocal (include/matching.h:297-311)
    int device = 0;
    std::vector<int> devices;       // more than one entry: the call is partitioned over these GPUs inside the library
                                    // (b200m_create_multi: source rows sharded, target replicated, NCCL over NVLink)
    int precision = B200M_PREC_TC_F16;
};

class Context {   // RAII b200m_ctx; one per host thread
public:
    explicit Context(int device = 0) {
        if (b200m_create(&ctx_, device) != 0) throw std::runtime_error(b200m_last_error(nullptr));
    }
    ~Context() { b200m_destroy(ctx_); }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    b200m_ctx *get() const { return ctx_; }
    void check(int rc) const {
        if (rc != 0) throw std::runtime_error(b200m_last_error(ctx_));
    }
    template <typename FeatureT>
    void upload(int side, const FeatureCloud<FeatureT> &cloud) {
        // &cloud.points[0] with stride sizeof(FeatureT): what pcl2cv reads (reference include/matching.h:556-558)
        check(b200m_upload(ctx_, side, reinterpret_cast<const float *>(cloud_data<FeatureT>(cloud)), cloud_size<FeatureT>(cloud),
                           sizeof(FeatureT), feature_dim<FeatureT>(), 0));
    }

private:
    b200m_ctx *ctx_ = nullptr;
};

// One context per host thread and device, created on first use and kept: the reference calls matchBF / matchFLANN /
// matchLocal once per scale and direction (include/matching.h:297-311), and a context owns its stream and every device
// buffer (grow-only), so only the first call pays for them.
inline Context &shared_context(int device) {
    thread_local std::map<int, std::unique_ptr<Context>> pool;
    auto &slot = pool[device];
    if (!slot) slot.reset(new Context(device));
    return *slot;
}

class Group {   // RAII b200m_group: one context + one host thread per device, inside the library
public:
    explicit Group(const std::vector<int> &devices) {
        if (b200m_create_multi(&g_, devices.data(), (int) devices.size()) != 0) throw std::runtime_error(b200m_group_last_error(nullptr));
    }
    ~Group() { b200m_destroy_multi(g_); }
    Group(const Group &) = delete;
    Group &operator=(const Group &) = delete;
    b200m_group *get() const { return g_; }
    void check(int rc) const {
        if (rc != 0) throw std::runtime_error(b200m_group_last_error(g_));
    }
    template <typename FeatureT>
    void upload(int side, const FeatureCloud<FeatureT> &cloud) {
        check(b200m_group_upload(g_, side, reinterpret_cast<const float *>(cloud_data<FeatureT>(cloud)), cloud_size<FeatureT>(cloud),
                                 sizeof(FeatureT), feature_dim<FeatureT>()));
    }

private:
    b200m_group *g_ = nullptr;
};

inline Group &shared_group(const std::vector<int> &devices) {
    thread_local std::map<std::vector<int>, std::unique_ptr<Group>> pool;
    auto &slot = pool[devices];
    if (!slot) slot.reset(new Group(devices));
    return *slot;
}

inline b200m_params make_params(const AlignmentParameters &p, int mode, int k) {
    b200m_params q;
    q.k = k;
    q.mode = mode;
    q.ratio_thr = p.ratio_thr;
    q.distance_thr = p.distance_thr;
    q.precision = p.precision;
    q.cand_cap = 0;
    q.n_gpus = 0;
    q.shard = B200M_SHARD_QUERY;
    return q;
}

// ---- batches: many (query / source, train / target) cloud pairs in one call (b200m_knn_batch / b200m_match_batch) ----
// Pair p's result is the one the per-pair call (matchBF, or upload + b200m_match) gives, with pair-local indices.  The batch
// replaces the descriptor sets of the shared context.
template <typename FeatureT>
using CloudPairs = std::vector<std::pair<FeatureCloud<FeatureT>, FeatureCloud<FeatureT>>>;

template <typename FeatureT>
std::vector<b200m_pair> batch_pairs(const CloudPairs<FeatureT> &pairs, size_t *n_src_total) {
    std::vector<b200m_pair> v(pairs.size());
    *n_src_total = 0;
    for (size_t i = 0; i < pairs.size(); ++i) {
        v[i].src = reinterpret_cast<const float *>(cloud_data<FeatureT>(pairs[i].first));
        v[i].n_src = cloud_size<FeatureT>(pairs[i].first);
        v[i].tgt = reinterpret_cast<const float *>(cloud_data<FeatureT>(pairs[i].second));
        v[i].n_tgt = cloud_size<FeatureT>(pairs[i].second);
        *n_src_total += v[i].n_src;
    }
    return v;
}

// matchBF of every pair: result[p] has one entry per query row of pair p
template <typename FeatureT>
std::vector<std::vector<MultivaluedCorrespondence>> knnBatch(const CloudPairs<FeatureT> &pairs, const AlignmentParameters &parameters) {
    size_t nq = 0;
    std::vector<b200m_pair> bp = batch_pairs<FeatureT>(pairs, &nq);
    const int k = parameters.randomness;
    std::vector<int32_t> idx(nq * k);
    std::vector<float> dist(nq * k);
    std::vector<int32_t> cnt(nq);
    b200m_params p = make_params(parameters, B200M_MODE_KNN_ONLY, k);
    Context &ctx = shared_context(parameters.device);
    ctx.check(b200m_knn_batch(ctx.get(), &p, bp.data(), (int) bp.size(), sizeof(FeatureT), feature_dim<FeatureT>(), idx.data(),
                              dist.data(), cnt.data()));
    std::vector<std::vector<MultivaluedCorrespondence>> out(bp.size());
    size_t row = 0;
    for (size_t q = 0; q < bp.size(); ++q) {
        out[q].resize(bp[q].n_src);
        for (size_t i = 0; i < bp[q].n_src; ++i, ++row) {
            out[q][i].match_indices.assign(idx.begin() + row * k, idx.begin() + row * k + cnt[row]);
            out[q][i].distances.assign(dist.begin() + row * k, dist.begin() + row * k + cnt[row]);
        }
    }
    return out;
}

struct BatchMatches {
    std::vector<CorrespondencesPtr> correspondences;   // per pair, ascending index_query, pair-local indices
    std::vector<float> average_distances;              // per pair: FeatureBasedMatcher::getAverageDistance()
};

// The k-list filter of every pair: mode B200M_MODE_ONE_SIDED / MUTUAL / RATIO / RATIO_MUTUAL, k = randomness (ratio modes:
// max(ratio_k, 2)), thresholds = distance_thr -- b200m_match on each pair alone.
template <typename FeatureT>
BatchMatches matchBatch(const CloudPairs<FeatureT> &pairs, const AlignmentParameters &parameters, int mode) {
    size_t nq = 0;
    std::vector<b200m_pair> bp = batch_pairs<FeatureT>(pairs, &nq);
    const bool ratio = mode == B200M_MODE_RATIO || mode == B200M_MODE_RATIO_MUTUAL;
    const int k = ratio ? std::max(parameters.ratio_k, 2) : parameters.randomness;
    b200m_params p = make_params(parameters, mode, k);
    Correspondences all(std::max<size_t>(nq * (mode == B200M_MODE_MUTUAL ? k : 1), 1));
    std::vector<size_t> offsets(bp.size() + 1);
    BatchMatches r;
    r.average_distances.resize(bp.size());
    Context &ctx = shared_context(parameters.device);
    ctx.check(b200m_match_batch(ctx.get(), &p, bp.data(), (int) bp.size(), sizeof(FeatureT), feature_dim<FeatureT>(), nullptr,
                                nullptr, reinterpret_cast<b200m_corr *>(all.data()), all.size(), offsets.data(),
                                r.average_distances.data()));
    for (size_t q = 0; q < bp.size(); ++q)
        r.correspondences.push_back(std::make_shared<Correspondences>(all.begin() + offsets[q], all.begin() + offsets[q + 1]));
    return r;
}

// matchBF<FeatureT> (reference include/matching.h:594-634): one entry per query, <= k matches, ascending L2.
template <typename FeatureT>
std::vector<MultivaluedCorrespondence> matchBF(const FeatureCloud<FeatureT> &query_features,
                                               const FeatureCloud<FeatureT> &train_features,
                                               const AlignmentParameters &parameters) {
    const size_t nq = cloud_size<FeatureT>(query_features);
    const int k = parameters.randomness;
    std::vector<int32_t> idx(nq * k);
    std::vector<float> dist(nq * k);
    std::vector<int32_t> cnt(nq);
    b200m_params p = make_params(parameters, B200M_MODE_KNN_ONLY, k);
    if (parameters.devices.size() > 1) {   // query rows sharded over the GPUs, train set replicated
        Group &g = shared_group(parameters.devices);
        g.upload<FeatureT>(0, query_features);
        g.upload<FeatureT>(1, train_features);
        g.check(b200m_group_knn(g.get(), &p, idx.data(), dist.data(), cnt.data()));
    } else {
        Context &ctx = shared_context(parameters.device);
        ctx.upload<FeatureT>(0, query_features);
        ctx.upload<FeatureT>(1, train_features);
        ctx.check(b200m_knn(ctx.get(), &p, 0, 0, 0, idx.data(), dist.data(), cnt.data()));
    }
    std::vector<MultivaluedCorrespondence> out(nq);
    for (size_t i = 0; i < nq; ++i) {
        out[i].match_indices.assign(idx.begin() + i * k, idx.begin() + i * k + cnt[i]);
        out[i].distances.assign(dist.begin() + i * k, dist.begin() + i * k + cnt[i]);
    }
    return out;
}

// matchFLANN<FeatureT> (reference include/matching.h:562-592): same exact result set.
template <typename FeatureT>
std::vector<MultivaluedCorrespondence> matchFLANN(const FeatureCloud<FeatureT> &query_features,
                                                  const FeatureCloud<FeatureT> &train_features,
                                                  const AlignmentParameters &parameters) {
    return matchBF<FeatureT>(query_features, train_features, parameters);
}

// matchLocal<FeatureT> with match_search_radius = inf (reference include/matching.h:637-678 as called by
// tests/flann_bf_matcher.h:66-72): plain brute force.
template <typename FeatureT>
std::vector<MultivaluedCorrespondence> matchLocal(const FeatureCloud<FeatureT> &query_features,
                                                  const FeatureCloud<FeatureT> &train_features,
                                                  const AlignmentParameters &parameters) {
    return matchBF<FeatureT>(query_features, train_features, parameters);
}

// The keypoints moved by `guess` (row-major 4x4): x' = ((g00 x + g01 y) + g02 z) + g03 in float, every product and sum
// rounded on its own (Eigen's affine product order).  `n` rows `in_stride` floats apart in, `out_stride` floats apart out;
// only the first three floats of an output row are written.
inline void moveKeypoints(const float *kps, size_t n, size_t in_stride, const std::array<float, 16> &guess, float *out,
                          size_t out_stride) {
    for (size_t i = 0; i < n; ++i) {
        const float *q = kps + i * in_stride;
        for (int r = 0; r < 3; ++r)
            out[i * out_stride + r] = guess[4 * r] * q[0] + guess[4 * r + 1] * q[1] + guess[4 * r + 2] * q[2] + guess[4 * r + 3];
    }
}

// The inverse of a guess (the pose of the reverse matchLocal call, inverse_tn): Gauss-Jordan with partial pivoting in
// double, rounded to float.
inline std::array<float, 16> invertGuess(const std::array<float, 16> &g) {
    double a[4][8];
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 8; ++c) a[r][c] = c < 4 ? (double) g[4 * r + c] : (c - 4 == r ? 1.0 : 0.0);
    for (int c = 0; c < 4; ++c) {
        int piv = c;
        for (int r = c + 1; r < 4; ++r)
            if (std::abs(a[r][c]) > std::abs(a[piv][c])) piv = r;
        if (a[piv][c] == 0.0) throw std::runtime_error("the guess is not invertible");
        for (int j = 0; j < 8; ++j) std::swap(a[c][j], a[piv][j]);
        const double d = a[c][c];
        for (int j = 0; j < 8; ++j) a[c][j] /= d;
        for (int r = 0; r < 4; ++r)
            if (r != c) {
                const double f = a[r][c];
                for (int j = 0; j < 8; ++j) a[r][j] -= f * a[c][j];
            }
    }
    std::array<float, 16> inv;
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) inv[4 * r + c] = (float) a[r][4 + c];
    return inv;
}

// matchLocal<FeatureT> as match_multiscale calls it when AlignmentParameters::guess is set (reference
// include/matching.h:378-383, :637-678): the query keypoints are moved by `guess` (row-major 4x4, the reference's
// Eigen::Matrix4f; pcl::transformPointCloudWithNormals, :644), and only train rows whose keypoint lies within
// parameters.match_search_radius of the moved query keypoint compete (radiusSearch on the train keypoint tree, :659).
// query_kps / train_kps: one keypoint per descriptor row, `kps_stride_bytes` apart (pcl::PointNormal rows: 48).
// In a PCL build pass the cloud already transformed by PCL and the identity as `guess` to keep PCL's own arithmetic.
template <typename FeatureT>
std::vector<MultivaluedCorrespondence> matchLocal(const float *query_kps, const float *train_kps, size_t kps_stride_bytes,
                                                  const FeatureCloud<FeatureT> &query_features,
                                                  const FeatureCloud<FeatureT> &train_features,
                                                  const AlignmentParameters &parameters, const std::array<float, 16> &guess) {
    Context &ctx = shared_context(parameters.device);
    ctx.upload<FeatureT>(0, query_features);
    ctx.upload<FeatureT>(1, train_features);
    const size_t nq = cloud_size<FeatureT>(query_features), fl = kps_stride_bytes / 4;
    const int k = parameters.randomness;
    std::vector<float> moved(nq * 3);
    moveKeypoints(query_kps, nq, fl, guess, moved.data(), 3);
    std::vector<float> train_xyz(cloud_size<FeatureT>(train_features) * 3);
    for (size_t j = 0; j < train_xyz.size() / 3; ++j)
        for (int r = 0; r < 3; ++r) train_xyz[3 * j + r] = train_kps[j * fl + r];
    std::vector<int32_t> idx(nq * k), cnt(nq);
    std::vector<float> dist(nq * k);
    b200m_params p = make_params(parameters, B200M_MODE_KNN_ONLY, k);
    ctx.check(b200m_knn_local(ctx.get(), &p, 0, moved.data(), train_xyz.data(), 12, parameters.match_search_radius, idx.data(),
                              dist.data(), cnt.data()));
    std::vector<MultivaluedCorrespondence> out(nq);
    for (size_t i = 0; i < nq; ++i) {
        out[i].match_indices.assign(idx.begin() + i * k, idx.begin() + i * k + cnt[i]);
        out[i].distances.assign(dist.begin() + i * k, dist.begin() + i * k + cnt[i]);
    }
    return out;
}

// match_multiscale (reference include/matching.h:264-354) over precomputed per-scale descriptors: one exact kNN per
// scale (k = parameters.randomness) over that scale's keypoint subset, per-scale row numbers renamed to keypoint ids
// through the scale's kps_indices_multiscale (:313-321), candidates concatenated per query keypoint in scale order, and
// the spatial vote over the train keypoints' xyz (:327-352) keeps at most ONE match per query keypoint.
//   query_features[s] / train_features[s]   kps_features_multiscale[s] of the two Storage objects (common scales only)
//   query_indices[s] / train_indices[s]     kps_indices_multiscale[s] (row of scale s -> keypoint id)
//   train_kps_xyz                           st_train.kps: n_train_kps rows, `xyz_stride_bytes` apart (pcl::PointXYZ: 16)
// Returns st_query.kps->size() entries, each empty or {one match index, its descriptor distance}.
template <typename FeatureT>
std::vector<MultivaluedCorrespondence> match_multiscale(const std::vector<FeatureCloud<FeatureT>> &query_features,
                                                        const std::vector<FeatureCloud<FeatureT>> &train_features,
                                                        const std::vector<std::vector<int>> &query_indices,
                                                        const std::vector<std::vector<int>> &train_indices,
                                                        size_t n_query_kps, const float *train_kps_xyz, size_t n_train_kps,
                                                        size_t xyz_stride_bytes, float iss_radius,
                                                        const AlignmentParameters &parameters) {
    const size_t n_scales = query_features.size();
    if (n_scales == 0 || train_features.size() != n_scales || query_indices.size() != n_scales || train_indices.size() != n_scales)
        throw std::runtime_error("match_multiscale: one descriptor cloud and one index map per scale and side are needed");
    Context &ctx = shared_context(parameters.device);
    const int k = parameters.randomness;
    ctx.check(b200m_multiscale_begin(ctx.get(), n_query_kps, (int) n_scales, k));
    b200m_params p = make_params(parameters, B200M_MODE_KNN_ONLY, k);
    static_assert(sizeof(int) == sizeof(int32_t), "index maps are passed as int32");
    for (size_t s = 0; s < n_scales; ++s) {
        if (query_indices[s].size() != cloud_size<FeatureT>(query_features[s]) ||
            train_indices[s].size() != cloud_size<FeatureT>(train_features[s]))
            throw std::runtime_error("match_multiscale: index map length != number of descriptors of the scale");
        ctx.upload<FeatureT>(0, query_features[s]);
        ctx.upload<FeatureT>(1, train_features[s]);
        ctx.check(b200m_multiscale_add(ctx.get(), &p, 0, (int) s, reinterpret_cast<const int32_t *>(query_indices[s].data()),
                                       reinterpret_cast<const int32_t *>(train_indices[s].data()), n_train_kps));
    }
    std::vector<int32_t> idx(n_query_kps), cnt(n_query_kps);
    std::vector<float> dist(n_query_kps);
    ctx.check(b200m_multiscale_vote(ctx.get(), train_kps_xyz, n_train_kps, xyz_stride_bytes, iss_radius, idx.data(), dist.data(),
                                    cnt.data()));
    std::vector<MultivaluedCorrespondence> out(n_query_kps);
    for (size_t i = 0; i < n_query_kps; ++i)
        if (cnt[i] > 0) {
            out[i].match_indices.push_back(idx[i]);
            out[i].distances.push_back(dist[i]);
        }
    return out;
}

// FeatureBasedMatcher (reference include/matching.h:25-42) at the descriptor seam.
class FeatureBasedMatcher {
public:
    using Ptr = std::shared_ptr<FeatureBasedMatcher>;
    virtual ~FeatureBasedMatcher() = default;
    virtual CorrespondencesPtr match() = 0;
    inline float getAverageDistance() const { return average_distance_; }
    virtual std::string getClassName() = 0;

protected:
    float average_distance_ = std::numeric_limits<float>::max();
};

template <typename FeatureT>
class FeatureBasedMatcherImpl : public FeatureBasedMatcher {
public:
    // The fields of FeatureBasedMatcherImpl<FeatureT>::Storage (reference include/matching.h:114-127) that match_impl
    // reads; `initialize` (downsampling, normals, feature estimation: :163-262) stays with the caller and fills them.
    struct Storage {
        const float *kps_xyz = nullptr;            // kps: keypoint coordinates, one row per keypoint
        size_t n_kps = 0;                          // kps->size()
        size_t kps_stride_bytes = 16;              // sizeof(PointN) (pcl::PointNormal: 48; pcl::PointXYZ: 16)
        std::vector<int> kps_indices;              // keypoint id -> index in pcd (finalize, :356-362); empty = identity
        std::vector<std::vector<int>> kps_indices_multiscale;          // [scale][row] -> keypoint id; empty = identity (one scale)
        std::vector<FeatureCloud<FeatureT>> kps_features_multiscale;   // [scale] descriptors of that scale's keypoints
        int min_log2_radius = 0, max_log2_radius = 0;                  // scales present: max - min + 1 entries above
        float iss_radius = 1.f;
        std::vector<float> thresholds;             // calculateSmoothedDensities(kps) (src/common.cpp:531-547); may be empty
    };

    // single-scale convenience: one descriptor per keypoint, identity maps
    static Storage makeStorage(FeatureCloud<FeatureT> features, const float *kps_xyz = nullptr, size_t kps_stride_bytes = 16,
                               float iss_radius = 1.f, std::vector<float> thresholds = {}, std::vector<int> kps_indices = {}) {
        Storage st;
        st.n_kps = cloud_size<FeatureT>(features);
        st.kps_features_multiscale.push_back(std::move(features));
        st.kps_xyz = kps_xyz;
        st.kps_stride_bytes = kps_stride_bytes;
        st.iss_radius = iss_radius;
        st.thresholds = std::move(thresholds);
        st.kps_indices = std::move(kps_indices);
        return st;
    }

    FeatureBasedMatcherImpl(Storage src, Storage tgt, AlignmentParameters parameters)
        : st_src_(std::move(src)), st_tgt_(std::move(tgt)), parameters_(std::move(parameters)) {}

    // match() (reference include/matching.h:148-161): match_impl + finalize
    CorrespondencesPtr match() override { return finalize(match_impl()); }

    template <typename F>
    friend std::vector<CorrespondencesPtr> matchMany(const std::vector<std::shared_ptr<FeatureBasedMatcherImpl<F>>> &matchers);

protected:
    virtual int mode() const = 0;

    // finalize (reference :356-362): keypoint ids -> indices in the clouds
    CorrespondencesPtr finalize(CorrespondencesPtr correspondences) const {
        for (auto &c : *correspondences) {
            if (!st_src_.kps_indices.empty()) c.index_query = st_src_.kps_indices[c.index_query];
            if (!st_tgt_.kps_indices.empty()) c.index_match = st_tgt_.kps_indices[c.index_match];
        }
        return correspondences;
    }

    // the scales common to both clouds (reference :268-270) as the library's per-scale rows; *lo = the first one's log2 radius
    std::vector<b200m_scale> commonScales(int *lo_out = nullptr) const {
        const int lo = std::max(st_src_.min_log2_radius, st_tgt_.min_log2_radius);
        const int hi = std::min(st_src_.max_log2_radius, st_tgt_.max_log2_radius);
        if (hi < lo) throw std::runtime_error("the two clouds have no scale in common");
        std::vector<b200m_scale> scales;
        static_assert(sizeof(int) == sizeof(int32_t), "index maps are passed as int32");
        for (int r = lo; r <= hi; ++r) {
            const size_t is = (size_t) (r - st_src_.min_log2_radius), it = (size_t) (r - st_tgt_.min_log2_radius);
            if (is >= st_src_.kps_features_multiscale.size() || it >= st_tgt_.kps_features_multiscale.size())
                throw std::runtime_error("kps_features_multiscale has fewer entries than scales");
            b200m_scale sc{};
            sc.src_desc = reinterpret_cast<const float *>(cloud_data<FeatureT>(st_src_.kps_features_multiscale[is]));
            sc.n_src = cloud_size<FeatureT>(st_src_.kps_features_multiscale[is]);
            sc.tgt_desc = reinterpret_cast<const float *>(cloud_data<FeatureT>(st_tgt_.kps_features_multiscale[it]));
            sc.n_tgt = cloud_size<FeatureT>(st_tgt_.kps_features_multiscale[it]);
            if (is < st_src_.kps_indices_multiscale.size()) {
                if (st_src_.kps_indices_multiscale[is].size() != sc.n_src) throw std::runtime_error("kps_indices_multiscale: length != descriptors of the scale");
                sc.src_map = reinterpret_cast<const int32_t *>(st_src_.kps_indices_multiscale[is].data());
            }
            if (it < st_tgt_.kps_indices_multiscale.size()) {
                if (st_tgt_.kps_indices_multiscale[it].size() != sc.n_tgt) throw std::runtime_error("kps_indices_multiscale: length != descriptors of the scale");
                sc.tgt_map = reinterpret_cast<const int32_t *>(st_tgt_.kps_indices_multiscale[it].data());
            }
            scales.push_back(sc);
        }
        if (lo_out) *lo_out = lo;
        return scales;
    }

    // the keypoint coordinates of both clouds; one candidate per keypoint (randomness 1, one scale): the vote is the identity
    // and needs none, `zeros` stands in for them
    void keypointRows(size_t n_scales, std::vector<float> &zeros, const float **sx, const float **tx, size_t *stride) const {
        *sx = st_src_.kps_xyz;
        *tx = st_tgt_.kps_xyz;
        *stride = st_src_.kps_stride_bytes;
        if (!*sx || !*tx) {
            if (parameters_.randomness != 1 || n_scales != 1 || mode() == B200M_MODE_CLUSTER)
                throw std::runtime_error("randomness * scales > 1 (or the cluster filter) needs the keypoint coordinates of both clouds: "
                                         "match_multiscale's spatial vote keeps one match per keypoint (include/matching.h:327-352)");
            zeros.assign(4 * std::max(st_src_.n_kps, st_tgt_.n_kps) + 4, 0.f);
            *sx = *tx = zeros.data();
            *stride = 16;
        } else if (st_src_.kps_stride_bytes != st_tgt_.kps_stride_bytes) {
            throw std::runtime_error("both keypoint clouds must have the same point stride");
        }
    }

    // with a guess: the keypoints of both clouds moved for the two matchLocal directions -- the source by the guess, the
    // target by its inverse -- in the keypoint rows' own stride
    void movedRows(std::vector<float> &ms, std::vector<float> &mt) const {
        if (!st_src_.kps_xyz || !st_tgt_.kps_xyz)
            throw std::runtime_error("a guess needs the keypoint coordinates of both clouds: matchLocal gates on them "
                                     "(include/matching.h:637-678)");
        const size_t fl = st_src_.kps_stride_bytes / 4;
        ms.assign(st_src_.n_kps * fl + 4, 0.f);
        mt.assign(st_tgt_.n_kps * fl + 4, 0.f);
        moveKeypoints(st_src_.kps_xyz, st_src_.n_kps, fl, *parameters_.guess, ms.data(), fl);
        moveKeypoints(st_tgt_.kps_xyz, st_tgt_.n_kps, fl, invertGuess(*parameters_.guess), mt.data(), fl);
    }

    // match_impl of the three implemented matchers: both match_multiscale calls, the vote, printDebugInfo's average
    // and the filter loop in one device-resident call
    virtual CorrespondencesPtr match_impl() {
        int lo = 0;
        std::vector<b200m_scale> scales = commonScales(&lo);
        std::vector<float> zeros;
        const float *sx, *tx;
        size_t stride;
        if (parameters_.guess && parameters_.devices.size() > 1)
            throw std::runtime_error("a guess runs on one GPU only (parameters.devices has several)");
        keypointRows(scales.size(), zeros, &sx, &tx, &stride);
        std::vector<float> ms, mt;
        if (parameters_.guess) movedRows(ms, mt);
        const bool thr = !st_src_.thresholds.empty() && !st_tgt_.thresholds.empty();
        b200m_params p = make_params(parameters_, mode(), parameters_.randomness);
        auto out = std::make_shared<Correspondences>(st_src_.n_kps);
        size_t n = 0;
        if (parameters_.guess) {   // matchLocal per scale and direction: a batch of one pair
            const b200m_wide_pair wp{scales.data(), (int) scales.size(), sx, st_src_.n_kps, tx, st_tgt_.n_kps, st_src_.iss_radius,
                                     st_tgt_.iss_radius};
            const b200m_local_pair lp{ms.data(), mt.data()};
            size_t offsets[2] = {0, 0};
            Context &ctx = shared_context(parameters_.device);
            ctx.check(b200m_match_multiscale_local_batch(
                ctx.get(), &p, &wp, &lp, 1, sizeof(FeatureT), feature_dim<FeatureT>(), stride, parameters_.cluster_k,
                parameters_.match_search_radius, thr ? st_src_.thresholds.data() : nullptr, thr ? st_tgt_.thresholds.data() : nullptr,
                reinterpret_cast<b200m_corr *>(out->data()), std::max<size_t>(out->size(), 1), offsets, &average_distance_));
            out->resize(offsets[1]);
            return out;
        }
        if (parameters_.devices.size() > 1) {
            // several GPUs: the library partitions the k-list matcher call (b200m_group_match).  That IS match_impl when every
            // keypoint has one candidate (randomness 1, one scale, identity maps: the vote keeps it); the voted multi-scale
            // form runs on one GPU.
            if (parameters_.randomness != 1 || scales.size() != 1 || scales[0].src_map || scales[0].tgt_map || mode() == B200M_MODE_CLUSTER)
                throw std::runtime_error("multi-GPU matcher classes: randomness 1, one scale, one-sided / lr only");
            Group &g = shared_group(parameters_.devices);
            g.upload<FeatureT>(0, st_src_.kps_features_multiscale[(size_t) (lo - st_src_.min_log2_radius)]);
            g.upload<FeatureT>(1, st_tgt_.kps_features_multiscale[(size_t) (lo - st_tgt_.min_log2_radius)]);
            g.check(b200m_group_match(g.get(), &p, thr ? st_src_.thresholds.data() : nullptr, thr ? st_tgt_.thresholds.data() : nullptr,
                                      reinterpret_cast<b200m_corr *>(out->data()), out->size(), &n, &average_distance_));
            out->resize(n);
            return out;
        }
        Context &ctx = shared_context(parameters_.device);
        ctx.check(b200m_match_multiscale(ctx.get(), &p, scales.data(), (int) scales.size(), sizeof(FeatureT), feature_dim<FeatureT>(),
                                         sx, st_src_.n_kps, tx, st_tgt_.n_kps, stride, st_src_.iss_radius, st_tgt_.iss_radius,
                                         parameters_.cluster_k, thr ? st_src_.thresholds.data() : nullptr,
                                         thr ? st_tgt_.thresholds.data() : nullptr, reinterpret_cast<b200m_corr *>(out->data()),
                                         out->size(), &n, &average_distance_));
        out->resize(n);
        return out;
    }

    Storage st_src_, st_tgt_;
    AlignmentParameters parameters_;
};

template <typename FeatureT>
class OneSidedMatcher : public FeatureBasedMatcherImpl<FeatureT> {   // reference include/matching.h:385-416
public:
    using FeatureBasedMatcherImpl<FeatureT>::FeatureBasedMatcherImpl;
    std::string getClassName() override { return "OneSidedMatcher"; }
protected:
    int mode() const override { return B200M_MODE_ONE_SIDED; }
};

template <typename FeatureT>
class LeftToRightMatcher : public FeatureBasedMatcherImpl<FeatureT> {   // reference include/matching.h:418-458
public:
    using FeatureBasedMatcherImpl<FeatureT>::FeatureBasedMatcherImpl;
    std::string getClassName() override { return "LeftToRightMatcher"; }
protected:
    int mode() const override { return B200M_MODE_MUTUAL; }
};

// ClusterMatcher (reference include/matching.h:480-551, the default matching_id): both Storages need kps_xyz.
template <typename FeatureT>
class ClusterMatcher : public FeatureBasedMatcherImpl<FeatureT> {
public:
    using FeatureBasedMatcherImpl<FeatureT>::FeatureBasedMatcherImpl;
    std::string getClassName() override { return "ClusterMatcher"; }
protected:
    int mode() const override { return B200M_MODE_CLUSTER; }
};

// RatioMatcher: a stub in the reference (include/matching.h:460-478, match_impl returns {}); defined here on the raw
// k-lists of a single scale (DESIGN.md section 6; parity unpinned: there is no reference behaviour).
template <typename FeatureT>
class RatioMatcher : public FeatureBasedMatcherImpl<FeatureT> {
public:
    using FeatureBasedMatcherImpl<FeatureT>::FeatureBasedMatcherImpl;
    std::string getClassName() override { return "RatioMatcher"; }
protected:
    int mode() const override { return B200M_MODE_RATIO; }
    CorrespondencesPtr match_impl() override {
        if (this->parameters_.guess) throw std::runtime_error("RatioMatcher: a guess is not supported (the reference's is a stub)");
        if (this->st_src_.kps_features_multiscale.size() != 1 || this->st_tgt_.kps_features_multiscale.size() != 1)
            throw std::runtime_error("RatioMatcher is defined on a single scale");
        Context &ctx = shared_context(this->parameters_.device);
        ctx.template upload<FeatureT>(0, this->st_src_.kps_features_multiscale[0]);
        ctx.template upload<FeatureT>(1, this->st_tgt_.kps_features_multiscale[0]);
        const int k = this->parameters_.ratio_k < 2 ? 2 : this->parameters_.ratio_k;
        b200m_params p = make_params(this->parameters_, B200M_MODE_RATIO, k);
        auto out = std::make_shared<Correspondences>(this->st_src_.n_kps);
        size_t n = 0;
        const bool thr = !this->st_src_.thresholds.empty() && !this->st_tgt_.thresholds.empty();
        ctx.check(b200m_match(ctx.get(), &p, thr ? this->st_src_.thresholds.data() : nullptr,
                              thr ? this->st_tgt_.thresholds.data() : nullptr, reinterpret_cast<b200m_corr *>(out->data()),
                              out->size(), &n, &this->average_distance_));
        out->resize(n);
        return out;
    }
};

// match() of many OneSided / LeftToRight / ClusterMatchers in one library call (b200m_match_multiscale_batch): multi-view
// registration, one scan against many submaps, an evaluation table.  All matchers must be of one class with the same
// parameters (the guess aside: each matcher may have its own) and keypoint point stride; each pair's common scales are
// built as match_impl builds them.  Either every matcher has a guess (b200m_match_multiscale_local_batch) or none has.
// result[i] equals matchers[i]->match(), finalize included, and matchers[i]->getAverageDistance() is set.  With several
// parameters.devices the pairs are spread over those GPUs (b200m_group_match_multiscale[_local]_batch; same results).
inline bool sameParameters(const AlignmentParameters &a, const AlignmentParameters &b) {
    return a.use_bfmatcher == b.use_bfmatcher && a.bf_block_size == b.bf_block_size && a.ratio_k == b.ratio_k &&
           a.cluster_k == b.cluster_k && a.randomness == b.randomness && a.distance_thr == b.distance_thr &&
           a.matching_id == b.matching_id && a.ratio_thr == b.ratio_thr && a.match_search_radius == b.match_search_radius &&
           a.device == b.device && a.devices == b.devices && a.precision == b.precision;
}

template <typename FeatureT>
std::vector<CorrespondencesPtr> matchMany(const std::vector<std::shared_ptr<FeatureBasedMatcherImpl<FeatureT>>> &matchers) {
    std::vector<CorrespondencesPtr> result;
    if (matchers.empty()) return result;
    const FeatureBasedMatcherImpl<FeatureT> &m0 = *matchers[0];
    const AlignmentParameters &pa = m0.parameters_;
    const int mode = m0.mode();
    if (mode != B200M_MODE_ONE_SIDED && mode != B200M_MODE_MUTUAL && mode != B200M_MODE_CLUSTER)
        throw std::runtime_error("matchMany: OneSided, LeftToRight and ClusterMatchers only (RatioMatcher: matchBatch)");
    const size_t n = matchers.size();
    std::vector<std::vector<b200m_scale>> scales(n);
    std::vector<std::vector<float>> zeros(n);
    std::vector<b200m_wide_pair> pairs(n);
    std::vector<b200m_local_pair> locals(n);
    std::vector<std::vector<float>> moved(2 * n);
    const bool guessed = pa.guess.has_value();
    std::vector<float> thr_src, thr_tgt;
    bool thr = false;
    size_t stride = 0, n_src = 0;
    for (size_t i = 0; i < n; ++i) {
        const FeatureBasedMatcherImpl<FeatureT> &m = *matchers[i];
        if (m.mode() != mode || matchers[i]->getClassName() != matchers[0]->getClassName() || !sameParameters(m.parameters_, pa))
            throw std::runtime_error("matchMany: every matcher must be of one class with the same AlignmentParameters");
        if (m.parameters_.guess.has_value() != guessed)
            throw std::runtime_error("matchMany: give every matcher a guess or none (the guessed and unguessed kNN are different calls)");
        scales[i] = m.commonScales();
        const float *sx, *tx;
        size_t st;
        m.keypointRows(scales[i].size(), zeros[i], &sx, &tx, &st);
        if (guessed) {
            m.movedRows(moved[2 * i], moved[2 * i + 1]);
            locals[i] = b200m_local_pair{moved[2 * i].data(), moved[2 * i + 1].data()};
        }
        if (i && st != stride) throw std::runtime_error("matchMany: every keypoint cloud must have the same point stride");
        stride = st;
        pairs[i] = b200m_wide_pair{scales[i].data(), (int) scales[i].size(), sx, m.st_src_.n_kps, tx, m.st_tgt_.n_kps,
                                   m.st_src_.iss_radius, m.st_tgt_.iss_radius};
        thr = thr || (!m.st_src_.thresholds.empty() && !m.st_tgt_.thresholds.empty());
        n_src += m.st_src_.n_kps;
    }
    if (thr) {   // a matcher without thresholds gets +inf ones: min(max(inf, .), distance_thr) = distance_thr, as with none
        for (size_t i = 0; i < n; ++i) {
            const FeatureBasedMatcherImpl<FeatureT> &m = *matchers[i];
            const bool own = !m.st_src_.thresholds.empty() && !m.st_tgt_.thresholds.empty();
            const float inf = std::numeric_limits<float>::infinity();
            if (own) {
                thr_src.insert(thr_src.end(), m.st_src_.thresholds.begin(), m.st_src_.thresholds.begin() + m.st_src_.n_kps);
                thr_tgt.insert(thr_tgt.end(), m.st_tgt_.thresholds.begin(), m.st_tgt_.thresholds.begin() + m.st_tgt_.n_kps);
            } else {
                thr_src.insert(thr_src.end(), m.st_src_.n_kps, inf);
                thr_tgt.insert(thr_tgt.end(), m.st_tgt_.n_kps, inf);
            }
        }
        thr_src.push_back(0.f);
        thr_tgt.push_back(0.f);
    }
    b200m_params p = make_params(pa, mode, pa.randomness);
    Correspondences all(std::max<size_t>(n_src, 1));
    std::vector<size_t> offsets(n + 1);
    std::vector<float> avg(n);
    const float *ts = thr ? thr_src.data() : nullptr, *tt = thr ? thr_tgt.data() : nullptr;
    b200m_corr *rec = reinterpret_cast<b200m_corr *>(all.data());
    if (pa.devices.size() > 1) {
        Group &g = shared_group(pa.devices);
        if (guessed)
            g.check(b200m_group_match_multiscale_local_batch(g.get(), &p, pairs.data(), locals.data(), (int) n, sizeof(FeatureT),
                                                             feature_dim<FeatureT>(), stride, pa.cluster_k, pa.match_search_radius, ts, tt,
                                                             rec, all.size(), offsets.data(), avg.data()));
        else
            g.check(b200m_group_match_multiscale_batch(g.get(), &p, pairs.data(), (int) n, sizeof(FeatureT), feature_dim<FeatureT>(),
                                                       stride, pa.cluster_k, ts, tt, rec, all.size(), offsets.data(), avg.data()));
    } else {
        Context &ctx = shared_context(pa.device);
        if (guessed)
            ctx.check(b200m_match_multiscale_local_batch(ctx.get(), &p, pairs.data(), locals.data(), (int) n, sizeof(FeatureT),
                                                         feature_dim<FeatureT>(), stride, pa.cluster_k, pa.match_search_radius, ts, tt,
                                                         rec, all.size(), offsets.data(), avg.data()));
        else
            ctx.check(b200m_match_multiscale_batch(ctx.get(), &p, pairs.data(), (int) n, sizeof(FeatureT), feature_dim<FeatureT>(), stride,
                                                   pa.cluster_k, ts, tt, rec, all.size(), offsets.data(), avg.data()));
    }
    for (size_t i = 0; i < n; ++i) {
        matchers[i]->average_distance_ = avg[i];
        result.push_back(matchers[i]->finalize(std::make_shared<Correspondences>(all.begin() + offsets[i], all.begin() + offsets[i + 1])));
    }
    return result;
}

// getFeatureBasedMatcherFromParameters (reference src/matching.cpp:21-76) for one feature type.
template <typename FeatureT>
FeatureBasedMatcher::Ptr getFeatureBasedMatcherFromParameters(typename FeatureBasedMatcherImpl<FeatureT>::Storage src,
                                                              typename FeatureBasedMatcherImpl<FeatureT>::Storage tgt,
                                                              const AlignmentParameters &parameters) {
    if (parameters.matching_id == "one_sided")
        return std::make_shared<OneSidedMatcher<FeatureT>>(std::move(src), std::move(tgt), parameters);
    if (parameters.matching_id == "lr")
        return std::make_shared<LeftToRightMatcher<FeatureT>>(std::move(src), std::move(tgt), parameters);
    if (parameters.matching_id == "ratio")
        return std::make_shared<RatioMatcher<FeatureT>>(std::move(src), std::move(tgt), parameters);
    if (parameters.matching_id == "cluster")
        return std::make_shared<ClusterMatcher<FeatureT>>(std::move(src), std::move(tgt), parameters);
    throw std::runtime_error("Matching method " + parameters.matching_id + " isn't supported by the B200 matcher");
}

}  // namespace b200match
