// multiscale.cu -- the tail of FeatureBasedMatcherImpl<FeatureT>::match_multiscale
// (reference include/matching.h:264-354): per-scale k-lists are remapped from per-scale row
// numbers to keypoint ids (:313-321), concatenated per query keypoint in scale order, and a
// spatial vote (:327-352) reduces every keypoint's candidates to at most one match.
//
//   ms_scatter_kernel   one thread per (per-scale query row, neighbour): k-list entries go to the
//                       keypoint's slot [kp][scale][k] with the train row remapped to its keypoint id.
//                       A keypoint occurs at most once per scale, so there are no write conflicts and
//                       walking the slots in scale order reproduces the reference's push_back order.
//   ms_vote_kernel      one thread per query keypoint: candidate m1 scores
//                       sum_{m2 >= m1, |p_m1 - p_m2| < 32 r} r / max(|p_m1 - p_m2|, r)   (r = iss_radius, p = train
//                       keypoint xyz), the best score wins, ties -> the smaller descriptor distance.  FP32 with
//                       separate roundings (the reference builds without FMA), sums in the reference's order.
#include <math.h>

#include "internal.cuh"

namespace {

__global__ void ms_scatter_kernel(size_t n_rows, int k, int scale, int n_scales, size_t n_query_kps, size_t n_train_kps,
                                  const int32_t *__restrict__ idx, const float *__restrict__ dist,
                                  const int32_t *__restrict__ count, const int32_t *__restrict__ query_map,
                                  const int32_t *__restrict__ train_map, size_t n_train_rows, long long train_offset,
                                  int32_t *__restrict__ s_idx, float *__restrict__ s_dist, int32_t *__restrict__ s_cnt,
                                  int *__restrict__ bad) {
    const size_t row = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const long long kp = query_map ? (long long) query_map[row] : (long long) row;
    if (kp < 0 || (size_t) kp >= n_query_kps) { atomicExch(bad, 1); return; }
    const int c = count[row];
    const size_t slot = ((size_t) kp * n_scales + scale) * k;
    for (int m = 0; m < c && m < k; ++m) {
        const long long j = (long long) idx[row * k + m] - train_offset;   // row of the train side of this scale
        long long tj = -1;
        if (j >= 0 && (size_t) j < n_train_rows) tj = train_map ? (long long) train_map[j] : j;
        if (tj < 0 || (size_t) tj >= n_train_kps) { atomicExch(bad, 2); tj = -1; }
        s_idx[slot + m] = (int32_t) tj;
        s_dist[slot + m] = dist[row * k + m];
    }
    s_cnt[(size_t) kp * n_scales + scale] = c < k ? c : k;
}

constexpr int kMaxVoteCands = 128;

// SEG (batch calls, wide_batch.cu): the query keypoints of many pairs back to back, iss_radius = radii[pair of kp].  A
// compile-time flag, so the single-pair instantiation is the kernel it was.
template <bool SEG>
__global__ void ms_vote_kernel(size_t n_query_kps, int n_scales, int k, const int32_t *__restrict__ s_idx,
                               const float *__restrict__ s_dist, const int32_t *__restrict__ s_cnt,
                               const float *__restrict__ xyz, size_t xyz_stride_floats, float iss_radius,
                               int32_t *__restrict__ out_idx, float *__restrict__ out_dist, int32_t *__restrict__ out_cnt,
                               const int32_t *__restrict__ kp_off = nullptr, int n_pairs = 0,
                               const float *__restrict__ radii = nullptr) {
    const size_t kp = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (kp >= n_query_kps) return;
    if constexpr (SEG) iss_radius = radii[pair_of(kp_off, n_pairs, (long long) kp)];
    // candidate m of the concatenated list = m-th entry when the scales' lists are walked in order
    const int32_t *ci = s_idx + kp * (size_t) n_scales * k;
    const float *cd = s_dist + kp * (size_t) n_scales * k;
    const int32_t *cc = s_cnt + kp * (size_t) n_scales;
    int n = 0;
    for (int s = 0; s < n_scales; ++s) n += cc[s];
    const float limit = __fmul_rn(32.f, iss_radius);
    float best_count = 0.f, best_dist = 0.f;
    int best_pos = -1;
    // outer walk over m1
    int s1 = 0, e1 = 0;
    for (int m1 = 0; m1 < n; ++m1) {
        while (e1 >= cc[s1]) { ++s1; e1 = 0; }
        const int p1 = s1 * k + e1;
        const int32_t j1 = ci[p1];
        float c = 0.f;
        if (j1 >= 0) {
            const float *a = xyz + (size_t) j1 * xyz_stride_floats;
            const float ax = a[0], ay = a[1], az = a[2];
            int s2 = s1, e2 = e1;
            for (int m2 = m1; m2 < n; ++m2) {
                while (e2 >= cc[s2]) { ++s2; e2 = 0; }
                const int32_t j2 = ci[s2 * k + e2];
                ++e2;
                if (j2 < 0) continue;
                const float *b = xyz + (size_t) j2 * xyz_stride_floats;
                const float dx = __fsub_rn(ax, b[0]), dy = __fsub_rn(ay, b[1]), dz = __fsub_rn(az, b[2]);
                // Eigen's Vector3f::norm(): the unrolled fixed-size reduction adds x^2 + (y^2 + z^2)
                const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dz, dz))));
                if (d < limit) c = __fadd_rn(c, __fdiv_rn(iss_radius, fmaxf(d, iss_radius)));
            }
        }
        const float dd = cd[p1];
        if (c > best_count || (c == best_count && dd < best_dist)) {
            best_count = c;
            best_dist = dd;
            best_pos = p1;
        }
        ++e1;
    }
    if (best_pos >= 0) {
        out_idx[kp] = ci[best_pos];
        out_dist[kp] = cd[best_pos];
        out_cnt[kp] = 1;
    } else {
        out_idx[kp] = -1;
        out_dist[kp] = 0.f;
        out_cnt[kp] = 0;
    }
}

}  // namespace

static MultiscaleState *ms_state(b200m_ctx *ctx) {
    if (!ctx->multiscale) ctx->multiscale = new MultiscaleState();
    return static_cast<MultiscaleState *>(ctx->multiscale);
}

void ms_free(MultiscaleState *ms) {
    if (!ms) return;
    DevBuf *b[] = {&ms->idx, &ms->dist, &ms->cnt, &ms->bad, &ms->qmap, &ms->tmap, &ms->xyz, &ms->oidx, &ms->odist, &ms->ocnt,
                   &ms->kidx, &ms->kdist, &ms->kcnt};
    for (DevBuf *x : b) x->release();
    delete ms;
}

void multiscale_release(b200m_ctx *ctx) {
    ms_free(static_cast<MultiscaleState *>(ctx->multiscale));
    ctx->multiscale = nullptr;
}

int ms_begin(b200m_ctx *ctx, MultiscaleState *ms, size_t n_query_kps, int n_scales, int k) {
    if (n_scales < 1 || n_scales > 32) return b200m_fail_msg(ctx, "b200m_multiscale_begin: n_scales must be in [1, 32]");
    if (k < 1 || k > B200M_MAX_K || n_scales * k > kMaxVoteCands)
        return b200m_fail_msg(ctx, "b200m_multiscale_begin: k in [1, 32] and n_scales * k <= 128");
    ms->n_query_kps = n_query_kps;
    ms->n_scales = n_scales;
    ms->k = k;
    const size_t slots = n_query_kps * (size_t) n_scales;
    CK(ms->idx.reserve(sizeof(int32_t) * slots * k));
    CK(ms->dist.reserve(sizeof(float) * slots * k));
    CK(ms->cnt.reserve(sizeof(int32_t) * slots));
    CK(ms->bad.reserve(sizeof(int)));
    if (slots) CK(cudaMemsetAsync(ms->cnt.p, 0, sizeof(int32_t) * slots, ctx->stream));   // a keypoint absent from a scale adds nothing
    CK(cudaMemsetAsync(ms->bad.p, 0, sizeof(int), ctx->stream));
    return 0;
}

int ms_add_device(b200m_ctx *ctx, MultiscaleState *ms, int scale, size_t n_rows, const int32_t *d_idx, const float *d_dist,
                  const int32_t *d_count, const int32_t *d_query_map, const int32_t *d_train_map, size_t n_train_rows,
                  int64_t train_index_offset, size_t n_train_kps) {
    if (!ms || ms->n_scales == 0) return b200m_fail_msg(ctx, "b200m_multiscale_add: call b200m_multiscale_begin first");
    if (scale < 0 || scale >= ms->n_scales) return b200m_fail_msg(ctx, "b200m_multiscale_add: scale out of range");
    if (n_rows == 0) return 0;
    if (!d_idx || !d_dist || !d_count) return b200m_fail_msg(ctx, "b200m_multiscale_add: null k-list pointer");
    ms_scatter_kernel<<<(unsigned) ((n_rows + 255) / 256), 256, 0, ctx->stream>>>(
        n_rows, ms->k, scale, ms->n_scales, ms->n_query_kps, n_train_kps, d_idx, d_dist, d_count, d_query_map, d_train_map,
        n_train_rows, (long long) train_index_offset, ms->idx.as<int32_t>(), ms->dist.as<float>(), ms->cnt.as<int32_t>(),
        ms->bad.as<int>());
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

int ms_vote_device(b200m_ctx *ctx, MultiscaleState *ms, const float *d_train_xyz, size_t xyz_stride_bytes, float iss_radius,
                   int32_t *d_idx, float *d_dist, int32_t *d_count) {
    if (!ms || ms->n_scales == 0) return b200m_fail_msg(ctx, "b200m_multiscale_vote: call b200m_multiscale_begin first");
    if (xyz_stride_bytes % 4 != 0 || xyz_stride_bytes < 12)
        return b200m_fail_msg(ctx, "b200m_multiscale_vote: xyz stride must be a multiple of 4 and >= 12 bytes");
    if (ms->n_query_kps == 0) return 0;
    if (!d_train_xyz || !d_idx || !d_dist || !d_count) return b200m_fail_msg(ctx, "b200m_multiscale_vote: null pointer");
    ms_vote_kernel<false><<<(unsigned) ((ms->n_query_kps + 127) / 128), 128, 0, ctx->stream>>>(
        ms->n_query_kps, ms->n_scales, ms->k, ms->idx.as<int32_t>(), ms->dist.as<float>(), ms->cnt.as<int32_t>(), d_train_xyz,
        xyz_stride_bytes / 4, iss_radius, d_idx, d_dist, d_count);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

int ms_vote_batch_device(b200m_ctx *ctx, MultiscaleState *ms, const float *d_train_xyz, size_t xyz_stride_bytes,
                         const int32_t *d_kp_off, int n_pairs, const float *d_radii, int32_t *d_idx, float *d_dist,
                         int32_t *d_count) {
    if (ms->n_query_kps == 0) return 0;
    ms_vote_kernel<true><<<(unsigned) ((ms->n_query_kps + 127) / 128), 128, 0, ctx->stream>>>(
        ms->n_query_kps, ms->n_scales, ms->k, ms->idx.as<int32_t>(), ms->dist.as<float>(), ms->cnt.as<int32_t>(), d_train_xyz,
        xyz_stride_bytes / 4, 0.f, d_idx, d_dist, d_count, d_kp_off, n_pairs, d_radii);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

extern "C" {

int b200m_multiscale_begin(b200m_ctx *ctx, size_t n_query_kps, int n_scales, int k) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    return ms_begin(ctx, ms_state(ctx), n_query_kps, n_scales, k);
}

int b200m_multiscale_add_device(b200m_ctx *ctx, int scale, size_t n_rows, const int32_t *d_idx, const float *d_dist,
                                const int32_t *d_count, const int32_t *d_query_map, const int32_t *d_train_map,
                                size_t n_train_rows, int64_t train_index_offset, size_t n_train_kps) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    return ms_add_device(ctx, static_cast<MultiscaleState *>(ctx->multiscale), scale, n_rows, d_idx, d_dist, d_count, d_query_map,
                         d_train_map, n_train_rows, train_index_offset, n_train_kps);
}

int b200m_multiscale_vote_device(b200m_ctx *ctx, const float *d_train_xyz, size_t xyz_stride_bytes, float iss_radius,
                                 int32_t *d_idx, float *d_dist, int32_t *d_count) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    return ms_vote_device(ctx, static_cast<MultiscaleState *>(ctx->multiscale), d_train_xyz, xyz_stride_bytes, iss_radius, d_idx,
                          d_dist, d_count);
}

// ---- host-buffer forms: what match_multiscale's loop body and tail become ---------------------------
int b200m_multiscale_add(b200m_ctx *ctx, const b200m_params *p, int direction, int scale, const int32_t *query_map,
                         const int32_t *train_map, size_t n_train_kps) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    MultiscaleState *ms = static_cast<MultiscaleState *>(ctx->multiscale);
    if (!ms || ms->n_scales == 0) return b200m_fail_msg(ctx, "b200m_multiscale_add: call b200m_multiscale_begin first");
    if (!p || p->k != ms->k) return b200m_fail_msg(ctx, "b200m_multiscale_add: params.k differs from b200m_multiscale_begin's k");
    if (direction != 0 && direction != 1) return b200m_fail_msg(ctx, "b200m_multiscale_add: direction must be 0 or 1");
    Side &q = ctx->side[direction], &t = ctx->side[1 - direction];
    const size_t n_rows = q.n;
    if (n_rows == 0) return 0;
    CK(ms->kidx.reserve(sizeof(int32_t) * n_rows * ms->k));
    CK(ms->kdist.reserve(sizeof(float) * n_rows * ms->k));
    CK(ms->kcnt.reserve(sizeof(int32_t) * n_rows));
    b200m_params pk = *p;
    pk.mode = B200M_MODE_KNN_ONLY;
    if (b200m_knn_device(ctx, &pk, direction, 0, n_rows, ms->kidx.as<int32_t>(), ms->kdist.as<float>(), ms->kcnt.as<int32_t>()))
        return 1;
    const int32_t *d_qmap = nullptr, *d_tmap = nullptr;
    if (query_map) {
        CK(ms->qmap.reserve(sizeof(int32_t) * n_rows));
        CK(cudaMemcpyAsync(ms->qmap.p, query_map, sizeof(int32_t) * n_rows, cudaMemcpyHostToDevice, ctx->stream));
        d_qmap = ms->qmap.as<int32_t>();
    }
    if (train_map && t.n) {
        CK(ms->tmap.reserve(sizeof(int32_t) * t.n));
        CK(cudaMemcpyAsync(ms->tmap.p, train_map, sizeof(int32_t) * t.n, cudaMemcpyHostToDevice, ctx->stream));
        d_tmap = ms->tmap.as<int32_t>();
    }
    if (b200m_multiscale_add_device(ctx, scale, n_rows, ms->kidx.as<int32_t>(), ms->kdist.as<float>(), ms->kcnt.as<int32_t>(),
                                    d_qmap, d_tmap, t.n, t.index_offset, n_train_kps))
        return 1;
    // the host maps may be reused by the caller as soon as this returns
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int b200m_multiscale_vote(b200m_ctx *ctx, const float *train_xyz, size_t n_train_kps, size_t xyz_stride_bytes,
                          float iss_radius, int32_t *idx, float *dist, int32_t *count) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    MultiscaleState *ms = static_cast<MultiscaleState *>(ctx->multiscale);
    if (!ms || ms->n_scales == 0) return b200m_fail_msg(ctx, "b200m_multiscale_vote: call b200m_multiscale_begin first");
    const size_t nq = ms->n_query_kps;
    if (nq == 0) return 0;
    if (!idx || !dist || !count || (n_train_kps && !train_xyz)) return b200m_fail_msg(ctx, "b200m_multiscale_vote: null pointer");
    if (xyz_stride_bytes % 4 != 0 || xyz_stride_bytes < 12)
        return b200m_fail_msg(ctx, "b200m_multiscale_vote: xyz stride must be a multiple of 4 and >= 12 bytes");
    const size_t xyz_bytes = n_train_kps ? (n_train_kps - 1) * xyz_stride_bytes + 12 : 0;
    CK(ms->xyz.reserve(n_train_kps * xyz_stride_bytes + 16));
    if (xyz_bytes) CK(cudaMemcpyAsync(ms->xyz.p, train_xyz, xyz_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(ms->oidx.reserve(sizeof(int32_t) * nq));
    CK(ms->odist.reserve(sizeof(float) * nq));
    CK(ms->ocnt.reserve(sizeof(int32_t) * nq));
    if (b200m_multiscale_vote_device(ctx, ms->xyz.as<float>(), xyz_stride_bytes, iss_radius, ms->oidx.as<int32_t>(),
                                     ms->odist.as<float>(), ms->ocnt.as<int32_t>()))
        return 1;
    int bad = 0;
    CK(cudaMemcpyAsync(idx, ms->oidx.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(dist, ms->odist.p, sizeof(float) * nq, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(count, ms->ocnt.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&bad, ms->bad.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (bad == 1) return b200m_fail_msg(ctx, "b200m_multiscale: a query index map entry is outside [0, n_query_kps)");
    if (bad == 2) return b200m_fail_msg(ctx, "b200m_multiscale: a train index map entry is outside [0, n_train_kps)");
    return 0;
}

}  // extern "C"
