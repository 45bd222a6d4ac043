// cluster.cu -- ClusterMatcher<FeatureT>::match_impl (reference include/matching.h:480-551), the reference's default
// matching_id: a forward pair (i, j) survives when the matches of i's 3-D neighbours land among j's 3-D neighbours,
// and vice versa.
//
//   knn3d_kernel         the 3-D neighbourhoods (pcl::search::KdTree<PointN>::nearestKSearch(index, cluster_k), :524-528):
//                        one warp per keypoint, brute force over all keypoints of the same cloud (10^4..10^5 points:
//                        10^10 three-term distances, milliseconds), the point itself included; FLANN's L2_Simple
//                        squared distance (sequential FP32 sum over x, y, z); the k best by (distance, lower index)
//                        are kept in a per-warp sorted list in shared memory, insertions done by the whole warp.
//   cluster_dist_kernel  calculateCorrespondenceDistance (:519-550) in both directions for every forward pair:
//                        1 - consistent / pairs; the pair's value max(d_i, d_j) if both are under the threshold, else -1.
//   The order-preserving compaction is filter.cu's (mode B200M_MODE_CLUSTER).
#include <limits.h>
#include <math.h>

#include "internal.cuh"

namespace {

constexpr int kKnn3dWarps = 8;
constexpr int kMaxClusterK = 64;

__device__ __forceinline__ bool lex_less(float d1, int i1, float d2, int i2) { return d1 < d2 || (d1 == d2 && i1 < i2); }

// SEG (batch calls): the points of many pairs back to back, seg_off[p] = first point of pair p; point i only scans its own
// pair's points [seg_off[p], seg_off[p + 1]) and reports global ids.  A compile-time flag, so the single-pair instantiation
// is the kernel it was.
template <bool SEG>
__global__ void __launch_bounds__(kKnn3dWarps * 32)
knn3d_kernel(const float *__restrict__ xyz, size_t stride_floats, size_t n, int k, int32_t *__restrict__ nbr,
             const int32_t *__restrict__ seg_off = nullptr, int n_seg = 0) {
    __shared__ float s_d[kKnn3dWarps][kMaxClusterK];
    __shared__ int s_i[kKnn3dWarps][kMaxClusterK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *ld = s_d[warp];
    int *li = s_i[warp];
    for (size_t i = (size_t) blockIdx.x * kKnn3dWarps + warp; i < n; i += (size_t) gridDim.x * kKnn3dWarps) {
        ld[lane] = INFINITY; li[lane] = INT_MAX;
        ld[lane + 32] = INFINITY; li[lane + 32] = INT_MAX;
        __syncwarp();
        const float ax = xyz[i * stride_floats], ay = xyz[i * stride_floats + 1], az = xyz[i * stride_floats + 2];
        float tau_d = INFINITY;
        int tau_i = INT_MAX;
        size_t first = 0, end = n;
        if constexpr (SEG) {
            const int p = pair_of(seg_off, n_seg, (long long) i);
            first = (size_t) seg_off[p];
            end = (size_t) seg_off[p + 1];
        }
        for (size_t base = first; base < end; base += 32) {
            const size_t j = base + lane;
            float d = INFINITY;
            if (j < end) {
                const float *b = xyz + j * stride_floats;
                const float dx = __fsub_rn(ax, b[0]), dy = __fsub_rn(ay, b[1]), dz = __fsub_rn(az, b[2]);
                d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
            }
            unsigned mask = __ballot_sync(0xffffffffu, j < end && lex_less(d, (int) j, tau_d, tau_i));
            while (mask) {
                const int b = __ffs((int) mask) - 1;
                mask &= mask - 1;
                const float db = __shfl_sync(0xffffffffu, d, b);
                const int jb = (int) (base + b);
                if (!lex_less(db, jb, tau_d, tau_i)) continue;   // the k-th entry moved since the ballot
                // position = number of kept entries before the new one; both halves of the list, whole warp
                const float e0d = ld[lane], e1d = ld[lane + 32];
                const int e0i = li[lane], e1i = li[lane + 32];
                const bool c0 = lane < k && lex_less(e0d, e0i, db, jb);
                const bool c1 = lane + 32 < k && lex_less(e1d, e1i, db, jb);
                const int p = __popc(__ballot_sync(0xffffffffu, c0)) + __popc(__ballot_sync(0xffffffffu, c1));
                __syncwarp();
                if (lane >= p && lane + 1 < k) { ld[lane + 1] = e0d; li[lane + 1] = e0i; }
                if (lane + 32 >= p && lane + 33 < k) { ld[lane + 33] = e1d; li[lane + 33] = e1i; }
                __syncwarp();
                if (lane == 0) { ld[p] = db; li[p] = jb; }
                __syncwarp();
                tau_d = ld[k - 1];
                tau_i = li[k - 1];
            }
        }
        for (int e = lane; e < k; e += 32) nbr[i * (size_t) k + e] = li[e] == INT_MAX ? -1 : li[e];
        __syncwarp();
    }
}

// calculateCorrespondenceDistance(i, j, ...) over the k-lists `idx/count` of i's side
__device__ float cluster_distance(long long i, long long j, int ck, int k, const int32_t *__restrict__ idx,
                                  const int32_t *__restrict__ count, size_t n_a, const int32_t *__restrict__ nbr_a,
                                  const int32_t *__restrict__ nbr_b) {
    const int32_t *ni = nbr_a + (size_t) i * ck, *nj = nbr_b + (size_t) j * ck;
    int consistent = 0, pairs = 0;
    for (int a = 0; a < ck; ++a) {
        const int ia = ni[a];
        if (ia < 0 || (size_t) ia >= n_a) continue;
        const int c = count[ia];
        for (int m = 0; m < c; ++m) {
            const int32_t match = idx[(size_t) ia * k + m];
            for (int b = 0; b < ck; ++b) {
                const int v = nj[b];
                if (v >= 0 && v == match) { consistent++; break; }
            }
            pairs++;
        }
    }
    if (pairs == 0) return 0.f;
    return __fsub_rn(1.f, __fdiv_rn((float) consistent, (float) pairs));
}

__global__ void cluster_dist_kernel(size_t n_src, size_t n_tgt, int k, int ck, float cluster_thr,
                                    const int32_t *__restrict__ fidx, const int32_t *__restrict__ fcount,
                                    const int32_t *__restrict__ ridx, const int32_t *__restrict__ rcount,
                                    const int32_t *__restrict__ nbr_src, const int32_t *__restrict__ nbr_tgt,
                                    float *__restrict__ cdist) {
    const size_t e = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_src * (size_t) k) return;
    const size_t i = e / k;
    const int slot = (int) (e % k);
    float out = -1.f;
    if (slot < fcount[i]) {
        const int32_t j = fidx[e];
        if (j >= 0 && (size_t) j < n_tgt) {
            const float di = cluster_distance((long long) i, j, ck, k, fidx, fcount, n_src, nbr_src, nbr_tgt);
            const float dj = cluster_distance(j, (long long) i, ck, k, ridx, rcount, n_tgt, nbr_tgt, nbr_src);
            if (di < cluster_thr && dj < cluster_thr) out = fmaxf(di, dj);
        }
    }
    cdist[e] = out;
}

}  // namespace

struct ClusterState {
    DevBuf nbr_src, nbr_tgt, cdist, xyz_src, xyz_tgt;
};

static ClusterState *cl_state(b200m_ctx *ctx) {
    if (!ctx->cluster) ctx->cluster = new ClusterState();
    return static_cast<ClusterState *>(ctx->cluster);
}

void cluster_release(b200m_ctx *ctx) {
    ClusterState *cs = static_cast<ClusterState *>(ctx->cluster);
    if (!cs) return;
    DevBuf *b[] = {&cs->nbr_src, &cs->nbr_tgt, &cs->cdist, &cs->xyz_src, &cs->xyz_tgt};
    for (DevBuf *x : b) x->release();
    delete cs;
    ctx->cluster = nullptr;
}

int cluster_filter_batch_device(b200m_ctx *ctx, const b200m_params *p, int cluster_k, float cluster_thr, size_t n_src, size_t n_tgt,
                                const int32_t *d_fidx, const float *d_fdist, const int32_t *d_fcount, const int32_t *d_ridx,
                                const int32_t *d_rcount, const float *d_src_xyz, const float *d_tgt_xyz, size_t xyz_stride_bytes,
                                const int32_t *d_src_off, const int32_t *d_tgt_off, int n_pairs, const float *d_thr_src,
                                const float *d_thr_tgt, b200m_corr *d_out, size_t cap, unsigned long long *d_n_out) {
    if (cluster_k < 1 || cluster_k > kMaxClusterK) return b200m_fail_msg(ctx, "b200m_cluster_filter: cluster_k must be in [1, 64]");
    const int k = p->k;
    ClusterState *cs = cl_state(ctx);
    cudaStream_t st = ctx->stream;
    if (n_src == 0 || n_tgt == 0) {
        CK(cudaMemsetAsync(d_n_out, 0, sizeof(unsigned long long), st));
        return 0;
    }
    CK(cs->nbr_src.reserve(sizeof(int32_t) * n_src * cluster_k));
    CK(cs->nbr_tgt.reserve(sizeof(int32_t) * n_tgt * cluster_k));
    CK(cs->cdist.reserve(sizeof(float) * n_src * k));
    StatTimer t(ctx, &ctx->stats.ms_filter);
    const size_t cap_blocks = (size_t) ctx->sm_count * 8;
    const size_t ns[2] = {n_src, n_tgt};
    const float *xyz[2] = {d_src_xyz, d_tgt_xyz};
    const int32_t *off[2] = {d_src_off, d_tgt_off};
    int32_t *nbr[2] = {cs->nbr_src.as<int32_t>(), cs->nbr_tgt.as<int32_t>()};
    for (int s = 0; s < 2; ++s) {
        const size_t want = (ns[s] + kKnn3dWarps - 1) / kKnn3dWarps;
        knn3d_kernel<true><<<(unsigned) (want < cap_blocks ? want : cap_blocks), kKnn3dWarps * 32, 0, st>>>(
            xyz[s], xyz_stride_bytes / 4, ns[s], cluster_k, nbr[s], off[s], n_pairs);
        CK(cudaGetLastError());
    }
    const size_t n_elems = n_src * (size_t) k;
    cluster_dist_kernel<<<(unsigned) ((n_elems + 127) / 128), 128, 0, st>>>(
        n_src, n_tgt, k, cluster_k, cluster_thr, d_fidx, d_fcount, d_ridx, d_rcount, nbr[0], nbr[1], cs->cdist.as<float>());
    CK(cudaGetLastError());
    CK(ctx->ws_scan.reserve(filter_scan_ws_bytes(n_src, k)));
    int launches = 3;
    CK(launch_filter(B200M_MODE_CLUSTER, k, p->ratio_thr, p->distance_thr, 0, n_src, d_fidx, d_fdist, d_fcount, nullptr, nullptr,
                     nullptr, 0, d_thr_src, d_thr_tgt, 0, 0, d_out, cap, d_n_out, nullptr, ctx->ws_scan.p, ctx->ws_scan.cap, st,
                     &launches, cs->cdist.as<float>()));
    ctx->stats.launches += launches;
    t.stop();
    return 0;
}

extern "C" {

int b200m_knn3d_device(b200m_ctx *ctx, const float *d_xyz, size_t n, size_t xyz_stride_bytes, int k, int32_t *d_nbr) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    if (k < 1 || k > kMaxClusterK) return b200m_fail_msg(ctx, "b200m_knn3d: k must be in [1, 64]");
    if (xyz_stride_bytes % 4 != 0 || xyz_stride_bytes < 12) return b200m_fail_msg(ctx, "b200m_knn3d: xyz stride must be a multiple of 4 and >= 12 bytes");
    if (n == 0) return 0;
    if (!d_xyz || !d_nbr) return b200m_fail_msg(ctx, "b200m_knn3d: null pointer");
    size_t want = (n + kKnn3dWarps - 1) / kKnn3dWarps, cap = (size_t) ctx->sm_count * 8;
    knn3d_kernel<false><<<(unsigned) (want < cap ? want : cap), kKnn3dWarps * 32, 0, ctx->stream>>>(d_xyz, xyz_stride_bytes / 4, n, k, d_nbr);
    CK(cudaGetLastError());
    ctx->stats.launches += 1;
    return 0;
}

int b200m_cluster_filter_device(b200m_ctx *ctx, const b200m_params *p, int cluster_k, float cluster_thr, size_t n_src, size_t n_tgt,
                                const int32_t *d_fidx, const float *d_fdist, const int32_t *d_fcount,
                                const int32_t *d_ridx, const int32_t *d_rcount, const float *d_src_xyz,
                                const float *d_tgt_xyz, size_t xyz_stride_bytes, const float *d_thr_src,
                                const float *d_thr_tgt, b200m_corr *d_out, size_t cap, unsigned long long *d_n_out,
                                float *d_avg) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    if (!p || p->k < 1 || p->k > B200M_MAX_K) return b200m_fail_msg(ctx, "b200m_cluster_filter: params.k must be in [1, 32]");
    if (cluster_k < 1 || cluster_k > kMaxClusterK) return b200m_fail_msg(ctx, "b200m_cluster_filter: cluster_k must be in [1, 64]");
    if (!d_n_out) return b200m_fail_msg(ctx, "b200m_cluster_filter: null n_out");
    if (ctx->side[0].index_offset || ctx->side[1].index_offset)   // the neighbourhood tables are addressed by the reported indices
        return b200m_fail_msg(ctx, "b200m_cluster_filter: descriptor sets uploaded with a non-zero index_offset are not supported");
    const int k = p->k;
    ClusterState *cs = cl_state(ctx);
    cudaStream_t st = ctx->stream;
    if (n_src == 0 || n_tgt == 0) {
        CK(cudaMemsetAsync(d_n_out, 0, sizeof(unsigned long long), st));
        return 0;
    }
    if (!d_fidx || !d_fdist || !d_fcount || !d_ridx || !d_rcount || !d_src_xyz || !d_tgt_xyz || (cap && !d_out))
        return b200m_fail_msg(ctx, "b200m_cluster_filter: null pointer");
    CK(cs->nbr_src.reserve(sizeof(int32_t) * n_src * cluster_k));
    CK(cs->nbr_tgt.reserve(sizeof(int32_t) * n_tgt * cluster_k));
    CK(cs->cdist.reserve(sizeof(float) * n_src * k));
    StatTimer t(ctx, &ctx->stats.ms_filter);
    if (b200m_knn3d_device(ctx, d_src_xyz, n_src, xyz_stride_bytes, cluster_k, cs->nbr_src.as<int32_t>())) return 1;
    if (b200m_knn3d_device(ctx, d_tgt_xyz, n_tgt, xyz_stride_bytes, cluster_k, cs->nbr_tgt.as<int32_t>())) return 1;
    const size_t n_elems = n_src * (size_t) k;
    cluster_dist_kernel<<<(unsigned) ((n_elems + 127) / 128), 128, 0, st>>>(
        n_src, n_tgt, k, cluster_k, cluster_thr, d_fidx, d_fcount, d_ridx, d_rcount, cs->nbr_src.as<int32_t>(),
        cs->nbr_tgt.as<int32_t>(), cs->cdist.as<float>());
    CK(cudaGetLastError());
    CK(ctx->ws_scan.reserve(filter_scan_ws_bytes(n_src, k)));
    int launches = 1;
    CK(launch_filter(B200M_MODE_CLUSTER, k, p->ratio_thr, p->distance_thr, 0, n_src, d_fidx, d_fdist, d_fcount, nullptr, nullptr,
                     nullptr, 0, d_thr_src, d_thr_tgt, ctx->side[0].index_offset, ctx->side[1].index_offset, d_out, cap, d_n_out, d_avg,
                     ctx->ws_scan.p,
                     ctx->ws_scan.cap, st, &launches, cs->cdist.as<float>()));
    ctx->stats.launches += launches;
    t.stop();
    return 0;
}

int b200m_match_cluster(b200m_ctx *ctx, const b200m_params *p, int cluster_k, const float *src_kps_xyz,
                        const float *tgt_kps_xyz, size_t xyz_stride_bytes, const float *thr_src, const float *thr_tgt,
                        b200m_corr *out, size_t cap, size_t *n_out, float *avg_first_dist) {
    if (!ctx) return b200m_fail_msg(nullptr, "null context");
    CK(cudaSetDevice(ctx->device));
    if (!p || !n_out) return b200m_fail_msg(ctx, "b200m_match_cluster: null params / n_out");
    *n_out = 0;
    if ((thr_src == nullptr) != (thr_tgt == nullptr)) return b200m_fail_msg(ctx, "b200m_match_cluster: give both threshold arrays or neither");
    if (xyz_stride_bytes % 4 != 0 || xyz_stride_bytes < 12) return b200m_fail_msg(ctx, "b200m_match_cluster: xyz stride must be a multiple of 4 and >= 12 bytes");
    Side &src = ctx->side[0], &tgt = ctx->side[1];
    const size_t nq = src.n, nt = tgt.n;
    const int k = p->k;
    cudaStream_t st = ctx->stream;
    if (nq == 0) {
        if (avg_first_dist) *avg_first_dist = 3.402823466e+38F;   // FLT_MAX, reference include/matching.h:41
        return 0;
    }
    if (!src_kps_xyz || (nt && !tgt_kps_xyz)) return b200m_fail_msg(ctx, "b200m_match_cluster: null keypoint coordinates");
    b200m_params pk = *p;
    pk.mode = B200M_MODE_KNN_ONLY;
    CK(ctx->ws_fidx.reserve(sizeof(int32_t) * nq * k));
    CK(ctx->ws_fdist.reserve(sizeof(float) * nq * k));
    CK(ctx->ws_fcnt.reserve(sizeof(int32_t) * nq));
    if (b200m_knn_device(ctx, &pk, 0, 0, nq, ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>())) return 1;
    if (nt) {
        CK(ctx->ws_ridx.reserve(sizeof(int32_t) * nt * k));
        CK(ctx->ws_rdist.reserve(sizeof(float) * nt * k));
        CK(ctx->ws_rcnt.reserve(sizeof(int32_t) * nt));
        if (b200m_knn_device(ctx, &pk, 1, 0, nt, ctx->ws_ridx.as<int32_t>(), ctx->ws_rdist.as<float>(), ctx->ws_rcnt.as<int32_t>())) return 1;
    }
    ClusterState *cs = cl_state(ctx);
    const size_t sb = (nq - 1) * xyz_stride_bytes + 12, tb = nt ? (nt - 1) * xyz_stride_bytes + 12 : 0;
    CK(cs->xyz_src.reserve(nq * xyz_stride_bytes + 16));
    CK(cs->xyz_tgt.reserve(nt * xyz_stride_bytes + 16));
    CK(cudaMemcpyAsync(cs->xyz_src.p, src_kps_xyz, sb, cudaMemcpyHostToDevice, st));
    if (tb) CK(cudaMemcpyAsync(cs->xyz_tgt.p, tgt_kps_xyz, tb, cudaMemcpyHostToDevice, st));
    const float *d_thr_s = nullptr, *d_thr_t = nullptr;
    if (thr_src && nt) {
        CK(ctx->ws_thr[0].reserve(sizeof(float) * nq));
        CK(ctx->ws_thr[1].reserve(sizeof(float) * nt));
        CK(cudaMemcpyAsync(ctx->ws_thr[0].p, thr_src, sizeof(float) * nq, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->ws_thr[1].p, thr_tgt, sizeof(float) * nt, cudaMemcpyHostToDevice, st));
        d_thr_s = ctx->ws_thr[0].as<float>();
        d_thr_t = ctx->ws_thr[1].as<float>();
    }
    CK(ctx->ws_misc.reserve(64));
    float *d_avg = ctx->ws_misc.as<float>();
    unsigned long long *d_n = reinterpret_cast<unsigned long long *>(ctx->ws_misc.as<char>() + 16);
    const size_t max_out = nq * (size_t) k;
    CK(ctx->ws_corr.reserve(sizeof(b200m_corr) * max_out));
    if (b200m_cluster_filter_device(ctx, p, cluster_k, 0.95f /* MATCHING_CLUSTER_THRESHOLD, include/common.h:52 */, nq, nt,
                                    ctx->ws_fidx.as<int32_t>(), ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>(),
                                    ctx->ws_ridx.as<int32_t>(), ctx->ws_rcnt.as<int32_t>(), cs->xyz_src.as<float>(),
                                    cs->xyz_tgt.as<float>(), xyz_stride_bytes, d_thr_s, d_thr_t, ctx->ws_corr.as<b200m_corr>(),
                                    max_out, d_n, avg_first_dist ? d_avg : nullptr))
        return 1;
    if (nt == 0 && avg_first_dist) CK(launch_average(ctx->ws_fdist.as<float>(), ctx->ws_fcnt.as<int32_t>(), nq, k, d_avg, st));
    struct { float avg; float pad[3]; unsigned long long n; } h;
    CK(cudaMemcpyAsync(&h, ctx->ws_misc.p, sizeof(h), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (avg_first_dist) *avg_first_dist = h.avg;
    *n_out = (size_t) h.n;
    if (h.n > cap) return b200m_fail_msg(ctx, "b200m_match_cluster: output capacity too small (" + std::to_string(h.n) + " correspondences)");
    if (h.n) {
        if (!out) return b200m_fail_msg(ctx, "b200m_match_cluster: null output buffer");
        CK(cudaMemcpyAsync(out, ctx->ws_corr.p, sizeof(b200m_corr) * h.n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return 0;
}

}  // extern "C"
