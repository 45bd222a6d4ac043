// filter.cu -- correspondence filters over the k-lists, emitted in the reference's
// order (ascending index_query, then list order) by an order-preserving compaction.
//
//   one-sided : OneSidedMatcher::match_impl     (reference include/matching.h:395-411)
//   mutual    : LeftToRightMatcher::match_impl  (:428-453), k-list form; the emitted
//               distance is the REVERSE list's (:443)
//   ratio     : RatioMatcher (stub in the reference, :470-473) as defined in DESIGN.md:
//               keep (i, j1, d1) iff d2 >= ratio_thr * d1 (FP32 product), needs 2 neighbours
//   threshold : min(max(thr_src[i], thr_tgt[j]), distance_thr)   (:404-405, :441-442)
//   average   : FeatureBasedMatcher::printDebugInfo (src/matching.cpp:3-19): FP32 running
//               sum of first-NN distances in index order -- kept sequential so the float
//               result is bit-identical to the reference's loop.
//   merge     : k best of n_lists k-lists per query by (dist, idx) -- the cross-block job of
//               updateMultivaluedCorrespondence (src/common.cpp:517-529), canonical tie rule.
//
// HBM-bound scans; algorithmic bytes: n_rows*k*8 (forward table) + gathered reverse rows
// + 16 B per emitted correspondence.
#include <limits.h>
#include <math.h>

#include "internal.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kItems = 4;
constexpr int kElemsPerBlock = kThreads * kItems;

struct FilterArgs {
    int mode, k, kk;
    float ratio_thr, distance_thr;
    size_t row_begin, n_rows, n_rev_rows;
    const int32_t *fidx; const float *fdist; const int32_t *fcount;
    const int32_t *ridx; const float *rdist; const int32_t *rcount;
    const float *thr_src; const float *thr_tgt;
    const float *cdist;   // cluster mode: per (row, slot) max cluster distance, negative = rejected (cluster.cu)
    long long src_offset, tgt_offset;   // index_offset of the two sides: reported indices carry them, table rows do not
};

__device__ __forceinline__ bool eval_elem(const FilterArgs &a, size_t e, b200m_corr &c) {
    const size_t local = e / a.kk;
    const int slot = (int) (e % a.kk);
    const int fc = a.fcount[local];
    if (slot >= fc) return false;
    const int32_t *fi = a.fidx + local * a.k;
    const float *fd = a.fdist + local * a.k;
    const size_t i_loc = a.row_begin + local;
    const long long i_glob = (long long) i_loc + a.src_offset;
    int32_t j = fi[slot];
    const long long j_loc = (long long) j - a.tgt_offset;   // row of the reverse table / threshold array
    float d = fd[slot];
    if (a.mode == B200M_MODE_RATIO || a.mode == B200M_MODE_RATIO_MUTUAL) {
        if (fc < 2) return false;
        if (!(fd[1] >= __fmul_rn(a.ratio_thr, fd[0]))) return false;
    }
    if (a.mode == B200M_MODE_CLUSTER) {   // ClusterMatcher::match_impl (:503-515): the emitted distance is max(d_i, d_j)
        const float cd = a.cdist[e];
        if (!(cd >= 0.f)) return false;
        d = cd;
    }
    if (a.mode == B200M_MODE_MUTUAL || a.mode == B200M_MODE_RATIO_MUTUAL) {
        if (j_loc < 0 || (size_t) j_loc >= a.n_rev_rows) return false;
        const int rc = a.rcount[j_loc];
        const int32_t *ri = a.ridx + (size_t) j_loc * a.k;
        bool hit = false;
        for (int m = 0; m < rc; ++m) {
            if ((long long) ri[m] == i_glob) {
                d = a.rdist[(size_t) j_loc * a.k + m];
                hit = true;
                break;
            }
        }
        if (!hit) return false;
    }
    float thr = a.distance_thr;
    if (a.thr_src && a.thr_tgt) {
        float t = fmaxf(a.thr_src[i_loc], j_loc >= 0 ? a.thr_tgt[j_loc] : a.distance_thr);
        thr = fminf(t, a.distance_thr);
    }
    c.index_query = (int32_t) i_glob;
    c.index_match = j;
    c.distance = d;
    c.threshold = thr;
    return true;
}

__global__ void __launch_bounds__(kThreads)
filter_count_kernel(FilterArgs a, size_t n_elems, unsigned *__restrict__ block_counts) {
    size_t base = (size_t) blockIdx.x * kElemsPerBlock + (size_t) threadIdx.x * kItems;
    unsigned c = 0;
    b200m_corr tmp;
#pragma unroll
    for (int u = 0; u < kItems; ++u)
        if (base + u < n_elems && eval_elem(a, base + u, tmp)) c++;
    __shared__ unsigned wsum[kThreads / 32];
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
        for (int w = 0; w < kThreads / 32; ++w) t += wsum[w];
        block_counts[blockIdx.x] = t;
    }
}

// single CTA: exclusive scan of block_counts -> block_offsets (64-bit), total -> n_out
__global__ void __launch_bounds__(1024)
filter_scan_kernel(const unsigned *__restrict__ block_counts, size_t n_blocks,
                   unsigned long long *__restrict__ block_offsets, unsigned long long *__restrict__ n_out) {
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long carry, chunk_total;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (size_t base = 0; base < n_blocks; base += 1024) {
        size_t i = base + threadIdx.x;
        unsigned long long v = i < n_blocks ? block_counts[i] : 0ull, inc = v;
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = wsum[lane], winc = w;
            for (int o = 1; o < 32; o <<= 1) {
                unsigned long long t = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o) winc += t;
            }
            wsum[lane] = winc - w;              // exclusive prefix of the warp sums
            if (lane == 31) chunk_total = winc;
        }
        __syncthreads();
        if (i < n_blocks) block_offsets[i] = carry + wsum[warp] + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) carry += chunk_total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_out = carry;
}

__global__ void __launch_bounds__(kThreads)
filter_scatter_kernel(FilterArgs a, size_t n_elems, const unsigned long long *__restrict__ block_offsets,
                      b200m_corr *__restrict__ out, size_t cap) {
    size_t base = (size_t) blockIdx.x * kElemsPerBlock + (size_t) threadIdx.x * kItems;
    b200m_corr c[kItems];
    bool f[kItems];
    unsigned cnt = 0;
#pragma unroll
    for (int u = 0; u < kItems; ++u) {
        f[u] = base + u < n_elems && eval_elem(a, base + u, c[u]);
        cnt += f[u] ? 1u : 0u;
    }
    __shared__ unsigned wsum[kThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned inc = cnt;
    for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    unsigned wpre = 0;
    for (int w = 0; w < warp; ++w) wpre += wsum[w];
    unsigned long long pos = block_offsets[blockIdx.x] + wpre + (inc - cnt);
#pragma unroll
    for (int u = 0; u < kItems; ++u) {
        if (f[u]) {
            if (pos < cap) out[pos] = c[u];
            pos++;
        }
    }
}

// FP32 running sum in index order (src/matching.cpp:6-11).  The additions are ONE dependent chain by definition (every
// partial sum is rounded before the next term is added), so the kernel is built around that chain: thread 0 adds the
// 4096 values of a shared-memory buffer with 128-bit loads and nothing else in its loop (~4 cycles per term, the FADD
// latency), while warps 1..7 fill the other buffer with the next 4096 first-neighbour distances.  A row without a
// neighbour contributes +0.0f, which leaves a non-negative (or non-finite) running sum unchanged bit for bit, so the
// chain needs no predicate; the rows that do count are tallied on the side.  (The first version -- one warp, 32 shuffles
// and predicated adds per 32 rows, loads not overlapped -- took ~6 ms for 500k rows; this one ~1.2 ms.)
// segs != null (batch calls): CTA s runs the same chain over rows [segs[s].x, segs[s].x + segs[s].y) into avg[s].
constexpr int kAvgChunk = 4096;
constexpr int kAvgThreads = 256;
__global__ void __launch_bounds__(kAvgThreads) average_kernel(const float *__restrict__ fdist, const int32_t *__restrict__ fcount,
                                                              size_t n_rows, int k, float *__restrict__ avg,
                                                              const int2 *__restrict__ segs) {
    if (segs) {
        const int2 sg = segs[blockIdx.x];
        fdist += (size_t) sg.x * k;
        fcount += sg.x;
        n_rows = (size_t) sg.y;
        avg += blockIdx.x;
    }
    __shared__ __align__(16) float buf[2][kAvgChunk];
    __shared__ unsigned long long n_with;
    const int tid = threadIdx.x;
    if (tid == 0) n_with = 0ull;
    unsigned long long mine = 0ull;
    const size_t n_chunks = (n_rows + kAvgChunk - 1) / kAvgChunk;
    auto fill = [&](size_t c, int first_thread, int n_threads) {
        float *b = buf[c & 1];
        const size_t base = c * kAvgChunk;
        for (int i = tid - first_thread; i < kAvgChunk; i += n_threads) {
            const size_t row = base + (size_t) i;
            const bool has = row < n_rows && fcount[row] > 0;
            b[i] = has ? fdist[row * (size_t) k] : 0.f;
            mine += has ? 1ull : 0ull;
        }
    };
    if (n_chunks) fill(0, 0, kAvgThreads);
    __syncthreads();
    float sum = 0.f;
    for (size_t c = 0; c < n_chunks; ++c) {
        if (tid >= 32) {
            if (c + 1 < n_chunks) fill(c + 1, 32, kAvgThreads - 32);
        } else if (tid == 0) {
            const float4 *b4 = reinterpret_cast<const float4 *>(buf[c & 1]);
#pragma unroll 8
            for (int i = 0; i < kAvgChunk / 4; ++i) {
                const float4 v = b4[i];
                sum = __fadd_rn(sum, v.x);
                sum = __fadd_rn(sum, v.y);
                sum = __fadd_rn(sum, v.z);
                sum = __fadd_rn(sum, v.w);
            }
        }
        __syncthreads();
    }
    if (mine) atomicAdd(&n_with, mine);
    __syncthreads();
    if (tid == 0) *avg = n_with == 0ull ? 3.402823466e+38F : __fdiv_rn(sum, (float) n_with);
}

__global__ void merge_kernel(int k, int n_lists, size_t nq, const int32_t *__restrict__ idx_in,
                             const float *__restrict__ dist_in, const int32_t *__restrict__ count_in,
                             int32_t *__restrict__ idx, float *__restrict__ dist, int32_t *__restrict__ count) {
    size_t q = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    int head[8];
    for (int l = 0; l < n_lists; ++l) head[l] = 0;
    int found = 0;
    for (int r = 0; r < k; ++r) {
        float bd = INFINITY;
        int bi = INT_MAX, bl = -1;
        for (int l = 0; l < n_lists; ++l) {
            size_t row = (size_t) l * nq + q;
            if (head[l] < count_in[row]) {
                float d = dist_in[row * k + head[l]];
                int i = idx_in[row * k + head[l]];
                if (d < bd || (d == bd && i < bi)) { bd = d; bi = i; bl = l; }
            }
        }
        if (bl < 0) break;
        head[bl]++;
        idx[q * k + r] = bi;
        dist[q * k + r] = bd;
        found = r + 1;
    }
    for (int r = found; r < k; ++r) { idx[q * k + r] = -1; dist[q * k + r] = 0.f; }
    count[q] = found;
}

}  // namespace

static size_t n_filter_blocks(size_t n_rows, int kk) {
    size_t n_elems = n_rows * (size_t) kk;
    return (n_elems + kElemsPerBlock - 1) / kElemsPerBlock;
}

size_t filter_scan_ws_bytes(size_t n_rows, int k) {
    size_t nb = n_filter_blocks(n_rows, k) + 1;
    return nb * (sizeof(unsigned) + sizeof(unsigned long long)) + 64;
}

cudaError_t launch_filter(int mode, int k, float ratio_thr, float distance_thr, size_t row_begin, size_t n_rows,
                          const int32_t *fidx, const float *fdist, const int32_t *fcount,
                          const int32_t *ridx, const float *rdist, const int32_t *rcount, size_t n_rev_rows,
                          const float *thr_src, const float *thr_tgt, int64_t src_offset, int64_t tgt_offset,
                          b200m_corr *out, size_t cap, unsigned long long *n_out, float *avg,
                          void *scan_ws, size_t scan_ws_bytes, cudaStream_t st, int *n_launches, const float *cdist) {
    FilterArgs a;
    a.mode = mode; a.k = k;
    a.kk = (mode == B200M_MODE_MUTUAL || mode == B200M_MODE_CLUSTER) ? k : 1;
    a.cdist = cdist;
    a.ratio_thr = ratio_thr; a.distance_thr = distance_thr;
    a.row_begin = row_begin; a.n_rows = n_rows; a.n_rev_rows = n_rev_rows;
    a.fidx = fidx; a.fdist = fdist; a.fcount = fcount;
    a.ridx = ridx; a.rdist = rdist; a.rcount = rcount;
    a.thr_src = thr_src; a.thr_tgt = thr_tgt; a.src_offset = src_offset; a.tgt_offset = tgt_offset;
    size_t n_elems = n_rows * (size_t) a.kk;
    size_t nb = n_filter_blocks(n_rows, a.kk);
    if (filter_scan_ws_bytes(n_rows, k) > scan_ws_bytes) return cudaErrorInvalidValue;
    unsigned long long *block_offsets = (unsigned long long *) scan_ws;
    unsigned *block_counts = (unsigned *) (block_offsets + nb + 1);
    if (nb > 0) {
        filter_count_kernel<<<(unsigned) nb, kThreads, 0, st>>>(a, n_elems, block_counts);
        filter_scan_kernel<<<1, 1024, 0, st>>>(block_counts, nb, block_offsets, n_out);
        filter_scatter_kernel<<<(unsigned) nb, kThreads, 0, st>>>(a, n_elems, block_offsets, out, cap);
        *n_launches += 3;
    } else {
        cudaError_t e = cudaMemsetAsync(n_out, 0, sizeof(unsigned long long), st);
        if (e != cudaSuccess) return e;
    }
    if (avg) {
        average_kernel<<<1, kAvgThreads, 0, st>>>(fdist, fcount, n_rows, k, avg, nullptr);
        *n_launches += 1;
    }
    return cudaGetLastError();
}

cudaError_t launch_average(const float *fdist, const int32_t *fcount, size_t n_rows, int k, float *avg,
                           cudaStream_t st) {
    average_kernel<<<1, kAvgThreads, 0, st>>>(fdist, fcount, n_rows, k, avg, nullptr);
    return cudaGetLastError();
}

cudaError_t launch_average_segments(const float *fdist, const int32_t *fcount, const int2 *segs, int n_segs, int k, float *avg,
                                    cudaStream_t st) {
    if (n_segs <= 0) return cudaSuccess;
    average_kernel<<<(unsigned) n_segs, kAvgThreads, 0, st>>>(fdist, fcount, 0, k, avg, segs);
    return cudaGetLastError();
}

cudaError_t launch_merge(int k, int n_lists, size_t nq, const int32_t *idx_in, const float *dist_in,
                         const int32_t *count_in, int32_t *idx, float *dist, int32_t *count, cudaStream_t st) {
    if (nq == 0) return cudaSuccess;
    if (n_lists > 8) return cudaErrorInvalidValue;
    merge_kernel<<<(unsigned) ((nq + 127) / 128), 128, 0, st>>>(k, n_lists, nq, idx_in, dist_in, count_in, idx, dist,
                                                                count);
    return cudaGetLastError();
}
