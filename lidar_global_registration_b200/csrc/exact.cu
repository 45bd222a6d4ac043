// exact.cu -- exact FP32 CUDA-core kernels.
//
// Arithmetic is the reference's own, bit for bit: pcl::L2_Norm as called by matchLocal
// (reference include/matching.h:663) == FLANN L2_Simple under matchFLANN (:581) --
//     s = 0; for d: diff = a[d]-b[d]; s = s + diff*diff;  dist = sqrt(s)
// sequential over d in FP32 with separate multiply and add (the reference builds for
// baseline x86-64: no FMA), so distances are BIT-IDENTICAL to the CPU oracle and the
// order (dist, index) -- KNNResult's "earlier stays first", include/matching.h:69-93 --
// is reproduced exactly, ties included.
//
//   exact_rows_kernel   one CTA per query row, all train rows: the universal exact path
//                       (B200M_PREC_F32_EXACT, and the fallback for rows whose candidate
//                       list overflowed).
//   rerank_kernel       one warp per query row over the candidate lists of the tensor-core
//                       pass (a certified superset of the exact top-k, see candidates_tc.cu):
//                       exact distances and the final (dist, idx) order.
#include <float.h>
#include <stdlib.h>
#include <limits.h>
#include <math.h>

#include "internal.cuh"

namespace {

__device__ __forceinline__ bool lex_less(float d1, int i1, float d2, int i2) {
    return d1 < d2 || (d1 == d2 && i1 < i2);
}

// pcl::L2_Norm's squared sum over a dp-padded row pair (padding columns are 0 on both
// sides and add +0.0f, which leaves s unchanged).  q in shared memory, t in global.
__device__ __forceinline__ float seq_sqdist(const float *__restrict__ q, const float *__restrict__ t, int dp) {
    float s = 0.f;
    const float4 *t4 = reinterpret_cast<const float4 *>(t);
    for (int c = 0; c < dp / 4; ++c) {
        float4 v = __ldg(t4 + c);
        float d0 = __fsub_rn(q[4 * c + 0], v.x);
        s = __fadd_rn(s, __fmul_rn(d0, d0));
        float d1 = __fsub_rn(q[4 * c + 1], v.y);
        s = __fadd_rn(s, __fmul_rn(d1, d1));
        float d2 = __fsub_rn(q[4 * c + 2], v.z);
        s = __fadd_rn(s, __fmul_rn(d2, d2));
        float d3 = __fsub_rn(q[4 * c + 3], v.w);
        s = __fadd_rn(s, __fmul_rn(d3, d3));
    }
    return s;
}

constexpr int kExactThreads = 256;

template <int KMAX>
__global__ void __launch_bounds__(kExactThreads)
exact_rows_kernel(const float *__restrict__ q_f32, const uint8_t *__restrict__ q_valid, int dp, int dim,
                  const float *__restrict__ t_f32, const uint8_t *__restrict__ t_valid, size_t nt,
                  long long t_off, size_t row_begin, size_t n_rows, const int32_t *__restrict__ row_list,
                  const int32_t *__restrict__ row_list_count, int k, int32_t *__restrict__ idx,
                  float *__restrict__ dist, int32_t *__restrict__ count, int split_max,
                  const int32_t *__restrict__ row_map, const int2 *__restrict__ seg_range) {
    extern __shared__ float smem[];
    float *sq = smem;                                   // [dp] query row
    float *red_d = smem + dp;                           // [warps]
    int *red_i = reinterpret_cast<int *>(red_d + kExactThreads / 32);
    int *red_w = red_i + kExactThreads / 32;            // winner thread id per warp
    __shared__ float win_d;
    __shared__ int win_i, win_t;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t total = row_list ? (size_t) *row_list_count : n_rows;
    if (row_list && split_max > 0 && total <= (size_t) split_max) return;   // few flagged rows: exact_rows_split_kernel has them

    for (size_t r = blockIdx.x; r < total; r += gridDim.x) {
        // `local` numbers the rows of this call (compacted when a row map is given); results are stored by original row
        const size_t local = row_list ? (size_t) row_list[r] : r;
        const size_t qi = row_map ? (size_t) row_map[local] : row_begin + local;
        const size_t orow = qi - row_begin;
        int32_t *oi = idx + orow * k;
        float *od = dist + orow * k;
        if (!q_valid[qi]) {   // non-finite query -> empty entry (reference include/matching.h:576)
            if (tid < k) { oi[tid] = -1; od[tid] = 0.f; }
            if (tid == 0) count[orow] = 0;
            continue;
        }
        __syncthreads();
        for (int d = tid; d < dp; d += kExactThreads) sq[d] = q_f32[qi * (size_t) dp + d];
        __syncthreads();

        float ld[KMAX];
        int li[KMAX];
#pragma unroll
        for (int m = 0; m < KMAX; ++m) { ld[m] = INFINITY; li[m] = INT_MAX; }
        size_t j_lo = 0, j_hi = nt;   // batch calls: the train rows of the query's own pair
        if (seg_range) {
            const int2 r = seg_range[qi / B200M_TILE_N];
            j_lo = (size_t) r.x;
            j_hi = (size_t) r.y;
        }
        for (size_t j = j_lo + tid; j < j_hi; j += kExactThreads) {
            if (!t_valid[j]) continue;   // invalid train rows are never candidates (:661)
            float d = __fsqrt_rn(seq_sqdist(sq, t_f32 + j * (size_t) dp, dp));
            if (lex_less(d, (int) j, ld[KMAX - 1], li[KMAX - 1])) {
                // sorted insertion, fully unrolled so the list stays in registers
                float cd = d;
                int ci = (int) j;
#pragma unroll
                for (int m = 0; m < KMAX; ++m) {
                    if (lex_less(cd, ci, ld[m], li[m])) {
                        float td = ld[m]; int ti = li[m];
                        ld[m] = cd; li[m] = ci;
                        cd = td; ci = ti;
                    }
                }
            }
        }
        // k rounds of block-wide arg-min over the per-thread list heads
        int head = 0, found = 0;
        for (int round = 0; round < k; ++round) {
            float hd = INFINITY;
            int hi = INT_MAX;
#pragma unroll
            for (int m = 0; m < KMAX; ++m)
                if (m == head) { hd = ld[m]; hi = li[m]; }
            float bd = hd;
            int bi = hi, bt = tid;
            for (int o = 16; o > 0; o >>= 1) {
                float od2 = __shfl_xor_sync(0xffffffffu, bd, o);
                int oi2 = __shfl_xor_sync(0xffffffffu, bi, o);
                int ot2 = __shfl_xor_sync(0xffffffffu, bt, o);
                if (lex_less(od2, oi2, bd, bi)) { bd = od2; bi = oi2; bt = ot2; }
            }
            if (lane == 0) { red_d[warp] = bd; red_i[warp] = bi; red_w[warp] = bt; }
            __syncthreads();
            if (tid == 0) {
                float wd = red_d[0];
                int wi = red_i[0], wt = red_w[0];
                for (int w = 1; w < kExactThreads / 32; ++w)
                    if (lex_less(red_d[w], red_i[w], wd, wi)) { wd = red_d[w]; wi = red_i[w]; wt = red_w[w]; }
                win_d = wd; win_i = wi; win_t = wt;
            }
            __syncthreads();
            if (win_i == INT_MAX) break;   // fewer than k valid train rows
            if (tid == win_t) head++;
            if (tid == 0) { oi[round] = (int32_t) (win_i + t_off); od[round] = win_d; }
            found = round + 1;
            __syncthreads();
        }
        if (tid >= found && tid < k) { oi[tid] = -1; od[tid] = 0.f; }
        if (tid == 0) count[orow] = found;
    }
}

// ---- matchLocal with a finite search radius (reference include/matching.h:637-678) ------------------------
// One CTA per query row over ALL train rows: the 3-D gate first -- FLANN's L2_Simple squared distance between the
// (guess-transformed) query keypoint and the train keypoint, strictly below radius^2 (KdTree::radiusSearch, :661) --
// then pcl::L2_Norm on the descriptors of the gated rows only.  radiusSearch returns its hits sorted by spatial distance
// and KNNResult keeps the earlier insertion first among equal descriptor distances, so the order is
// (descriptor distance, spatial distance, index).
__device__ __forceinline__ bool lex3_less(float d1, float s1, int i1, float d2, float s2, int i2) {
    return d1 < d2 || (d1 == d2 && (s1 < s2 || (s1 == s2 && i1 < i2)));
}

template <int KMAX>
__global__ void __launch_bounds__(kExactThreads)
local_rows_kernel(const float *__restrict__ q_f32, const uint8_t *__restrict__ q_valid, int dp,
                  const float *__restrict__ t_f32, const uint8_t *__restrict__ t_valid, size_t nt, long long t_off,
                  size_t n_rows, const float *__restrict__ q_xyz, const float *__restrict__ t_xyz, size_t xyz_stride_floats,
                  float r2, int k, int32_t *__restrict__ idx, float *__restrict__ dist, int32_t *__restrict__ count) {
    extern __shared__ float smem[];
    float *sq = smem;
    float *red_d = smem + dp;
    float *red_s = red_d + kExactThreads / 32;
    int *red_i = reinterpret_cast<int *>(red_s + kExactThreads / 32);
    int *red_w = red_i + kExactThreads / 32;
    __shared__ float win_d, win_s;
    __shared__ int win_i, win_t;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (size_t qi = blockIdx.x; qi < n_rows; qi += gridDim.x) {
        int32_t *oi = idx + qi * k;
        float *od = dist + qi * k;
        if (!q_valid[qi]) {   // non-finite query -> empty entry (:658)
            if (tid < k) { oi[tid] = -1; od[tid] = 0.f; }
            if (tid == 0) count[qi] = 0;
            continue;
        }
        __syncthreads();
        for (int d = tid; d < dp; d += kExactThreads) sq[d] = q_f32[qi * (size_t) dp + d];
        __syncthreads();
        const float ax = q_xyz[qi * xyz_stride_floats], ay = q_xyz[qi * xyz_stride_floats + 1], az = q_xyz[qi * xyz_stride_floats + 2];
        float ld[KMAX], ls[KMAX];
        int li[KMAX];
#pragma unroll
        for (int m = 0; m < KMAX; ++m) { ld[m] = INFINITY; ls[m] = INFINITY; li[m] = INT_MAX; }
        for (size_t j = tid; j < nt; j += kExactThreads) {
            const float *b = t_xyz + j * xyz_stride_floats;
            const float dx = __fsub_rn(ax, b[0]), dy = __fsub_rn(ay, b[1]), dz = __fsub_rn(az, b[2]);
            const float s = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
            if (!(s < r2) || !t_valid[j]) continue;
            float cd = __fsqrt_rn(seq_sqdist(sq, t_f32 + j * (size_t) dp, dp));
            float cs = s;
            int ci = (int) j;
            if (lex3_less(cd, cs, ci, ld[KMAX - 1], ls[KMAX - 1], li[KMAX - 1])) {
#pragma unroll
                for (int m = 0; m < KMAX; ++m) {
                    if (lex3_less(cd, cs, ci, ld[m], ls[m], li[m])) {
                        float td = ld[m], tsp = ls[m]; int ti = li[m];
                        ld[m] = cd; ls[m] = cs; li[m] = ci;
                        cd = td; cs = tsp; ci = ti;
                    }
                }
            }
        }
        int head = 0, found = 0;
        for (int round = 0; round < k; ++round) {
            float hd = INFINITY, hs = INFINITY;
            int hi = INT_MAX;
#pragma unroll
            for (int m = 0; m < KMAX; ++m)
                if (m == head) { hd = ld[m]; hs = ls[m]; hi = li[m]; }
            float bd = hd, bs = hs;
            int bi = hi, bt = tid;
            for (int o = 16; o > 0; o >>= 1) {
                float od2 = __shfl_xor_sync(0xffffffffu, bd, o);
                float os2 = __shfl_xor_sync(0xffffffffu, bs, o);
                int oi2 = __shfl_xor_sync(0xffffffffu, bi, o);
                int ot2 = __shfl_xor_sync(0xffffffffu, bt, o);
                if (lex3_less(od2, os2, oi2, bd, bs, bi)) { bd = od2; bs = os2; bi = oi2; bt = ot2; }
            }
            if (lane == 0) { red_d[warp] = bd; red_s[warp] = bs; red_i[warp] = bi; red_w[warp] = bt; }
            __syncthreads();
            if (tid == 0) {
                float wd = red_d[0], ws = red_s[0];
                int wi = red_i[0], wt = red_w[0];
                for (int w = 1; w < kExactThreads / 32; ++w)
                    if (lex3_less(red_d[w], red_s[w], red_i[w], wd, ws, wi)) { wd = red_d[w]; ws = red_s[w]; wi = red_i[w]; wt = red_w[w]; }
                win_d = wd; win_s = ws; win_i = wi; win_t = wt;
            }
            __syncthreads();
            if (win_i == INT_MAX) break;
            if (tid == win_t) head++;
            if (tid == 0) { oi[round] = (int32_t) (win_i + t_off); od[round] = win_d; }
            found = round + 1;
            __syncthreads();
        }
        if (tid >= found && tid < k) { oi[tid] = -1; od[tid] = 0.f; }
        if (tid == 0) count[qi] = found;
    }
}

// ---- exact rows, split over the whole grid (a FEW flagged rows) -------------------------------
// The one-CTA-per-row kernel above streams the entire train set through a single SM per row -- 700 MB at 15 GB/s for
// SHOT-352 x 500k, tens of milliseconds for one overflowed row.  Here every CTA scans its slice of the train set for
// every flagged row and leaves a sorted partial k-list; the CTA that finishes a row last merges the partials.
constexpr int kSplitMaxRows = 256;

template <int KMAX>
__device__ __forceinline__ void block_select(float (&ld)[KMAX], int (&li)[KMAX], int k, float *red_d, int *red_i, int *red_w,
                                             float *win_d, int *win_i, int *win_t, float *out_d, int *out_i, int *found_out) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int head = 0, found = 0;
    for (int round = 0; round < k; ++round) {
        float hd = INFINITY;
        int hi = INT_MAX;
#pragma unroll
        for (int m = 0; m < KMAX; ++m)
            if (m == head) { hd = ld[m]; hi = li[m]; }
        float bd = hd;
        int bi = hi, bt = tid;
        for (int o = 16; o > 0; o >>= 1) {
            float od2 = __shfl_xor_sync(0xffffffffu, bd, o);
            int oi2 = __shfl_xor_sync(0xffffffffu, bi, o);
            int ot2 = __shfl_xor_sync(0xffffffffu, bt, o);
            if (lex_less(od2, oi2, bd, bi)) { bd = od2; bi = oi2; bt = ot2; }
        }
        if (lane == 0) { red_d[warp] = bd; red_i[warp] = bi; red_w[warp] = bt; }
        __syncthreads();
        if (tid == 0) {
            float wd = red_d[0];
            int wi = red_i[0], wt = red_w[0];
            for (int w = 1; w < kExactThreads / 32; ++w)
                if (lex_less(red_d[w], red_i[w], wd, wi)) { wd = red_d[w]; wi = red_i[w]; wt = red_w[w]; }
            *win_d = wd; *win_i = wi; *win_t = wt;
        }
        __syncthreads();
        if (*win_i == INT_MAX) break;
        if (tid == *win_t) head++;
        if (tid == 0) { out_i[round] = *win_i; out_d[round] = *win_d; }
        found = round + 1;
        __syncthreads();
    }
    *found_out = found;
}

template <int KMAX>
__global__ void __launch_bounds__(kExactThreads)
exact_rows_split_kernel(const float *__restrict__ q_f32, int dp, const float *__restrict__ t_f32,
                        const uint8_t *__restrict__ t_valid, size_t nt, long long t_off, size_t row_begin,
                        const int32_t *__restrict__ row_list, const int32_t *__restrict__ row_list_count, int k,
                        int32_t *__restrict__ part_i, float *__restrict__ part_d, unsigned int *__restrict__ done,
                        int32_t *__restrict__ idx, float *__restrict__ dist, int32_t *__restrict__ count,
                        const int32_t *__restrict__ row_map, const int2 *__restrict__ seg_range) {
    extern __shared__ float smem[];
    float *sq = smem;
    float *red_d = smem + dp;
    int *red_i = reinterpret_cast<int *>(red_d + kExactThreads / 32);
    int *red_w = red_i + kExactThreads / 32;
    __shared__ float win_d;
    __shared__ int win_i, win_t, is_last;
    const int total = *row_list_count;
    if (total <= 0 || total > kSplitMaxRows) return;   // many flagged rows: the one-CTA-per-row kernel takes them
    const int tid = threadIdx.x;
    const int S = (int) gridDim.x;
    for (int r = 0; r < total; ++r) {
        const size_t local = (size_t) row_list[r];
        const size_t qi = row_map ? (size_t) row_map[local] : row_begin + local;
        const size_t orow = qi - row_begin;
        size_t a = 0, b = nt;   // batch calls: the train rows of the query's own pair, sliced over the grid
        if (seg_range) {
            const int2 sr = seg_range[qi / B200M_TILE_N];
            a = (size_t) sr.x;
            b = (size_t) sr.y;
        }
        const size_t chunk = (b - a + S - 1) / S;
        const size_t j0 = a + (size_t) blockIdx.x * chunk, j1 = j0 + chunk < b ? j0 + chunk : b;
        __syncthreads();
        for (int d = tid; d < dp; d += kExactThreads) sq[d] = q_f32[qi * (size_t) dp + d];
        __syncthreads();
        float ld[KMAX];
        int li[KMAX];
#pragma unroll
        for (int m = 0; m < KMAX; ++m) { ld[m] = INFINITY; li[m] = INT_MAX; }
        for (size_t j = j0 + tid; j < j1; j += kExactThreads) {
            if (!t_valid[j]) continue;
            float d = __fsqrt_rn(seq_sqdist(sq, t_f32 + j * (size_t) dp, dp));
            if (lex_less(d, (int) j, ld[KMAX - 1], li[KMAX - 1])) {
                float cd = d;
                int ci = (int) j;
#pragma unroll
                for (int m = 0; m < KMAX; ++m) {
                    if (lex_less(cd, ci, ld[m], li[m])) {
                        float td = ld[m]; int ti = li[m];
                        ld[m] = cd; li[m] = ci;
                        cd = td; ci = ti;
                    }
                }
            }
        }
        int32_t *pi = part_i + ((size_t) r * S + blockIdx.x) * k;
        float *pd = part_d + ((size_t) r * S + blockIdx.x) * k;
        int found = 0;
        block_select<KMAX>(ld, li, k, red_d, red_i, red_w, &win_d, &win_i, &win_t, pd, pi, &found);
        if (tid >= found && tid < k) { pi[tid] = INT_MAX; pd[tid] = INFINITY; }
        __threadfence();
        __syncthreads();
        if (tid == 0) is_last = atomicAdd(&done[r], 1u) == (unsigned) (S - 1);
        __syncthreads();
        if (!is_last) continue;
        __threadfence();
        // merge: S sorted partial lists of k entries; every thread folds a strided share into its own sorted list
#pragma unroll
        for (int m = 0; m < KMAX; ++m) { ld[m] = INFINITY; li[m] = INT_MAX; }
        const int n_part = S * k;
        const volatile int32_t *vi = part_i + (size_t) r * S * k;
        const volatile float *vd = part_d + (size_t) r * S * k;
        for (int e = tid; e < n_part; e += kExactThreads) {
            float cd = vd[e];
            int ci = vi[e];
            if (ci == INT_MAX) continue;
            if (lex_less(cd, ci, ld[KMAX - 1], li[KMAX - 1])) {
#pragma unroll
                for (int m = 0; m < KMAX; ++m) {
                    if (lex_less(cd, ci, ld[m], li[m])) {
                        float td = ld[m]; int ti = li[m];
                        ld[m] = cd; li[m] = ci;
                        cd = td; ci = ti;
                    }
                }
            }
        }
        __shared__ float fin_d[B200M_MAX_K];
        __shared__ int fin_i[B200M_MAX_K];
        block_select<KMAX>(ld, li, k, red_d, red_i, red_w, &win_d, &win_i, &win_t, fin_d, fin_i, &found);
        __syncthreads();
        int32_t *oi = idx + orow * k;
        float *od = dist + orow * k;
        if (tid < k) {
            oi[tid] = tid < found ? (int32_t) (fin_i[tid] + t_off) : -1;
            od[tid] = tid < found ? fin_d[tid] : 0.f;
        }
        if (tid == 0) { count[orow] = found; done[r] = 0u; }   // counter ready for the next call
    }
}

// ---- re-rank -----------------------------------------------------------------
// One warp per query row (persistent warps, grid-stride over rows).  The row's candidates are taken 32 at a time:
// lane c owns candidate c.  Every lane issues ONE bulk asynchronous copy (cp.async.bulk, the TMA engine's 1-D form)
// of its candidate's whole FP32 row from HBM into the warp's shared-memory slab, all of them -- and the query row
// -- completing on the warp's mbarrier, so a warp has its entire gather (up to 32 rows, 45 KB for SHOT-352) in
// flight at once instead of a load/store round trip per 128 bytes.  Each lane then runs the reference's sequential
// FP32 chain over its own slab row with 128-bit shared loads; the slab pitch is an odd number of 16-byte units, so
// the 32 lanes' loads are bank-conflict free.
constexpr int kMaxLists = 32;   // train splits x epilogue column halves

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void bar_wait_parity(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}

// bytes between consecutive slab rows: the row itself, padded so that (pitch / 16) is odd
__host__ __device__ inline int rerank_pitch_bytes(int dp) { return (dp / 4) % 2 ? dp * 4 : dp * 4 + 16; }
// Slab rows per warp.  Short rows: one per lane.  Long rows (RoPS, SHOT): 8 -- the live candidates of a row (after
// pruning, typically k plus a few) are compacted into the slab, a full slab of 32 x 1.4 KB would leave room for only four
// warps per SM, and this kernel lives on the number of gathers in flight, not on lanes.  Rows over 4 KB (USC-1960: a
// 7856-byte pitch) keep 8 too: 3 warps x 8 slots hold 24 of the 27 rows that fit in 220 KB with one query row per warp,
// and no other slot count holds more (4: 5 x 4 = 20, 6: 4 x 6 = 24, 12: 2 x 12 = 24).
__host__ __device__ inline int rerank_slots(int dp) { return rerank_pitch_bytes(dp) <= 256 ? 32 : 8; }
__host__ __device__ inline size_t rerank_warp_bytes(int dp) { return (size_t) (rerank_slots(dp) + 1) * rerank_pitch_bytes(dp); }   // + the query

// Row metadata travels through a three-deep software pipeline so that no warp ever waits on a dependent chain of
// global loads: the list lengths of row r+2 and the candidate indices of row r+1 are in flight while row r's slab is
// being filled and consumed.
struct RerankLens {   // stage 1: issued two rows ahead
    int len;          // lanes 0..n_lists-1: appended entries of list `lane` (may exceed cap: overflow)
    int qv;           // q_valid of the row (rows of a row map are valid by construction)
    long long qi;     // original row number of the query
    float thr;        // lanes 0..n_lists-1: final append threshold of list `lane` (+inf when values were not recorded)
};
struct RerankRow {    // stage 2: issued one row ahead
    int total;        // candidates over all lists (capped lists)
    int my_len;       // capped length of list `lane`
    int j0;           // candidate of this lane in the first group of 32 (-1: none or pruned); range-checked, validity not yet
    float thr;        // pruning threshold of the row
    long long qi;     // original row number of the query
    bool overflow, qv;
};

__device__ __forceinline__ RerankLens rerank_fetch_lens(size_t local, size_t n_rows, size_t row_begin,
                                                        const int32_t *__restrict__ cand_cnt,
                                                        const float *__restrict__ cand_thr,
                                                        const uint8_t *__restrict__ q_valid, int n_lists, int lane,
                                                        const int32_t *__restrict__ row_map) {
    RerankLens m;
    m.len = 0;
    m.qv = 0;
    m.qi = 0;
    m.thr = INFINITY;
    if (local < n_rows) {
        if (lane < n_lists) {
            m.len = __ldg(cand_cnt + (size_t) lane * n_rows + local);
            if (cand_thr) m.thr = __ldg(cand_thr + (size_t) lane * n_rows + local);
        }
        if (row_map) {
            m.qi = (long long) __ldg(row_map + local);
            m.qv = 1;
        } else {
            m.qi = (long long) (row_begin + local);
            m.qv = q_valid[row_begin + local];
        }
    }
    return m;
}

// position `c` of the concatenated (capped) lists -> (list, offset); warp-uniform walk, every lane takes part
__device__ __forceinline__ void rerank_locate(int c, int my_len, int n_lists, int &l_sel, int &c_sel) {
    bool placed = false;
    l_sel = 0;
    c_sel = c;
    for (int l = 0; l < n_lists; ++l) {
        const int cl = __shfl_sync(0xffffffffu, my_len, l);
        if (!placed) {
            if (c_sel < cl) { placed = true; l_sel = l; }
            else c_sel -= cl;
        }
    }
}

// Every list's final threshold bounds the accumulator of every exact top-k member (DESIGN.md "Certified
// candidates"), so an entry whose recorded value is not under the smallest of them cannot be one.
__device__ __forceinline__ float rerank_row_thr(const RerankLens &m) {
    float t = m.thr;
    for (int o = 16; o > 0; o >>= 1) t = fminf(t, __shfl_xor_sync(0xffffffffu, t, o));
    return t;
}

__device__ __forceinline__ RerankRow rerank_fetch_row(const RerankLens &m, size_t local, size_t n_rows,
                                                      const int32_t *__restrict__ cand_idx,
                                                      const float *__restrict__ cand_val, int n_lists, int cap, size_t nt,
                                                      int lane) {
    RerankRow r;
    r.qv = m.qv != 0;
    r.qi = m.qi;
    r.overflow = __any_sync(0xffffffffu, m.len > cap);
    r.my_len = m.len > cap ? cap : m.len;
    int t = r.my_len;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    r.total = t;
    int l_sel, c_sel;
    rerank_locate(lane, r.my_len, n_lists, l_sel, c_sel);
    r.j0 = -1;
    r.thr = rerank_row_thr(m);
    if (local < n_rows && r.qv && !r.overflow && lane < r.total) {
        const size_t e = ((size_t) l_sel * n_rows + local) * cap + c_sel;
        const int j = __ldg(cand_idx + e);
        const bool keep = cand_val ? __ldg(cand_val + e) < r.thr : true;
        r.j0 = (j < 0 || (size_t) j >= nt || !keep) ? -1 : j;
    }
    return r;
}

template <int KMAX>
__global__ void __launch_bounds__(512)
rerank_kernel(const float *__restrict__ q_f32, const uint8_t *__restrict__ q_valid, int dp, int dim,
              const float *__restrict__ t_f32, const uint8_t *__restrict__ t_valid, size_t nt, long long t_off,
              size_t row_begin, size_t n_rows, int k,
              const int32_t *__restrict__ cand_idx, const int32_t *__restrict__ cand_cnt, int n_lists, int cap,
              const float *__restrict__ cand_val, const float *__restrict__ cand_thr,
              int32_t *__restrict__ idx, float *__restrict__ dist, int32_t *__restrict__ count,
              int32_t *__restrict__ flag_rows, int32_t *__restrict__ counters, const int32_t *__restrict__ row_map) {
    extern __shared__ __align__(128) uint8_t rr_smem[];
    __shared__ unsigned long long blk_cands;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int pitch = rerank_pitch_bytes(dp);
    const uint32_t row_bytes = (uint32_t) dp * 4u;
    // per-warp slab: [32 candidate rows][pitch] then the query row; the warps' mbarriers sit behind all slabs
    uint8_t *slab = rr_smem + (size_t) warp * rerank_warp_bytes(dp);
    const uint32_t slab_u = smem_addr(slab);
    const int G = rerank_slots(dp);
    const uint32_t sq_u = slab_u + (uint32_t) G * (uint32_t) pitch;
    const float4 *sq4 = reinterpret_cast<const float4 *>(slab + (size_t) G * pitch);
    const uint32_t bar = smem_addr(rr_smem + (size_t) n_warps * rerank_warp_bytes(dp)) + 8u * (uint32_t) warp;
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x == 0) blk_cands = 0ull;
    __syncthreads();
    uint32_t phase = 0;
    unsigned long long my_cands = 0ull;
    const size_t stride = (size_t) gridDim.x * n_warps;
    size_t local = (size_t) blockIdx.x * n_warps + warp;
    // pipeline prologue
    RerankRow cur = rerank_fetch_row(rerank_fetch_lens(local, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map), local,
                                     n_rows, cand_idx, cand_val, n_lists, cap, nt, lane);
    RerankLens nxt_lens = rerank_fetch_lens(local + stride, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map);
    for (; local < n_rows; local += stride) {
        // `local` numbers the rows of this call (and its candidate lists); results are stored by original row
        const size_t qi = (size_t) cur.qi;
        const size_t orow = qi - row_begin;
        int32_t *oi = idx + orow * k;
        float *od = dist + orow * k;
        const bool work = cur.qv && !cur.overflow;
        float ld[KMAX];
        int li[KMAX];
#pragma unroll
        for (int m = 0; m < KMAX; ++m) { ld[m] = INFINITY; li[m] = INT_MAX; }
        bool first = true;   // the query row rides with the first pass that gathers anything
        RerankRow nxt;
        if (!work || cur.total == 0) {
            nxt = rerank_fetch_row(nxt_lens, local + stride, n_rows, cand_idx, cand_val, n_lists, cap, nt, lane);
            nxt_lens = rerank_fetch_lens(local + 2 * stride, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map);
        } else {
            for (int base = 0; base < cur.total; base += 32) {
                int j = cur.j0;
                if (base > 0) {   // list positions beyond the first 32 (rare): fetched on the spot
                    int l_sel, c_sel;
                    rerank_locate(base + lane, cur.my_len, n_lists, l_sel, c_sel);
                    j = -1;
                    if (base + lane < cur.total) {
                        const size_t e = ((size_t) l_sel * n_rows + local) * cap + c_sel;
                        j = cand_idx[e];
                        if (j < 0 || (size_t) j >= nt || (cand_val && !(cand_val[e] < cur.thr))) j = -1;
                    }
                }
                // live candidates, compacted: the n-th live lane uses slab row n (mod G), G at a time
                const unsigned live = __ballot_sync(0xffffffffu, j >= 0);
                const int n_live = __popc(live);
                const int slot = __popc(live & ((1u << lane) - 1u));
                my_cands += (unsigned long long) n_live;   // train rows evaluated exactly (entries the final threshold pruned are not)
                for (int p0 = 0; p0 < n_live; p0 += G) {
                    const bool mine = j >= 0 && slot >= p0 && slot < p0 + G;
                    // earlier (generic-proxy) reads of the slab are ordered before the asynchronous writes that follow
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    if (lane == 0) {
                        const int n_pass = n_live - p0 < G ? n_live - p0 : G;
                        const uint32_t tx = (uint32_t) (n_pass + (first ? 1 : 0)) * row_bytes;
                        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tx) : "memory");
                        if (first) bulk_g2s(sq_u, q_f32 + qi * (size_t) dp, row_bytes, bar);
                    }
                    __syncwarp();   // the expectation is posted before any copy can complete
                    const float4 *my4 = reinterpret_cast<const float4 *>(slab + (size_t) (slot - p0) * pitch);
                    if (mine) bulk_g2s(slab_u + (uint32_t) (slot - p0) * (uint32_t) pitch, t_f32 + (size_t) j * dp, row_bytes, bar);
                    if (first) {
                        // metadata of the rows behind this one: their loads land while this row's slab fills
                        nxt = rerank_fetch_row(nxt_lens, local + stride, n_rows, cand_idx, cand_val, n_lists, cap, nt, lane);
                        nxt_lens = rerank_fetch_lens(local + 2 * stride, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map);
                        first = false;
                    }
                    bar_wait_parity(bar, phase);
                    phase ^= 1u;
                    if (mine) {
                        float s = 0.f;
#pragma unroll 4
                        for (int d4 = 0; d4 < dp / 4; ++d4) {
                            const float4 a = sq4[d4], b = my4[d4];
                            float df = __fsub_rn(a.x, b.x);
                            s = __fadd_rn(s, __fmul_rn(df, df));
                            df = __fsub_rn(a.y, b.y);
                            s = __fadd_rn(s, __fmul_rn(df, df));
                            df = __fsub_rn(a.z, b.z);
                            s = __fadd_rn(s, __fmul_rn(df, df));
                            df = __fsub_rn(a.w, b.w);
                            s = __fadd_rn(s, __fmul_rn(df, df));
                        }
                        float cd = __fsqrt_rn(s);
                        int ci = j;
                        // invalid (non-finite) train rows are never candidates (reference :661); only such a row -- or an
                        // overflowing sum -- can give a non-finite distance, so validity is looked up on that path alone
                        const bool ok = cd < INFINITY || t_valid[j] != 0;
                        if (ok && lex_less(cd, ci, ld[KMAX - 1], li[KMAX - 1])) {
#pragma unroll
                            for (int m = 0; m < KMAX; ++m) {
                                if (lex_less(cd, ci, ld[m], li[m])) {
                                    float td = ld[m]; int ti = li[m];
                                    ld[m] = cd; li[m] = ci;
                                    cd = td; ci = ti;
                                }
                            }
                        }
                    }
                    __syncwarp();
                }
            }
            if (first) {   // every candidate was pruned or invalid: nothing was gathered
                nxt = rerank_fetch_row(nxt_lens, local + stride, n_rows, cand_idx, cand_val, n_lists, cap, nt, lane);
                nxt_lens = rerank_fetch_lens(local + 2 * stride, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map);
            }
        }
        // k rounds of warp arg-min over the per-lane list heads
        int head = 0, found = 0;
        if (work) {
            for (int round = 0; round < k; ++round) {
                float hd = INFINITY;
                int hi = INT_MAX;
#pragma unroll
                for (int m = 0; m < KMAX; ++m)
                    if (m == head) { hd = ld[m]; hi = li[m]; }
                float wd = hd;
                int wi = hi;
                for (int o = 16; o > 0; o >>= 1) {
                    float od2 = __shfl_xor_sync(0xffffffffu, wd, o);
                    int oi2 = __shfl_xor_sync(0xffffffffu, wi, o);
                    if (lex_less(od2, oi2, wd, wi)) { wd = od2; wi = oi2; }
                }
                if (wi == INT_MAX) break;
                if (hi == wi) head++;   // candidate indices are unique per row
                if (lane == 0) { oi[round] = (int32_t) (wi + t_off); od[round] = wd; }
                found = round + 1;
            }
        }
        // a non-finite query has an empty entry (reference include/matching.h:576); overflowed rows are redone exactly
        for (int m = found + lane; m < k; m += 32) { oi[m] = -1; od[m] = 0.f; }
        if (lane == 0) {
            count[orow] = found;
            if (cur.qv && cur.overflow) {
                int pos = atomicAdd(counters, 1);
                flag_rows[pos] = (int32_t) local;
            }
        }
        cur = nxt;
    }
    if (lane == 0 && my_cands) atomicAdd(&blk_cands, my_cands);
    __syncthreads();
    if (threadIdx.x == 0 && blk_cands)
        atomicAdd(reinterpret_cast<unsigned long long *>(counters + 2), blk_cands);
}

// ---- re-rank over CHUNK entries (candidate kernel EPI = 4 / 5) ---------------------------------------------------------
// A list entry names 32 consecutive train rows (a chunk of the candidate kernel's columns) and carries the chunk's smallest
// accumulator.  Entries whose minimum is not under the row's final threshold are dropped (DESIGN.md section 4: no exact top-k
// member lives in such a chunk) -- of the ~k ln(N/k) entries of a row about k + margin survive, scattered over the lists, so
// the survivors of ALL list positions are first compacted into a small per-warp array and then fetched G chunks per pass:
// every chunk by ONE bulk copy (32 contiguous FP32 rows, 4.6 KB for FPFH-33), lane l runs the reference's sequential FP32
// chain over row l of every chunk of the pass -- up to four chains per lane in flight.  Same per-lane sorted lists and warp
// arg-min as rerank_kernel; same metadata pipeline for the first 32 list positions, the rest are loaded four groups at a time.
constexpr int kChunkRows = 32;
constexpr int kChunkPassMax = 4;
constexpr int kChunkPassBytes = 9216;   // slab bytes per warp and pass: two FPFH-33 chunks, so that sixteen warps fit an SM
constexpr int kSurvCap = 64;
inline int chunk_pass(int dp) {
    static const int forced = getenv("B200M_CHUNK_PASS") ? atoi(getenv("B200M_CHUNK_PASS")) : 0;   // tuning override: 1..4
    const int g = forced > 0 ? forced : kChunkPassBytes / (kChunkRows * dp * 4);
    return g < 1 ? 1 : g > kChunkPassMax ? kChunkPassMax : g;
}
// slab of G chunks + the query row + the survivor array
__host__ __device__ inline size_t chunk_warp_bytes(int dp, int G) { return (size_t) (G * kChunkRows + 1) * dp * 4 + kSurvCap * 4; }

template <int KMAX>
__global__ void __launch_bounds__(512)
rerank_chunks_kernel(const float *__restrict__ q_f32, const uint8_t *__restrict__ q_valid, int dp, int dim,
                     const float *__restrict__ t_f32, const uint8_t *__restrict__ t_valid, size_t nt, long long t_off,
                     size_t row_begin, size_t n_rows, int k,
                     const int32_t *__restrict__ cand_idx, const int32_t *__restrict__ cand_cnt, int n_lists, int cap,
                     const float *__restrict__ cand_val, const float *__restrict__ cand_thr,
                     int32_t *__restrict__ idx, float *__restrict__ dist, int32_t *__restrict__ count,
                     int32_t *__restrict__ flag_rows, int32_t *__restrict__ counters, const int32_t *__restrict__ row_map,
                     int G /* chunks per pass */) {
    extern __shared__ __align__(128) uint8_t rr_smem[];
    __shared__ unsigned long long blk_cands;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const uint32_t row_bytes = (uint32_t) dp * 4u;
    const uint32_t chunk_bytes = (uint32_t) kChunkRows * row_bytes;
    // per-warp: [G chunks][32 rows][dp], the query row, the survivors' first train rows; the warps' mbarriers sit behind all of it
    uint8_t *slab = rr_smem + (size_t) warp * chunk_warp_bytes(dp, G);
    const uint32_t slab_u = smem_addr(slab);
    const uint32_t sq_u = slab_u + (uint32_t) G * chunk_bytes;
    const float4 *sq4 = reinterpret_cast<const float4 *>(slab + (size_t) G * chunk_bytes);
    volatile int *surv = reinterpret_cast<volatile int *>(slab + (size_t) G * chunk_bytes + row_bytes);
    const float4 *my4 = reinterpret_cast<const float4 *>(slab + (size_t) lane * row_bytes);   // row `lane` of chunk 0
    const int chunk4 = (int) (chunk_bytes / 16u);
    const uint32_t bar = smem_addr(rr_smem + (size_t) n_warps * chunk_warp_bytes(dp, G)) + 8u * (uint32_t) warp;
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x == 0) blk_cands = 0ull;
    __syncthreads();
    uint32_t phase = 0;
    unsigned long long my_cands = 0ull;
    const size_t stride = (size_t) gridDim.x * n_warps;
    size_t local = (size_t) blockIdx.x * n_warps + warp;
    RerankRow cur = rerank_fetch_row(rerank_fetch_lens(local, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map), local,
                                     n_rows, cand_idx, cand_val, n_lists, cap, nt, lane);
    RerankLens nxt_lens = rerank_fetch_lens(local + stride, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map);
    for (; local < n_rows; local += stride) {
        const size_t qi = (size_t) cur.qi;
        const size_t orow = qi - row_begin;
        int32_t *oi = idx + orow * k;
        float *od = dist + orow * k;
        const bool work = cur.qv && !cur.overflow;
        float ld[KMAX];
        int li[KMAX];
#pragma unroll
        for (int m = 0; m < KMAX; ++m) { ld[m] = INFINITY; li[m] = INT_MAX; }
        bool first = true;   // the query row rides with the first pass that gathers anything
        RerankRow nxt;
        // exact distances of the rows of the compacted survivors surv[0 .. n_surv)
        auto gather = [&](int n_surv) {
            __syncwarp();   // surv[] written
            my_cands += (unsigned long long) n_surv * kChunkRows;   // train rows evaluated exactly
            for (int p0 = 0; p0 < n_surv; p0 += G) {
                const int n_pass = n_surv - p0 < G ? n_surv - p0 : G;
                const bool mine = lane < n_pass;
                const int j = mine ? surv[p0 + lane] : 0;
                const unsigned my_rows = mine ? (nt - (size_t) j < (size_t) kChunkRows ? (unsigned) (nt - (size_t) j) : (unsigned) kChunkRows) : 0u;
                const unsigned pass_rows = __reduce_add_sync(0xffffffffu, my_rows);
                // earlier (generic-proxy) reads of the slab are ordered before the asynchronous writes that follow
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                if (lane == 0) {
                    const uint32_t tx = (pass_rows + (first ? 1u : 0u)) * row_bytes;
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tx) : "memory");
                    if (first) bulk_g2s(sq_u, q_f32 + qi * (size_t) dp, row_bytes, bar);
                }
                __syncwarp();   // the expectation is posted before any copy can complete
                if (mine) bulk_g2s(slab_u + (uint32_t) lane * chunk_bytes, t_f32 + (size_t) j * dp, my_rows * row_bytes, bar);
                if (first) {
                    // metadata of the rows behind this one: their loads land while this row's slab fills
                    nxt = rerank_fetch_row(nxt_lens, local + stride, n_rows, cand_idx, cand_val, n_lists, cap, nt, lane);
                    nxt_lens = rerank_fetch_lens(local + 2 * stride, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map);
                    first = false;
                }
                int cj[kChunkPassMax];   // first train row of every chunk of the pass
#pragma unroll
                for (int i = 0; i < kChunkPassMax; ++i) cj[i] = i < n_pass ? surv[p0 + i] : -1;
                bar_wait_parity(bar, phase);
                phase ^= 1u;
                float s[kChunkPassMax];
#pragma unroll
                for (int i = 0; i < kChunkPassMax; ++i) s[i] = 0.f;
#pragma unroll 2
                for (int d4 = 0; d4 < dp / 4; ++d4) {
                    const float4 a = sq4[d4];
#pragma unroll
                    for (int i = 0; i < kChunkPassMax; ++i) {
                        if (i < n_pass) {   // warp-uniform
                            const float4 b = my4[i * chunk4 + d4];
                            float df = __fsub_rn(a.x, b.x);
                            s[i] = __fadd_rn(s[i], __fmul_rn(df, df));
                            df = __fsub_rn(a.y, b.y);
                            s[i] = __fadd_rn(s[i], __fmul_rn(df, df));
                            df = __fsub_rn(a.z, b.z);
                            s[i] = __fadd_rn(s[i], __fmul_rn(df, df));
                            df = __fsub_rn(a.w, b.w);
                            s[i] = __fadd_rn(s[i], __fmul_rn(df, df));
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < kChunkPassMax; ++i) {
                    if (i < n_pass && (size_t) (cj[i] + lane) < nt) {
                        float cd = __fsqrt_rn(s[i]);
                        int ci = cj[i] + lane;
                        // invalid (non-finite) train rows are never candidates (reference :661); only such a row -- or an
                        // overflowing sum -- can give a non-finite distance, so validity is looked up on that path alone
                        const bool ok = cd < INFINITY || t_valid[ci] != 0;
                        if (ok && lex_less(cd, ci, ld[KMAX - 1], li[KMAX - 1])) {
#pragma unroll
                            for (int m = 0; m < KMAX; ++m) {
                                if (lex_less(cd, ci, ld[m], li[m])) {
                                    float td = ld[m]; int ti = li[m];
                                    ld[m] = cd; li[m] = ci;
                                    cd = td; ci = ti;
                                }
                            }
                        }
                    }
                }
                __syncwarp();   // slab and surv[] reads done before the next pass / the next compaction
            }
        };
        if (work && cur.total > 0) {
            int n_surv = 0;
            const int n_groups = (cur.total + 31) >> 5;
            for (int g0 = 0; g0 < n_groups; g0 += 4) {
                // the entries of up to four groups of 32 list positions: all loads in flight before the first is looked at
                int jg[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int g = g0 + u;
                    jg[u] = -1;
                    if (g == 0) jg[u] = cur.j0;   // came with the metadata pipeline
                    else if (g < n_groups) {
                        int l_sel, c_sel;
                        rerank_locate(g * 32 + lane, cur.my_len, n_lists, l_sel, c_sel);
                        if (g * 32 + lane < cur.total) {
                            const size_t e = ((size_t) l_sel * n_rows + local) * cap + c_sel;
                            const int j = cand_idx[e];
                            const float v = cand_val[e];
                            jg[u] = (j < 0 || (size_t) j >= nt || !(v < cur.thr)) ? -1 : j;
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (g0 + u < n_groups) {
                        const unsigned live = __ballot_sync(0xffffffffu, jg[u] >= 0);
                        const int n = __popc(live);
                        if (n_surv + n > kSurvCap) {
                            gather(n_surv);
                            n_surv = 0;
                        }
                        if (jg[u] >= 0) surv[n_surv + __popc(live & ((1u << lane) - 1u))] = jg[u];
                        n_surv += n;
                    }
                }
            }
            gather(n_surv);
        }
        if (first) {   // nothing was gathered for this row
            nxt = rerank_fetch_row(nxt_lens, local + stride, n_rows, cand_idx, cand_val, n_lists, cap, nt, lane);
            nxt_lens = rerank_fetch_lens(local + 2 * stride, n_rows, row_begin, cand_cnt, cand_thr, q_valid, n_lists, lane, row_map);
        }
        // k rounds of warp arg-min over the per-lane list heads
        int head = 0, found = 0;
        if (work) {
            for (int round = 0; round < k; ++round) {
                float hd = INFINITY;
                int hi = INT_MAX;
#pragma unroll
                for (int m = 0; m < KMAX; ++m)
                    if (m == head) { hd = ld[m]; hi = li[m]; }
                float wd = hd;
                int wi = hi;
                for (int o = 16; o > 0; o >>= 1) {
                    float od2 = __shfl_xor_sync(0xffffffffu, wd, o);
                    int oi2 = __shfl_xor_sync(0xffffffffu, wi, o);
                    if (lex_less(od2, oi2, wd, wi)) { wd = od2; wi = oi2; }
                }
                if (wi == INT_MAX) break;
                if (hi == wi) head++;   // a train row is evaluated once per query row (chunks are disjoint)
                if (lane == 0) { oi[round] = (int32_t) (wi + t_off); od[round] = wd; }
                found = round + 1;
            }
        }
        for (int m = found + lane; m < k; m += 32) { oi[m] = -1; od[m] = 0.f; }
        if (lane == 0) {
            count[orow] = found;
            if (cur.qv && cur.overflow) {
                int pos = atomicAdd(counters, 1);
                flag_rows[pos] = (int32_t) local;
            }
        }
        cur = nxt;
    }
    if (lane == 0 && my_cands) atomicAdd(&blk_cands, my_cands);
    __syncthreads();
    if (threadIdx.x == 0 && blk_cands)
        atomicAdd(reinterpret_cast<unsigned long long *>(counters + 2), blk_cands);
}

template <int KMAX>
cudaError_t launch_exact_t(const float *q_f32, const uint8_t *q_valid, int dp, int dim, const float *t_f32,
                           const uint8_t *t_valid, size_t nt, int64_t t_off, size_t row_begin, size_t n_rows,
                           const int32_t *row_list, const int32_t *row_list_count, int k, int32_t *idx, float *dist,
                           int32_t *count, int blocks, int split_blocks, int32_t *part_i, float *part_d,
                           unsigned int *done, const int32_t *row_map, cudaStream_t st, const int2 *seg_range) {
    size_t smem = sizeof(float) * dp + (sizeof(float) + 2 * sizeof(int)) * (kExactThreads / 32);
    const bool split = row_list && split_blocks > 0 && part_i && part_d && done;
    if (split) {
        exact_rows_split_kernel<KMAX><<<split_blocks, kExactThreads, smem, st>>>(
            q_f32, dp, t_f32, t_valid, nt, (long long) t_off, row_begin, row_list, row_list_count, k, part_i, part_d, done,
            idx, dist, count, row_map, seg_range);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    exact_rows_kernel<KMAX><<<blocks, kExactThreads, smem, st>>>(q_f32, q_valid, dp, dim, t_f32, t_valid, nt,
                                                                 (long long) t_off, row_begin, n_rows, row_list,
                                                                 row_list_count, k, idx, dist, count,
                                                                 split ? kSplitMaxRows : 0, row_map, seg_range);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_exact_rows(const float *q_f32, const uint8_t *q_valid, int dp, int dim,
                              const float *t_f32, const uint8_t *t_valid, size_t nt, int64_t t_index_offset,
                              size_t row_begin, size_t n_rows, const int32_t *row_list, const int32_t *row_list_count,
                              int k, int32_t *idx, float *dist, int32_t *count, int max_blocks, int split_blocks,
                              int32_t *part_i, float *part_d, unsigned int *done, const int32_t *row_map, cudaStream_t st,
                              const int2 *seg_range) {
    if (n_rows == 0) return cudaSuccess;
    int blocks = (int) (n_rows < (size_t) max_blocks ? n_rows : (size_t) max_blocks);
#define B200M_EXACT_CASE(K)                                                                                   \
    return launch_exact_t<K>(q_f32, q_valid, dp, dim, t_f32, t_valid, nt, t_index_offset, row_begin, n_rows,  \
                             row_list, row_list_count, k, idx, dist, count, blocks, split_blocks, part_i, part_d, \
                             done, row_map, st, seg_range)
    if (k <= 1) B200M_EXACT_CASE(1);
    if (k <= 2) B200M_EXACT_CASE(2);
    if (k <= 4) B200M_EXACT_CASE(4);
    if (k <= 8) B200M_EXACT_CASE(8);
    if (k <= 16) B200M_EXACT_CASE(16);
    B200M_EXACT_CASE(32);
#undef B200M_EXACT_CASE
}

cudaError_t launch_local_rows(const float *q_f32, const uint8_t *q_valid, int dp, const float *t_f32,
                              const uint8_t *t_valid, size_t nt, int64_t t_index_offset, size_t n_rows,
                              const float *q_xyz, const float *t_xyz, size_t xyz_stride_bytes, float radius, int k,
                              int32_t *idx, float *dist, int32_t *count, int max_blocks, cudaStream_t st) {
    if (n_rows == 0) return cudaSuccess;
    const int blocks = (int) (n_rows < (size_t) max_blocks ? n_rows : (size_t) max_blocks);
    const size_t smem = sizeof(float) * dp + (2 * sizeof(float) + 2 * sizeof(int)) * (kExactThreads / 32);
    const float r2 = radius * radius;   // radiusSearch is handed radius * radius (FP32 product)
#define B200M_LOCAL_CASE(K)                                                                                            \
    do {                                                                                                               \
        local_rows_kernel<K><<<blocks, kExactThreads, smem, st>>>(q_f32, q_valid, dp, t_f32, t_valid, nt,              \
                                                                  (long long) t_index_offset, n_rows, q_xyz, t_xyz,    \
                                                                  xyz_stride_bytes / 4, r2, k, idx, dist, count);      \
        return cudaGetLastError();                                                                                     \
    } while (0)
    if (k <= 1) B200M_LOCAL_CASE(1);
    if (k <= 2) B200M_LOCAL_CASE(2);
    if (k <= 4) B200M_LOCAL_CASE(4);
    if (k <= 8) B200M_LOCAL_CASE(8);
    if (k <= 16) B200M_LOCAL_CASE(16);
    B200M_LOCAL_CASE(32);
#undef B200M_LOCAL_CASE
}

size_t exact_split_ws_entries(int split_blocks, int k) { return (size_t) kSplitMaxRows * (size_t) split_blocks * (size_t) k; }
int exact_split_max_rows() { return kSplitMaxRows; }

cudaError_t launch_rerank(const float *q_f32, const uint8_t *q_valid, int dp, int dim,
                          const float *t_f32, const uint8_t *t_valid, size_t nt, int64_t t_index_offset,
                          size_t row_begin, size_t n_rows, int k,
                          const int32_t *cand_idx, const int32_t *cand_cnt, int n_lists, int cap,
                          const float *cand_val, const float *cand_thr,
                          int32_t *idx, float *dist, int32_t *count,
                          int32_t *flag_rows, int32_t *counters, int sm_count, const int32_t *row_map, int chunk_entries,
                          cudaStream_t st) {
    if (n_rows == 0) return cudaSuccess;
    if (n_lists > kMaxLists) return cudaErrorInvalidValue;
    if (chunk_entries) {
        if (!cand_val || !cand_thr) return cudaErrorInvalidValue;
        const int G = chunk_pass(dp);
        const size_t per_warp = chunk_warp_bytes(dp, G) + 8;
        int warps = (int) ((220 * 1024) / per_warp);
        if (warps > 16) warps = 16;
        if (warps < 1) return cudaErrorInvalidValue;
        const size_t smem = (size_t) warps * per_warp;
        const size_t want = (n_rows + warps - 1) / warps;
        const unsigned blocks = (unsigned) (want < (size_t) sm_count ? want : (size_t) sm_count);
#define B200M_RERANK_CHUNK_CASE(K)                                                                              \
    do {                                                                                                        \
        cudaError_t e = cudaFuncSetAttribute(rerank_chunks_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                             (int) smem);                                                       \
        if (e != cudaSuccess) return e;                                                                         \
        rerank_chunks_kernel<K><<<blocks, warps * 32, smem, st>>>(                                              \
            q_f32, q_valid, dp, dim, t_f32, t_valid, nt, (long long) t_index_offset, row_begin, n_rows, k,      \
            cand_idx, cand_cnt, n_lists, cap, cand_val, cand_thr, idx, dist, count, flag_rows, counters,        \
            row_map, G);                                                                                        \
        return cudaGetLastError();                                                                              \
    } while (0)
        if (k <= 1) B200M_RERANK_CHUNK_CASE(1);
        if (k <= 2) B200M_RERANK_CHUNK_CASE(2);
        if (k <= 4) B200M_RERANK_CHUNK_CASE(4);
        if (k <= 8) B200M_RERANK_CHUNK_CASE(8);
        if (k <= 16) B200M_RERANK_CHUNK_CASE(16);
        B200M_RERANK_CHUNK_CASE(32);
#undef B200M_RERANK_CHUNK_CASE
    }
    // one CTA per SM holding as many warps (each with its own gather slab) as shared memory allows
    const size_t per_warp = rerank_warp_bytes(dp) + 8;
    int warps = (int) ((220 * 1024) / per_warp);
    if (warps > 16) warps = 16;
    if (warps < 1) return cudaErrorInvalidValue;   // dp <= 2048 needs at most 74 KB per warp
    const size_t smem = (size_t) warps * per_warp;
    size_t want = (n_rows + warps - 1) / warps;
    // small descriptors leave room for two CTAs per SM
    const size_t max_blocks = (size_t) sm_count * (smem <= 100 * 1024 ? 2 : 1);
    unsigned blocks = (unsigned) (want < max_blocks ? want : max_blocks);
#define B200M_RERANK_CASE(K)                                                                                    \
    do {                                                                                                        \
        cudaError_t e = cudaFuncSetAttribute(rerank_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                             (int) smem);                                                       \
        if (e != cudaSuccess) return e;                                                                         \
        rerank_kernel<K><<<blocks, warps * 32, smem, st>>>(                                                     \
            q_f32, q_valid, dp, dim, t_f32, t_valid, nt, (long long) t_index_offset, row_begin, n_rows, k,      \
            cand_idx, cand_cnt, n_lists, cap, cand_val, cand_thr, idx, dist, count, flag_rows, counters,        \
            row_map);                                                                                           \
        return cudaGetLastError();                                                                              \
    } while (0)
    if (k <= 1) B200M_RERANK_CASE(1);
    if (k <= 2) B200M_RERANK_CASE(2);
    if (k <= 4) B200M_RERANK_CASE(4);
    if (k <= 8) B200M_RERANK_CASE(8);
    if (k <= 16) B200M_RERANK_CASE(16);
    B200M_RERANK_CASE(32);
#undef B200M_RERANK_CASE
}
