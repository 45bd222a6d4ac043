// candidates_tc.cu -- the tensor-core candidate pass (sm_100a: TMA + tcgen05.mma + TMEM).
//
// Replaces the O(Nq*Nt*D) inner loop of cv::BFMatcher::knnMatch as called by matchBF
// (reference include/matching.h:612) and the kd-tree search of matchFLANN (:581).
//
// For a tile of 128 query rows the CTA streams every 256-row train tile through
//     acc[i][j] = sum_d (-2*a16[i][d]) * b16[j][d] + 1*nb_hi[j] + 1*nb_mid[j] + 1*nb_lo[j]
//               = |b16_j|^2 - 2 a16_i.b16_j                      (FP16 operands, FP32 accumulate in TMEM)
// i.e. the squared distance minus the per-row constant |a16_i|^2.  Operands are the K-major,
// 128B-swizzled tiles written by pack.cu and fetched by TMA; one elected thread issues
// tcgen05.mma (M=128, N=256, K=16) into one of two 256-column TMEM accumulators while the four
// epilogue warps drain the other with tcgen05.ld (lane == query row, so a thread owns a row).
//
// Selection is a running-threshold filter, never a top-k' truncation: each row keeps the k
// smallest accumulator VALUES seen so far (tk[]) and appends the index of every column with
//     acc <= thr(tk[k-1])
// to the row's candidate list in HBM.  thr(T) over-approximates, by the FP16 rounding of both
// rows (eta), the tensor-core accumulation slop and the FP32 rounding of the reference's own
// sequential sum (gamma), the largest accumulator an exact top-k member can have once k
// values <= T are known (derivation in DESIGN.md "Certified candidates").  Since tk[k-1] only
// decreases, the list is a superset of the exact top-k BY CONSTRUCTION; the exact FP32 re-rank
// (exact.cu) then reproduces the reference's distances and (dist, index) order bit for bit.
// A row whose list overflows its `cap` slots is re-done by the exact row kernel.
//
// Work decomposition: grid = (query tiles, train splits); each split writes its own list.
#include <cuda.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include "internal.cuh"

namespace {

// threads per CTA = 64 + 128 * EH (+ 32 in split-N mode): warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, then 4 * EH
// epilogue warps, then (split-N) the issuer of the second column half
constexpr int kATileBytes = B200M_TILE_M * 128;   // one 64-half K atom of the query tile
constexpr int kStageBytes = B200M_TILE_N * 128;   // one 64-half K atom of a train tile
constexpr int kTmemCols = 512;
constexpr int kTailBytes = 8576;         // barriers (<= 33 x 8 B) + TMEM slot + published thresholds (up to 4 x 128 x 4 B) + row
                                         // constants (2 KB) + the lists' published smallest values (4 KB)
constexpr int kMaxStages = 12;
constexpr int kMaxKAtoms = 10;           // A resident in shared memory (kp <= 640)
constexpr int kMaxKAtomsStreamed = 32;   // K-streamed form: A and B through the ring (kp <= 2048)
constexpr int kMaxLists = 16;
// Cycle stamps (B200M_TC_DEBUG & 1024) exist only in a library built with -DB200M_TC_TRACE (B200M_TC_TRACE=1 in the
// environment of build.py): their local arrays slow every debug instantiation down, also with the flag off.
#ifdef B200M_TC_TRACE
constexpr bool kTraceBuild = true;
#else
constexpr bool kTraceBuild = false;
#endif
constexpr int kTraceTile0 = 300, kTraceTiles = 12;   // which tiles of a sweep get cycle stamps
constexpr long long kWaitLimitCycles = 4000000000LL;   // ~2 s: a wedged pipeline traps instead of hanging the GPU

struct TcParams {
    int ka;               // 64-half K atoms per row (kp / 64)
    int ksteps;           // K=16 MMA steps actually needed: ceil((dim + 3) / 16)
    int stages;           // B ring depth
    int cluster;          // CTAs per cluster sharing every train tile by TMA multicast (1, 2 or 4)
    int pair;             // 1: CTA-pair mode (cta_group::2, M=256 across two SMs, each CTA holds half of B); cluster == 2
    int stage_bytes;      // bytes of one B stage in this CTA's shared memory (32 KB, or 16 KB in pair mode)
    int lean;             // 1: the MMA issuer runs the fully unrolled loop for one-atom descriptors (PAIR, 12 stages)
    int n_ttiles;         // 256-row train tiles
    int tiles_per_split;
    int q_row0;           // first query row of this call (row_begin)
    int n_rows;           // query rows of this call
    int k;
    int cap;              // candidate slots per row and list
    int dim;
    float bmax;           // max |b16| over the train side
    const float *q_norm16;
    int32_t *cand_idx;    // [n_lists][n_rows][cap]
    int32_t *cand_cnt;    // [n_lists][n_rows]
    float *cand_val;      // [n_lists][n_rows][cap] accumulator value of every entry, or null (EH = 1 kernels only)
    float *cand_thr;      // [n_lists][n_rows] the row's final append threshold (written when cand_val is)
    float *dump;          // debug: raw accumulators of one tile [128][256]
    int sweep_lag;        // tiles between consecutive followers of the rotated sweep; 0: every pair starts at tile 0
    int *sweep_hint;      // [train splits] how many tiles the most advanced CTA pair of a split has swept since the launch began
                          // (chunk-entry kernels: a pair starts a fixed distance behind it and wraps around)
    const int2 *seg_range;   // batch calls (or null): [query row / 256] = {first, end} train row of that query block's pair; the
                             // CTA then sweeps split `blockIdx.y` of that pair's train tiles only
    int debug_flags;      // timing experiments only (B200M_TC_DEBUG): 1 = epilogue skips its work, 2 = no MMAs issued,
                          // 4 = no B loads (pair mode), 8 / 16 = ring limited to 4 / 6 stages, 32 = epilogue only
                          // drains TMEM (no filtering), 64 / 128 = force EH = 1 / 2, 256 = fast path only,
                          // 512 = per-warp cycle totals, 1024 = cycle stamps of a few tiles (CTA pair 0),
                          // (n << 12) = n K steps per tile, 32768 = one accumulator, 65536 = no operand ring,
                          // 131072 / 262144 = service-scheduler / all epilogue warps skip a quarter of their columns
    const PrepDev *prep;  // DP kernels: the prepare step's device decision (usable) and norm bounds (bmax[train_side])
    int train_side;
};

// ---- PTX wrappers -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// A wedged pipeline traps after ~2 s instead of hanging the GPU (the launch then fails with cudaErrorLaunchFailure).  No
// printf on the time-out path: with a call there ptxas keeps nothing in uniform registers across the waits and re-derives
// every MMA descriptor per tile (126 instead of 81 instructions between two tiles' first MMAs in the issuer warps, a
// 32-byte larger stack frame) -- no measurable change in kernel time, but nothing to pay for (profiles/r02_notes.md 11).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > kWaitLimitCycles) __trap();
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *tmap, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_mcast(uint32_t dst, const CUtensorMap *tmap, uint32_t bar, int c0, int c1,
                                                  uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
        " [%0], [%1, {%4, %5}], [%2], %3;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "h"(cta_mask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap *tmap, uint32_t leader_bar, int c0, int c1) {
    // CTA-pair form: the bytes land in THIS CTA's shared memory, the transaction count goes to the leader's barrier
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_commit_mcast(uint32_t bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(cta_mask)
                 : "memory");
}
__device__ __forceinline__ void tc_commit_2sm_mcast(uint32_t bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(cta_mask)
                 : "memory");
}
// One MMA, issued only when `enable` is set (a predicated instruction instead of a branch keeps the issue loop
// straight-line); `accumulate` = 0 overwrites the accumulator.
__device__ __forceinline__ void tc_mma_f16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate, uint32_t enable) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.ne.b32 q, %5, 0;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(enable)
        : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate, uint32_t enable) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.ne.b32 q, %5, 0;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(enable)
        : "memory");
}
template <bool PAIR>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate,
                                       uint32_t enable) {
    if (PAIR) tc_mma_f16_2sm(tmem_d, desc_a, desc_b, idesc, accumulate, enable);
    else tc_mma_f16(tmem_d, desc_a, desc_b, idesc, accumulate, enable);
}
// true in exactly one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
// the same load with the destination registers tied to their previous contents ("+r"): the software-pipelined drain of
// the chunk epilogue loads into the SAME two register windows over and over, and with plain outputs ptxas gives every
// load a fresh 32-register tuple that overlaps a live one (35 register moves per tile to shuffle values out of the way)
__device__ __forceinline__ void tmem_ld_32x32b_x32_inplace(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
          "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
          "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
          "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// The same wait, tied to the 32 registers of the load it completes: in the software-pipelined drain of the chunk epilogue
// (EPI = 4) arithmetic on OTHER registers sits between a load and its wait, so nothing but this dependency keeps the
// compiler from scheduling the uses of r[] in front of the wait.
__device__ __forceinline__ void tmem_ld_wait_for(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                      "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]));
    asm volatile("" : "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                      "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31]));
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format, cute::UMMA::SmemDescriptor):
// start>>4 | LBO(ignored for swizzled K-major)=1 <<16 | SBO = 1024 B (8 rows x 128 B) >>4 <<32 | version 1 <<46 |
// layout SWIZZLE_128B (2) <<61.
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
    uint64_t d = (uint64_t) ((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t) 1 << 16;
    d |= (uint64_t) (1024 >> 4) << 32;
    d |= (uint64_t) 1 << 46;
    d |= (uint64_t) 2 << 61;
    return d;
}
// kind::f16 instruction descriptor: D=F32 (bit 4), A=B=F16 (0), K-major both, N>>3 at bit 17, M>>4 at bit 24.
constexpr uint32_t kInstrDesc = (1u << 4) | ((uint32_t) (B200M_TILE_N >> 3) << 17) | ((uint32_t) (B200M_TILE_M >> 4) << 24);
// CTA-pair form: M = 256 (128 rows from each CTA's A tile), N = 256 (128 train rows from each CTA's B stage)
constexpr uint32_t kInstrDescPair = (1u << 4) | ((uint32_t) (B200M_TILE_N >> 3) << 17) | ((uint32_t) ((2 * B200M_TILE_M) >> 4) << 24);

// ---- per-row selection state ------------------------------------------------------------------
// Shared-memory words are addressed through the shared window (32-bit addresses, ld/st/atom.shared) -- generic
// pointers would cost an address conversion per access inside the tile loop.
__device__ __forceinline__ float lds_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
template <int KT>
struct RowState {
    float tk[KT];   // k smallest accumulator values this thread has seen (of distinct columns), ascending
    float T;        // tk[k - 1], cached: the k-th smallest (+inf until k values are known)
    float thr;      // effective append threshold: min(own threshold, the partner thread's published one)
    uint32_t s_const;     // shared: the row's certificate constants {na, eta, slop, gfac} (read when the threshold is re-derived:
                          // rare, so they stay out of the register file)
    int cnt;              // entries appended to this thread's own list (may run past cap: overflow)
    uint32_t s_pub_own;   // shared (EH = 2): where this thread publishes its two smallest values; the row's slots (one per list,
                          // 8 bytes each) sit in one 32-byte line, so the other lists' slots follow from this address
    uint32_t s_thr_own;   // shared: where this thread publishes its own threshold (EH = 2: read by the thread that
                          // filters the other half of this row's columns)
};

// Largest accumulator value an exact top-k member can have, given k accumulators <= T exist
// (DESIGN.md "Certified candidates"); monotone in T, +inf for T = +inf.  sqrt.approx (2^-22 rel.)
// is covered by the 2^-20 guard terms.
__device__ __forceinline__ float cand_threshold(float T, float na, float eta, float slop, float gfac) {
    float x;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(x) : "f"(fmaxf(T + na + slop, 0.f)));
    float R = fmaf(x * 1.0000009537f + eta, gfac, eta);
    float R2 = R * R;
    return (R2 - na) + slop + 9.5367431640625e-7f * (R2 + na);
}

__device__ __forceinline__ float min3(float a, float b, float c) { return fminf(fminf(a, b), c); }   // one FMNMX3

template <int KT>
__device__ __forceinline__ float kth_smallest(const RowState<KT> &st, int k) {
    float T = st.tk[KT - 1];
#pragma unroll
    for (int s = 0; s < KT - 1; ++s)
        if (s == k - 1) T = st.tk[s];
    return T;
}
// branch-free sorted insertion of one value (2 * KT min/max ops)
template <int KT>
__device__ __forceinline__ void tk_insert(RowState<KT> &st, float v) {
#pragma unroll
    for (int s = 0; s < KT; ++s) {
        const float lo = fminf(st.tk[s], v);
        v = fmaxf(st.tk[s], v);
        st.tk[s] = lo;
    }
}
// The threads that share a row (EH = 2: two or four private lists over disjoint columns) each know only the k smallest
// values of their OWN columns; the k-th smallest of the row is at most the k-th smallest of any set of values of distinct
// columns, so a thread merges the two smallest values the other lists have published into a copy of its own list before it
// derives the threshold -- without this every list converges like a search over a quarter of the columns and the row
// collects about twice the candidates (and hits) it needs.  Stale values only make the bound looser.
template <int KT, int EH>
__device__ __forceinline__ void retighten(RowState<KT> &st, int k) {
    st.T = kth_smallest<KT>(st, k);
    float T = st.T;
    if (EH == 2) {
        asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(st.s_pub_own), "f"(st.tk[0]), "f"(KT > 1 ? st.tk[KT > 1 ? 1 : 0] : INFINITY) : "memory");
        RowState<KT> m;
#pragma unroll
        for (int s = 0; s < KT; ++s) m.tk[s] = st.tk[s];
        const uint32_t row_slots = st.s_pub_own & ~31u, li = (st.s_pub_own >> 3) & 3u;
#pragma unroll
        for (uint32_t j = 1; j < 4; ++j) {
            float a, b;
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(a), "=f"(b) : "r"(row_slots + 8u * ((li + j) & 3u)) : "memory");
            tk_insert<KT>(m, a);
            tk_insert<KT>(m, b);
        }
        T = kth_smallest<KT>(m, k);
    }
    float na, eta, slop, gfac;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(na), "=f"(eta), "=f"(slop), "=f"(gfac) : "r"(st.s_const) : "memory");
    const float thr_own = cand_threshold(T, na, eta, slop, gfac);
    st.thr = fminf(st.thr, thr_own);
    if (EH == 2) sts_f32(st.s_thr_own, thr_own);
}
// A chunk minimum enters the k-smallest list only if it can move the k-th smallest; the threshold is re-derived only
// when it did (a hit inside the certificate's margin, T <= v < thr(T), changes nothing).
template <int KT>
__device__ __forceinline__ void tk_offer(RowState<KT> &st, float m) {
    if (m < st.T) tk_insert<KT>(st, m);
}
template <int KT, int EH>
__device__ __forceinline__ void retighten_if_moved(RowState<KT> &st, int k) {
    if (kth_smallest<KT>(st, k) < st.T) retighten<KT, EH>(st, k);
}

#define F(i) __uint_as_float(r[i])
// element i (runtime index) of 32 registers through a select tree: no dynamic register indexing, no local memory
__device__ __forceinline__ float select32(const uint32_t (&r)[32], int i) {
    float s16[16], s8[8], s4[4];
#pragma unroll
    for (int j = 0; j < 16; ++j) s16[j] = (i & 16) ? F(16 + j) : F(j);
#pragma unroll
    for (int j = 0; j < 8; ++j) s8[j] = (i & 8) ? s16[8 + j] : s16[j];
#pragma unroll
    for (int j = 0; j < 4; ++j) s4[j] = (i & 4) ? s8[4 + j] : s8[j];
    const float s2a = (i & 2) ? s4[2] : s4[0], s2b = (i & 2) ? s4[3] : s4[1];
    return (i & 1) ? s2b : s2a;
}
// Warm-up path (a row that has not yet seen k columns, i.e. its first tile): every column under the running
// threshold is appended and inserted one at a time, the threshold tightening as soon as k values are known.  The
// value is fetched through a select tree (no dynamic register indexing, no local memory).
template <int KT, int EH>
__device__ __forceinline__ void warmup_chunk(const uint32_t (&r)[32], int col0, RowState<KT> &st, int k,
                                             int32_t *__restrict__ out, float *__restrict__ out_v, int cap) {
    const float thr0 = st.thr;
    uint32_t mask = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) mask |= (F(i) < thr0) ? (1u << i) : 0u;
    while (mask) {
        const int i = __ffs((int) mask) - 1;
        mask &= mask - 1;
        const float v = select32(r, i);
        if (v < st.thr) {   // the threshold may have tightened since the mask was taken
            const int slot = st.cnt++;
            if (slot < cap) {
                out[slot] = col0 + i;
                if (EH == 1) out_v[slot] = v;
            }
            tk_insert<KT>(st, v);
            retighten<KT, EH>(st, k);
        }
    }
}

// Steady-state append: every column of the chunk under the (already re-tightened) threshold goes to the list.
// EH = 1 kernels (long descriptors: the epilogue has slack, the re-rank gather is what costs) also record the
// accumulator value, so that the re-rank can drop every entry that the row's FINAL threshold no longer admits.
template <int EH>
__device__ __forceinline__ void append_chunk(const uint32_t (&r)[32], int col0, float thr, int &cnt,
                                             int32_t *__restrict__ out, float *__restrict__ out_v, int cap) {
    uint32_t mask = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) mask |= (F(i) < thr) ? (1u << i) : 0u;
    while (mask) {
        const int i = __ffs((int) mask) - 1;
        mask &= mask - 1;
        const int slot = cnt++;
        if (slot < cap) {
            out[slot] = col0 + i;
            if (EH == 1) out_v[slot] = select32(r, i);
        }
    }
}

// minimum of 32 accumulators: one dependent chain of 16 three-input min ops (one live temporary; the four chains of a
// 128-column batch are independent, which is all the instruction-level parallelism the half-rate min pipe can use)
__device__ __forceinline__ float min32(const uint32_t (&r)[32]) {
    float m = min3(F(0), F(1), F(2));
#pragma unroll
    for (int i = 3; i < 31; i += 2) m = min3(m, F(i), F(i + 1));
    return fminf(m, F(31));
}
#undef F

// 128 accumulators of one row, already in registers (the TMEM buffer has been handed back to the MMA issuer).
// Fast path: their minimum against the row threshold -- 66 min ops, one compare, one branch per 128 columns.
// Rare path: the four chunk minima (four distinct columns) go into the row's k-smallest list, the threshold is
// re-derived, and the columns under it are appended.  Tracking only chunk minima keeps the list an upper bound of the
// true k smallest -- all the certificate needs -- and misses a tightening only when two of the k smallest fall into
// one 32-column chunk.
// The four 32-column chunks sit at train rows col0, col0 + 32, col0 + hi, col0 + hi + 32 (hi = 64: 128 consecutive columns;
// hi = 128 in the split-N kernel, where a warp's columns 64..127 come from the other CTA's half of the train tile).
template <int KT, int EH>
__device__ __forceinline__ void process128(const uint32_t (&r0)[32], const uint32_t (&r1)[32], const uint32_t (&r2)[32],
                                           const uint32_t (&r3)[32], int col0, int hi, RowState<KT> &st, int k,
                                           int32_t *__restrict__ out, float *__restrict__ out_v, int cap) {
    const float m0 = min32(r0), m1 = min32(r1), m2 = min32(r2), m3 = min32(r3);
    if (fminf(min3(m0, m1, m2), m3) < st.thr) {   // inactive rows carry thr = -inf
        if (st.T == INFINITY) {
            if (m0 < st.thr) warmup_chunk<KT, EH>(r0, col0, st, k, out, out_v, cap);
            if (m1 < st.thr) warmup_chunk<KT, EH>(r1, col0 + 32, st, k, out, out_v, cap);
            if (m2 < st.thr) warmup_chunk<KT, EH>(r2, col0 + hi, st, k, out, out_v, cap);
            if (m3 < st.thr) warmup_chunk<KT, EH>(r3, col0 + hi + 32, st, k, out, out_v, cap);
        } else {
            tk_offer<KT>(st, m0);
            tk_offer<KT>(st, m1);
            tk_offer<KT>(st, m2);
            tk_offer<KT>(st, m3);
            retighten_if_moved<KT, EH>(st, k);
            const float thr = st.thr;
            if (m0 < thr) append_chunk<EH>(r0, col0, thr, st.cnt, out, out_v, cap);
            if (m1 < thr) append_chunk<EH>(r1, col0 + 32, thr, st.cnt, out, out_v, cap);
            if (m2 < thr) append_chunk<EH>(r2, col0 + hi, thr, st.cnt, out, out_v, cap);
            if (m3 < thr) append_chunk<EH>(r3, col0 + hi + 32, thr, st.cnt, out, out_v, cap);
        }
    }
}

// ---- 64-column batches (the sixteen-warp epilogues: EH = 2, no accumulator values recorded) ----
// The work of a batch is split into what needs the accumulator VALUES (scan64: the minima and, on a hit, bit masks of the
// columns under the threshold -- two-level: eight-column group minima first, so that a typical hit costs 16 + 8 compares
// instead of 64) and what does not (apply64: appends from the masks, k-smallest list, threshold).  The alternating-tile
// epilogue runs only scan64 of its first batch before the accumulators go back to the MMA issuer.
// (Tried and measured slower, C2 launch 3.78 -> 5.50 ms: moving 12 of every 32 columns of the "any column under the
// threshold?" test to FMA-pipe indicators sat(2^40 (thr - v)) summed with FADDs, to relieve the half-rate ALU pipe the four
// epilogue warps of a scheduler share -- profiles/r02_notes.md.)
struct Hit64 {
    uint32_t mask0, mask1;   // columns of the two 32-column chunks under the threshold at scan time
    float m0, m1;            // chunk minima
};
#define F(i) __uint_as_float(r[i])
__device__ __forceinline__ uint32_t mask_below(const uint32_t (&r)[32], float thr) {
    uint32_t mask = 0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const float pg = fminf(min3(min3(F(8 * g), F(8 * g + 1), F(8 * g + 2)), F(8 * g + 3), F(8 * g + 4)),
                               min3(F(8 * g + 5), F(8 * g + 6), F(8 * g + 7)));
        if (pg < thr) {
#pragma unroll
            for (int i = 8 * g; i < 8 * g + 8; ++i) mask |= (F(i) < thr) ? (1u << i) : 0u;
        }
    }
    return mask;
}
#undef F
__device__ __forceinline__ void append_mask(uint32_t mask, int col0, int &cnt, int32_t *__restrict__ out, int cap) {
    while (mask) {
        const int i = __ffs((int) mask) - 1;
        mask &= mask - 1;
        const int slot = cnt++;
        if (slot < cap) out[slot] = col0 + i;
    }
}
// needs the values.  Returns true when apply64 has work to do.  A row that has not yet seen k columns (its first
// tile) goes through the warm-up path right here, values in hand.
template <int KT>
__device__ __forceinline__ bool scan64(const uint32_t (&r0)[32], const uint32_t (&r1)[32], int col0, RowState<KT> &st, int k,
                                       int32_t *__restrict__ out, int cap, Hit64 &h) {
    h.m0 = min32(r0);
    h.m1 = min32(r1);
    h.mask0 = h.mask1 = 0u;
    if (!(fminf(h.m0, h.m1) < st.thr)) return false;   // inactive rows carry thr = -inf
    if (st.T == INFINITY) {
        if (h.m0 < st.thr) warmup_chunk<KT, 2>(r0, col0, st, k, out, nullptr, cap);
        if (h.m1 < st.thr) warmup_chunk<KT, 2>(r1, col0 + 32, st, k, out, nullptr, cap);
        st.T = kth_smallest<KT>(st, k);
        return false;
    }
    if (h.m0 < st.thr) h.mask0 = mask_below(r0, st.thr);
    if (h.m1 < st.thr) h.mask1 = mask_below(r1, st.thr);
    return true;
}
// needs only the masks and minima: may run after the accumulators have gone back (the masks were taken with a threshold
// at least as loose as the current one, so the list stays a superset)
template <int KT>
__device__ __forceinline__ void apply64(const Hit64 &h, int col0, RowState<KT> &st, int k, int32_t *__restrict__ out, int cap) {
    append_mask(h.mask0, col0, st.cnt, out, cap);
    append_mask(h.mask1, col0 + 32, st.cnt, out, cap);
    tk_offer<KT>(st, h.m0);
    tk_offer<KT>(st, h.m1);
    retighten_if_moved<KT, 2>(st, k);
}
template <int KT>
__device__ __forceinline__ void process64(const uint32_t (&r0)[32], const uint32_t (&r1)[32], int col0, RowState<KT> &st, int k,
                                          int32_t *__restrict__ out, int cap) {
    Hit64 h;
    if (scan64<KT>(r0, r1, col0, st, k, out, cap, h)) apply64<KT>(h, col0, st, k, out, cap);
}

// minimum of a 32-column chunk held as two 16-register halves: 16 min ops
__device__ __forceinline__ float min16x2(const uint32_t (&a)[16], const uint32_t (&b)[16]) {
    float m = min3(__uint_as_float(a[0]), __uint_as_float(a[1]), __uint_as_float(a[2]));
#pragma unroll
    for (int i = 3; i < 15; i += 2) m = min3(m, __uint_as_float(a[i]), __uint_as_float(a[i + 1]));
    m = min3(m, __uint_as_float(a[15]), __uint_as_float(b[0]));
#pragma unroll
    for (int i = 1; i < 15; i += 2) m = min3(m, __uint_as_float(b[i]), __uint_as_float(b[i + 1]));
    return fminf(m, __uint_as_float(b[15]));
}
// ---- chunk entries (EPI = 4) ----------------------------------------------------------------------------------------------
// A list entry is a 32-column CHUNK (its first train row and its minimum), not a column: the epilogue never finds out WHICH
// column of a chunk is under the threshold -- that search (group minima, 8..32 compares, bit masks, one append per column:
// 50-150 ALU-pipe instructions run by one lane of a diverged warp) was most of the hit path, and the hit path was a third of
// the instructions of the FPFH kernel.  The accumulators are dead as soon as their chunk minimum exists, so nothing of the
// hit path sits between a TMEM load and the hand-back, and no value registers are live in it.  The re-rank drops every entry
// whose minimum is not under the row's FINAL threshold (about k + margin of the ~k ln(N/k) entries survive) and runs the
// exact FP32 distance over all 32 train rows of a surviving chunk (one contiguous bulk copy: rerank_chunks_kernel, exact.cu).
// Superset argument: an exact top-k member j has v_j < thr(T_final) <= thr(T_run); its chunk's minimum is <= v_j, so the
// chunk was appended and survives the pruning.  The k-smallest list holds chunk minima: values of distinct columns.
template <int KT>
__device__ __forceinline__ void append_entry(float m, int col, RowState<KT> &st, int32_t *__restrict__ out,
                                             float *__restrict__ out_v, int cap) {
    const int slot = st.cnt++;
    if (slot < cap) {
        out[slot] = col;
        out_v[slot] = m;
    }
}
template <int KT>
__device__ __forceinline__ void chunk_hits(float m0, float m1, float m2, float m3, int c0, int c1, int c2, int c3,
                                           RowState<KT> &st, int k, int32_t *__restrict__ out, float *__restrict__ out_v,
                                           int cap) {
    tk_offer<KT>(st, m0);
    tk_offer<KT>(st, m1);
    tk_offer<KT>(st, m2);
    tk_offer<KT>(st, m3);
    retighten_if_moved<KT, 2>(st, k);   // (fewer than k values known: T and thr stay +inf, every chunk is appended)
    const float thr = st.thr;
    if (m0 < thr) append_entry<KT>(m0, c0, st, out, out_v, cap);
    if (m1 < thr) append_entry<KT>(m1, c1, st, out, out_v, cap);
    if (m2 < thr) append_entry<KT>(m2, c2, st, out, out_v, cap);
    if (m3 < thr) append_entry<KT>(m3, c3, st, out, out_v, cap);
}

// PAIR: CTA-pair mode (tcgen05.mma cta_group::2, M = 256 across two SMs, each CTA holds half of every train tile).
// EH:   epilogue column halves.  1 = four epilogue warps, a thread owns a whole row; 2 = eight warps (two per
//       scheduler), warp w drains TMEM lanes 32*(w%4).. (hardware rule) and the column half (w-2)/4 of every tile.
// DBG:  compiles the timing experiments (TcParams::debug_flags) and the accumulator dump in; the production
//       instantiation carries none of it in its loops.
// SPLITN: (pair mode, EH = 2, one-atom descriptors) every 256-column accumulator is two independent 128-column halves:
//       MMAs of N = 128 issued by one issuer warp per half (warp 1 and the extra warp 10), a full / empty barrier pair per
//       (buffer, half), handed back by the eight epilogue warps (four per CTA) that own the half.  Four hand-off chains
//       of 192 MMA cycles are in flight instead of two of 384, and a slow epilogue warp only holds up its own half.
//       Column c of half h is train row h*64 + c of the tile for c < 64 (CTA 0's stage rows) and 128 + h*64 + (c - 64)
//       beyond (CTA 1's).
// EPI:  (split-N only) 1 or 2 = sixteen epilogue warps holding 64 accumulators each (20 warps x 96 registers fit the
//       register file; four private candidate lists per row and train split).
//       1 ("alternating tiles"): a warp is bound to ONE accumulator buffer and drains the 128 columns of its half of every
//         second tile in two 64-column batches; the half goes back to the issuer after the second batch has been loaded,
//         i.e. the filtering of the first batch sits on the hand-off chain (measured: drain-only 2.44 ms per C2 launch,
//         fast path only 2.78 ms, full kernel 3.91 ms -- the append / threshold path of the first batch stalls the chain).
//       2 ("quarter columns"): a warp owns 64 columns of EVERY tile; the half of the accumulator (N = 128 MMA) goes back
//         as soon as both of its 64-column warps have their values in registers, all filtering happens off the chain.
//       4, 5 ("chunk entries", the default): alternating tiles, but a list entry is a 32-column chunk (first train row,
//         minimum) instead of a column -- see chunk_hits; drained by 32-column (4) or 16-column (5) TMEM loads.
// SEG:  (batch calls, production instantiations only) the CTA's train tiles come from TcParams::seg_range.  A compile-time
//       switch, not a runtime test of the pointer: either half of the lookup (the load, or the early exit) changes the register
//       allocation of the whole kernel -- the chunk-entry epilogue then spills more and the C2 launch runs 3.25 -> 3.50 ms on
//       one B200 (profiles/r03_ab_c2_seg_runtime.log).  SEG = false compiles to the single-pair kernel as it was.
// KS:   (pair mode, EH = 1, kp > 640: 11..32 K atoms) K-streamed operands.  The query tile no longer stays resident: a ring
//       stage holds this CTA's A atom (128 rows x 64 halves, 16 KB) followed by its half of the B atom (16 KB), and the
//       producer loads ka stages per train tile.  The certificate's accumulation slop grows with the K steps (DESIGN.md §4).
// DP:   (batch plans, next to the SEG instantiations only) device prepare: the train side's norm bound comes from
//       TcParams::prep instead of TcParams::bmax, and data outside the certificate's window (prep->usable == 0) leaves every
//       list of the CTA's rows overflowed (count cap + 1, threshold +inf) before anything else, so that the re-rank flags
//       every valid row and the exact fallback answers it.  A compile-time switch for the reason SEG is one.
template <int KT, bool PAIR, int EH, bool SPLITN, int EPI, bool DBG, bool SEG, bool KS = false, bool DP = false>
__global__ void __launch_bounds__(EPI ? 640 : 64 + 128 * EH + (SPLITN ? 32 : 0), 1)
tc_candidates_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_t,
                     const TcParams p) {
    static_assert(!KS || (PAIR && EH == 1 && !SPLITN && EPI == 0), "the K-streamed form is a pair-mode, EH = 1 kernel");
    const int dflags = DBG ? p.debug_flags : 0;
    float *const dump = DBG ? p.dump : nullptr;
    constexpr bool ALT = EPI != 0;   // the sixteen-warp layouts (warp roles, register re-division, four lists per row)
    constexpr bool QE = EPI == 2;
    constexpr bool CHK = EPI == 4 || EPI == 5;   // alternating tiles, list entries are 32-column chunks (first train row, minimum);
                                                 // 4: chunk-by-chunk drain (next load in flight under a min chain), 5: two loads per wait
    constexpr int kEpiWarps = 4 * EH * (ALT ? 2 : 1);
    constexpr int kEpiThreads = 32 * kEpiWarps;
    constexpr int kListsPerSplit = EH * (ALT ? 2 : 1);   // private candidate lists per row and train split
    // Warp roles.  ALT: warps 0..3 are the service warpgroup (TMA producer, the two MMA issuers, one idle warp) and the
    // sixteen epilogue warps form warpgroups 1..4, so that the register file can be re-divided per warpgroup
    // (setmaxnreg): 640 threads start with 96 registers each, the service warpgroup drops to 64, the epilogue rises to 104 -- the pool a CTA can re-divide is what it was launched with: 128 x 64 + 512 x 104 = 640 x 96.
    constexpr int kEpiWarp0 = ALT ? 4 : 2;           // first epilogue warp (TMEM lane quarter = warp & 3 either way)
    constexpr int kIssuer2 = ALT ? 2 : 2 + kEpiWarps;   // SPLITN: the warp that issues the second column half
    constexpr uint32_t kAcc = SPLITN ? 4u : 2u;      // accumulator hand-off units: buffers, or (buffer, half) pairs
    static_assert(!SPLITN || (PAIR && EH == 2), "split-N is a pair-mode, two-column-half kernel");
    static_assert(!ALT || SPLITN, "the alternating-tile epilogue is a split-N kernel");
    constexpr int kColsPerWarp = B200M_TILE_N / EH;
    // Everything in shared memory is addressed through the shared window (32-bit addresses).  The operand tiles need
    // 1024-byte alignment (128B-swizzle atoms of 8 rows); the dynamic segment starts at a 1024-aligned window offset as
    // long as the kernel has no static shared memory, and the round-up below keeps it correct if that ever changes
    // (the launch reserves the slack).
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t smem_u = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sA_u = smem_u;
    const uint32_t sB_u = KS ? sA_u : sA_u + (uint32_t) (p.ka * kATileBytes);   // KS: the ring starts the segment
    const uint32_t bars_u = sB_u + (uint32_t) (p.stages * p.stage_bytes);
    // barrier map: [0..S) full, [S..2S) empty, 2S a_full, then tmem_full[kAcc], tmem_empty[kAcc], the TMEM slot, thresholds
    const int stages = p.stages;
    const uint32_t bar_full0 = bars_u;
    const uint32_t bar_empty0 = bar_full0 + 8u * (uint32_t) stages;
    const uint32_t bar_a = bar_full0 + 8u * (uint32_t) (2 * stages);
    const uint32_t bar_tfull0 = bar_a + 8u;
    const uint32_t bar_tempty0 = bar_tfull0 + 8u * kAcc;                  // SPLITN: index buf * 2 + half
    const uint32_t tmem_slot = bar_tempty0 + 8u * kAcc;
    const uint32_t s_start = tmem_slot + 4u;                              // first tile of this CTA pair's sweep (CHK kernels)
    const uint32_t s_thr = (tmem_slot + 8u + 15u) & ~15u;                // published thresholds: [2][128] f32 per column half; ALT: [128][4]
    const uint32_t s_rowc = s_thr + 2048u;                               // [128][4] f32: per-row certificate constants
    const uint32_t s_pub = (s_rowc + 2048u + 31u) & ~31u;                // [128 rows][4 lists] x {smallest, second smallest} f32; a row's
                                                                         // four slots share one 32-byte line (retighten relies on it)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qtile = blockIdx.x, split = blockIdx.y;
    int seg_t0 = 0, seg_tiles = p.n_ttiles, tps = p.tiles_per_split;
    if constexpr (SEG) {
        // batch: the train tiles of this query block's pair (segments start at multiples of 256 rows on both sides, so the
        // two CTAs of a pair -- 256 query rows -- share one range), divided over the splits as a whole array is
        const int2 r = p.seg_range[(p.q_row0 + qtile * B200M_TILE_M) / B200M_TILE_N];
        seg_t0 = r.x / B200M_TILE_N;
        seg_tiles = (r.y + B200M_TILE_N - 1) / B200M_TILE_N - seg_t0;
        tps = (seg_tiles + (int) gridDim.y - 1) / (int) gridDim.y;
    }
    const int t0 = dump ? p.tiles_per_split : seg_t0 + split * tps;   // dump mode: tiles_per_split holds the tile id
    const int t1 = dump ? t0 + 1 : min(seg_t0 + seg_tiles, t0 + tps);
    const int ka = p.ka;
    if (DP && !p.prep->usable) {
        // outside the window: both CTAs of a pair read the same word and leave here, before any barrier, TMEM allocation
        // or pipeline exists, as below
        const int local = qtile * B200M_TILE_M + (int) threadIdx.x;
        if (threadIdx.x < B200M_TILE_M && local < p.n_rows) {
            for (int l = 0; l < kListsPerSplit; ++l) {
                const size_t list_row = (size_t) (split * kListsPerSplit + l) * p.n_rows + local;
                p.cand_cnt[list_row] = p.cap + 1;
                if (p.cand_thr) p.cand_thr[list_row] = INFINITY;
            }
        }
        return;
    }
    if (SEG && t1 <= t0) {
        // batch: a pair with fewer train tiles than there are splits (or none) leaves this CTA nothing to sweep.  Its rows'
        // lists are empty, with the final threshold an empty list has; the range is the same for both CTAs of a pair, so
        // both leave here, before any barrier, TMEM allocation or pipeline exists.
        const int local = qtile * B200M_TILE_M + (int) threadIdx.x;
        if (threadIdx.x < B200M_TILE_M && local < p.n_rows) {
            for (int l = 0; l < kListsPerSplit; ++l) {
                const size_t list_row = (size_t) (split * kListsPerSplit + l) * p.n_rows + local;
                p.cand_cnt[list_row] = 0;
                if (p.cand_thr) p.cand_thr[list_row] = INFINITY;
            }
        }
        return;
    }

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_q)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_t)) : "memory");
        for (int s = 0; s < stages; ++s) {
            mbar_init(bar_full0 + 8u * s, 1);
            // multicast mode: every CTA of the cluster must have read the stage; pair mode: one commit frees it
            mbar_init(bar_empty0 + 8u * s, SPLITN ? 2u : PAIR ? 1u : (uint32_t) p.cluster);   // SPLITN: both issuers commit
        }
        mbar_init(bar_a, 1);
        for (int b = 0; b < (int) kAcc; ++b) {
            mbar_init(bar_tfull0 + 8u * b, 1);
            // one arrival per epilogue WARP (a per-thread count serialises hundreds of barrier updates per tile);
            // pair mode: both CTAs' epilogue warps report to the leader, whose MMA thread owns the accumulators
            mbar_init(bar_tempty0 + 8u * b, QE ? 16u : SPLITN ? 8u : PAIR ? 2u * kEpiWarps : (uint32_t) kEpiWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        if (PAIR) {   // the same warp of both CTAs of the pair allocates
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                         "r"(kTmemCols)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                         "r"(kTmemCols)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    // Chunk-entry kernels can sweep the train tiles of their split in ROTATED order (the selection does not care in which
    // order the tiles come).  Started at tile 0, the CTA pairs of a long launch spread over the whole operand array (C4:
    // 256 MB against 126 MB of L2) and re-read it from DRAM -- 577 GB per launch against 0.5 GB of operands
    // (profiles/r02d_ncu_c4_cand.txt).  With p.sweep_lag > 0 every pair follows the most advanced one at a distance of its
    // own: the leaders report how far they have come (a running maximum of "tiles since the launch began"), a pair that starts
    // reads it and begins 16 + lag * (pair number mod 64) tiles behind -- everybody moves at the same speed, so all running
    // pairs stay inside one window (lag 20: ~1300 tiles, 42 MB), the front runner's misses fill L2 for the rest, and no two
    // pairs ask for the same line at the same time (pairs in exact lockstep do: their misses are not merged and DRAM traffic
    // doubles).  Measured on C4: DRAM reads 577 -> 88 GB per launch, 417 -> 372 ms; a window that is too narrow (lag 8) or
    // wider than L2 (lag 48+) is slower than no rotation.  The leader publishes the start tile to both CTAs of the pair.
    if (CHK && threadIdx.x == 0 && (p.cluster == 1 || cluster_ctarank() == 0u)) {
        const int nt_all = t1 - t0;
        int v_start = 0;
        if (!dump && nt_all > 1 && p.sweep_lag > 0) {
            int front;
            asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(front) : "l"(p.sweep_hint + split) : "memory");
            v_start = front - 16 - p.sweep_lag * (int) ((blockIdx.x >> 1) & 63u);
        }
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(s_start), "r"(v_start) : "memory");
        if (p.cluster > 1) asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(map_to_cta(s_start, 1)), "r"(v_start) : "memory");
    }
    tc_fence_before();
    if (p.cluster > 1) cluster_sync_all();   // peers' barriers are initialised before any multicast lands
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = lds_u32(tmem_slot);
    const uint32_t crank = p.cluster > 1 ? cluster_ctarank() : 0u;
    const int sweep_v0 = CHK ? (int) lds_u32(s_start) : 0;   // this pair's position when it starts, in tiles since the launch began
    const int sweep_start = CHK && t1 - t0 > 1 ? ((sweep_v0 % (t1 - t0)) + (t1 - t0)) % (t1 - t0) : 0;   // ... as a tile of the split
    const uint16_t cmask = (uint16_t) ((1u << p.cluster) - 1u);

    // setmaxnreg is a warpgroup-aligned instruction: all four warps of a warpgroup execute the SAME instruction, so the
    // service warpgroup re-divides its registers before its warps part ways.
    const bool is_service = ALT ? warp < 4 : (warp < 2 || (SPLITN && warp == kIssuer2));
    if (is_service) {
    if (ALT) asm volatile("setmaxnreg.dec.sync.aligned.u32 64;" ::: "memory");
    if (warp == 0) {
        // ===== TMA producer: the whole warp walks the ring (warp-uniform control flow keeps addresses and barrier
        // handles in uniform registers), one elected lane issues =====
        const int q_row = p.q_row0 + qtile * B200M_TILE_M;
        if (PAIR) {
            // CTA-pair mode: each CTA keeps its own 128 query rows and HALF of every train tile (its 128 rows);
            // all transaction bytes are counted on the leader's barriers, which the leader's MMA thread waits on.
            const uint32_t lead_a = map_to_cta(bar_a, 0);
            const uint32_t lead_full0 = map_to_cta(bar_full0, 0);
            const int row_off = (int) crank * (B200M_TILE_N / 2);
            if (!KS && elect_one()) {
                if (crank == 0) mbar_arrive_expect_tx(bar_a, (uint32_t) (2 * ka * kATileBytes));
                for (int a = 0; a < ka; ++a) tma_load_2d_2sm(sA_u + (uint32_t) (a * kATileBytes), &tmap_q, lead_a, a * 64, q_row);
            }
            __syncwarp();
            uint32_t s = 0, ph = 1;
            // opaque register copies of the ring's addresses (see the epilogue: keeps ptxas from re-deriving them per tile)
            uint32_t r_empty = bar_empty0, r_full = bar_full0, r_lead_full = lead_full0, r_sb = sB_u;
            asm volatile("" : "+r"(r_empty), "+r"(r_full), "+r"(r_lead_full), "+r"(r_sb));
            // pair mode: half a train tile per CTA (KS: behind this CTA's query atom)
            const uint32_t stage_bytes = (uint32_t) (KS ? kATileBytes + kStageBytes / 2 : kStageBytes / 2);
            const uint32_t b_off = KS ? (uint32_t) kATileBytes : 0u;
            int t = t0 + sweep_start;   // rotated sweep (chunk-entry kernels; 0 otherwise): t0 + start, ..., t1 - 1, t0, ...
            for (int lt = (dflags & 65536) ? t1 - t0 : 0; lt < t1 - t0; ++lt) {
                for (int a = 0; a < ka; ++a) {
                    mbar_wait(r_empty + 8u * s, ph);
                    if (elect_one()) {
                        if (dflags & 4) {   // timing experiment: no B traffic at all
                            if (crank == 0) mbar_arrive(r_full + 8u * s);
                        } else {
                            if (crank == 0) mbar_arrive_expect_tx(r_full + 8u * s, 2u * stage_bytes);
                            if (KS) tma_load_2d_2sm(r_sb + s * stage_bytes, &tmap_q, r_lead_full + 8u * s, a * 64, q_row);
                            tma_load_2d_2sm(r_sb + s * stage_bytes + b_off, &tmap_t, r_lead_full + 8u * s, a * 64,
                                            t * B200M_TILE_N + row_off);
                        }
                        // every 32 tiles the leader says where it is: pairs that start from now on start there
                        if (CHK && crank == 0 && a == 0 && (lt & 31) == 16 && !dump && p.sweep_lag > 0)
                            asm volatile("red.relaxed.gpu.global.max.s32 [%0], %1;" ::"l"(p.sweep_hint + split), "r"(sweep_v0 + lt) : "memory");
                    }
                    __syncwarp();
                    if (++s == (uint32_t) stages) { s = 0; ph ^= 1u; }
                }
                if (++t == t1) t = t0;
            }
        } else {
            if (elect_one()) {
                mbar_arrive_expect_tx(bar_a, (uint32_t) (ka * kATileBytes));
                for (int a = 0; a < ka; ++a) tma_load_2d(sA_u + (uint32_t) (a * kATileBytes), &tmap_q, bar_a, a * 64, q_row);
            }
            __syncwarp();
            const int slice = B200M_TILE_N / p.cluster;
            uint32_t s = 0, ph = 1;
            for (int t = t0; t < t1; ++t) {
                for (int a = 0; a < ka; ++a) {
                    mbar_wait(bar_empty0 + 8u * s, ph);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(bar_full0 + 8u * s, (uint32_t) kStageBytes);
                        if (p.cluster == 1) {
                            tma_load_2d(sB_u + s * (uint32_t) kStageBytes, &tmap_t, bar_full0 + 8u * s, a * 64, t * B200M_TILE_N);
                        } else {
                            // this CTA fetches its 1/cluster slice of the tile and multicasts it into every peer
                            tma_load_2d_mcast(sB_u + s * (uint32_t) kStageBytes + crank * (uint32_t) (slice * 128), &tmap_t,
                                              bar_full0 + 8u * s, a * 64, t * B200M_TILE_N + (int) crank * slice, cmask);
                        }
                    }
                    __syncwarp();
                    if (++s == (uint32_t) stages) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 1 || (SPLITN && warp == kIssuer2)) {
        // ===== MMA issuer.  One MMA (K = 16) is 128 tensor-pipe cycles, so the issue loop has to stay far below that
        // per instruction: warp-uniform control flow, ring position kept as counters (no divisions), descriptors
        // advanced by adding to their low word, the four K steps of an atom unrolled. =====
        if (!PAIR || crank == 0) {   // pair mode: the leader CTA issues for both SMs
            if (!KS) mbar_wait(bar_a, 0);
            tc_fence_after();
            const uint64_t desc_a0 = make_kmajor_sw128_desc(sA_u);
            const uint64_t desc_b0 = make_kmajor_sw128_desc(sB_u);
            const uint32_t a_step = (uint32_t) (kATileBytes >> 4), b_step = (uint32_t) (p.stage_bytes >> 4);
            const uint32_t nk_full = (dflags & 2) ? 0u : 4u;
            const uint32_t nk_last = (dflags & 2) ? 0u : (uint32_t) (p.ksteps - 4 * (ka - 1));   // K steps of the last atom (1..4)
            constexpr uint32_t idesc = PAIR ? kInstrDescPair : kInstrDesc;
            if (SPLITN) {
                // one issuer per column half: N = 128 MMAs on this CTA pair's rows [half*64, half*64 + 64) of every stage
                // (8 KB into each CTA's half tile), accumulator columns [buf*256 + half*128, +128); the unrolled loop of
                // the one-atom case below with the half's constants
                const uint32_t hf = warp == 1 ? 0u : 1u;
                constexpr uint32_t idesc_h = (1u << 4) | ((uint32_t) ((B200M_TILE_N / 2) >> 3) << 17) |
                                             ((uint32_t) ((2 * B200M_TILE_M) >> 4) << 24);
                const uint64_t desc_bh = desc_b0 + (uint64_t) (hf * (uint32_t) ((64 * 128) >> 4));
                const uint32_t tmem_h = tmem_base + hf * (uint32_t) (B200M_TILE_N / 2);
                const int nt = t1 - t0;
                // (timing experiment, debug instantiation: (n << 12) forces n K steps per tile)
                const uint32_t nk = (DBG && (dflags & 2) == 0 && (((uint32_t) dflags >> 12) & 7u)) ? (((uint32_t) dflags >> 12) & 7u) : nk_last;
                uint32_t ph = 0;
                int lt = 0;
                // trace builds: cycle stamps of kTraceTiles tiles -- before the waits, operands landed, half handed back, issued
                const bool trace = kTraceBuild && (dflags & 1024) && blockIdx.x == 0 && blockIdx.y == 0;
                long long tr[kTraceBuild ? kTraceTiles : 1][4];
                while (lt < nt) {
#pragma unroll
                    for (int i = 0; i < kMaxStages; ++i) {
                        if (lt + i < nt) {
                            const uint32_t buf = (uint32_t) (i & 1);
                            const int ti = lt + i - kTraceTile0;
                            const bool tr_on = trace && ti >= 0 && ti < kTraceTiles;
                            if (kTraceBuild && tr_on) tr[ti][0] = clock64();
                            mbar_wait(bar_full0 + 8u * (uint32_t) i, ph);
                            if (kTraceBuild && tr_on) tr[ti][1] = clock64();
                            mbar_wait(bar_tempty0 + 8u * (buf * 2u + hf), (uint32_t) (((i >> 1) & 1) ^ 1));
                            tc_fence_after();
                            if (kTraceBuild && tr_on) tr[ti][2] = clock64();
                            if (elect_one()) {
                                const uint64_t db = desc_bh + (uint64_t) ((uint32_t) i * (uint32_t) ((kStageBytes / 2) >> 4));
                                const uint32_t tmem_d = tmem_h + buf * (uint32_t) B200M_TILE_N;
                                tc_mma<PAIR>(tmem_d, desc_a0, db, idesc_h, 0u, (uint32_t) (nk > 0));
                                tc_mma<PAIR>(tmem_d, desc_a0 + 2, db + 2, idesc_h, 1u, (uint32_t) (nk > 1));
                                tc_mma<PAIR>(tmem_d, desc_a0 + 4, db + 4, idesc_h, 1u, (uint32_t) (nk > 2));
                                tc_mma<PAIR>(tmem_d, desc_a0 + 6, db + 6, idesc_h, 1u, (uint32_t) (nk > 3));
                                // the accumulator's commit first: it is on the hand-off chain, the operand ring is 12 stages deep
                                tc_commit_2sm_mcast(bar_tfull0 + 8u * (buf * 2u + hf), (uint16_t) 3);
                                tc_commit_2sm_mcast(bar_empty0 + 8u * (uint32_t) i, (uint16_t) 3);
                            }
                            __syncwarp();
                            if (kTraceBuild && tr_on) tr[ti][3] = clock64();
                        }
                    }
                    lt += kMaxStages;
                    ph ^= 1u;
                }
                if (kTraceBuild && trace && lane == 0)
                    for (int i = 0; i < kTraceTiles && kTraceTile0 + i < nt; ++i)
                        printf("b200match trace issuer half %u tile %d: %lld %lld %lld %lld\n", hf, kTraceTile0 + i, tr[i][0], tr[i][1],
                               tr[i][2], tr[i][3]);
            } else if (PAIR && EH == 2 && p.lean && !(DBG && (dflags & ~(1 | 32 | 256 | 512 | 131072 | 262144)))) {
                // One-atom descriptors (FPFH-33: 3 MMAs = 384 tensor-pipe cycles per tile).  The general loop below costs
                // this warp ~100 dependent instructions per tile (stage index in a vector register: R2UR moves, address
                // arithmetic, descriptor adds) -- ~630 cycles when it has its scheduler to itself, far more while the two
                // epilogue warps on the same scheduler stream their min chains, and all of it sits on the accumulator
                // hand-off chain.  Here the ring is unrolled over its 12 stages: stage, accumulator buffer, barrier
                // addresses and even the accumulator barrier's parity (lt = 12 r + i, (lt >> 1) & 1 = (i >> 1) & 1) are
                // immediates of the unrolled body.
                static_assert(kMaxStages == 12, "unrolled issue loop is written for a 12-stage ring");
                const int nt = t1 - t0;
                const uint32_t nk = nk_last;
                uint32_t ph = 0;
                int lt = 0;
                while (lt < nt) {
#pragma unroll
                    for (int i = 0; i < kMaxStages; ++i) {
                        if (lt + i < nt) {
                            const uint32_t buf = (uint32_t) (i & 1);
                            mbar_wait(bar_full0 + 8u * (uint32_t) i, ph);
                            mbar_wait(bar_tempty0 + 8u * buf, (uint32_t) (((i >> 1) & 1) ^ 1));
                            tc_fence_after();
                            if (elect_one()) {
                                const uint64_t db = desc_b0 + (uint64_t) ((uint32_t) i * (uint32_t) ((kStageBytes / 2) >> 4));
                                const uint32_t tmem_d = tmem_base + buf * (uint32_t) B200M_TILE_N;
                                tc_mma<PAIR>(tmem_d, desc_a0, db, idesc, 0u, (uint32_t) (nk > 0));
                                tc_mma<PAIR>(tmem_d, desc_a0 + 2, db + 2, idesc, 1u, (uint32_t) (nk > 1));
                                tc_mma<PAIR>(tmem_d, desc_a0 + 4, db + 4, idesc, 1u, (uint32_t) (nk > 2));
                                tc_mma<PAIR>(tmem_d, desc_a0 + 6, db + 6, idesc, 1u, (uint32_t) (nk > 3));
                                tc_commit_2sm_mcast(bar_empty0 + 8u * (uint32_t) i, (uint16_t) 3);
                                tc_commit_2sm_mcast(bar_tfull0 + 8u * buf, (uint16_t) 3);
                            }
                            __syncwarp();
                        }
                    }
                    lt += kMaxStages;
                    ph ^= 1u;
                }
            } else {
            uint32_t s = 0, ph = 0;
            const bool trace = kTraceBuild && (dflags & 1024) && blockIdx.x == 0 && blockIdx.y == 0;   // cycle stamps of kTraceTiles tiles
            const uint32_t nk_force = ((uint32_t) dflags >> 12) & 7u;   // timing experiment: K steps per tile forced to 1..4
            const bool one_buf = (dflags & 32768) != 0;                 // timing experiment: every tile into accumulator 0
            const bool no_ring = (dflags & 65536) != 0;                 // timing experiment: no operand ring (no full wait, no empty commit)
            long long tr[kTraceTiles][7];
            if (trace)
                for (int i = 0; i < kTraceTiles; ++i)
                    for (int j = 0; j < 7; ++j) tr[i][j] = 0;
            for (int lt = 0; lt < t1 - t0; ++lt) {
                const uint32_t buf = (uint32_t) lt & 1u;
                const uint32_t tmem_d = tmem_base + (one_buf ? 0u : buf * (uint32_t) B200M_TILE_N);
                const int ti = lt - kTraceTile0;
                const bool tr_on = trace && ti >= 0 && ti < kTraceTiles;
                for (int a = 0; a < ka; ++a) {
                    if (!no_ring) mbar_wait(bar_full0 + 8u * s, ph);
                    // KS: A atom at the start of the stage, the B half behind it
                    const uint64_t da = KS ? desc_b0 + (uint64_t) (s * b_step) : desc_a0 + (uint64_t) ((uint32_t) a * a_step);
                    const uint64_t db = KS ? da + (uint64_t) (kATileBytes >> 4) : desc_b0 + (uint64_t) (s * b_step);
                    // K steps of this atom: 4, or what is left of the row in the last one; +32 B (2 descriptor
                    // units) per K = 16 step inside the 128 B swizzle atom
                    uint32_t nk = a + 1 < ka ? nk_full : nk_last;
                    if (nk_force) nk = nk_force;
                    // The accumulator buffer is waited for LAST, with the operands landed and the descriptors built:
                    // for short descriptors the hand-back of the buffer by the epilogue is the critical path, and
                    // everything between that arrival and the first MMA is latency on it.
                    if (tr_on && a == 0) tr[ti][0] = clock64();   // operands landed
                    if (a == 0) mbar_wait(bar_tempty0 + 8u * buf, (((uint32_t) lt >> 1) & 1u) ^ 1u);
                    tc_fence_after();
                    if (tr_on && a == 0) tr[ti][1] = clock64();   // accumulator buffer handed back
                    if (elect_one()) {
                        tc_mma<PAIR>(tmem_d, da, db, idesc, (uint32_t) (a != 0), (uint32_t) (nk > 0));
                        if (tr_on && a == 0) tr[ti][2] = clock64();
                        tc_mma<PAIR>(tmem_d, da + 2, db + 2, idesc, 1u, (uint32_t) (nk > 1));
                        if (tr_on && a == 0) tr[ti][3] = clock64();
                        tc_mma<PAIR>(tmem_d, da + 4, db + 4, idesc, 1u, (uint32_t) (nk > 2));
                        tc_mma<PAIR>(tmem_d, da + 6, db + 6, idesc, 1u, (uint32_t) (nk > 3));
                        if (tr_on && a == 0) tr[ti][4] = clock64();
                        // frees the B stage once these MMAs have read it (in every CTA that writes into it)
                        if (!no_ring) {
                            if (PAIR) tc_commit_2sm_mcast(bar_empty0 + 8u * s, (uint16_t) 3);
                            else if (p.cluster == 1) tc_commit(bar_empty0 + 8u * s);
                            else tc_commit_mcast(bar_empty0 + 8u * s, cmask);
                        }
                        if (tr_on && a == 0) tr[ti][5] = clock64();
                    }
                    __syncwarp();
                    if (++s == (uint32_t) stages) { s = 0; ph ^= 1u; }
                }
                if (elect_one()) {   // accumulators of this tile complete (in both CTAs of a pair)
                    if (PAIR) tc_commit_2sm_mcast(bar_tfull0 + 8u * buf, (uint16_t) 3);
                    else tc_commit(bar_tfull0 + 8u * buf);
                    if (tr_on) tr[ti][6] = clock64();   // MMAs and commits issued
                }
                __syncwarp();
            }
            if (trace) {
                // the stamps live in whichever lane was elected (the same one every time); the others hold zeros
                for (int i = 0; i < kTraceTiles && kTraceTile0 + i < t1 - t0; ++i)
                    if (tr[i][6] != 0 && tr[i][2] != 0)
                        printf("b200match trace mma tile %d: %lld %lld %lld %lld %lld %lld %lld\n", kTraceTile0 + i, tr[i][0],
                               tr[i][1], tr[i][2], tr[i][3], tr[i][4], tr[i][5], tr[i][6]);
            }
            }   // general issue loop
        }
    }
    } else {
        if (ALT) asm volatile("setmaxnreg.inc.sync.aligned.u32 104;" ::: "memory");
        // ===== epilogue: a thread owns one TMEM lane (query row) and kColsPerWarp columns of every tile.  With EH = 2
        // the two threads of a row share its candidate list (shared-memory counter) and exchange thresholds. =====
        const int quarter = warp & 3;
        const int half = ((warp - kEpiWarp0) >> 2) & 1;
        // EPI 1: the accumulator buffer (tile parity) this warp is bound to; EPI 2: which 64 columns of its 128-column half
        const int bsel = ALT ? (warp - kEpiWarp0) >> 3 : 0;
        const int row_in_tile = quarter * 32 + lane;
        const int local = qtile * B200M_TILE_M + row_in_tile;
        const bool active = local < p.n_rows;
        RowState<KT> st;
#pragma unroll
        for (int s = 0; s < KT; ++s) st.tk[s] = INFINITY;
        st.thr = active ? INFINITY : -INFINITY;
        st.T = INFINITY;
        st.cnt = 0;
        st.s_thr_own = ALT ? s_thr + 4u * (uint32_t) (row_in_tile * 4 + bsel * 2 + half)
                           : s_thr + 4u * (uint32_t) (half * B200M_TILE_M + row_in_tile);
        const uint32_t s_thr_peer = ALT ? s_thr + 16u * (uint32_t) row_in_tile   // the row's four published thresholds
                                        : s_thr + 4u * (uint32_t) ((half ^ 1) * B200M_TILE_M + row_in_tile);
        sts_f32(st.s_thr_own, st.thr);
        st.s_pub_own = s_pub + 32u * (uint32_t) row_in_tile + 8u * (uint32_t) (bsel * 2 + half);
        if (EH == 2) {   // nothing published yet (slots of lists that do not exist stay at +inf)
            if (!ALT) asm volatile("st.shared.v2.f32 [%0], {%1, %1};" ::"r"(st.s_pub_own + 16u), "f"(INFINITY) : "memory");
            asm volatile("st.shared.v2.f32 [%0], {%1, %1};" ::"r"(st.s_pub_own), "f"(INFINITY) : "memory");
        }
        {
            const float na = active ? p.q_norm16[p.q_row0 + local] : 0.f;
            const float ab = sqrtf(na) + (DP ? p.prep->bmax[p.train_side] : p.bmax);
            st.s_const = s_rowc + 16u * (uint32_t) row_in_tile;
            // every thread of the row writes the same four values
            sts_f32(st.s_const, na);
            sts_f32(st.s_const + 4u, ab * 4.8828125e-4f * 1.001953125f + 2.384185791015625e-7f * sqrtf((float) p.dim));
            // accumulation slop: measured bound 2^-16 ab^2 up to 40 K steps; KS: 2^-21 ab^2 per K step (DESIGN.md §4)
            sts_f32(st.s_const + 8u, KS ? ab * ab * ((float) p.ksteps * 4.76837158203125e-7f) + 1e-6f
                                        : ab * ab * 1.52587890625e-5f + 1e-6f);
            sts_f32(st.s_const + 12u, 1.f + 2.2f * (float) (p.dim + 4) * 5.9604644775390625e-8f);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");   // shared row state initialised
        // every epilogue thread owns a private candidate list: [split][column half][row][cap]
        const size_t list_row = (size_t) (split * kListsPerSplit + bsel * 2 + half) * p.n_rows + (active ? local : 0);
        int32_t *const out = p.cand_idx + list_row * p.cap;
        float *const out_v = (EH == 1 || CHK) ? p.cand_val + list_row * p.cap : nullptr;
        const int k = p.k, cap = p.cap;
        const uint32_t lane_base = tmem_base + ((uint32_t) (quarter * 32) << 16) + (uint32_t) (half * kColsPerWarp);
        // SPLITN: this warp's hand-off barriers are those of its column half (index buf * 2 + half)
        const uint32_t acc_stride = SPLITN ? 16u : 8u;
        const uint32_t tfull_mine = bar_tfull0 + (SPLITN ? 8u * (uint32_t) half : 0u) + ((EPI == 1 || CHK) ? 16u * (uint32_t) bsel : 0u);
        const uint32_t tempty_mine = bar_tempty0 + (SPLITN ? 8u * (uint32_t) half : 0u) + ((EPI == 1 || CHK) ? 16u * (uint32_t) bsel : 0u);
        const uint32_t tempty_dst0 = PAIR ? map_to_cta(tempty_mine, 0) : tempty_mine;
        // The addresses the tile loop needs, as opaque register values: left to itself ptxas re-derives them on every tile
        // (shared-window base from %cluster_ctaid, kernel parameters from constant memory, threadIdx: ~40 instructions,
        // half of them a dependent chain in front of the barrier test and of the first TMEM load) -- on the hand-off
        // chain of every tile.
        uint32_t e_tfull = tfull_mine, e_tempty = tempty_dst0, e_tmem = lane_base, e_peer = s_thr_peer;
        asm volatile("" : "+r"(e_tfull), "+r"(e_tempty), "+r"(e_tmem), "+r"(e_peer));
        if constexpr (QE) {
            // ===== quarter-column epilogue: 64 columns of every tile; hand back first, filter afterwards =====
            uint32_t r0[32], r1[32];
            const uint32_t tcol = e_tmem + (uint32_t) bsel * 64u;
            // train rows of the warp's columns: TMEM columns 0..63 of a half are tile rows half*64 + c (CTA 0's stage rows),
            // columns 64..127 are rows 128 + half*64 + c (CTA 1's)
            int col_base = t0 * B200M_TILE_N + bsel * 128 + half * 64;
            for (int lt = 0; lt < t1 - t0; ++lt, col_base += B200M_TILE_N) {
                const uint32_t buf = (uint32_t) lt & 1u;
                mbar_wait(e_tfull + 16u * buf, ((uint32_t) lt >> 1) & 1u);
                tc_fence_after();
                if (!(dflags & 1)) {
                    const uint32_t taddr = tcol + buf * (uint32_t) B200M_TILE_N;
                    tmem_ld_32x32b_x32(taddr, r0);
                    tmem_ld_32x32b_x32(taddr + 32u, r1);
                    tmem_ld_wait();
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(e_tempty + 16u * buf);
                {   // what the row's other three threads have learnt (own entry included: harmless)
                    float t0_, t1_, t2_, t3_;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(t0_), "=f"(t1_), "=f"(t2_), "=f"(t3_) : "r"(e_peer) : "memory");
                    st.thr = fminf(st.thr, fminf(fminf(t0_, t1_), fminf(t2_, t3_)));
                }
                if (dflags & (1 | 32)) continue;
                if (dflags & 256) {   // timing experiment: fast path only
                    if (fminf(min32(r0), min32(r1)) < st.thr) st.cnt += 1;
                    continue;
                }
                process64<KT>(r0, r1, col_base, st, k, out, cap);
            }
        } else if constexpr (CHK) {
            // ===== chunk-entry epilogue: alternating tiles (this warp owns accumulator buffer `bsel`), drained one 32-column
            // chunk at a time with the next chunk's TMEM load in flight under the min chain of the current one; the half goes
            // back to its MMA issuer when the fourth load has landed; the whole hit path runs after that, on four floats. =====
            uint32_t r0[32], r1[32];
            uint32_t qa[16], qb[16], qc[16], qd[16];   // EPI = 5: the same drain in 16-column loads
#pragma unroll
            for (int i = 0; i < 32; ++i) r0[i] = r1[i] = 0u;   // (the in-place loads formally read their destinations)
            const uint32_t taddr = e_tmem + (uint32_t) bsel * (uint32_t) B200M_TILE_N;
            // train rows of the warp's columns: 0..63 -> tile row half*64 + c (CTA 0's stage rows), 64..127 -> 128 + half*64 + c;
            // the sweep is rotated: local tile lt is train tile t0 + (sweep_start + lt) mod (t1 - t0)
            // (kept as ONE running register: the wrap test compares against t1 * 256, half * 64 < 256 does not disturb it)
            int col_next = (t0 + sweep_start + bsel) * B200M_TILE_N + half * 64;
            if (col_next >= t1 * B200M_TILE_N) col_next -= (t1 - t0) * B200M_TILE_N;
            uint32_t par = 0;
            for (int lt = bsel; lt < t1 - t0; lt += 2) {
                const int col_base = col_next;
                col_next += 2 * B200M_TILE_N;
                if (col_next >= t1 * B200M_TILE_N) col_next -= (t1 - t0) * B200M_TILE_N;
                mbar_wait(e_tfull, par);
                par ^= 1u;
                tc_fence_after();
                float m0 = INFINITY, m1 = INFINITY, m2 = INFINITY, m3 = INFINITY;
                if (EPI == 5) {
                    if (!(dflags & 1)) {
                        tmem_ld_32x32b_x16(taddr, qa);
                        tmem_ld_32x32b_x16(taddr + 16u, qb);
                        tmem_ld_wait();
                        tmem_ld_32x32b_x16(taddr + 32u, qc);
                        tmem_ld_32x32b_x16(taddr + 48u, qd);
                        if (!(dflags & 32)) m0 = min16x2(qa, qb);
                        tmem_ld_wait();
                        tmem_ld_32x32b_x16(taddr + 64u, qa);
                        tmem_ld_32x32b_x16(taddr + 80u, qb);
                        if (!(dflags & 32)) m1 = min16x2(qc, qd);
                        tmem_ld_wait();
                        tmem_ld_32x32b_x16(taddr + 96u, qc);
                        tmem_ld_32x32b_x16(taddr + 112u, qd);
                        if (!(dflags & 32)) m2 = min16x2(qa, qb);
                        tmem_ld_wait();
                    }
                } else if (!(dflags & 1)) {
                    tmem_ld_32x32b_x32_inplace(taddr, r0);
                    tmem_ld_wait_for(r0);
                    tmem_ld_32x32b_x32_inplace(taddr + 32u, r1);
                    if (!(dflags & 32)) m0 = min32(r0);
                    tmem_ld_wait_for(r1);
                    tmem_ld_32x32b_x32_inplace(taddr + 64u, r0);
                    if (!(dflags & 32)) m1 = min32(r1);
                    tmem_ld_wait_for(r0);
                    tmem_ld_32x32b_x32_inplace(taddr + 96u, r1);
                    if (!(dflags & 32)) m2 = min32(r0);
                    tmem_ld_wait_for(r1);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(e_tempty);
                if (dflags & (1 | 32)) continue;
                m3 = EPI == 5 ? min16x2(qc, qd) : min32(r1);
                {   // what the row's other three threads have learnt (own entry included: harmless)
                    float t0_, t1_, t2_, t3_;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(t0_), "=f"(t1_), "=f"(t2_), "=f"(t3_) : "r"(e_peer) : "memory");
                    st.thr = fminf(st.thr, fminf(fminf(t0_, t1_), fminf(t2_, t3_)));
                }
                if (fminf(min3(m0, m1, m2), m3) < st.thr) {   // inactive rows carry thr = -inf
                    if (dflags & 256) { st.cnt += 1; continue; }   // timing experiment: fast path only
                    chunk_hits<KT>(m0, m1, m2, m3, col_base, col_base + 32, col_base + 128, col_base + 160, st, k, out, out_v, cap);
                }
            }
        } else if constexpr (ALT) {
            // ===== alternating-tile epilogue: this warp owns accumulator buffer `bsel`, i.e. tiles bsel, bsel + 2, ...
            // Of the first 64-column batch only what needs the values (minima, hit masks) runs before the second batch is
            // loaded and the half goes back to its MMA issuer; appends and threshold upkeep of both batches run after. =====
            uint32_t r0[32], r1[32];
            const uint32_t taddr = e_tmem + (uint32_t) bsel * (uint32_t) B200M_TILE_N;
            // train rows of the warp's columns: 0..63 -> tile row half*64 + c (CTA 0's stage rows), 64..127 -> 128 + half*64 + c
            int col_base = (t0 + bsel) * B200M_TILE_N + half * 64;
            uint32_t par = 0;
            // B200M_TC_DEBUG & 512: where this warp's cycles go -- [phase: first 64 tiles / the rest][wait for the accumulators,
            // values in registers + first scan (on the hand-off chain), everything after the hand-back], and how many
            // batches took the hit path in some lane
            const bool prof = DBG && (dflags & 512) != 0;
            long long cyc[2][3] = {{0, 0, 0}, {0, 0, 0}};
            int hits[2][2] = {{0, 0}, {0, 0}};
            // trace builds: accumulators seen, first batch scanned, second batch in registers, handed back, iteration done
            const bool etrace = kTraceBuild && (dflags & 1024) && blockIdx.x < 2 && blockIdx.y == 0;
            long long etr[kTraceBuild ? kTraceTiles / 2 + 1 : 1][5];
            for (int lt = bsel; lt < t1 - t0; lt += 2, col_base += 2 * B200M_TILE_N) {
                const int ph = lt < 64 ? 0 : 1;
                long long c0 = prof ? clock64() : 0;
                mbar_wait(e_tfull, par);
                par ^= 1u;
                tc_fence_after();
                if (prof) { const long long c1 = clock64(); cyc[ph][0] += c1 - c0; c0 = c1; }
                const int eti = (lt - kTraceTile0) >> 1;
                const bool etr_on = kTraceBuild && etrace && lt >= kTraceTile0 && lt < kTraceTile0 + kTraceTiles;
                if (kTraceBuild && etr_on) etr[eti][0] = clock64();
                Hit64 h0;
                bool hit0 = false;
                if (!(dflags & 1)) {
                    tmem_ld_32x32b_x32(taddr, r0);
                    tmem_ld_32x32b_x32(taddr + 32u, r1);
                    tmem_ld_wait();
                    if (!(dflags & 32)) {
                        if (dflags & 256) {   // timing experiment: fast path only
                            if (fminf(min32(r0), min32(r1)) < st.thr) st.cnt += 1;
                        } else if ((dflags & (2048 | 4096)) && st.T != INFINITY) {
                            // timing experiments (results invalid): no hit masks for the first batch -- the hand-off chain
                            // carries the plain min pass only; threshold upkeep from the chunk minima stays
                            h0.m0 = min32(r0);
                            h0.m1 = min32(r1);
                            h0.mask0 = h0.mask1 = 0u;
                            hit0 = fminf(h0.m0, h0.m1) < st.thr;
                        } else {
                            hit0 = scan64<KT>(r0, r1, col_base, st, k, out, cap, h0);
                        }
                    }
                    if (kTraceBuild && etr_on) etr[eti][1] = clock64();
                    tmem_ld_32x32b_x32(taddr + 64u, r0);
                    tmem_ld_32x32b_x32(taddr + 96u, r1);
                    tmem_ld_wait();
                    if (kTraceBuild && etr_on) etr[eti][2] = clock64();
                }
                // all 128 columns are in registers or reduced to masks: the half goes back to its MMA issuer
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(e_tempty);
                if (kTraceBuild && etr_on) etr[eti][3] = clock64();
                if (prof) {
                    const long long c1 = clock64();
                    cyc[ph][1] += c1 - c0;
                    c0 = c1;
                    if (__any_sync(0xffffffffu, hit0)) ++hits[ph][0];
                }
                if (dflags & (1 | 32)) continue;
                if (dflags & 256) {
                    if (fminf(min32(r0), min32(r1)) < st.thr) st.cnt += 1;
                    continue;
                }
                if (hit0) apply64<KT>(h0, col_base, st, k, out, cap);
                {   // what the row's other three threads have learnt (own entry included: harmless)
                    float t0_, t1_, t2_, t3_;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(t0_), "=f"(t1_), "=f"(t2_), "=f"(t3_) : "r"(e_peer) : "memory");
                    st.thr = fminf(st.thr, fminf(fminf(t0_, t1_), fminf(t2_, t3_)));
                }
                if ((dflags & 4096) && st.T != INFINITY) {   // timing experiment: no masks / appends for the second batch either
                    Hit64 h1;
                    h1.m0 = min32(r0);
                    h1.m1 = min32(r1);
                    h1.mask0 = h1.mask1 = 0u;
                    if (fminf(h1.m0, h1.m1) < st.thr) apply64<KT>(h1, col_base + 128, st, k, out, cap);
                } else if (prof) {
                    Hit64 h1;
                    const bool hit1 = scan64<KT>(r0, r1, col_base + 128, st, k, out, cap, h1);
                    if (hit1) apply64<KT>(h1, col_base + 128, st, k, out, cap);
                    if (__any_sync(0xffffffffu, hit1)) ++hits[ph][1];
                    cyc[ph][2] += clock64() - c0;
                } else {
                    process64<KT>(r0, r1, col_base + 128, st, k, out, cap);
                }
                if (kTraceBuild && etr_on) etr[eti][4] = clock64();
            }
            if (kTraceBuild && etrace && lane == 0)
                for (int i = 0; i < kTraceTiles / 2; ++i) {
                    const int tile = kTraceTile0 + 2 * i + ((bsel ^ (kTraceTile0 & 1)) & 1);
                    if (tile < t1 - t0)
                        printf("b200match trace epi cta %d warp %d buf %d half %d tile %d: %lld %lld %lld %lld %lld\n", blockIdx.x, warp, bsel,
                               half, tile, etr[i][0], etr[i][1], etr[i][2], etr[i][3], etr[i][4]);
                }
            if (prof && lane == 0 && blockIdx.x < 2 && blockIdx.y == 0)
                printf("b200match epi-prof cta %d warp %2d (buf %d half %d) tiles<64: wait %lld chain %lld after %lld hits %d/%d | rest: "
                       "wait %lld chain %lld after %lld hits %d/%d of %d batches each\n", blockIdx.x, warp, bsel, half, cyc[0][0],
                       cyc[0][1], cyc[0][2], hits[0][0], hits[0][1], cyc[1][0], cyc[1][1], cyc[1][2], hits[1][0], hits[1][1],
                       (t1 - t0 - 64) / 2);
        } else {
        uint32_t r0[32], r1[32], r2[32], r3[32];
        long long c_wait = 0, c_ld = 0, c_fast = 0, c_slow = 0;   // B200M_TC_DEBUG & 512: where this warp's cycles go
        int n_slow = 0;
        const bool prof = (dflags & 512) != 0;
        // first train row of this warp's columns in the current tile, and where its upper 64 columns continue
        int col_base = t0 * B200M_TILE_N + half * (SPLITN ? 64 : kColsPerWarp);
        const int col_hi = SPLITN ? 128 : 64;
        const bool trace = kTraceBuild && (dflags & 1024) && blockIdx.x < 2 && blockIdx.y == 0;
        long long tr[kTraceTiles][4];
        for (int lt = 0; lt < t1 - t0; ++lt, col_base += B200M_TILE_N) {
            const uint32_t buf = (uint32_t) lt & 1u;
            const int ti = lt - kTraceTile0;
            const bool tr_on = trace && ti >= 0 && ti < kTraceTiles;
            long long c0 = prof ? clock64() : 0;
            mbar_wait(e_tfull + acc_stride * buf, ((uint32_t) lt >> 1) & 1u);
            tc_fence_after();
            if (tr_on) tr[ti][0] = clock64();   // accumulators seen complete
            if (prof) { long long c1 = clock64(); c_wait += c1 - c0; c0 = c1; }
            const uint32_t taddr = e_tmem + buf * (uint32_t) B200M_TILE_N;
            // 128 columns at a time: four TMEM loads in flight, one wait.  The accumulator buffer goes back to the MMA
            // issuer as soon as this warp's last load has landed in registers -- the filtering below then overlaps the
            // MMAs of the tile after next instead of sitting on their critical path.
#pragma unroll 1
            for (int h = 0; h < kColsPerWarp / 128; ++h) {
                // timing experiments (with the fast-path-only flag 256): 131072 = the warps that share a scheduler with the
                // TMA producer / MMA issuer (quarters 0, 1) skip a quarter of their columns, 262144 = every warp does
                const bool skip4 = DBG && (((dflags & 131072) && quarter < 2) || (dflags & 262144));
                if (!(dflags & 1)) {
                    tmem_ld_32x32b_x32(taddr + (uint32_t) (h * 128), r0);
                    tmem_ld_32x32b_x32(taddr + (uint32_t) (h * 128 + 32), r1);
                    tmem_ld_32x32b_x32(taddr + (uint32_t) (h * 128 + 64), r2);
                    if (!skip4) tmem_ld_32x32b_x32(taddr + (uint32_t) (h * 128 + 96), r3);
                    tmem_ld_wait();
                }
                if (prof) { long long c1 = clock64(); c_ld += c1 - c0; c0 = c1; }
                if (tr_on && h == kColsPerWarp / 128 - 1) tr[ti][1] = clock64();   // last TMEM load landed
                if (h == kColsPerWarp / 128 - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (PAIR) mbar_arrive_cluster(e_tempty + acc_stride * buf);
                        else mbar_arrive(e_tempty + acc_stride * buf);
                    }
                }
                if (tr_on && h == kColsPerWarp / 128 - 1) tr[ti][2] = clock64();   // buffer handed back
                if (EH == 2) st.thr = fminf(st.thr, lds_f32(e_peer));   // pick up what the partner thread has learnt
                if (dflags & (1 | 32)) continue;
                if (dump) {   // debug: raw accumulators of this tile
                    float *d = dump + ((size_t) qtile * B200M_TILE_M + row_in_tile) * B200M_TILE_N +
                               half * (SPLITN ? 64 : kColsPerWarp) + h * 128;
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        d[i] = __uint_as_float(r0[i]);
                        d[32 + i] = __uint_as_float(r1[i]);
                        d[col_hi + i] = __uint_as_float(r2[i]);
                        d[col_hi + 32 + i] = __uint_as_float(r3[i]);
                    }
                }
                if (dflags & 256) {   // timing experiment: fast path only
                    float m = fminf(fminf(min32(r0), min32(r1)), min32(r2));
                    if (!skip4) m = fminf(m, min32(r3));
                    if (m < st.thr) st.cnt += 1;
                    if (tr_on) tr[ti][3] = clock64();
                    continue;
                }
                const float thr_before = st.thr;
                process128<KT, EH>(r0, r1, r2, r3, col_base + h * 128, col_hi, st, k, out, out_v, cap);
                if (tr_on) tr[ti][3] = clock64();   // filtering done
                if (prof) {
                    long long c1 = clock64();
                    const bool slow = __any_sync(0xffffffffu, st.thr != thr_before);
                    if (slow) { c_slow += c1 - c0; ++n_slow; } else c_fast += c1 - c0;
                    c0 = c1;
                }
            }
        }
        if (prof && lane == 0 && blockIdx.x < 2 && blockIdx.y == 0)
            printf("b200match epi-prof cta %d warp %d tiles %d: wait %lld ld %lld fast %lld slow %lld (entries that tightened: %d)\n",
                   blockIdx.x, warp, t1 - t0, c_wait, c_ld, c_fast, c_slow, n_slow);
        if (trace && lane == 0)
            for (int i = 0; i < kTraceTiles && kTraceTile0 + i < t1 - t0; ++i)
                printf("b200match trace epi cta %d warp %d tile %d: %lld %lld %lld %lld\n", blockIdx.x, warp, kTraceTile0 + i,
                       tr[i][0], tr[i][1], tr[i][2], tr[i][3]);
        }   // !ALT
        if ((dflags & 256) && st.cnt == -1) p.cand_cnt[0] = 0;   // keeps the experiment's arithmetic alive
        if (active && !dump) {
            p.cand_cnt[list_row] = st.cnt;
            if (EH == 1 || CHK) p.cand_thr[list_row] = st.thr;
        }
    }
    tc_fence_before();
    if (p.cluster > 1) cluster_sync_all();   // no peer may still multicast into, or arrive on, this CTA's shared memory
    else __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        if (PAIR)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// ---- host side ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct TmapCache {
    EncodeTiledFn encode = nullptr;
    struct Entry {
        const void *ptr = nullptr;
        size_t n_pad = 0;
        int kp = 0, box_rows = 0;
        CUtensorMap map;
    } e[4];   // [side][as_query]
};

int get_tmap(b200m_ctx *ctx, int side, bool as_query, int cluster, const CUtensorMap **out, const void *q_ops = nullptr,
             size_t q_pad = 0) {
    TmapCache *tc = static_cast<TmapCache *>(ctx->tmap_cache);
    if (!tc) {
        tc = new TmapCache();
        ctx->tmap_cache = tc;
    }
    if (!tc->encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
            return b200m_fail_msg(ctx, "cuTensorMapEncodeTiled is not available from the driver");
        tc->encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    Side &sd = ctx->side[side];
    const void *ptr = as_query ? (q_ops ? q_ops : sd.op_query.p) : sd.op_train.p;
    const size_t rows = as_query && q_ops ? q_pad : sd.n_pad;
    const int box_rows = as_query ? B200M_TILE_M : B200M_TILE_N / cluster;
    TmapCache::Entry &en = tc->e[side * 2 + (as_query ? 1 : 0)];
    if (en.ptr != ptr || en.n_pad != rows || en.kp != sd.kp || en.box_rows != box_rows) {
        cuuint64_t dims[2] = {(cuuint64_t) sd.kp, (cuuint64_t) rows};
        cuuint64_t strides[1] = {(cuuint64_t) sd.kp * 2};
        cuuint32_t box[2] = {64, (cuuint32_t) box_rows};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = tc->encode(&en.map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(ptr), dims, strides, box,
                                estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return b200m_fail_msg(ctx, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int) r));
        en.ptr = ptr;
        en.n_pad = rows;
        en.kp = sd.kp;
        en.box_rows = box_rows;
    }
    *out = &en.map;
    return 0;
}

template <int KT, bool PAIR, int EH, bool SPLITN, int EPI, bool DBG, bool SEG, bool KS = false, bool DP = false>
int launch_tc(b200m_ctx *ctx, const CUtensorMap *mq, const CUtensorMap *mt, const TcParams &p, dim3 grid, size_t smem) {
    CK(cudaFuncSetAttribute(tc_candidates_kernel<KT, PAIR, EH, SPLITN, EPI, DBG, SEG, KS, DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(EPI ? 640 : 64 + 128 * EH + (SPLITN ? 32 : 0), 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned) p.cluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, tc_candidates_kernel<KT, PAIR, EH, SPLITN, EPI, DBG, SEG, KS, DP>, *mq, *mt, p);
    if (e != cudaSuccess) {
        cudaGetLastError();   // do not leave the launch error behind for the next call
        return b200m_fail_msg(ctx, std::string("tc_candidates launch failed: ") + cudaGetErrorString(e) + " (grid " +
                                       std::to_string(grid.x) + "x" + std::to_string(grid.y) + ", cluster " +
                                       std::to_string(p.cluster) + ", pair " + std::to_string(p.pair) + ", smem " +
                                       std::to_string(smem) + ", stages " + std::to_string(p.stages) + ")");
    }
    return 0;
}

}  // namespace

// kp <= 640: the A-resident kernels (any mode); 640 < kp <= 2048 (dim <= 2045): the K-streamed kernel, which exists in
// pair mode only.  Everything else is answered on the exact path.
bool tc_supported(const b200m_ctx *ctx, int dim, int k) {
    int kp = (dim + B200M_AUG_COLS + 63) / 64 * 64;
    if (k > 16) return false;
    return kp / 64 <= kMaxKAtoms || (ctx->tc_pair && kp / 64 <= kMaxKAtomsStreamed);
}

void tc_release(b200m_ctx *ctx) {
    delete static_cast<TmapCache *>(ctx->tmap_cache);
    ctx->tmap_cache = nullptr;
}

int tc_candidates(b200m_ctx *ctx, int direction, size_t row_begin, size_t n_rows, int k, int cap_request,
                  int *n_lists_out, int *cap_out, int *has_values_out, float *dump, size_t dump_t_tile,
                  const void *q_ops, const float *q_norm, size_t q_pad, const SegTable *seg) {
    Side &q = ctx->side[direction], &t = ctx->side[1 - direction];
    const int n_qtiles = (int) ((n_rows + B200M_TILE_M - 1) / B200M_TILE_M);
    // Default = CTA-pair mode (cta_group::2): the two CTAs of a cluster form one M=256 MMA, each keeps its own 128
    // query rows and HALF of every train tile, so per SM the B stream (TMA writes and MMA reads of shared memory, and
    // L2->SM traffic) is halved -- a single-CTA M=128 x N=256 SS-mode MMA is shared-memory-bandwidth bound.
    // B200M_TC_MODE=mcast / B200M_TC_CLUSTER select the cta_group::1 path with TMA multicast (kept for comparison).
    int pair = ctx->tc_pair;
    int cluster = pair ? 2 : (ctx->tc_cluster > 0 ? ctx->tc_cluster : 2);
    const CUtensorMap *mq = nullptr, *mt = nullptr;
    if (get_tmap(ctx, direction, true, 1, &mq, q_ops, q_pad)) return 1;
    if (get_tmap(ctx, 1 - direction, false, cluster, &mt)) return 1;

    TcParams p{};
    p.cluster = cluster;
    p.pair = pair;
    p.ka = q.kp / 64;
    // long descriptors (kp > 640): the query tile does not fit next to a useful ring, both operands are streamed
    const bool ks = p.ka > kMaxKAtoms;
    if (ks && (!pair || p.ka > kMaxKAtomsStreamed)) return b200m_fail_msg(ctx, "tc_candidates: descriptor too long for this mode");
    p.stage_bytes = ks ? kATileBytes + kStageBytes / 2 : pair ? kStageBytes / 2 : kStageBytes;
    p.ksteps = (q.dim + B200M_AUG_COLS + 15) / 16;
    const size_t smem_limit = 227 * 1024;
    const size_t a_bytes = ks ? 0 : (size_t) p.ka * kATileBytes;   // the resident query tile
    const size_t fixed = a_bytes + 1024 /*alignment*/ + kTailBytes /*barriers + per-row shared state*/;
    int stages = (int) ((smem_limit - fixed) / p.stage_bytes);
    if (stages > kMaxStages) stages = kMaxStages;
    if ((ctx->tc_debug & 8) && stages > 4) stages = 4;     // timing experiment: shallow ring
    if ((ctx->tc_debug & 16) && stages > 6) stages = 6;
    if (stages < 2) return b200m_fail_msg(ctx, "tc_candidates: descriptor too long for the shared-memory pipeline");
    p.stages = stages;
    p.n_ttiles = (int) (t.n_pad / B200M_TILE_N);
    // tiles one query block sweeps: all of them, or (batch) those of the largest pair -- splits, list capacity and the
    // rotated sweep's default are chosen from this
    const int sweep_tiles = seg ? seg->max_tiles : p.n_ttiles;
    // Short descriptors (FPFH: 3 MMAs per tile) are bound by the epilogue's latency chain: two epilogue warps per
    // scheduler.  Long ones (SHOT: 23 MMAs per tile) hide a four-warp epilogue, and there a thread that owns its whole row
    // also records the accumulator values so that the re-rank can prune by the row's final threshold.
    int eh = p.ka <= 2 ? 2 : 1;
    if (ctx->tc_debug & 64) eh = 1;
    if ((ctx->tc_debug & 128) && !ks) eh = 2;
    // One-atom descriptors (FPFH) in pair mode with the full 12-stage ring: fully unrolled issue loop (B200M_TC_LEAN=0
    // falls back to the general loop).
    p.lean = (pair && p.ka == 1 && stages == kMaxStages && ctx->tc_lean != 0) ? 1 : 0;
    // split-N (two 128-column halves per accumulator, an issuer warp per half) for one-atom descriptors: C2 launch
    // 4.18 -> 3.92 ms; B200M_TC_SPLITN=0 selects the single N = 256 MMA per tile (comparison)
    const bool splitn = p.lean && eh == 2 && ctx->tc_splitn != 0 && !dump;
    // ... with sixteen epilogue warps of 64 accumulators each.  B200M_TC_ALT: 4 / 5 (default) alternating tiles with CHUNK
    // entries -- a list entry is a 32-column chunk and its minimum, the re-rank evaluates the surviving chunks' rows -- drained
    // by 32-column (4) or 16-column (5) TMEM loads; 1 alternating tiles, 2 quarter columns of every tile (both: column entries);
    // 0 eight warps of 128 accumulators, every warp on every tile.  (A third column-entry layout, hit chunks handed to a worker
    // warp through a shared-memory ring, was exact and slower -- profiles/r02_notes.md section 5 -- and is gone.)  Measured per
    // launch, same boxes (profiles/r02_cand_epilogue_modes.log, r02_cand_chunk_entries.log): C2 k = 2 -- 4.10 (0) / 3.75 (1) /
    // 3.85 (2) / 3.08 (4) / 3.03 ms (5); C4 k = 5 -- 492 (0) / 530 (1) / 438 (2) / 398 (4) / 459 ms (5: spills at KT = 8).
    const int alt_pick = ctx->tc_alt >= 0 ? ctx->tc_alt : (k <= 2 ? 5 : 4);
    const int epi = splitn ? (alt_pick == 1 ? 1 : alt_pick == 4 ? 4 : alt_pick == 5 ? 5 : alt_pick != 0 ? 2 : 0) : 0;
    const bool alt = epi != 0;
    const int lists_per_split = eh * (alt ? 2 : 1);
    int n_splits = 1;
    if (!dump) {
        // Train splits balance the waves of CTAs: a (cluster of) query tile(s) is a work unit that occupies its SMs for
        // the whole sweep, so e.g. 245 units on 74 cluster slots run 4 waves at 83 % -- three splits run 10 waves at 99 %.
        // Each split costs a CTA prologue (about 4 tiles' worth) and a candidate list of its own (about 2 % more work
        // downstream), and keeps at least 8 train tiles.
        const long long units = (n_qtiles + cluster - 1) / cluster, slots = ctx->sm_count / cluster > 0 ? ctx->sm_count / cluster : 1;
        int max_splits = sweep_tiles / 8 > 0 ? sweep_tiles / 8 : 1;
        if (max_splits > kMaxLists) max_splits = kMaxLists;
        if (max_splits * lists_per_split > 32) max_splits = 32 / lists_per_split;   // the re-rank reads at most 32 lists per row
        double best = 0;
        for (int sp = 1; sp <= max_splits; ++sp) {
            const long long waves = (units * sp + slots - 1) / slots;
            const double cost = (double) waves * ((sweep_tiles + sp - 1) / sp + 4) * (1.0 + 0.02 * (sp - 1));
            if (sp == 1 || cost < best) { best = cost; n_splits = sp; }
        }
        if (ctx->tc_splits > 0) n_splits = ctx->tc_splits < max_splits ? ctx->tc_splits : max_splits;   // B200M_TC_SPLITS: tuning override
    }
    p.tiles_per_split = (sweep_tiles + n_splits - 1) / n_splits;
    n_splits = (sweep_tiles + p.tiles_per_split - 1) / p.tiles_per_split;
    p.seg_range = seg && !dump ? seg->range : nullptr;
    p.q_row0 = (int) row_begin;
    p.n_rows = (int) n_rows;
    p.k = k;
    p.dim = q.dim;
    p.bmax = ctx->prep.max_norm[1 - direction];
    // device prepare (batch plans): the bound and the routing come from the device; only the SEG kernels have the DP form
    const bool dp = ctx->device_prepare;
    if (dp && (!seg || dump)) return b200m_fail_msg(ctx, "tc_candidates: device prepare is a batch form");
    p.prep = dp ? ctx->prep.red.as<PrepDev>() : nullptr;
    p.train_side = 1 - direction;
    p.q_norm16 = q_ops ? q_norm : q.norm16.as<float>();
    // A list receives a column whenever it is under the running threshold: for columns in random order that is a
    // record process, E = k (ln(n / k) + 1) appends with variance about E, n = the columns the list's thread sees.
    // cap = E + 8 sqrt(E) + 16 puts an overflow beyond 8 sigma; overflowed rows (adversarial column orders) are
    // still answered exactly, by the CUDA-core fallback.
    int cap = cap_request;
    if (cap <= 0) {
        const double n_list = (double) p.tiles_per_split * B200M_TILE_N / lists_per_split;
        const double expect = k * (log(fmax(n_list / k, 2.0)) + 1.0);
        cap = (int) (expect + 8.0 * sqrt(expect) + 16.0);
        cap = (cap + 7) / 8 * 8;
    }
    if (cap < k) cap = k;
    p.cap = cap;
    const int n_lists = n_splits * lists_per_split;
    CK(ctx->ws_cand_idx.reserve(sizeof(int32_t) * (size_t) n_lists * n_rows * (size_t) cap));
    CK(ctx->ws_cand_cnt.reserve(sizeof(int32_t) * (size_t) n_lists * n_rows));
    p.cand_idx = ctx->ws_cand_idx.as<int32_t>();
    p.cand_cnt = ctx->ws_cand_cnt.as<int32_t>();
    p.cand_val = nullptr;
    p.cand_thr = nullptr;
    if (eh == 1 || epi >= 4) {
        CK(ctx->ws_cand_val.reserve(sizeof(float) * (size_t) n_lists * n_rows * (size_t) cap));
        CK(ctx->ws_cand_thr.reserve(sizeof(float) * (size_t) n_lists * n_rows));
        p.cand_val = ctx->ws_cand_val.as<float>();
        p.cand_thr = ctx->ws_cand_thr.as<float>();
    }
    // 0: column entries without values; 1: column entries + accumulator values + final thresholds (the re-rank prunes);
    // 2: CHUNK entries (first train row of a 32-row chunk, chunk minimum) + final thresholds
    *has_values_out = epi >= 4 ? 2 : eh == 1 ? 1 : 0;
    p.dump = dump;
    CK(ctx->ws_sweep_hint.reserve(sizeof(int) * 64));   // per launch: the front runner's progress starts at zero
    if (epi >= 4) CK(cudaMemsetAsync(ctx->ws_sweep_hint.p, 0, sizeof(int) * 64, ctx->stream));
    // default: rotate when the train operands do NOT fit L2 (C4: 256 MB; measured 417 -> 372 ms per launch with 16-24 tiles
    // between followers, 8 and >= 48 are slower than no rotation; operands that fit L2 show no difference) --
    // profiles/r02_notes.md section 14.  B200M_TC_SWEEP_LAG overrides (0 = off).
    p.sweep_lag = ctx->tc_sweep_lag >= 0 ? ctx->tc_sweep_lag
                                         : ((size_t) sweep_tiles * B200M_TILE_N * (size_t) t.kp * 2 > (size_t) 96 << 20 ? 20 : 0);
    p.sweep_hint = ctx->ws_sweep_hint.as<int>();
    p.debug_flags = ctx->tc_debug;
    if (dump) p.tiles_per_split = (int) dump_t_tile;
    const size_t smem = a_bytes + (size_t) stages * p.stage_bytes + 1024 + kTailBytes;
    dim3 grid((unsigned) (dump ? cluster : (n_qtiles + cluster - 1) / cluster * cluster), (unsigned) n_splits, 1);
    int kt = k <= 1 ? 1 : k <= 2 ? 2 : k <= 4 ? 4 : k <= 8 ? 8 : 16;
    int rc;
    // batch launches (p.seg_range) run the production kernels with the segment lookup: the timing experiments of
    // B200M_TC_DEBUG do not apply to them, and dump mode is single-pair only
    const bool dbg = dump != nullptr || ctx->tc_debug != 0;
#define B200M_TC_CASE2(KT_, DBG_, SEG_, DP_)                                                                     \
    rc = pair ? (eh == 2 ? (epi == 5 ? launch_tc<KT_, true, 2, true, 5, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem)   \
                            : epi == 4 ? launch_tc<KT_, true, 2, true, 4, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem) \
                            : epi == 2 ? launch_tc<KT_, true, 2, true, 2, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem) \
                            : epi == 1 ? launch_tc<KT_, true, 2, true, 1, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem) \
                            : splitn ? launch_tc<KT_, true, 2, true, 0, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem)   \
                                     : launch_tc<KT_, true, 2, false, 0, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem)) \
                         : launch_tc<KT_, true, 1, false, 0, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem))             \
              : (eh == 2 ? launch_tc<KT_, false, 2, false, 0, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem)             \
                         : launch_tc<KT_, false, 1, false, 0, DBG_, SEG_, false, DP_>(ctx, mq, mt, p, grid, smem))
#define B200M_TC_CASE_KS(KT_)                                                                                  \
    if (p.seg_range && dp) rc = launch_tc<KT_, true, 1, false, 0, false, true, true, true>(ctx, mq, mt, p, grid, smem); \
    else if (p.seg_range) rc = launch_tc<KT_, true, 1, false, 0, false, true, true>(ctx, mq, mt, p, grid, smem);   \
    else if (dbg) rc = launch_tc<KT_, true, 1, false, 0, true, false, true>(ctx, mq, mt, p, grid, smem);           \
    else rc = launch_tc<KT_, true, 1, false, 0, false, false, true>(ctx, mq, mt, p, grid, smem);
#define B200M_TC_CASE(KT_)                                         \
    if (ks) { B200M_TC_CASE_KS(KT_) }                                 \
    else if (p.seg_range && dp) { B200M_TC_CASE2(KT_, false, true, true); } \
    else if (p.seg_range) { B200M_TC_CASE2(KT_, false, true, false); } \
    else if (dbg) { B200M_TC_CASE2(KT_, true, false, false); }        \
    else { B200M_TC_CASE2(KT_, false, false, false); }
    switch (kt) {
        case 1: B200M_TC_CASE(1); break;
        case 2: B200M_TC_CASE(2); break;
        case 4: B200M_TC_CASE(4); break;
        case 8: B200M_TC_CASE(8); break;
        default: B200M_TC_CASE(16); break;
    }
#undef B200M_TC_CASE
#undef B200M_TC_CASE_KS
#undef B200M_TC_CASE2
    if (rc) return rc;
    ctx->stats.launches += 1;
    ctx->stats.candidate_launches += 1;
    *n_lists_out = n_lists;
    *cap_out = cap;
    return 0;
}
