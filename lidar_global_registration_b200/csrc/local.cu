// local.cu -- matchLocal with a finite match_search_radius (reference include/matching.h:637-678) over a CELL LIST of the
// train keypoints, instead of testing the 3-D gate against every train row for every query.
//
// The reference asks a kd-tree for the train keypoints within match_search_radius of the (guess-transformed) query keypoint
// (pcd_tree->radiusSearch, :659-661) and runs pcl::L2_Norm over the descriptors of those rows only (:663-668).  Here the
// train keypoints are binned once into a uniform grid whose cells are at least one radius wide (counting sort: histogram,
// scan, scatter -- all on the device), and a warp per query row walks the 27 cells around its keypoint: the same FP32 gate
// (FLANN's L2_Simple squared distance < radius^2), the same sequential FP32 descriptor distance, the same order
// (descriptor distance, spatial distance, index) as the brute-force gate kernel in exact.cu, which stays as the path for
// radii that cover most of the cloud.  Work per query drops from Nt gate tests to the population of 27 cells.
//
// The batch form (launch_local_cells_batch, used by b200m_match_multiscale_local_batch) bins every pair's train keypoints
// into that pair's own grid: one launch sequence per scale and direction for all pairs, no host round trip (DESIGN.md
// section 3.13).
//
// This is deliberately NOT a tensor-core path: the gate is a per-pair predicate, and a column that fails it must not
// tighten a row's running threshold -- the candidate kernel's epilogue would have to evaluate a 3-D distance per
// accumulator, which costs more than the distance itself at these candidate counts (DESIGN.md section 3.10).
#include <limits.h>
#include <math.h>
#include <string.h>

#include <algorithm>

#include "internal.cuh"

namespace {

constexpr int kMaxCellsPerAxis = 256;
constexpr int kLocalWarps = 8;

struct Grid {
    float ox, oy, oz;    // origin (bounding-box minimum of the finite train keypoints)
    float inv;           // 1 / cell edge
    int nx, ny, nz;
};

struct SegGrid {           // a batch pair's grid: its cells are [cell0, cell0 + nx * ny * nz) of the batch's cell table
    Grid g;
    long long cell0;
};

__device__ __forceinline__ int cell_coord(float v, float o, float inv, int n) {
    const float c = floorf((v - o) * inv);
    // keypoints outside the box (queries only) are clamped one cell beyond it, where nothing is stored
    return c < -1.f ? -2 : c > (float) n ? n + 1 : (int) c;
}

// bounding box of the finite train keypoints: per-block min/max, folded by atomics on ordered integers
__device__ __forceinline__ int f2ord(float f) {
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

__global__ void bbox_kernel(const float *__restrict__ xyz, size_t stride, size_t n, int *__restrict__ box /*[6] min xyz, max xyz*/) {
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        const float *p = xyz + i * stride;
        if (isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2])) {
#pragma unroll
            for (int a = 0; a < 3; ++a) { lo[a] = fminf(lo[a], p[a]); hi[a] = fmaxf(hi[a], p[a]); }
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(box + a, f2ord(lo[a]));
            atomicMax(box + 3 + a, f2ord(hi[a]));
        }
    }
}

__device__ __forceinline__ long long train_cell(const Grid &g, const float *p) {
    if (!(isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]))) return -1;   // can never pass the gate
    int cx = cell_coord(p[0], g.ox, g.inv, g.nx), cy = cell_coord(p[1], g.oy, g.inv, g.ny), cz = cell_coord(p[2], g.oz, g.inv, g.nz);
    cx = min(max(cx, 0), g.nx - 1);   // the maximum corner falls on the upper edge
    cy = min(max(cy, 0), g.ny - 1);
    cz = min(max(cz, 0), g.nz - 1);
    return ((long long) cz * g.ny + cy) * g.nx + cx;
}

// SEG (batch): row i is filed in its pair's grid (block_pair[i / 256] -> grids[pair]) and cell table
template <bool SEG>
__global__ void cell_count_kernel(Grid g0, const float *__restrict__ xyz, size_t stride, const uint8_t *__restrict__ valid, size_t n,
                                  int *__restrict__ counts, const SegGrid *__restrict__ grids = nullptr,
                                  const int32_t *__restrict__ block_pair = nullptr) {
    const size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !valid[i]) return;
    Grid g = g0;
    if constexpr (SEG) {
        const SegGrid &sg = grids[block_pair[i / B200M_TILE_N]];
        g = sg.g;
        counts += sg.cell0;
    }
    const long long c = train_cell(g, xyz + i * stride);
    if (c >= 0) atomicAdd(counts + c, 1);
}

// exclusive scan of `counts` (n_cells entries) into `starts` (n_cells + 1), single CTA.
// SEG (batch): CTA p scans pair p's cells, which start at cell_base(p); its starts begin at the pair's first train row.
template <bool SEG>
__global__ void __launch_bounds__(1024) cell_scan_kernel(const int *__restrict__ counts, size_t n_cells, int *__restrict__ starts,
                                                         const SegGrid *__restrict__ grids = nullptr,
                                                         const int4 *__restrict__ rows = nullptr, int t_side = 0) {
    __shared__ int wsum[32];
    __shared__ int carry;
    if constexpr (SEG) {
        const SegGrid &sg = grids[blockIdx.x];
        counts += sg.cell0;
        starts += sg.cell0;
        n_cells = (size_t) sg.g.nx * sg.g.ny * sg.g.nz;
        if (threadIdx.x == 0) carry = t_side ? rows[blockIdx.x].z : rows[blockIdx.x].x;
    } else {
        if (threadIdx.x == 0) carry = 0;
    }
    __syncthreads();
    for (size_t base = 0; base < n_cells; base += 1024) {
        const size_t i = base + threadIdx.x;
        const int v = i < n_cells ? counts[i] : 0;
        int x = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if ((threadIdx.x & 31) >= o) x += y;
        }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = x;
        __syncthreads();
        if (threadIdx.x < 32) {
            int w = wsum[threadIdx.x];
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, w, o);
                if ((int) threadIdx.x >= o) w += y;
            }
            wsum[threadIdx.x] = w;
        }
        __syncthreads();
        const int before = carry + ((threadIdx.x >> 5) ? wsum[(threadIdx.x >> 5) - 1] : 0) + x - v;
        if (i < n_cells) starts[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) starts[n_cells] = carry;
}

template <bool SEG>
__global__ void cell_fill_kernel(Grid g0, const float *__restrict__ xyz, size_t stride, const uint8_t *__restrict__ valid, size_t n,
                                 const int *__restrict__ starts, int *__restrict__ cursor, int32_t *__restrict__ rows,
                                 const SegGrid *__restrict__ grids = nullptr, const int32_t *__restrict__ block_pair = nullptr) {
    const size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !valid[i]) return;
    Grid g = g0;
    if constexpr (SEG) {
        const SegGrid &sg = grids[block_pair[i / B200M_TILE_N]];
        g = sg.g;
        starts += sg.cell0;
        cursor += sg.cell0;
    }
    const long long c = train_cell(g, xyz + i * stride);
    if (c >= 0) rows[starts[c] + atomicAdd(cursor + c, 1)] = (int32_t) i;
}

__device__ __forceinline__ float seq_sqdist_s(const float *__restrict__ q, const float *__restrict__ t, int dp) {
    float s = 0.f;   // the reference's sequential chain (pcl::L2_Norm): separate roundings, no FMA
    const float4 *t4 = reinterpret_cast<const float4 *>(t);
    for (int c = 0; c < dp / 4; ++c) {
        const float4 v = __ldg(t4 + c);
        const float d0 = __fsub_rn(q[4 * c + 0], v.x);
        s = __fadd_rn(s, __fmul_rn(d0, d0));
        const float d1 = __fsub_rn(q[4 * c + 1], v.y);
        s = __fadd_rn(s, __fmul_rn(d1, d1));
        const float d2 = __fsub_rn(q[4 * c + 2], v.z);
        s = __fadd_rn(s, __fmul_rn(d2, d2));
        const float d3 = __fsub_rn(q[4 * c + 3], v.w);
        s = __fadd_rn(s, __fmul_rn(d3, d3));
    }
    return s;
}
__device__ __forceinline__ bool lex3(float d1, float s1, int i1, float d2, float s2, int i2) {
    return d1 < d2 || (d1 == d2 && (s1 < s2 || (s1 == s2 && i1 < i2)));
}

// one warp per query row: the query descriptor in the warp's shared slab, lanes stride over the rows of the 27 cells
// SEG (batch): the query row's grid is its pair's (q_block_pair[row / 256] -> grids[pair]); `rows` holds global train rows.
template <int KMAX, bool SEG>
__global__ void __launch_bounds__(kLocalWarps * 32)
local_cells_kernel(Grid g, const float *__restrict__ q_f32, const uint8_t *__restrict__ q_valid, int dp,
                   const float *__restrict__ t_f32, long long t_off, size_t n_rows, const float *__restrict__ q_xyz,
                   const float *__restrict__ t_xyz, size_t stride, float r2, int k, const int *__restrict__ starts,
                   const int32_t *__restrict__ rows, int32_t *__restrict__ idx, float *__restrict__ dist, int32_t *__restrict__ count,
                   const SegGrid *__restrict__ grids = nullptr, const int32_t *__restrict__ q_block_pair = nullptr,
                   const int *__restrict__ seg_starts = nullptr) {
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *sq = smem + (size_t) warp * dp;
    for (size_t qi = (size_t) blockIdx.x * kLocalWarps + warp; qi < n_rows; qi += (size_t) gridDim.x * kLocalWarps) {
        if constexpr (SEG) {   // g and starts are this row's pair's
            const SegGrid &sg = grids[q_block_pair[qi / B200M_TILE_N]];
            g = sg.g;
            starts = seg_starts + sg.cell0;
        }
        int32_t *oi = idx + qi * k;
        float *od = dist + qi * k;
        const float ax = q_xyz[qi * stride], ay = q_xyz[qi * stride + 1], az = q_xyz[qi * stride + 2];
        if (!q_valid[qi] || !(isfinite(ax) && isfinite(ay) && isfinite(az))) {   // non-finite query -> empty entry (:658)
            for (int m = lane; m < k; m += 32) { oi[m] = -1; od[m] = 0.f; }
            if (lane == 0) count[qi] = 0;
            continue;
        }
        __syncwarp();
        for (int d = lane; d < dp; d += 32) sq[d] = q_f32[qi * (size_t) dp + d];
        __syncwarp();
        float ld[KMAX], ls[KMAX];
        int li[KMAX];
#pragma unroll
        for (int m = 0; m < KMAX; ++m) { ld[m] = INFINITY; ls[m] = INFINITY; li[m] = INT_MAX; }
        const int cx = cell_coord(ax, g.ox, g.inv, g.nx), cy = cell_coord(ay, g.oy, g.inv, g.ny), cz = cell_coord(az, g.oz, g.inv, g.nz);
        for (int z = max(cz - 1, 0); z <= min(cz + 1, g.nz - 1); ++z)
            for (int y = max(cy - 1, 0); y <= min(cy + 1, g.ny - 1); ++y) {
                const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.nx - 1);
                if (x1 < x0) continue;
                // the (up to three) cells of a row of the grid are contiguous in the sorted list
                const size_t c0 = ((size_t) z * g.ny + y) * g.nx;
                for (int e = starts[c0 + x0] + lane; e < starts[c0 + x1 + 1]; e += 32) {
                    const int j = rows[e];
                    const float *b = t_xyz + (size_t) j * stride;
                    const float dx = __fsub_rn(ax, b[0]), dy = __fsub_rn(ay, b[1]), dz = __fsub_rn(az, b[2]);
                    const float s = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
                    if (!(s < r2)) continue;
                    float cd = __fsqrt_rn(seq_sqdist_s(sq, t_f32 + (size_t) j * dp, dp));
                    float cs = s;
                    int ci = j;
                    if (lex3(cd, cs, ci, ld[KMAX - 1], ls[KMAX - 1], li[KMAX - 1])) {
#pragma unroll
                        for (int m = 0; m < KMAX; ++m) {
                            if (lex3(cd, cs, ci, ld[m], ls[m], li[m])) {
                                const float td = ld[m], tsp = ls[m];
                                const int ti = li[m];
                                ld[m] = cd; ls[m] = cs; li[m] = ci;
                                cd = td; cs = tsp; ci = ti;
                            }
                        }
                    }
                }
            }
        // k rounds of warp arg-min over the per-lane list heads
        int head = 0, found = 0;
        for (int round = 0; round < k; ++round) {
            float hd = INFINITY, hs = INFINITY;
            int hi = INT_MAX;
#pragma unroll
            for (int m = 0; m < KMAX; ++m)
                if (m == head) { hd = ld[m]; hs = ls[m]; hi = li[m]; }
            float bd = hd, bs = hs;
            int bi = hi, bl = lane;
            for (int o = 16; o > 0; o >>= 1) {
                const float od2 = __shfl_xor_sync(0xffffffffu, bd, o), os2 = __shfl_xor_sync(0xffffffffu, bs, o);
                const int oi2 = __shfl_xor_sync(0xffffffffu, bi, o), ol2 = __shfl_xor_sync(0xffffffffu, bl, o);
                if (lex3(od2, os2, oi2, bd, bs, bi)) { bd = od2; bs = os2; bi = oi2; bl = ol2; }
            }
            if (bi == INT_MAX) break;
            if (lane == bl) head++;
            if (lane == 0) { oi[round] = (int32_t) ((long long) bi + t_off); od[round] = bd; }
            found = round + 1;
        }
        for (int m = found + lane; m < k; m += 32) { oi[m] = -1; od[m] = 0.f; }
        if (lane == 0) count[qi] = found;
    }
}

// ---- batch form: every pair in its own grid (launch_local_cells_batch) ----------------------------------------------------
// One xyz row per padded descriptor row of both sides of one scale: query rows [0, n_q), then train rows [n_q, n_q + n_t).
// A row's keypoint is found through its pair (block table), its side's index map and the pair's first keypoint; gap rows
// and out-of-range map entries (flagged) get NaN, so they can never pass the gate.  Also resets the per-pair boxes.
__global__ void seg_gather_kernel(size_t n_q, size_t n_t, int q_side, int scale, int n_pairs, const int4 *__restrict__ rows,
                                  const int32_t *__restrict__ q_blk, const int32_t *__restrict__ t_blk,
                                  const int32_t *__restrict__ q_map, const int32_t *__restrict__ t_map,
                                  const int32_t *__restrict__ q_kp_off, const int32_t *__restrict__ t_kp_off,
                                  const float *__restrict__ q_xyz, const float *__restrict__ t_xyz, size_t stride,
                                  float4 *__restrict__ out, int *__restrict__ box, unsigned long long *__restrict__ bad) {
    const size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (size_t) n_pairs * 6) box[i] = i % 6 < 3 ? INT_MAX : INT_MIN;
    if (i >= n_q + n_t) return;
    const bool tr = i >= n_q;
    const size_t row = tr ? i - n_q : i;
    const int side = tr ? 1 - q_side : q_side;
    const int p = (tr ? t_blk : q_blk)[row / B200M_TILE_N];
    const int4 r = rows[p];
    const long long r0 = side ? r.z : r.x, rn = side ? r.w : r.y;
    float4 v = make_float4(NAN, NAN, NAN, NAN);
    if ((long long) row - r0 < rn) {
        const int32_t *off = tr ? t_kp_off : q_kp_off;
        const long long kp = (tr ? t_map : q_map)[row], n_kp = off[p + 1] - off[p];
        if (kp < 0 || kp >= n_kp) {
            flag_bad(bad, scale, p, side);
        } else {
            const float *x = (tr ? t_xyz : q_xyz) + (size_t) (off[p] + kp) * stride;
            v = make_float4(x[0], x[1], x[2], 0.f);
        }
    }
    out[i] = v;
}

// box of the finite train keypoints per pair: CTA b = train block b, which lies inside one pair
__global__ void __launch_bounds__(256) seg_bbox_kernel(const float4 *__restrict__ xyz, const int32_t *__restrict__ t_blk,
                                                       int *__restrict__ box) {
    __shared__ float red[8][6];
    const float4 v = xyz[(size_t) blockIdx.x * B200M_TILE_N + threadIdx.x];
    const bool fin = isfinite(v.x) && isfinite(v.y) && isfinite(v.z);
    float m[6] = {fin ? v.x : INFINITY, fin ? v.y : INFINITY, fin ? v.z : INFINITY,
                  fin ? v.x : -INFINITY, fin ? v.y : -INFINITY, fin ? v.z : -INFINITY};
#pragma unroll
    for (int a = 0; a < 6; ++a)
        for (int o = 16; o > 0; o >>= 1) {
            const float w = __shfl_xor_sync(0xffffffffu, m[a], o);
            m[a] = a < 3 ? fminf(m[a], w) : fmaxf(m[a], w);
        }
    if ((threadIdx.x & 31) == 0)
        for (int a = 0; a < 6; ++a) red[threadIdx.x >> 5][a] = m[a];
    __syncthreads();
    if (threadIdx.x < 6) {
        const int a = threadIdx.x;
        float x = red[0][a];
        for (int w = 1; w < 8; ++w) x = a < 3 ? fminf(x, red[w][a]) : fmaxf(x, red[w][a]);
        int *b = box + 6 * t_blk[blockIdx.x] + a;
        if (a < 3) atomicMin(b, f2ord(x)); else atomicMax(b, f2ord(x));
    }
}

// CTA p: pair p's grid from its box -- cells at least radius * (1 + 1e-4) wide (the 27 cells around a keypoint cover its
// ball), at most kMaxCellsPerAxis per axis, and at most as many cells as the pair has padded train rows (its share of the
// cell table, sized on the host from the row counts alone) -- then zeroes the pair's cell counters.
__global__ void __launch_bounds__(256) seg_grid_kernel(const int *__restrict__ box, const int4 *__restrict__ rows, int t_side,
                                                       float radius, SegGrid *__restrict__ grids, int *__restrict__ counts,
                                                       int *__restrict__ cursor) {
    __shared__ SegGrid sg;
    const int p = blockIdx.x;
    if (threadIdx.x == 0) {
        const int4 r = rows[p];
        const long long budget = (long long) ((t_side ? r.w : r.y) + B200M_TILE_N - 1) / B200M_TILE_N * B200M_TILE_N;
        Grid g{0.f, 0.f, 0.f, 0.f, 1, 1, 1};   // one cell (inv = 0): no finite train keypoint, or a ball that covers the cloud
        float lo[3], hi[3];
        for (int a = 0; a < 3; ++a) { lo[a] = ord2f(box[6 * p + a]); hi[a] = ord2f(box[6 * p + 3 + a]); }
        if (budget == 0) {
            g.nx = g.ny = g.nz = 0;
        } else if (hi[0] >= lo[0]) {
            g.ox = lo[0]; g.oy = lo[1]; g.oz = lo[2];
            float cell = fabsf(radius) * 1.0001f;
            for (int a = 0; a < 3; ++a) cell = fmaxf(cell, (hi[a] - lo[a]) / (float) kMaxCellsPerAxis);
            for (;;) {
                const float inv = 1.f / cell;
                if (!(inv < INFINITY)) break;   // radius 0 (or below FLT_MIN) and a one-point cloud
                const int nx = (int) floorf((hi[0] - lo[0]) * inv) + 1, ny = (int) floorf((hi[1] - lo[1]) * inv) + 1,
                          nz = (int) floorf((hi[2] - lo[2]) * inv) + 1;
                if ((long long) nx * ny * nz <= budget) {
                    g.inv = inv; g.nx = nx; g.ny = ny; g.nz = nz;
                    break;
                }
                cell *= 1.25f;
            }
        }
        sg.g = g;
        sg.cell0 = (long long) (t_side ? r.z : r.x) + p;   // pair p's cells follow the padded rows + 1 of the pairs before it
        grids[p] = sg;
    }
    __syncthreads();
    const long long n = (long long) sg.g.nx * sg.g.ny * sg.g.nz;
    for (long long c = threadIdx.x; c < n; c += blockDim.x) {
        counts[sg.cell0 + c] = 0;
        cursor[sg.cell0 + c] = 0;
    }
}

struct LocalState {
    DevBuf box, counts, starts, cursor, rows;
    DevBuf seg_xyz, seg_grids;   // batch form: gathered coordinates (query rows, then train rows), box + grid per pair
};

}  // namespace

void local_release(b200m_ctx *ctx) {
    LocalState *ls = static_cast<LocalState *>(ctx->local);
    if (!ls) return;
    DevBuf *b[] = {&ls->box, &ls->counts, &ls->starts, &ls->cursor, &ls->rows, &ls->seg_xyz, &ls->seg_grids};
    for (DevBuf *x : b) x->release();
    delete ls;
    ctx->local = nullptr;
}

// Returns 0 when the cell-list path ran, 1 on error, 2 when the radius is too large for a grid to pay (the caller then
// runs the brute-force gate kernel).
int launch_local_cells(b200m_ctx *ctx, int direction, const float *d_query_xyz, const float *d_train_xyz, size_t xyz_stride_bytes,
                       float radius, int k, int32_t *d_idx, float *d_dist, int32_t *d_count) {
    Side &q = ctx->side[direction], &t = ctx->side[1 - direction];
    if (!(radius > 0.f) || !isfinite(radius) || t.n < (size_t) ctx->local_min_rows || t.n >= (size_t) INT_MAX) return 2;
    if (!ctx->local) ctx->local = new LocalState();
    LocalState *ls = static_cast<LocalState *>(ctx->local);
    cudaStream_t st = ctx->stream;
    const size_t stride = xyz_stride_bytes / 4;
    CK(ls->box.reserve(32));
    const int init[6] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN};
    CK(cudaMemcpyAsync(ls->box.p, init, sizeof(init), cudaMemcpyHostToDevice, st));
    bbox_kernel<<<ctx->sm_count * 2, 256, 0, st>>>(d_train_xyz, stride, t.n, ls->box.as<int>());
    CK(cudaGetLastError());
    int box[6];
    CK(cudaMemcpyAsync(box, ls->box.p, sizeof(box), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));   // the grid's shape decides the launch geometry (one host round trip)
    ctx->stats.launches += 1;
    auto ord2f_h = [](int i) { int j = i >= 0 ? i : i ^ 0x7fffffff; float f; memcpy(&f, &j, 4); return f; };
    float lo[3], hi[3];
    for (int a = 0; a < 3; ++a) { lo[a] = ord2f_h(box[a]); hi[a] = ord2f_h(box[3 + a]); }
    if (!(hi[0] >= lo[0])) return 2;   // no finite train keypoint
    // cells at least one radius wide (so the 27 cells around a keypoint cover its ball), at most kMaxCellsPerAxis per axis
    float cell = radius * 1.0001f;
    for (int a = 0; a < 3; ++a) cell = fmaxf(cell, (hi[a] - lo[a]) / (float) kMaxCellsPerAxis);
    Grid g;
    g.ox = lo[0]; g.oy = lo[1]; g.oz = lo[2];
    g.inv = 1.f / cell;
    g.nx = (int) floorf((hi[0] - lo[0]) * g.inv) + 1;
    g.ny = (int) floorf((hi[1] - lo[1]) * g.inv) + 1;
    g.nz = (int) floorf((hi[2] - lo[2]) * g.inv) + 1;
    const size_t n_cells = (size_t) g.nx * g.ny * g.nz;
    if (n_cells < 64) return 2;        // the ball covers most of the cloud: the plain gate kernel is as good
    CK(ls->counts.reserve(sizeof(int) * n_cells));
    CK(ls->cursor.reserve(sizeof(int) * n_cells));
    CK(ls->starts.reserve(sizeof(int) * (n_cells + 1)));
    CK(ls->rows.reserve(sizeof(int32_t) * t.n));
    CK(cudaMemsetAsync(ls->counts.p, 0, sizeof(int) * n_cells, st));
    CK(cudaMemsetAsync(ls->cursor.p, 0, sizeof(int) * n_cells, st));
    const unsigned nb = (unsigned) ((t.n + 255) / 256);
    cell_count_kernel<false><<<nb, 256, 0, st>>>(g, d_train_xyz, stride, t.valid.as<uint8_t>(), t.n, ls->counts.as<int>());
    cell_scan_kernel<false><<<1, 1024, 0, st>>>(ls->counts.as<int>(), n_cells, ls->starts.as<int>());
    cell_fill_kernel<false><<<nb, 256, 0, st>>>(g, d_train_xyz, stride, t.valid.as<uint8_t>(), t.n, ls->starts.as<int>(),
                                                ls->cursor.as<int>(), ls->rows.as<int32_t>());
    CK(cudaGetLastError());
    const size_t smem = sizeof(float) * (size_t) q.dp * kLocalWarps;
    size_t want = (q.n + kLocalWarps - 1) / kLocalWarps;
    const size_t cap = (size_t) ctx->sm_count * 8;
    const unsigned blocks = (unsigned) (want < cap ? want : cap);
    const float r2 = radius * radius;   // radiusSearch is handed radius * radius (FP32 product)
#define B200M_LOCALC_CASE(K)                                                                                                   \
    do {                                                                                                                       \
        if (smem > 48 * 1024) /* rows over 1536 floats */                                                                    \
            CK(cudaFuncSetAttribute(local_cells_kernel<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));   \
        local_cells_kernel<K, false><<<blocks, kLocalWarps * 32, smem, st>>>(                                                  \
            g, q.f32.as<float>(), q.valid.as<uint8_t>(), q.dp, t.f32.as<float>(), (long long) t.index_offset, q.n, d_query_xyz, \
            d_train_xyz, stride, r2, k, ls->starts.as<int>(), ls->rows.as<int32_t>(), d_idx, d_dist, d_count);                 \
        CK(cudaGetLastError());                                                                                                \
        ctx->stats.launches += 4;                                                                                              \
        return 0;                                                                                                              \
    } while (0)
    if (k <= 1) B200M_LOCALC_CASE(1);
    if (k <= 2) B200M_LOCALC_CASE(2);
    if (k <= 4) B200M_LOCALC_CASE(4);
    if (k <= 8) B200M_LOCALC_CASE(8);
    if (k <= 16) B200M_LOCALC_CASE(16);
    B200M_LOCALC_CASE(32);
#undef B200M_LOCALC_CASE
}

// The gated kNN of one scale and direction of a batch call for every pair at once (b200m_match_multiscale_local_batch):
// gather, per-pair boxes and grids, count, per-pair scan, fill, then a warp per query row in its pair's grid.  The launch
// count does not depend on the number of pairs and nothing goes back to the host.  Train indices are global padded rows.
int launch_local_cells_batch(b200m_ctx *ctx, const LocalBatch &a, int32_t *d_idx, float *d_dist, int32_t *d_count) {
    const int qs = a.direction, ts = 1 - a.direction;
    Side &q = ctx->side[qs], &t = ctx->side[ts];
    const size_t nq = q.n, nt = t.n;   // padded rows (stage_batch)
    if (!nq) return 0;
    if (!ctx->local) ctx->local = new LocalState();
    LocalState *ls = static_cast<LocalState *>(ctx->local);
    cudaStream_t st = ctx->stream;
    const size_t n_cells = nt + (size_t) a.n_pairs + 1;
    CK(ls->seg_xyz.reserve(sizeof(float4) * (nq + nt)));
    CK(ls->box.reserve(sizeof(int) * 6 * (size_t) a.n_pairs));
    CK(ls->seg_grids.reserve(sizeof(SegGrid) * (size_t) a.n_pairs));
    CK(ls->counts.reserve(sizeof(int) * n_cells));
    CK(ls->cursor.reserve(sizeof(int) * n_cells));
    CK(ls->starts.reserve(sizeof(int) * n_cells));
    CK(ls->rows.reserve(sizeof(int32_t) * (nt + 1)));
    float4 *xq = ls->seg_xyz.as<float4>(), *xt = xq + nq;
    const SegGrid *grids = ls->seg_grids.as<SegGrid>();
    const size_t stride = a.xyz_stride_bytes / 4;
    const size_t n_gather = std::max(nq + nt, (size_t) a.n_pairs * 6);
    seg_gather_kernel<<<(unsigned) ((n_gather + 255) / 256), 256, 0, st>>>(
        nq, nt, qs, a.scale, a.n_pairs, a.rows, a.blk[qs], a.blk[ts], a.map[qs], a.map[ts], a.kp_off[qs], a.kp_off[ts], a.q_xyz,
        a.t_xyz, stride, xq, ls->box.as<int>(), a.bad);
    int launches = 1;
    const Grid none{};
    if (nt) {
        seg_bbox_kernel<<<(unsigned) (nt / B200M_TILE_N), 256, 0, st>>>(xt, a.blk[ts], ls->box.as<int>());
        launches += 1;
    }
    seg_grid_kernel<<<(unsigned) a.n_pairs, 256, 0, st>>>(ls->box.as<int>(), a.rows, ts, a.radius, ls->seg_grids.as<SegGrid>(),
                                                          ls->counts.as<int>(), ls->cursor.as<int>());
    launches += 1;
    if (nt) {
        cell_count_kernel<true><<<(unsigned) (nt / 256), 256, 0, st>>>(none, &xt->x, 4, t.valid.as<uint8_t>(), nt, ls->counts.as<int>(),
                                                                       grids, a.blk[ts]);
        launches += 1;
    }
    cell_scan_kernel<true><<<(unsigned) a.n_pairs, 1024, 0, st>>>(ls->counts.as<int>(), 0, ls->starts.as<int>(), grids, a.rows, ts);
    launches += 1;
    if (nt) {
        cell_fill_kernel<true><<<(unsigned) (nt / 256), 256, 0, st>>>(none, &xt->x, 4, t.valid.as<uint8_t>(), nt, ls->starts.as<int>(),
                                                                      ls->cursor.as<int>(), ls->rows.as<int32_t>(), grids, a.blk[ts]);
        launches += 1;
    }
    CK(cudaGetLastError());
    const size_t smem = sizeof(float) * (size_t) q.dp * kLocalWarps;
    const size_t want = (nq + kLocalWarps - 1) / kLocalWarps, cap = (size_t) ctx->sm_count * 8;
    const unsigned blocks = (unsigned) (want < cap ? want : cap);
    const float r2 = a.radius * a.radius;   // radiusSearch is handed radius * radius (FP32 product)
    ctx->stats.launches += launches + 1;
#define B200M_LOCALB_CASE(K)                                                                                                    \
    do {                                                                                                                        \
        if (smem > 48 * 1024) /* rows over 1536 floats */                                                                     \
            CK(cudaFuncSetAttribute(local_cells_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));     \
        local_cells_kernel<K, true><<<blocks, kLocalWarps * 32, smem, st>>>(                                                    \
            none, q.f32.as<float>(), q.valid.as<uint8_t>(), q.dp, t.f32.as<float>(), 0, nq, &xq->x, &xt->x, 4, r2, a.k,         \
            nullptr, ls->rows.as<int32_t>(), d_idx, d_dist, d_count, grids, a.blk[qs], ls->starts.as<int>());                  \
        CK(cudaGetLastError());                                                                                                 \
        return 0;                                                                                                               \
    } while (0)
    if (a.k <= 1) B200M_LOCALB_CASE(1);
    if (a.k <= 2) B200M_LOCALB_CASE(2);
    if (a.k <= 4) B200M_LOCALB_CASE(4);
    if (a.k <= 8) B200M_LOCALB_CASE(8);
    if (a.k <= 16) B200M_LOCALB_CASE(16);
    B200M_LOCALB_CASE(32);
#undef B200M_LOCALB_CASE
}
