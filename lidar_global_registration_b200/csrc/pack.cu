// pack.cu -- descriptor upload kernels: the GPU replacement of pcl2cv<FeatureT>
// (reference include/matching.h:553-560), done ONCE per descriptor set instead of once
// per (query block, train block) pair.
//
//   pack_f32      AoS rows (stride sizeof(FeatureT)) -> dense FP32 [n][dp] + validity byte
//                 (pcl::PointRepresentation::isValid: every value finite).
//   tc_prepare    common centre + power-of-two scale for both sides, then the two FP16
//                 operand tiles per side for the tcgen05 candidate kernel:
//                     as query : [-2*x16 , 1, 1, 1, 0..]          (A operand, K-major)
//                     as train : [   x16 , nb_hi, nb_mid, nb_lo, 0..]  (B operand, K-major)
//                 so that  A.B = |b16|^2 - 2 a16.b16  comes out of the tensor core with
//                 the train-row norm already fused in.  Invalid / padding train rows carry
//                 the FP16 sentinel 60000 in nb_hi so they can never look near.
//
// All HBM-bound: algorithmic bytes per row = stride_in + 4*dp + 1 (pack_f32) and
// 4*dp + 2*2*kp + 4 (operand pack) -- see DESIGN.md.
#include <float.h>
#include <math.h>
#include <string.h>

#include "internal.cuh"

namespace {

constexpr int kPackWarps = 16;       // warps per CTA of the persistent pack kernel
constexpr int kWarpsPerBlock = 8;    // operand pack: one warp per row

// column statistics of one CTA: [sum | min | max][dp] then the number of valid rows
__host__ __device__ inline size_t stats_floats(int dp) { return (size_t) 3 * dp + 1; }

// One warp per row, persistent over the rows.  NI = ceil(dp / 32) values per lane stay in registers: the row is dense-
// copied, its validity decided (every value finite), and -- for valid rows only -- folded into the lane's running
// column sum / min / max, from which tc_prepare derives the common centre and the FP16 scale without reading the data
// again.
// SEG (device batch calls): `aos` is unused; row `row` of the padded layout belongs to set seg_blk[row / 256], which
// starts at padded row sets[.].first and has sets[.].rows rows at sets[.].base + local * stride_floats.  The rows after
// a set's last row (up to its next multiple of 256) are written as the staging path's 0xFF bytes pack: NaN (all ones)
// in the descriptor columns, 0 in the padding columns, invalid.
template <int NI, bool SEG>
__global__ void __launch_bounds__(kPackWarps * 32)
pack_f32_kernel(const float *__restrict__ aos, size_t n, size_t stride_floats, int dim, int dp,
                float *__restrict__ f32, uint8_t *__restrict__ valid, float *__restrict__ stats,
                const int32_t *__restrict__ seg_blk, const SetRef *__restrict__ sets) {
    extern __shared__ float sh[];   // [3][dp]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float sum[NI], mn[NI], mx[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i) { sum[i] = 0.f; mn[i] = INFINITY; mx[i] = -INFINITY; }
    float cnt = 0.f;
    for (size_t row = (size_t) blockIdx.x * kPackWarps + warp; row < n; row += (size_t) gridDim.x * kPackWarps) {
        float *dst = f32 + row * (size_t) dp;
        float v[NI];
        bool ok = true;
        if constexpr (SEG) {
            const SetRef set = sets[seg_blk[row / B200M_TILE_N]];
            const size_t local = row - (size_t) set.first;
            const bool gap = local >= (size_t) set.rows;
            const float *src = set.base + (gap ? 0 : local) * stride_floats;
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int d = lane + 32 * i;
                v[i] = d < dim ? (gap ? __int_as_float(-1) : __ldg(src + d)) : 0.f;
                ok = ok && isfinite(v[i]);
            }
        } else {
            const float *src = aos + row * stride_floats;
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int d = lane + 32 * i;
                v[i] = d < dim ? __ldg(src + d) : 0.f;
                ok = ok && isfinite(v[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < NI; ++i) {
            const int d = lane + 32 * i;
            if (d < dp) dst[d] = v[i];
        }
        ok = __all_sync(0xffffffffu, ok);
        if (lane == 0) valid[row] = ok ? 1 : 0;
        if (ok) {
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                sum[i] += v[i];
                mn[i] = fminf(mn[i], v[i]);
                mx[i] = fmaxf(mx[i], v[i]);
            }
            cnt += 1.f;
        }
    }
    // fold the warps of the CTA, one after the other
    for (int d = threadIdx.x; d < dp; d += blockDim.x) { sh[d] = 0.f; sh[dp + d] = INFINITY; sh[2 * dp + d] = -INFINITY; }
    __shared__ float sh_cnt;
    if (threadIdx.x == 0) sh_cnt = 0.f;
    __syncthreads();
    for (int w = 0; w < kPackWarps; ++w) {
        if (warp == w) {
#pragma unroll
            for (int i = 0; i < NI; ++i) {
                const int d = lane + 32 * i;
                if (d < dp) {
                    sh[d] += sum[i];
                    sh[dp + d] = fminf(sh[dp + d], mn[i]);
                    sh[2 * dp + d] = fmaxf(sh[2 * dp + d], mx[i]);
                }
            }
            if (lane == 0) sh_cnt += cnt;
        }
        __syncthreads();
    }
    float *out = stats + (size_t) blockIdx.x * stats_floats(dp);
    for (int d = threadIdx.x; d < 3 * dp; d += blockDim.x) out[d] = sh[d];
    if (threadIdx.x == 0) out[3 * dp] = sh_cnt;
}

// Long rows (dp > 1024: NI = 64 would not fit the register file, NI = 32 already spills) in two passes.  First the copy and
// the validity, one warp per row walking the row in 32-column slices, with the same SEG handling as pack_f32_kernel.
template <bool SEG>
__global__ void __launch_bounds__(kPackWarps * 32)
pack_f32_long_kernel(const float *__restrict__ aos, size_t n, size_t stride_floats, int dim, int dp,
                     float *__restrict__ f32, uint8_t *__restrict__ valid,
                     const int32_t *__restrict__ seg_blk, const SetRef *__restrict__ sets) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (size_t row = (size_t) blockIdx.x * kPackWarps + warp; row < n; row += (size_t) gridDim.x * kPackWarps) {
        float *dst = f32 + row * (size_t) dp;
        const float *src = aos + row * stride_floats;
        bool gap = false;
        if constexpr (SEG) {
            const SetRef set = sets[seg_blk[row / B200M_TILE_N]];
            const size_t local = row - (size_t) set.first;
            gap = local >= (size_t) set.rows;
            src = set.base + (gap ? 0 : local) * stride_floats;
        }
        bool ok = true;
        for (int d = lane; d < dp; d += 32) {
            const float v = d < dim ? (gap ? __int_as_float(-1) : __ldg(src + d)) : 0.f;
            ok = ok && isfinite(v);
            dst[d] = v;
        }
        ok = __all_sync(0xffffffffu, ok);
        if (lane == 0) valid[row] = ok ? 1 : 0;
    }
}

// ... then the column statistics of the rows just written, in the layout pack_f32_kernel leaves: CTA b of the grid folds
// the valid rows of its contiguous share of the rows, a thread per column (coalesced across the threads of a row).  The
// summation order differs from the short form; the centre only has to be some centre (DESIGN.md §4).
__global__ void __launch_bounds__(kPackWarps * 32)
pack_stats_long_kernel(const float *__restrict__ f32, const uint8_t *__restrict__ valid, size_t n, int dp,
                       float *__restrict__ stats) {
    const size_t per = (n + gridDim.x - 1) / gridDim.x;
    const size_t r0 = min(n, (size_t) blockIdx.x * per), r1 = min(n, r0 + per);
    float *out = stats + (size_t) blockIdx.x * stats_floats(dp);
    for (int d = threadIdx.x; d < dp; d += blockDim.x) {
        float s = 0.f, mn = INFINITY, mx = -INFINITY;
        for (size_t r = r0; r < r1; ++r) {
            if (!valid[r]) continue;
            const float v = __ldg(f32 + r * (size_t) dp + d);
            s += v;
            mn = fminf(mn, v);
            mx = fmaxf(mx, v);
        }
        out[d] = s;
        out[dp + d] = mn;
        out[2 * dp + d] = mx;
    }
    if (threadIdx.x == 0) {
        float cnt = 0.f;
        for (size_t r = r0; r < r1; ++r) cnt += valid[r] ? 1.f : 0.f;
        out[3 * dp] = cnt;
    }
}

// power of two s with maxabs*s in (0.5, 1]; all-equal data (maxabs == 0) keeps s = 1
__host__ __device__ inline float scale_for(float maxabs) {
    float scale = 1.f;
    if (maxabs > 0.f && isfinite(maxabs)) {
        int ex;
        float fr = frexpf(maxabs, &ex);   // maxabs = fr * 2^ex, fr in [0.5, 1)
        if (fr == 0.5f) ex -= 1;          // exactly a power of two -> map to 1.0
        scale = ldexpf(1.f, -ex);
    }
    return scale;
}

// The certificate's window (DESIGN.md §4); data outside it stays on the exact path.  Upper edge: the reference's FP32 sum
// of D squared differences, each at most (2 maxabs)^2, stays finite.  Lower edge: the subnormal rounding of those terms (at
// most 2^-150 each, D 2^-150 s^2 in scaled units) stays under 2^-25, inside the 1e-6 that slop carries on top of the
// accumulator bound.  The host (launch_tc_prepare) and the device (prep_decide_kernel) decide with this one function.
__host__ __device__ inline bool tc_window(float maxabs, float scale, int dim) {
    const double m = maxabs, s = scale, gam = (dim + 4) * 0x1p-24;
    return isfinite(maxabs) && isfinite(scale) && scale > 0.f &&
           (maxabs == 0.f || (dim * 4.0 * m * m * (1.0 + gam) < (double) FLT_MAX && dim * s * s <= 0x1p125));
}

// Combine the per-CTA column statistics of both sides: CTA b owns columns 32b..32b+31, its eight warps each fold
// every eighth partial; -> mean[dp] and (atomicMax) the largest centred magnitude.
__global__ void __launch_bounds__(256)
prep_finalize_kernel(const float *__restrict__ sa, int ga, const float *__restrict__ sb, int gb, int dp, int dim,
                     float *__restrict__ mean, PrepDev *__restrict__ out) {
    __shared__ double sh_s[8][32], sh_c[8];
    __shared__ float sh_lo[8][32], sh_hi[8][32];
    const int col = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int d = blockIdx.x * 32 + col;
    const size_t sf = stats_floats(dp);
    double s = 0, c = 0;
    float lo = INFINITY, hi = -INFINITY;
    for (int side = 0; side < 2; ++side) {
        const float *st = side ? sb : sa;
        const int g_n = side ? gb : ga;
        for (int g = slice; g < g_n; g += 8) {
            const float *row = st + (size_t) g * sf;
            c += (double) row[3 * dp];
            if (d < dp) {
                s += (double) row[d];
                lo = fminf(lo, row[dp + d]);
                hi = fmaxf(hi, row[2 * dp + d]);
            }
        }
    }
    sh_s[slice][col] = s;
    sh_lo[slice][col] = lo;
    sh_hi[slice][col] = hi;
    if (col == 0) sh_c[slice] = c;
    __syncthreads();
    if (slice == 0 && d < dp) {
        for (int w = 1; w < 8; ++w) {
            s += sh_s[w][col];
            lo = fminf(lo, sh_lo[w][col]);
            hi = fmaxf(hi, sh_hi[w][col]);
        }
        double cc = 0;
        for (int w = 0; w < 8; ++w) cc += sh_c[w];
        const float mu = cc > 0 ? (float) (s / cc) : 0.f;
        mean[d] = mu;
        if (d < dim && cc > 0) {
            const float e = fabsf(fmaxf(hi - mu, mu - lo));   // NaN keeps its (positive) bit pattern: larger than +inf as an int
            atomicMax(&out->maxabs_bits, __float_as_int(e));
        }
    }
}

// One warp per (padded) row, persistent over the rows: FP16 operand rows + |x16|^2.  A lane converts four consecutive
// values at a time (128-bit loads, 64-bit stores); the scale word is read once per warp and the side's largest norm
// leaves through ONE atomic per warp (a per-row atomic on the line that also holds the scale serialises the kernel
// in a single L2 slice: 0.9 ms instead of 0.25 ms for 500k SHOT rows).
// NS: 128-column sweeps of the row held in registers (5: kp <= 640; 16: the long form, kp <= 2048).
template <int NS>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
pack_operands_kernel(const float *__restrict__ f32, const uint8_t *__restrict__ valid, size_t n, size_t n_pad,
                     int dim, int dp, int kp, const float *__restrict__ mean, PrepDev *__restrict__ prep, int side,
                     __half *__restrict__ op_query, __half *__restrict__ op_train, float *__restrict__ norm16) {
    const int lane = threadIdx.x & 31;
    const float scale = scale_for(__int_as_float(prep->maxabs_bits));
    float4 mu[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        const int d0 = 4 * lane + 128 * i;
        mu[i] = d0 < dp ? __ldg(reinterpret_cast<const float4 *>(mean + d0)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float max_nf = 0.f;
    const size_t stride = (size_t) gridDim.x * kWarpsPerBlock;
    for (size_t row = (size_t) blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5); row < n_pad; row += stride) {
        const bool ok = row < n && valid[row];
        __half *oq = op_query + row * (size_t) kp;
        __half *ot = op_train + row * (size_t) kp;
        const float *src = f32 + row * (size_t) dp;
        double nrm = 0.0;
        // the descriptor columns (dp is a multiple of 4, kp of 64; columns dim..dp-1 of f32 are zero): every load of
        // the row is issued before the first conversion (at most NS 128-column sweeps)
        float4 v[NS];
#pragma unroll
        for (int i = 0; i < NS; ++i) {
            const int d0 = 4 * lane + 128 * i;
            v[i] = (row < n && d0 < dp) ? __ldg(reinterpret_cast<const float4 *>(src + d0)) : mu[i];   // x - mu = 0 beyond the row
        }
#pragma unroll
        for (int i = 0; i < NS; ++i) {
            const int d0 = 4 * lane + 128 * i;
            if (d0 >= kp) break;
            const float x[4] = {(v[i].x - mu[i].x) * scale, (v[i].y - mu[i].y) * scale, (v[i].z - mu[i].z) * scale,
                                (v[i].w - mu[i].w) * scale};
            __half ht[4], hq[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int d = d0 + e;
                if (d < dim) {
                    ht[e] = __float2half_rn(ok ? x[e] : 0.f);
                    const float xf = __half2float(ht[e]);
                    hq[e] = __float2half_rn(-2.f * xf);   // exact: |x| <= 1, power-of-two factor
                    nrm += (double) xf * (double) xf;
                } else {
                    ht[e] = __float2half_rn(0.f);   // the three norm columns are filled in below
                    hq[e] = __float2half_rn(d < dim + B200M_AUG_COLS ? 1.f : 0.f);   // 1s pick up the norm pieces of the train row
                }
            }
            *reinterpret_cast<uint2 *>(oq + d0) = *reinterpret_cast<const uint2 *>(hq);
            *reinterpret_cast<uint2 *>(ot + d0) = *reinterpret_cast<const uint2 *>(ht);
        }
        for (int o = 16; o > 0; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
        __syncwarp();
        if (lane == 0) {
            float nf = ok ? (float) nrm : 0.f;
            norm16[row] = nf;
            float hi_src = ok ? nf : B200M_SENTINEL;
            __half hi = __float2half_rn(hi_src);
            float r1 = hi_src - __half2float(hi);
            __half mid = __float2half_rn(r1);
            float r2 = r1 - __half2float(mid);
            __half lo = __float2half_rn(r2);
            ot[dim + 0] = hi;
            ot[dim + 1] = mid;
            ot[dim + 2] = lo;
            if (ok) max_nf = fmaxf(max_nf, nf);
        }
    }
    if (lane == 0 && max_nf > 0.f) atomicMax(&prep->max_norm_bits[side], __float_as_int(sqrtf(max_nf)));
}

// device_prepare: the routing decision and the norm bounds, from the statistics and operand passes before it (one thread)
__global__ void prep_decide_kernel(PrepDev *__restrict__ prep, int dim) {
    const float maxabs = __int_as_float(prep->maxabs_bits);
    prep->usable = tc_window(maxabs, scale_for(maxabs), dim) ? 1 : 0;
    prep->bmax[0] = __int_as_float(prep->max_norm_bits[0]);
    prep->bmax[1] = __int_as_float(prep->max_norm_bits[1]);
}

}  // namespace

int pack_stats_blocks(int sm_count) { return sm_count * 2; }
size_t pack_stats_bytes(int sm_count, int dp) { return sizeof(float) * (size_t) pack_stats_blocks(sm_count) * stats_floats(dp); }

cudaError_t launch_pack_f32(const float *aos, size_t n, size_t stride_bytes, int dim, int dp,
                            float *f32, uint8_t *valid, float *stats, int sm_count, cudaStream_t st,
                            const int32_t *seg_blk, const SetRef *sets) {
    if (n == 0) return cudaSuccess;
    const unsigned blocks = (unsigned) pack_stats_blocks(sm_count);
    const size_t smem = sizeof(float) * 3 * (size_t) dp;
    const int ni = (dp + 31) / 32;
    if (ni > 32) {   // long rows: copy + validity, then the column statistics over what was written
        if (sets)
            pack_f32_long_kernel<true><<<blocks, kPackWarps * 32, 0, st>>>(aos, n, stride_bytes / 4, dim, dp, f32, valid, seg_blk, sets);
        else
            pack_f32_long_kernel<false><<<blocks, kPackWarps * 32, 0, st>>>(aos, n, stride_bytes / 4, dim, dp, f32, valid, nullptr,
                                                                            nullptr);
        pack_stats_long_kernel<<<blocks, kPackWarps * 32, 0, st>>>(f32, valid, n, dp, stats);
        return cudaGetLastError();
    }
#define B200M_PACK_CASE(NI)                                                                                          \
    do {                                                                                                             \
        if (sets)                                                                                                    \
            pack_f32_kernel<NI, true><<<blocks, kPackWarps * 32, smem, st>>>(aos, n, stride_bytes / 4, dim, dp, f32, \
                                                                             valid, stats, seg_blk, sets);           \
        else                                                                                                         \
            pack_f32_kernel<NI, false><<<blocks, kPackWarps * 32, smem, st>>>(aos, n, stride_bytes / 4, dim, dp, f32,\
                                                                              valid, stats, nullptr, nullptr);       \
    } while (0)
    if (ni <= 2) B200M_PACK_CASE(2);
    else if (ni <= 5) B200M_PACK_CASE(5);
    else if (ni <= 11) B200M_PACK_CASE(11);
    else if (ni <= 16) B200M_PACK_CASE(16);
    else B200M_PACK_CASE(32);
#undef B200M_PACK_CASE
    return cudaGetLastError();
}

cudaError_t launch_tc_prepare(b200m_ctx *ctx) {
    Side &a = ctx->side[0], &b = ctx->side[1];
    TcPrep &pr = ctx->prep;
    cudaStream_t st = ctx->stream;
    const int dp = a.dp, dim = a.dim;
    cudaError_t e;
    if ((e = pr.red.reserve(sizeof(PrepDev))) != cudaSuccess) return e;
    if ((e = pr.mean.reserve(sizeof(float) * dp)) != cudaSuccess) return e;
    PrepDev *dev = pr.red.as<PrepDev>();
    const int ga = a.n ? pack_stats_blocks(ctx->sm_count) : 0, gb = b.n ? pack_stats_blocks(ctx->sm_count) : 0;
    if ((e = cudaMemsetAsync(dev, 0, sizeof(PrepDev), st)) != cudaSuccess) return e;
    prep_finalize_kernel<<<(dp + 31) / 32, 256, 0, st>>>(a.stats.as<float>(), ga, b.stats.as<float>(), gb, dp, dim,
                                                         pr.mean.as<float>(), dev);
    ctx->stats.launches += 1;
    for (int s = 0; s < 2; ++s) {
        Side &sd = ctx->side[s];
        if (sd.n_pad == 0) continue;
        size_t opb = sizeof(__half) * sd.n_pad * (size_t) sd.kp;
        if ((e = sd.op_query.reserve(opb)) != cudaSuccess) return e;
        if ((e = sd.op_train.reserve(opb)) != cudaSuccess) return e;
        if ((e = sd.norm16.reserve(sizeof(float) * sd.n_pad)) != cudaSuccess) return e;
        size_t want = (sd.n_pad + kWarpsPerBlock - 1) / kWarpsPerBlock, cap_blocks = (size_t) ctx->sm_count * 8;
        unsigned blocks = (unsigned) (want < cap_blocks ? want : cap_blocks);
        if (sd.kp <= 640)
            pack_operands_kernel<5><<<blocks, kWarpsPerBlock * 32, 0, st>>>(
                sd.f32.as<float>(), sd.valid.as<uint8_t>(), sd.n, sd.n_pad, dim, dp, sd.kp, pr.mean.as<float>(), dev, s,
                sd.op_query.as<__half>(), sd.op_train.as<__half>(), sd.norm16.as<float>());
        else
            pack_operands_kernel<16><<<blocks, kWarpsPerBlock * 32, 0, st>>>(
                sd.f32.as<float>(), sd.valid.as<uint8_t>(), sd.n, sd.n_pad, dim, dp, sd.kp, pr.mean.as<float>(), dev, s,
                sd.op_query.as<__half>(), sd.op_train.as<__half>(), sd.norm16.as<float>());
        ctx->stats.launches += 1;
    }
    if (ctx->device_prepare) {   // no round trip: the candidate kernel's DP form reads the decision from PrepDev
        prep_decide_kernel<<<1, 1, 0, st>>>(dev, dim);
        ctx->stats.launches += 1;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        pr.ver[0] = a.version;
        pr.ver[1] = b.version;
        pr.ready = true;
        return cudaSuccess;
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    // the one host round trip of the prepare step: scale, usability and the per-side norm bounds
    PrepDev h;
    if ((e = cudaMemcpyAsync(&h, dev, sizeof(h), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    float maxabs;
    memcpy(&maxabs, &h.maxabs_bits, 4);
    const float scale = scale_for(maxabs);
    pr.scale = scale;
    pr.usable = tc_window(maxabs, scale, dim);
    memcpy(&pr.max_norm[0], &h.max_norm_bits[0], 4);
    memcpy(&pr.max_norm[1], &h.max_norm_bits[1], 4);
    pr.ver[0] = a.version;
    pr.ver[1] = b.version;
    pr.ready = true;
    return cudaSuccess;
}
