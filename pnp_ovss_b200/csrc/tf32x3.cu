// tf32x3.cu -- operand preparation for fp32-grade GEMMs on the TF32 tensor cores (SURVEY 8f.1: the model pass,
// BITM:386-404, whose dense contractions stay torch's -- cuBLAS TF32 GEMMs -- while everything around them is here).
//
// y = x W^T is computed as ONE TF32 GEMM of depth 3K on an exact split of both operands:
//     x = x_hi + x_lo,  W = W_hi + W_lo    (hi = x rounded to TF32's 10 explicit mantissa bits; lo = x - hi is exact)
//     [x_hi | x_lo | x_hi] (M x 3K)  times  [W_hi | W_hi | W_lo]^T (3K x N)  =  x_hi W_hi + x_lo W_hi + x_hi W_lo
// (the dropped x_lo W_lo term is 2^-22 relative; accumulation is fp32 inside the tensor core).  The kernels below write
// the tripled activation operand straight from its producer, so the split costs no extra pass over HBM:
//     split3            x                        -> [hi | lo | hi]
//     layernorm_split3  LayerNorm(x) (VIT:70-71) -> [hi | lo | hi]   (one warp per row, row held in registers)
//     gelu_split3       GELU(x + bias) (exact erf, VIT:35-40)  -> [hi | lo | hi]
// All three are pure HBM streams (4 B read, 12 B written per element) with 128-bit accesses.
//
// "3xFP16" is the same idea on the fp16 tensor cores (twice the TF32 rate, half the operand bytes):
//     x = h + l 2^-11 with h = fp16(x), l = fp16((x - h) 2^11)  (22-23 significant bits; fp16's range: |x| <= 65504 / 2^a)
//     [h 2^a | l | h] (M x 3K)  times  [W_h 2^b | W_h | W_l]^T,  a + b = 11   =   2^11 (h W_h + 2^-11 (l W_h + h W_l))
// i.e. ONE fp16 GEMM with fp32 accumulation whose result carries a factor 2^11 that the consumer kernels here take back
// (in_scale / residual_scale) -- powers of two, so nothing is rounded by the scaling.  b is chosen per weight matrix as large
// as its largest entry allows, which leaves a = 0 (no loss of activation range) for any realistic weight.
#include <cuda_fp16.h>
#include <math.h>

#include "common.cuh"

namespace pnp {

__device__ __forceinline__ float tf32_hi(float x) {
    // round to nearest (ties away) at bit 13.  Where the carry would leave the finite range x is kept (lo = 0): from
    // |x| = 0x1.ffep+127 (0x7F7FF000) up, +-inf, and NaN -- whose arithmetic form 0x7FFFFFFF would carry into the sign bit
    // and round to -0
    float hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
    return (fabsf(x) < 0x1.ffep+127f) ? hi : x;
}

// ---- operand writers.  kHalf == false: fp32 [hi | lo | hi] for the 3xTF32 GEMM; kHalf == true: fp16 [hi*2^a | lo*2^11 | hi]
// for the 3xFP16 GEMM (see the header of this file), `hi_scale` = 2^a, `flag` raised when a value does not fit fp16.
template <bool kHalf>
struct Split3;

template <>
struct Split3<false> {
    typedef float out_t;
    static __device__ __forceinline__ void store(float *__restrict__ row_out, int K, int k, float4 v, float, int *) {
        float4 hi = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
        // lo = v - hi exactly; where hi fell back to v itself (inf, NaN, overflow) the difference is defined as 0, not inf - inf
        float4 lo = make_float4(hi.x == v.x ? 0.f : v.x - hi.x, hi.y == v.y ? 0.f : v.y - hi.y, hi.z == v.z ? 0.f : v.z - hi.z,
                                hi.w == v.w ? 0.f : v.w - hi.w);
        stg_stream4(row_out + k, hi);
        stg_stream4(row_out + K + k, lo);
        stg_stream4(row_out + 2 * K + k, hi);
    }
};

// (x0, x1) -> packed (h, l) pairs: h = fp16(x), l = fp16((x - h) 2^11); x - h is exact in fp32 and |(x - h) 2^11| <= |x| / 2.
// Packed cvt.rn.f16x2.f32 conversions: one instruction per pair.
__device__ __forceinline__ void split_half2(float x0, float x1, __half2 &h, __half2 &l) {
    h = __floats2half2_rn(x0, x1);
    const float2 hf = __half22float2(h);
    l = __floats2half2_rn((x0 - hf.x) * 2048.0f, (x1 - hf.y) * 2048.0f);
}
// either half of a packed pair is inf or NaN (exponent field all ones): 0x7C00 + 0x0400 carries into the half's sign bit
__device__ __forceinline__ bool half2_nonfinite(__half2 v) {
    const unsigned u = *reinterpret_cast<const unsigned *>(&v);
    return (((u & 0x7C007C00u) + 0x04000400u) & 0x80008000u) != 0u;
}

template <>
struct Split3<true> {
    typedef __half out_t;
    static __device__ __forceinline__ void store(__half *__restrict__ row_out, int K, int k, float4 v, float hi_scale, int *flag) {
        __half2 h01, h23, l01, l23;
        split_half2(v.x, v.y, h01, l01);
        split_half2(v.z, v.w, h23, l23);
        // h * 2^a in half arithmetic: exact (a power of two) unless it overflows, which -- like an inf / NaN input -- raises the flag
        __half2 s01 = h01, s23 = h23;
        if (hi_scale != 1.0f) {
            const __half2 sc = __float2half2_rn(hi_scale);
            s01 = __hmul2(h01, sc);
            s23 = __hmul2(h23, sc);
        }
        const bool bad = half2_nonfinite(s01) || half2_nonfinite(s23);
        *reinterpret_cast<uint2 *>(row_out + k) = make_uint2(*reinterpret_cast<unsigned *>(&s01), *reinterpret_cast<unsigned *>(&s23));
        *reinterpret_cast<uint2 *>(row_out + K + k) = make_uint2(*reinterpret_cast<unsigned *>(&l01), *reinterpret_cast<unsigned *>(&l23));
        *reinterpret_cast<uint2 *>(row_out + 2 * K + k) = make_uint2(*reinterpret_cast<unsigned *>(&h01), *reinterpret_cast<unsigned *>(&h23));
        if (bad && flag) *flag = 1;
    }
};

// Rows are walked by CTAs (grid-stride), the float4 pieces of a row by the CTA's threads: no division per item.
template <bool kHalf>
__global__ void __launch_bounds__(256) split3_kernel(const float *__restrict__ x, typename Split3<kHalf>::out_t *__restrict__ out,
                                                     long long M, int K, float in_scale, float hi_scale, int *__restrict__ flag) {
    for (long long m = blockIdx.x; m < M; m += gridDim.x) {
        const float *xr = x + m * K;
        typename Split3<kHalf>::out_t *orow = out + m * 3 * K;
        for (int k = threadIdx.x * 4; k < K; k += blockDim.x * 4) {
            float4 v = ldg_stream4(xr + k);
            v.x *= in_scale; v.y *= in_scale; v.z *= in_scale; v.w *= in_scale;
            Split3<kHalf>::store(orow, K, k, v, hi_scale, flag);
        }
    }
}

__device__ __forceinline__ float gelu_erf(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }

template <bool kHalf>
__global__ void __launch_bounds__(256) gelu_split3_kernel(const float *__restrict__ x, const float *__restrict__ bias,
                                                          typename Split3<kHalf>::out_t *__restrict__ out, long long M, int K,
                                                          float in_scale, float hi_scale, int *__restrict__ flag) {
    for (long long m = blockIdx.x; m < M; m += gridDim.x) {
        const float *xr = x + m * K;
        typename Split3<kHalf>::out_t *orow = out + m * 3 * K;
        for (int k = threadIdx.x * 4; k < K; k += blockDim.x * 4) {
            float4 v = ldg_stream4(xr + k);
            v.x *= in_scale; v.y *= in_scale; v.z *= in_scale; v.w *= in_scale;
            if (bias) {
                const float4 b = __ldg(reinterpret_cast<const float4 *>(bias + k));
                v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
            }
            Split3<kHalf>::store(orow, K, k, make_float4(gelu_erf(v.x), gelu_erf(v.y), gelu_erf(v.z), gelu_erf(v.w)), hi_scale, flag);
        }
    }
}

// One warp per row; the row (K <= 128*kChunks floats) stays in registers between the mean, the variance and the write.
// Optional residual: x = x + res * res_scale (+ res_bias) is formed first and written back to x_out (the running hidden state),
// so the residual add, the LayerNorm and the operand split are one pass.
template <int kChunks, bool kHalf>
__global__ void __launch_bounds__(256, kChunks <= 8 ? 3 : 1) layernorm_split3_kernel(const float *__restrict__ x, const float *__restrict__ res, float res_scale,
                                                               const float *__restrict__ res_bias, float *__restrict__ x_out,
                                                               const float *__restrict__ gamma, const float *__restrict__ beta,
                                                               float eps, typename Split3<kHalf>::out_t *__restrict__ out3,
                                                               float *__restrict__ out1, long long M, int K, float hi_scale,
                                                               int *__restrict__ flag, int ld3, float tail_one) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    for (long long m = blockIdx.x * (long long)wpb + (threadIdx.x >> 5); m < M; m += (long long)gridDim.x * wpb) {
        if (kHalf && out3 && ld3 > 3 * K && lane == 0) {
            // bias columns of the GEMM operand: [tail_one, 1, 0 x 6] against the weight rows [b_h 2^11 / tail_one, b_l, 0 x 6]
            __half t[8];
            t[0] = __float2half_rn(tail_one);
            t[1] = __float2half_rn(1.0f);
#pragma unroll
            for (int i = 2; i < 8; ++i) t[i] = __float2half_rn(0.f);
            *reinterpret_cast<uint4 *>(reinterpret_cast<__half *>(out3) + m * ld3 + 3 * K) = *reinterpret_cast<const uint4 *>(t);
        }
        float4 v[kChunks];
        float sum = 0.f;
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
            const int k = (lane + 32 * c) * 4;
            if (k < K) {
                float4 t = ldg_stream4(x + m * K + k);
                if (res) {
                    const float4 r = ldg_stream4(res + m * K + k);
                    t.x = fmaf(r.x, res_scale, t.x); t.y = fmaf(r.y, res_scale, t.y); t.z = fmaf(r.z, res_scale, t.z); t.w = fmaf(r.w, res_scale, t.w);
                    if (res_bias) {
                        const float4 b = __ldg(reinterpret_cast<const float4 *>(res_bias + k));
                        t.x += b.x; t.y += b.y; t.z += b.z; t.w += b.w;
                    }
                    if (x_out) *reinterpret_cast<float4 *>(x_out + m * K + k) = t;
                }
                v[c] = t;
                sum += (t.x + t.y) + (t.z + t.w);
            } else {
                v[c] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        // corrected two-pass moments: the second pass also sums the deviations from the fp32 mean m0; their mean r moves the
        // mean to m0 + r and takes r^2 out of the variance.  On a (near-)constant row rstd is about rsqrt(eps), and it would
        // otherwise multiply m0's rounding error into the output (3e-5 |gamma| for a row of 0.3 at K = 768, eps = 1e-6).
        const float mean0 = warp_sum(sum) / (float)K;
        float sq = 0.f, dev = 0.f;
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
            if ((lane + 32 * c) * 4 < K) {
                const float a = v[c].x - mean0, b = v[c].y - mean0, cc = v[c].z - mean0, d = v[c].w - mean0;
                dev += (a + b) + (cc + d);
                sq += (a * a + b * b) + (cc * cc + d * d);
            }
        }
        dev = warp_sum(dev);
        const float r = dev / (float)K;
        const float mean = mean0 + r;
        const float rstd = rsqrtf(fmaxf(warp_sum(sq) - dev * r, 0.f) / (float)K + eps);
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
            const int k = (lane + 32 * c) * 4;
            if (k < K) {
                const float4 g = __ldg(reinterpret_cast<const float4 *>(gamma + k));
                const float4 b = __ldg(reinterpret_cast<const float4 *>(beta + k));
                const float4 y = make_float4((v[c].x - mean) * rstd * g.x + b.x, (v[c].y - mean) * rstd * g.y + b.y,
                                             (v[c].z - mean) * rstd * g.z + b.z, (v[c].w - mean) * rstd * g.w + b.w);
                if (out3) Split3<kHalf>::store(out3 + m * ld3, K, k, y, hi_scale, flag);
                if (out1) stg_stream4(out1 + m * K + k, y);
            }
        }
    }
}

}  // namespace pnp

using namespace pnp;

static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

namespace {
template <bool kHalf>
int run_split3(const float *x, void *out3, long long M, int K, float in_scale, float hi_scale, int *flag, cudaStream_t st) {
    const int grid = (int)std::max<long long>(1, std::min<long long>(M, (long long)kNumSMs * 16));   // CTAs walk rows
    typedef typename Split3<kHalf>::out_t out_t;
    PNP_LAUNCH(kTf32Split, st, (split3_kernel<kHalf><<<grid, 256, 0, st>>>(x, reinterpret_cast<out_t *>(out3), M, K, in_scale, hi_scale, flag)));
    return launch_status();
}
template <bool kHalf>
int run_gelu_split3(const float *x, const float *bias, void *out3, long long M, int K, float in_scale, float hi_scale, int *flag,
                    cudaStream_t st) {
    const int grid = (int)std::max<long long>(1, std::min<long long>(M, (long long)kNumSMs * 16));   // CTAs walk rows
    typedef typename Split3<kHalf>::out_t out_t;
    PNP_LAUNCH(kGeluSplit, st, (gelu_split3_kernel<kHalf><<<grid, 256, 0, st>>>(x, bias, reinterpret_cast<out_t *>(out3), M, K, in_scale, hi_scale, flag)));
    return launch_status();
}
template <bool kHalf>
int run_layernorm_split3(const float *x, const float *residual, float res_scale, const float *residual_bias, float *x_out,
                         const float *gamma, const float *beta, float eps, void *out3, float *out1, long long M, int K,
                         float hi_scale, int *flag, int ld3, float tail_one, cudaStream_t st) {
    const int wpb = 8;
    const int grid = (int)std::max<long long>(1, std::min<long long>((M + wpb - 1) / wpb, (long long)kNumSMs * 8));
    const int chunks = (K + 127) / 128;
    typedef typename Split3<kHalf>::out_t out_t;
#define PNP_LN(C)                                                                                                             \
    PNP_LAUNCH(kLayernormSplit, st, (layernorm_split3_kernel<C, kHalf><<<grid, 32 * wpb, 0, st>>>(                             \
                                        x, residual, res_scale, residual_bias, x_out, gamma, beta, eps, reinterpret_cast<out_t *>(out3), \
                                        out1, M, K, hi_scale, flag, ld3, tail_one)))
    if (chunks <= 6) PNP_LN(6);
    else if (chunks <= 8) PNP_LN(8);
    else PNP_LN(16);
#undef PNP_LN
    return launch_status();
}
bool ln_args_ok(const float *x, const float *residual, const float *residual_bias, const float *x_out, const float *gamma,
                const float *beta, const void *out3, const float *out1, long long M, int K) {
    return x && gamma && beta && (out3 || out1) && M >= 0 && K >= 4 && K % 4 == 0 && K <= 128 * 16 && aligned16(x) &&
           (!out3 || aligned16(out3)) && (!out1 || aligned16(out1)) && aligned16(gamma) && aligned16(beta) &&
           (!residual || aligned16(residual)) && (!residual_bias || (residual && aligned16(residual_bias))) &&
           (!x_out || (residual && aligned16(x_out)));
}
}  // namespace

extern "C" int pnp_tf32_split3(const float *x, float *out3, long long M, int K, pnp_stream_t stream) {
    if (!x || !out3 || M < 0 || K < 4 || K % 4 || !aligned16(x) || !aligned16(out3)) return PNP_ERR_INVALID_ARGUMENT;
    if (M == 0) return PNP_OK;
    return run_split3<false>(x, out3, M, K, 1.0f, 1.0f, nullptr, as_stream(stream));
}

extern "C" int pnp_gelu_tf32_split3(const float *x, const float *bias, float *out3, long long M, int K, pnp_stream_t stream) {
    if (!x || !out3 || M < 0 || K < 4 || K % 4 || !aligned16(x) || !aligned16(out3) || (bias && !aligned16(bias)))
        return PNP_ERR_INVALID_ARGUMENT;
    if (M == 0) return PNP_OK;
    return run_gelu_split3<false>(x, bias, out3, M, K, 1.0f, 1.0f, nullptr, as_stream(stream));
}

extern "C" int pnp_layernorm_tf32_split3(const float *x, const float *residual, const float *residual_bias, float *x_out,
                                         const float *gamma, const float *beta, float eps, float *out3, float *out1, long long M,
                                         int K, pnp_stream_t stream) {
    if (!ln_args_ok(x, residual, residual_bias, x_out, gamma, beta, out3, out1, M, K)) return PNP_ERR_INVALID_ARGUMENT;
    if (M == 0) return PNP_OK;
    return run_layernorm_split3<false>(x, residual, 1.0f, residual_bias, x_out, gamma, beta, eps, out3, out1, M, K, 1.0f, nullptr,
                                       3 * K, 0.f, as_stream(stream));
}

extern "C" int pnp_fp16_split3(const float *x, float in_scale, float hi_scale, uint16_t *out3, int *overflow_flag, long long M, int K,
                               pnp_stream_t stream) {
    if (!x || !out3 || M < 0 || K < 4 || K % 4 || !aligned16(x) || (reinterpret_cast<uintptr_t>(out3) & 7)) return PNP_ERR_INVALID_ARGUMENT;
    if (M == 0) return PNP_OK;
    return run_split3<true>(x, out3, M, K, in_scale, hi_scale, overflow_flag, as_stream(stream));
}

extern "C" int pnp_gelu_fp16_split3(const float *x, float in_scale, const float *bias, float hi_scale, uint16_t *out3,
                                    int *overflow_flag, long long M, int K, pnp_stream_t stream) {
    if (!x || !out3 || M < 0 || K < 4 || K % 4 || !aligned16(x) || (reinterpret_cast<uintptr_t>(out3) & 7) || (bias && !aligned16(bias)))
        return PNP_ERR_INVALID_ARGUMENT;
    if (M == 0) return PNP_OK;
    return run_gelu_split3<true>(x, bias, out3, M, K, in_scale, hi_scale, overflow_flag, as_stream(stream));
}

extern "C" int pnp_layernorm_fp16_split3(const float *x, const float *residual, float residual_scale, const float *residual_bias,
                                         float *x_out, const float *gamma, const float *beta, float eps, float hi_scale,
                                         uint16_t *out3, int ld_out3, float bias_one, float *out1, int *overflow_flag, long long M,
                                         int K, pnp_stream_t stream) {
    // the 8 bias columns of a row go out as one 16-byte store at half offset m (3K + 8) + 3K: 16-byte aligned for every m
    // only when K % 8 == 0
    if (out3 && ld_out3 != 3 * K && (ld_out3 != 3 * K + 8 || K % 8 || !aligned16(out3))) return PNP_ERR_INVALID_ARGUMENT;
    if (!x || !gamma || !beta || (!out3 && !out1) || M < 0 || K < 4 || K % 4 || K > 128 * 16 || !aligned16(x) ||
        (out3 && (reinterpret_cast<uintptr_t>(out3) & 7)) || (out1 && !aligned16(out1)) || !aligned16(gamma) || !aligned16(beta) ||
        (residual && !aligned16(residual)) || (residual_bias && (!residual || !aligned16(residual_bias))) ||
        (x_out && (!residual || !aligned16(x_out))))
        return PNP_ERR_INVALID_ARGUMENT;
    if (M == 0) return PNP_OK;
    return run_layernorm_split3<true>(x, residual, residual_scale, residual_bias, x_out, gamma, beta, eps, out3, out1, M, K, hi_scale,
                                      overflow_flag, out3 ? ld_out3 : 3 * K, bias_one, as_stream(stream));
}
