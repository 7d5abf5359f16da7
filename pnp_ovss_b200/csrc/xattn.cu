// xattn.cu -- (a) block-8 cross-attention softmax fused with capture, and its backward fused with GradCAM.
// Replaces MED:267-283 (softmax + save_attention_map + register_hook) and BITM:415-433 (cam*clamp(grad)*mask).
//
// One warp owns one [K]-wide row (K = P*P+1 = 442 / 785 / 1025): the row lives in registers between the
// max, the sum and the normalisation, so scores are read once and probs written once (8 B/element forward,
// 12 B/element backward + the GradCAM side-write).  Rows are only 8-byte aligned (K is odd or 2 mod 4), so
// accesses are lane-strided 32-bit: each warp instruction still covers one fully used 128-byte line.
#include "common.cuh"

namespace pnp {

template <int kItems>  // row fits 32*kItems elements
__global__ void __launch_bounds__(256) softmax_fwd_kernel(const float *__restrict__ scores, const float *__restrict__ key_mask,
                                                          float *__restrict__ probs, long long n_rows, int rows_per_batch,
                                                          int K, float scale) {
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    for (long long row = blockIdx.x * (long long)warps_per_block + (threadIdx.x >> 5); row < n_rows;
         row += (long long)gridDim.x * warps_per_block) {
        const float *src = scores + row * K;
        const float *km = key_mask ? key_mask + (row / rows_per_batch) * K : nullptr;
        float v[kItems];
        float mx = -INFINITY;
#pragma unroll
        for (int i = 0; i < kItems; ++i) {
            int k = lane + 32 * i;
            if (k < K) {
                float s = __fmul_rn(src[k], scale);
                if (km) s = __fadd_rn(s, km[k]);
                v[i] = s;
                mx = fmaxf(mx, s);
            } else {
                v[i] = -INFINITY;
            }
        }
        mx = warp_max(mx);
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < kItems; ++i) {
            float e = (lane + 32 * i < K) ? expf(v[i] - mx) : 0.f;
            v[i] = e;
            sum += e;
        }
        sum = warp_sum(sum);
        float *dst = probs + row * K;
#pragma unroll
        for (int i = 0; i < kItems; ++i) {
            int k = lane + 32 * i;
            if (k < K) dst[k] = __fdiv_rn(v[i], sum);
        }
    }
}

// Backward + GradCAM.  kFull: every (b,h,t) row gets dscores; rows of `head` with t>=1 also emit GradCAM.
// !kFull: only those GradCAM rows are visited (frozen-weights mode) and nothing else is read.
template <int kItems, bool kFull>
__global__ void __launch_bounds__(256) softmax_bwd_gradcam_kernel(const float *__restrict__ probs, const float *__restrict__ dprobs,
                                                                  float *__restrict__ dscores, const int64_t *__restrict__ token_mask,
                                                                  int token_mask_stride, float *__restrict__ gradcam,
                                                                  long long n_rows, int heads, int T, int K, float scale, int head) {
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    for (long long r = blockIdx.x * (long long)warps_per_block + (threadIdx.x >> 5); r < n_rows;
         r += (long long)gridDim.x * warps_per_block) {
        long long row;  // index into [B,heads,T]
        int b, h, t;
        if (kFull) {
            row = r;
            t = (int)(row % T);
            h = (int)((row / T) % heads);
            b = (int)(row / ((long long)T * heads));
        } else {
            b = (int)(r / (T - 1));
            t = (int)(r % (T - 1)) + 1;
            h = head;
            row = ((long long)b * heads + h) * T + t;
        }
        const float *p = probs + row * K;
        const float *dp = dprobs + row * K;
        const bool cam_row = gradcam != nullptr && h == head && t >= 1;
        float m = 0.f;
        if (cam_row) m = (float)token_mask[(long long)b * token_mask_stride + t];
        float *g = cam_row ? gradcam + ((long long)b * (T - 1) + (t - 1)) * (K - 1) : nullptr;
        float pv[kItems], dv[kItems];
        float inner = 0.f;
#pragma unroll
        for (int i = 0; i < kItems; ++i) {
            int k = lane + 32 * i;
            if (k < K) {
                pv[i] = p[k];
                dv[i] = dp[k];
                if (kFull) inner = fmaf(pv[i], dv[i], inner);
                if (cam_row && k >= 1) {
                    // BITM:427: cams * grads.clamp(0) * mask   (left to right, separately rounded).  torch's clamp
                    // keeps a NaN gradient NaN; fmaxf alone would turn it into 0.
                    const float dc = dv[i] != dv[i] ? dv[i] : fmaxf(dv[i], 0.f);
                    g[k - 1] = __fmul_rn(__fmul_rn(pv[i], dc), m);
                }
            } else {
                pv[i] = 0.f;
                dv[i] = 0.f;
            }
        }
        if (kFull) {
            inner = warp_sum(inner);
            float *ds = dscores + row * K;
#pragma unroll
            for (int i = 0; i < kItems; ++i) {
                int k = lane + 32 * i;
                if (k < K) ds[k] = pv[i] * (dv[i] - inner) * scale;
            }
        }
    }
}

}  // namespace pnp

using namespace pnp;

extern "C" int pnp_xattn_softmax_fwd(const float *scores, const float *key_mask, float *probs, int B, int heads, int T,
                                     int K, float scale, pnp_stream_t stream) {
    if (!scores || !probs || B < 0 || heads < 1 || T < 1 || K < 1 || K > 32 * 36) return PNP_ERR_INVALID_ARGUMENT;
    long long n_rows = (long long)B * heads * T;
    if (n_rows == 0) return PNP_OK;
    cudaStream_t st = as_stream(stream);
    int grid = (int)min((long long)kNumSMs * 8, (n_rows + 7) / 8);
    if (K <= 32 * 16)
        PNP_LAUNCH(kSoftmaxFwd, st, softmax_fwd_kernel<16><<<grid, 256, 0, st>>>(scores, key_mask, probs, n_rows, heads * T, K, scale));
    else
        PNP_LAUNCH(kSoftmaxFwd, st, softmax_fwd_kernel<36><<<grid, 256, 0, st>>>(scores, key_mask, probs, n_rows, heads * T, K, scale));
    return launch_status();
}

extern "C" int pnp_xattn_softmax_bwd_gradcam(const float *probs, const float *dprobs, float *dscores,
                                             const int64_t *token_mask, int token_mask_stride, float *gradcam, int B,
                                             int heads, int T, int K, float scale, int head, pnp_stream_t stream) {
    if (!probs || !dprobs || B < 0 || heads < 1 || T < 1 || K < 2 || K > 32 * 36) return PNP_ERR_INVALID_ARGUMENT;
    if (!dscores && !gradcam) return PNP_ERR_INVALID_ARGUMENT;
    if (gradcam && (!token_mask || token_mask_stride < T || head < 0 || head >= heads)) return PNP_ERR_INVALID_ARGUMENT;
    cudaStream_t st = as_stream(stream);
    const bool full = dscores != nullptr;
    long long n_rows = full ? (long long)B * heads * T : (long long)B * (T - 1);
    if (n_rows == 0) return PNP_OK;
    int grid = (int)min((long long)kNumSMs * 8, (n_rows + 7) / 8);
    const bool small = K <= 32 * 16;
    if (full) {
        if (small)
            PNP_LAUNCH(kSoftmaxBwdGradcam, st, softmax_bwd_gradcam_kernel<16, true><<<grid, 256, 0, st>>>(probs, dprobs, dscores, token_mask, token_mask_stride,
                                                                       gradcam, n_rows, heads, T, K, scale, head));
        else
            PNP_LAUNCH(kSoftmaxBwdGradcam, st, softmax_bwd_gradcam_kernel<36, true><<<grid, 256, 0, st>>>(probs, dprobs, dscores, token_mask, token_mask_stride,
                                                                       gradcam, n_rows, heads, T, K, scale, head));
    } else {
        if (small)
            PNP_LAUNCH(kSoftmaxBwdGradcam, st, softmax_bwd_gradcam_kernel<16, false><<<grid, 256, 0, st>>>(probs, dprobs, dscores, token_mask, token_mask_stride,
                                                                        gradcam, n_rows, heads, T, K, scale, head));
        else
            PNP_LAUNCH(kSoftmaxBwdGradcam, st, softmax_bwd_gradcam_kernel<36, false><<<grid, 256, 0, st>>>(probs, dprobs, dscores, token_mask, token_mask_stride,
                                                                        gradcam, n_rows, heads, T, K, scale, head));
    }
    return launch_status();
}
