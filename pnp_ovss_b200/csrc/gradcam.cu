// gradcam.cu -- (b) token->class merge and (c) one Salience DropOut round.
// Replaces DRV:810-853 / DRV:656-701 (merge) and DRV:589-603, 623-647, 716-721 (DropOut bookkeeping).
// Both are a few MB per batch: latency-bound, one launch per batch, one CTA per image (or image x class).
#include "common.cuh"

namespace pnp {

__global__ void __launch_bounds__(256) token_merge_kernel(const float *__restrict__ gradcam, const int32_t *__restrict__ seg_start,
                                                          const int32_t *__restrict__ seg_len, const float *__restrict__ seg_div,
                                                          float *__restrict__ class_maps, int Tm, int PP, int C, int row_offset) {
    const int c = blockIdx.x, b = blockIdx.y;
    const int start = seg_start[b * C + c], len = seg_len[b * C + c];
    const float div = seg_div[b * C + c];
    const float *g = gradcam + ((long long)b * Tm + row_offset + start) * PP;
    float *out = class_maps + ((long long)b * C + c) * PP;
    for (int p = threadIdx.x; p < PP; p += blockDim.x) {
        float acc = 0.f;
        if (len > 0) {
            acc = g[p];  // first piece is copied, continuations are added in order (DRV:826, 837-841)
            for (int i = 1; i < len; ++i) acc = __fadd_rn(acc, g[(long long)i * PP + p]);
            if (div != 1.0f) acc = __fdiv_rn(acc, div);  // DRV:845
        }
        out[p] = acc;
    }
}

constexpr int kMaxCells = 1024;  // P*P <= 1024 (P <= 32)

// Order-preserving key of a DropOut score under numpy's sort order: -0 ties with +0, and every NaN ties with the
// others above +inf (np.argsort puts NaN last).
__device__ __forceinline__ unsigned int score_key(float s) {
    if (s != s) return 0xFFFFFFFFu;
    const unsigned int u = __float_as_uint(s == 0.f ? 0.f : s);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(512) salience_dropout_round_kernel(const float *__restrict__ gradcam, float *__restrict__ ensemble_r,
                                                                     float *__restrict__ agg, int32_t *__restrict__ chosen,
                                                                     int chosen_stride, int n_prev, float *__restrict__ imgs,
                                                                     float *__restrict__ norm_imgs, int Tm, int P, int patch,
                                                                     int row_lo, int row_hi, int save_len, int round) {
    __shared__ unsigned int s_key[kMaxCells];
    __shared__ unsigned char s_dropped[kMaxCells];
    __shared__ int s_new[32];
    const int b = blockIdx.x;
    const int PP = P * P;
    const int S = P * patch;
    for (int p = threadIdx.x; p < PP; p += blockDim.x) s_dropped[p] = 0;
    __syncthreads();
    int32_t *my_chosen = chosen + (long long)b * chosen_stride;
    for (int i = threadIdx.x; i < n_prev; i += blockDim.x) {
        int idx = my_chosen[i];
        if (idx >= 0 && idx < PP) s_dropped[idx] = 1;
    }
    __syncthreads();

    // DRV:623-635 + DRV:716-721: pred = map with dropped cells zeroed; agg = m0 + sum_r m_r (m0 twice)
    const float *g = gradcam + (long long)b * Tm * PP;
    for (int i = threadIdx.x; i < Tm * PP; i += blockDim.x) {
        int p = i % PP;
        float v = s_dropped[p] ? 0.f : g[i];
        long long o = (long long)b * Tm * PP + i;
        if (ensemble_r) ensemble_r[o] = v;
        if (agg) agg[o] = (round == 0) ? __fadd_rn(v, v) : __fadd_rn(agg[o], v);
    }

    // DRV:638-642: score = sum over class-token rows of the UNZEROED map, then dropped cells := 0
    for (int p = threadIdx.x; p < PP; p += blockDim.x) {
        float acc = 0.f;
        for (int t = row_lo; t < row_hi; ++t) acc = __fadd_rn(acc, g[(long long)t * PP + p]);
        s_key[p] = score_key(s_dropped[p] ? 0.f : acc);
    }
    __syncthreads();

    // DRV:643-647: argsort(score, kind="stable")[-save_len:] by rank counting (ties: larger index ranks higher).
    // (key, index) is a total order, so the ranks are a permutation of 0..PP-1 and every s_new slot is written
    // exactly once, whatever the scores hold.
    for (int p = threadIdx.x; p < PP; p += blockDim.x) {
        const unsigned int kp = s_key[p];
        int rank = 0;
        for (int q = 0; q < PP; ++q) {
            const unsigned int kq = s_key[q];
            rank += (kq > kp) || (kq == kp && q > p);
        }
        if (rank < save_len) s_new[save_len - 1 - rank] = p;
    }
    __syncthreads();
    if ((int)threadIdx.x < save_len) my_chosen[n_prev + threadIdx.x] = s_new[threadIdx.x];

    // DRV:597-603: zero the 16x16 pixel blocks of the new cells for the next round's model pass
    const int per_cell = 3 * patch * patch;
    for (int i = threadIdx.x; i < save_len * per_cell; i += blockDim.x) {
        int j = i / per_cell, e = i % per_cell;
        int ch = e / (patch * patch), dy = (e / patch) % patch, dx = e % patch;
        int cell = s_new[j];
        int y = (cell / P) * patch + dy, x = (cell % P) * patch + dx;
        if (imgs) imgs[(((long long)b * 3 + ch) * S + y) * S + x] = 0.f;
        if (norm_imgs) norm_imgs[(((long long)b * S + y) * S + x) * 3 + ch] = 0.f;
    }
}

}  // namespace pnp

using namespace pnp;

extern "C" int pnp_token_merge(const float *gradcam, const int32_t *seg_start, const int32_t *seg_len, const float *seg_div,
                               float *class_maps, int B, int Tm, int PP, int C, int row_offset, pnp_stream_t stream) {
    if (!gradcam || !seg_start || !seg_len || !seg_div || !class_maps || B < 0 || C < 0 || Tm < 1 || PP < 1 || row_offset < 0)
        return PNP_ERR_INVALID_ARGUMENT;
    if (B == 0 || C == 0) return PNP_OK;
    if (B > 65535) return PNP_ERR_INVALID_ARGUMENT;
    cudaStream_t st = as_stream(stream);
    PNP_LAUNCH(kTokenMerge, st, token_merge_kernel<<<dim3(C, B), 256, 0, st>>>(gradcam, seg_start, seg_len, seg_div, class_maps, Tm, PP,
                                                                               C, row_offset));
    return launch_status();
}

extern "C" int pnp_salience_dropout_round(const float *gradcam, float *ensemble_r, float *agg, int32_t *chosen,
                                          int chosen_stride, int n_prev, float *imgs, float *norm_imgs, int B, int Tm,
                                          int P, int patch, int row_lo, int row_hi, int save_len, int round,
                                          pnp_stream_t stream) {
    if (!gradcam || !chosen || B < 0 || Tm < 1 || P < 1 || P * P > kMaxCells || patch < 1 || save_len < 1 || save_len > 32 ||
        save_len > P * P || n_prev < 0 || n_prev + save_len > chosen_stride || row_lo < 0 || row_hi > Tm || round < 0)
        return PNP_ERR_INVALID_ARGUMENT;
    if (B == 0) return PNP_OK;
    cudaStream_t st = as_stream(stream);
    PNP_LAUNCH(kDropoutRound, st, salience_dropout_round_kernel<<<B, 512, 0, st>>>(gradcam, ensemble_r, agg, chosen, chosen_stride,
                                                                                   n_prev, imgs, norm_imgs, Tm, P, patch, row_lo,
                                                                                   row_hi, save_len, round));
    return launch_status();
}
