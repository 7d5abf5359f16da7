// confusion.cu -- (f) argmax over channels, relabel LUT, mIoU confusion-matrix histogram.
// Replaces DRV:387 / DRV:1073 (argmax), DRV:390-399 / DRV:468-480 (relabel), DRV:1106-1112 (_fast_hist).
// HBM-bound: argmax streams C*N floats once with 128-bit loads; the histogram streams labels + gt once (128-bit loads, four
// pixels per thread, when N % 4 == 0) and keeps its bins in shared memory, fed by warp-aggregated atomics (one atomic per
// distinct bin per warp).
#include "common.cuh"

namespace pnp {

// ------------------------------------------------------------------ argmax over channels, 4 pixels/thread
// first maximum wins; NaN counts as the maximum and the first NaN wins (numpy.argmax / torch.argmax).
__device__ __forceinline__ void argmax_step(float v, int c, float &best, int &bi) {
    if (!(best != best) && (v > best || v != v)) {
        best = v;
        bi = c;
    }
}

__global__ void __launch_bounds__(256) argmax_channels_vec4(const float *__restrict__ maps, int32_t *__restrict__ labels,
                                                            int C, int N4, long long total4) {
    // maps [B,C,N], N = 4*N4; one thread owns 4 consecutive pixels of one image
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
        long long b = i / N4;
        int q = (int)(i - b * N4);
        const float *base = maps + (b * C) * (long long)N4 * 4 + (long long)q * 4;
        float4 best = ldg_stream4(base);
        int4 bi = make_int4(0, 0, 0, 0);
        for (int c = 1; c < C; ++c) {
            float4 v = ldg_stream4(base + (long long)c * N4 * 4);
            argmax_step(v.x, c, best.x, bi.x);
            argmax_step(v.y, c, best.y, bi.y);
            argmax_step(v.z, c, best.z, bi.z);
            argmax_step(v.w, c, best.w, bi.w);
        }
        *reinterpret_cast<int4 *>(labels + i * 4) = bi;
    }
}

__global__ void __launch_bounds__(256) argmax_channels_scalar(const float *__restrict__ maps, int32_t *__restrict__ labels,
                                                              int C, int N, long long total) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        long long b = i / N;
        int p = (int)(i - b * N);
        const float *base = maps + (b * C) * (long long)N + p;
        float best = base[0];
        int bi = 0;
        for (int c = 1; c < C; ++c) argmax_step(base[(long long)c * N], c, best, bi);
        labels[i] = bi;
    }
}

// ------------------------------------------------------------------ confusion matrix
// Warp-aggregated increment: lanes holding the same bin elect a leader which adds the group's size.
template <typename CounterT>
__device__ __forceinline__ void warp_aggregated_inc(CounterT *bins, int bin, bool valid) {
    unsigned active = __ballot_sync(0xffffffffu, valid);
    if (!valid) return;
    unsigned peers = __match_any_sync(active, bin);
    int leader = __ffs(peers) - 1;
    if ((int)(threadIdx.x & 31) == leader) atomicAdd(&bins[bin], (CounterT)__popc(peers));
}

// kVec: N % 4 == 0 and 16-byte aligned arrays -> every thread owns 4 consecutive pixels of one image per round and moves
// them with one 128-bit load per input array (labels, ground truth) and one 128-bit store (pred_out).
template <bool kSmemBins, bool kVec>
__global__ void __launch_bounds__(512) confusion_kernel(const int32_t *__restrict__ labels, const float *__restrict__ gt,
                                                        const int32_t *__restrict__ lut, int lut_stride,
                                                        float *__restrict__ pred_out, unsigned long long *__restrict__ hist,
                                                        int32_t *__restrict__ bad_count, int N, long long total,
                                                        int n_class) {
    extern __shared__ unsigned int s_bins[];
    constexpr int V = kVec ? 4 : 1;
    const int n_bins = n_class * n_class;
    if (kSmemBins) {
        for (int i = threadIdx.x; i < n_bins; i += blockDim.x) s_bins[i] = 0u;
        __syncthreads();
    }
    int bad = 0;
    // every lane of a warp runs the same number of iterations (match_any needs convergent warps)
    const long long items = total / V;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long rounds = (items + stride - 1) / stride;
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    for (long long r = 0; r < rounds; ++r, i += stride) {
        const bool in_range = i < items;
        int lab[V];
        float g[V];
        bool valid[V];
        int bin[V];
        float pred_f[V];
#pragma unroll
        for (int v = 0; v < V; ++v) { valid[v] = false; bin[v] = 0; pred_f[v] = 0.f; lab[v] = 0; g[v] = -1.f; }
        if (in_range) {
            if (kVec) {
                const int4 l4 = __ldg(reinterpret_cast<const int4 *>(labels) + i);
                const float4 g4 = __ldg(reinterpret_cast<const float4 *>(gt) + i);
                lab[0] = l4.x; lab[V > 1 ? 1 : 0] = l4.y; lab[V > 2 ? 2 : 0] = l4.z; lab[V > 3 ? 3 : 0] = l4.w;
                g[0] = g4.x; g[V > 1 ? 1 : 0] = g4.y; g[V > 2 ? 2 : 0] = g4.z; g[V > 3 ? 3 : 0] = g4.w;
            } else {
                lab[0] = labels[i];
                g[0] = gt[i];
            }
            const long long b = (i * V) / N;   // N % V == 0: the V pixels of an item belong to one image
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const int pred = lut ? __ldg(lut + b * lut_stride + lab[v]) : lab[v];
                pred_f[v] = (float)pred;
                if (g[v] >= 0.0f && g[v] < (float)n_class) {  // DRV:1107 mask, evaluated on the float32 ground truth
                    if (pred >= 0 && pred < n_class) {
                        valid[v] = true;
                        bin[v] = n_class * (int)g[v] + pred;  // .astype(int) truncates toward zero
                    } else {
                        ++bad;
                    }
                }
            }
            if (pred_out) {
                if (kVec) reinterpret_cast<float4 *>(pred_out)[i] = make_float4(pred_f[0], pred_f[V > 1 ? 1 : 0], pred_f[V > 2 ? 2 : 0], pred_f[V > 3 ? 3 : 0]);
                else pred_out[i] = pred_f[0];
            }
        }
#pragma unroll
        for (int v = 0; v < V; ++v) {
            if (kSmemBins)
                warp_aggregated_inc<unsigned int>(s_bins, bin[v], valid[v]);
            else
                warp_aggregated_inc<unsigned long long>(hist, bin[v], valid[v]);
        }
    }
    if (bad_count && bad) atomicAdd(bad_count, bad);
    if (kSmemBins) {
        __syncthreads();
        for (int k = threadIdx.x; k < n_bins; k += blockDim.x) {
            unsigned int v = s_bins[k];
            if (v) atomicAdd(&hist[k], (unsigned long long)v);
        }
    }
}

// ------------------------------------------------------------------ label map + confidence (no ground truth)
// ids[p] = lut[b, labels[p]], conf[p] = Q[p, labels[p]] (Q pixel-major [B,N,Cp]); a label outside [0, lut_stride) gives -1 in
// both.  kVec: N % 4 == 0 and 16-byte aligned labels / ids / conf -> four consecutive pixels of one image per thread, one
// 128-bit streaming load of labels and one 128-bit store per output.  The lut and Q reads are gathers (one word per pixel).
// Timed by the in-situ profiler as the relabel stage it stands in for (kConfusion).
__device__ __forceinline__ void label_one(int lab, long long b, long long pix, const int32_t *__restrict__ lut, int lut_stride,
                                          const float *__restrict__ Q, int Cp, int &id, float &conf) {
    id = -1;
    conf = -1.f;
    if (lab >= 0 && lab < lut_stride) {
        id = __ldg(lut + b * lut_stride + lab);
        if (Q) conf = __ldg(Q + pix * Cp + lab);
    }
}

template <bool kVec>
__global__ void __launch_bounds__(256) label_map_kernel(const int32_t *__restrict__ labels, const int32_t *__restrict__ lut,
                                                        int lut_stride, const float *__restrict__ Q, int Cp,
                                                        int32_t *__restrict__ ids_out, float *__restrict__ conf_out, int N,
                                                        long long total) {
    constexpr int V = kVec ? 4 : 1;
    const long long items = total / V;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < items; i += (long long)gridDim.x * blockDim.x) {
        const long long p0 = i * V;
        const long long b = p0 / N;   // N % V == 0: the V pixels of an item belong to one image
        int lab[V], id[V];
        float conf[V];
        if (kVec) {   // int32 moved through the f32 streaming load / store: bit patterns pass unchanged
            const float4 l4 = ldg_stream4(reinterpret_cast<const float *>(labels) + p0);
            lab[0] = __float_as_int(l4.x); lab[V > 1 ? 1 : 0] = __float_as_int(l4.y);
            lab[V > 2 ? 2 : 0] = __float_as_int(l4.z); lab[V > 3 ? 3 : 0] = __float_as_int(l4.w);
        } else {
            lab[0] = __ldg(labels + p0);
        }
#pragma unroll
        for (int v = 0; v < V; ++v) label_one(lab[v], b, p0 + v, lut, lut_stride, Q, Cp, id[v], conf[v]);
        if (kVec) {
            stg_stream4(reinterpret_cast<float *>(ids_out) + p0, make_float4(__int_as_float(id[0]), __int_as_float(id[V > 1 ? 1 : 0]),
                                                                              __int_as_float(id[V > 2 ? 2 : 0]), __int_as_float(id[V > 3 ? 3 : 0])));
            if (conf_out) stg_stream4(conf_out + p0, make_float4(conf[0], conf[V > 1 ? 1 : 0], conf[V > 2 ? 2 : 0], conf[V > 3 ? 3 : 0]));
        } else {
            ids_out[p0] = id[0];
            if (conf_out) conf_out[p0] = conf[0];
        }
    }
}

}  // namespace pnp

using namespace pnp;

extern "C" int pnp_argmax_channels(const float *maps, int32_t *labels, int B, int C, int N, pnp_stream_t stream) {
    if (!maps || !labels || B < 0 || C < 1 || N < 1) return PNP_ERR_INVALID_ARGUMENT;
    if (B == 0) return PNP_OK;
    cudaStream_t st = as_stream(stream);
    const bool vec = (N % 4 == 0) && ((reinterpret_cast<uintptr_t>(maps) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(labels) & 15) == 0);
    if (vec) {
        long long total4 = (long long)B * (N / 4);
        int grid = (int)min((long long)kNumSMs * 16, (total4 + 255) / 256);
        PNP_LAUNCH(kArgmax, st, argmax_channels_vec4<<<grid, 256, 0, st>>>(maps, labels, C, N / 4, total4));
    } else {
        long long total = (long long)B * N;
        int grid = (int)min((long long)kNumSMs * 16, (total + 255) / 256);
        PNP_LAUNCH(kArgmax, st, argmax_channels_scalar<<<grid, 256, 0, st>>>(maps, labels, C, N, total));
    }
    return launch_status();
}

extern "C" int pnp_confusion_accumulate(const int32_t *labels, const float *gt, const int32_t *lut, int lut_stride,
                                        float *pred_out, int64_t *hist, int32_t *bad_count, int B, int N, int n_class,
                                        pnp_stream_t stream) {
    if (!labels || !gt || !hist || B < 0 || N < 1 || n_class < 1 || n_class > 30000) return PNP_ERR_INVALID_ARGUMENT;
    if (B == 0) return PNP_OK;
    cudaStream_t st = as_stream(stream);
    long long total = (long long)B * N;
    size_t smem = (size_t)n_class * n_class * sizeof(unsigned int);
    auto aligned = [](const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    const bool vec = (N % 4 == 0) && aligned(labels) && aligned(gt) && (!pred_out || aligned(pred_out));
    const long long items = vec ? total / 4 : total;
    int grid = (int)std::max<long long>(1, std::min<long long>((long long)kNumSMs * 2, (items + 511) / 512));
    unsigned long long *h = reinterpret_cast<unsigned long long *>(hist);
    if (smem <= 200 * 1024) {
        if (smem > 48 * 1024) {
            cudaError_t e = vec ? allow_smem(confusion_kernel<true, true>, smem) : allow_smem(confusion_kernel<true, false>, smem);
            if (e != cudaSuccess) return cuda_err(e);
            grid = (int)std::max<long long>(1, std::min<long long>((long long)kNumSMs, (items + 511) / 512));
        }
        if (vec)
            PNP_LAUNCH(kConfusion, st, (confusion_kernel<true, true><<<grid, 512, smem, st>>>(labels, gt, lut, lut_stride, pred_out, h, bad_count, N, total, n_class)));
        else
            PNP_LAUNCH(kConfusion, st, (confusion_kernel<true, false><<<grid, 512, smem, st>>>(labels, gt, lut, lut_stride, pred_out, h, bad_count, N, total, n_class)));
    } else {
        if (vec)
            PNP_LAUNCH(kConfusion, st, (confusion_kernel<false, true><<<grid, 512, 0, st>>>(labels, gt, lut, lut_stride, pred_out, h, bad_count, N, total, n_class)));
        else
            PNP_LAUNCH(kConfusion, st, (confusion_kernel<false, false><<<grid, 512, 0, st>>>(labels, gt, lut, lut_stride, pred_out, h, bad_count, N, total, n_class)));
    }
    return launch_status();
}

extern "C" int pnp_label_map(const int32_t *labels, const int32_t *lut, int lut_stride, const float *Q, int Cp, int32_t *ids_out,
                             float *conf_out, int B, int N, pnp_stream_t stream) {
    if (!labels || !lut || !ids_out || lut_stride < 1 || B < 0 || N < 1) return PNP_ERR_INVALID_ARGUMENT;
    if ((Q == nullptr) != (conf_out == nullptr)) return PNP_ERR_INVALID_ARGUMENT;
    if (Q && Cp < lut_stride) return PNP_ERR_INVALID_ARGUMENT;   // every label the lut accepts must be a channel of Q
    if (B == 0) return PNP_OK;
    cudaStream_t st = as_stream(stream);
    auto aligned = [](const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    const bool vec = (N % 4 == 0) && aligned(labels) && aligned(ids_out) && (!conf_out || aligned(conf_out));
    const long long total = (long long)B * N;
    const long long items = vec ? total / 4 : total;
    const int grid = (int)std::max<long long>(1, std::min<long long>((long long)kNumSMs * 16, (items + 255) / 256));
    if (vec)
        PNP_LAUNCH(kConfusion, st, (label_map_kernel<true><<<grid, 256, 0, st>>>(labels, lut, lut_stride, Q, Cp, ids_out, conf_out, N, total)));
    else
        PNP_LAUNCH(kConfusion, st, (label_map_kernel<false><<<grid, 256, 0, st>>>(labels, lut, lut_stride, Q, Cp, ids_out, conf_out, N, total)));
    return launch_status();
}
