// upsample_blur.cu -- (d) threshold + bilinear upsample (+Scale_0_1) + background, and the Gaussian blur.
// Replaces DRV:348-380 / DRV:424-455 / DRV:1078-1094 and DRV:1149-1153 (scipy gaussian_filter) + DRV:1005-1011.
//
// upsample: the PxP grids are tiny (L1-resident); the kernel is a pure HBM write stream of C'*H*W floats with
//           128-bit stores -- the algorithmic minimum 4*C'*N bytes per image.
// blur:     separable, smem-tiled.  Pass V (axis 0) stages a 64-column strip of the map with its reflected halo
//           in shared memory and register-blocks 16 output rows per thread; pass H (axis 1) stages 32 full rows,
//           maps lanes to rows (odd pitch -> conflict-free) and register-blocks 16 output columns per thread,
//           then stores through shared memory so global writes are coalesced 128-bit.  Min/max of each blurred
//           map is reduced in the same pass (order-preserving uint keys + atomicMin/Max), so the reference's
//           (y-min)/(max-min) costs 2 scalars per channel in the consumer instead of another pass over HBM.
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace pnp {

// ============================================================================================ upsample
constexpr int kMaxP2 = 1024;

// K1: per (b,c): min-max threshold of the PxP map; optional min/max of its upsampled image (for Scale_0_1)
__global__ void __launch_bounds__(256) threshold_prep_kernel(const float *__restrict__ class_maps, float *__restrict__ masked,
                                                             float *__restrict__ scale_params, int C, int P, int H, int W,
                                                             float threshold, int rescale, const int32_t *__restrict__ n_classes) {
    __shared__ float s_grid[kMaxP2];
    __shared__ float s_red[2][8];
    __shared__ float s_mm[2];
    const int c = blockIdx.x, b = blockIdx.y;
    const int PP = P * P;
    const long long base = ((long long)b * C + c) * PP;
    if (n_classes) {   // a batch padded to C classes: image b has n_classes[b] of them (and is rescaled only with more than one)
        const int Cb = n_classes[b];
        if (c >= Cb) return;
        rescale = rescale && Cb > 1;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    float mn = INFINITY, mx = -INFINITY;
    for (int p = threadIdx.x; p < PP; p += blockDim.x) {
        float v = class_maps[base + p];
        s_grid[p] = v;
        mn = nan_min(mn, v);
        mx = nan_max(mx, v);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mn = nan_min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = nan_max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) { s_red[0][warp] = mn; s_red[1][warp] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = s_red[0][0], z = s_red[1][0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { a = nan_min(a, s_red[0][w]); z = nan_max(z, s_red[1][w]); }
        s_mm[0] = a; s_mm[1] = z;
    }
    __syncthreads();
    mn = s_mm[0];
    const float range = __fsub_rn(s_mm[1], mn);
    // DRV:425-433: th = (x-min)/(max-min) >= threshold (0/0 -> NaN -> False); pred = x * th
    for (int p = threadIdx.x; p < PP; p += blockDim.x) {
        float v = s_grid[p];
        float nrm = __fdiv_rn(__fsub_rn(v, mn), range);
        float keep = (nrm >= threshold) ? v : __fmul_rn(v, 0.0f);
        s_grid[p] = keep;
        masked[base + p] = keep;
    }
    if (!rescale) return;
    __syncthreads();
    // min/max of the upsampled image (needed by Scale_0_1, DRV:1078-1094): evaluate, never store
    const float rh = (H > 1) ? (float)(P - 1) / (float)(H - 1) : 0.f;
    const float rw = (W > 1) ? (float)(P - 1) / (float)(W - 1) : 0.f;
    mn = INFINITY; mx = -INFINITY;
    for (int i = threadIdx.x; i < H * W; i += blockDim.x) {
        int y = i / W, x = i - y * W;
        float sy = rh * y, sx = rw * x;
        int y0 = min((int)sy, P - 1), x0 = min((int)sx, P - 1);
        int y1 = min(y0 + 1, P - 1), x1 = min(x0 + 1, P - 1);
        float ly = fminf(fmaxf(sy - y0, 0.f), 1.f), lx = fminf(fmaxf(sx - x0, 0.f), 1.f);
        float hy = 1.f - ly, hx = 1.f - lx;
        float top = __fadd_rn(__fmul_rn(hx, s_grid[y0 * P + x0]), __fmul_rn(lx, s_grid[y0 * P + x1]));
        float bot = __fadd_rn(__fmul_rn(hx, s_grid[y1 * P + x0]), __fmul_rn(lx, s_grid[y1 * P + x1]));
        float v = __fadd_rn(__fmul_rn(hy, top), __fmul_rn(ly, bot));
        mn = nan_min(mn, v);
        mx = nan_max(mx, v);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mn = nan_min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = nan_max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __syncthreads();
    if (lane == 0) { s_red[0][warp] = mn; s_red[1][warp] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = s_red[0][0], z = s_red[1][0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { a = nan_min(a, s_red[0][w]); z = nan_max(z, s_red[1][w]); }
        scale_params[((long long)b * C + c) * 2 + 0] = a;
        scale_params[((long long)b * C + c) * 2 + 1] = __fsub_rn(z, a);  // max of (x - min)
    }
}

// K2: write out[b, bg + c, y, x..x+VEC) for all c, plus the background channel.
// kBgOnly: evaluate every channel exactly as above but store ONLY the background indicator, to out [B,H,W] (the fused
// low-rank path blurs the class channels from their PxP grids and needs the full-resolution values just for this test).
template <int VEC, bool kBgOnly = false>
__global__ void __launch_bounds__(256) upsample_write_kernel(const float *__restrict__ masked, const float *__restrict__ scale_params,
                                                             float *__restrict__ out, int C, int P, int H, int W, int rescale,
                                                             int with_background, const int32_t *__restrict__ n_classes = nullptr) {
    const int b = blockIdx.y;
    const int PP = P * P;
    const int Cb = n_classes ? n_classes[b] : C;          // classes image b really has (the batch is padded to C)
    if (n_classes) rescale = rescale && Cb > 1;
    const int Wq = W / VEC;
    const long long N = (long long)H * W;
    const int Cout = C + (with_background ? 1 : 0);
    const float rh = (H > 1) ? (float)(P - 1) / (float)(H - 1) : 0.f;
    const float rw = (W > 1) ? (float)(P - 1) / (float)(W - 1) : 0.f;
    const float *grid0 = masked + (long long)b * C * PP;
    float *out_b = out + (long long)b * (kBgOnly ? 1 : Cout) * N;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < H * Wq; q += gridDim.x * blockDim.x) {
        const int y = q / Wq, xb = (q - y * Wq) * VEC;
        const float sy = rh * y;
        const int y0 = min((int)sy, P - 1), y1 = min(y0 + 1, P - 1);
        const float ly = fminf(fmaxf(sy - y0, 0.f), 1.f), hy = 1.f - ly;
        int x0[VEC], x1[VEC];
        float lx[VEC], hx[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            float sx = rw * (xb + v);
            x0[v] = min((int)sx, P - 1);
            x1[v] = min(x0[v] + 1, P - 1);
            lx[v] = fminf(fmaxf(sx - x0[v], 0.f), 1.f);
            hx[v] = 1.f - lx[v];
        }
        float vmax[VEC];
        bool vnan[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) { vmax[v] = -INFINITY; vnan[v] = false; }
        for (int c = 0; c < Cb; ++c) {
            if (kBgOnly) {
                // background = (no NaN) && (max over classes == 0): a pixel is decided (not background) as soon as one class
                // is positive or NaN, and dense maps decide every pixel within the first few classes
                bool all_decided = true;
#pragma unroll
                for (int v = 0; v < VEC; ++v) all_decided = all_decided && (vnan[v] || vmax[v] > 0.f);
                if (all_decided) break;
            }
            const float *g = grid0 + c * PP;
            float mn = 0.f, rg = 1.f;
            if (rescale) { mn = scale_params[((long long)b * C + c) * 2]; rg = scale_params[((long long)b * C + c) * 2 + 1]; }
            float r[VEC];
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                float top = __fadd_rn(__fmul_rn(hx[v], __ldg(g + y0 * P + x0[v])), __fmul_rn(lx[v], __ldg(g + y0 * P + x1[v])));
                float bot = __fadd_rn(__fmul_rn(hx[v], __ldg(g + y1 * P + x0[v])), __fmul_rn(lx[v], __ldg(g + y1 * P + x1[v])));
                float val = __fadd_rn(__fmul_rn(hy, top), __fmul_rn(ly, bot));
                if (rescale) val = __fdiv_rn(__fsub_rn(val, mn), rg);  // Scale_0_1: AA -= min; AA /= max
                r[v] = val;
                vnan[v] = vnan[v] || (val != val);
                vmax[v] = fmaxf(vmax[v], val);
            }
            if (!kBgOnly) {
                float *dst = out_b + (long long)(c + (with_background ? 1 : 0)) * N + (long long)y * W + xb;
                if (VEC == 4)
                    stg_stream4(dst, make_float4(r[0], r[1], r[2], r[3]));
                else
                    dst[0] = r[0];
            }
        }
        if (with_background) {  // DRV:446-450: background = (max over classes == 0); torch.max propagates NaN
            float r[VEC];
#pragma unroll
            for (int v = 0; v < VEC; ++v) r[v] = (!vnan[v] && vmax[v] == 0.f) ? 1.f : 0.f;
            float *dst = out_b + (long long)y * W + xb;
            if (VEC == 4)
                stg_stream4(dst, make_float4(r[0], r[1], r[2], r[3]));
            else
                dst[0] = r[0];
        }
    }
}

// ============================================================================================ blur
__host__ __device__ __forceinline__ int reflect_index(int i, int n) {  // scipy mode='reflect': d c b a | a b c d | d c b a
    if (n == 1) return 0;
    int period = 2 * n;
    i %= period;
    if (i < 0) i += period;
    return i < n ? i : period - 1 - i;
}

constexpr int kTapPad = 16;  // weights are zero-padded so register-blocked loops never branch on the tap count

// weights[j] = exp(-0.5 x^2 / sigma^2) / sum, x = j - lw (float64 like scipy's _gaussian_kernel1d), stored fp32;
// also resets the per-map min/max keys.
__global__ void blur_prologue_kernel(float *__restrict__ weights, unsigned *__restrict__ mm_keys, int n_maps, int lw, int n_w_padded,
                                     double sigma) {
    __shared__ double s_sum;
    const int taps = 2 * lw + 1;
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int j = 0; j < taps; ++j) {
            double x = (double)(j - lw);
            s += exp(-0.5 / (sigma * sigma) * (x * x));
        }
        s_sum = s;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < n_w_padded; j += blockDim.x) {
        double x = (double)(j - lw);
        weights[j] = (j < taps) ? (float)(exp(-0.5 / (sigma * sigma) * (x * x)) / s_sum) : 0.f;
    }
    for (int i = threadIdx.x; i < n_maps; i += blockDim.x) {
        mm_keys[2 * i + 0] = 0xffffffffu;  // running min key
        mm_keys[2 * i + 1] = 0u;           // running max key
    }
}

// acc[r] += sum_j w[j] * v[(j + r) * kStride] over the taps = 2 lw + 1 taps, in chunks of 8 taps (one FMA order for every
// pass and variant).  taps is odd, so the last chunk is partial: its padding taps (weight 0) are skipped rather than
// multiplied, because the staged values they would meet are live data past the tap window, and 0 * NaN or 0 * inf would put
// a NaN up to 7 px beyond the footprint of a non-finite input.  For finite data the result is the same bit for bit.
// kWindowTail: the last chunk loads its sliding window once and predicates the FMAs (the loads of a full chunk; pass V), else
// it runs tap by tap (16 loads a tap, but fewer live registers: the paired pass-H kernel, capped at 40, spills the window).
// Measured on a B200 (profiles/time_blur_passes.py, DESIGN.md section 5), tap by tap is also the faster tail for both pass-H
// kernels.
template <int R, int kStride, bool kWindowTail>
__device__ __forceinline__ void blur_taps(float (&acc)[R], const float *__restrict__ v, const float *__restrict__ w, int taps) {
    int jc = 0;
    for (; jc + 8 <= taps; jc += 8) {
        float vv[R + 7], ww[8];
#pragma unroll
        for (int i = 0; i < R + 7; ++i) vv[i] = v[(jc + i) * kStride];
#pragma unroll
        for (int i = 0; i < 8; ++i) ww[i] = w[jc + i];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = fmaf(ww[i], vv[i + r], acc[r]);
    }
    if (kWindowTail) {   // the last 1..7 taps
        const int rem = taps - jc;
        float vv[R + 6], ww[7];
#pragma unroll
        for (int i = 0; i < R + 6; ++i) vv[i] = v[(jc + i) * kStride];
#pragma unroll
        for (int i = 0; i < 7; ++i) ww[i] = w[jc + i];
#pragma unroll
        for (int i = 0; i < 7; ++i)
            if (i < rem)
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = fmaf(ww[i], vv[i + r], acc[r]);
        return;
    }
    for (; jc < taps; ++jc) {   // the last 1..7 taps, one at a time
        const float wj = w[jc];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = fmaf(wj, v[(jc + r) * kStride], acc[r]);
    }
}

constexpr int kVCols = 64;   // columns per CTA in pass V
constexpr int kVRows = 16;   // output rows per thread per sweep
constexpr int kVGroups = 8;  // row groups per CTA (kVCols * kVGroups = 512 threads)

// pass V: out[y][x] = sum_j w[j] * in[reflect(y + j - lw)][x]
__global__ void __launch_bounds__(kVCols *kVGroups) blur_vertical_kernel(const float *__restrict__ in, float *__restrict__ out,
                                                                         const float *__restrict__ weights, int H, int W, int lw,
                                                                         int tile_rows, int n_w_padded) {
    extern __shared__ float smem[];
    float *s_w = smem;                    // [n_w_padded]
    float *s_in = smem + n_w_padded;      // [tile_rows + 2*lw + kTapPad + kVRows][kVCols]
    const int map = blockIdx.z;
    const int x_base = blockIdx.x * kVCols;
    const int y_base = blockIdx.y * tile_rows;
    const int rows_here = min(tile_rows, H - y_base);
    const int n_virtual = rows_here + 2 * lw;
    const int n_alloc = tile_rows + 2 * lw + kTapPad + kVRows;
    const float *src = in + (long long)map * H * W;
    for (int j = threadIdx.x; j < n_w_padded; j += blockDim.x) s_w[j] = weights[j];
    const int cx = threadIdx.x % kVCols;
    const int gx = x_base + cx;
    for (int r = threadIdx.x / kVCols; r < n_alloc; r += kVGroups) {
        float v = 0.f;
        if (r < n_virtual && gx < W) v = src[(long long)reflect_index(y_base - lw + r, H) * W + gx];
        s_in[r * kVCols + cx] = v;
    }
    __syncthreads();
    float *dst = out + (long long)map * H * W;
    const int grp = threadIdx.x / kVCols;
    for (int yl = grp * kVRows; yl < rows_here; yl += kVGroups * kVRows) {
        float acc[kVRows];
#pragma unroll
        for (int r = 0; r < kVRows; ++r) acc[r] = 0.f;
        blur_taps<kVRows, kVCols, true>(acc, s_in + yl * kVCols + cx, s_w, 2 * lw + 1);
        if (gx < W) {
#pragma unroll
            for (int r = 0; r < kVRows; ++r)
                if (yl + r < rows_here) dst[(long long)(y_base + yl + r) * W + gx] = acc[r];
        }
    }
}

// ---- pass V, TMA variant: the strip (with its reflected halo rows) is brought in by 1-D bulk async copies
// (cp.async.bulk, one 128-byte row segment each, source row = reflect(y)) that complete on an mbarrier, so no thread
// spends issue slots or registers on the tile load; 32-column strips keep the tile at <= 72 KB -> 3 CTAs per SM whose
// load and FMA phases overlap each other.  Needs W % 4 == 0 and 16-byte aligned maps (else the plain kernel runs).
constexpr int kTCols = 32;
constexpr int kTGroups = 8;  // 256 threads

__device__ __forceinline__ void mbar_init(unsigned long long *mbar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(mbar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *mbar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(mbar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *mbar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tWAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}" ::"r"((unsigned)__cvta_generic_to_shared(mbar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void *smem_dst, const void *gmem_src, unsigned bytes, unsigned long long *mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (unsigned)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(mbar))
                 : "memory");
}

__global__ void __launch_bounds__(kTCols *kTGroups) blur_vertical_tma_kernel(const float *__restrict__ in, float *__restrict__ out,
                                                                             const float *__restrict__ weights, int H, int W, int lw,
                                                                             int tile_rows, int n_w_padded) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long s_mbar;
    float *s_w = smem;                // [n_w_padded]  (a multiple of 8 floats: the tile stays 32-byte aligned)
    float *s_in = smem + n_w_padded;  // [tile_rows + 2*lw + kTapPad + kVRows][kTCols]
    const int map = blockIdx.z;
    const int x_base = blockIdx.x * kTCols;
    const int y_base = blockIdx.y * tile_rows;
    const int rows_here = min(tile_rows, H - y_base);
    const int n_virtual = rows_here + 2 * lw;
    const int n_alloc = tile_rows + 2 * lw + kTapPad + kVRows;
    const int cols_here = min(kTCols, W - x_base);  // multiple of 4
    const float *src = in + (long long)map * H * W;
    if (threadIdx.x == 0) {
        mbar_init(&s_mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // warp 0 programs the bulk copies
        if (threadIdx.x == 0) mbar_expect_tx(&s_mbar, (unsigned)(n_virtual * cols_here * 4));
        __syncwarp();
        for (int r = threadIdx.x; r < n_virtual; r += 32)
            bulk_copy_g2s(s_in + r * kTCols, src + (long long)reflect_index(y_base - lw + r, H) * W + x_base, (unsigned)(cols_here * 4),
                          &s_mbar);
    }
    // everything the copies do not write: weights, padding rows, columns past the image edge
    for (int j = threadIdx.x; j < n_w_padded; j += blockDim.x) s_w[j] = weights[j];
    const int cx = threadIdx.x % kTCols;
    for (int r = threadIdx.x / kTCols; r < n_alloc; r += kTGroups)
        if (r >= n_virtual || cx >= cols_here) s_in[r * kTCols + cx] = 0.f;
    __syncthreads();
    mbar_wait(&s_mbar, 0);
    float *dst = out + (long long)map * H * W;
    const int grp = threadIdx.x / kTCols;
    const int gx = x_base + cx;
    for (int yl = grp * kVRows; yl < rows_here; yl += kTGroups * kVRows) {
        float acc[kVRows];
#pragma unroll
        for (int r = 0; r < kVRows; ++r) acc[r] = 0.f;
        blur_taps<kVRows, kTCols, true>(acc, s_in + yl * kTCols + cx, s_w, 2 * lw + 1);
        if (gx < W) {
#pragma unroll
            for (int r = 0; r < kVRows; ++r)
                if (yl + r < rows_here) dst[(long long)(y_base + yl + r) * W + gx] = acc[r];
        }
    }
}

constexpr int kHRows = 32;    // rows per CTA in pass H (one per lane)
constexpr int kHCols = 16;    // output columns per thread per sweep
constexpr int kHGroupsMax = 32;  // column groups (warps) per CTA: as many as one sweep over the tile needs, up to 1024 threads

// pass H: out[y][x] = sum_j w[j] * in[y][reflect(x + j - lw)], + min/max of the result
template <int kMaxWarps, int kMinCtas>
__global__ void __launch_bounds__(kHRows *kMaxWarps, kMinCtas) blur_horizontal_kernel(const float *__restrict__ in, float *__restrict__ out,
                                                                           const float *__restrict__ weights,
                                                                           unsigned *__restrict__ mm_keys, int H, int W, int lw,
                                                                           int tile_cols, int pitch, int n_w_padded) {
    extern __shared__ float smem[];
    float *s_w = smem;                                   // [n_w_padded]
    float *s_in = smem + n_w_padded;                     // [kHRows][pitch]
    const int n_groups = blockDim.x >> 5;                // warps of this CTA, one column group of kHCols outputs each
    float *s_out = s_in + kHRows * pitch;                // [kHRows][n_groups*kHCols + 1]
    const int kOutPitch = n_groups * kHCols + 1;
    __shared__ unsigned s_mm[2];
    const int map = blockIdx.z;
    const int y_base = blockIdx.y * kHRows;
    const int x_base = blockIdx.x * tile_cols;
    const int cols_here = min(tile_cols, W - x_base);
    const int n_virtual = cols_here + 2 * lw;
    const float *src = in + (long long)map * H * W;
    float *dst = out + (long long)map * H * W;
    if (threadIdx.x == 0) { s_mm[0] = 0xffffffffu; s_mm[1] = 0u; }
    for (int j = threadIdx.x; j < n_w_padded; j += blockDim.x) s_w[j] = weights[j];
    for (int i = threadIdx.x; i < kHRows * pitch; i += blockDim.x) {
        int r = i / pitch, v = i - r * pitch;
        float val = 0.f;
        int gy = y_base + r;
        if (v < n_virtual && gy < H) val = src[(long long)gy * W + reflect_index(x_base - lw + v, W)];
        s_in[i] = val;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int gy = y_base + lane;
    float mn = INFINITY, mx = -INFINITY;
    bool has_nan = false, seen = false;   // seen: this thread wrote a pixel (mn == inf also means a map of +inf)
    for (int sweep = 0; sweep < cols_here; sweep += n_groups * kHCols) {
        const int xl = sweep + grp * kHCols;
        if (xl < cols_here) {
            float acc[kHCols];
#pragma unroll
            for (int r = 0; r < kHCols; ++r) acc[r] = 0.f;
            blur_taps<kHCols, 1, false>(acc, s_in + lane * pitch + xl, s_w, 2 * lw + 1);
#pragma unroll
            for (int r = 0; r < kHCols; ++r) s_out[lane * kOutPitch + grp * kHCols + r] = acc[r];
        }
        __syncthreads();
        // coalesced write-back of this sweep's [kHRows][<=256] block, tracking min/max
        const int sweep_cols = min(n_groups * kHCols, cols_here - sweep);
        for (int i = threadIdx.x; i < kHRows * sweep_cols; i += blockDim.x) {
            int r = i / sweep_cols, c = i - r * sweep_cols;
            if (y_base + r < H) {
                float v = s_out[r * kOutPitch + c];
                dst[(long long)(y_base + r) * W + x_base + sweep + c] = v;
                seen = true;
                has_nan = has_nan || (v != v);
                mn = fminf(mn, v);
                mx = fmaxf(mx, v);
            }
        }
        __syncthreads();
    }
    (void)gy;
    unsigned kmin = has_nan ? 0u : f2key(mn), kmax = has_nan ? 0xffffffffu : f2key(mx);
    if (!seen) { kmin = 0xffffffffu; kmax = 0u; }
    for (int o = 16; o > 0; o >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, o));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
    }
    if (lane == 0) { atomicMin(&s_mm[0], kmin); atomicMax(&s_mm[1], kmax); }
    __syncthreads();
    if (threadIdx.x == 0) {
        atomicMin(&mm_keys[2 * map + 0], s_mm[0]);
        atomicMax(&mm_keys[2 * map + 1], s_mm[1]);
    }
}

// decode keys -> (min, max) floats; optional in-place normalisation (y - min) / (max - min)
__global__ void blur_minmax_decode_kernel(const unsigned *__restrict__ mm_keys, float *__restrict__ minmax, int n_maps) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_maps) {
        minmax[2 * i + 0] = key2f(mm_keys[2 * i + 0]);
        minmax[2 * i + 1] = key2f(mm_keys[2 * i + 1]);
    }
}

__global__ void __launch_bounds__(256) blur_normalize_kernel(float *__restrict__ maps, const float *__restrict__ minmax, long long HW,
                                                             long long total) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        long long m = i / HW;
        float mn = minmax[2 * m], mx = minmax[2 * m + 1];
        // DRV:1151-1152: att -= att.min(); att /= att.max()
        maps[i] = __fdiv_rn(__fsub_rn(maps[i], mn), __fsub_rn(mx, mn));
    }
}


// ============================================================================================ fused low-rank (d) group
// The maps that get blurred are bilinear upsamples of PxP grids (thresholded BEFORE upsampling, DRV:425-437), and both the
// upsample and the separable Gaussian are linear and separable, so for a class channel
//     blur(upsample(m)) = (G U_y) m (G U_x)^T = A_y m A_x^T          A_y: H x P,  A_x: W x P   (reflect boundary folded in)
// -- about 2 P multiply-adds per output instead of 2 (2 lw + 1) (42 against 270 at 336 px), and no full-resolution input or
// intermediate at all.  Scale_0_1 (DRV:1078-1094) is an affine map per channel and G's rows sum to one, so it commutes with
// the blur and cancels in the min-max normalisation that follows it (DRV:1151-1152): the class channels never need it.
// Only the background channel -- a non-linear indicator of the full-resolution values (DRV:446-450) -- keeps the direct
// path: indicator at full resolution (same arithmetic as the direct kernels, bit-exact), then the tap-by-tap blur.
//   pass A (one CTA per (image, class)):  T = A_y m (H x P, also stored for pass B), min/max of Y = T A_x^T, never stored
//   pass B (one CTA per row segment):     Y recomputed for every channel of a pixel, normalised, then either
//                                         unary = -log(clip(softmax_c)) written pixel-major for the CRF (DRV:1057-1063),
//                                         or the argmax label (blur-only mode, DRV:1018-1025), or the maps themselves.
constexpr int kLrMaxP = 32;

__global__ void __launch_bounds__(128) lowrank_operator_kernel(float *__restrict__ Ay, float *__restrict__ AxT, int H, int W, int P,
                                                               int PPAD, int lw, double sigma) {
    extern __shared__ double s_w[];   // [2 lw + 1] Gaussian weights (float64, scipy _gaussian_kernel1d), built by the whole CTA
    __shared__ double s_part[128];
    const int taps = 2 * lw + 1;
    double part = 0.0;
    for (int j = threadIdx.x; j < taps; j += blockDim.x) {
        const double x = (double)(j - lw);
        const double w = exp(-0.5 / (sigma * sigma) * (x * x));
        s_w[j] = w;
        part += w;
    }
    s_part[threadIdx.x] = part;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) s_part[threadIdx.x] += s_part[threadIdx.x + o];
        __syncthreads();
    }
    const double inv_sum = 1.0 / s_part[0];
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= H + W) return;
    const bool is_y = t < H;
    const int n = is_y ? H : W, pos = is_y ? t : t - H;
    const float r = (n > 1) ? (float)(P - 1) / (float)(n - 1) : 0.f;  // align_corners=True scale, as upsample_write_kernel
    double acc[kLrMaxP];
#pragma unroll
    for (int i = 0; i < kLrMaxP; ++i) acc[i] = 0.0;
    for (int j = 0; j < taps; ++j) {
        const double w = s_w[j] * inv_sum;
        const int src = reflect_index(pos + j - lw, n);
        const float sp = r * src;
        const int i0 = min((int)sp, P - 1), i1 = min(i0 + 1, P - 1);
        const float l = fminf(fmaxf(sp - i0, 0.f), 1.f), h = 1.f - l;
        acc[i0] += w * (double)h;
        acc[i1] += w * (double)l;
    }
    for (int i = 0; i < PPAD; ++i) {
        const float v = (i < P) ? (float)acc[i] : 0.f;
        if (is_y) Ay[(size_t)pos * PPAD + i] = v;
        else AxT[(size_t)i * W + pos] = v;
    }
}

// Y = sum_j t[j] * ax[j], j ascending, one fmaf chain: pass A and pass B must produce bit-identical values
template <int PPAD>
__device__ __forceinline__ float lr_dot(const float *__restrict__ t_row, const float (&ax)[PPAD]) {
    float y = 0.f;
#pragma unroll
    for (int q = 0; q < PPAD / 4; ++q) {
        const float4 t = *reinterpret_cast<const float4 *>(t_row + 4 * q);
        y = fmaf(t.x, ax[4 * q + 0], y);
        y = fmaf(t.y, ax[4 * q + 1], y);
        y = fmaf(t.z, ax[4 * q + 2], y);
        y = fmaf(t.w, ax[4 * q + 3], y);
    }
    return y;
}

template <int PPAD>
__global__ void __launch_bounds__(512) lowrank_minmax_kernel(const float *__restrict__ masked, const float *__restrict__ Ay,
                                                             const float *__restrict__ AxT, float *__restrict__ T,
                                                             float *__restrict__ norm, float *__restrict__ minmax_out, int C, int P,
                                                             int H, int W, int rows_chunk, int out_channel_offset, int out_channels,
                                                             const int32_t *__restrict__ n_classes) {
    extern __shared__ __align__(16) float lr_smem[];
    if (n_classes && (int)blockIdx.x >= n_classes[blockIdx.y]) return;   // a class this image does not have
    float *s_m = lr_smem;                   // [PPAD][PPAD] the thresholded grid, zero padded
    float *s_T = lr_smem + PPAD * PPAD;     // [rows_chunk][PPAD]
    __shared__ float s_red[2][16];
    __shared__ int s_nan;
    const int c = blockIdx.x, b = blockIdx.y;
    const float *m = masked + ((size_t)b * C + c) * P * P;
    for (int e = threadIdx.x; e < PPAD * PPAD; e += blockDim.x) {
        const int i = e / PPAD, j = e - i * PPAD;
        s_m[e] = (i < P && j < P) ? m[i * P + j] : 0.f;
    }
    if (threadIdx.x == 0) s_nan = 0;
    float mn = INFINITY, mx = -INFINITY;
    bool has_nan = false;
    float *Tc = T + ((size_t)b * C + c) * H * PPAD;
    for (int y0 = 0; y0 < H; y0 += rows_chunk) {
        const int rows = min(rows_chunk, H - y0);
        __syncthreads();
        for (int e = threadIdx.x; e < rows * PPAD; e += blockDim.x) {   // T[y][j] = sum_i Ay[y][i] m[i][j]
            const int y = e / PPAD, j = e - y * PPAD;
            const float *a = Ay + (size_t)(y0 + y) * PPAD;
            float acc = 0.f;
            for (int i = 0; i < P; ++i) acc = fmaf(__ldg(a + i), s_m[i * PPAD + j], acc);
            s_T[e] = acc;
            Tc[(size_t)y0 * PPAD + e] = acc;
        }
        __syncthreads();
        for (int x = threadIdx.x; x < W; x += blockDim.x) {
            float ax[PPAD];
#pragma unroll
            for (int j = 0; j < PPAD; ++j) ax[j] = __ldg(AxT + (size_t)j * W + x);
            int y = 0;
            for (; y + 1 < rows; y += 2) {   // two independent FMA chains in flight
                const float v0 = lr_dot<PPAD>(s_T + y * PPAD, ax);
                const float v1 = lr_dot<PPAD>(s_T + (y + 1) * PPAD, ax);
                has_nan = has_nan || (v0 != v0) || (v1 != v1);
                mn = fminf(mn, fminf(v0, v1));
                mx = fmaxf(mx, fmaxf(v0, v1));
            }
            if (y < rows) {
                const float v = lr_dot<PPAD>(s_T + y * PPAD, ax);
                has_nan = has_nan || (v != v);
                mn = fminf(mn, v);
                mx = fmaxf(mx, v);
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (has_nan) s_nan = 1;
    if ((threadIdx.x & 31) == 0) { s_red[0][threadIdx.x >> 5] = mn; s_red[1][threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)((blockDim.x + 31) >> 5); ++w) { mn = fminf(mn, s_red[0][w]); mx = fmaxf(mx, s_red[1][w]); }
        if (s_nan) mn = mx = __int_as_float(0x7fc00000);
        const size_t k = (size_t)b * C + c;
        norm[2 * k + 0] = mn;
        norm[2 * k + 1] = __fdiv_rn(1.0f, __fsub_rn(mx, mn));   // 1/0 = inf: a constant map normalises to 0 * inf = NaN (0/0 in DRV:1152)
        if (minmax_out) {
            const size_t ko = (size_t)b * out_channels + out_channel_offset + c;
            minmax_out[2 * ko + 0] = mn;
            minmax_out[2 * ko + 1] = mx;
        }
    }
}

constexpr float kUnaryClipHi = 11.512925464970229f;  // -log(1e-5): np.clip(p, 1e-5, 1) seen from the log side

template <int PPAD>
__global__ void __launch_bounds__(128) lowrank_unary_kernel(const float *__restrict__ T, const float *__restrict__ AxT,
                                                            const float *__restrict__ norm, const float *__restrict__ bg_blur,
                                                            const float *__restrict__ bg_minmax, float *__restrict__ unary,
                                                            int32_t *__restrict__ labels, float *__restrict__ maps_out, int C, int H,
                                                            int W, int with_bg, int Cp, const int32_t *__restrict__ n_classes) {
    extern __shared__ __align__(16) float lr_smem[];
    const int TP = blockDim.x;
    // a batch padded to C classes: the channels image b does not have are dead -- value -inf (never the maximum, exp = 0 in the
    // softmax) and unary +inf (Q = 0 in every mean-field iteration, so they add exact zeros to every sum)
    const int Cb = n_classes ? n_classes[blockIdx.z] : C;
    const int Cc = C + with_bg;
    const int pitch = Cp + 1;                    // odd: thread-per-row accesses hit 32 different banks
    float *s_T = lr_smem;                        // [C][PPAD] row y of every channel's T
    float2 *s_norm = reinterpret_cast<float2 *>(s_T + (size_t)C * PPAD);   // [C] (min, 1/(max-min))
    float *s_tile = reinterpret_cast<float *>(s_norm + C);                 // [TP][Cp + 1]
    const int b = blockIdx.z, y = blockIdx.y, x0 = blockIdx.x * TP;
    const int x = x0 + threadIdx.x;
    const size_t N = (size_t)H * W;
    {   // T rows of all channels: C segments of PPAD contiguous floats, copied as float4
        const int q_per = PPAD / 4;
        for (int e = threadIdx.x; e < Cb * q_per; e += TP) {
            const int c = e / q_per, q = e - c * q_per;
            reinterpret_cast<float4 *>(s_T)[e] = __ldg(reinterpret_cast<const float4 *>(T + (((size_t)b * C + c) * H + y) * PPAD) + q);
        }
    }
    for (int e = threadIdx.x; e < Cb; e += TP) s_norm[e] = __ldg(reinterpret_cast<const float2 *>(norm) + (size_t)b * C + e);
    __syncthreads();
    float *row = s_tile + threadIdx.x * pitch;
    if (x < W) {
        float ax[PPAD];
#pragma unroll
        for (int j = 0; j < PPAD; ++j) ax[j] = __ldg(AxT + (size_t)j * W + x);
        float mxv = -INFINITY;
        if (with_bg) {
            const float mn = bg_minmax[2 * b], hi = bg_minmax[2 * b + 1];
            const float v = __fmul_rn(__fsub_rn(bg_blur[(size_t)b * N + (size_t)y * W + x], mn), __fdiv_rn(1.0f, __fsub_rn(hi, mn)));
            row[0] = v;
            mxv = fmaxf(mxv, v);
        }
        float *rc = row + with_bg;
        for (int c = Cb; c < C; ++c) rc[c] = -INFINITY;
#pragma unroll 2
        for (int c = 0; c < Cb; ++c) {
            const float yv = lr_dot<PPAD>(s_T + c * PPAD, ax);
            const float2 nm = s_norm[c];
            const float v = __fmul_rn(__fsub_rn(yv, nm.x), nm.y);   // (y - min) / (max - min), DRV:1151-1152
            rc[c] = v;
            mxv = fmaxf(mxv, v);
        }
        if (maps_out) {
            float *mo = maps_out + (size_t)b * Cc * N + (size_t)y * W + x;
            for (int c = 0; c < Cc; ++c) mo[(size_t)c * N] = row[c];
        }
        if (labels) {   // np.argmax / torch.argmax: first maximum, NaN counts as the maximum and the first NaN wins
            float best = row[0];
            int bi = 0;
            for (int c = 1; c < Cc; ++c) {
                const float v = row[c];
                if (!(best != best) && (v > best || v != v)) { best = v; bi = c; }
            }
            labels[(size_t)b * N + (size_t)y * W + x] = bi;
        }
        if (unary) {
            // U_c = -log(clip(softmax_c(v), 1e-5, 1)) = clamp(log(sum_k e^(v_k - max)) - (v_c - max), 0, -log 1e-5): one log per
            // pixel and no division instead of a division and a log per channel.  A NaN in any channel (fmaxf skips it) turns
            // the sum, hence every channel's unary, into NaN -- the softmax of a column holding a NaN.
            float sum = 0.f;
            for (int c = 0; c < Cc; ++c) sum += __expf(row[c] - mxv);
            const bool has_nan = sum != sum;
            const float shift = __logf(sum) + mxv;
            for (int c = 0; c < Cb + with_bg; ++c) {
                const float u = fminf(fmaxf(shift - row[c], 0.f), kUnaryClipHi);
                row[c] = has_nan ? __int_as_float(0x7fc00000) : u;
            }
            for (int c = Cb + with_bg; c < Cc; ++c) row[c] = INFINITY;
            for (int c = Cc; c < Cp; ++c) row[c] = n_classes ? INFINITY : 0.f;   // padded-batch mode: the CRF runs over all Cp channels
        }
    }
    if (!unary) return;
    __syncthreads();
    // coalesced copy-out of the [n_here][Cp] block; (pixel, channel) advance incrementally -- no division per element
    const int n_here = min(TP, W - x0);
    float *ub = unary + ((size_t)b * N + (size_t)y * W + x0) * Cp;
    const int step_p = TP / Cp, step_c = TP - step_p * Cp;
    int pp = threadIdx.x / Cp, c = threadIdx.x - pp * Cp;
    for (int i = threadIdx.x; i < n_here * Cp; i += TP) {
        ub[i] = s_tile[pp * pitch + c];
        pp += step_p;
        c += step_c;
        if (c >= Cp) { c -= Cp; ++pp; }
    }
}

static inline int blur_radius(double sigma) { return (int)(4.0 * sigma + 0.5); }  // scipy: int(truncate * sd + 0.5)
static inline int blur_padded_taps(int lw) { return (int)align_up((size_t)(2 * lw + 1), 8) + kTapPad; }

}  // namespace pnp

using namespace pnp;

extern "C" size_t pnp_threshold_upsample_workspace_bytes(int B, int C, int P) {
    if (B < 0 || C < 0 || P < 0) return 0;
    return align_up((size_t)B * C * P * P * sizeof(float), 256) + align_up((size_t)B * C * 2 * sizeof(float), 256);
}

extern "C" int pnp_threshold_upsample(const float *class_maps, float *out, void *workspace, size_t workspace_bytes, int B,
                                      int C, int P, int H, int W, float threshold, int rescale, int with_background,
                                      pnp_stream_t stream) {
    if (!class_maps || !out || !workspace || B < 0 || C < 1 || P < 1 || P * P > kMaxP2 || H < 1 || W < 1 || B > 65535)
        return PNP_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < pnp_threshold_upsample_workspace_bytes(B, C, P)) return PNP_ERR_WORKSPACE;
    if (B == 0) return PNP_OK;
    // Quirk kept: with ONE class F.interpolate(...).squeeze() is 2-D and Scale_0_1 returns 2-D input untouched
    // (DRV:1079-1080), so the rescale silently does not happen.
    if (C == 1) rescale = 0;
    cudaStream_t st = as_stream(stream);
    float *masked = reinterpret_cast<float *>(workspace);
    float *params = reinterpret_cast<float *>(reinterpret_cast<char *>(workspace) + align_up((size_t)B * C * P * P * sizeof(float), 256));
    PNP_LAUNCH(kThresholdPrep, st, threshold_prep_kernel<<<dim3(C, B), 256, 0, st>>>(class_maps, masked, params, C, P, H, W, threshold, rescale, nullptr));
    int rc = launch_status();
    if (rc != PNP_OK) return rc;
    const bool vec = (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    if (vec) {
        int gx = max(1, min(ceil_div((long long)H * (W / 4), 256), ceil_div(kNumSMs * 8, B)));
        PNP_LAUNCH(kUpsampleWrite, st, upsample_write_kernel<4><<<dim3(gx, B), 256, 0, st>>>(masked, params, out, C, P, H, W, rescale, with_background));
    } else {
        int gx = max(1, min(ceil_div((long long)H * W, 256), ceil_div(kNumSMs * 8, B)));
        PNP_LAUNCH(kUpsampleWrite, st, upsample_write_kernel<1><<<dim3(gx, B), 256, 0, st>>>(masked, params, out, C, P, H, W, rescale, with_background));
    }
    return launch_status();
}

namespace {
struct BlurPlan {
    int lw, n_w_padded, tile_rows, tile_cols, pitch, tile_rows_tma, h_groups;
    size_t smem_v, smem_h, smem_v_tma;
    size_t off_keys, off_tmp, total;
};
constexpr size_t kSmemBudget = 200 * 1024;

bool make_blur_plan(int n_maps, int H, int W, double sigma, BlurPlan &p) {
    if (!(sigma > 0.0) || n_maps < 0 || H < 1 || W < 1) return false;
    p.lw = blur_radius(sigma);
    if (p.lw > 4096) return false;
    p.n_w_padded = blur_padded_taps(p.lw);
    // pass V: whole column strip if it fits, else row tiles
    size_t fixed_rows = 2 * (size_t)p.lw + kTapPad + kVRows;
    size_t max_rows = (kSmemBudget - p.n_w_padded * sizeof(float)) / (kVCols * sizeof(float));
    if (max_rows <= fixed_rows + kVRows) return false;
    p.tile_rows = (int)std::min<size_t>((size_t)H, (max_rows - fixed_rows) / kVRows * kVRows);
    p.smem_v = (p.n_w_padded + (p.tile_rows + fixed_rows) * kVCols) * sizeof(float);
    // pass V, TMA variant: 32-column strips, <= 72 KB per CTA so that three CTAs share an SM
    {
        const size_t budget = 72 * 1024;
        size_t rows_max = (budget - p.n_w_padded * sizeof(float)) / (kTCols * sizeof(float));
        p.tile_rows_tma = rows_max > fixed_rows + kVRows ? (int)std::min<size_t>((size_t)H, (rows_max - fixed_rows) / kVRows * kVRows) : 0;
        p.smem_v_tma = (p.n_w_padded + (p.tile_rows_tma + fixed_rows) * kTCols) * sizeof(float);
    }
    // pass H: full rows if they fit, else column tiles
    // one warp per 16-column group so that a tile is one sweep (336 columns: 21 warps instead of 16 + 5 in two sweeps)
    const int groups_cap = kHGroupsMax;
    size_t out_floats = (size_t)kHRows * (groups_cap * kHCols + 1);  // worst case while the tile width is being chosen
    size_t max_pitch = (kSmemBudget - (p.n_w_padded + out_floats) * sizeof(float)) / (kHRows * sizeof(float));
    size_t fixed_cols = 2 * (size_t)p.lw + kTapPad + kHCols;
    if (max_pitch <= fixed_cols + kHCols + 1) return false;
    p.tile_cols = (int)std::min<size_t>((size_t)W, (max_pitch - 1 - fixed_cols) / kHCols * kHCols);
    p.pitch = (int)(p.tile_cols + fixed_cols) | 1;
    {   // warps per CTA: spread the tile's column groups evenly over the fewest sweeps
        const int n_col_groups = (p.tile_cols + kHCols - 1) / kHCols;
        const int sweeps = (n_col_groups + groups_cap - 1) / groups_cap;
        p.h_groups = (n_col_groups + sweeps - 1) / sweeps;
    }
    out_floats = (size_t)kHRows * (p.h_groups * kHCols + 1);
    p.smem_h = (p.n_w_padded + (size_t)kHRows * p.pitch + out_floats) * sizeof(float);
    p.off_keys = align_up(p.n_w_padded * sizeof(float), 256);
    p.off_tmp = p.off_keys + align_up((size_t)n_maps * 2 * sizeof(unsigned), 256);
    p.total = p.off_tmp + align_up((size_t)n_maps * H * W * sizeof(float), 256);
    return true;
}
}  // namespace

extern "C" size_t pnp_gaussian_blur_workspace_bytes(int n_maps, int H, int W, double sigma) {
    BlurPlan p;
    return make_blur_plan(n_maps, H, W, sigma, p) ? p.total : 0;
}

namespace {
// enqueue prologue (weights + key reset) + pass V + pass H + key decode (+ normalisation)
int blur_impl(const float *in, float *out, float *minmax, float *weights, unsigned *keys, float *tmp, const BlurPlan &p, int n_maps,
              int H, int W, double sigma, int normalize, cudaStream_t st) {
    cudaError_t e = allow_smem(blur_vertical_kernel, p.smem_v);
    if (e != cudaSuccess) return cuda_err(e);
    // up to 21 warps (tiles of <= 336 columns) two CTAs share an SM: cap the registers for that; wider tiles own the SM
    const bool h_pair = p.h_groups <= 21 && 2 * (p.smem_h + 1024) <= 227 * 1024;
    e = h_pair ? allow_smem(blur_horizontal_kernel<21, 2>, p.smem_h) : allow_smem(blur_horizontal_kernel<kHGroupsMax, 1>, p.smem_h);
    if (e != cudaSuccess) return cuda_err(e);
    blur_prologue_kernel<<<1, 256, 0, st>>>(weights, keys, n_maps, p.lw, p.n_w_padded, sigma);
    const bool tma_ok = p.tile_rows_tma > 0 && (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(in) & 15) == 0);
    if (tma_ok) {
        e = allow_smem(blur_vertical_tma_kernel, p.smem_v_tma);
        if (e != cudaSuccess) return cuda_err(e);
        PNP_LAUNCH(kBlurVertical, st, blur_vertical_tma_kernel<<<dim3(ceil_div(W, kTCols), ceil_div(H, p.tile_rows_tma), n_maps), kTCols * kTGroups, p.smem_v_tma, st>>>(
            in, tmp, weights, H, W, p.lw, p.tile_rows_tma, p.n_w_padded));
    } else {
        PNP_LAUNCH(kBlurVertical, st, blur_vertical_kernel<<<dim3(ceil_div(W, kVCols), ceil_div(H, p.tile_rows), n_maps), kVCols * kVGroups, p.smem_v, st>>>(
            in, tmp, weights, H, W, p.lw, p.tile_rows, p.n_w_padded));
    }
    const dim3 h_grid(ceil_div(W, p.tile_cols), ceil_div(H, kHRows), n_maps);
    if (h_pair)
        PNP_LAUNCH(kBlurHorizontal, st, (blur_horizontal_kernel<21, 2><<<h_grid, kHRows * p.h_groups, p.smem_h, st>>>(
            tmp, out, weights, keys, H, W, p.lw, p.tile_cols, p.pitch, p.n_w_padded)));
    else
        PNP_LAUNCH(kBlurHorizontal, st, (blur_horizontal_kernel<kHGroupsMax, 1><<<h_grid, kHRows * p.h_groups, p.smem_h, st>>>(
            tmp, out, weights, keys, H, W, p.lw, p.tile_cols, p.pitch, p.n_w_padded)));
    blur_minmax_decode_kernel<<<ceil_div(n_maps, 256), 256, 0, st>>>(keys, minmax, n_maps);
    if (normalize) {
        long long total = (long long)n_maps * H * W;
        int grid = (int)std::min<long long>((long long)kNumSMs * 16, (total + 255) / 256);
        PNP_LAUNCH(kBlurNormalize, st, blur_normalize_kernel<<<grid, 256, 0, st>>>(out, minmax, (long long)H * W, total));
    }
    return launch_status();
}
}  // namespace

extern "C" int pnp_gaussian_blur(const float *in, float *out, float *minmax, void *workspace, size_t workspace_bytes,
                                 int n_maps, int H, int W, double sigma, int normalize, pnp_stream_t stream) {
    BlurPlan p;
    if (!in || !out || !minmax || !workspace || in == out || !make_blur_plan(n_maps, H, W, sigma, p)) return PNP_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < p.total) return PNP_ERR_WORKSPACE;
    if (n_maps == 0) return PNP_OK;
    if (n_maps > 65535) return PNP_ERR_INVALID_ARGUMENT;
    char *ws = reinterpret_cast<char *>(workspace);
    return blur_impl(in, out, minmax, reinterpret_cast<float *>(ws), reinterpret_cast<unsigned *>(ws + p.off_keys),
                     reinterpret_cast<float *>(ws + p.off_tmp), p, n_maps, H, W, sigma, normalize, as_stream(stream));
}

// ------------------------------------------------------------------------------------------------ fused low-rank entry point
namespace {
struct LowrankPlan {
    BlurPlan blur;   // direct blur of the B background maps (planned only with_background)
    int lw, PPAD, rows_chunk, threads_a, tile_pix;
    size_t smem_a, smem_b;
    size_t off_masked, off_params, off_ay, off_axt, off_T, off_norm, off_bg, off_bgblur, off_bgmm, off_blur_ws, total;
};

bool make_lowrank_plan(int B, int C, int P, int H, int W, double sigma, int with_background, LowrankPlan &p) {
    if (B < 0 || C < 1 || P < 1 || P > kLrMaxP || H < 1 || W < 1 || !(sigma > 0.0)) return false;
    // only the background maps take the direct blur: without them its size limits do not apply
    p.blur = BlurPlan{};
    if (with_background && !make_blur_plan(B, H, W, sigma, p.blur)) return false;
    // lowrank_operator_kernel keeps the 2 lw + 1 float64 weights in dynamic shared memory, next to its 1 KB s_part, within the
    // 48 KB a CTA gets without opting in: lw <= 3007
    if (!(4.0 * sigma + 0.5 < (48 * 1024 - 128 * sizeof(double)) / (2 * sizeof(double)))) return false;
    p.lw = blur_radius(sigma);
    p.PPAD = P <= 24 ? 24 : (P <= 28 ? 28 : 32);
    p.rows_chunk = std::min(H, 512);   // <= 64 KB of T per chunk
    {   // pass A: one thread per column, as few sweeps over x as possible
        const int sweeps = (W + 511) / 512;
        p.threads_a = std::min(512, std::max(64, (int)align_up((size_t)((W + sweeps - 1) / sweeps), 32)));
    }
    p.smem_a = ((size_t)p.PPAD * p.PPAD + (size_t)p.rows_chunk * p.PPAD) * sizeof(float);
    const int Cp = (C + (with_background ? 1 : 0) + 3) / 4 * 4;
    p.tile_pix = Cp <= 64 ? 128 : 64;
    p.smem_b = ((size_t)C * p.PPAD + 2 * (size_t)C + (size_t)p.tile_pix * (Cp + 1)) * sizeof(float);  // s_T, s_norm (float2), s_tile
    if (p.smem_b > 200 * 1024) {
        p.tile_pix = 32;
        p.smem_b = ((size_t)C * p.PPAD + 2 * (size_t)C + (size_t)p.tile_pix * (Cp + 1)) * sizeof(float);  // s_T, s_norm (float2), s_tile
        if (p.smem_b > 200 * 1024) return false;
    }
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return o; };
    p.off_masked = take((size_t)B * C * P * P * sizeof(float));
    p.off_params = take((size_t)B * C * 2 * sizeof(float));
    p.off_ay = take((size_t)H * p.PPAD * sizeof(float));
    p.off_axt = take((size_t)W * p.PPAD * sizeof(float));
    p.off_T = take((size_t)B * C * H * p.PPAD * sizeof(float));
    p.off_norm = take((size_t)B * C * 2 * sizeof(float));
    p.off_bg = take(with_background ? (size_t)B * H * W * sizeof(float) : 0);
    p.off_bgblur = take(with_background ? (size_t)B * H * W * sizeof(float) : 0);
    p.off_bgmm = take(with_background ? (size_t)B * 2 * sizeof(float) : 0);
    p.off_blur_ws = take(with_background ? p.blur.total : 0);
    p.total = off;
    return true;
}

template <int PPAD>
int launch_lowrank(const LowrankPlan &p, char *ws, float *unary, int32_t *labels, float *maps_out, float *minmax_out, int B, int C,
                   int P, int H, int W, int with_background, const int32_t *n_classes, cudaStream_t st) {
    const float *masked = reinterpret_cast<const float *>(ws + p.off_masked);
    const float *Ay = reinterpret_cast<const float *>(ws + p.off_ay), *AxT = reinterpret_cast<const float *>(ws + p.off_axt);
    float *T = reinterpret_cast<float *>(ws + p.off_T), *norm = reinterpret_cast<float *>(ws + p.off_norm);
    const int Cc = C + (with_background ? 1 : 0), Cp = (Cc + 3) / 4 * 4;
    cudaError_t e = allow_smem(lowrank_minmax_kernel<PPAD>, p.smem_a);
    if (e != cudaSuccess) return cuda_err(e);
    e = allow_smem(lowrank_unary_kernel<PPAD>, p.smem_b);
    if (e != cudaSuccess) return cuda_err(e);
    PNP_LAUNCH(kLowrankBlur, st, (lowrank_minmax_kernel<PPAD><<<dim3(C, B), p.threads_a, p.smem_a, st>>>(
        masked, Ay, AxT, T, norm, minmax_out, C, P, H, W, p.rows_chunk, with_background ? 1 : 0, Cc, n_classes)));
    PNP_LAUNCH(kLowrankUnary, st, (lowrank_unary_kernel<PPAD><<<dim3(ceil_div(W, p.tile_pix), H, B), p.tile_pix, p.smem_b, st>>>(
        T, AxT, norm, with_background ? reinterpret_cast<const float *>(ws + p.off_bgblur) : nullptr,
        with_background ? reinterpret_cast<const float *>(ws + p.off_bgmm) : nullptr, unary, labels, maps_out, C, H, W,
        with_background ? 1 : 0, Cp, n_classes)));
    return launch_status();
}
}  // namespace

extern "C" size_t pnp_lowrank_blur_workspace_bytes(int B, int C, int P, int H, int W, double sigma, int with_background) {
    LowrankPlan p;
    return make_lowrank_plan(B, C, P, H, W, sigma, with_background, p) ? p.total : 0;
}

extern "C" int pnp_lowrank_blur_unary(const float *class_maps, float *unary, int32_t *labels, float *maps_out, float *minmax_out,
                                      void *workspace, size_t workspace_bytes, int B, int C, int P, int H, int W, float threshold,
                                      int rescale, int with_background, double sigma, pnp_stream_t stream) {
    return pnp_lowrank_blur_unary_padded(class_maps, nullptr, unary, labels, maps_out, minmax_out, workspace, workspace_bytes, B, C, P, H, W,
                                         threshold, rescale, with_background, sigma, stream);
}

extern "C" int pnp_lowrank_blur_unary_padded(const float *class_maps, const int32_t *n_classes, float *unary, int32_t *labels,
                                             float *maps_out, float *minmax_out, void *workspace, size_t workspace_bytes, int B, int C,
                                             int P, int H, int W, float threshold, int rescale, int with_background, double sigma,
                                             pnp_stream_t stream) {
    LowrankPlan p;
    if (!class_maps || !workspace || (!unary && !labels && !maps_out) || B > 65535 || H > 65535 ||
        !make_lowrank_plan(B, C, P, H, W, sigma, with_background, p))
        return PNP_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < p.total) return PNP_ERR_WORKSPACE;
    if (B == 0) return PNP_OK;
    cudaStream_t st = as_stream(stream);
    char *ws = reinterpret_cast<char *>(workspace);
    float *masked = reinterpret_cast<float *>(ws + p.off_masked), *params = reinterpret_cast<float *>(ws + p.off_params);
    // Scale_0_1 only matters for the background test (it cancels in every class channel, see above); with ONE class the
    // reference's rescale silently does not happen (DRV:1079-1080), as in pnp_threshold_upsample
    const int bg_rescale = (rescale && with_background && (n_classes || C > 1)) ? 1 : 0;   // per image in the kernels when n_classes is given
    char *bws = ws + p.off_blur_ws;
    lowrank_operator_kernel<<<ceil_div(H + W, 128), 128, (2 * p.lw + 1) * sizeof(double), st>>>(
        reinterpret_cast<float *>(ws + p.off_ay), reinterpret_cast<float *>(ws + p.off_axt), H, W, P, p.PPAD, p.lw, sigma);
    PNP_LAUNCH(kThresholdPrep, st, threshold_prep_kernel<<<dim3(C, B), 256, 0, st>>>(class_maps, masked, params, C, P, H, W, threshold, bg_rescale, n_classes));
    int rc = launch_status();
    if (rc != PNP_OK) return rc;
    if (with_background) {
        float *bg = reinterpret_cast<float *>(ws + p.off_bg);
        const bool vec = (W % 4 == 0);
        const int per = vec ? H * (W / 4) : H * W;
        const int gx = std::max(1, std::min(ceil_div(per, 256), ceil_div(kNumSMs * 8, B)));
        if (vec)
            PNP_LAUNCH(kUpsampleWrite, st, (upsample_write_kernel<4, true><<<dim3(gx, B), 256, 0, st>>>(masked, params, bg, C, P, H, W, bg_rescale, 1, n_classes)));
        else
            PNP_LAUNCH(kUpsampleWrite, st, (upsample_write_kernel<1, true><<<dim3(gx, B), 256, 0, st>>>(masked, params, bg, C, P, H, W, bg_rescale, 1, n_classes)));
        const bool timed = prof::on(kBackgroundBlur, st);
        if (timed) prof::begin(kBackgroundBlur, st);
        rc = blur_impl(bg, reinterpret_cast<float *>(ws + p.off_bgblur), reinterpret_cast<float *>(ws + p.off_bgmm),
                       reinterpret_cast<float *>(bws), reinterpret_cast<unsigned *>(bws + p.blur.off_keys),
                       reinterpret_cast<float *>(bws + p.blur.off_tmp), p.blur, B, H, W, sigma, 0, st);
        if (timed) prof::end(kBackgroundBlur, st);
        if (rc != PNP_OK) return rc;
        if (minmax_out) {   // channel 0 of each image = the background map's (min, max)
            const int Cc = C + 1;
            cudaError_t e = cudaMemcpy2DAsync(minmax_out, (size_t)Cc * 2 * sizeof(float), ws + p.off_bgmm, 2 * sizeof(float),
                                              2 * sizeof(float), B, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) return cuda_err(e);
        }
    }
    switch (p.PPAD) {
        case 24: return launch_lowrank<24>(p, ws, unary, labels, maps_out, minmax_out, B, C, P, H, W, with_background, n_classes, st);
        case 28: return launch_lowrank<28>(p, ws, unary, labels, maps_out, minmax_out, B, C, P, H, W, with_background, n_classes, st);
        default: return launch_lowrank<32>(p, ws, unary, labels, maps_out, minmax_out, B, C, P, H, W, with_background, n_classes, st);
    }
}
