// crf.cu -- (e) part 2: filtering on the permutohedral lattice and dense-CRF mean-field inference.
// Replaces pydensecrf's DenseCRF2D.inference (DRV:1071) and unary_from_softmax (DRV:1057-1063).
//
// Data layout: per-pixel / per-vertex channel vectors are contiguous ([B,N,Cp], [rows,Cp], Cp = 4*ceil(C/4)), so
// every gather moves whole rows with 128-bit accesses; one thread owns one float4 chunk of one row.
//   splat   gather over the vertex's CSR row (pixels in ascending order): values[v] = sum w * (norm * Q[pix])
//   blur    values'[v] = values[v] + 0.5 (values[n1] + values[n2]) along each of the d+1 axes (ping-pong), two axes
//           per launch (the first recomputed at the two neighbours) so the intermediate lattice stays out of HBM
//   update  per pixel: slice every kernel's lattice, add the weighted messages to -U, softmax over channels,
//           write Q (and, on the last iteration, the argmax label) -- one pass over Q/U per iteration.
// splat / blur / slice of pnp_crf_filter are written with explicit __fmul_rn/__fadd_rn in the reference's order (it is
// compiled without FMA contraction), so the filter is bit-identical to the sequential CPU restatement.  The mean-field
// update of the standard [Gaussian, bilateral] pair folds alpha, norm and the kernel weight into the barycentric weights
// and uses FMA / __expf (its inputs already carry expf ulps); the marginals stay within 1e-3 of the restatement (tests).
#include <math.h>

#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "lattice.cuh"

namespace pnp {

__device__ __forceinline__ float4 f4_mul(float4 a, float s) {
    return make_float4(__fmul_rn(a.x, s), __fmul_rn(a.y, s), __fmul_rn(a.z, s), __fmul_rn(a.w, s));
}
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) {
    return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
}

__device__ __forceinline__ float4 ld_gather4(const float *p) {  // ordered (volatile) 128-bit gather through L1
    float4 r;
    asm volatile("ld.global.ca.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
// rows of a value buffer that one image (shared lattice) or the whole batch (batched lattice) occupies
__host__ __device__ __forceinline__ long long value_rows(const LatticeView &L, int B) {
    return L.shared ? (long long)B * (L.M + 1) : (long long)L.M + 1;
}

// ------------------------------------------------------------------------------------------ splat
// grid.y = image for shared lattices (1 otherwise).  One thread owns one float4 chunk of one vertex row and walks the
// vertex's CSR entries (pixels in ascending order) four at a time (four row gathers in flight), adding them in entry
// order with separately rounded mul/add (bit-identical to the sequential reference).  ncu: the kernel is bound by L1
// wavefronts of the row gathers, so staging through shared memory (cp.async) only adds to that pipe.
constexpr int kSplatBatch = 4;

__global__ void __launch_bounds__(256) splat_kernel(LatticeView L, const float *__restrict__ x, float *__restrict__ values, int Cp,
                                                    int normalized) {
    const int nch = Cp >> 2;
    const int b = blockIdx.y;
    const float *xb = L.shared ? x + (size_t)b * L.N * Cp : x;
    float *vb = L.shared ? values + (size_t)b * (L.M + 1) * L.vp : values;
    const long long total = (long long)(L.M + 1) * nch;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int v = (int)(idx / nch), ch = (int)(idx - (long long)v * nch);
        if (v == L.M) {  // sentinel row 0 stays zero
            *reinterpret_cast<float4 *>(vb + 4 * ch) = make_float4(0.f, 0.f, 0.f, 0.f);
            continue;
        }
        // vertices are visited in first-touch order: neighbours in memory are neighbours in the image, which keeps the
        // row gathers in L1/L2 (sorting vertices by row length to balance warps cost 2x the DRAM traffic: profiles/)
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        const int end = __ldg(L.row_ptr + v + 1);
        int k = __ldg(L.row_ptr + v);
        for (; k + kSplatBatch <= end; k += kSplatBatch) {  // kSplatBatch gathers in flight, accumulated in entry order
            int lp[kSplatBatch];
            float w[kSplatBatch], nr[kSplatBatch];
            float4 xv[kSplatBatch];
#pragma unroll
            for (int i = 0; i < kSplatBatch; ++i) {
                lp[i] = __ldg(L.csr_pix + k + i);
                w[i] = __ldg(L.csr_w + k + i);
                nr[i] = normalized ? __ldg(L.csr_norm + k + i) : 1.f;
            }
#pragma unroll
            for (int i = 0; i < kSplatBatch; ++i) xv[i] = *reinterpret_cast<const float4 *>(xb + (size_t)lp[i] * Cp + 4 * ch);
#pragma unroll
            for (int i = 0; i < kSplatBatch; ++i) {
                if (normalized) xv[i] = f4_mul(xv[i], nr[i]);
                acc = f4_add(acc, f4_mul(xv[i], w[i]));
            }
        }
        for (; k < end; ++k) {
            const int lp = __ldg(L.csr_pix + k);
            float4 xv = *reinterpret_cast<const float4 *>(xb + (size_t)lp * Cp + 4 * ch);
            if (normalized) xv = f4_mul(xv, __ldg(L.csr_norm + k));
            acc = f4_add(acc, f4_mul(xv, __ldg(L.csr_w + k)));
        }
        *reinterpret_cast<float4 *>(vb + (size_t)(v + 1) * L.vp + 4 * ch) = acc;
    }
}

// ------------------------------------------------------------------------------------------ blur along one axis
__global__ void __launch_bounds__(256) blur_axis_kernel(LatticeView L, const float *__restrict__ old_v, float *__restrict__ new_v, int axis,
                                                        int Cp) {
    const int nch = Cp >> 2;
    const int b = blockIdx.y;
    const long long img_off = L.shared ? (long long)b * (L.M + 1) * L.vp : 0;
    const float *ob = old_v + img_off;
    float *nb = new_v + img_off;
    const int2 *nbr = reinterpret_cast<const int2 *>(L.nbr) + (size_t)axis * L.vertex_stride;
    const long long total = (long long)(L.M + 1) * nch;
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (idx >= total) return;
    // software pipeline over the grid-stride loop: the neighbour indices of the NEXT item are fetched while the rows
    // of the current one are in flight (ncu: the kernel otherwise stalls on the index -> address -> row chain)
    int v = (int)(idx / nch), ch = (int)(idx - (long long)v * nch);
    int2 n = (v < L.M) ? nbr[v] : make_int2(0, 0);
    while (true) {
        const long long idx_next = idx + stride;
        const bool more = idx_next < total;
        int v_next = 0, ch_next = 0;
        int2 n_next = make_int2(0, 0);
        if (more) {
            v_next = (int)(idx_next / nch);
            ch_next = (int)(idx_next - (long long)v_next * nch);
            if (v_next < L.M) n_next = nbr[v_next];
        }
        if (v == L.M) {
            *reinterpret_cast<float4 *>(nb + 4 * ch) = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            const float4 c = *reinterpret_cast<const float4 *>(ob + (long long)(v + 1) * L.vp + 4 * ch);
            const float4 a1 = *reinterpret_cast<const float4 *>(ob + (long long)n.x * L.vp + 4 * ch);
            const float4 a2 = *reinterpret_cast<const float4 *>(ob + (long long)n.y * L.vp + 4 * ch);
            // new = old + 0.5f * (n1 + n2)   (plain cached accesses: streaming hints measured 4 % slower, profiles/README.md)
            *reinterpret_cast<float4 *>(nb + (long long)(v + 1) * L.vp + 4 * ch) = f4_add(c, f4_mul(f4_add(a1, a2), 0.5f));
        }
        if (!more) break;
        idx = idx_next; v = v_next; ch = ch_next; n = n_next;
    }
}

// Two consecutive axis passes in one launch (temporal fusion through the 126 MB L2): new = B_b(B_a(old)).  The first
// pass is recomputed on the fly at the vertex and at its two axis-b neighbours (9 row gathers instead of 3 + 3), so the
// intermediate lattice is never written to or read back from HBM: DRAM traffic per pair of axes drops from
// 2 x (read + write) to one read + one write.  Every B_a value is computed with the same operations in the same order as
// the single-axis kernel, so the result is bit-identical to two separate passes.
__device__ __forceinline__ float4 blur_row(const float *__restrict__ ob, int row, int2 n, int vp, int ch) {
    const float4 c = *reinterpret_cast<const float4 *>(ob + (size_t)row * vp + 4 * ch);
    const float4 a1 = *reinterpret_cast<const float4 *>(ob + (size_t)n.x * vp + 4 * ch);
    const float4 a2 = *reinterpret_cast<const float4 *>(ob + (size_t)n.y * vp + 4 * ch);
    return f4_add(c, f4_mul(f4_add(a1, a2), 0.5f));
}

__global__ void __launch_bounds__(256) blur_axis2_kernel(LatticeView L, const float *__restrict__ old_v, float *__restrict__ new_v,
                                                         int axis_a, int axis_b, int Cp) {
    const int nch = Cp >> 2;
    const int b = blockIdx.y;
    const long long img_off = L.shared ? (long long)b * (L.M + 1) * L.vp : 0;
    const float *ob = old_v + img_off;
    float *nb = new_v + img_off;
    const int2 *nbr_a = reinterpret_cast<const int2 *>(L.nbr) + (size_t)axis_a * L.vertex_stride;
    const int2 *nbr_b = reinterpret_cast<const int2 *>(L.nbr) + (size_t)axis_b * L.vertex_stride;
    const long long total = (long long)(L.M + 1) * nch;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int v = (int)(idx / nch), ch = (int)(idx - (long long)v * nch);
        if (v == L.M) {
            *reinterpret_cast<float4 *>(nb + 4 * ch) = make_float4(0.f, 0.f, 0.f, 0.f);
            continue;
        }
        const int2 nb2 = nbr_b[v];  // axis-b neighbours of v (+1 shifted, 0 = none)
        const int2 na_v = nbr_a[v];
        const int2 na_1 = nb2.x ? nbr_a[nb2.x - 1] : make_int2(0, 0);
        const int2 na_2 = nb2.y ? nbr_a[nb2.y - 1] : make_int2(0, 0);
        const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 t_v = blur_row(ob, v + 1, na_v, L.vp, ch);
        const float4 t_1 = nb2.x ? blur_row(ob, nb2.x, na_1, L.vp, ch) : zero;  // the sentinel row stays zero after pass a
        const float4 t_2 = nb2.y ? blur_row(ob, nb2.y, na_2, L.vp, ch) : zero;
        *reinterpret_cast<float4 *>(nb + (size_t)(v + 1) * L.vp + 4 * ch) = f4_add(t_v, f4_mul(f4_add(t_1, t_2), 0.5f));
    }
}

// slice one lattice at (pixel gp of image b, chunk ch): sum_j (w_j * values[o_j]) * alpha, optionally * norm.
// DP1 = d+1 is a template parameter so the d+1 gathers are all in flight before the (ordered) accumulation.
template <int DP1>
__device__ __forceinline__ float4 slice_pixel_t(const LatticeView &L, const float *__restrict__ values, int b, int pix, int gp, int ch,
                                                int Cp, bool normalized) {
    const int lp = L.shared ? pix : gp;
    const float *vb = L.shared ? values + (size_t)b * (L.M + 1) * L.vp : values;
    int o[DP1];
    float w[DP1];
    float4 v[DP1];
#pragma unroll
    for (int j = 0; j < DP1; ++j) {
        o[j] = __ldg(L.offset + (size_t)lp * DP1 + j) + 1;
        w[j] = __ldg(L.bary + (size_t)lp * DP1 + j);
    }
#pragma unroll
    for (int j = 0; j < DP1; ++j) v[j] = *reinterpret_cast<const float4 *>(vb + (size_t)o[j] * L.vp + 4 * ch);
    float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < DP1; ++j) out = f4_add(out, f4_mul(f4_mul(v[j], w[j]), L.alpha));
    if (normalized) out = f4_mul(out, __ldg(L.norm + lp));
    return out;
}

__device__ __forceinline__ float4 slice_pixel(const LatticeView &L, const float *__restrict__ values, int b, int pix, long long gp,
                                              int ch, int Cp, bool normalized) {
    if (L.Dp1 == 3) return slice_pixel_t<3>(L, values, b, pix, (int)gp, ch, Cp, normalized);
    return slice_pixel_t<6>(L, values, b, pix, (int)gp, ch, Cp, normalized);
}

__global__ void __launch_bounds__(256) slice_kernel(LatticeView L, const float *__restrict__ values, float *__restrict__ y, int B, int Cp,
                                                    int normalized) {
    const int nch = Cp >> 2;
    const long long total = (long long)B * L.N * nch;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long gp = idx / nch;
        const int ch = (int)(idx - gp * nch);
        const int b = (int)(gp / L.N), pix = (int)(gp - (long long)b * L.N);
        *reinterpret_cast<float4 *>(y + gp * Cp + 4 * ch) = slice_pixel(L, values, b, pix, gp, ch, Cp, normalized != 0);
    }
}

// ------------------------------------------------------------------------------------------ mean-field update
constexpr int kMaxKernels = 4;
struct MeanFieldParams {
    LatticeView lat[kMaxKernels];
    const float *values[kMaxKernels];
    float weight[kMaxKernels];
    int n_kernels;
};

__device__ __forceinline__ void argmax_first(float v, int c, float &best, int &bi) {
    if (!(best != best) && (v > best || v != v)) { best = v; bi = c; }
}

// Q = softmax_c(-U + sum_k w_k * norm_k . slice_k(values_k)); 256 threads = TP pixels x nch chunks
template <bool kLabels>
__global__ void __launch_bounds__(256) meanfield_update_kernel(MeanFieldParams P, const float *__restrict__ unary, float *__restrict__ Q,
                                                               int32_t *__restrict__ labels, int B, int N, int C, int Cp) {
    __shared__ float s_a[256];
    __shared__ float s_b[256];
    __shared__ int s_i[256];
    const int nch = Cp >> 2;
    const int TP = 256 / nch;
    const int pl = threadIdx.x / nch, ch = threadIdx.x - pl * nch;
    const long long n_pix = (long long)B * N;
    const long long n_tiles = (n_pix + TP - 1) / TP;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long gp = tile * TP + pl;
        const bool active = pl < TP && gp < n_pix;
        float t[4] = {0.f, 0.f, 0.f, 0.f};
        float mx = -INFINITY;
        if (active) {
            const int b = (int)(gp / N), pix = (int)(gp - (long long)b * N);
            const float4 u = *reinterpret_cast<const float4 *>(unary + gp * Cp + 4 * ch);
            float4 acc = make_float4(-u.x, -u.y, -u.z, -u.w);
            for (int k = 0; k < P.n_kernels; ++k) {
                float4 s = slice_pixel(P.lat[k], P.values[k], b, pix, gp, ch, Cp, true);
                acc = f4_add(acc, f4_mul(s, P.weight[k]));  // tmp1 -= (-w * K Q)
            }
            t[0] = acc.x; t[1] = acc.y; t[2] = acc.z; t[3] = acc.w;
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (4 * ch + i < C) mx = fmaxf(mx, t[i]);
        }
        s_a[threadIdx.x] = mx;
        __syncthreads();
        float e[4] = {0.f, 0.f, 0.f, 0.f};
        float part = 0.f;
        if (active) {
            float m = s_a[pl * nch];
            for (int k = 1; k < nch; ++k) m = fmaxf(m, s_a[pl * nch + k]);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (4 * ch + i < C) {
                    e[i] = expf(t[i] - m);
                    part += e[i];
                }
            }
        }
        s_b[threadIdx.x] = part;
        __syncthreads();
        float q[4] = {0.f, 0.f, 0.f, 0.f};
        if (active) {
            float sum = 0.f;
            for (int k = 0; k < nch; ++k) sum += s_b[pl * nch + k];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (4 * ch + i < C) q[i] = __fdiv_rn(e[i], sum);
            *reinterpret_cast<float4 *>(Q + gp * Cp + 4 * ch) = make_float4(q[0], q[1], q[2], q[3]);
        }
        if (kLabels) {
            __syncthreads();  // s_a is reused
            float best = q[0];
            int bi = 4 * ch;
#pragma unroll
            for (int i = 1; i < 4; ++i)
                if (4 * ch + i < C) argmax_first(q[i], 4 * ch + i, best, bi);
            s_a[threadIdx.x] = best;
            s_i[threadIdx.x] = bi;
            __syncthreads();
            if (active && ch == 0) {
                for (int k = 1; k < nch; ++k) argmax_first(s_a[pl * nch + k], s_i[pl * nch + k], best, bi);
                labels[gp] = bi;
            }
        }
        __syncthreads();
    }
}


// Warp-level variant for Cp <= 128 (nch <= 32 chunks): the nch lanes of a pixel sit in one warp, so the softmax
// reductions are shuffles -- no shared memory, no block barrier, warps never wait for each other's gathers.
// A CTA owns whole 16x16 pixel tiles, so the lattice rows its pixels share stay in L1 between its sub-iterations.
constexpr int kTile = 16;

// index-aware argmax merge for out-of-order traversal: larger value wins, equal values -> smaller channel index wins,
// NaN beats every number and the NaN with the smallest index wins (numpy/torch "first maximum, NaN counts as maximum")
__device__ __forceinline__ void argmax_merge(float v, int c, float &best, int &bi) {
    const bool vnan = v != v, bnan = best != best;
    const bool take = bnan ? (vnan && c < bi) : (vnan || v > best || (v == best && c < bi));
    if (take) { best = v; bi = c; }
}

// A pixel's nch float4 chunks are spread over LPP lanes, CPL chunks per lane (chunk = lane_in_pixel + k*LPP), PW = 32/LPP
// pixels per warp.  The host picks (LPP, CPL) to waste the fewest lanes and, among equals, the most chunks per lane (fewer
// shuffle rounds, more pixels per warp): 21 channels (nch 6) -> 1 lane x 6 chunks, 32 pixels per warp; 81 channels (nch 21)
// -> 4 lanes x 6 chunks, 8 pixels (32.3 ms per pass against 36.9 for 7 x 3); 150 channels (nch 38) -> 10 lanes x 4 chunks.
template <bool kLabels, bool kFast, int CPL>
__device__ __forceinline__ void meanfield_update_warp_body(const MeanFieldParams &P, const float *__restrict__ unary,
                                                           float *__restrict__ Q, int32_t *__restrict__ labels, int B, int H, int W,
                                                           int C, int Cp, int LPP) {
    const int nch = Cp >> 2;
    const int PW = 32 / LPP;                       // pixels per warp
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int pl = lane / LPP, li = lane - pl * LPP;
    const int base_lane = pl * LPP;
    const bool lane_used = pl < PW;
    const int N = H * W;
    const int tiles_x = (W + kTile - 1) / kTile, tiles_y = (H + kTile - 1) / kTile;
    const int tiles_per_image = tiles_x * tiles_y;
    const int n_tiles = B * tiles_per_image;
    const int pix_per_iter = (blockDim.x >> 5) * PW;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int b = tile / tiles_per_image;
        const int t = tile - b * tiles_per_image;
        const int ty = t / tiles_x, tx = t - ty * tiles_x;
        for (int sub = 0; sub < kTile * kTile; sub += pix_per_iter) {
            const int within = sub + warp * PW + pl;
            const int y = ty * kTile + within / kTile, x = tx * kTile + (within % kTile);
            const bool active = lane_used && within < kTile * kTile && y < H && x < W;
            const int pix = y * W + x;
            const int gp = b * N + pix;
            float t4[CPL][4];
            float mx = -INFINITY;
            if (kFast) {
                // [spatial d=2 shared, bilateral d=5 batched].  Loads are unconditional (idle lanes read pixel 0 / chunk 0);
                // alpha, norm and the kernel weight are folded into the barycentric weights (the exactly-ordered variant
                // lives in slice_pixel_t / pnp_crf_filter).  Offsets and weights are loaded once per pixel and reused
                // by the lane's CPL chunks.
                const int spix = active ? pix : 0, sgp = active ? gp : 0, sb = active ? b : 0;
                const LatticeView &A = P.lat[0];
                const LatticeView &Bl = P.lat[1];
                int oa[3], ob[6];
                float wa[3], wb[6];
#pragma unroll
                for (int j = 0; j < 3; ++j) { oa[j] = __ldg(A.offset + (size_t)spix * 3 + j) + 1; wa[j] = __ldg(A.bary + (size_t)spix * 3 + j); }
#pragma unroll
                for (int j = 0; j < 3; ++j) {  // 6 ints / 6 floats per pixel, 8-byte aligned
                    const int2 o2 = __ldg(reinterpret_cast<const int2 *>(Bl.offset + (size_t)sgp * 6) + j);
                    const float2 w2 = __ldg(reinterpret_cast<const float2 *>(Bl.bary + (size_t)sgp * 6) + j);
                    ob[2 * j] = o2.x + 1; ob[2 * j + 1] = o2.y + 1;
                    wb[2 * j] = w2.x; wb[2 * j + 1] = w2.y;
                }
                const float ca = A.alpha * __ldg(A.norm + spix) * P.weight[0];
                const float cb = Bl.alpha * __ldg(Bl.norm + sgp) * P.weight[1];
#pragma unroll
                for (int j = 0; j < 3; ++j) wa[j] *= ca;
#pragma unroll
                for (int j = 0; j < 6; ++j) wb[j] *= cb;
                const float *va0 = P.values[0] + (size_t)sb * (A.M + 1) * A.vp;
                const float *vb0 = P.values[1];
#pragma unroll
                for (int k = 0; k < CPL; ++k) {
                    const int ch = li + k * LPP;
                    const int sch = (lane_used && ch < nch) ? ch : 0;
                    const float4 u = ldg_stream4(unary + (size_t)sgp * Cp + 4 * sch);
                    // The 9 row gathers are volatile (ordered) loads and the accumulation chain STARTS with the gather
                    // issued last, so all nine are in flight before the first FFMA can retire (ptxas otherwise
                    // interleaves load/FFMA pairs to save registers and serialises the L2 latencies).
                    float4 ga[3], gb[6];
#pragma unroll
                    for (int j = 0; j < 3; ++j) ga[j] = ld_gather4(va0 + (size_t)oa[j] * A.vp + 4 * sch);
#pragma unroll
                    for (int j = 0; j < 6; ++j) gb[j] = ld_gather4(vb0 + (size_t)ob[j] * Bl.vp + 4 * sch);
                    float4 acc = make_float4(-u.x, -u.y, -u.z, -u.w);
#pragma unroll
                    for (int j = 5; j >= 0; --j) {
                        acc.x = fmaf(gb[j].x, wb[j], acc.x); acc.y = fmaf(gb[j].y, wb[j], acc.y);
                        acc.z = fmaf(gb[j].z, wb[j], acc.z); acc.w = fmaf(gb[j].w, wb[j], acc.w);
                    }
#pragma unroll
                    for (int j = 2; j >= 0; --j) {
                        acc.x = fmaf(ga[j].x, wa[j], acc.x); acc.y = fmaf(ga[j].y, wa[j], acc.y);
                        acc.z = fmaf(ga[j].z, wa[j], acc.z); acc.w = fmaf(ga[j].w, wa[j], acc.w);
                    }
                    t4[k][0] = acc.x; t4[k][1] = acc.y; t4[k][2] = acc.z; t4[k][3] = acc.w;
                    if (active && ch < nch) {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            if (4 * ch + i < C) mx = fmaxf(mx, t4[k][i]);
                    }
                }
            } else {
#pragma unroll
                for (int k = 0; k < CPL; ++k) {
                    const int ch = li + k * LPP;
                    t4[k][0] = t4[k][1] = t4[k][2] = t4[k][3] = 0.f;
                    if (active && ch < nch) {
                        const float4 u = ldg_stream4(unary + (size_t)gp * Cp + 4 * ch);
                        float4 acc = make_float4(-u.x, -u.y, -u.z, -u.w);
                        for (int kk = 0; kk < P.n_kernels; ++kk) {
                            float4 s = slice_pixel(P.lat[kk], P.values[kk], b, pix, gp, ch, Cp, true);
                            acc = f4_add(acc, f4_mul(s, P.weight[kk]));  // tmp1 -= (-w * K Q)
                        }
                        t4[k][0] = acc.x; t4[k][1] = acc.y; t4[k][2] = acc.z; t4[k][3] = acc.w;
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            if (4 * ch + i < C) mx = fmaxf(mx, t4[k][i]);
                    }
                }
            }
            float m = -INFINITY;
            for (int k = 0; k < LPP; ++k) m = fmaxf(m, __shfl_sync(0xffffffffu, mx, base_lane + k));
            float e[CPL][4];
            float part = 0.f;
#pragma unroll
            for (int k = 0; k < CPL; ++k) {
                const int ch = li + k * LPP;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    e[k][i] = 0.f;
                    if (active && ch < nch && 4 * ch + i < C) {
                        e[k][i] = kFast ? __expf(t4[k][i] - m) : expf(t4[k][i] - m);
                        part += e[k][i];
                    }
                }
            }
            float sum = 0.f;
            for (int k = 0; k < LPP; ++k) sum += __shfl_sync(0xffffffffu, part, base_lane + k);
            const float rs = __frcp_rn(sum);
            float best = 0.f;
            int bi = 0x7fffffff;
            bool have = false;
#pragma unroll
            for (int k = 0; k < CPL; ++k) {
                const int ch = li + k * LPP;
                if (active && ch < nch) {
                    float q[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        q[i] = 0.f;
                        if (4 * ch + i < C) {
                            q[i] = kFast ? e[k][i] * rs : __fdiv_rn(e[k][i], sum);
                            if (kLabels) {
                                if (!have) { best = q[i]; bi = 4 * ch + i; have = true; }
                                else argmax_merge(q[i], 4 * ch + i, best, bi);
                            }
                        }
                    }
                    *reinterpret_cast<float4 *>(Q + (size_t)gp * Cp + 4 * ch) = make_float4(q[0], q[1], q[2], q[3]);
                }
            }
            if (kLabels) {
                // lanes without a real channel carry (-inf, INT_MAX) and can never win
                if (!have) { best = -INFINITY; bi = 0x7fffffff; }
                float rb = __shfl_sync(0xffffffffu, best, base_lane);
                int ri = __shfl_sync(0xffffffffu, bi, base_lane);
                for (int k = 1; k < LPP; ++k) {
                    float ob2 = __shfl_sync(0xffffffffu, best, base_lane + k);
                    int oi = __shfl_sync(0xffffffffu, bi, base_lane + k);
                    argmax_merge(ob2, oi, rb, ri);
                }
                if (active && li == 0) labels[gp] = ri;
            }
        }
    }
}

// Two entry points around the same body.  The plain one lets ptxas take the ~105 registers the six-chunk variants want
// (2 CTAs per SM): fastest for narrow rows (21 channels: 5.35 against 5.52 ms per pass).  The occ3 one caps registers at 80
// (3 CTAs per SM, ~30 bytes of spills): with rows of 300+ bytes the kernel is latency-bound at 25 % occupancy (ncu: 0.49
// eligible warps per scheduler) and the third CTA buys 9-18 % (150 ch: 38.2 -> 31.2, 81 ch @448: 31.6 -> 28.9 ms per pass).
template <bool kLabels, bool kFast, int CPL>
__global__ void __launch_bounds__(256) meanfield_update_warp_kernel(MeanFieldParams P, const float *__restrict__ unary,
                                                                    float *__restrict__ Q, int32_t *__restrict__ labels, int B, int H,
                                                                    int W, int C, int Cp, int LPP) {
    meanfield_update_warp_body<kLabels, kFast, CPL>(P, unary, Q, labels, B, H, W, C, Cp, LPP);
}
template <bool kLabels, bool kFast, int CPL>
__global__ void __launch_bounds__(256, 3) meanfield_update_warp_occ3_kernel(MeanFieldParams P, const float *__restrict__ unary,
                                                                            float *__restrict__ Q, int32_t *__restrict__ labels, int B,
                                                                            int H, int W, int C, int Cp, int LPP) {
    meanfield_update_warp_body<kLabels, kFast, CPL>(P, unary, Q, labels, B, H, W, C, Cp, LPP);
}

// ------------------------------------------------------------------------------------------ unary + layout helpers
// one thread per pixel; channel-major reads are coalesced across the warp, pixel-major writes go through smem
constexpr int kUnaryPix = 128;

__global__ void __launch_bounds__(kUnaryPix) unary_from_maps_kernel(const float *__restrict__ maps, const float *__restrict__ minmax,
                                                                    float *__restrict__ unary, int C, int Cp, int N) {
    extern __shared__ float s_tile[];  // [kUnaryPix][Cp+1]
    const int b = blockIdx.y;
    const int pitch = Cp + 1;
    const int p0 = blockIdx.x * kUnaryPix;
    const int p = p0 + threadIdx.x;
    const float *mb = maps + (long long)b * C * N;
    float *row = s_tile + threadIdx.x * pitch;
    if (p < N) {
        float mx = -INFINITY;
        bool has_nan = false;
        for (int c = 0; c < C; ++c) {
            float v = mb[(long long)c * N + p];
            if (minmax) {
                float mn = minmax[((long long)b * C + c) * 2], hi = minmax[((long long)b * C + c) * 2 + 1];
                v = __fdiv_rn(__fsub_rn(v, mn), __fsub_rn(hi, mn));  // DRV:1151-1152
            }
            row[c] = v;
            has_nan = has_nan || (v != v);
            mx = fmaxf(mx, v);
        }
        float sum = 0.f;
        for (int c = 0; c < C; ++c) {
            float e = expf(row[c] - mx);
            row[c] = e;
            sum += e;
        }
        for (int c = 0; c < C; ++c) {
            float pr = __fdiv_rn(row[c], sum);             // F.softmax(mask, dim=0), DRV:1057
            pr = fminf(fmaxf(pr, 1e-5f), 1.0f);            // np.clip(sm, 1e-5, 1.0)
            float u = -logf(pr);
            row[c] = has_nan ? __int_as_float(0x7fc00000) : u;  // softmax of a NaN column is NaN everywhere
        }
        for (int c = C; c < Cp; ++c) row[c] = 0.f;
    }
    __syncthreads();
    const int n_here = min(kUnaryPix, N - p0);
    float *ub = unary + ((long long)b * N + p0) * Cp;
    for (int i = threadIdx.x; i < n_here * Cp; i += blockDim.x) {
        int pp = i / Cp, c = i - pp * Cp;
        ub[i] = s_tile[pp * pitch + c];
    }
}

// Many-channel variant (C > 32): the one-thread-per-pixel kernel above needs a [128][C+1] shared tile, which at 150-171
// channels leaves 2 CTAs per SM.  Here pass A reduces max and sum per pixel (same arithmetic, same order), pass B
// revisits the maps in 32-channel slabs and transposes each slab through a [128][33] tile.
__global__ void __launch_bounds__(kUnaryPix) unary_stats_kernel(const float *__restrict__ maps, const float *__restrict__ minmax,
                                                                float2 *__restrict__ stats, int C, int N) {
    const int b = blockIdx.y;
    const int p = blockIdx.x * kUnaryPix + threadIdx.x;
    if (p >= N) return;
    const float *mb = maps + (long long)b * C * N + p;
    const float *mm = minmax ? minmax + (long long)b * C * 2 : nullptr;
    float mx = -INFINITY;
    bool has_nan = false;
    for (int c = 0; c < C; ++c) {
        float v = mb[(long long)c * N];
        if (mm) v = __fdiv_rn(__fsub_rn(v, mm[2 * c]), __fsub_rn(mm[2 * c + 1], mm[2 * c]));
        has_nan = has_nan || (v != v);
        mx = fmaxf(mx, v);
    }
    float sum = 0.f;
    for (int c = 0; c < C; ++c) {
        float v = mb[(long long)c * N];
        if (mm) v = __fdiv_rn(__fsub_rn(v, mm[2 * c]), __fsub_rn(mm[2 * c + 1], mm[2 * c]));
        sum += expf(v - mx);
    }
    stats[(long long)b * N + p] = make_float2(has_nan ? __int_as_float(0x7fc00000) : mx, sum);
}

constexpr int kUnarySlab = 32;

__global__ void __launch_bounds__(kUnaryPix) unary_write_kernel(const float *__restrict__ maps, const float *__restrict__ minmax,
                                                                const float2 *__restrict__ stats, float *__restrict__ unary, int C,
                                                                int Cp, int N) {
    __shared__ float s_tile[kUnaryPix][kUnarySlab + 1];
    const int b = blockIdx.z;
    const int p0 = blockIdx.x * kUnaryPix, c0 = blockIdx.y * kUnarySlab;
    const int p = p0 + threadIdx.x;
    const int n_c = min(kUnarySlab, Cp - c0);
    if (p < N) {
        const float2 st = stats[(long long)b * N + p];
        const bool has_nan = st.x != st.x;
        for (int j = 0; j < n_c; ++j) {
            const int c = c0 + j;
            float u = 0.f;  // padding channels
            if (c < C) {
                float v = maps[((long long)b * C + c) * N + p];
                if (minmax) {
                    float mn = minmax[((long long)b * C + c) * 2], hi = minmax[((long long)b * C + c) * 2 + 1];
                    v = __fdiv_rn(__fsub_rn(v, mn), __fsub_rn(hi, mn));
                }
                float pr = __fdiv_rn(expf(v - st.x), st.y);
                pr = fminf(fmaxf(pr, 1e-5f), 1.0f);
                u = has_nan ? __int_as_float(0x7fc00000) : -logf(pr);
            }
            s_tile[threadIdx.x][j] = u;
        }
    }
    __syncthreads();
    const int n_here = min(kUnaryPix, N - p0);
    for (int i = threadIdx.x; i < n_here * n_c; i += blockDim.x) {
        const int pp = i / n_c, j = i - pp * n_c;
        unary[((long long)b * N + p0 + pp) * Cp + c0 + j] = s_tile[pp][j];
    }
}

// [B,C,N] <-> [B,N,Cp] in 32-channel slabs through a [128][33] shared tile (any channel count)
__global__ void __launch_bounds__(kUnaryPix) pack_cn_to_nc_kernel(const float *__restrict__ src, float *__restrict__ dst, int C, int Cp, int N) {
    __shared__ float s_tile[kUnaryPix][kUnarySlab + 1];
    const int b = blockIdx.z, p0 = blockIdx.x * kUnaryPix, c0 = blockIdx.y * kUnarySlab, p = p0 + threadIdx.x;
    const int n_c = min(kUnarySlab, Cp - c0);
    if (p < N)
        for (int j = 0; j < n_c; ++j) s_tile[threadIdx.x][j] = (c0 + j < C) ? src[((long long)b * C + c0 + j) * N + p] : 0.f;
    __syncthreads();
    const int n_here = min(kUnaryPix, N - p0);
    for (int i = threadIdx.x; i < n_here * n_c; i += blockDim.x) {
        const int pp = i / n_c, j = i - pp * n_c;
        dst[((long long)b * N + p0 + pp) * Cp + c0 + j] = s_tile[pp][j];
    }
}

__global__ void __launch_bounds__(kUnaryPix) unpack_nc_to_cn_kernel(const float *__restrict__ src, float *__restrict__ dst, int C, int Cp, int N) {
    __shared__ float s_tile[kUnaryPix][kUnarySlab + 1];
    const int b = blockIdx.z, p0 = blockIdx.x * kUnaryPix, c0 = blockIdx.y * kUnarySlab, p = p0 + threadIdx.x;
    const int n_c = min(kUnarySlab, Cp - c0);
    const int n_here = min(kUnaryPix, N - p0);
    for (int i = threadIdx.x; i < n_here * n_c; i += blockDim.x) {
        const int pp = i / n_c, j = i - pp * n_c;
        s_tile[pp][j] = src[((long long)b * N + p0 + pp) * Cp + c0 + j];
    }
    __syncthreads();
    if (p < N)
        for (int j = 0; j < n_c; ++j)
            if (c0 + j < C) dst[((long long)b * C + c0 + j) * N + p] = s_tile[threadIdx.x][j];
}

// ------------------------------------------------------------------------------------------ host helpers
// CTAs per SM of the grid-stride kernels.  Measured on B200: the lattice blur is fastest with exactly one resident wave
// (8 CTAs x 148 SMs: every SM streams one contiguous slice, no tail), the splat with many more CTAs than fit (its CSR rows
// differ in length, so late CTAs fill the holes), the mean-field update with 8.
constexpr int kMultBlur = 8;
// Splat: the wider the rows, the more CTAs.  Measured per CRF pass (10 launches, profiles/time_other_configs.py; grid = 148 SMs x mult
// CTAs of 256 threads, grid-stride): 21 channels  64: 4.69 ms, 512: 5.26;  59 channels  128: 9.2, 256: 9.3, 512: 9.9;
// 81 channels @448  64: 24.5, 128: 21.3, 256: 19.6, 512: 20.0;  150 channels  64: 24.0, 128: 21.0, 256: 19.6, 512: 19.3, 1024: 20.4,
// one chunk per CTA (4096): 23.2.  (ncu at 150 channels, mult 64: 8.6 GB of DRAM reads per launch for 2.4 GB of Q, L2 hit rate 30 %:
// every CTA of a long grid-stride loop hops through the whole batch.  Handing chunks of consecutive vertices out in order from a
// global counter to one resident wave was also measured: 21.7 ms at 150 channels -- better than mult 64, worse than mult 256.)
static inline int mult_splat(int nch) { return nch <= 8 ? 64 : (nch <= 16 ? 128 : 256); }
// Update: one resident wave for narrow rows; with wide rows more, shorter-lived CTAs hide the gather latency a little better
// (per CRF pass, mult 8 / 16 / 32 / 64: 21 channels 5.36 / 5.36 / 5.42 / 5.48 ms, 81 channels @448 29.2 / 28.1 / 27.0 / 27.3, 150
// channels 31.2 / 30.3 / 29.2 / 28.8).
static inline int mult_update(int nch) { return nch <= 8 ? 8 : 32; }
static inline int grid_for(long long work_items, int threads, int mult = 16) {
    return (int)std::max<long long>(1, std::min<long long>((work_items + threads - 1) / threads, (long long)kNumSMs * mult));
}

// Vertex-value rows are packed at Cp floats (vp = Cp).  Padding rows so that none straddles a 128-byte line was measured on
// B200 and does not pay: the gather kernels do not speed up and the HBM-bound lattice blur slows by 9 % (profiles/README.md).
static inline LatticeView view_for(const pnp_lattice *lat, int Cp) {
    LatticeView L = make_view(lat);
    L.vp = Cp;
    return L;
}

static bool lattice_ok(const pnp_lattice *lat, int B) {
    if (!lat || lat->n_vertices < 0 || !lat->offset) return false;
    if (!lat->shared && lat->n_images != B) return false;
    return true;
}

// enqueue splat + (d+1) blurs; returns the buffer holding the blurred values
static const float *run_splat_blur(const LatticeView &L, const float *x, float *va, float *vb, int B, int Cp, int normalized,
                                   cudaStream_t st) {
    const int nch = Cp / 4;
    const int gy = L.shared ? B : 1;
    const int div = L.shared ? std::min(B, 8) : 1;
    const int gx_splat = std::max(1, grid_for((long long)(L.M + 1) * nch, 256, mult_splat(nch)) / div);
    const int gx = std::max(1, grid_for((long long)(L.M + 1) * nch, 256, kMultBlur) / div);
    const int id_splat = L.shared ? kSplatSpatial : kSplatBilateral;
    const int id_blur = L.shared ? kBlurAxisSpatial : kBlurAxisBilateral;
    PNP_LAUNCH(id_splat, st, splat_kernel<<<dim3(gx_splat, gy), 256, 0, st>>>(L, x, va, Cp, normalized));
    float *src = va, *dst = vb;
    // Two axes per launch halve the HBM traffic of the blur but re-gather the first axis at both neighbours; measured on
    // B200 that pays up to ~340-byte rows (21 ch: 0.187 vs 0.232 ms, 81 ch @448: 23.6 vs 27.5 ms per pass) and loses with
    // 600-byte rows (150 ch: 44.4 vs 38.6 ms), where one launch per axis already runs at the HBM roofline.
    int j = 0;
    if (Cp <= 112) {
        for (; j + 1 < L.Dp1; j += 2) {  // axes (0,1), (2,3), (4,5): two passes per launch
            PNP_LAUNCH(id_blur, st, blur_axis2_kernel<<<dim3(gx, gy), 256, 0, st>>>(L, src, dst, j, j + 1, Cp));
            std::swap(src, dst);
        }
    }
    for (; j < L.Dp1; ++j) {
        PNP_LAUNCH(id_blur, st, blur_axis_kernel<<<dim3(gx, gy), 256, 0, st>>>(L, src, dst, j, Cp));
        std::swap(src, dst);
    }
    return src;
}

static size_t unary_smem(int Cp) { return (size_t)kUnaryPix * (Cp + 1) * sizeof(float); }

}  // namespace pnp

using namespace pnp;

extern "C" size_t pnp_crf_scratch_bytes(const pnp_lattice *const *lattices, int n_kernels, int B, int Cp) {
    if (!lattices || n_kernels < 1 || n_kernels > kMaxKernels || B < 1 || Cp < 4 || Cp % 4) return 0;
    size_t total = 0;
    for (int k = 0; k < n_kernels; ++k) {
        if (!lattice_ok(lattices[k], B)) return 0;
        LatticeView L = view_for(lattices[k], Cp);
        total += 2 * align_up((size_t)value_rows(L, B) * L.vp * sizeof(float), 256);
    }
    return total;
}

extern "C" int pnp_crf_filter(const pnp_lattice *lat, const float *x, float *y, void *scratch, size_t scratch_bytes, int B,
                              int Cp, int normalized, pnp_stream_t stream) {
    if (!x || !y || !scratch || B < 1 || Cp < 4 || Cp % 4 || Cp > 1024 || !lattice_ok(lat, B)) return PNP_ERR_INVALID_ARGUMENT;
    const pnp_lattice *one[1] = {lat};
    if (scratch_bytes < pnp_crf_scratch_bytes(one, 1, B, Cp)) return PNP_ERR_WORKSPACE;
    cudaStream_t st = as_stream(stream);
    LatticeView L = view_for(lat, Cp);
    size_t buf = align_up((size_t)value_rows(L, B) * L.vp * sizeof(float), 256);
    float *va = reinterpret_cast<float *>(scratch);
    float *vb = reinterpret_cast<float *>(reinterpret_cast<char *>(scratch) + buf);
    const float *blurred = run_splat_blur(L, x, va, vb, B, Cp, normalized, st);
    slice_kernel<<<grid_for((long long)B * L.N * (Cp / 4), 256), 256, 0, st>>>(L, blurred, y, B, Cp, normalized);
    return launch_status();
}

extern "C" int pnp_crf_inference(const pnp_lattice *const *lattices, const float *weights, int n_kernels,
                                 const float *unary, float *Q, void *scratch, size_t scratch_bytes, int32_t *labels, int B,
                                 int C, int Cp, int n_iter, pnp_stream_t stream) {
    if (!lattices || !weights || !unary || !Q || !scratch || n_kernels < 1 || n_kernels > kMaxKernels || B < 1 || C < 1 ||
        Cp < C || Cp % 4 || Cp > 1024 || n_iter < 0)
        return PNP_ERR_INVALID_ARGUMENT;
    size_t need = pnp_crf_scratch_bytes(lattices, n_kernels, B, Cp);
    if (need == 0) return PNP_ERR_INVALID_ARGUMENT;
    if (scratch_bytes < need) return PNP_ERR_WORKSPACE;
    const int N = lattices[0]->n_pixels;
    for (int k = 1; k < n_kernels; ++k)
        if (lattices[k]->n_pixels != N) return PNP_ERR_INVALID_ARGUMENT;
    cudaStream_t st = as_stream(stream);

    MeanFieldParams P;
    float *va[kMaxKernels], *vb[kMaxKernels];
    char *p = reinterpret_cast<char *>(scratch);
    for (int k = 0; k < kMaxKernels; ++k) {
        if (k < n_kernels) {
            P.lat[k] = view_for(lattices[k], Cp);
            P.weight[k] = weights[k];
            size_t buf = align_up((size_t)value_rows(P.lat[k], B) * P.lat[k].vp * sizeof(float), 256);
            va[k] = reinterpret_cast<float *>(p);
            vb[k] = reinterpret_cast<float *>(p + buf);
            p += 2 * buf;
        } else {
            P.lat[k] = P.lat[0];
            P.weight[k] = 0.f;
            va[k] = vb[k] = nullptr;
        }
        P.values[k] = nullptr;
    }
    const int TP = 256 / (Cp / 4);
    const long long n_tiles = ((long long)B * N + TP - 1) / TP;
    const int grid = (int)std::max<long long>(1, std::min<long long>(n_tiles, (long long)kNumSMs * 8));
    const int Wimg = lattices[0]->width, Himg = Wimg > 0 ? N / Wimg : 0;
    // lanes per pixel / chunks per lane: the split of the nch chunks over a warp that idles the fewest lanes
    const int nch_all = Cp / 4;
    int LPP = 0, CPL = 0;
    {
        double best_eff = 0.0;
        for (int cpl = 1; cpl <= 6; ++cpl) {
            if (cpl == 5) continue;
            int lpp = (nch_all + cpl - 1) / cpl;
            if (lpp > 32) continue;
            double eff = (double)(32 / lpp) * nch_all / (32.0 * cpl);
            if (eff >= best_eff - 1e-9) { best_eff = eff; LPP = lpp; CPL = cpl; }  // ties: more chunks per lane wins (measured)
        }
    }
    const bool occ3 = (CPL == 4 || CPL == 6) && nch_all >= 12;   // rows of >= 192 bytes
    const bool warp_path = CPL > 0 && Wimg > 0 && (long long)Himg * Wimg == N && (long long)B * N < (1ll << 31) / Cp;
    const int grid_w = (int)std::max<long long>(
        1, std::min<long long>((long long)B * ((Himg + kTile - 1) / kTile) * ((Wimg + kTile - 1) / kTile), (long long)kNumSMs * mult_update(nch_all)));
    auto launch_warp = [&](auto labels_tag, auto fast_tag) {
        constexpr bool kL = decltype(labels_tag)::value, kF = decltype(fast_tag)::value;
        if (occ3) {
            if (CPL == 4) PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_warp_occ3_kernel<kL, kF, 4><<<grid_w, 256, 0, st>>>(P, unary, Q, labels, B, Himg, Wimg, C, Cp, LPP));
            else PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_warp_occ3_kernel<kL, kF, 6><<<grid_w, 256, 0, st>>>(P, unary, Q, labels, B, Himg, Wimg, C, Cp, LPP));
            return;
        }
        switch (CPL) {
            case 1: PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_warp_kernel<kL, kF, 1><<<grid_w, 256, 0, st>>>(P, unary, Q, labels, B, Himg, Wimg, C, Cp, LPP)); break;
            case 2: PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_warp_kernel<kL, kF, 2><<<grid_w, 256, 0, st>>>(P, unary, Q, labels, B, Himg, Wimg, C, Cp, LPP)); break;
            case 3: PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_warp_kernel<kL, kF, 3><<<grid_w, 256, 0, st>>>(P, unary, Q, labels, B, Himg, Wimg, C, Cp, LPP)); break;
            case 4: PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_warp_kernel<kL, kF, 4><<<grid_w, 256, 0, st>>>(P, unary, Q, labels, B, Himg, Wimg, C, Cp, LPP)); break;
            default: PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_warp_kernel<kL, kF, 6><<<grid_w, 256, 0, st>>>(P, unary, Q, labels, B, Himg, Wimg, C, Cp, LPP)); break;
        }
    };
    auto update = [&](bool with_labels) {
        const bool fast = warp_path && P.n_kernels == 2 && P.lat[0].Dp1 == 3 && P.lat[0].shared && P.lat[1].Dp1 == 6 && !P.lat[1].shared;
        if (warp_path) {
            if (with_labels && fast) launch_warp(std::true_type{}, std::true_type{});
            else if (with_labels) launch_warp(std::true_type{}, std::false_type{});
            else if (fast) launch_warp(std::false_type{}, std::true_type{});
            else launch_warp(std::false_type{}, std::false_type{});
        } else {
            if (with_labels)
                PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_kernel<true><<<grid, 256, 0, st>>>(P, unary, Q, labels, B, N, C, Cp));
            else
                PNP_LAUNCH(kMeanfieldUpdate, st, meanfield_update_kernel<false><<<grid, 256, 0, st>>>(P, unary, Q, labels, B, N, C, Cp));
        }
    };

    // Q0 = softmax(-U)
    P.n_kernels = 0;
    update(n_iter == 0 && labels != nullptr);
    for (int it = 0; it < n_iter; ++it) {
        for (int k = 0; k < n_kernels; ++k) P.values[k] = run_splat_blur(P.lat[k], Q, va[k], vb[k], B, Cp, 1, st);
        P.n_kernels = n_kernels;
        update(it == n_iter - 1 && labels != nullptr);
    }
    return launch_status();
}

extern "C" size_t pnp_crf_unary_workspace_bytes(int B, int C, int N) {
    if (B < 1 || C < 1 || N < 1) return 0;
    return C > kUnarySlab ? align_up((size_t)B * N * sizeof(float2), 256) : 0;
}

extern "C" int pnp_crf_unary_from_maps(const float *maps, const float *minmax, float *unary, void *workspace, size_t workspace_bytes,
                                       int B, int C, int N, pnp_stream_t stream) {
    if (!maps || !unary || B < 1 || C < 1 || N < 1 || B > 65535) return PNP_ERR_INVALID_ARGUMENT;
    const int Cp = (C + 3) / 4 * 4;
    cudaStream_t st = as_stream(stream);
    if (C > kUnarySlab) {  // many channels: two passes, 32-channel slabs
        if (!workspace || workspace_bytes < pnp_crf_unary_workspace_bytes(B, C, N)) return PNP_ERR_WORKSPACE;
        float2 *stats = reinterpret_cast<float2 *>(workspace);
        const bool timed = prof::on(kCrfUnary, st);
        if (timed) prof::begin(kCrfUnary, st);
        unary_stats_kernel<<<dim3(ceil_div(N, kUnaryPix), B), kUnaryPix, 0, st>>>(maps, minmax, stats, C, N);
        unary_write_kernel<<<dim3(ceil_div(N, kUnaryPix), ceil_div(Cp, kUnarySlab), B), kUnaryPix, 0, st>>>(maps, minmax, stats, unary, C,
                                                                                                           Cp, N);
        if (timed) prof::end(kCrfUnary, st);
        return launch_status();
    }
    size_t smem = unary_smem(Cp);
    cudaError_t e = allow_smem(unary_from_maps_kernel, smem);
    if (e != cudaSuccess) return cuda_err(e);
    PNP_LAUNCH(kCrfUnary, st, unary_from_maps_kernel<<<dim3(ceil_div(N, kUnaryPix), B), kUnaryPix, smem, st>>>(maps, minmax, unary, C, Cp, N));
    return launch_status();
}

extern "C" int pnp_crf_pack_cn_to_nc(const float *src_cn, float *dst_nc, int B, int C, int N, pnp_stream_t stream) {
    if (!src_cn || !dst_nc || B < 1 || C < 1 || N < 1 || B > 65535) return PNP_ERR_INVALID_ARGUMENT;
    const int Cp = (C + 3) / 4 * 4;
    pack_cn_to_nc_kernel<<<dim3(ceil_div(N, kUnaryPix), ceil_div(Cp, kUnarySlab), B), kUnaryPix, 0, as_stream(stream)>>>(src_cn, dst_nc, C, Cp, N);
    return launch_status();
}

extern "C" int pnp_crf_unpack_nc_to_cn(const float *src_nc, float *dst_cn, int B, int C, int N, pnp_stream_t stream) {
    if (!src_nc || !dst_cn || B < 1 || C < 1 || N < 1 || B > 65535) return PNP_ERR_INVALID_ARGUMENT;
    const int Cp = (C + 3) / 4 * 4;
    unpack_nc_to_cn_kernel<<<dim3(ceil_div(N, kUnaryPix), ceil_div(Cp, kUnarySlab), B), kUnaryPix, 0, as_stream(stream)>>>(src_nc, dst_cn, C, Cp, N);
    return launch_status();
}
