// lattice.cu -- (e) part 1: permutohedral lattice construction on the GPU.
// Replaces what pydensecrf's addPairwiseGaussian / addPairwiseBilateral do on the CPU (DRV:1068-1069):
// Permutohedral::init (embed, hash, neighbours) and DenseKernel::initLattice (symmetric normalisation).
//
// Pipeline (all on one stream, no host round trip until pnp_lattice_finish):
//   embed      per pixel: elevate -> nearest remainder-0 point -> rank -> barycentric -> d+1 vertex keys, each key
//              packed into 64 bits and inserted into an open-addressing table with atomicCAS.  Lanes of a warp that
//              hold the same key (neighbouring pixels share vertices) are grouped with __match_any_sync and only the
//              group leader touches the table ("warp-level hashing"); it also records the smallest entry id that
//              touched the slot.
//   number     flag = "this (pixel, remainder) entry touched its slot first"; an exclusive scan over the flags in
//              entry order numbers the vertices exactly like the sequential reference's hash table (insertion
//              order), so offsets are bit-identical to the CPU lattice and vertices first met by nearby pixels are
//              nearby in memory.
//   neighbours per vertex and axis: unpack key, step +-1 along the axis, look the two keys up.
//   CSR        entries grouped by vertex (count, scan, fill) and each row sorted by entry id: the splat becomes a
//              gather that sums contributions in pixel order -- deterministic, atomic-free, and the same fp32
//              summation order as the sequential reference.
//   norm       K applied to a field of ones (scalar splat / blur / slice), then 1/sqrt(. + 1e-20).
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "lattice.cuh"

namespace pnp {

// ------------------------------------------------------------------------------------------ device scan
constexpr int kScanThreads = 256;
constexpr int kScanItems = 16;
constexpr int kScanChunk = kScanThreads * kScanItems;

__global__ void __launch_bounds__(kScanThreads) scan_reduce_kernel(const int32_t *__restrict__ in, int32_t *__restrict__ block_sums,
                                                                   long long n) {
    __shared__ int s_warp[kScanThreads / 32];
    long long base = (long long)blockIdx.x * kScanChunk;
    int sum = 0;
    for (int i = threadIdx.x; i < kScanChunk; i += kScanThreads) {
        long long idx = base + i;
        if (idx < n) sum += in[idx];
    }
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < kScanThreads / 32; ++w) t += s_warp[w];
        block_sums[blockIdx.x] = t;
    }
}

// exclusive scan of block sums in place by ONE block; writes the grand total to *total_out (optional)
__global__ void __launch_bounds__(1024) scan_spine_kernel(int32_t *__restrict__ block_sums, int nb, int32_t *__restrict__ total_out) {
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < nb; base += 1024) {
        int i = base + threadIdx.x;
        int v = (i < nb) ? block_sums[i] : 0;
        int incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane];
            int wi = w;
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            s_warp[lane] = wi - w;  // exclusive warp offsets
        }
        __syncthreads();
        int carry = s_carry;
        int excl = carry + s_warp[warp] + incl - v;
        if (i < nb) block_sums[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total_out) *total_out = s_carry;
}

// out[i] = exclusive prefix of in[0..i); in may alias out.  block_sums already exclusive-scanned.
__global__ void __launch_bounds__(kScanThreads) scan_apply_kernel(const int32_t *in, int32_t *out,
                                                                  const int32_t *__restrict__ block_sums, long long n) {
    __shared__ int s_warp[kScanThreads / 32];
    const long long base = (long long)blockIdx.x * kScanChunk + (long long)threadIdx.x * kScanItems;
    int v[kScanItems];
    int sum = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
        long long idx = base + k;
        v[k] = (idx < n) ? in[idx] : 0;
        sum += v[k];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = sum;
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int warp_off = 0;
    for (int w = 0; w < warp; ++w) warp_off += s_warp[w];
    int run = block_sums[blockIdx.x] + warp_off + incl - sum;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
        long long idx = base + k;
        if (idx < n) out[idx] = run;
        run += v[k];
    }
}

static int exclusive_scan(const int32_t *in, int32_t *out, int32_t *block_sums, long long n, int32_t *total_out, cudaStream_t st) {
    int nb = (int)((n + kScanChunk - 1) / kScanChunk);
    if (nb < 1) nb = 1;
    scan_reduce_kernel<<<nb, kScanThreads, 0, st>>>(in, block_sums, n);
    scan_spine_kernel<<<1, 1024, 0, st>>>(block_sums, nb, total_out);
    scan_apply_kernel<<<nb, kScanThreads, 0, st>>>(in, out, block_sums, n);
    return launch_status();
}

// ------------------------------------------------------------------------------------------ key packing
constexpr unsigned long long kEmptyKey = ~0ull;

template <int D>
struct KeyPack {
    static constexpr int kBits = (D <= 3) ? 16 : 12;  // r (3 bits) + D * kBits <= 63
    static constexpr int kBias = 1 << (kBits - 1);
    // coords c[i] = q[i]*(D+1) + r  ->  r | (q[i]+bias) << (3 + i*kBits)
    __device__ static bool pack(const int *c, int r, unsigned long long &key) {
        key = (unsigned long long)r;
        bool ok = true;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            int q = (c[i] - r) / (D + 1) + kBias;  // exact: c[i] == r (mod D+1)
            ok = ok && (q >= 0) && (q < (1 << kBits));
            key |= (unsigned long long)(unsigned)(q & ((1 << kBits) - 1)) << (3 + i * kBits);
        }
        return ok;
    }
    __device__ static void unpack(unsigned long long key, int *c, int &r) {
        r = (int)(key & 7ull);
#pragma unroll
        for (int i = 0; i < D; ++i) {
            int q = (int)((key >> (3 + i * kBits)) & ((1ull << kBits) - 1)) - kBias;
            c[i] = q * (D + 1) + r;
        }
    }
};

__device__ __forceinline__ unsigned hash64(unsigned long long k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdULL;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ULL;
    k ^= k >> 33;
    return (unsigned)k;
}

__device__ __forceinline__ int table_insert(unsigned long long *table, unsigned cap_mask, unsigned long long key) {
    unsigned h = hash64(key) & cap_mask;
    while (true) {
        unsigned long long prev = atomicCAS(&table[h], kEmptyKey, key);
        if (prev == kEmptyKey || prev == key) return (int)h;
        h = (h + 1) & cap_mask;
    }
}

__device__ __forceinline__ int table_find(const unsigned long long *table, unsigned cap_mask, unsigned long long key) {
    unsigned h = hash64(key) & cap_mask;
    while (true) {
        unsigned long long cur = table[h];
        if (cur == key) return (int)h;
        if (cur == kEmptyKey) return -1;
        h = (h + 1) & cap_mask;
    }
}

// ------------------------------------------------------------------------------------------ embed
struct EmbedParams {
    const uint8_t *rgb;  // [n_images,H,W,3] or null
    int W, N;            // N = H*W
    long long n_lp;      // lattice pixels = n_images*N
    float sx, sy, sr, sg, sb;
    float scale_factor[5];
    unsigned cap_mask;   // per-image table capacity - 1
};

template <int D>
__global__ void __launch_bounds__(256) lattice_embed_kernel(EmbedParams prm, unsigned long long *__restrict__ table,
                                                            int32_t *__restrict__ first, int32_t *__restrict__ offset,
                                                            float *__restrict__ bary, int32_t *__restrict__ counters) {
    const long long lp = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const bool valid = lp < prm.n_lp;
    const int lane = threadIdx.x & 31;
    int img = 0;
    int rem0[D + 1], rank[D + 1];
    float b[D + 2];
    if (valid) {
        img = (int)(lp / prm.N);
        const int pix = (int)(lp - (long long)img * prm.N);
        const int y = pix / prm.W, x = pix - y * prm.W;
        float f[D];
        f[0] = __fdiv_rn((float)x, prm.sx);
        f[1] = __fdiv_rn((float)y, prm.sy);
        if (D == 5) {
            const uint8_t *c = prm.rgb + lp * 3;
            f[D - 3] = __fdiv_rn((float)c[0], prm.sr);
            f[D - 2] = __fdiv_rn((float)c[1], prm.sg);
            f[D - 1] = __fdiv_rn((float)c[2], prm.sb);
        }
        // elevate onto the hyperplane sum = 0 (every product / sum separately rounded: the reference is built
        // without FMA contraction)
        float el[D + 1];
        float sm = 0.f;
#pragma unroll
        for (int j = D; j > 0; --j) {
            float cf = __fmul_rn(f[j - 1], prm.scale_factor[j - 1]);
            el[j] = __fsub_rn(sm, __fmul_rn((float)j, cf));
            sm = __fadd_rn(sm, cf);
        }
        el[0] = sm;
        // nearest remainder-0 lattice point
        const float down_factor = 1.0f / (D + 1);
        const float up_factor = (float)(D + 1);
        int sum = 0;
#pragma unroll
        for (int i = 0; i <= D; ++i) {
            float v = __fmul_rn(down_factor, el[i]);
            float up = __fmul_rn(ceilf(v), up_factor);
            float down = __fmul_rn(floorf(v), up_factor);
            int rd2 = (__fsub_rn(up, el[i]) < __fsub_rn(el[i], down)) ? (int)(short)up : (int)(short)down;
            rem0[i] = rd2;
            sum = (int)__fadd_rn((float)sum, __fmul_rn((float)rd2, down_factor));  // int += float, truncating
        }
        // rank of the residuals
#pragma unroll
        for (int i = 0; i <= D; ++i) rank[i] = 0;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            float di = __fsub_rn(el[i], (float)rem0[i]);
#pragma unroll
            for (int j = i + 1; j <= D; ++j) {
                if (di < __fsub_rn(el[j], (float)rem0[j]))
                    rank[i]++;
                else
                    rank[j]++;
            }
        }
        // back onto the plane
#pragma unroll
        for (int i = 0; i <= D; ++i) {
            rank[i] += sum;
            if (rank[i] < 0) {
                rank[i] += D + 1;
                rem0[i] += D + 1;
            } else if (rank[i] > D) {
                rank[i] -= D + 1;
                rem0[i] -= D + 1;
            }
        }
        // barycentric coordinates (accumulated in coordinate order, like the reference)
#pragma unroll
        for (int k = 0; k <= D + 1; ++k) b[k] = 0.f;
#pragma unroll
        for (int i = 0; i <= D; ++i) {
            float v = __fmul_rn(__fsub_rn(el[i], (float)rem0[i]), down_factor);
            const int k0 = D - rank[i];
#pragma unroll
            for (int k = 0; k <= D + 1; ++k) {
                if (k == k0) b[k] = __fadd_rn(b[k], v);
                if (k == k0 + 1) b[k] = __fsub_rn(b[k], v);
            }
        }
        b[0] = __fadd_rn(b[0], __fadd_rn(1.0f, b[D + 1]));
    }
    // d+1 simplex vertices: hash-insert with warp-level de-duplication (all 32 lanes take part in the votes)
    unsigned long long *my_table = table + (size_t)img * ((size_t)prm.cap_mask + 1);
    const unsigned img_peers = __match_any_sync(0xffffffffu, img);
#pragma unroll
    for (int r = 0; r <= D; ++r) {
        unsigned long long key = kEmptyKey - 1 - (unsigned long long)lane;  // distinct dummy for idle lanes
        bool ok = true;
        if (valid) {
            int c[D];
#pragma unroll
            for (int i = 0; i < D; ++i) c[i] = rem0[i] + ((rank[i] <= D - r) ? r : r - (D + 1));
            ok = KeyPack<D>::pack(c, r, key);
            if (!ok) {
                atomicOr(&counters[1], 1);
                key = kEmptyKey - 1 - (unsigned long long)lane;
            }
        }
        const unsigned peers = __match_any_sync(0xffffffffu, key) & img_peers;
        const int leader = __ffs(peers) - 1;
        const long long e = lp * (D + 1) + r;
        int slot = -1;
        if (valid && ok && lane == leader) {
            int h = table_insert(my_table, prm.cap_mask, key);
            slot = img * (int)(prm.cap_mask + 1) + h;
            atomicMin(&first[slot], (int)e);
        }
        slot = __shfl_sync(0xffffffffu, slot, leader);
        if (valid) {
            offset[e] = ok ? slot : 0;
            bary[e] = b[r];
        }
    }
}

// flag[e] = 1 iff entry e is the first to touch its slot
__global__ void __launch_bounds__(256) lattice_flag_kernel(const int32_t *__restrict__ offset, const int32_t *__restrict__ first,
                                                           int32_t *__restrict__ flag, long long n_entries) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_entries; e += (long long)gridDim.x * blockDim.x)
        flag[e] = (first[offset[e]] == (int)e) ? 1 : 0;
}

// first touchers publish the dense id of their slot and remember the key
__global__ void __launch_bounds__(256) lattice_assign_kernel(const int32_t *__restrict__ offset, const int32_t *__restrict__ first,
                                                             const int32_t *__restrict__ prefix, const unsigned long long *__restrict__ table,
                                                             int32_t *__restrict__ slot_id, unsigned long long *__restrict__ keys_dense,
                                                             long long n_entries) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_entries; e += (long long)gridDim.x * blockDim.x) {
        int slot = offset[e];
        if (first[slot] == (int)e) {
            int id = prefix[e];
            slot_id[slot] = id;
            keys_dense[id] = table[slot];
        }
    }
}

// vstart[b] = first vertex id of image b; vstart[n_images] = M
__global__ void lattice_vstart_kernel(const int32_t *__restrict__ prefix, const int32_t *__restrict__ counters, int32_t *__restrict__ vstart,
                                      int n_images, long long entries_per_image) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < n_images) vstart[b] = prefix[(long long)b * entries_per_image];
    if (b == n_images) vstart[b] = counters[0];
}

// offset: slot -> dense id; count entries per vertex
__global__ void __launch_bounds__(256) lattice_offsets_kernel(int32_t *__restrict__ offset, const int32_t *__restrict__ slot_id,
                                                              int32_t *__restrict__ row_cnt, long long n_entries) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_entries; e += (long long)gridDim.x * blockDim.x) {
        int id = slot_id[offset[e]];
        offset[e] = id;
        atomicAdd(&row_cnt[id], 1);
    }
}

__global__ void __launch_bounds__(256) csr_fill_kernel(const int32_t *__restrict__ offset, const int32_t *__restrict__ row_ptr,
                                                       int32_t *__restrict__ cursor, int32_t *__restrict__ csr_tmp, long long n_entries) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_entries; e += (long long)gridDim.x * blockDim.x) {
        int id = offset[e];
        int pos = row_ptr[id] + atomicAdd(&cursor[id], 1);
        csr_tmp[pos] = (int)e;
    }
}

// Sort each row by entry id (rank counting; entries are distinct) and emit (pixel, weight) in that order.
// Rows up to kShortRow entries: one 8-lane group per row.  Longer rows are left to csr_sort_long_kernel.
constexpr int kShortRow = 256;
constexpr int kGroup = 8;

__global__ void __launch_bounds__(256) csr_sort_short_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ csr_tmp,
                                                             const float *__restrict__ bary, int32_t *__restrict__ csr_pix,
                                                             float *__restrict__ csr_w, int32_t *counters, int32_t *__restrict__ long_rows,
                                                             int Dp1) {
    const int M = counters[0];
    const int sub = threadIdx.x % kGroup;
    int longest = 0;
    for (long long v = (blockIdx.x * (long long)blockDim.x + threadIdx.x) / kGroup; v < M;
         v += (long long)gridDim.x * blockDim.x / kGroup) {
        const int beg = row_ptr[v], len = row_ptr[v + 1] - beg;
        longest = max(longest, len);
        if (len > kShortRow) {  // left to csr_sort_long_kernel, which walks this compact list
            if (sub == 0) long_rows[atomicAdd(&counters[3], 1)] = (int)v;
            continue;
        }
        for (int i = sub; i < len; i += kGroup) {
            const int e = csr_tmp[beg + i];
            int rank = 0;
            for (int k = 0; k < len; ++k) rank += (csr_tmp[beg + k] < e);
            csr_pix[beg + rank] = e / Dp1;
            csr_w[beg + rank] = bary[e];
        }
    }
    for (int o = 16; o > 0; o >>= 1) longest = max(longest, __shfl_xor_sync(0xffffffffu, longest, o));
    if ((threadIdx.x & 31) == 0 && longest > 0) atomicMax(&counters[2], longest);
}

__global__ void __launch_bounds__(256) csr_sort_long_kernel(const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ csr_tmp,
                                                            const float *__restrict__ bary, int32_t *__restrict__ csr_pix,
                                                            float *__restrict__ csr_w, const int32_t *__restrict__ counters,
                                                            const int32_t *__restrict__ long_rows, int Dp1) {
    const int n_long = counters[3];
    for (int i_row = blockIdx.x; i_row < n_long; i_row += gridDim.x) {
        const int v = long_rows[i_row];
        const int beg = row_ptr[v], len = row_ptr[v + 1] - beg;
        for (int i = threadIdx.x; i < len; i += blockDim.x) {
            const int e = csr_tmp[beg + i];
            int rank = 0;
            for (int k = 0; k < len; ++k) rank += (csr_tmp[beg + k] < e);
            csr_pix[beg + rank] = e / Dp1;
            csr_w[beg + rank] = bary[e];
        }
    }
}

// blur neighbours: for vertex v and axis j, the vertices at key -+ (1,..,1) +- (D+1) e_j
template <int D>
__global__ void __launch_bounds__(256) lattice_neighbors_kernel(const unsigned long long *__restrict__ keys_dense,
                                                                const unsigned long long *__restrict__ table,
                                                                const int32_t *__restrict__ slot_id, const int32_t *__restrict__ vstart,
                                                                const int32_t *__restrict__ counters, int32_t *__restrict__ nbr,
                                                                int n_images, unsigned cap_mask, int vertex_stride) {
    const int M = counters[0];
    for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < M; v += (long long)gridDim.x * blockDim.x) {
        // image of this vertex: largest b with vstart[b] <= v
        int lo = 0, hi = n_images - 1;
        while (lo < hi) {
            int mid = (lo + hi + 1) >> 1;
            if (vstart[mid] <= v) lo = mid; else hi = mid - 1;
        }
        const unsigned long long *my_table = table + (size_t)lo * ((size_t)cap_mask + 1);
        const int slot_base = lo * (int)(cap_mask + 1);
        int c[D], r;
        KeyPack<D>::unpack(keys_dense[v], c, r);
#pragma unroll
        for (int j = 0; j <= D; ++j) {
            int c1[D], c2[D];
#pragma unroll
            for (int i = 0; i < D; ++i) { c1[i] = c[i] - 1; c2[i] = c[i] + 1; }
            if (j < D) {
#pragma unroll
                for (int i = 0; i < D; ++i)
                    if (i == j) { c1[i] = c[i] + D; c2[i] = c[i] - D; }
            }
            const int r1 = (r + D) % (D + 1), r2 = (r + 1) % (D + 1);
            unsigned long long k1, k2;
            int n1 = 0, n2 = 0;
            if (KeyPack<D>::pack(c1, r1, k1)) {
                int h = table_find(my_table, cap_mask, k1);
                if (h >= 0) n1 = slot_id[slot_base + h] + 1;
            }
            if (KeyPack<D>::pack(c2, r2, k2)) {
                int h = table_find(my_table, cap_mask, k2);
                if (h >= 0) n2 = slot_id[slot_base + h] + 1;
            }
            reinterpret_cast<int2 *>(nbr)[(size_t)j * vertex_stride + v] = make_int2(n1, n2);
        }
    }
}


// ------------------------------------------------------------------------------------------ norm = 1/sqrt(K 1 + 1e-20)
__global__ void __launch_bounds__(256) norm_splat_kernel(const int32_t *__restrict__ row_ptr, const float *__restrict__ csr_w,
                                                         const int32_t *__restrict__ counters, float *__restrict__ values) {
    const int M = counters[0];
    for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v <= M; v += (long long)gridDim.x * blockDim.x) {
        if (v == M) { values[0] = 0.f; continue; }  // sentinel row
        float acc = 0.f;
        for (int k = row_ptr[v]; k < row_ptr[v + 1]; ++k) acc = __fadd_rn(acc, csr_w[k]);  // w * 1.0f
        values[v + 1] = acc;
    }
}

__global__ void __launch_bounds__(256) norm_blur_kernel(const float *__restrict__ old_v, float *__restrict__ new_v,
                                                        const int32_t *__restrict__ nbr_axis, const int32_t *__restrict__ counters) {
    const int M = counters[0];
    for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v <= M; v += (long long)gridDim.x * blockDim.x) {
        if (v == M) { new_v[0] = 0.f; continue; }
        int2 n = reinterpret_cast<const int2 *>(nbr_axis)[v];
        new_v[v + 1] = __fadd_rn(old_v[v + 1], __fmul_rn(0.5f, __fadd_rn(old_v[n.x], old_v[n.y])));
    }
}

__global__ void __launch_bounds__(256) norm_slice_kernel(const float *__restrict__ values, const int32_t *__restrict__ offset,
                                                         const float *__restrict__ bary, float *__restrict__ norm, long long n_lp,
                                                         int Dp1, float alpha) {
    for (long long lp = blockIdx.x * (long long)blockDim.x + threadIdx.x; lp < n_lp; lp += (long long)gridDim.x * blockDim.x) {
        float out = 0.f;
        for (int j = 0; j < Dp1; ++j) {
            int o = offset[lp * Dp1 + j] + 1;
            float w = bary[lp * Dp1 + j];
            out = __fadd_rn(out, __fmul_rn(__fmul_rn(w, values[o]), alpha));
        }
        norm[lp] = (float)(1.0 / sqrt((double)out + 1e-20));
    }
}

__global__ void __launch_bounds__(256) csr_norm_fill_kernel(const int32_t *__restrict__ csr_pix, const float *__restrict__ norm,
                                                            float *__restrict__ csr_norm, long long n_entries) {
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n_entries; k += (long long)gridDim.x * blockDim.x)
        csr_norm[k] = norm[csr_pix[k]];
}

// ------------------------------------------------------------------------------------------ host side
static inline unsigned long long table_capacity(int d, int n_pixels) {
    unsigned long long need = 2ull * (unsigned long long)n_pixels * (d + 1);
    unsigned long long cap = 1024;
    while (cap < need) cap <<= 1;
    return cap;
}

struct BuildLayout {
    size_t off_table, off_first, off_slot_id, off_keys, off_prefix, off_block_sums, off_row_cnt, off_csr_tmp, off_vstart, off_va,
        off_vb, total;
};

static BuildLayout build_layout(int d, int n_images, int n_pixels) {
    BuildLayout L;
    const size_t n_entries = (size_t)n_images * n_pixels * (d + 1);
    const size_t slots = (size_t)n_images * table_capacity(d, n_pixels);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes, 256); return r; };
    L.off_table = take(slots * 8);
    L.off_first = take(slots * 4);
    L.off_slot_id = take(slots * 4);
    L.off_keys = take(n_entries * 8);
    L.off_prefix = take(n_entries * 4);
    L.off_block_sums = take(((n_entries + kScanChunk - 1) / kScanChunk + 1) * 4);
    L.off_row_cnt = take((n_entries + 1) * 4);
    L.off_csr_tmp = take(n_entries * 4);
    L.off_vstart = take(((size_t)n_images + 1) * 4);
    L.off_va = take((n_entries + 1) * 4);
    L.off_vb = take((n_entries + 1) * 4);
    L.total = o;
    return L;
}

}  // namespace pnp

using namespace pnp;

// The build addresses the hash tables of all images as one int32 slot index (img * capacity + h in lattice_embed_kernel and
// lattice_neighbors_kernel), and numbers entries with int32 ids below the 0x7f7f7f7f fill of `first`.
static bool lattice_shape_ok(int d, int n_images, int n_pixels) {
    if ((d != 2 && d != 5) || n_images < 1 || n_pixels < 1) return false;
    if ((size_t)n_images * n_pixels * (d + 1) >= 0x7f000000ull) return false;
    return (unsigned long long)n_images * table_capacity(d, n_pixels) <= 0x7fffffffull;
}

extern "C" size_t pnp_lattice_storage_bytes(int d, int n_images, int n_pixels) {
    if (!lattice_shape_ok(d, n_images, n_pixels)) return 0;
    const size_t n_entries = (size_t)n_images * n_pixels * (d + 1);
    size_t o = 0;
    o += align_up(n_entries * 4, 256);                        // offset
    o += align_up(n_entries * 4, 256);                        // bary
    o += align_up((size_t)(d + 1) * n_entries * 2 * 4, 256);  // nbr
    o += align_up((n_entries + 1) * 4, 256);                  // row_ptr
    o += align_up(n_entries * 4, 256);                        // csr_pix
    o += align_up(n_entries * 4, 256);                        // csr_w
    o += align_up(n_entries * 4, 256);                        // csr_norm
    o += align_up((size_t)n_images * n_pixels * 4, 256);      // norm
    o += 256;                                                 // counters
    return o;
}

extern "C" size_t pnp_lattice_build_workspace_bytes(int d, int n_images, int n_pixels) {
    if (!lattice_shape_ok(d, n_images, n_pixels)) return 0;
    return build_layout(d, n_images, n_pixels).total;
}

extern "C" int pnp_lattice_init(pnp_lattice *lat, void *storage, size_t storage_bytes, int d, int n_images, int n_pixels,
                                int shared) {
    if (!lat || !storage || !lattice_shape_ok(d, n_images, n_pixels)) return PNP_ERR_INVALID_ARGUMENT;
    if (shared && n_images != 1) return PNP_ERR_INVALID_ARGUMENT;
    if ((reinterpret_cast<uintptr_t>(storage) & 255) != 0) return PNP_ERR_INVALID_ARGUMENT;
    const size_t n_entries = (size_t)n_images * n_pixels * (d + 1);
    if (storage_bytes < pnp_lattice_storage_bytes(d, n_images, n_pixels)) return PNP_ERR_WORKSPACE;
    char *p = reinterpret_cast<char *>(storage);
    auto take = [&](size_t bytes) { char *r = p; p += align_up(bytes, 256); return r; };
    lat->d = d;
    lat->n_images = n_images;
    lat->n_pixels = n_pixels;
    lat->shared = shared ? 1 : 0;
    lat->n_vertices = -1;
    lat->max_row = -1;
    lat->vertex_stride = (int)n_entries;
    lat->width = 0;
    lat->offset = reinterpret_cast<int32_t *>(take(n_entries * 4));
    lat->bary = reinterpret_cast<float *>(take(n_entries * 4));
    lat->nbr = reinterpret_cast<int32_t *>(take((size_t)(d + 1) * n_entries * 2 * 4));
    lat->row_ptr = reinterpret_cast<int32_t *>(take((n_entries + 1) * 4));
    lat->csr_pix = reinterpret_cast<int32_t *>(take(n_entries * 4));
    lat->csr_w = reinterpret_cast<float *>(take(n_entries * 4));
    lat->csr_norm = reinterpret_cast<float *>(take(n_entries * 4));
    lat->norm = reinterpret_cast<float *>(take((size_t)n_images * n_pixels * 4));
    lat->counters = reinterpret_cast<int32_t *>(take(256));
    return PNP_OK;
}

template <int D>
static int build_impl(pnp_lattice *lat, const uint8_t *rgb, int H, int W, float sx, float sy, float sr, float sg, float sb,
                      char *ws, cudaStream_t st) {
    const int N = lat->n_pixels;
    const long long n_lp = (long long)lat->n_images * N;
    const long long n_entries = n_lp * (D + 1);
    const BuildLayout L = build_layout(D, lat->n_images, N);
    const unsigned cap = (unsigned)table_capacity(D, N);  // n_images * cap <= INT32_MAX (lattice_shape_ok)
    const size_t slots = (size_t)lat->n_images * cap;
    auto *table = reinterpret_cast<unsigned long long *>(ws + L.off_table);
    auto *first = reinterpret_cast<int32_t *>(ws + L.off_first);
    auto *slot_id = reinterpret_cast<int32_t *>(ws + L.off_slot_id);
    auto *keys_dense = reinterpret_cast<unsigned long long *>(ws + L.off_keys);
    auto *prefix = reinterpret_cast<int32_t *>(ws + L.off_prefix);
    auto *block_sums = reinterpret_cast<int32_t *>(ws + L.off_block_sums);
    auto *row_cnt = reinterpret_cast<int32_t *>(ws + L.off_row_cnt);
    auto *csr_tmp = reinterpret_cast<int32_t *>(ws + L.off_csr_tmp);
    auto *vstart = reinterpret_cast<int32_t *>(ws + L.off_vstart);
    auto *va = reinterpret_cast<float *>(ws + L.off_va);
    auto *vb = reinterpret_cast<float *>(ws + L.off_vb);

    cudaError_t e;
    const bool timed = prof::on(kLatticeBuild, st);
    if (timed) prof::begin(kLatticeBuild, st);
    if ((e = cudaMemsetAsync(table, 0xFF, slots * 8, st)) != cudaSuccess) return cuda_err(e);
    if ((e = cudaMemsetAsync(first, 0x7F, slots * 4, st)) != cudaSuccess) return cuda_err(e);
    if ((e = cudaMemsetAsync(lat->counters, 0, 256, st)) != cudaSuccess) return cuda_err(e);
    if ((e = cudaMemsetAsync(row_cnt, 0, (size_t)(n_entries + 1) * 4, st)) != cudaSuccess) return cuda_err(e);

    EmbedParams prm;
    prm.rgb = rgb;
    prm.W = W;
    prm.N = N;
    prm.n_lp = n_lp;
    prm.sx = sx; prm.sy = sy; prm.sr = sr; prm.sg = sg; prm.sb = sb;
    // Permutohedral::init: scale_factor[i] = 1/sqrt((i+2)(i+1)) * (float)(sqrt(2/3) * (d+1))
    const float inv_std_dev = (float)(sqrt(2.0 / 3.0) * (D + 1));
    for (int i = 0; i < 5; ++i) prm.scale_factor[i] = (i < D) ? (float)(1.0 / sqrt((double)((i + 2) * (i + 1))) * inv_std_dev) : 0.f;
    prm.cap_mask = cap - 1;

    const int big_grid = (int)std::min<long long>((n_entries + 255) / 256, (long long)kNumSMs * 32);
    lattice_embed_kernel<D><<<ceil_div(n_lp, 256), 256, 0, st>>>(prm, table, first, lat->offset, lat->bary, lat->counters);
    lattice_flag_kernel<<<big_grid, 256, 0, st>>>(lat->offset, first, prefix, n_entries);
    int rc = exclusive_scan(prefix, prefix, block_sums, n_entries, lat->counters + 0, st);
    if (rc != PNP_OK) return rc;
    lattice_assign_kernel<<<big_grid, 256, 0, st>>>(lat->offset, first, prefix, table, slot_id, keys_dense, n_entries);
    lattice_vstart_kernel<<<ceil_div(lat->n_images + 1, 256), 256, 0, st>>>(prefix, lat->counters, vstart, lat->n_images,
                                                                            (long long)N * (D + 1));
    lattice_offsets_kernel<<<big_grid, 256, 0, st>>>(lat->offset, slot_id, row_cnt, n_entries);
    // row_ptr = exclusive scan of the per-vertex counts (zeros past M keep row_ptr[M..] = n_entries)
    rc = exclusive_scan(row_cnt, lat->row_ptr, block_sums, n_entries + 1, nullptr, st);
    if (rc != PNP_OK) return rc;
    if ((e = cudaMemsetAsync(row_cnt, 0, (size_t)(n_entries + 1) * 4, st)) != cudaSuccess) return cuda_err(e);
    csr_fill_kernel<<<big_grid, 256, 0, st>>>(lat->offset, lat->row_ptr, row_cnt, csr_tmp, n_entries);
    // rows longer than kShortRow are rare (flat-coloured regions); prefix (free again) holds their compact list
    csr_sort_short_kernel<<<big_grid, 256, 0, st>>>(lat->row_ptr, csr_tmp, lat->bary, lat->csr_pix, lat->csr_w, lat->counters,
                                                    prefix, D + 1);
    csr_sort_long_kernel<<<kNumSMs * 8, 256, 0, st>>>(lat->row_ptr, csr_tmp, lat->bary, lat->csr_pix, lat->csr_w, lat->counters,
                                                      prefix, D + 1);
    lattice_neighbors_kernel<D><<<big_grid, 256, 0, st>>>(keys_dense, table, slot_id, vstart, lat->counters, lat->nbr,
                                                          lat->n_images, cap - 1, lat->vertex_stride);
    // normalisation: K applied to ones
    norm_splat_kernel<<<big_grid, 256, 0, st>>>(lat->row_ptr, lat->csr_w, lat->counters, va);
    float *src = va, *dst = vb;
    for (int j = 0; j <= D; ++j) {
        norm_blur_kernel<<<big_grid, 256, 0, st>>>(src, dst, lat->nbr + (size_t)j * lat->vertex_stride * 2, lat->counters);
        std::swap(src, dst);
    }
    const float alpha = 1.0f / (1 + powf(2, -D));
    norm_slice_kernel<<<(int)std::min<long long>((n_lp + 255) / 256, (long long)kNumSMs * 32), 256, 0, st>>>(
        src, lat->offset, lat->bary, lat->norm, n_lp, D + 1, alpha);
    csr_norm_fill_kernel<<<big_grid, 256, 0, st>>>(lat->csr_pix, lat->norm, lat->csr_norm, n_entries);
    if (timed) prof::end(kLatticeBuild, st);
    return launch_status();
}

extern "C" int pnp_lattice_build(pnp_lattice *lat, const uint8_t *rgb, int H, int W, float sx, float sy, float sr, float sg,
                                 float sb, void *workspace, size_t workspace_bytes, pnp_stream_t stream) {
    if (!lat || !workspace || H < 1 || W < 1 || (long long)H * W != lat->n_pixels) return PNP_ERR_INVALID_ARGUMENT;
    if (!(sx > 0.f) || !(sy > 0.f)) return PNP_ERR_INVALID_ARGUMENT;
    if ((lat->d == 5) != (rgb != nullptr)) return PNP_ERR_INVALID_ARGUMENT;
    if (lat->d == 5 && (!(sr > 0.f) || !(sg > 0.f) || !(sb > 0.f))) return PNP_ERR_INVALID_ARGUMENT;
    const size_t need = pnp_lattice_build_workspace_bytes(lat->d, lat->n_images, lat->n_pixels);
    if (need == 0) return PNP_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < need) return PNP_ERR_WORKSPACE;
    if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return PNP_ERR_INVALID_ARGUMENT;
    char *ws = reinterpret_cast<char *>(workspace);
    lat->width = W;
    if (lat->d == 2) return build_impl<2>(lat, rgb, H, W, sx, sy, sr, sg, sb, ws, as_stream(stream));
    return build_impl<5>(lat, rgb, H, W, sx, sy, sr, sg, sb, ws, as_stream(stream));
}

extern "C" int pnp_lattice_finish(pnp_lattice *lat, pnp_stream_t stream) {
    if (!lat || !lat->counters) return PNP_ERR_INVALID_ARGUMENT;
    int32_t host[8];
    cudaError_t e = cudaMemcpyAsync(host, lat->counters, sizeof(host), cudaMemcpyDeviceToHost, as_stream(stream));
    if (e != cudaSuccess) return cuda_err(e);
    e = cudaStreamSynchronize(as_stream(stream));
    if (e != cudaSuccess) return cuda_err(e);
    lat->n_vertices = host[0];
    lat->max_row = host[2];
    if (host[1] != 0) return PNP_ERR_INVALID_ARGUMENT;
    return PNP_OK;
}
