// attention.cu -- ViT self-attention softmax(Q K^T / sqrt(d)) V at fp32-grade accuracy on the 5th-generation tensor cores (tcgen05.mma,
// accumulators in tensor memory); VIT:93-119, the attention of every encoder block (SURVEY 8f.1: the model pass).
//
// Same idea as the 3xFP16 GEMM operands (tf32x3.cu): every fp32 operand is split exactly into x = h + l 2^-11 (h = fp16(x),
// l = fp16((x - h) 2^11)) and each product a b is evaluated as  a_h b_h + 2^-11 (a_l b_h + a_h b_l)  with fp32 accumulation, the main
// term and the two corrections in separate accumulators (the tensor core adds with truncation: the 2^-11-sized corrections must not
// sit in the main chain).  That holds for both contractions: S = Q K^T and O = P V, with the probabilities P split the same way after
// the fp32 online softmax in the exp2 domain.
// Two passes.  (1) attention_split_kernel: k and v are split once per (image, head) into fp16 (hi, lo) pairs in a workspace.
// (2) attention_tc5_kernel, flash-attention structure: nothing of size L x L touches HBM.  HBM traffic: q, k, v read once, the k / v
// splits written once and read once (K/V tiles hit in L2 across the query tiles of a head), O written once.
//
// One CTA = 128 query rows of one (image, head) = the 128 lanes of tensor memory; thread t owns row t.  Keys stream in tiles of 64.
// Per tile:  S = Q K^T   : 8 tcgen05.mma (M 128, K 16) from shared memory: Q_h [K_h; K_l] as one N = 128 MMA per k-step into TMEM
//                          columns [0,64) main, [64,128) corr, then Q_l K_h onto corr
//            softmax     : every thread reads its row of S with tcgen05.ld, p = exp2(s - m), writes P as fp16 (hi, lo) to shared memory
//            O += P V    : 8 tcgen05.mma likewise (P_h [V_h | V_l], P_l V_h) into TMEM columns [128,192) main, [192,256) corr; O stays
//                          in tensor memory over all key tiles and is rescaled there only when a row's maximum grows by more than 2^8
// Operands sit in shared memory in the un-swizzled canonical core-matrix layouts (8 rows x 16 bytes = 128 contiguous bytes):
// Q, K and P K-major; V MN-major, i.e. its row-major [key][dim] 16-byte pieces are only re-tiled, never transposed.
// 256 TMEM columns and 112 KB of shared memory per CTA: two CTAs per SM, one's softmax under the other's MMAs.
// Inside a CTA the tensor pipe runs ahead of the threads: S_{j+1} is issued as soon as every thread has read S_j (K tiles are
// double-buffered), and O_{j-1} is waited for one tile late, so neither MMA group is waited for right after its issue.
// K and V tiles are copied from the split workspace with cp.async as soon as the MMAs reading the buffer they replace have committed.
#include <cuda_fp16.h>
#include <math.h>

#include "common.cuh"

namespace pnp {

constexpr int kAttD = 64;          // head dimension (ViT-L/16: 1024 / 16)
constexpr int kAttTile = 64;       // keys per tile of the main kernel: the workspace rows are padded to a multiple of it

// (x0, x1) -> packed half2 of the hi parts and of the 2^11-scaled lo parts (packed cvt.rn.f16x2.f32 conversions)
__device__ __forceinline__ void split2(float x0, float x1, unsigned &hi, unsigned &lo) {
    const __half2 hh = __floats2half2_rn(x0, x1);
    const float2 hf = __half22float2(hh);
    const __half2 ll = __floats2half2_rn((x0 - hf.x) * 2048.0f, (x1 - hf.y) * 2048.0f);
    hi = *reinterpret_cast<const unsigned *>(&hh);
    lo = *reinterpret_cast<const unsigned *>(&ll);
}

// ---- pass 1: fp32 k, v -> fp16 (hi, lo) pairs, four [B, H, Lp, 64] planes k_hi, k_lo, v_hi, v_lo with Lp = L rounded up to the
// tile (rows past L zero).  k and v are multiplied by in_scale (a power of two: exact); q is split by the main kernel.
// Done once per (image, head) instead of once per query tile inside the main kernel (4 query tiles share every K/V tile at L = 442).
__global__ void __launch_bounds__(256) attention_split_kernel(const float *__restrict__ qkv, __half *__restrict__ ws, int L, int Lp, int H,
                                                              int B, float in_scale, int *__restrict__ flag) {
    // grid = (Lp, B): one CTA per token row; its k and v parts are 2 x H x 64 contiguous floats of qkv.  No per-item divisions.
    const size_t plane = (size_t)B * H * Lp * kAttD;                 // one [B,H,Lp,64] fp16 array
    const int l = blockIdx.x, b = blockIdx.y;
    const int per_which = H * (kAttD / 4);                           // float4 pieces of the k (or v) part of one row
    bool bad = false;
    for (int i = threadIdx.x; i < 2 * per_which; i += blockDim.x) {
        const int which = i >= per_which, j = i - which * per_which;   // 0 k, 1 v
        const int h = j >> 4, c4 = (j & 15) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (l < L) v = ldg_stream4(qkv + (((size_t)b * L + l) * 3 + 1 + which) * H * kAttD + 4 * j);
        v.x *= in_scale; v.y *= in_scale; v.z *= in_scale; v.w *= in_scale;
        bad = bad || !(fabsf(v.x) <= 65504.f && fabsf(v.y) <= 65504.f && fabsf(v.z) <= 65504.f && fabsf(v.w) <= 65504.f);
        unsigned h01, l01, h23, l23;
        split2(v.x, v.y, h01, l01);
        split2(v.z, v.w, h23, l23);
        const size_t o = (((size_t)b * H + h) * Lp + l) * kAttD + c4;
        *reinterpret_cast<uint2 *>(ws + (size_t)(2 * which) * plane + o) = make_uint2(h01, h23);
        *reinterpret_cast<uint2 *>(ws + (size_t)(2 * which + 1) * plane + o) = make_uint2(l01, l23);
    }
    if (bad && flag) *flag = 1;
}

namespace tc5 {

constexpr int BM = 128;            // query rows per CTA = TMEM lanes
constexpr int BN = 64;             // keys per tile
constexpr int D = 64;              // head dimension
constexpr int NS = 256;            // softmax threads: two per query row
constexpr int NT = NS + 32;        // + the warp whose lane 0 issues every tcgen05.mma
constexpr int HC = 32;             // columns (keys of S, dims of O) per thread
constexpr uint32_t LBO = 128;      // bytes between core matrices along K (adjacent)
constexpr uint32_t SBO = 1024;     // bytes between 8-row groups along M/N (8 K-chunks of a 64-wide tile)
constexpr uint32_t OFF_QH = 0, OFF_QL = 16384, OFF_K = 32768 /* 2 stages x (hi 8 KB, lo 8 KB) */, OFF_VH = 65536, OFF_VL = 73728,
                   OFF_PH = 81920, OFF_PL = 98304, OFF_BAR = 114688, OFF_XCH = OFF_BAR + 64, SMEM_BYTES = OFF_XCH + 512;
static_assert(2 * (SMEM_BYTES + 1024) <= 233472, "two CTAs per SM");
constexpr uint32_t TM_S_MAIN = 0, TM_S_CORR = 64, TM_O_MAIN = 128, TM_O_CORR = 192, TM_COLS = 256;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor, no swizzle: start >> 4 | LBO >> 4 at 16 | SBO >> 4 at 32 | version 1 at 46
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(LBO >> 4) << 16) | ((uint64_t)(SBO >> 4) << 32) | (1ull << 46);
}
// instruction descriptor, kind::f16: D fp32 (bit 4), A/B fp16, A K-major, B major at bit 16, N >> 3 at 17, M >> 4 at 24
constexpr uint32_t kIdescS = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
constexpr uint32_t kIdescS2 = (1u << 4) | ((uint32_t)(2 * BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);             // N = 128: hi and lo stacked
constexpr uint32_t kIdescO2 = (1u << 4) | (1u << 16) | ((uint32_t)(2 * D >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
static_assert(TM_S_CORR == TM_S_MAIN + BN && TM_O_CORR == TM_O_MAIN + D && OFF_VL == OFF_VH + 8192, "stacked-N MMAs need adjacent halves");
constexpr uint32_t kIdescO = (1u << 4) | (1u << 16) | ((uint32_t)(D >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
                 "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
                 : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (int spin = 0; spin < (1 << 26); ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done)
                     : "r"(bar), "r"(parity)
                     : "memory");
        if (done) return;
    }
    __trap();   // an MMA group that never commits is a bug: fail the launch instead of hanging the GPU
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void st_shared8(uint32_t addr, unsigned a, unsigned b) {
    asm volatile("st.shared.v2.b32 [%0], {%1,%2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}

__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void *gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait0() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void st_shared16(uint32_t addr, unsigned a, unsigned b, unsigned c, unsigned d) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// 16 consecutive 32-bit columns of this thread's TMEM lane, store
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%16], {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15};" ::"r"(__float_as_uint(v[0])),
                 "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
                 "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])),
                 "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])),
                 "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])), "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

constexpr float kRescaleThreshold = 8.0f;   // O and l are rescaled only when a row's maximum has grown by more than 2^8 (exp2 domain)

// ws: the workspace of attention_split_kernel, [4][B,H,Lp,64] fp16 planes (k_hi, k_lo, v_hi, v_lo), Lp a multiple of 64.
// 288 threads.  Warps 0-7 (softmax): thread t works on query row t & 127 (TMEM lane) and on the column half t >> 7 of S (keys) and
// of O (dims); the two threads of a row exchange their partial row maximum through shared memory once per tile and their row sums
// once at the end; they also copy the K / V tiles (cp.async).  Warp 8: lane 0 issues every tcgen05.mma (an issue blocks for ~100
// cycles per MMA -- measured, profiles/experiments/probe_umma_timing.cu -- so it must not sit in a softmax thread's instruction stream).
// O accumulates in tensor memory over all key tiles (the MMAs of tile j add to it).  The softmax subtracts a reference m_used that is
// refreshed -- and O, l rescaled through tcgen05.ld / tcgen05.st -- only when the row maximum has outgrown it by more than 2^8: p stays
// below 256, which fp16 (hi, lo) pairs hold as exactly as values below 1, and the result is the same softmax (any common shift is).
// Hand-offs are mbarriers only: s_full / o_full (tcgen05.commit: an MMA group has finished), s_free (all 256 softmax threads have
// read S_j), p_full (all 256 have written their part of P_j, finished any rescale of O and seen their copies land).
__global__ void __launch_bounds__(NT, 2) attention_tc5_kernel(const float *__restrict__ qkv, const __half *__restrict__ ws,
                                                              float *__restrict__ out, __half *__restrict__ out3, int L, int Lp, int H, int B,
                                                              float q_scale, float hi_scale, int *__restrict__ flag) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * BM;
    const uint32_t bar_s = sbase + OFF_BAR, bar_o = sbase + OFF_BAR + 8, bar_s_free = sbase + OFF_BAR + 16, bar_p_full = sbase + OFF_BAR + 24;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + OFF_BAR + 32);
    const int n_tiles = Lp / BN;

    if (t == 0) {
        mbar_init(bar_s, 1);
        mbar_init(bar_o, 1);
        mbar_init(bar_s_free, NS);
        mbar_init(bar_p_full, NS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == NS / 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }

    if (warp == NS / 32) {
        // ================================================================ MMA warp: lane 0 issues, the others wait at the end
        tc_fence_before();
        __syncthreads();                 // Q, K_0, K_1, V_0 are staged, TMEM is allocated, the barriers are initialised
        tc_fence_after();
        const uint32_t tmem = *tmem_slot;
        if (lane == 0) {
            // descriptors of the first k-step of every operand; k-step s is 256 bytes further: + 16 in the start-address field
            const uint64_t d_qh = make_desc(sbase + OFF_QH), d_ql = make_desc(sbase + OFF_QL), d_ph = make_desc(sbase + OFF_PH),
                           d_pl = make_desc(sbase + OFF_PL), d_vh = make_desc(sbase + OFF_VH), d_k0 = make_desc(sbase + OFF_K);
            auto issue_s = [&](int tile) {   // S = Q K_tile^T : main = Qh Kh, corr = Ql Kh + Qh Kl
                const uint64_t d_kh = d_k0 + (uint64_t)((tile & 1) * (16384 >> 4));
                // B = [Kh ; Kl] stacked along N (the lo stage follows the hi stage: 8 more 8-row groups at the same SBO): one N = 128
                // MMA per k-step gives Qh Kh in columns [0,64) and Qh Kl in [64,128); Ql Kh is added to the second half.  An MMA
                // costs ~100 cycles for N = 64 and N = 128 alike: 8 MMAs, not 12.
#pragma unroll
                for (int s = 0; s < D / 16; ++s) umma(tmem + TM_S_MAIN, d_qh + 16 * s, d_kh + 16 * s, kIdescS2, s > 0);
#pragma unroll
                for (int s = 0; s < D / 16; ++s) umma(tmem + TM_S_CORR, d_ql + 16 * s, d_kh + 16 * s, kIdescS, 1);
                umma_commit(bar_s);
            };
            issue_s(0);
            for (int j = 0; j < n_tiles; ++j) {
                const uint32_t par = (uint32_t)(j & 1);
                if (j + 1 < n_tiles) {       // S_{j+1} once all 256 have read S_j (K_{j+1} landed before they arrived at p_full(j-1))
                    mbar_wait(bar_s_free, par);
                    tc_fence_after();
                    issue_s(j + 1);
                }
                mbar_wait(bar_p_full, par);  // P_j and V_j are in shared memory, O has been rescaled where it had to be
                tc_fence_after();
#pragma unroll
                for (int s2 = 0; s2 < BN / 16; ++s2) umma(tmem + TM_O_MAIN, d_ph + 16 * s2, d_vh + 16 * s2, kIdescO2, (j | s2) > 0);   // B = [Vh | Vl]
#pragma unroll
                for (int s2 = 0; s2 < BN / 16; ++s2) umma(tmem + TM_O_CORR, d_pl + 16 * s2, d_vh + 16 * s2, kIdescO, 1);
                umma_commit(bar_o);
            }
        }
        __syncwarp();
        tc_fence_before();
        __syncthreads();                 // the softmax warps have read the final O (which also means: every MMA has completed)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TM_COLS) : "memory");
        return;
    }

    // ==================================================================== softmax warps
    const int row = t & (BM - 1), hh = t >> 7;            // TMEM lane / column half
    // [256] partial row maxima, rounded up to bf16: both threads of a row must subtract the SAME bound, and any bound >= the
    // maximum is exact for a softmax; 16 bits keep two CTAs per SM inside the 228 KB
    unsigned short *xch = reinterpret_cast<unsigned short *>(smem + OFF_XCH);
    float *xch_l = reinterpret_cast<float *>(smem + OFF_K);   // [256] row sums (after the last S group the K stages are free)

    // ---- K / V tile copies: 512 16-byte pieces per array, 2 per thread; piece (key, c = dim / 8)
    const size_t plane = (size_t)B * H * Lp * D;
    const __half *head = ws + ((size_t)b * H + h) * Lp * D;
    auto load_k = [&](int tile) {   // into stage tile & 1
        const uint32_t stage = sbase + OFF_K + (uint32_t)(tile & 1) * 16384;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int idx = t + NS * i, key = idx >> 3, c = idx & 7;
            const uint32_t dst = (uint32_t)(key >> 3) * SBO + (uint32_t)c * LBO + (uint32_t)(key & 7) * 16;   // K-major: rows = keys
            const __half *src = head + (size_t)(tile * BN + key) * D + c * 8;
            cp_async16(stage + dst, src);
            cp_async16(stage + 8192 + dst, src + plane);
        }
    };
    auto load_v = [&](int tile) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int idx = t + NS * i, key = idx >> 3, c = idx & 7;
            const uint32_t dst = (uint32_t)c * SBO + (uint32_t)(key >> 3) * LBO + (uint32_t)(key & 7) * 16;   // MN-major: 8 dims contiguous
            const __half *src = head + 2 * plane + (size_t)(tile * BN + key) * D + c * 8;   // planes v_hi, v_lo
            cp_async16(sbase + OFF_VH + dst, src);
            cp_async16(sbase + OFF_VL + dst, src + plane);
        }
    };
    load_k(0);
    if (n_tiles > 1) load_k(1);
    load_v(0);
    cp_async_commit();

    // ---- the CTA's 128 query rows, pre-multiplied by in_scale * softmax_scale * log2(e), as K-major (hi, lo) rows; 16 threads read
    // one row's 256 bytes (coalesced); all eight loads of a thread are in flight before the first conversion
    bool q_bad = false;   // a scaled q value outside fp16's range (or NaN): its hi part would be inf
    {
        const float *qb = qkv + (size_t)b * L * (size_t)(3 * H * D) + (size_t)h * D;
        float4 a[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int idx = t + NS * i, r = idx >> 4, f = idx & 15;
            a[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (q0 + r < L) a[i] = __ldg(reinterpret_cast<const float4 *>(qb + (size_t)(q0 + r) * (size_t)(3 * H * D) + 4 * f));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int idx = t + NS * i, r = idx >> 4, f = idx & 15;
            const float x0 = a[i].x * q_scale, x1 = a[i].y * q_scale, x2 = a[i].z * q_scale, x3 = a[i].w * q_scale;
            q_bad = q_bad || !(fabsf(x0) <= 65504.f && fabsf(x1) <= 65504.f && fabsf(x2) <= 65504.f && fabsf(x3) <= 65504.f);
            unsigned h0, h1, l0, l1;
            split2(x0, x1, h0, l0);
            split2(x2, x3, h1, l1);
            const uint32_t off = (uint32_t)(r >> 3) * SBO + (uint32_t)(f >> 1) * LBO + (uint32_t)(r & 7) * 16 + (uint32_t)(f & 1) * 8;
            st_shared8(sbase + OFF_QH + off, h0, h1);
            st_shared8(sbase + OFF_QL + off, l0, l1);
        }
    }
    cp_async_wait0();
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(hh * HC);

    float m_used = -INFINITY, l = 0.f;
    const uint32_t p_row = (uint32_t)(row >> 3) * SBO + (uint32_t)(row & 7) * 16 + (uint32_t)(hh * (HC / 8)) * LBO;

    for (int j = 0; j < n_tiles; ++j) {
        const int k0 = j * BN + hh * HC;     // first key of this thread's half of the tile
        // ---- S_j is ready (issued one tile ago); its K stage is free for tile j + 2
        mbar_wait(bar_s, (uint32_t)(j & 1));
        tc_fence_after();
        if (j + 2 < n_tiles) load_k(j + 2);
        float s[HC];
        {
            float a0[16], c0[16], a1[16], c1[16];
            tmem_ld16(lane_addr + TM_S_MAIN, a0);
            tmem_ld16(lane_addr + TM_S_CORR, c0);
            tmem_ld16(lane_addr + TM_S_MAIN + 16, a1);
            tmem_ld16(lane_addr + TM_S_CORR + 16, c1);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                s[i] = fmaf(c0[i], 1.0f / 2048.0f, a0[i]);
                s[16 + i] = fmaf(c1[i], 1.0f / 2048.0f, a1[i]);
            }
        }
        if (k0 + HC > L) {   // only the last tile holds keys past L
#pragma unroll
            for (int i = 0; i < HC; ++i)
                if (k0 + i >= L) s[i] = -INFINITY;
        }
        float mx = s[0];
#pragma unroll
        for (int i = 1; i < HC; ++i) mx = fmaxf(mx, s[i]);
        {
            const unsigned u = __float_as_uint(mx);
            const unsigned up = (u & 0x80000000u) ? (u & 0xFFFF0000u) : ((u + 0xFFFFu) & 0xFFFF0000u);   // towards +inf
            mx = __uint_as_float(up);
            xch[t] = (unsigned short)(up >> 16);
        }
        // the two warps that share these 32 rows meet at a named barrier (ids 1..4, 64 threads) and read each other's bound
        asm volatile("bar.sync %0, 64;" ::"r"(1 + (warp & 3)) : "memory");
        mx = fmaxf(mx, __uint_as_float((unsigned)xch[t ^ BM] << 16));
        // ---- this thread is done with S_j (and with its partner's xch slot: the slot is rewritten only after S_{j+1} has been
        // committed, which needs this arrival).  The tensor pipe starts on S_{j+1} once all 256 have arrived.
        tc_fence_before();
        mbar_arrive(bar_s_free);

        // ---- P V_{j-1} has committed: the P and V buffers are free, and O may be rescaled
        if (j > 0) {
            mbar_wait(bar_o, (uint32_t)((j - 1) & 1));
            tc_fence_after();
            load_v(j);
        }
        cp_async_commit();
        // a row whose maximum has outgrown its reference by more than 2^8 gets a new reference; O (in TMEM) and l follow.  Both
        // threads of a row see the same mx and take the same decision for their column halves; the branch is uniform per warp
        // because tcgen05.ld / st are warp-wide.  Tile 0 only sets the reference (O is still empty).
        const bool grow = mx > m_used + kRescaleThreshold;   // also true on tile 0 (m_used = -inf)
        if (j > 0 && __any_sync(0xffffffffu, grow)) {
            const float alpha = grow ? ex2_approx(m_used - mx) : 1.0f;
#pragma unroll
            for (int c0 = 0; c0 < HC; c0 += 16) {
                float a[16], cr[16];
                tmem_ld16(lane_addr + TM_O_MAIN + c0, a);
                tmem_ld16(lane_addr + TM_O_CORR + c0, cr);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) { a[i] *= alpha; cr[i] *= alpha; }
                tmem_st16(lane_addr + TM_O_MAIN + c0, a);
                tmem_st16(lane_addr + TM_O_CORR + c0, cr);
            }
            tmem_st_wait();
            l *= alpha;
        }
        if (grow) m_used = mx;

        // ---- p = exp2(s - m_used) as fp16 (hi, lo) pairs, K-major rows of P
        float sum = 0.f;
#pragma unroll
        for (int c = 0; c < HC / 8; ++c) {
            unsigned ph[4], pl[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float p0 = ex2_approx(s[8 * c + 2 * i] - m_used), p1 = ex2_approx(s[8 * c + 2 * i + 1] - m_used);
                sum += p0 + p1;
                split2(p0, p1, ph[i], pl[i]);
            }
            st_shared16(sbase + OFF_PH + p_row + c * LBO, ph[0], ph[1], ph[2], ph[3]);
            st_shared16(sbase + OFF_PL + p_row + c * LBO, pl[0], pl[1], pl[2], pl[3]);
        }
        l += sum;

        // ---- P V_j may be issued once all 256 are here
        cp_async_wait0();          // this thread's pieces of V_j (and K_{j+2}) have landed
        fence_async_smem();
        tc_fence_before();
        mbar_arrive(bar_p_full);
    }
    mbar_wait(bar_o, (uint32_t)((n_tiles - 1) & 1));
    tc_fence_after();
    float o[HC];
#pragma unroll
    for (int c0 = 0; c0 < HC; c0 += 16) {
        float a[16], cr[16];
        tmem_ld16(lane_addr + TM_O_MAIN + c0, a);
        tmem_ld16(lane_addr + TM_O_CORR + c0, cr);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) o[c0 + i] = fmaf(cr[i], 1.0f / 2048.0f, a[i]);
    }
    xch_l[t] = l;
    tc_fence_before();
    __syncthreads();

    // ---- normalise; the rows go through shared memory (the V and P buffers are free) so that the global stores are whole
    // 256-byte (fp32) / 128-byte (fp16) row segments.  16-byte pieces are XOR-swizzled by the row: conflict-free both ways.
    const float inv = 1.0f / (l + xch_l[t ^ BM]);
    const int Dm = H * D;
    // The bound both threads of a row subtract is bf16, so it can sit one bf16 ulp above the row maximum: the largest p of the row is
    // then as small as 2^-ulp.  For |m_used| < 2^11 the ulp is at most 8 and p_max >= 2^-8 stays in fp16's normal range; beyond it
    // the (hi, lo) pairs of P lose bits or flush to zero.  m_used only grows; tiles taken under an earlier, coarser bound weigh at
    // most 2^-8 after the rescale that replaced it (2^-2048 if it was below -4096), so the final bound is the one to test.
    bool bad = q_bad || !(fabsf(m_used) < 2048.f);
#pragma unroll
    for (int i = 0; i < HC; ++i) o[i] *= inv;
    const uint32_t stage = sbase + OFF_VH;
    if (out) {
#pragma unroll
        for (int c = 0; c < HC / 4; ++c) {   // fp32 [128][16 pieces]
            const int piece = hh * (HC / 4) + c;
            st_shared16(stage + (uint32_t)row * 256 + (uint32_t)((piece ^ (row & 7)) * 16), __float_as_uint(o[4 * c]), __float_as_uint(o[4 * c + 1]),
                        __float_as_uint(o[4 * c + 2]), __float_as_uint(o[4 * c + 3]));
        }
        asm volatile("bar.sync 5, %0;" ::"n"(NS) : "memory");
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int idx = t + NS * i, r = idx >> 4, piece = idx & 15;
            if (q0 + r < L) {
                const uint4 v = *reinterpret_cast<const uint4 *>(smem + OFF_VH + r * 256 + ((piece ^ (r & 7)) * 16));
                *reinterpret_cast<uint4 *>(out + ((size_t)b * L + q0 + r) * Dm + (size_t)h * D + 4 * piece) = v;
            }
        }
        if (out3) asm volatile("bar.sync 5, %0;" ::"n"(NS) : "memory");
    }
    if (out3) {   // [h * hi_scale | l | h] of the attention output, ready for the projection GEMM: three fp16 [128][8 pieces] arrays
        const __half2 hs2 = __float2half2_rn(hi_scale);
#pragma unroll
        for (int c = 0; c < HC / 8; ++c) {
            unsigned hv[4], lv[4], sc[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float x0 = o[8 * c + 2 * k], x1 = o[8 * c + 2 * k + 1];
                split2(x0, x1, hv[k], lv[k]);
                const __half2 hsv = __hmul2(*reinterpret_cast<__half2 *>(&hv[k]), hs2);   // a power of two: exact
                sc[k] = *reinterpret_cast<const unsigned *>(&hsv);
                bad = bad || !(fabsf(x0 * hi_scale) <= 65504.f && fabsf(x1 * hi_scale) <= 65504.f);
            }
            const int piece = hh * (HC / 8) + c;
            const uint32_t off = (uint32_t)row * 128 + (uint32_t)((piece ^ (row & 7)) * 16);
            st_shared16(stage + off, sc[0], sc[1], sc[2], sc[3]);
            st_shared16(stage + 16384 + off, lv[0], lv[1], lv[2], lv[3]);
            st_shared16(stage + 32768 + off, hv[0], hv[1], hv[2], hv[3]);
        }
        asm volatile("bar.sync 5, %0;" ::"n"(NS) : "memory");
#pragma unroll
        for (int i = 0; i < 12; ++i) {
            const int idx = t + NS * i, arr = idx >> 10, r = (idx >> 3) & (BM - 1), piece = idx & 7;
            if (q0 + r < L) {
                const uint4 v = *reinterpret_cast<const uint4 *>(smem + OFF_VH + arr * 16384 + r * 128 + ((piece ^ (r & 7)) * 16));
                *reinterpret_cast<uint4 *>(out3 + ((size_t)b * L + q0 + r) * 3 * Dm + (size_t)arr * Dm + (size_t)h * D + 8 * piece) = v;
            }
        }
    }
    if (bad && flag) *flag = 1;
}

}  // namespace tc5

}  // namespace pnp

using namespace pnp;

extern "C" size_t pnp_attention_fp16x3_workspace_bytes(int B, int L, int H, int D) {
    if (B < 0 || L < 1 || H < 1 || D != kAttD) return 0;
    const size_t Lp = (size_t)ceil_div(L, kAttTile) * kAttTile;
    return 4 * (size_t)B * H * Lp * kAttD * sizeof(__half);   // k_hi, k_lo, v_hi, v_lo
}

extern "C" int pnp_attention_fp16x3(const float *qkv, float in_scale, float softmax_scale, float *out, uint16_t *out3, float out3_hi_scale,
                                    void *workspace, size_t workspace_bytes, int *overflow_flag, int B, int L, int H, int D,
                                    pnp_stream_t stream) {
    if (!qkv || (!out && !out3) || (out3 && (reinterpret_cast<uintptr_t>(out3) & 3)) || !workspace || B < 0 || L < 1 || H < 1 || D != kAttD || B > 65535 || H > 65535 ||
        (reinterpret_cast<uintptr_t>(qkv) & 15) || (out && (reinterpret_cast<uintptr_t>(out) & 7)) || (reinterpret_cast<uintptr_t>(workspace) & 15) ||
        !(in_scale > 0.f))
        return PNP_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < pnp_attention_fp16x3_workspace_bytes(B, L, H, D)) return PNP_ERR_WORKSPACE;
    if (B == 0) return PNP_OK;
    cudaStream_t st = as_stream(stream);
    const int Lp = ceil_div(L, kAttTile) * kAttTile;
    const cudaError_t e = allow_smem(tc5::attention_tc5_kernel, tc5::SMEM_BYTES);
    if (e != cudaSuccess) return cuda_err(e);
    __half *ws = reinterpret_cast<__half *>(workspace);
    const bool timed = prof::on(kAttention, st);
    if (timed) prof::begin(kAttention, st);
    attention_split_kernel<<<dim3(Lp, B), 256, 0, st>>>(qkv, ws, L, Lp, H, B, in_scale, overflow_flag);
    const float q_scale = in_scale * softmax_scale * 1.4426950408889634f;
    tc5::attention_tc5_kernel<<<dim3(ceil_div(L, tc5::BM), H, B), tc5::NT, tc5::SMEM_BYTES, st>>>(
        qkv, ws, out, reinterpret_cast<__half *>(out3), L, Lp, H, B, q_scale, out3_hi_scale, overflow_flag);
    if (timed) prof::end(kAttention, st);
    return launch_status();
}
