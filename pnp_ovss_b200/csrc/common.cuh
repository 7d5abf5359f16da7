// common.cuh -- shared device/host helpers for libpnp_ovss_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <mutex>
#include <unordered_set>

#include "../../include/pnp_ovss_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libpnp_ovss_b200 is written for sm_100a (B200); compile with -gencode arch=compute_100a,code=sm_100a"
#endif

namespace pnp {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; persistent grids are sized in multiples of this

static inline int cuda_err(cudaError_t e) { return e == cudaSuccess ? PNP_OK : PNP_ERR_CUDA_BASE - (int)e; }
static inline int launch_status() { return cuda_err(cudaGetLastError()); }
static inline cudaStream_t as_stream(pnp_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---- opt-in to more than 48 KB of dynamic shared memory: granted ONCE per kernel, at the device maximum (the attribute only bounds
// what a launch may ask for; it is process-wide state, so setting it per launch to that launch's size races between host threads)
constexpr int kMaxOptinSmemBytes = 232448;   // B200: 227 KB per CTA
inline cudaError_t allow_smem_ptr(const void *kernel) {
    static std::mutex mu;
    static std::unordered_set<const void *> granted;
    std::lock_guard<std::mutex> lock(mu);
    if (granted.count(kernel)) return cudaSuccess;
    cudaFuncAttributes attr;
    cudaError_t e = cudaFuncGetAttributes(&attr, kernel);     // static + dynamic share the 227 KB
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxOptinSmemBytes - (int)attr.sharedSizeBytes);
    if (e == cudaSuccess) granted.insert(kernel);
    return e;
}
template <typename K>
inline cudaError_t allow_smem(K kernel, size_t bytes) {
    if (bytes > (size_t)kMaxOptinSmemBytes) return cudaErrorInvalidValue;
    return allow_smem_ptr(reinterpret_cast<const void *>(kernel));
}

// ---- streaming 128-bit global accesses (read-once / write-once data: keep L1 clean) ----
__device__ __forceinline__ float4 ldg_stream4(const float *p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream4(float *p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

// ---- warp reductions ----
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- order-preserving float <-> uint32 keys for atomicMin/atomicMax; NaN is sticky ----
// A NaN is stored as the largest key on the max side and as the smallest on the min side:
// key 0xffffffff decodes to u = 0x7fffffff (NaN); key 0 decodes to u = 0xffffffff (NaN): both stay NaN.
__device__ __forceinline__ unsigned f2key(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(unsigned k) {
    unsigned u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(u);
}

// min/max that propagate NaN like torch.min/max and numpy
__device__ __forceinline__ float nan_min(float a, float b) { return (a != a || b != b) ? __int_as_float(0x7fc00000) : fminf(a, b); }
__device__ __forceinline__ float nan_max(float a, float b) { return (a != a || b != b) ? __int_as_float(0x7fc00000) : fmaxf(a, b); }


// ---- optional in-situ kernel timing (pnp_profile_*): bench.py brackets the launches of selected kernel classes
// with CUDA events on their own stream, inside the timed region.  Off (mask 0) it costs one predictable branch.
enum KernelId {
    kSoftmaxFwd = 1, kSoftmaxBwdGradcam = 2, kTokenMerge = 3, kDropoutRound = 4, kThresholdPrep = 5, kUpsampleWrite = 6,
    kBlurVertical = 7, kBlurHorizontal = 8, kBlurNormalize = 9, kLatticeBuild = 10, kCrfUnary = 11, kSplatBilateral = 12,
    kBlurAxisBilateral = 13, kMeanfieldUpdate = 14, kArgmax = 15, kConfusion = 16, kSplatSpatial = 17, kBlurAxisSpatial = 18,
    kTf32Split = 19, kGeluSplit = 20, kLayernormSplit = 21, kLowrankBlur = 22, kLowrankUnary = 23, kBackgroundBlur = 24,
    kAttention = 25, kNumKernelIds = 26
};
namespace prof {
extern unsigned g_mask;
extern bool g_filter;           // when set, only launches on g_filter_stream are timed
extern cudaStream_t g_filter_stream;
void begin(int id, cudaStream_t st);
void end(int id, cudaStream_t st);
static inline bool on(int id, cudaStream_t st) { return (g_mask & (1u << id)) && (!g_filter || st == g_filter_stream); }
}  // namespace prof
#define PNP_LAUNCH(id, st, ...)                         \
    do {                                                \
        if (pnp::prof::on((id), (st))) {                \
            pnp::prof::begin((id), (st));               \
            __VA_ARGS__;                                \
            pnp::prof::end((id), (st));                 \
        } else {                                        \
            __VA_ARGS__;                                \
        }                                               \
    } while (0)

}  // namespace pnp
