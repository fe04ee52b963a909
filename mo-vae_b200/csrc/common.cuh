// Shared host/device helpers for the movae_b200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <type_traits>

#include "../../include/movae_b200.h"

namespace movae {

// thread-local error text returned by movae_last_error()
void set_error(const char* fmt, ...);
int fail_cuda(cudaError_t e, const char* what);   // formats "CUDA error ..." and returns MOVAE_ERR_CUDA
int sm_count();                                    // cached multiProcessorCount of the current device (0 on failure)

#define MOVAE_CUDA_TRY(expr)                                        \
    do {                                                            \
        cudaError_t _e = (expr);                                    \
        if (_e != cudaSuccess) return ::movae::fail_cuda(_e, #expr); \
    } while (0)

#define MOVAE_REQUIRE(cond, code, ...)          \
    do {                                        \
        if (!(cond)) {                          \
            ::movae::set_error(__VA_ARGS__);    \
            return (code);                      \
        }                                       \
    } while (0)

// Grid of a persistent launch of `kern` with `threads` threads per CTA: as many CTAs as the device holds at once (SMs x
// occupancy), at most one per tile and at most `cap`.  The occupancy is cached per kernel instantiation, host thread and
// device: a cache keyed on the kernel's type alone would mix up the instantiations that share one.
template <auto kern>
int persistent_grid(int threads, int64_t n_tiles, int64_t cap, unsigned int* grid) {
    static thread_local int occ_dev = -1, occ = 0;
    int dev = 0;
    MOVAE_CUDA_TRY(cudaGetDevice(&dev));
    if (occ_dev != dev) {
        MOVAE_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, 0));
        if (occ < 1) occ = 1;
        occ_dev = dev;
    }
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    int64_t g = (int64_t)sms * occ;
    if (g > n_tiles) g = n_tiles;
    if (g > cap) g = cap;
    *grid = g > 1 ? (unsigned int)g : 1u;
    return MOVAE_OK;
}

// Lets `kern` launch with `bytes` of dynamic shared memory (more than 48 KB needs this opt-in).  The attribute belongs to
// the device current when it is set, so it is set once per kernel instantiation, host thread and device, as above.
template <auto kern>
int allow_dynamic_smem(int bytes) {
    static thread_local int attr_dev = -1;
    int dev = 0;
    MOVAE_CUDA_TRY(cudaGetDevice(&dev));
    if (attr_dev != dev) {
        MOVAE_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        attr_dev = dev;
    }
    return MOVAE_OK;
}

// Returns f(std::integral_constant<int, K>{}) for K = k; k is 1 .. MOVAE_MAX_K (larger k take MOVAE_MAX_K).
template <int K = 1, class F>
int dispatch_k(int k, F&& f) {
    if constexpr (K == MOVAE_MAX_K) return f(std::integral_constant<int, K>{});
    else return k == K ? f(std::integral_constant<int, K>{}) : dispatch_k<K + 1>(k, f);
}

// 128-bit streaming load: read-only path, do not allocate in L1 (each byte is used once per pass)
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_stream_f1(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
// The same loads with an L2 eviction priority.  The policy is a 64-bit descriptor from createpolicy; keep it warp-uniform
// (it then travels in a uniform register: LDG.E.NA.128.CONSTANT desc[URx][...]).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ float4 ld_stream_f4(const float4* p, uint64_t pol) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ float ld_stream_f1(const float* p, uint64_t pol) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
    return v;
}
// streaming store (evict-first): the write-back is not re-read by this step
__device__ __forceinline__ void st_stream_f4(float4* p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

// ---- k x k Gramian exchange over peer memory (include/movae_b200.h, "P-sharded aggregation") ----------
// One buffer per rank, mapped by every peer (CUDA IPC).  `slots` / `flags` are written by the PEERS (rank r writes
// slots[*][r] and flags[*][r] of every buffer); `step`, `bar_epoch` are this rank's own device-side sequence numbers:
// nothing about the exchange is a kernel argument that changes from step to step, so the launches are CUDA-graph
// capturable and a replayed graph keeps counting.
struct XchgBuffer {
    double slots[2][MOVAE_MAX_WORLD][MOVAE_MAX_K * MOVAE_MAX_K];
    unsigned long long flags[2][MOVAE_MAX_WORLD];
    unsigned long long bar_flags[MOVAE_MAX_WORLD];
    unsigned long long step;         // exchanges this rank has published so far
    unsigned long long bar_epoch;    // device barriers this rank has entered so far
};
struct P2PArgs {
    int rank, world;                    // world == 0: exchange disabled
    XchgBuffer* peers[MOVAE_MAX_WORLD];
};
__host__ __device__ inline P2PArgs p2p_disabled() {
    P2PArgs a;
    a.rank = 0;
    a.world = 0;
    for (int i = 0; i < MOVAE_MAX_WORLD; ++i) a.peers[i] = nullptr;
    return a;
}
int make_p2p_args(const movae_p2p_ctx* ctx, P2PArgs* out);   // validates; defined in p2p.cu

__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_relaxed_sys_f64(double* p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned int* p, unsigned int v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Waits until *flag >= want (system scope: the flag is written by a peer GPU).  Returns false when the peer did not
// show up within `timeout_ns` (a dead or desynchronised rank must not hang the GPU forever).
__device__ __forceinline__ bool wait_flag_sys(const unsigned long long* flag, unsigned long long want,
                                              unsigned long long timeout_ns) {
    if (ld_acquire_sys_u64(flag) >= want) return true;
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys_u64(flag) < want) {
        if (global_timer_ns() - t0 > timeout_ns) return false;
    }
    return true;
}
constexpr unsigned long long kExchangeTimeoutNs = 20ull * 1000ull * 1000ull * 1000ull;   // 20 s

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace movae
