// Internal helpers shared by the libhgr.so translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "hgr.h"

namespace hgr {

int set_error(int code, const char *fmt, ...);
extern std::atomic<uint64_t> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

#define HGR_REQUIRE(cond, ...)                                      \
    do {                                                            \
        if (!(cond)) return hgr::set_error(HGR_ERR_INVALID, __VA_ARGS__); \
    } while (0)

#define HGR_CUDA_OK(expr)                                                                            \
    do {                                                                                             \
        cudaError_t e_ = (expr);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return hgr::set_error(HGR_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                                  __FILE__, __LINE__);                                               \
    } while (0)

#define HGR_LAUNCH_OK(name)                                                                               \
    do {                                                                                                  \
        cudaError_t e_ = cudaGetLastError();                                                              \
        if (e_ != cudaSuccess)                                                                            \
            return hgr::set_error(HGR_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e_)); \
        hgr::count_launch();                                                                              \
    } while (0)

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- device helpers ------------------------------------------------------------------------
// streaming (read-once) loads: keep them out of L1 so gathered embedding rows stay there
__device__ __forceinline__ int ld_stream_i32(const int *p) {
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_stream_f32(const float *p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ld_stream_f4(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}

// One 16-byte store to a MULTICAST address: the NVSwitch delivers it to the copy of every GPU bound to the multicast object.
__device__ __forceinline__ void st_multicast_f4(float4 *mc_addr, float4 v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

// Philox4x32-10 (counter-based: the value depends on (seed, counter) only, never on the launch geometry)
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0;
    c[1] = n1;
    c[2] = n2;
    c[3] = n3;
}

__device__ __forceinline__ void philox4x32_10(uint64_t seed, uint64_t ctr_lo, uint32_t ctr_hi, uint32_t (&out)[4]) {
    uint32_t c[4] = {(uint32_t)ctr_lo, (uint32_t)(ctr_lo >> 32), ctr_hi, 0x9E3779B9u};
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) out[j] = c[j];
}

template <int WIDTH>
__device__ __forceinline__ float group_sum(float v, unsigned mask) {
#pragma unroll
    for (int o = WIDTH / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o, WIDTH);
    return v;
}

}  // namespace hgr
