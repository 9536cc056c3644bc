// Shared helpers for the TEAM head kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/team_b200.h"

namespace team {

constexpr int D = TEAM_D;               // 512
constexpr int NUM_SMS = 148;            // B200
constexpr float LN_EPS = 1e-5f;
constexpr float NORM_EPS = 1e-12f;

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
void count_launch();

#define TEAM_CUDA_CHECK(expr)                                   \
    do {                                                        \
        cudaError_t _e = (expr);                                \
        if (_e != cudaSuccess) return team::cuda_fail(_e, #expr); \
    } while (0)

// one per kernel launch: counts it (team_launch_count) and checks the launch status
#define TEAM_LAUNCH_CHECK(name)                                 \
    do {                                                        \
        team::count_launch();                                   \
        cudaError_t _e = cudaGetLastError();                    \
        if (_e != cudaSuccess) return team::cuda_fail(_e, name); \
    } while (0)

#define TEAM_REQUIRE(cond, ...)                                 \
    do {                                                        \
        if (!(cond)) { team::set_error(__VA_ARGS__); return TEAM_EINVAL; } \
    } while (0)

// Programmatic dependent launch: every kernel of the library releases its dependents at once and then waits
// for its own prerequisites before touching global memory, so launch latency, block scheduling and the
// prologue (barrier init, TMEM alloc, parameter loads) of kernel N+1 overlap the tail of kernel N.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(block, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<Args&&>(args)...);
}
// launch + count + status check (the kernel must start with pdl_trigger(); pdl_wait();)
#define TEAM_LAUNCH(kernel, grid, block, smem, st, ...)                                         \
    do {                                                                                        \
        cudaError_t _e = team::launch_pdl(kernel, (unsigned)(grid), (unsigned)(block), (size_t)(smem), st, __VA_ARGS__); \
        team::count_launch();                                                                   \
        if (_e != cudaSuccess) return team::cuda_fail(_e, #kernel);                             \
    } while (0)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// 128-bit streaming load that does not pollute L1 (inputs read exactly once).
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ld_stream_u2(const void* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

__device__ __forceinline__ uint2 pack_bf16x4(float4 v) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<const uint32_t*>(&a);
    o.y = *reinterpret_cast<const uint32_t*>(&b);
    return o;
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace team
