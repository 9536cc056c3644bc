// Per-row / per-sample CUDA-core kernels of the fusion head (softmax, LayerNorm, table-query
// rows, normalisation) - warp-per-row with 128-bit loads and shuffle reductions.
// Lane l of a warp owns float4 columns {l, l+32, l+64, l+96} of a 512-wide row.
#pragma once
#include "head.cuh"

namespace team {

constexpr float INV_TAU = 0.04419417382415922f;      // 1/sqrt(512)  (convs/projections.py:57)
constexpr int TR_WARPS = 8;                           // warps per CTA in the table-row kernels (thread t owns columns 2t,2t+1)

struct PtrList {
    const float* p[TEAM_MAX_TASKS];
    int n;
};

__device__ __forceinline__ void ld_row(const float* p, int lane, float4 (&v)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = reinterpret_cast<const float4*>(p)[lane + 32 * i];
}
__device__ __forceinline__ void st_row(float* p, int lane, const float4 (&v)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) reinterpret_cast<float4*>(p)[lane + 32 * i] = v[i];
}
// 512-wide row from its bf16 shadow when there is one (BF16 mode: the fp32 copy of a pure GEMM operand is not
// materialised), else from the fp32 buffer; same lane -> column mapping as ld_row
__device__ __forceinline__ void ld_row_any(const float* f, const __nv_bfloat16* h, int lane, float4 (&v)[4]) {
    if (h != nullptr) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint2 u = reinterpret_cast<const uint2*>(h)[lane + 32 * i];
            v[i] = make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
        }
    } else {
        ld_row(f, lane, v);
    }
}
// bf16 shadow of a 512-wide row (same lane -> column mapping); p may be null (F32 mode)
__device__ __forceinline__ void st_row_h(__nv_bfloat16* p, int lane, const float4 (&v)[4]) {
    if (p == nullptr) return;
#pragma unroll
    for (int i = 0; i < 4; ++i) reinterpret_cast<uint2*>(p)[lane + 32 * i] = pack_bf16x4(v[i]);
}
// ---- 512-wide row arithmetic on packed fp32 pairs (sm_100 FFMA2 / FADD2 / FMUL2: one instruction per two
// lanes of a float4, rounding identical to the scalar fmaf / add / mul)
__device__ __forceinline__ float2 xy(const float4& v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 zw(const float4& v) { return make_float2(v.z, v.w); }
__device__ __forceinline__ float4 f4(float2 a, float2 b) { return make_float4(a.x, a.y, b.x, b.y); }
__device__ __forceinline__ float4 fma4(float4 a, float4 b, float4 c) {
    return f4(__ffma2_rn(xy(a), xy(b), xy(c)), __ffma2_rn(zw(a), zw(b), zw(c)));
}
__device__ __forceinline__ float4 fma4s(float a, float4 b, float4 c) {
    const float2 aa = make_float2(a, a);
    return f4(__ffma2_rn(aa, xy(b), xy(c)), __ffma2_rn(aa, zw(b), zw(c)));
}
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return f4(__fadd2_rn(xy(a), xy(b)), __fadd2_rn(zw(a), zw(b))); }
__device__ __forceinline__ float4 mul4(float4 a, float4 b) { return f4(__fmul2_rn(xy(a), xy(b)), __fmul2_rn(zw(a), zw(b))); }
__device__ __forceinline__ float4 mul4s(float a, float4 b) {
    const float2 aa = make_float2(a, a);
    return f4(__fmul2_rn(aa, xy(b)), __fmul2_rn(aa, zw(b)));
}
__device__ __forceinline__ float4 add4s(float a, float4 b) {
    const float2 aa = make_float2(a, a);
    return f4(__fadd2_rn(aa, xy(b)), __fadd2_rn(aa, zw(b)));
}

__device__ __forceinline__ float dot_part(const float4 (&a)[4], const float4 (&b)[4]) {
    float2 s0 = __fmul2_rn(xy(a[0]), xy(b[0])), s1 = __fmul2_rn(zw(a[0]), zw(b[0]));
#pragma unroll
    for (int i = 1; i < 4; ++i) { s0 = __ffma2_rn(xy(a[i]), xy(b[i]), s0); s1 = __ffma2_rn(zw(a[i]), zw(b[i]), s1); }
    const float2 s = __fadd2_rn(s0, s1);
    return s.x + s.y;
}
__device__ __forceinline__ float sum_part(const float4 (&a)[4]) {
    float2 s0 = __fadd2_rn(xy(a[0]), zw(a[0])), s1 = __fadd2_rn(xy(a[1]), zw(a[1]));
    s0 = __fadd2_rn(s0, __fadd2_rn(xy(a[2]), zw(a[2])));
    s1 = __fadd2_rn(s1, __fadd2_rn(xy(a[3]), zw(a[3])));
    const float2 s = __fadd2_rn(s0, s1);
    return s.x + s.y;
}
__device__ __forceinline__ void axpy_row(float4 (&y)[4], float a, const float4 (&x)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = fma4s(a, x[i], y[i]);
}
__device__ __forceinline__ void add_row(float4 (&y)[4], const float4 (&x)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = add4(y[i], x[i]);
}
__device__ __forceinline__ void scale_row(float4 (&y)[4], float a) {
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = mul4s(a, y[i]);
}
__device__ __forceinline__ void shift_row(float4 (&y)[4], float a) {            // y += a
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = add4s(a, y[i]);
}
__device__ __forceinline__ void zero_row(float4 (&y)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// LayerNorm over a 512-wide row held by one warp (eps 1e-5, biased variance).
__device__ __forceinline__ void ln_forward(const float4 (&u)[4], const float4 (&g)[4], const float4 (&be)[4],
                                           float4 (&xh)[4], float& rstd, float4 (&o)[4]) {
    const float mean = warp_sum(sum_part(u)) * (1.0f / D);
#pragma unroll
    for (int i = 0; i < 4; ++i) xh[i] = add4s(-mean, u[i]);
    const float var = warp_sum(dot_part(xh, xh)) * (1.0f / D);
    rstd = 1.0f / sqrtf(var + LN_EPS);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        xh[i] = mul4s(rstd, xh[i]);
        o[i] = fma4(xh[i], g[i], be[i]);
    }
}
// du = rstd * (gg - mean(gg) - xh * mean(gg*xh)),  gg = go * gamma
__device__ __forceinline__ void ln_backward(const float4 (&go)[4], const float4 (&xh)[4], float rstd,
                                            const float4 (&g)[4], float4 (&du)[4]) {
    float4 gg[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) gg[i] = mul4(go[i], g[i]);
    const float m1 = warp_sum(sum_part(gg)) * (1.0f / D);
    const float m2 = warp_sum(dot_part(gg, xh)) * (1.0f / D);
#pragma unroll
    for (int i = 0; i < 4; ++i) du[i] = mul4s(rstd, fma4s(-m2, xh[i], add4s(-m1, gg[i])));
}

__device__ __forceinline__ int clamp_state(int64_t s) { return s < 0 ? 0 : (s > 9 ? 9 : (int)s); }

}  // namespace team
