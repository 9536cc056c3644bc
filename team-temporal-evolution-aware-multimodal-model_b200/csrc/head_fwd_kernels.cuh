// Forward kernels of the fusion head (Proof_Net.forward_tri_modal, utils/inc_net.py:528-580;
// sel_attn, convs/projections.py:64-87) in the factorised form of DESIGN.md section 3:
//   * the C prototype rows, P prompt rows and the 10 state-table rows ("step rows") are
//     projected ONCE per step instead of once per sample;
//   * fc is folded into V (VF = V Wfc^T), so attention outputs are convex combinations of
//     VF rows and fc is never applied to the 3+C returned rows of every sample;
//   * queries that are step rows (prototype outputs, state output) reuse a per-step
//     softmax partial (m, Z, NF) over the M shared keys; only 3 own keys are per sample.
#pragma once
#include "head_kernels.cuh"

namespace team {

// ------------------------------------------------------------------ step prologue: sum_t W_t, sum_t b_t, operand staging
// ONE launch: blocks [0, sum_blocks) sum the per-task projection weights/biases (fp32 + bf16 shadow); the
// remaining blocks copy/convert the listed fp32 matrices (caller inputs, attention weights) into the
// workspace (optional fp32 copy, optional bf16 shadow).  Both lists travel by value (graph-capturable).
struct PrepSum {
    PtrList W[3], Bv[3];
    float* Wout[3];
    __nv_bfloat16* Wh[3];
    float* bout[3];
    int n;                     // how many of the 3 projections to sum
};
struct ConvSeg {
    const float* src;
    float* dstf;               // optional fp32 copy
    __nv_bfloat16* dsth;       // optional bf16 shadow
    int64_t n4;                // float4 count (rows * cols / 4; both sides contiguous)
    int blk0;                  // first conversion block of this segment
};
constexpr int PREP_MAX_SEGS = 12;
struct ConvList {
    ConvSeg s[PREP_MAX_SEGS];
    int n;
    int sum_blocks;
};
constexpr int PREP_SUM_BLOCKS_PER_W = D * D / 4 / 256;      // 256

__global__ void __launch_bounds__(256)
prep_kernel(const __grid_constant__ PrepSum ps, const __grid_constant__ ConvList cl) {
    pdl_trigger();
    pdl_wait();
    if ((int)blockIdx.x < cl.sum_blocks) {
        const int k = blockIdx.x / PREP_SUM_BLOCKS_PER_W;
        const int i = (blockIdx.x % PREP_SUM_BLOCKS_PER_W) * 256 + threadIdx.x;        // float4 index
        const PtrList& W = ps.W[k];
        // summation order t = 0, 1, 2, ... like torch.stack(...).sum(1); loads batched 4 deep to overlap their latency
        float4 s = __ldg(reinterpret_cast<const float4*>(W.p[0]) + i);
        int t = 1;
        for (; t + 4 <= W.n; t += 4) {
            float4 a[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) a[q] = __ldg(reinterpret_cast<const float4*>(W.p[t + q]) + i);
#pragma unroll
            for (int q = 0; q < 4; ++q) { s.x += a[q].x; s.y += a[q].y; s.z += a[q].z; s.w += a[q].w; }
        }
        for (; t < W.n; ++t) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(W.p[t]) + i);
            s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
        }
        reinterpret_cast<float4*>(ps.Wout[k])[i] = s;
        if (ps.Wh[k] != nullptr) reinterpret_cast<uint2*>(ps.Wh[k])[i] = pack_bf16x4(s);
        if (i < D / 4) {
            const PtrList& Bv = ps.Bv[k];
            float4 b = __ldg(reinterpret_cast<const float4*>(Bv.p[0]) + i);
            for (int t = 1; t < Bv.n; ++t) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(Bv.p[t]) + i);
                b.x += a.x; b.y += a.y; b.z += a.z; b.w += a.w;
            }
            reinterpret_cast<float4*>(ps.bout[k])[i] = b;
        }
        return;
    }
    const int cb = (int)blockIdx.x - cl.sum_blocks;
    int si = 0;
    for (int q = 1; q < cl.n; ++q)
        if (cb >= cl.s[q].blk0) si = q;
    const ConvSeg& sg = cl.s[si];
    const int64_t i = (int64_t)(cb - sg.blk0) * 256 + threadIdx.x;
    if (i >= sg.n4) return;
    const float4 v = __ldg(reinterpret_cast<const float4*>(sg.src) + i);
    if (sg.dstf != nullptr) reinterpret_cast<float4*>(sg.dstf)[i] = v;
    if (sg.dsth != nullptr) reinterpret_cast<uint2*>(sg.dsth)[i] = pack_bf16x4(v);
}

// ------------------------------------------------------------------ row L2-normalise (F.normalize)
// For every segment: X[r] = Z[r] / max(|Z[r]|, 1e-12) (fp32 + bf16 shadow); inv[r] = 1/max(|Z[r]|,eps).
// warp per row, 8 rows per block, one launch for all row sets of a step.
struct NormSeg {
    const float* Z;
    float* X;
    __nv_bfloat16* Xh;
    float* inv;
    int64_t rows;
    int blk0;
};
struct NormList {
    NormSeg s[4];
    int n;
    int do_normalize;
};
__global__ void __launch_bounds__(256)
rows_normalize_kernel(const __grid_constant__ NormList nl) {
    pdl_trigger();
    pdl_wait();
    int si = 0;
    for (int q = 1; q < nl.n; ++q)
        if ((int)blockIdx.x >= nl.s[q].blk0) si = q;
    const NormSeg& sg = nl.s[si];
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)((int)blockIdx.x - sg.blk0) * 8 + (threadIdx.x >> 5);
    if (r >= sg.rows) return;
    float4 v[4];
    ld_row(sg.Z + r * D, lane, v);
    float s = 1.0f;
    if (nl.do_normalize) {
        const float ss = warp_sum(dot_part(v, v));
        s = 1.0f / fmaxf(sqrtf(ss), NORM_EPS);
        scale_row(v, s);
    }
    st_row(sg.X + r * D, lane, v);
    st_row_h(sg.Xh != nullptr ? sg.Xh + r * D : nullptr, lane, v);
    if (sg.inv != nullptr && lane == 0) sg.inv[r] = s;
}

// out[r] = table[clamp(ids[r])]  (state-embedding style gather of 512-wide rows)
__global__ void __launch_bounds__(256)
gather_rows_kernel(const float* __restrict__ table, const int64_t* __restrict__ ids, int64_t n_rows, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= n_rows) return;
    float4 v[4];
    ld_row(table + (size_t)clamp_state(ids[r]) * D, lane, v);
    st_row(out + r * D, lane, v);
}

// prompts of all tasks -> S rows [C, C+P); zero rows [Ns, Nsp)
__global__ void __launch_bounds__(128)
fill_prompt_rows_kernel(PtrList prompts, int ppt, int C, int Ns, int Nsp, float* __restrict__ S,
                        __nv_bfloat16* __restrict__ Sh) {
    pdl_trigger();
    pdl_wait();
    const int r = blockIdx.x;                    // 0 .. P + (Nsp-Ns) - 1
    const int P = prompts.n * ppt;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    int dst;
    if (r < P) {
        v = reinterpret_cast<const float4*>(prompts.p[r / ppt] + (size_t)(r % ppt) * D)[threadIdx.x];
        dst = C + r;
    } else {
        dst = Ns + (r - P);
    }
    reinterpret_cast<float4*>(S + (size_t)dst * D)[threadIdx.x] = v;
    if (Sh != nullptr) reinterpret_cast<uint2*>(Sh + (size_t)dst * D)[threadIdx.x] = pack_bf16x4(v);
}

// ------------------------------------------------------------------ per-step softmax partials of step-row queries
// For every step row r: m_r = max_j<M TT[r][j]/tau, P[r][j] = exp(TT[r][j]/tau - m_r) (0 for j>=M), Z_r = sum_j P.
// Warps past the Nsp step rows (optional, Xf != null) write the TABLE rows of the Gram formulation of the table-query
// rows (head_table_gram.cuh) behind the VF rows of the step - extra B-operand rows of W0 = VFo x [VFs ; s ; n]^T:
//   Xf[tr]      = s_tr = S_r + b_fc                       (tr < 32: r = the C prototype rows, then the ten state rows)
//   Xf[32 + tr] = n_tr = sum_{j<M} P[r][j] VFs_j           (table_nf_kernel below)
// rows past Rt are zero.
__global__ void __launch_bounds__(256)
table_prep_kernel(const float* __restrict__ TT, int M, int Nsp, float* __restrict__ mt, float* __restrict__ Zt,
                  float* __restrict__ Pt, __nv_bfloat16* __restrict__ Pth, const float* __restrict__ S,
                  const float* __restrict__ bfc, const float* __restrict__ VFsf, const __nv_bfloat16* __restrict__ VFsh,
                  int C, int xrows, float* __restrict__ Xf, __nv_bfloat16* __restrict__ Xh) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= Nsp) {
        if (Xf == nullptr) return;
        const int x = r - Nsp, Rt = C + 10;
        if (x < xrows) {                                   // s rows (and the zero padding of both tables)
            float4 v[4];
            zero_row(v);
            if (x < Rt) {
                float4 b[4];
                ld_row(S + (size_t)(x < C ? x : M + x - C) * D, lane, v);
                ld_row(bfc, lane, b);
                add_row(v, b);
            } else {
                st_row(Xf + (size_t)(xrows + x) * D, lane, v);
                st_row_h(Xh != nullptr ? Xh + (size_t)(xrows + x) * D : nullptr, lane, v);
            }
            st_row(Xf + (size_t)x * D, lane, v);
            st_row_h(Xh != nullptr ? Xh + (size_t)x * D : nullptr, lane, v);
            return;
        }
        return;
    }
    float mx = -INFINITY;
    for (int j = lane; j < M; j += 32) mx = fmaxf(mx, TT[(size_t)r * Nsp + j] * INV_TAU);
    mx = warp_max(mx);
    float z = 0.f;
    for (int j = lane; j < Nsp; j += 32) {
        float p = 0.f;
        if (j < M) { p = expf(TT[(size_t)r * Nsp + j] * INV_TAU - mx); z += p; }
        Pt[(size_t)r * Nsp + j] = p;
        if (Pth != nullptr) Pth[(size_t)r * Nsp + j] = __float2bfloat16_rn(p);
    }
    z = warp_sum(z);
    if (lane == 0) { mt[r] = mx; Zt[r] = z; }
}

// n rows of the Gram formulation: Xn[tr] = sum_{j<M} P[r(tr)][j] VFs_j, one CTA per table row, thread = (float4 column,
// half of the j range).  Operands rounded to bf16 in BF16 mode (VFsh != null) - exactly what the tensor-core product
// Pt x VFs of GEMM wave 4 multiplies - fp32 accumulation.  Recomputes the row's softmax numerators itself, so it only
// depends on GEMM wave 3 and runs beside table_prep_kernel.
__global__ void __launch_bounds__(256)
table_nf_kernel(const float* __restrict__ TT, int M, int Nsp, int C, const float* __restrict__ VFsf,
                const __nv_bfloat16* __restrict__ VFsh, float* __restrict__ Xn, __nv_bfloat16* __restrict__ Xnh) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) float nf_smem[];          // p[M] | half sums [128] float4
    float* p = nf_smem;
    float4* part = reinterpret_cast<float4*>(nf_smem + ((M + 3) / 4) * 4);
    const int tr = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int rr = tr < C ? tr : M + tr - C;
    float mx = -INFINITY;
    for (int j = lane; j < M; j += 32) mx = fmaxf(mx, TT[(size_t)rr * Nsp + j] * INV_TAU);
    mx = warp_max(mx);
    for (int j = tid; j < M; j += blockDim.x) {
        float v = expf(TT[(size_t)rr * Nsp + j] * INV_TAU - mx);
        if (VFsh != nullptr) v = __bfloat162float(__float2bfloat16_rn(v));
        p[j] = v;
    }
    __syncthreads();
    const int c4 = tid & 127, half = tid >> 7;
    const int jmid = (M + 1) / 2;
    const int j0 = half == 0 ? 0 : jmid, j1 = half == 0 ? jmid : M;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (VFsh != nullptr) {
#pragma unroll 8
        for (int j = j0; j < j1; ++j) {
            const uint2 u = reinterpret_cast<const uint2*>(VFsh + (size_t)j * D)[c4];
            const float pj = p[j];
            acc.x = fmaf(pj, bf16_lo(u.x), acc.x); acc.y = fmaf(pj, bf16_hi(u.x), acc.y);
            acc.z = fmaf(pj, bf16_lo(u.y), acc.z); acc.w = fmaf(pj, bf16_hi(u.y), acc.w);
        }
    } else {
#pragma unroll 8
        for (int j = j0; j < j1; ++j) {
            const float4 v = reinterpret_cast<const float4*>(VFsf + (size_t)j * D)[c4];
            const float pj = p[j];
            acc.x = fmaf(pj, v.x, acc.x); acc.y = fmaf(pj, v.y, acc.y); acc.z = fmaf(pj, v.z, acc.z); acc.w = fmaf(pj, v.w, acc.w);
        }
    }
    if (half == 1) part[c4] = acc;
    __syncthreads();
    if (half == 0) {
        const float4 o = part[c4];
        acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
        reinterpret_cast<float4*>(Xn + (size_t)tr * D)[c4] = acc;
        if (Xnh != nullptr) reinterpret_cast<uint2*>(Xnh + (size_t)tr * D)[c4] = pack_bf16x4(acc);
    }
}

// ------------------------------------------------------------------ softmax of the own (image/text) query rows
// keys: M shared step rows, the sample's state-table row (column M+sid), own image key, own text key.
__global__ void __launch_bounds__(256)
attn_own_kernel(HeadDims d, const float* __restrict__ SQ, const float* __restrict__ QKVo,
                const __nv_bfloat16* __restrict__ QKVoh, const int64_t* __restrict__ state_ids, float* __restrict__ Aext, __nv_bfloat16* __restrict__ Aexth,
                float* __restrict__ aown) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= d.B2) return;
    const int b = row < d.B ? row : row - d.B;
    const int scol = d.M + clamp_state(state_ids[b]);
    float4 q[4], k[4];
    const bool hq = QKVoh != nullptr;
    ld_row_any(QKVo + (size_t)row * 3 * D, hq ? QKVoh + (size_t)row * 3 * D : nullptr, lane, q);
    ld_row_any(QKVo + (size_t)b * 3 * D + D, hq ? QKVoh + (size_t)b * 3 * D + D : nullptr, lane, k);
    const float s_img = warp_sum(dot_part(q, k)) * INV_TAU;
    ld_row_any(QKVo + (size_t)(d.B + b) * 3 * D + D, hq ? QKVoh + (size_t)(d.B + b) * 3 * D + D : nullptr, lane, k);
    const float s_txt = warp_sum(dot_part(q, k)) * INV_TAU;
    float mx = fmaxf(s_img, s_txt);
    for (int j = lane; j < d.Nsp; j += 32)
        if (j < d.M || j == scol) mx = fmaxf(mx, SQ[(size_t)row * d.Nsp + j] * INV_TAU);
    mx = warp_max(mx);
    float z = 0.f;
    for (int j = lane; j < d.Nsp; j += 32) {
        float p = 0.f;
        if (j < d.M || j == scol) { p = expf(SQ[(size_t)row * d.Nsp + j] * INV_TAU - mx); z += p; }
        Aext[(size_t)row * d.Nsp + j] = p;
    }
    const float p_img = expf(s_img - mx), p_txt = expf(s_txt - mx);
    z = warp_sum(z) + p_img + p_txt;
    const float iz = 1.0f / z;
    for (int j = lane; j < d.Nsp; j += 32) {
        const float a = Aext[(size_t)row * d.Nsp + j] * iz;
        Aext[(size_t)row * d.Nsp + j] = a;
        if (Aexth != nullptr) Aexth[(size_t)row * d.Nsp + j] = __float2bfloat16_rn(a);
    }
    if (lane == 0) { aown[2 * row] = p_img * iz; aown[2 * row + 1] = p_txt * iz; }
}

// ------------------------------------------------------------------ fc-space output + residual + LayerNorm, own rows
__global__ void __launch_bounds__(256)
ln_own_fwd_kernel(HeadDims d, float* __restrict__ Ybo, const float* __restrict__ aown,
                  const float* __restrict__ VFo, const float* __restrict__ Xo, const float* __restrict__ bfc,
                  const float* __restrict__ gamma, const float* __restrict__ beta,
                  float* __restrict__ out_image, float* __restrict__ out_text) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= d.B2) return;
    const int b = row < d.B ? row : row - d.B;
    float4 y[4], t[4], g[4], be[4], xh[4], o[4];
    ld_row(Ybo + (size_t)row * D, lane, y);
    ld_row(VFo + (size_t)b * D, lane, t);
    axpy_row(y, aown[2 * row], t);
    ld_row(VFo + (size_t)(d.B + b) * D, lane, t);
    axpy_row(y, aown[2 * row + 1], t);
    st_row(Ybo + (size_t)row * D, lane, y);               // Ybar (without bias): needed by the backward
    ld_row(bfc, lane, t); add_row(y, t);
    ld_row(Xo + (size_t)row * D, lane, t); add_row(y, t);
    ld_row(gamma, lane, g); ld_row(beta, lane, be);
    float rstd;
    ln_forward(y, g, be, xh, rstd, o);
    st_row((row < d.B ? out_image : out_text) + (size_t)b * D, lane, o);
}

// ------------------------------------------------------------------ table-query rows (prototype + state outputs)
// The C prototype queries and the state query of one sample share the per-step softmax partial (m_r, Z_r, NF_r)
// over the M shared keys; only the three own keys (image, text, state) are per sample.
// One CTA (TQ_WARPS warps) works on one sample at a time; warp w owns the rows j = w, w + TQ_WARPS, ...
// (j < C: prototype row j, j == C: the state row).  The softmax weights of a warp's rows are computed
// lane-parallel (lane k -> k-th row of the warp) and broadcast with shuffles inside the row loop.
constexpr int TQ_WARPS = 4;

struct TableRowW {
    float c_w;             // c / den   (weight of the shared partial NF_r)
    float a_i, a_t, a_s;   // attention on the own image / text / state keys
    int r;                 // step-row id of this query
};

__device__ __forceinline__ TableRowW table_row_weights(const HeadDims& d, int b, int j, int srow,
        const float* __restrict__ SK, const float* __restrict__ TT, const float* __restrict__ mt,
        const float* __restrict__ Zt) {
    TableRowW o;
    const int r = j < d.C ? j : srow;
    o.r = r;
    const float s_i = SK[(size_t)b * d.Nsp + r] * INV_TAU;
    const float s_t = SK[(size_t)(d.B + b) * d.Nsp + r] * INV_TAU;
    const float s_s = TT[(size_t)r * d.Nsp + srow] * INV_TAU;
    const float mr = mt[r];
    const float m2 = fmaxf(fmaxf(mr, s_i), fmaxf(s_t, s_s));
    const float c = expf(mr - m2), p_i = expf(s_i - m2), p_t = expf(s_t - m2), p_s = expf(s_s - m2);
    const float w = 1.0f / (c * Zt[r] + p_i + p_t + p_s);
    o.c_w = c * w; o.a_i = p_i * w; o.a_t = p_t * w; o.a_s = p_s * w;
    return o;
}
__device__ __forceinline__ TableRowW shfl_row_weights(const TableRowW& v, int src) {
    TableRowW o;
    o.c_w = __shfl_sync(0xffffffffu, v.c_w, src); o.a_i = __shfl_sync(0xffffffffu, v.a_i, src);
    o.a_t = __shfl_sync(0xffffffffu, v.a_t, src); o.a_s = __shfl_sync(0xffffffffu, v.a_s, src);
    o.r = __shfl_sync(0xffffffffu, v.r, src);
    return o;
}

// out_proto[b] = gamma .* (1/C) sum_{j<C} xhat_bj + beta  (LayerNorm is affine in xhat, so gamma/beta are applied once);
// out_state[b] = gamma .* xhat_bC + beta.
__global__ void __launch_bounds__(TQ_WARPS * 32)
table_rows_fwd_kernel(HeadDims d, const float* __restrict__ SK, const float* __restrict__ TT,
                      const float* __restrict__ mt, const float* __restrict__ Zt, const float* __restrict__ NFt,
                      const float* __restrict__ VFo, const float* __restrict__ VFs, const float* __restrict__ S,
                      const float* __restrict__ bfc, const float* __restrict__ gamma, const float* __restrict__ beta,
                      const int64_t* __restrict__ state_ids, float* __restrict__ out_proto,
                      float* __restrict__ out_state) {
    pdl_trigger();
    pdl_wait();
    __shared__ __align__(16) float slot[TQ_WARPS][D];          // 8 KB
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4 bf[4];
    ld_row(bfc, lane, bf);
    const int nrows = d.C + 1 > warp ? (d.C + 1 - warp + TQ_WARPS - 1) / TQ_WARPS : 0;     // rows of this warp
    const float invC = 1.0f / (float)d.C;
    for (int b = blockIdx.x; b < d.B; b += gridDim.x) {
        const int srow = d.M + clamp_state(state_ids[b]);
        float4 vi[4], vt[4], vs[4], acc[4];
        ld_row(VFo + (size_t)b * D, lane, vi);
        ld_row(VFo + (size_t)(d.B + b) * D, lane, vt);
        ld_row(VFs + (size_t)srow * D, lane, vs);
        zero_row(acc);
        for (int k0 = 0; k0 < nrows; k0 += 32) {
            TableRowW mine;
            mine.c_w = mine.a_i = mine.a_t = mine.a_s = 0.f; mine.r = 0;
            if (k0 + lane < nrows) mine = table_row_weights(d, b, warp + (k0 + lane) * TQ_WARPS, srow, SK, TT, mt, Zt);
            const int kn = min(32, nrows - k0);
            for (int k = 0; k < kn; ++k) {
                const TableRowW rw = shfl_row_weights(mine, k);
                const int j = warp + (k0 + k) * TQ_WARPS;
                float4 u[4], t[4];
                ld_row(NFt + (size_t)rw.r * D, lane, u);
                ld_row(S + (size_t)rw.r * D, lane, t);
                scale_row(u, rw.c_w);
                axpy_row(u, rw.a_i, vi); axpy_row(u, rw.a_t, vt); axpy_row(u, rw.a_s, vs);
                add_row(u, bf); add_row(u, t);
                const float mean = warp_sum(sum_part(u)) * (1.0f / D);
                shift_row(u, -mean);
                const float var = warp_sum(dot_part(u, u)) * (1.0f / D);
                const float rstd = 1.0f / sqrtf(var + LN_EPS);
                if (j < d.C) {
                    axpy_row(acc, rstd, u);
                } else {
                    float4 g[4], be[4];
                    ld_row(gamma, lane, g); ld_row(beta, lane, be);
#pragma unroll
                    for (int i = 0; i < 4; ++i) u[i] = fma4(mul4s(rstd, u[i]), g[i], be[i]);
                    st_row(out_state + (size_t)b * D, lane, u);
                }
            }
        }
        st_row(slot[warp], lane, acc);
        __syncthreads();
        {
            const int t = threadIdx.x;                              // float4 column t of the 512-wide row
            float4 s = reinterpret_cast<const float4*>(slot[0])[t];
#pragma unroll
            for (int w = 1; w < TQ_WARPS; ++w) {
                const float4 a = reinterpret_cast<const float4*>(slot[w])[t];
                s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
            }
            const float4 g = reinterpret_cast<const float4*>(gamma)[t], be = reinterpret_cast<const float4*>(beta)[t];
            s.x = fmaf(s.x * invC, g.x, be.x); s.y = fmaf(s.y * invC, g.y, be.y);
            s.z = fmaf(s.z * invC, g.z, be.z); s.w = fmaf(s.w * invC, g.w, be.w);
            reinterpret_cast<float4*>(out_proto + (size_t)b * D)[t] = s;
        }
        __syncthreads();
    }
}

}  // namespace team
