// Kernels of the two forwards whose text rows are shared by the whole batch (head.cu: shared_rows_fwd).  Step rows:
// [Tn class-text rows | C prototype rows | P prompt rows | 10 state-table rows]; only the image row is per sample.
//  - PROOF fusion (Proof_Net.forward / forward_transformer, utils/inc_net.py:436-492): tokens of sample b =
//    [image_b | Tn text | C prototypes | P prompts]; the state rows stay zero and no query sees them.  Outputs: the
//    image row of every sample and the BATCH MEANS of the text / prototype rows (utils/inc_net.py:458-459).
//  - class-text form of forward_tri_modal (utils/inc_net.py:528-580 with text rows != batch): tokens of sample b =
//    [image_b | Tn text | state_b | C prototypes | P prompts]; the state-table row of the sample (column M + sid) is
//    one more per-sample key.  Outputs per sample: image row, MEAN over the Tn text rows, state row, MEAN over the C
//    prototype rows.
// As in the tri-modal head, the shared rows are projected once per step, their softmax over the M = Tn + C + P shared
// keys is a per-step partial (m_r, Z_r, NF_r), and the only per-sample keys they see are those of the sample.
#pragma once
#include "head_bwd_kernels.cuh"

namespace team {

// softmax of the own (image) query over the M shared keys, the sample's state key (column M + sid; none when
// state_ids is null) and its own key
__global__ void __launch_bounds__(256)
image_attn_own_kernel(int B, int M, int Nsp, const float* __restrict__ SQ, const float* __restrict__ QKVo,
                      const __nv_bfloat16* __restrict__ QKVoh, const int64_t* __restrict__ state_ids,
                      float* __restrict__ Aext, __nv_bfloat16* __restrict__ Aexth, float* __restrict__ aown) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= B) return;
    const int scol = state_ids != nullptr ? M + clamp_state(state_ids[row]) : -1;
    float4 q[4], k[4];
    const bool hq = QKVoh != nullptr;
    ld_row_any(QKVo + (size_t)row * 3 * D, hq ? QKVoh + (size_t)row * 3 * D : nullptr, lane, q);
    ld_row_any(QKVo + (size_t)row * 3 * D + D, hq ? QKVoh + (size_t)row * 3 * D + D : nullptr, lane, k);
    const float s_own = warp_sum(dot_part(q, k)) * INV_TAU;
    float mx = s_own;
    for (int j = lane; j < Nsp; j += 32)
        if (j < M || j == scol) mx = fmaxf(mx, SQ[(size_t)row * Nsp + j] * INV_TAU);
    mx = warp_max(mx);
    float z = 0.f;
    for (int j = lane; j < Nsp; j += 32) {
        float p = 0.f;
        if (j < M || j == scol) { p = expf(SQ[(size_t)row * Nsp + j] * INV_TAU - mx); z += p; }
        Aext[(size_t)row * Nsp + j] = p;
    }
    const float p_own = expf(s_own - mx);
    z = warp_sum(z) + p_own;
    const float iz = 1.0f / z;
    for (int j = lane; j < Nsp; j += 32) {
        const float a = Aext[(size_t)row * Nsp + j] * iz;
        Aext[(size_t)row * Nsp + j] = a;
        if (Aexth != nullptr) Aexth[(size_t)row * Nsp + j] = __float2bfloat16_rn(a);
    }
    if (lane == 0) aown[row] = p_own * iz;
}

// out_image[b] = LayerNorm(Aext_b VFs + a_own VF_b + bfc + x_b)
__global__ void __launch_bounds__(256)
proof_ln_own_fwd_kernel(int B, const float* __restrict__ Ybo, const float* __restrict__ aown,
                        const float* __restrict__ VFo, const float* __restrict__ Xo, const float* __restrict__ bfc,
                        const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ out_image) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= B) return;
    float4 y[4], t[4], g[4], be[4], xh[4], o[4];
    ld_row(Ybo + (size_t)row * D, lane, y);
    ld_row(VFo + (size_t)row * D, lane, t);
    axpy_row(y, aown[row], t);
    ld_row(bfc, lane, t); add_row(y, t);
    ld_row(Xo + (size_t)row * D, lane, t); add_row(y, t);
    ld_row(gamma, lane, g); ld_row(beta, lane, be);
    float rstd;
    ln_forward(y, g, be, xh, rstd, o);
    st_row(out_image + (size_t)row * D, lane, o);
}

// Shared-row queries r < R (text rows, then prototype rows): per sample b
//   u_br = c_w NF_r + a_i VF_b + S_r + bfc,   xhat_br = (u - mean) rstd
// and the sum over the samples [b0, b1) of this CTA goes to partials[cta][r] (fixed partition, fixed order).
// Warp w owns the rows r = w, w + PT_WARPS, ...; the row's NF / S+bfc stay in registers over the sample loop.
constexpr int PT_WARPS = 8;
__global__ void __launch_bounds__(PT_WARPS * 32)
proof_table_rows_fwd_kernel(int B, int R, int Nsp, int per_cta, const float* __restrict__ SK,
                            const float* __restrict__ mt, const float* __restrict__ Zt, const float* __restrict__ NFt,
                            const float* __restrict__ VFo, const float* __restrict__ S, const float* __restrict__ bfc,
                            float* __restrict__ partials) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b0 = blockIdx.x * per_cta, b1 = min(B, b0 + per_cta);
    float4 bf[4];
    ld_row(bfc, lane, bf);
    for (int r = warp; r < R; r += PT_WARPS) {
        float4 nf[4], sr[4], acc[4];
        ld_row(NFt + (size_t)r * D, lane, nf);
        ld_row(S + (size_t)r * D, lane, sr);
        add_row(sr, bf);
        zero_row(acc);
        const float mr = mt[r], zr = Zt[r];
        for (int b = b0; b < b1; ++b) {
            const float s_i = SK[(size_t)b * Nsp + r] * INV_TAU;
            const float m2 = fmaxf(mr, s_i);
            const float c = expf(mr - m2), p_i = expf(s_i - m2);
            const float w = 1.0f / (c * zr + p_i);
            float4 u[4], v[4];
            ld_row(VFo + (size_t)b * D, lane, v);
#pragma unroll
            for (int i = 0; i < 4; ++i) u[i] = fma4s(c * w, nf[i], fma4s(p_i * w, v[i], sr[i]));
            const float mean = warp_sum(sum_part(u)) * (1.0f / D);
            shift_row(u, -mean);
            const float var = warp_sum(dot_part(u, u)) * (1.0f / D);
            axpy_row(acc, 1.0f / sqrtf(var + LN_EPS), u);
        }
        st_row(partials + ((size_t)blockIdx.x * R + r) * D, lane, acc);
    }
}

// out[r] = gamma .* (1/B) sum_p partials[p][r] + beta; rows [0, Tn) -> out_text, [Tn, R) -> out_proto.
// block = row r, 128 float4 columns x 4 interleaved partial groups folded in a fixed order.
__global__ void __launch_bounds__(512)
proof_finalize_kernel(const float* __restrict__ partials, int nparts, int R, int Tn, float inv_B,
                      const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ out_text,
                      float* __restrict__ out_proto) {
    pdl_trigger();
    pdl_wait();
    __shared__ float4 fold[4][128];
    const int r = blockIdx.x, c = threadIdx.x & 127, g = threadIdx.x >> 7;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int p = g; p < nparts; p += 4) {
        const float4 a = reinterpret_cast<const float4*>(partials + ((size_t)p * R + r) * D)[c];
        s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
    }
    fold[g][c] = s;
    __syncthreads();
    if (g == 0) {
        float4 t = fold[0][c];
        for (int q = 1; q < 4; ++q) { t.x += fold[q][c].x; t.y += fold[q][c].y; t.z += fold[q][c].z; t.w += fold[q][c].w; }
        const float4 ga = reinterpret_cast<const float4*>(gamma)[c], be = reinterpret_cast<const float4*>(beta)[c];
        t.x = fmaf(t.x * inv_B, ga.x, be.x); t.y = fmaf(t.y * inv_B, ga.y, be.y);
        t.z = fmaf(t.z * inv_B, ga.z, be.z); t.w = fmaf(t.w * inv_B, ga.w, be.w);
        float* dst = r < Tn ? out_text + (size_t)r * D : out_proto + (size_t)(r - Tn) * D;
        reinterpret_cast<float4*>(dst)[c] = t;
    }
}

// table-query rows of one sample (warp per sample): Tn text rows, C prototype rows, the state row.
// row r (step-row id): u = c_w NF_r + a_i VF_b + a_s VFs_srow + S_r + bfc -> LayerNorm; softmax over
// {M shared keys (partial m_r, Z_r), own image key SK[b][r], state key TT[r][srow]}.
__global__ void __launch_bounds__(256)
ct_table_rows_fwd_kernel(int B, int Tn, int C, int M, int Nsp, const float* __restrict__ SK,
                         const float* __restrict__ TT, const float* __restrict__ mt, const float* __restrict__ Zt,
                         const float* __restrict__ NFt, const float* __restrict__ VFo, const float* __restrict__ VFs,
                         const float* __restrict__ S, const float* __restrict__ bfc, const float* __restrict__ gamma,
                         const float* __restrict__ beta, const int64_t* __restrict__ state_ids,
                         float* __restrict__ out_text, float* __restrict__ out_state, float* __restrict__ out_proto) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    const int srow = M + clamp_state(state_ids[b]);
    float4 vi[4], vs[4], bf[4], g[4], be[4], acc_t[4], acc_p[4];
    ld_row(VFo + (size_t)b * D, lane, vi);
    ld_row(VFs + (size_t)srow * D, lane, vs);
    ld_row(bfc, lane, bf); ld_row(gamma, lane, g); ld_row(beta, lane, be);
    zero_row(acc_t); zero_row(acc_p);
    const int R = Tn + C;
    for (int j = 0; j <= R; ++j) {
        const int r = j < R ? j : srow;
        const float s_i = SK[(size_t)b * Nsp + r] * INV_TAU;
        const float s_s = TT[(size_t)r * Nsp + srow] * INV_TAU;
        const float mr = mt[r];
        const float m2 = fmaxf(mr, fmaxf(s_i, s_s));
        const float c = expf(mr - m2), p_i = expf(s_i - m2), p_s = expf(s_s - m2);
        const float w = 1.0f / (c * Zt[r] + p_i + p_s);
        float4 u[4], t[4];
        ld_row(NFt + (size_t)r * D, lane, u);
        ld_row(S + (size_t)r * D, lane, t);
#pragma unroll
        for (int i = 0; i < 4; ++i) u[i] = fma4s(c * w, u[i], fma4s(p_i * w, vi[i], fma4s(p_s * w, vs[i], add4(t[i], bf[i]))));
        const float mean = warp_sum(sum_part(u)) * (1.0f / D);
        shift_row(u, -mean);
        const float var = warp_sum(dot_part(u, u)) * (1.0f / D);
        const float rstd = 1.0f / sqrtf(var + LN_EPS);
        if (j < Tn) axpy_row(acc_t, rstd, u);
        else if (j < R) axpy_row(acc_p, rstd, u);
        else {
#pragma unroll
            for (int i = 0; i < 4; ++i) u[i] = fma4(mul4s(rstd, u[i]), g[i], be[i]);
            st_row(out_state + (size_t)b * D, lane, u);
        }
    }
    const float it = 1.0f / (float)Tn, ip = 1.0f / (float)C;
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc_t[i] = fma4(mul4s(it, acc_t[i]), g[i], be[i]); acc_p[i] = fma4(mul4s(ip, acc_p[i]), g[i], be[i]); }
    st_row(out_text + (size_t)b * D, lane, acc_t);
    st_row(out_proto + (size_t)b * D, lane, acc_p);
}

}  // namespace team
