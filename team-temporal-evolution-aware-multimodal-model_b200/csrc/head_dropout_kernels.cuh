// Train-mode dropout of sel_attn in the fused tri-modal head (team_dropout, include/team_b200.h).
//
// The masks are the ones team_mha_fwd draws on the token tensor [image | text | state | C prototypes | P prompts]
// (L = 3 + C + P) of every sample: probability (b L + i) L + j of the stream (seed, offset), fc element (b L + i) 512 + c of
// (seed, offset + 1).  Query token i: 0 image, 1 text, 2 state, 3 + r prototype r.  Key token j: 0 / 1 / 2 the sample's own
// image / text / state key, 3 + col the shared column col < M.  In the head's [., Nsp] probability rows the shared column
// col sits at col and the state key at M + sid.
//
// With a mask the shared part of a table query is no longer sample-independent, so every (sample, table row) gets its
// own probability row: Wd[b (C+1) + r] = mask .* (the undropped probabilities of the row), and the shared-key output is
// the product Wd VFs (GEMM wave 4).  The backward is the VJP of that: dWd = dYt VFs^T and dVFs = Ad^T dYo + Wd^T dYt
// are products, the softmax backward of every row is folded over the batch in a fixed order into the step-level score
// gradient dTT that GEMM wave 7 consumes.  The undropped probabilities are kept (Aext, Pt and the row scalars), so the
// softmax backward needs no mask regeneration: dS_j = (Ad_j dA_j - A_j (dY . Ybar_dropped)) / tau.
#pragma once
#include "head_kernels.cuh"
#include "head_fwd_kernels.cuh"
#include "head_bwd_kernels.cuh"

namespace team {

struct DropArgs {
    Philox attn;                  // stream (seed, offset); the fc stream is (seed, offset + 1)
    uint32_t thr;                 // p * 2^32
    float inv_keep;               // 1 / (1 - p)
    const uint64_t* offset_dev;   // overrides attn.offset when not null
    int L;                        // tokens per sample, 3 + C + P
};
constexpr int DROP_NSC = 8;      // row scalars of a table-query row: c_w, a_i, a_t, a_s (undropped), a_i, a_t (dropped), rowdot, -

__device__ __forceinline__ Philox drop_stream(const DropArgs& da, int which) {
    Philox g = da.attn;
    if (da.offset_dev != nullptr) g.offset = *da.offset_dev;
    g.offset += (uint64_t)which;
    return g;
}
// keep-scales of the four fc elements of float4 column c4 of token row `tok` (= b L + i)
__device__ __forceinline__ float4 fc_scales(const Philox& g, const DropArgs& da, int64_t tok, int c4) {
    uint32_t q[4];
    philox4(g, ((uint64_t)tok * D + 4 * (uint64_t)c4) >> 2, q);
    return make_float4(q[0] >= da.thr ? da.inv_keep : 0.f, q[1] >= da.thr ? da.inv_keep : 0.f,
                       q[2] >= da.thr ? da.inv_keep : 0.f, q[3] >= da.thr ? da.inv_keep : 0.f);
}
__device__ __forceinline__ void fc_mask_row(const Philox& g, const DropArgs& da, int64_t tok, int lane, float4 (&m)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) m[i] = fc_scales(g, da, tok, lane + 32 * i);
}

// ------------------------------------------------------------------ masked probability rows (forward)
// blocks [0, own_blocks): own query rows (warp per row): Ad = mask .* Aext, aownd = mask .* aown.
// the rest: table-query rows t = b (C+1) + r (warp per row): Wd[t] = mask .* undropped probabilities (shared columns
// P_rj c_w, state key a_s at M + sid), row scalars in tsc.
__global__ void __launch_bounds__(256)
drop_probs_kernel(HeadDims d, DropArgs da, int own_blocks, const float* __restrict__ Aext, const float* __restrict__ aown,
                  const int64_t* __restrict__ state_ids, const float* __restrict__ SK, const float* __restrict__ TT,
                  const float* __restrict__ mt, const float* __restrict__ Zt, const float* __restrict__ Pt,
                  float* __restrict__ Ad, __nv_bfloat16* __restrict__ Adh, float* __restrict__ aownd,
                  float* __restrict__ Wd, __nv_bfloat16* __restrict__ Wdh, float* __restrict__ tsc) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const Philox g = drop_stream(da, 0);
    const int64_t L = da.L;
    if ((int)blockIdx.x < own_blocks) {
        const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
        if (row >= d.B2) return;
        const int b = row < d.B ? row : row - d.B, i = row < d.B ? 0 : 1;
        const int scol = d.M + clamp_state(state_ids[b]);
        const uint64_t tb = (uint64_t)(((int64_t)b * L + i) * L);
        for (int j = lane; j < d.Nsp; j += 32) {
            float v = 0.f;
            if (j < d.M || j == scol) v = Aext[(size_t)row * d.Nsp + j] * drop_scale(g, tb + (j < d.M ? 3 + j : 2), da.thr, da.inv_keep);
            Ad[(size_t)row * d.Nsp + j] = v;
            if (Adh != nullptr) Adh[(size_t)row * d.Nsp + j] = __float2bfloat16_rn(v);
        }
        if (lane < 2) aownd[2 * row + lane] = aown[2 * row + lane] * drop_scale(g, tb + lane, da.thr, da.inv_keep);
        return;
    }
    const int R1 = d.C + 1;
    const int64_t t = (int64_t)((int)blockIdx.x - own_blocks) * 8 + (threadIdx.x >> 5);
    if (t >= (int64_t)d.B * R1) return;
    const int b = (int)(t / R1), r = (int)(t % R1);
    const int srow = d.M + clamp_state(state_ids[b]);
    const TableRowW rw = table_row_weights(d, b, r, srow, SK, TT, mt, Zt);
    const uint64_t tb = (uint64_t)(((int64_t)b * L + (r < d.C ? 3 + r : 2)) * L);
    for (int j = lane; j < d.Nsp; j += 32) {
        float v = 0.f;
        if (j < d.M) v = Pt[(size_t)rw.r * d.Nsp + j] * rw.c_w * drop_scale(g, tb + 3 + j, da.thr, da.inv_keep);
        else if (j == srow) v = rw.a_s * drop_scale(g, tb + 2, da.thr, da.inv_keep);
        Wd[t * d.Nsp + j] = v;
        if (Wdh != nullptr) Wdh[t * d.Nsp + j] = __float2bfloat16_rn(v);
    }
    if (lane == 0) {
        float* sc = tsc + t * DROP_NSC;
        sc[0] = rw.c_w; sc[1] = rw.a_i; sc[2] = rw.a_t; sc[3] = rw.a_s;
        sc[4] = rw.a_i * drop_scale(g, tb + 0, da.thr, da.inv_keep);
        sc[5] = rw.a_t * drop_scale(g, tb + 1, da.thr, da.inv_keep);
        sc[6] = 0.f; sc[7] = 0.f;
    }
}

// ------------------------------------------------------------------ fc output, fc dropout, residual, LayerNorm (forward)
// blocks [0, own_blocks): own rows (warp per row) -> out_image / out_text; Ybo becomes Ybar (dropped, without bias).
// the rest: one warp per sample, its C + 1 table rows -> out_proto (mean of the prototype rows) / out_state; Yt becomes
// Ybar of every table row.
__global__ void __launch_bounds__(256)
drop_ln_fwd_kernel(HeadDims d, DropArgs da, int own_blocks, float* __restrict__ Ybo, const float* __restrict__ aownd,
                   float* __restrict__ Yt, const float* __restrict__ tsc, const float* __restrict__ VFo,
                   const float* __restrict__ Xo, const float* __restrict__ S, const float* __restrict__ bfc,
                   const float* __restrict__ gamma, const float* __restrict__ beta, const int64_t* __restrict__ state_ids,
                   float* __restrict__ out_image, float* __restrict__ out_text, float* __restrict__ out_state,
                   float* __restrict__ out_proto) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const Philox g = drop_stream(da, 1);
    const int64_t L = da.L;
    float4 y[4], t[4], m[4], bf[4], gm[4], be[4], xh[4], o[4];
    ld_row(bfc, lane, bf); ld_row(gamma, lane, gm); ld_row(beta, lane, be);
    if ((int)blockIdx.x < own_blocks) {
        const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
        if (row >= d.B2) return;
        const int b = row < d.B ? row : row - d.B, i = row < d.B ? 0 : 1;
        ld_row(Ybo + (size_t)row * D, lane, y);
        ld_row(VFo + (size_t)b * D, lane, t);
        axpy_row(y, aownd[2 * row], t);
        ld_row(VFo + (size_t)(d.B + b) * D, lane, t);
        axpy_row(y, aownd[2 * row + 1], t);
        st_row(Ybo + (size_t)row * D, lane, y);
        add_row(y, bf);
        fc_mask_row(g, da, (int64_t)b * L + i, lane, m);
#pragma unroll
        for (int k = 0; k < 4; ++k) y[k] = mul4(y[k], m[k]);
        ld_row(Xo + (size_t)row * D, lane, t); add_row(y, t);
        float rstd;
        ln_forward(y, gm, be, xh, rstd, o);
        st_row((row < d.B ? out_image : out_text) + (size_t)b * D, lane, o);
        return;
    }
    const int b = ((int)blockIdx.x - own_blocks) * 8 + (threadIdx.x >> 5);
    if (b >= d.B) return;
    const int R1 = d.C + 1, srow = d.M + clamp_state(state_ids[b]);
    float4 vi[4], vt[4], acc[4];
    ld_row(VFo + (size_t)b * D, lane, vi);
    ld_row(VFo + (size_t)(d.B + b) * D, lane, vt);
    zero_row(acc);
    for (int r = 0; r < R1; ++r) {
        const int64_t tr = (int64_t)b * R1 + r;
        const int rt = r < d.C ? r : srow;
        ld_row(Yt + tr * D, lane, y);
        axpy_row(y, tsc[tr * DROP_NSC + 4], vi);
        axpy_row(y, tsc[tr * DROP_NSC + 5], vt);
        st_row(Yt + tr * D, lane, y);
        add_row(y, bf);
        fc_mask_row(g, da, (int64_t)b * L + (r < d.C ? 3 + r : 2), lane, m);
#pragma unroll
        for (int k = 0; k < 4; ++k) y[k] = mul4(y[k], m[k]);
        ld_row(S + (size_t)rt * D, lane, t); add_row(y, t);
        float rstd;
        ln_forward(y, gm, be, xh, rstd, o);
        if (r < d.C) add_row(acc, xh);
        else st_row(out_state + (size_t)b * D, lane, o);
    }
    const float invC = 1.0f / (float)d.C;
#pragma unroll
    for (int k = 0; k < 4; ++k) o[k] = fma4(mul4s(invC, acc[k]), gm[k], be[k]);
    st_row(out_proto + (size_t)b * D, lane, o);
}

// ------------------------------------------------------------------ backward of the own rows
// As ln_own_bwd_kernel, through the fc mask and the masked probabilities: dYo = mask .* du (the fc-output gradient),
// rowdot = dYo . Ybar (Ybar dropped), dsown = (aownd dA - aown rowdot) / tau; per-CTA partials of dgamma, dbeta, dbfc.
__global__ void __launch_bounds__(256)
drop_ln_own_bwd_kernel(HeadDims d, DropArgs da, const float* __restrict__ Ybo, const float* __restrict__ Xo,
                       const float* __restrict__ VFo, const float* __restrict__ aown, const float* __restrict__ aownd,
                       const float* __restrict__ bfc, const float* __restrict__ gamma, const float* __restrict__ beta,
                       const float* __restrict__ g_image, const float* __restrict__ g_text, float* __restrict__ dYo,
                       __nv_bfloat16* __restrict__ dYoh, float* __restrict__ dXo, float* __restrict__ rowdot,
                       float* __restrict__ dsown, float* __restrict__ dVFo, float* __restrict__ partials,
                       const float* __restrict__ g_own) {
    pdl_trigger();
    pdl_wait();
    __shared__ __align__(16) float fold[3][8][D];        // 48 KB
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Philox g = drop_stream(da, 1);
    float4 dgam[4], dbet[4], dbf[4], bf[4], gm[4], be[4];
    zero_row(dgam); zero_row(dbet); zero_row(dbf);
    ld_row(bfc, lane, bf); ld_row(gamma, lane, gm); ld_row(beta, lane, be);
    for (int b = blockIdx.x * 8 + warp; b < d.B; b += gridDim.x * 8) {
        float4 accI[4], accT[4], vi[4], vt[4];
        zero_row(accI); zero_row(accT);
        ld_row(VFo + (size_t)b * D, lane, vi);
        ld_row(VFo + (size_t)(d.B + b) * D, lane, vt);
#pragma unroll 1
        for (int which = 0; which < 2; ++which) {
            const int row = which ? d.B + b : b;
            float4 ybar[4], u[4], t[4], m[4], xh[4], o[4], du[4];
            ld_row(Ybo + (size_t)row * D, lane, ybar);
            fc_mask_row(g, da, (int64_t)b * da.L + which, lane, m);
#pragma unroll
            for (int k = 0; k < 4; ++k) u[k] = mul4(add4(ybar[k], bf[k]), m[k]);
            ld_row(Xo + (size_t)row * D, lane, t); add_row(u, t);
            float rstd;
            ln_forward(u, gm, be, xh, rstd, o);
            ld_row((which ? g_text : g_image) + (size_t)b * D, lane, u);
#pragma unroll
            for (int k = 0; k < 4; ++k) dgam[k] = fma4(u[k], xh[k], dgam[k]);
            add_row(dbet, u);
            ln_backward(u, xh, rstd, gm, du);
            if (g_own != nullptr) {
                ld_row(g_own + (size_t)row * D, lane, t);
                add_row(t, du);
                st_row(dXo + (size_t)row * D, lane, t);
            } else {
                st_row(dXo + (size_t)row * D, lane, du);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) du[k] = mul4(du[k], m[k]);
            add_row(dbf, du);
            st_row(dYo + (size_t)row * D, lane, du);
            st_row_h(dYoh != nullptr ? dYoh + (size_t)row * D : nullptr, lane, du);
            const float rd = warp_sum(dot_part(du, ybar));
            const float da_i = warp_sum(dot_part(du, vi));
            const float da_t = warp_sum(dot_part(du, vt));
            const float k0 = aownd[2 * row], k1 = aownd[2 * row + 1];
            if (lane == 0) {
                rowdot[row] = rd;
                dsown[2 * row] = (k0 * da_i - aown[2 * row] * rd) * INV_TAU;
                dsown[2 * row + 1] = (k1 * da_t - aown[2 * row + 1] * rd) * INV_TAU;
            }
            axpy_row(accI, k0, du);
            axpy_row(accT, k1, du);
        }
        st_row(dVFo + (size_t)b * D, lane, accI);
        st_row(dVFo + (size_t)(d.B + b) * D, lane, accT);
    }
    st_row(fold[0][warp], lane, dgam);
    st_row(fold[1][warp], lane, dbet);
    st_row(fold[2][warp], lane, dbf);
    __syncthreads();
    float* rec = partials + (size_t)blockIdx.x * OWN_PARTIAL_LEN;
    for (int i = threadIdx.x; i < 3 * D; i += blockDim.x) {
        const int q = i / D, c = i % D;
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += fold[q][w][c];
        rec[i] = s;
    }
}

// ------------------------------------------------------------------ backward of the table-query rows
// One warp per sample, its C + 1 rows in order: LayerNorm backward -> du (the residual gradient of the step row, dU) and
// dYt = mask .* du; rowdot = dYt . Ybar; own-key score gradients into dSK (every entry of the sample's two dSK rows is
// written); own-key part of dVF into dVFo (image and text row of the sample, complete rows); per-CTA partials of dgamma,
// dbeta, dbfc.  g_proto may be null (zero cotangent).
__global__ void __launch_bounds__(256)
drop_table_bwd_kernel(HeadDims d, DropArgs da, const float* __restrict__ Yt, float* __restrict__ tsc,
                      const float* __restrict__ VFo, const float* __restrict__ S, const float* __restrict__ bfc,
                      const float* __restrict__ gamma, const float* __restrict__ beta, const int64_t* __restrict__ state_ids,
                      const float* __restrict__ g_proto, const float* __restrict__ g_state, float* __restrict__ dYt,
                      __nv_bfloat16* __restrict__ dYth, float* __restrict__ dU, float* __restrict__ dSK,
                      __nv_bfloat16* __restrict__ dSKh, float* __restrict__ dVFo, float* __restrict__ partials) {
    pdl_trigger();
    pdl_wait();
    __shared__ __align__(16) float fold[3][8][D];        // 48 KB
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const Philox g = drop_stream(da, 1);
    const int R1 = d.C + 1;
    const float invC = 1.0f / (float)d.C;
    float4 dgam[4], dbet[4], dbf[4];
    zero_row(dgam); zero_row(dbet); zero_row(dbf);
    for (int b = blockIdx.x * 8 + warp; b < d.B; b += gridDim.x * 8) {
        const int srow = d.M + clamp_state(state_ids[b]);
        for (int j = lane; j < d.Nsp; j += 32) {
            dSK[(size_t)b * d.Nsp + j] = 0.f; dSK[(size_t)(d.B + b) * d.Nsp + j] = 0.f;
            if (dSKh != nullptr) { dSKh[(size_t)b * d.Nsp + j] = __float2bfloat16_rn(0.f); dSKh[(size_t)(d.B + b) * d.Nsp + j] = __float2bfloat16_rn(0.f); }
        }
        __syncwarp();
        float4 accI[4], accT[4], vi[4], vt[4];
        zero_row(accI); zero_row(accT);
        ld_row(VFo + (size_t)b * D, lane, vi);
        ld_row(VFo + (size_t)(d.B + b) * D, lane, vt);
#pragma unroll 1
        for (int r = 0; r < R1; ++r) {
            const int64_t tr = (int64_t)b * R1 + r;
            const int rt = r < d.C ? r : srow;
            float4 ybar[4], u[4], t[4], m[4], xh[4], du[4];
            ld_row(Yt + tr * D, lane, ybar);
            fc_mask_row(g, da, (int64_t)b * da.L + (r < d.C ? 3 + r : 2), lane, m);
            ld_row(bfc, lane, t);
#pragma unroll
            for (int k = 0; k < 4; ++k) u[k] = mul4(add4(ybar[k], t[k]), m[k]);
            ld_row(S + (size_t)rt * D, lane, t); add_row(u, t);
            const float mean = warp_sum(sum_part(u)) * (1.0f / D);
#pragma unroll
            for (int k = 0; k < 4; ++k) xh[k] = add4s(-mean, u[k]);
            const float rstd = 1.0f / sqrtf(warp_sum(dot_part(xh, xh)) * (1.0f / D) + LN_EPS);
            scale_row(xh, rstd);
            if (r < d.C) {                     // go = g_proto / C (zero when g_proto is null)
                if (g_proto != nullptr) { ld_row(g_proto + (size_t)b * D, lane, u); scale_row(u, invC); } else { zero_row(u); }
            } else {
                ld_row(g_state + (size_t)b * D, lane, u);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) dgam[k] = fma4(u[k], xh[k], dgam[k]);
            add_row(dbet, u);
            ld_row(gamma, lane, t);
            ln_backward(u, xh, rstd, t, du);
            st_row(dU + tr * D, lane, du);
#pragma unroll
            for (int k = 0; k < 4; ++k) du[k] = mul4(du[k], m[k]);
            add_row(dbf, du);
            st_row(dYt + tr * D, lane, du);
            st_row_h(dYth != nullptr ? dYth + tr * D : nullptr, lane, du);
            const float rd = warp_sum(dot_part(du, ybar));
            const float da_i = warp_sum(dot_part(du, vi));
            const float da_t = warp_sum(dot_part(du, vt));
            const float* sc = tsc + tr * DROP_NSC;
            const float a_i = sc[1], a_t = sc[2], k_i = sc[4], k_t = sc[5];
            if (lane == 0) {
                const float ds_i = (k_i * da_i - a_i * rd) * INV_TAU, ds_t = (k_t * da_t - a_t * rd) * INV_TAU;
                dSK[(size_t)b * d.Nsp + rt] = ds_i;
                dSK[(size_t)(d.B + b) * d.Nsp + rt] = ds_t;
                if (dSKh != nullptr) { dSKh[(size_t)b * d.Nsp + rt] = __float2bfloat16_rn(ds_i); dSKh[(size_t)(d.B + b) * d.Nsp + rt] = __float2bfloat16_rn(ds_t); }
                tsc[tr * DROP_NSC + 6] = rd;
            }
            axpy_row(accI, k_i, du);
            axpy_row(accT, k_t, du);
        }
        st_row(dVFo + (size_t)b * D, lane, accI);
        st_row(dVFo + (size_t)(d.B + b) * D, lane, accT);
    }
    st_row(fold[0][warp], lane, dgam);
    st_row(fold[1][warp], lane, dbet);
    st_row(fold[2][warp], lane, dbf);
    __syncthreads();
    float* rec = partials + (size_t)blockIdx.x * OWN_PARTIAL_LEN;
    for (int i = threadIdx.x; i < 3 * D; i += blockDim.x) {
        const int q = i / D, c = i % D;
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += fold[q][w][c];
        rec[i] = s;
    }
}

// dS = (Ad .* dA - Aext rowdot) / tau in place over dA (fp32 + bf16 shadow); the own-query softmax backward through the mask
__global__ void __launch_bounds__(256)
drop_ds_kernel(int64_t n4, int Nsp4, const float* __restrict__ Aext, const float* __restrict__ Ad, const float* __restrict__ rowdot,
               float* __restrict__ dA, __nv_bfloat16* __restrict__ dSh, int write_f) {
    pdl_trigger();
    pdl_wait();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const float rd = rowdot[i / Nsp4];
    const float4 a = reinterpret_cast<const float4*>(Aext)[i], k = reinterpret_cast<const float4*>(Ad)[i];
    float4 v = reinterpret_cast<const float4*>(dA)[i];
    v.x = (k.x * v.x - a.x * rd) * INV_TAU; v.y = (k.y * v.y - a.y * rd) * INV_TAU;
    v.z = (k.z * v.z - a.z * rd) * INV_TAU; v.w = (k.w * v.w - a.w * rd) * INV_TAU;
    if (write_f) reinterpret_cast<float4*>(dA)[i] = v;
    if (dSh != nullptr) reinterpret_cast<uint2*>(dSh)[i] = pack_bf16x4(v);
}

// ------------------------------------------------------------------ fixed-order batch folds of the table-query rows
// blocks [0, tt_blocks): thread = (step row q, column j) of dTT: sum over the samples (in order) of the score gradient
//   (Wd dWd - A rowdot) / tau of the table row that queries with step row q (prototype q < C: every sample; state row
//   M + s: the samples with state s); other step rows 0.  fp32 + bf16 shadow.
// blocks [tt_blocks, tt_blocks + Nsp): step row q of Rfull = the residual gradients dU of the same rows, summed in order.
// last block: dgamma, dbeta (table + own partials, in order) and dbfc_parts[0] (the rest of dbfc_parts zero).
__global__ void __launch_bounds__(256)
drop_fold_kernel(HeadDims d, int tt_blocks, const float* __restrict__ Wd, const float* __restrict__ dWd,
                 const float* __restrict__ Pt, const float* __restrict__ tsc, const int64_t* __restrict__ state_ids,
                 const float* __restrict__ dU, const float* __restrict__ tpart, int ntp, const float* __restrict__ opart, int nop,
                 float* __restrict__ dTT, __nv_bfloat16* __restrict__ dTTh, float* __restrict__ Rfull,
                 float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ dbfc_parts) {
    pdl_trigger();
    pdl_wait();
    const int R1 = d.C + 1;
    if ((int)blockIdx.x < tt_blocks) {
        const int e = blockIdx.x * 256 + threadIdx.x;
        if (e >= d.Nsp * d.Nsp) return;
        const int q = e / d.Nsp, j = e % d.Nsp;
        const bool proto = q < d.C, state = q >= d.M && q < d.Ns;
        float s = 0.f;
        if (proto || state) {
            const int r = proto ? q : d.C;
            const float p = j < d.M ? Pt[(size_t)q * d.Nsp + j] : 0.f;
            for (int b = 0; b < d.B; ++b) {
                const int scol = d.M + clamp_state(state_ids[b]);
                if (state && scol != q) continue;
                const int64_t t = (int64_t)b * R1 + r;
                const float* sc = tsc + t * DROP_NSC;
                const float a = j < d.M ? p * sc[0] : (j == scol ? sc[3] : 0.f);
                s += (Wd[t * d.Nsp + j] * dWd[t * d.Nsp + j] - a * sc[6]) * INV_TAU;
            }
        }
        dTT[e] = s;
        if (dTTh != nullptr) dTTh[e] = __float2bfloat16_rn(s);
        return;
    }
    const int t = threadIdx.x;
    if ((int)blockIdx.x < tt_blocks + d.Nsp) {
        const int q = (int)blockIdx.x - tt_blocks;
        if (t >= D / 4) return;
        const bool proto = q < d.C, state = q >= d.M && q < d.Ns;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        if (proto || state) {
            const int r = proto ? q : d.C;
            for (int b = 0; b < d.B; ++b) {
                if (state && d.M + clamp_state(state_ids[b]) != q) continue;
                const float4 v = reinterpret_cast<const float4*>(dU + ((int64_t)b * R1 + r) * D)[t];
                s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
            }
        }
        reinterpret_cast<float4*>(Rfull + (size_t)q * D)[t] = s;
        return;
    }
    for (int c = t; c < D; c += blockDim.x) {
        float v[3];
        for (int k = 0; k < 3; ++k) {
            float s = 0.f;
            for (int p = 0; p < ntp; ++p) s += tpart[(size_t)p * OWN_PARTIAL_LEN + k * D + c];
            for (int p = 0; p < nop; ++p) s += opart[(size_t)p * OWN_PARTIAL_LEN + k * D + c];
            v[k] = s;
        }
        dgamma[c] = v[0]; dbeta[c] = v[1]; dbfc_parts[c] = v[2];
        for (int q = 1; q < EXP_SUM_BLOCKS; ++q) dbfc_parts[(size_t)q * D + c] = 0.f;
    }
}

}  // namespace team
