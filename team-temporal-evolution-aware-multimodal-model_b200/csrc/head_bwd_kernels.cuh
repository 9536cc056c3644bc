// Backward kernels of the fusion head (hand-written VJP of head_fwd_kernels.cuh; replaces
// autograd through utils/inc_net.py:528-580 + convs/projections.py:64-87 at models/proof.py:444).
// All batch reductions (shared-row gradients, LayerNorm/bias gradients) are two-pass and
// fixed-order: per-CTA partial records, then reduce_partials_kernel -> bit-reproducible.
#pragma once
#include "head_fwd_kernels.cuh"

namespace team {

// ---- per-CTA partial record of table_rows_bwd (floats): [dvfst 10xD][dgam D][dbet D][scal Rt x TQ_NSC]
// scal row tr (table-query row: tr < C prototype row, tr = C + s the state row of state s):
//   0..3  R coefficients: sum_b alpha*m1, sum_b beta*cw, sum_b beta, sum_b beta*mean
//   4..7  the same, each term weighted by cw (G coefficients)
//   8     h:  sum_b cw * <dY, Ybar>
//   10..19 dTT state columns, 20..29 sum_b beta*a_s by state (R), 30..39 the same weighted by cw (G)
constexpr int TQ_NSC = 40;
struct TabOff {
    size_t dvfst, dgam, dbet, scal, len;
};
__host__ __device__ inline TabOff tab_offsets(const HeadDims& d) {
    TabOff o;
    o.dvfst = 0;
    o.dgam = (size_t)10 * D;
    o.dbet = o.dgam + D;
    o.scal = o.dbet + D;
    o.len = (o.scal + (size_t)d.Rt * TQ_NSC + 3) / 4 * 4;
    return o;
}
__host__ __device__ inline size_t table_bwd_smem_floats(const HeadDims& d) {
    return (size_t)(5 + 2 + 4 * TQ_WARPS + 1 + 10) * D + (size_t)d.Rt * TQ_NSC + 16;
}

// ------------------------------------------------------------------ table-query rows, backward
// Same work split as table_rows_fwd_kernel (one sample per CTA iteration, warp w owns rows w, w+4, ...).
// Per row it recomputes the forward (Ybar, LayerNorm), forms dY = LN-backward of the row's cotangent and emits
//   * the score gradients of the three own keys (dSK, dTT state columns),
//   * the per-sample sums  sum_j a_i dY, sum_j a_t dY (-> dVFo) and sum_j a_s dY (-> dVF of the state-table row),
//   * LayerNorm gamma/beta gradients,
// and, instead of accumulating the batch reductions R_r = sum_b dY_br and G_r = sum_b cw_br dY_br as 512-wide
// vectors, their COEFFICIENTS:  dY = alpha (gg - m1) - beta (u - mean)  with  u = cw NF_r + S_r + bfc + a_i VI_b +
// a_t VT_b + a_s VS_b,  so  R = A1^T GG + A23^T VFo  (one two-segment tensor-core GEMM, K = 2B each) plus
// rank-1 / table-row corrections assembled from the scalar sums in `scal` (expand_table_kernel).
// A1 / A23 are [2B, ldA]: column tr holds the R coefficient, column ldA/2 + tr the G coefficient.
// g_proto = NULL is a zero prototype cotangent: the prototype rows are still visited, with dY = 0 (a branch that skips
// them makes ptxas spill more of this register-bound kernel).
// dynamic smem: vec[5][D] (VI, VT, VS, gamma.*g_proto/C, gamma.*g_state) | lnp[2][D] (gamma, bfc) | slots[TQ_WARPS][4][D] | xst[D] |
//               dvfst[10][D] | scal[Rt][TQ_NSC] | red[16]
__global__ void __launch_bounds__(TQ_WARPS * 32, 3)
table_rows_bwd_kernel(HeadDims d, const float* __restrict__ SK, const float* __restrict__ TT,
                      const float* __restrict__ mt, const float* __restrict__ Zt, const float* __restrict__ NFt,
                      const float* __restrict__ VFo, const float* __restrict__ VFs, const float* __restrict__ S,
                      const float* __restrict__ bfc, const float* __restrict__ gamma,
                      const int64_t* __restrict__ state_ids, const float* __restrict__ g_proto,
                      const float* __restrict__ g_state, float* __restrict__ dSK, __nv_bfloat16* __restrict__ dSKh,
                      float* __restrict__ dVFo, float* __restrict__ GG, __nv_bfloat16* __restrict__ GGh,
                      float* __restrict__ A1, __nv_bfloat16* __restrict__ A1h, float* __restrict__ A23,
                      __nv_bfloat16* __restrict__ A23h, int ldA, float* __restrict__ partials) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) float tb_smem[];
    float* vec = tb_smem;                                     // [5][D]
    float* lnp = vec + 5 * D;                                 // [2][D]
    float* slots = lnp + 2 * D;                               // [TQ_WARPS][4][D]
    float* xst = slots + 4 * TQ_WARPS * D;                    // [D]
    float* dvfst = xst + D;                                   // [10][D]
    float* scal = dvfst + 10 * D;                             // [Rt][TQ_NSC]
    float* red = scal + d.Rt * TQ_NSC;                        // [16]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const TabOff off = tab_offsets(d);
    const int gcol = ldA / 2;
    for (int i = tid; i < 10 * D; i += blockDim.x) dvfst[i] = 0.f;
    for (int i = tid; i < d.Rt * TQ_NSC; i += blockDim.x) scal[i] = 0.f;
    reinterpret_cast<float4*>(lnp)[tid] = reinterpret_cast<const float4*>(gamma)[tid];
    reinterpret_cast<float4*>(lnp + D)[tid] = reinterpret_cast<const float4*>(bfc)[tid];
    float4 dgam = make_float4(0.f, 0.f, 0.f, 0.f), dbet = dgam;         // float4 column tid
    const int nrows = d.C + 1 > warp ? (d.C + 1 - warp + TQ_WARPS - 1) / TQ_WARPS : 0;
    const float invC = d.C > 1 ? 1.0f / (float)d.C : 1.0f;
    const __nv_bfloat16 hz = __float2bfloat16_rn(0.f);
    for (int b = blockIdx.x; b < d.B; b += gridDim.x) {
        const int sid = clamp_state(state_ids[b]);
        const int srow = d.M + sid;
        float4 gp_raw, gs_raw;                                // this thread's float4 column of g_proto/C and g_state
        __syncthreads();                                      // previous sample's slots / vec fully consumed
        {   // stage the sample's vectors; GG rows (cotangent .* gamma) for the coefficient GEMM; zero the sparse rows
            const float4 g4 = reinterpret_cast<const float4*>(lnp)[tid];
            float4 gp = g_proto != nullptr ? reinterpret_cast<const float4*>(g_proto + (size_t)b * D)[tid] : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 gs = reinterpret_cast<const float4*>(g_state + (size_t)b * D)[tid];
            gp.x *= invC; gp.y *= invC; gp.z *= invC; gp.w *= invC;
            reinterpret_cast<float4*>(vec)[tid] = reinterpret_cast<const float4*>(VFo + (size_t)b * D)[tid];
            reinterpret_cast<float4*>(vec + D)[tid] = reinterpret_cast<const float4*>(VFo + (size_t)(d.B + b) * D)[tid];
            reinterpret_cast<float4*>(vec + 2 * D)[tid] = reinterpret_cast<const float4*>(VFs + (size_t)srow * D)[tid];
            const float4 ggp = mul4(gp, g4), ggs = mul4(gs, g4);
            reinterpret_cast<float4*>(vec + 3 * D)[tid] = ggp;
            reinterpret_cast<float4*>(vec + 4 * D)[tid] = ggs;
            gp_raw = gp; gs_raw = gs;
            reinterpret_cast<float4*>(GG + (size_t)b * D)[tid] = ggp;
            reinterpret_cast<float4*>(GG + (size_t)(d.B + b) * D)[tid] = ggs;
            if (GGh != nullptr) {
                reinterpret_cast<uint2*>(GGh + (size_t)b * D)[tid] = pack_bf16x4(ggp);
                reinterpret_cast<uint2*>(GGh + (size_t)(d.B + b) * D)[tid] = pack_bf16x4(ggs);
            }
            const float sp = warp_sum(ggp.x + ggp.y + ggp.z + ggp.w), ss = warp_sum(ggs.x + ggs.y + ggs.z + ggs.w);
            if (lane == 0) { red[2 * warp] = sp; red[2 * warp + 1] = ss; }
            dbet.x += gp.x * d.C + gs.x; dbet.y += gp.y * d.C + gs.y; dbet.z += gp.z * d.C + gs.z; dbet.w += gp.w * d.C + gs.w;
            for (int i = tid; i < d.Nsp; i += blockDim.x) {
                dSK[(size_t)b * d.Nsp + i] = 0.f;
                dSK[(size_t)(d.B + b) * d.Nsp + i] = 0.f;
                if (dSKh != nullptr) { dSKh[(size_t)b * d.Nsp + i] = hz; dSKh[(size_t)(d.B + b) * d.Nsp + i] = hz; }
            }
            for (int i = tid; i < ldA; i += blockDim.x) {
                A1[(size_t)b * ldA + i] = 0.f; A1[(size_t)(d.B + b) * ldA + i] = 0.f;
                A23[(size_t)b * ldA + i] = 0.f; A23[(size_t)(d.B + b) * ldA + i] = 0.f;
                if (A1h != nullptr) {
                    A1h[(size_t)b * ldA + i] = hz; A1h[(size_t)(d.B + b) * ldA + i] = hz;
                    A23h[(size_t)b * ldA + i] = hz; A23h[(size_t)(d.B + b) * ldA + i] = hz;
                }
            }
        }
        __syncthreads();
        float m1p = 0.f, m1s = 0.f;
#pragma unroll
        for (int w = 0; w < TQ_WARPS; ++w) { m1p += red[2 * w]; m1s += red[2 * w + 1]; }
        m1p *= (1.0f / D); m1s *= (1.0f / D);
        float4 acc_i[4], acc_t[4], acc_s[4], xs[4];
        zero_row(acc_i); zero_row(acc_t); zero_row(acc_s); zero_row(xs);
        for (int k0 = 0; k0 < nrows; k0 += 32) {
            TableRowW mine;
            mine.c_w = mine.a_i = mine.a_t = mine.a_s = 0.f; mine.r = 0;
            if (k0 + lane < nrows) mine = table_row_weights(d, b, warp + (k0 + lane) * TQ_WARPS, srow, SK, TT, mt, Zt);
            const int kn = min(32, nrows - k0);
            float k_alpha = 0.f, k_beta = 0.f, k_mean = 0.f, k_m1 = 0.f, k_yy = 0.f, k_i = 0.f, k_t = 0.f, k_s = 0.f;
            for (int k = 0; k < kn; ++k) {
                const TableRowW rw = shfl_row_weights(mine, k);
                const int j = warp + (k0 + k) * TQ_WARPS;
                const bool is_proto = j < d.C;
                float4 ybar[4], xh[4], t[4];
                ld_row(NFt + (size_t)rw.r * D, lane, ybar); scale_row(ybar, rw.c_w);
                ld_row(vec, lane, t); axpy_row(ybar, rw.a_i, t);
                ld_row(vec + D, lane, t); axpy_row(ybar, rw.a_t, t);
                ld_row(vec + 2 * D, lane, t); axpy_row(ybar, rw.a_s, t);
                ld_row(S + (size_t)rw.r * D, lane, xh); add_row(xh, ybar);
                ld_row(lnp + D, lane, t); add_row(xh, t);
                const float mean = warp_sum(sum_part(xh)) * (1.0f / D);
                shift_row(xh, -mean);
                const float var = warp_sum(dot_part(xh, xh)) * (1.0f / D);
                const float rstd = 1.0f / sqrtf(var + LN_EPS);
                scale_row(xh, rstd);
                // gg = cotangent .* gamma (staged) ; dY = rstd (gg - m1 - xh m2)
                float4 gg[4];
                ld_row(vec + (is_proto ? 3 : 4) * D, lane, gg);
                const float m1 = is_proto ? m1p : m1s;
                const float m2 = warp_sum(dot_part(gg, xh)) * (1.0f / D);
#pragma unroll
                for (int i = 0; i < 4; ++i) gg[i] = mul4s(rstd, fma4s(-m2, xh[i], add4s(-m1, gg[i])));
                float p_yy = dot_part(gg, ybar);
                ld_row(vec, lane, t);
                float p_i = dot_part(gg, t);
                axpy_row(acc_i, rw.a_i, gg);
                ld_row(vec + D, lane, t);
                float p_t = dot_part(gg, t);
                axpy_row(acc_t, rw.a_t, gg);
                ld_row(vec + 2 * D, lane, t);
                float p_s = dot_part(gg, t);
                axpy_row(acc_s, rw.a_s, gg);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {            // four reductions interleaved
                    p_yy += __shfl_xor_sync(0xffffffffu, p_yy, o); p_i += __shfl_xor_sync(0xffffffffu, p_i, o);
                    p_t += __shfl_xor_sync(0xffffffffu, p_t, o); p_s += __shfl_xor_sync(0xffffffffu, p_s, o);
                }
                if (is_proto) add_row(xs, xh); else st_row(xst, lane, xh);
                if (lane == k) {                              // lane k keeps the (warp-uniform) scalars of its row
                    k_alpha = rstd; k_beta = rstd * rstd * m2; k_mean = mean; k_m1 = m1;
                    k_yy = p_yy; k_i = p_i; k_t = p_t; k_s = p_s;
                }
            }
            // scalar outputs of the chunk's rows, one row per lane
            if (lane < kn) {
                const int j = warp + (k0 + lane) * TQ_WARPS;
                const bool is_proto = j < d.C;
                const int tr = is_proto ? j : d.C + sid;
                const float cw = mine.c_w;
                const float v_i = mine.a_i * (k_i - k_yy) * INV_TAU, v_t = mine.a_t * (k_t - k_yy) * INV_TAU;
                dSK[(size_t)b * d.Nsp + mine.r] = v_i;
                dSK[(size_t)(d.B + b) * d.Nsp + mine.r] = v_t;
                if (dSKh != nullptr) {
                    dSKh[(size_t)b * d.Nsp + mine.r] = __float2bfloat16_rn(v_i);
                    dSKh[(size_t)(d.B + b) * d.Nsp + mine.r] = __float2bfloat16_rn(v_t);
                }
                const size_t ra = (size_t)(is_proto ? b : d.B + b) * ldA;        // GG row this query's cotangent lives in
                const size_t r0 = (size_t)b * ldA, r1 = (size_t)(d.B + b) * ldA;
                const float c23i = -k_beta * mine.a_i, c23t = -k_beta * mine.a_t;
                A1[ra + tr] = k_alpha; A1[ra + gcol + tr] = cw * k_alpha;
                A23[r0 + tr] = c23i; A23[r0 + gcol + tr] = cw * c23i;
                A23[r1 + tr] = c23t; A23[r1 + gcol + tr] = cw * c23t;
                if (A1h != nullptr) {
                    A1h[ra + tr] = __float2bfloat16_rn(k_alpha); A1h[ra + gcol + tr] = __float2bfloat16_rn(cw * k_alpha);
                    A23h[r0 + tr] = __float2bfloat16_rn(c23i); A23h[r0 + gcol + tr] = __float2bfloat16_rn(cw * c23i);
                    A23h[r1 + tr] = __float2bfloat16_rn(c23t); A23h[r1 + gcol + tr] = __float2bfloat16_rn(cw * c23t);
                }
                float* sc = scal + tr * TQ_NSC;               // row tr is only ever touched by this lane's warp
                const float e0 = k_alpha * k_m1, e1 = k_beta * cw, e2 = k_beta, e3 = k_beta * k_mean, e4 = k_beta * mine.a_s;
                sc[0] += e0; sc[1] += e1; sc[2] += e2; sc[3] += e3;
                sc[4] += cw * e0; sc[5] += cw * e1; sc[6] += cw * e2; sc[7] += cw * e3;
                sc[8] += cw * k_yy;
                sc[10 + sid] += mine.a_s * (k_s - k_yy) * INV_TAU;
                sc[20 + sid] += e4;
                sc[30 + sid] += cw * e4;
            }
            __syncwarp();
        }
        st_row(slots + (warp * 4 + 0) * D, lane, acc_i);
        st_row(slots + (warp * 4 + 1) * D, lane, acc_t);
        st_row(slots + (warp * 4 + 2) * D, lane, acc_s);
        st_row(slots + (warp * 4 + 3) * D, lane, xs);
        __syncthreads();
        {
            float4 f[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                f[q] = reinterpret_cast<const float4*>(slots + q * D)[tid];
#pragma unroll
                for (int w = 1; w < TQ_WARPS; ++w) {
                    const float4 a = reinterpret_cast<const float4*>(slots + (w * 4 + q) * D)[tid];
                    f[q].x += a.x; f[q].y += a.y; f[q].z += a.z; f[q].w += a.w;
                }
            }
            reinterpret_cast<float4*>(dVFo + (size_t)b * D)[tid] = f[0];
            reinterpret_cast<float4*>(dVFo + (size_t)(d.B + b) * D)[tid] = f[1];
            float4 o = reinterpret_cast<float4*>(dvfst + sid * D)[tid];
            o.x += f[2].x; o.y += f[2].y; o.z += f[2].z; o.w += f[2].w;
            reinterpret_cast<float4*>(dvfst + sid * D)[tid] = o;
            // dgamma += (g_proto/C) .* sum_{j<C} xhat_j + g_state .* xhat_state
            const float4 xq = reinterpret_cast<const float4*>(xst)[tid];
            dgam = fma4(gp_raw, f[3], fma4(gs_raw, xq, dgam));
        }
    }
    __syncthreads();
    float* rec = partials + (size_t)blockIdx.x * off.len;
    for (int i = tid; i < 10 * D; i += blockDim.x) rec[off.dvfst + i] = dvfst[i];
    reinterpret_cast<float4*>(rec + off.dgam)[tid] = dgam;
    reinterpret_cast<float4*>(rec + off.dbet)[tid] = dbet;
    for (int i = tid; i < d.Rt * TQ_NSC; i += blockDim.x) rec[off.scal + i] = scal[i];
    for (size_t i = off.scal + (size_t)d.Rt * TQ_NSC + tid; i < off.len; i += blockDim.x) rec[i] = 0.f;
}

// out[i] = sum_p partials[p][i] in fixed order (RP_GROUPS interleaved lanes of p, folded in order); up to two
// independent jobs per launch (blocks [0, blocks0) -> job 0, the rest -> job 1).
struct ReduceJob {
    const float* partials;
    float* out;
    size_t len4;
    int n_partials;
};
struct ReduceJobs {
    ReduceJob j[2];
    int blocks0;
};
constexpr int RP_COLS = 32;       // float4 columns per block
constexpr int RP_GROUPS = 32;     // partial-interleaved groups per block
__global__ void __launch_bounds__(RP_COLS * RP_GROUPS)
reduce_partials_kernel(const __grid_constant__ ReduceJobs rj) {
    pdl_trigger();
    pdl_wait();
    __shared__ float4 fold[RP_GROUPS][RP_COLS];
    const bool second = (int)blockIdx.x >= rj.blocks0;
    const ReduceJob& job = rj.j[second ? 1 : 0];
    const int c = threadIdx.x % RP_COLS, g = threadIdx.x / RP_COLS;
    const size_t i = (size_t)((int)blockIdx.x - (second ? rj.blocks0 : 0)) * RP_COLS + c;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < job.len4) {
        const float4* base = reinterpret_cast<const float4*>(job.partials) + i;
        int p = g;
        for (; p + 3 * RP_GROUPS < job.n_partials; p += 4 * RP_GROUPS) {       // 4 loads in flight
            float4 a[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) a[q] = base[(size_t)(p + q * RP_GROUPS) * job.len4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { s.x += a[q].x; s.y += a[q].y; s.z += a[q].z; s.w += a[q].w; }
        }
        for (; p < job.n_partials; p += RP_GROUPS) {
            const float4 a = base[(size_t)p * job.len4];
            s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
        }
    }
    fold[g][c] = s;
    __syncthreads();
    if (g == 0 && i < job.len4) {
        float4 r = fold[0][c];
        for (int q = 1; q < RP_GROUPS; ++q) { r.x += fold[q][c].x; r.y += fold[q][c].y; r.z += fold[q][c].z; r.w += fold[q][c].w; }
        reinterpret_cast<float4*>(job.out)[i] = r;
    }
}

constexpr int EXP_SUM_BLOCKS = 8;
__device__ __forceinline__ void combine_table_row(const HeadDims& d, const TabOff& off, const float* __restrict__ red,
        const float* __restrict__ RG, int gcol, const float* __restrict__ NFt, const float* __restrict__ S,
        const float* __restrict__ VFs, const float4 bf, int tr, int r, int t, float4& Rv, float4& Gv) {
    const float* sc = red + off.scal + (size_t)tr * TQ_NSC;
    const float4 nf = reinterpret_cast<const float4*>(NFt + (size_t)r * D)[t];
    float4 sb = reinterpret_cast<const float4*>(S + (size_t)r * D)[t];
    sb.x += bf.x; sb.y += bf.y; sb.z += bf.z; sb.w += bf.w;
    Rv = reinterpret_cast<const float4*>(RG + (size_t)tr * D)[t];
    Gv = reinterpret_cast<const float4*>(RG + (size_t)(gcol + tr) * D)[t];
    const float r0 = sc[3] - sc[0], g0 = sc[7] - sc[4];
    Rv.x += r0 - sc[1] * nf.x - sc[2] * sb.x; Rv.y += r0 - sc[1] * nf.y - sc[2] * sb.y;
    Rv.z += r0 - sc[1] * nf.z - sc[2] * sb.z; Rv.w += r0 - sc[1] * nf.w - sc[2] * sb.w;
    Gv.x += g0 - sc[5] * nf.x - sc[6] * sb.x; Gv.y += g0 - sc[5] * nf.y - sc[6] * sb.y;
    Gv.z += g0 - sc[5] * nf.z - sc[6] * sb.z; Gv.w += g0 - sc[5] * nf.w - sc[6] * sb.w;
    for (int s = 0; s < 10; ++s) {
        const float wr = sc[20 + s], wg = sc[30 + s];
        if (wr == 0.f && wg == 0.f) continue;
        const float4 v = reinterpret_cast<const float4*>(VFs + (size_t)(d.M + s) * D)[t];
        Rv.x -= wr * v.x; Rv.y -= wr * v.y; Rv.z -= wr * v.z; Rv.w -= wr * v.w;
        Gv.x -= wg * v.x; Gv.y -= wg * v.y; Gv.z -= wg * v.z; Gv.w -= wg * v.w;
    }
}

__global__ void __launch_bounds__(128)
expand_table_kernel(HeadDims d, const float* __restrict__ red, const float* __restrict__ own_red,
                    const float* __restrict__ RG, int gcol, const float* __restrict__ NFt, const float* __restrict__ S,
                    const float* __restrict__ VFs, const float* __restrict__ bfc,
                    float* __restrict__ Rfull, float* __restrict__ Gfull, __nv_bfloat16* __restrict__ Gfullh,
                    float* __restrict__ hfull, float* __restrict__ dTT, float* __restrict__ dVFs,
                    const float* __restrict__ dVFs_a, float* __restrict__ dgamma, float* __restrict__ dbeta,
                    float* __restrict__ dbfc_parts) {
    pdl_trigger();
    pdl_wait();
    const TabOff off = tab_offsets(d);
    const int r = blockIdx.x, t = threadIdx.x;
    const float4 bf = reinterpret_cast<const float4*>(bfc)[t];
    if (r >= d.Nsp) {
        // blocks Nsp .. Nsp+EXP_SUM_BLOCKS-1: fixed-order partial sums of R over the table rows (-> dbfc, finish_bwd_kernel);
        // the first of them also folds dgamma / dbeta
        const int q = r - d.Nsp;
        if (q == 0) {
            const float4 a = reinterpret_cast<const float4*>(red + off.dgam)[t], b = reinterpret_cast<const float4*>(own_red)[t];
            reinterpret_cast<float4*>(dgamma)[t] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
            const float4 c = reinterpret_cast<const float4*>(red + off.dbet)[t], e = reinterpret_cast<const float4*>(own_red + D)[t];
            reinterpret_cast<float4*>(dbeta)[t] = make_float4(c.x + e.x, c.y + e.y, c.z + e.z, c.w + e.w);
        }
        float4 s = q == 0 ? reinterpret_cast<const float4*>(own_red + 2 * D)[t] : make_float4(0.f, 0.f, 0.f, 0.f);
        for (int tr = q; tr < d.Rt; tr += EXP_SUM_BLOCKS) {
            float4 Rv, Gv;
            combine_table_row(d, off, red, RG, gcol, NFt, S, VFs, bf, tr, tr < d.C ? tr : d.M + (tr - d.C), t, Rv, Gv);
            s.x += Rv.x; s.y += Rv.y; s.z += Rv.z; s.w += Rv.w;
        }
        reinterpret_cast<float4*>(dbfc_parts + (size_t)q * D)[t] = s;
        return;
    }
    const bool is_state = r >= d.M && r < d.Ns;
    const int tr = r < d.C ? r : (is_state ? d.C + (r - d.M) : -1);
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 Rv = z, Gv = z;
    if (tr >= 0) combine_table_row(d, off, red, RG, gcol, NFt, S, VFs, bf, tr, r, t, Rv, Gv);
    reinterpret_cast<float4*>(Rfull + (size_t)r * D)[t] = Rv;
    reinterpret_cast<float4*>(Gfull + (size_t)r * D)[t] = Gv;
    if (Gfullh != nullptr) reinterpret_cast<uint2*>(Gfullh + (size_t)r * D)[t] = pack_bf16x4(Gv);
    {   // dVFs = Aext^T dYo (wave 5) + the state-table part of the table rows; wave 6 adds Pt^T G
        float4 v = reinterpret_cast<const float4*>(dVFs_a + (size_t)r * D)[t];
        if (is_state) {
            const float4 a = reinterpret_cast<const float4*>(red + off.dvfst + (size_t)(r - d.M) * D)[t];
            v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
        }
        reinterpret_cast<float4*>(dVFs + (size_t)r * D)[t] = v;
    }
    if (t == 0) hfull[r] = tr >= 0 ? red[off.scal + (size_t)tr * TQ_NSC + 8] : 0.f;
    for (int j = t; j < d.Nsp; j += blockDim.x)
        dTT[(size_t)r * d.Nsp + j] = (tr >= 0 && j >= d.M && j < d.Ns) ? red[off.scal + (size_t)tr * TQ_NSC + 10 + (j - d.M)] : 0.f;
}

// ------------------------------------------------------------------ own rows: LayerNorm + softmax-output backward
__global__ void __launch_bounds__(256)
ln_own_bwd_kernel(HeadDims d, const float* __restrict__ Ybo, const float* __restrict__ Xo,
                  const float* __restrict__ VFo, const float* __restrict__ aown, const float* __restrict__ bfc,
                  const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ g_image,
                  const float* __restrict__ g_text, float* __restrict__ dYo, __nv_bfloat16* __restrict__ dYoh,
                  float* __restrict__ dXo, float* __restrict__ rowdot, float* __restrict__ dsown,
                  float* __restrict__ dVFo, __nv_bfloat16* __restrict__ dVFoh, float* __restrict__ partials,
                  const float* __restrict__ g_own) {
    pdl_trigger();
    pdl_wait();
    __shared__ __align__(16) float fold[3][8][D];        // 48 KB
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4 dgam[4], dbet[4], dbf[4];
    zero_row(dgam); zero_row(dbet); zero_row(dbf);
    for (int b = blockIdx.x * 8 + warp; b < d.B; b += gridDim.x * 8) {
        float4 accI[4], accT[4], vi[4], vt[4];
        zero_row(accI); zero_row(accT);
        ld_row(VFo + (size_t)b * D, lane, vi);
        ld_row(VFo + (size_t)(d.B + b) * D, lane, vt);
#pragma unroll 1
        for (int which = 0; which < 2; ++which) {
            const int row = which ? d.B + b : b;
            float4 ybar[4], u[4], t[4], xh[4], du[4];
            ld_row(Ybo + (size_t)row * D, lane, ybar);
            ld_row(Xo + (size_t)row * D, lane, u); add_row(u, ybar);
            ld_row(bfc, lane, t); add_row(u, t);
            const float mean = warp_sum(sum_part(u)) * (1.0f / D);
#pragma unroll
            for (int i = 0; i < 4; ++i) { xh[i].x = u[i].x - mean; xh[i].y = u[i].y - mean; xh[i].z = u[i].z - mean; xh[i].w = u[i].w - mean; }
            const float var = warp_sum(dot_part(xh, xh)) * (1.0f / D);
            const float rstd = 1.0f / sqrtf(var + LN_EPS);
            scale_row(xh, rstd);
            ld_row((which ? g_text : g_image) + (size_t)b * D, lane, u);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                dgam[i].x = fmaf(u[i].x, xh[i].x, dgam[i].x); dgam[i].y = fmaf(u[i].y, xh[i].y, dgam[i].y);
                dgam[i].z = fmaf(u[i].z, xh[i].z, dgam[i].z); dgam[i].w = fmaf(u[i].w, xh[i].w, dgam[i].w);
            }
            add_row(dbet, u);
            ld_row(gamma, lane, t);
            ln_backward(u, xh, rstd, t, du);
            add_row(dbf, du);
            st_row(dYo + (size_t)row * D, lane, du);
            st_row_h(dYoh != nullptr ? dYoh + (size_t)row * D : nullptr, lane, du);
            if (g_own != nullptr) {       // extra cotangent on the normalised own rows themselves (the ClipLoss branch, head.cuh)
                float4 gx[4];
                ld_row(g_own + (size_t)row * D, lane, gx);
                add_row(gx, du);
                st_row(dXo + (size_t)row * D, lane, gx);
            } else {
                st_row(dXo + (size_t)row * D, lane, du);
            }
            const float rd = warp_sum(dot_part(du, ybar));
            const float da_i = warp_sum(dot_part(du, vi));
            const float da_t = warp_sum(dot_part(du, vt));
            const float a0 = aown[2 * row], a1 = aown[2 * row + 1];
            if (lane == 0) {
                rowdot[row] = rd;
                dsown[2 * row] = a0 * (da_i - rd) * INV_TAU;
                dsown[2 * row + 1] = a1 * (da_t - rd) * INV_TAU;
            }
            axpy_row(accI, a0, du);
            axpy_row(accT, a1, du);
        }
        // own-row part of dVF (image row, text row): kept apart from the table-row part that table_rows_bwd writes
        // concurrently into dVFo; add_rows_kernel sums the two (and writes the bf16 shadow) later
        (void)dVFoh;
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

// a += b (fp32, in place) with the bf16 shadow of the sum; n4 float4 elements
__global__ void __launch_bounds__(256)
add_rows_kernel(int64_t n4, float* __restrict__ a, const float* __restrict__ b, __nv_bfloat16* __restrict__ ah) {
    pdl_trigger();
    pdl_wait();
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n4) return;
    float4 x = reinterpret_cast<const float4*>(a)[i];
    const float4 y = reinterpret_cast<const float4*>(b)[i];
    x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w;
    reinterpret_cast<float4*>(a)[i] = x;
    if (ah != nullptr) reinterpret_cast<uint2*>(ah)[i] = pack_bf16x4(x);
}

// dS = A .* (dA - rowdot) / tau, in place over dA (fp32 + bf16 shadow); 4 columns per thread (Nsp % 16 == 0)
__global__ void __launch_bounds__(256)
ds_kernel(int64_t n4, int Nsp4, const float* __restrict__ Aext, const float* __restrict__ rowdot, float* __restrict__ dA,
          __nv_bfloat16* __restrict__ dSh, int write_f) {
    pdl_trigger();
    pdl_wait();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const float rd = rowdot[i / Nsp4];
    const float4 a = reinterpret_cast<const float4*>(Aext)[i];
    float4 v = reinterpret_cast<const float4*>(dA)[i];
    v.x = a.x * (v.x - rd) * INV_TAU; v.y = a.y * (v.y - rd) * INV_TAU;
    v.z = a.z * (v.z - rd) * INV_TAU; v.w = a.w * (v.w - rd) * INV_TAU;
    if (write_f) reinterpret_cast<float4*>(dA)[i] = v;
    if (dSh != nullptr) reinterpret_cast<uint2*>(dSh)[i] = pack_bf16x4(v);
}

// own-query x own-key score gradients (the 2x2 per-sample block): INITIAL values of the dQ / dK rows of the own rows
// (fp32); the GEMMs that produce the rest of dKo (wave 5) and dQo (wave 7) accumulate on top (beta = 1) and write
// the bf16 shadows, so this kernel sits beside the table-query rows instead of between two GEMM waves.
__global__ void __launch_bounds__(256)
own_own_bwd_kernel(HeadDims d, const float* __restrict__ QKVo, const __nv_bfloat16* __restrict__ QKVoh,
                   const float* __restrict__ dsown, float* __restrict__ dQKVo, __nv_bfloat16* __restrict__ dQKVoh) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= d.B) return;
    const size_t r0 = (size_t)b * 3 * D, r1 = (size_t)(d.B + b) * 3 * D;
    float4 q0[4], q1[4], k0[4], k1[4], t[4];
    const bool hq = QKVoh != nullptr;
    ld_row_any(QKVo + r0, hq ? QKVoh + r0 : nullptr, lane, q0); ld_row_any(QKVo + r1, hq ? QKVoh + r1 : nullptr, lane, q1);
    ld_row_any(QKVo + r0 + D, hq ? QKVoh + r0 + D : nullptr, lane, k0); ld_row_any(QKVo + r1 + D, hq ? QKVoh + r1 + D : nullptr, lane, k1);
    const float s00 = dsown[2 * b], s01 = dsown[2 * b + 1];
    const float s10 = dsown[2 * (d.B + b)], s11 = dsown[2 * (d.B + b) + 1];
    (void)dQKVoh;
    zero_row(t); axpy_row(t, s00, k0); axpy_row(t, s01, k1); st_row(dQKVo + r0, lane, t);
    zero_row(t); axpy_row(t, s10, k0); axpy_row(t, s11, k1); st_row(dQKVo + r1, lane, t);
    zero_row(t); axpy_row(t, s00, q0); axpy_row(t, s10, q1); st_row(dQKVo + r0 + D, lane, t);
    zero_row(t); axpy_row(t, s01, q0); axpy_row(t, s11, q1); st_row(dQKVo + r1 + D, lane, t);
}

// dTT[r][j] += P[r][j] * (GV[r][j] - h[r]) / tau   for j < M; the bf16 shadow is written for every element
__global__ void __launch_bounds__(256)
dtt_kernel(int Nsp, int M, const float* __restrict__ Pt, const float* __restrict__ GV, const float* __restrict__ h,
           float* __restrict__ dTT, __nv_bfloat16* __restrict__ dTTh) {
    pdl_trigger();
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Nsp * Nsp) return;
    const int r = i / Nsp, j = i % Nsp;
    float v = dTT[i];
    if (j < M) { v += Pt[i] * (GV[i] - h[r]) * INV_TAU; dTT[i] = v; }
    if (dTTh != nullptr) dTTh[i] = __float2bfloat16_rn(v);
}

// dz = inv * (dx - x (x.dx)) for up to four row sets in one launch (fp32 + bf16 shadow), plus per-block column
// sums of dz (fixed order inside the block) for the projection-bias gradients.
//   segment: dz[r] <- from dx[src_row(r)], X[xrow(r)], inv[xrow(r)] with xrow(r) = r + x_off
struct NrmSeg {
    const float* dXsrc;        // [.,D] source gradient rows (row r + x_off)
    const float* X;            // normalised rows
    const float* inv;
    float* dZ;                 // [rows,D] output
    __nv_bfloat16* dZh;
    float* partial;            // [nblocks][D] column sums of this segment's blocks
    int64_t rows;
    int64_t src_off;           // row offset into dXsrc / X / inv
    int rows_per_block;        // multiple of 8
    int blk0;
};
struct NrmList {
    NrmSeg s[4];
    int n;
    int identity;              // 1: dz = dx (no normalisation in the forward)
};
__global__ void __launch_bounds__(256)
nrm_bwd_kernel(const __grid_constant__ NrmList nl) {
    pdl_trigger();
    pdl_wait();
    __shared__ __align__(16) float fold[8][D];
    int si = 0;
    for (int q = 1; q < nl.n; ++q)
        if ((int)blockIdx.x >= nl.s[q].blk0) si = q;
    const NrmSeg& sg = nl.s[si];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lb = (int)blockIdx.x - sg.blk0;
    const int64_t r_begin = (int64_t)lb * sg.rows_per_block;
    const int64_t r_end = min(sg.rows, r_begin + sg.rows_per_block);
    float4 acc[4];
    zero_row(acc);
    for (int64_t r = r_begin + warp; r < r_end; r += 8) {
        const int64_t xr = r + sg.src_off;
        float4 x[4], dx[4];
        if (!nl.identity) ld_row(sg.X + xr * D, lane, x);
        ld_row(sg.dXsrc + xr * D, lane, dx);
        if (!nl.identity) {
            const float dt = warp_sum(dot_part(x, dx));
            const float s = sg.inv[xr];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                dx[i].x = s * (dx[i].x - x[i].x * dt); dx[i].y = s * (dx[i].y - x[i].y * dt);
                dx[i].z = s * (dx[i].z - x[i].z * dt); dx[i].w = s * (dx[i].w - x[i].w * dt);
            }
        }
        st_row(sg.dZ + r * D, lane, dx);
        st_row_h(sg.dZh != nullptr ? sg.dZh + r * D : nullptr, lane, dx);
        add_row(acc, dx);
    }
    st_row(fold[warp], lane, acc);
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += fold[w][c];
        sg.partial[(size_t)lb * D + c] = s;
    }
}

// last launch of the backward: projection-bias gradients from the nrm_bwd partials (fixed order) and the
// prompt-row gradients (rows [C, C+P) of the step-row gradient).
//   blocks 0..2: b_img = sum(part[0]) + sum(part[2]); b_text = sum(part[1]); b_state = sum(part[3])
//   block 3    : dbfc = sum of the expand_table partial sums
//   blocks 4.. : four prompt rows each
struct FinishArgs {
    const float* part[4];
    int nblk[4];
    float *b_img, *b_text, *b_state;
    const float* Rfull;
    float* prompts;            // may be null
    int C, P;
    const float* dbfc_parts;   // [EXP_SUM_BLOCKS][D] or null
    float* dbfc;
};
__global__ void __launch_bounds__(512)
finish_bwd_kernel(const __grid_constant__ FinishArgs fa) {
    pdl_trigger();
    pdl_wait();
    __shared__ float4 fold[4][128];
    const int t = threadIdx.x & 127, g = threadIdx.x >> 7;     // 4 groups of 128 threads, each a quarter of the partials
    if (blockIdx.x == 3) {
        if (fa.dbfc_parts != nullptr && g == 0) {
            float4 r = reinterpret_cast<const float4*>(fa.dbfc_parts)[t];
            for (int q = 1; q < EXP_SUM_BLOCKS; ++q) {
                const float4 a = reinterpret_cast<const float4*>(fa.dbfc_parts + (size_t)q * D)[t];
                r.x += a.x; r.y += a.y; r.z += a.z; r.w += a.w;
            }
            reinterpret_cast<float4*>(fa.dbfc)[t] = r;
        }
        return;
    }
    if (blockIdx.x < 3) {
        const int k = blockIdx.x;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        const int segs[2] = {k == 0 ? 0 : (k == 1 ? 1 : 3), k == 0 ? 2 : -1};
        for (int q = 0; q < 2; ++q) {
            if (segs[q] < 0 || fa.part[segs[q]] == nullptr) continue;
            const float* p = fa.part[segs[q]];
            const int n = fa.nblk[segs[q]];
            const int per = (n + 3) / 4, b0 = g * per, b1 = min(n, b0 + per);
            for (int b = b0; b < b1; ++b) {
                const float4 a = reinterpret_cast<const float4*>(p + (size_t)b * D)[t];
                s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
            }
        }
        fold[g][t] = s;
        __syncthreads();
        if (g == 0) {
            float4 r = fold[0][t];
#pragma unroll
            for (int q = 1; q < 4; ++q) { r.x += fold[q][t].x; r.y += fold[q][t].y; r.z += fold[q][t].z; r.w += fold[q][t].w; }
            float* out = k == 0 ? fa.b_img : (k == 1 ? fa.b_text : fa.b_state);
            if (out != nullptr) reinterpret_cast<float4*>(out)[t] = r;
        }
        return;
    }
    // prompt rows: 4 rows per block
    const int r = (blockIdx.x - 4) * 4 + g;
    if (fa.prompts != nullptr && r < fa.P)
        reinterpret_cast<float4*>(fa.prompts + (size_t)r * D)[t] = reinterpret_cast<const float4*>(fa.Rfull + (size_t)(fa.C + r) * D)[t];
}

}  // namespace team
