// Standalone MultiHeadAttention.forward (convs/projections.py:64-87, n_head = 1, d_model = d_k = d_v = 512) with its
// autograd backward, for callers that hand sel_attn arbitrary [B, L, 512] token tensors: the differentiable PROOF fusion
// (Proof_Net.forward / forward_transformer, utils/inc_net.py:436-492) and the class-text form of forward_tri_modal
// (:544-547) are composed from it in inc_net.py.  The learner's own per-batch path does not come through here - it runs
// the factorised head of head.cu, which never materialises the [B, L, 512] token tensor.
//
//   Q = q_in Wq^T, K = k_in Wk^T, V = v_in Wv^T            dense projections: tcgen05 GEMM (mode BF16) / fp32 FFMA GEMM
//   A = softmax(Q K^T / sqrt(512))  per sample              batched fp32 GEMM + warp-per-row softmax (log_softmax of the
//   O = A V                                                 reference is discarded by its caller)
//   out = LayerNorm(drop(O Wfc^T + b_fc) + q_in)           with A := drop(A) in train mode: counter-based masks, see Philox below
//
// The backward is the hand-written VJP; every batch reduction (weight gradients through split-K GEMMs, bias / LayerNorm
// gradients through per-CTA partials folded in CTA order) has a fixed order, so results are run-to-run reproducible.
#include "common.cuh"
#include "gemm.cuh"

namespace team {

// ------------------------------------------------------------------------------------------------ dropout masks
// Train-mode dropout of the block (attention probabilities and fc output, p = 0.1 in the reference: convs/projections.py:28,
// :62, :84) as COUNTER-BASED masks: element i of a tensor is kept iff philox4x32-10(key = seed, counter = (i / 4, offset))
// [i % 4] * 2^-32 >= p.  Nothing is stored: the backward regenerates the mask from the same (seed, offset).  The stream is
// this library's own (torch's Philox offsets depend on its launch geometry and cannot be reproduced), so parity in train
// mode is checked against the reference math with the SAME masks (oracle/team_oracle.py:philox_keep_mask) and statistically.
struct Philox {
    uint32_t k0, k1;
    uint64_t offset;
};
__host__ __device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1, n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
// the four 32-bit outputs of counter block `blk`
__host__ __device__ __forceinline__ void philox4(const Philox& g, uint64_t blk, uint32_t (&c)[4]) {
    c[0] = (uint32_t)blk; c[1] = (uint32_t)(blk >> 32); c[2] = (uint32_t)g.offset; c[3] = (uint32_t)(g.offset >> 32);
    uint32_t k0 = g.k0, k1 = g.k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
// keep-scale of element idx: 0 (dropped) or 1 / (1 - p); thr = p * 2^32
__device__ __forceinline__ float drop_scale(const Philox& g, uint64_t idx, uint32_t thr, float inv_keep) {
    uint32_t c[4];
    philox4(g, idx >> 2, c);
    return c[idx & 3] >= thr ? inv_keep : 0.f;
}

// ------------------------------------------------------------------------------------------------ batched fp32 GEMM
// C_b[M,N] = alpha * op(A_b) op(B_b) (+ beta * C_b), b = blockIdx.z; TA: A stored [K,M]; TB: B stored [N,K].
// 64x64x16 tiles, 256 threads, 4x4 micro-tile; guarded scalar loads (row lengths such as L = 141 are not multiples of 4).
constexpr int BG_M = 64, BG_N = 64, BG_K = 16;

template <bool TA, bool TB>
__global__ void __launch_bounds__(256)
bgemm_f32_kernel(int M, int N, int K, float alpha, const float* __restrict__ A, int64_t lda, int64_t sA,
                 const float* __restrict__ B, int64_t ldb, int64_t sB, float beta, float* __restrict__ C, int64_t ldc, int64_t sC) {
    __shared__ float As[BG_K][BG_M + 4];
    __shared__ float Bs[BG_K][BG_N + 4];
    pdl_trigger();
    pdl_wait();
    const int t = threadIdx.x;
    const int m0 = blockIdx.y * BG_M, n0 = blockIdx.x * BG_N;
    A += (int64_t)blockIdx.z * sA;
    B += (int64_t)blockIdx.z * sB;
    C += (int64_t)blockIdx.z * sC;
    const int tx = t & 15, ty = t >> 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < K; k0 += BG_K) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int idx = t + 256 * e;                 // 1024 elements of each operand tile
            if (!TA) {                                   // A[m][k]: k fastest
                const int kk = idx & 15, mm = idx >> 4;
                const int m = m0 + mm, k = k0 + kk;
                As[kk][mm] = (m < M && k < K) ? A[(int64_t)m * lda + k] : 0.f;
            } else {                                     // A[k][m]: m fastest
                const int mm = idx & 63, kk = idx >> 6;
                const int m = m0 + mm, k = k0 + kk;
                As[kk][mm] = (m < M && k < K) ? A[(int64_t)k * lda + m] : 0.f;
            }
            if (TB) {                                    // B[n][k]: k fastest
                const int kk = idx & 15, nn = idx >> 4;
                const int n = n0 + nn, k = k0 + kk;
                Bs[kk][nn] = (n < N && k < K) ? B[(int64_t)n * ldb + k] : 0.f;
            } else {                                     // B[k][n]: n fastest
                const int nn = idx & 63, kk = idx >> 6;
                const int n = n0 + nn, k = k0 + kk;
                Bs[kk][nn] = (n < N && k < K) ? B[(int64_t)k * ldb + n] : 0.f;
            }
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BG_K; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][4 * ty]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][4 * tx]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + 4 * ty + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + 4 * tx + j;
            if (n >= N) continue;
            float* dst = C + (int64_t)m * ldc + n;
            float v = alpha * acc[i][j];
            if (beta != 0.f) v = fmaf(beta, *dst, v);
            *dst = v;
        }
    }
}

static int bgemm(cudaStream_t st, bool ta, bool tb, int64_t batch, int M, int N, int K, float alpha, const float* A, int64_t lda,
                 int64_t sA, const float* B, int64_t ldb, int64_t sB, float beta, float* C, int64_t ldc, int64_t sC) {
    if (batch <= 0 || M <= 0 || N <= 0) return TEAM_OK;
    for (int64_t b0 = 0; b0 < batch; b0 += 65535) {          // gridDim.z limit
        const unsigned nb = (unsigned)(batch - b0 < 65535 ? batch - b0 : 65535);
        const dim3 grid((unsigned)((N + BG_N - 1) / BG_N), (unsigned)((M + BG_M - 1) / BG_M), nb);
        const float *Ab = A + b0 * sA, *Bb = B + b0 * sB;
        float* Cb = C + b0 * sC;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid; cfg.blockDim = dim3(256, 1, 1); cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        cudaError_t e;
        if (!ta && tb) e = cudaLaunchKernelEx(&cfg, bgemm_f32_kernel<false, true>, M, N, K, alpha, Ab, lda, sA, Bb, ldb, sB, beta, Cb, ldc, sC);
        else if (!ta && !tb) e = cudaLaunchKernelEx(&cfg, bgemm_f32_kernel<false, false>, M, N, K, alpha, Ab, lda, sA, Bb, ldb, sB, beta, Cb, ldc, sC);
        else if (ta && !tb) e = cudaLaunchKernelEx(&cfg, bgemm_f32_kernel<true, false>, M, N, K, alpha, Ab, lda, sA, Bb, ldb, sB, beta, Cb, ldc, sC);
        else e = cudaLaunchKernelEx(&cfg, bgemm_f32_kernel<true, true>, M, N, K, alpha, Ab, lda, sA, Bb, ldb, sB, beta, Cb, ldc, sC);
        count_launch();
        if (e != cudaSuccess) return cuda_fail(e, "bgemm_f32_kernel");
    }
    return TEAM_OK;
}

// ------------------------------------------------------------------------------------------------ row kernels
// softmax over the last dimension, in place, warp per row (any row length)
// Ad (optional): the probabilities after attention dropout (what multiplies V); S keeps the softmax itself (its backward needs it)
__global__ void __launch_bounds__(256) mha_softmax_kernel(float* __restrict__ S, int64_t rows, int len, float* __restrict__ Ad,
                                                         Philox rng, uint32_t thr, float inv_keep) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    float* p = S + row * len;
    float m = -INFINITY;
    for (int i = lane; i < len; i += 32) m = fmaxf(m, p[i]);
    m = warp_max(m);
    float z = 0.f;
    for (int i = lane; i < len; i += 32) { const float e = __expf(p[i] - m); p[i] = e; z += e; }
    z = warp_sum(z);
    const float inv = 1.f / z;
    for (int i = lane; i < len; i += 32) {
        const float a = p[i] * inv;
        p[i] = a;
        if (Ad != nullptr) Ad[row * len + i] = a * drop_scale(rng, (uint64_t)(row * len + i), thr, inv_keep);
    }
}
// dS = A .* (dA - sum_j dA_j A_j) * scale, in place on dA
// (with attention dropout dA arrives as the gradient of the DROPPED probabilities: the mask is regenerated and applied first)
__global__ void __launch_bounds__(256) mha_softmax_bwd_kernel(const float* __restrict__ A, float* __restrict__ dA, int64_t rows, int len, float scale,
                                                             int drop, Philox rng, uint32_t thr, float inv_keep) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const float* a = A + row * len;
    float* g = dA + row * len;
    float dot = 0.f;
    for (int i = lane; i < len; i += 32) {
        float gi = g[i];
        if (drop) { gi *= drop_scale(rng, (uint64_t)(row * len + i), thr, inv_keep); g[i] = gi; }
        dot = fmaf(a[i], gi, dot);
    }
    dot = warp_sum(dot);
    for (int i = lane; i < len; i += 32) g[i] = a[i] * (g[i] - dot) * scale;
}

// out = LayerNorm(Y + R) * gamma + beta; Y is overwritten with xhat (what the backward needs), rstd per row
__global__ void __launch_bounds__(256)
mha_add_ln_fwd_kernel(float* __restrict__ Y, const float* __restrict__ R, const float* __restrict__ gamma, const float* __restrict__ beta,
                      float* __restrict__ out, float* __restrict__ rstd, int64_t rows, int drop, Philox rng, uint32_t thr, float inv_keep) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    float4 v[4];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = 4 * (lane + 32 * i);
        float4 y = *reinterpret_cast<const float4*>(Y + row * D + c);
        const float4 r = *reinterpret_cast<const float4*>(R + row * D + c);
        if (drop) {                                        // dropout(fc(output)), convs/projections.py:84: one counter block per float4
            uint32_t q[4];
            philox4(rng, (uint64_t)(row * D + c) >> 2, q);
            y.x *= q[0] >= thr ? inv_keep : 0.f; y.y *= q[1] >= thr ? inv_keep : 0.f;
            y.z *= q[2] >= thr ? inv_keep : 0.f; y.w *= q[3] >= thr ? inv_keep : 0.f;
        }
        v[i] = make_float4(y.x + r.x, y.y + r.y, y.z + r.z, y.w + r.w);
        s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
    const float mean = warp_sum(s) * (1.f / D);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
        q += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
    }
    const float rs = rsqrtf(warp_sum(q) * (1.f / D) + LN_EPS);
    if (lane == 0) rstd[row] = rs;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = 4 * (lane + 32 * i);
        const float4 g = *reinterpret_cast<const float4*>(gamma + c), b = *reinterpret_cast<const float4*>(beta + c);
        const float4 xh = make_float4(v[i].x * rs, v[i].y * rs, v[i].z * rs, v[i].w * rs);
        *reinterpret_cast<float4*>(Y + row * D + c) = xh;
        *reinterpret_cast<float4*>(out + row * D + c) = make_float4(fmaf(xh.x, g.x, b.x), fmaf(xh.y, g.y, b.y), fmaf(xh.z, g.z, b.z), fmaf(xh.w, g.w, b.w));
    }
}

// LayerNorm backward of rows [blockIdx.x * rows_per_cta, ...): dpre = rstd (g.dy - mean(g.dy) - xhat mean(g.dy.xhat));
// per-CTA partial sums of dgamma = dy.xhat, dbeta = dy, db_fc = dpre  ->  partial[cta][3][512] (folded in CTA order).
constexpr int MHA_LNB_WARPS = 8;
__global__ void __launch_bounds__(MHA_LNB_WARPS * 32)
mha_ln_bwd_kernel(const float* __restrict__ dY, const float* __restrict__ XH, const float* __restrict__ rstd, const float* __restrict__ gamma,
                  float* __restrict__ dPre, float* __restrict__ partial, int64_t rows, int rows_per_cta,
                  float* __restrict__ dFc, Philox rng, uint32_t thr, float inv_keep) {
    __shared__ float red[MHA_LNB_WARPS][3][D];
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t r1 = r0 + rows_per_cta < rows ? r0 + rows_per_cta : rows;
    float4 g[4], ag[4], ab[4], ap[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        g[i] = *reinterpret_cast<const float4*>(gamma + 4 * (lane + 32 * i));
        ag[i] = ab[i] = ap[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int64_t row = r0 + warp; row < r1; row += MHA_LNB_WARPS) {
        float4 dy[4], xh[4];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = 4 * (lane + 32 * i);
            dy[i] = *reinterpret_cast<const float4*>(dY + row * D + c);
            xh[i] = *reinterpret_cast<const float4*>(XH + row * D + c);
            ag[i].x = fmaf(dy[i].x, xh[i].x, ag[i].x); ag[i].y = fmaf(dy[i].y, xh[i].y, ag[i].y);
            ag[i].z = fmaf(dy[i].z, xh[i].z, ag[i].z); ag[i].w = fmaf(dy[i].w, xh[i].w, ag[i].w);
            ab[i].x += dy[i].x; ab[i].y += dy[i].y; ab[i].z += dy[i].z; ab[i].w += dy[i].w;
            dy[i].x *= g[i].x; dy[i].y *= g[i].y; dy[i].z *= g[i].z; dy[i].w *= g[i].w;          // g . dy
            s1 += dy[i].x + dy[i].y + dy[i].z + dy[i].w;
            s2 += dy[i].x * xh[i].x + dy[i].y * xh[i].y + dy[i].z * xh[i].z + dy[i].w * xh[i].w;
        }
        s1 = warp_sum(s1) * (1.f / D);
        s2 = warp_sum(s2) * (1.f / D);
        const float rs = rstd[row];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = 4 * (lane + 32 * i);
            const float4 o = make_float4(rs * (dy[i].x - s1 - xh[i].x * s2), rs * (dy[i].y - s1 - xh[i].y * s2),
                                         rs * (dy[i].z - s1 - xh[i].z * s2), rs * (dy[i].w - s1 - xh[i].w * s2));
            *reinterpret_cast<float4*>(dPre + row * D + c) = o;
            float4 f = o;
            if (dFc != nullptr) {                          // gradient of the fc output through its dropout mask (dPre itself is the residual's)
                uint32_t q[4];
                philox4(rng, (uint64_t)(row * D + c) >> 2, q);
                f.x *= q[0] >= thr ? inv_keep : 0.f; f.y *= q[1] >= thr ? inv_keep : 0.f;
                f.z *= q[2] >= thr ? inv_keep : 0.f; f.w *= q[3] >= thr ? inv_keep : 0.f;
                *reinterpret_cast<float4*>(dFc + row * D + c) = f;
            }
            ap[i].x += f.x; ap[i].y += f.y; ap[i].z += f.z; ap[i].w += f.w;
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = 4 * (lane + 32 * i);
        *reinterpret_cast<float4*>(&red[warp][0][c]) = ag[i];
        *reinterpret_cast<float4*>(&red[warp][1][c]) = ab[i];
        *reinterpret_cast<float4*>(&red[warp][2][c]) = ap[i];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 3 * D; e += MHA_LNB_WARPS * 32) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < MHA_LNB_WARPS; ++w) s += red[w][e / D][e % D];                         // fixed warp order
        partial[(size_t)blockIdx.x * 3 * D + e] = s;
    }
}
// out_k[c] = sum over CTAs (in order) of partial[cta][k][c]
__global__ void __launch_bounds__(256) mha_fold_kernel(const float* __restrict__ partial, int nctas, float* __restrict__ o0, float* __restrict__ o1, float* __restrict__ o2) {
    pdl_trigger();
    pdl_wait();
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= 3 * D) return;
    float s = 0.f;
    for (int b = 0; b < nctas; ++b) s += partial[(size_t)b * 3 * D + e];
    float* o = e < D ? o0 : (e < 2 * D ? o1 : o2);
    if (o != nullptr) o[e % D] = s;
}
// y += x (float4)
__global__ void __launch_bounds__(256) mha_add_kernel(float* __restrict__ y, const float* __restrict__ x, int64_t n4) {
    pdl_trigger();
    pdl_wait();
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n4) return;
    float4 a = reinterpret_cast<float4*>(y)[i];
    const float4 b = reinterpret_cast<const float4*>(x)[i];
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    reinterpret_cast<float4*>(y)[i] = a;
}

// mean over the middle dimension of x[outer][red][inner] -> out[outer][inner] (serial, fixed order) and its backward
__global__ void __launch_bounds__(256) mean_mid_kernel(const float* __restrict__ x, float* __restrict__ out, int64_t outer, int64_t red, int64_t inner) {
    pdl_trigger();
    pdl_wait();
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= outer * inner) return;
    const int64_t o = i / inner, c = i % inner;
    const float* p = x + o * red * inner + c;
    float s = 0.f;
    for (int64_t r = 0; r < red; ++r) s += p[r * inner];
    out[i] = s / (float)red;
}
__global__ void __launch_bounds__(256) mean_mid_bwd_kernel(const float* __restrict__ g, float* __restrict__ dx, int64_t outer, int64_t red, int64_t inner) {
    pdl_trigger();
    pdl_wait();
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= outer * red * inner) return;
    const int64_t o = i / (red * inner), c = i % inner;
    dx[i] = g[o * inner + c] / (float)red;
}

// ------------------------------------------------------------------------------------------------ dense products
// C[M,N] = op(A) op(B) (+ bias) (+ beta C) on the mode's GEMM engine.  ta: A stored [K,M]; tb: B stored [N,K].
// BF16 mode stages both operands to bf16 first; shapes the tcgen05 engine cannot take run on the fp32 engine.
struct Dense {
    cudaStream_t st;
    int mode;
    void* gws; size_t gws_bytes;           // split-K workspace of the engine
    __nv_bfloat16 *ha, *hb;                // bf16 staging of the two operands (mode BF16)
};
static int dense(const Dense& e, bool ta, bool tb, int64_t M, int64_t N, int64_t K, const float* A, int64_t lda, const float* B, int64_t ldb,
                 float beta, float* C, int64_t ldc, const float* bias) {
    if (M <= 0 || N <= 0) return TEAM_OK;
    const bool tc = e.mode == TEAM_MODE_BF16 && K % 8 == 0 && lda % 8 == 0 && ldb % 8 == 0 && K >= 64;
    int rc;
    if (tc) {
        const int64_t ar = ta ? K : M, ac = ta ? M : K, br = tb ? N : K, bc = tb ? K : N;
        if ((rc = to_bf16(e.st, A, lda, ar, (int)ac, e.ha, nullptr, lda))) return rc;
        if ((rc = to_bf16(e.st, B, ldb, br, (int)bc, e.hb, nullptr, ldb))) return rc;
    }
    Wave wv;
    seg(wv.add(M, N, beta, Mat{C, nullptr, ldc}, bias), ta, Mat{const_cast<float*>(A), e.ha, lda}, !tb, Mat{const_cast<float*>(B), e.hb, ldb}, K);
    return run_wave(e.st, tc ? e.mode : TEAM_MODE_F32, wv, e.gws, e.gws_bytes);
}

struct MhaPlan {
    int64_t Rq, Rk;
    float *Q, *K, *V, *A, *Ad, *O, *XH, *rstd;            // saved by the forward (Ad: probabilities after attention dropout)
    float *dPre, *dFc, *dO, *dA, *dQ, *dK, *dV, *partial; // backward scratch (dFc: dPre through the fc-output dropout mask)
    __nv_bfloat16 *ha, *hb;
    void* gws; size_t gws_bytes;
    int ln_ctas, ln_rows_per_cta;
    size_t total;
};
static MhaPlan mha_plan(int64_t B, int64_t Lq, int64_t Lk, void* base) {
    MhaPlan p;
    p.Rq = B * Lq; p.Rk = B * Lk;
    size_t off = 0;
    auto take = [&](size_t bytes) { void* r = base ? (char*)base + off : nullptr; off += align_up(bytes, 256); return r; };
    const size_t fq = (size_t)p.Rq * D * 4, fk = (size_t)p.Rk * D * 4, fa = (size_t)B * Lq * Lk * 4;
    p.Q = (float*)take(fq); p.K = (float*)take(fk); p.V = (float*)take(fk);
    p.A = (float*)take(fa); p.Ad = (float*)take(fa); p.O = (float*)take(fq); p.XH = (float*)take(fq); p.rstd = (float*)take((size_t)p.Rq * 4);
    p.dPre = (float*)take(fq); p.dFc = (float*)take(fq); p.dO = (float*)take(fq); p.dA = (float*)take(fa);
    p.dQ = (float*)take(fq); p.dK = (float*)take(fk); p.dV = (float*)take(fk);
    int64_t ctas = (p.Rq + 63) / 64;
    if (ctas > 4 * NUM_SMS) ctas = 4 * NUM_SMS;
    if (ctas < 1) ctas = 1;
    p.ln_ctas = (int)ctas;
    p.ln_rows_per_cta = (int)((p.Rq + ctas - 1) / ctas);
    p.ln_ctas = (int)((p.Rq + p.ln_rows_per_cta - 1) / p.ln_rows_per_cta);
    p.partial = (float*)take((size_t)p.ln_ctas * 3 * D * 4);
    const int64_t rmax = p.Rq > p.Rk ? p.Rq : p.Rk;
    p.ha = (__nv_bfloat16*)take((size_t)(rmax > D ? rmax : D) * D * 2);
    p.hb = (__nv_bfloat16*)take((size_t)(rmax > D ? rmax : D) * D * 2);
    const size_t g = gemm_f32_workspace_bytes(D, D, rmax);                 // weight gradients: K = rows (split-K)
    p.gws_bytes = align_up(g > 256 ? g : 256, 256);                       // floor: keeps team_mha_workspace_bytes as callers size it
    p.gws = take(p.gws_bytes);
    p.total = off;
    return p;
}

struct MhaDrop {
    bool on;
    Philox attn, fc;
    uint32_t thr;
    float inv_keep;
};
static MhaDrop mha_drop(float p, uint64_t seed, uint64_t offset) {
    MhaDrop d;
    d.on = p > 0.f;
    d.attn = Philox{(uint32_t)seed, (uint32_t)(seed >> 32), offset};
    d.fc = Philox{(uint32_t)seed, (uint32_t)(seed >> 32), offset + 1};
    const double t = (double)p * 4294967296.0;
    d.thr = t >= 4294967295.0 ? 4294967295u : (uint32_t)t;
    d.inv_keep = p < 1.f ? 1.f / (1.f - p) : 0.f;
    return d;
}

static int mha_check(int mode, int64_t B, int64_t Lq, int64_t Lk) {
    TEAM_REQUIRE(mode == TEAM_MODE_F32 || mode == TEAM_MODE_BF16, "mha: bad mode %d", mode);
    TEAM_REQUIRE(B >= 1 && Lq >= 1 && Lk >= 1 && Lq <= 4096 && Lk <= 4096 && B * Lq < (1ll << 31) && B * Lk < (1ll << 31),
                 "mha: shape out of range (batch %lld, len_q %lld, len_k %lld)", (long long)B, (long long)Lq, (long long)Lk);
    return TEAM_OK;
}

}  // namespace team

using namespace team;

extern "C" size_t team_mha_workspace_bytes(int64_t batch, int64_t len_q, int64_t len_k) {
    if (batch < 1 || len_q < 1 || len_k < 1) return 0;
    return mha_plan(batch, len_q, len_k, nullptr).total;
}

extern "C" int team_mha_fwd(int mode, int64_t batch, int64_t len_q, int64_t len_k, const float* q_in, const float* k_in,
                            const float* v_in, const float* w_q, const float* w_k, const float* w_v, const float* w_fc,
                            const float* b_fc, const float* ln_g, const float* ln_b, float dropout_p, uint64_t seed,
                            uint64_t offset, float* out, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = mha_check(mode, batch, len_q, len_k);
    if (rc) return rc;
    TEAM_REQUIRE(q_in && k_in && v_in && w_q && w_k && w_v && w_fc && b_fc && ln_g && ln_b && out, "mha fwd: null pointer");
    TEAM_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "mha fwd: dropout_p %g outside [0, 1)", (double)dropout_p);
    const MhaDrop dr = mha_drop(dropout_p, seed, offset);
    TEAM_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "mha: workspace must be 256-byte aligned");
    const MhaPlan p = mha_plan(batch, len_q, len_k, workspace);
    if (workspace_bytes < p.total) { set_error("mha fwd: workspace %zu < %zu bytes", workspace_bytes, p.total); return TEAM_EWORKSPACE; }
    const cudaStream_t st = (cudaStream_t)stream;
    const int Lq = (int)len_q, Lk = (int)len_k;
    const Dense e{st, mode, p.gws, p.gws_bytes, p.ha, p.hb};
    if ((rc = dense(e, false, true, p.Rq, D, D, q_in, D, w_q, D, 0.f, p.Q, D, nullptr))) return rc;
    if ((rc = dense(e, false, true, p.Rk, D, D, k_in, D, w_k, D, 0.f, p.K, D, nullptr))) return rc;
    if ((rc = dense(e, false, true, p.Rk, D, D, v_in, D, w_v, D, 0.f, p.V, D, nullptr))) return rc;
    // scores / temperature (temperature = sqrt(d_k), convs/projections.py:53), softmax over the keys, A V
    if ((rc = bgemm(st, false, true, batch, Lq, Lk, D, 1.f / sqrtf((float)D), p.Q, D, (int64_t)Lq * D, p.K, D, (int64_t)Lk * D, 0.f, p.A, Lk, (int64_t)Lq * Lk))) return rc;
    TEAM_LAUNCH(mha_softmax_kernel, (p.Rq + 7) / 8, 256, 0, st, p.A, p.Rq, Lk, dr.on ? p.Ad : (float*)nullptr, dr.attn, dr.thr, dr.inv_keep);
    const float* Ause = dr.on ? p.Ad : p.A;
    if ((rc = bgemm(st, false, false, batch, Lq, D, Lk, 1.f, Ause, Lk, (int64_t)Lq * Lk, p.V, D, (int64_t)Lk * D, 0.f, p.O, D, (int64_t)Lq * D))) return rc;
    if ((rc = dense(e, false, true, p.Rq, D, D, p.O, D, w_fc, D, 0.f, p.XH, D, b_fc))) return rc;
    TEAM_LAUNCH(mha_add_ln_fwd_kernel, (p.Rq + 7) / 8, 256, 0, st, p.XH, q_in, ln_g, ln_b, out, p.rstd, p.Rq, dr.on ? 1 : 0, dr.fc, dr.thr, dr.inv_keep);
    return TEAM_OK;
}

// g_* of the inputs may be NULL (not needed); when q_in, k_in and v_in are one tensor the caller adds the three.
extern "C" int team_mha_bwd(int mode, int64_t batch, int64_t len_q, int64_t len_k, const float* q_in, const float* k_in,
                            const float* v_in, const float* w_q, const float* w_k, const float* w_v, const float* w_fc,
                            const float* ln_g, float dropout_p, uint64_t seed, uint64_t offset, const float* g_out,
                            float* g_q_in, float* g_k_in, float* g_v_in, float* g_w_q, float* g_w_k, float* g_w_v,
                            float* g_w_fc, float* g_b_fc, float* g_ln_g, float* g_ln_b, void* workspace,
                            size_t workspace_bytes, void* stream) {
    int rc = mha_check(mode, batch, len_q, len_k);
    if (rc) return rc;
    TEAM_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "mha bwd: dropout_p %g outside [0, 1)", (double)dropout_p);
    const MhaDrop dr = mha_drop(dropout_p, seed, offset);
    TEAM_REQUIRE(q_in && k_in && v_in && w_q && w_k && w_v && w_fc && ln_g && g_out, "mha bwd: null pointer");
    TEAM_REQUIRE(g_w_q && g_w_k && g_w_v && g_w_fc && g_b_fc && g_ln_g && g_ln_b, "mha bwd: null gradient buffer");
    TEAM_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "mha: workspace must be 256-byte aligned");
    const MhaPlan p = mha_plan(batch, len_q, len_k, workspace);
    if (workspace_bytes < p.total) { set_error("mha bwd: workspace %zu < %zu bytes", workspace_bytes, p.total); return TEAM_EWORKSPACE; }
    const cudaStream_t st = (cudaStream_t)stream;
    const int Lq = (int)len_q, Lk = (int)len_k;
    const Dense e{st, mode, p.gws, p.gws_bytes, p.ha, p.hb};
    // LayerNorm backward (+ residual branch), b_fc / gamma / beta gradients
    TEAM_LAUNCH(mha_ln_bwd_kernel, p.ln_ctas, MHA_LNB_WARPS * 32, 0, st, g_out, p.XH, p.rstd, ln_g, p.dPre, p.partial, p.Rq, p.ln_rows_per_cta,
                dr.on ? p.dFc : (float*)nullptr, dr.fc, dr.thr, dr.inv_keep);
    TEAM_LAUNCH(mha_fold_kernel, (3 * D + 255) / 256, 256, 0, st, p.partial, p.ln_ctas, g_ln_g, g_ln_b, g_b_fc);
    // fc: dWfc = dFc^T O, dO = dFc Wfc  (dFc = dPre through the fc-output dropout mask; = dPre without dropout)
    const float* dFc = dr.on ? p.dFc : p.dPre;
    const float* Ause = dr.on ? p.Ad : p.A;
    if ((rc = dense(e, true, false, D, D, p.Rq, dFc, D, p.O, D, 0.f, g_w_fc, D, nullptr))) return rc;
    if ((rc = dense(e, false, false, p.Rq, D, D, dFc, D, w_fc, D, 0.f, p.dO, D, nullptr))) return rc;
    // attention core: dA = dO V^T, dV = A^T dO, dS = softmax', dQ = dS K, dK = dS^T Q  (dS carries 1 / temperature)
    if ((rc = bgemm(st, false, true, batch, Lq, Lk, D, 1.f, p.dO, D, (int64_t)Lq * D, p.V, D, (int64_t)Lk * D, 0.f, p.dA, Lk, (int64_t)Lq * Lk))) return rc;
    if ((rc = bgemm(st, true, false, batch, Lk, D, Lq, 1.f, Ause, Lk, (int64_t)Lq * Lk, p.dO, D, (int64_t)Lq * D, 0.f, p.dV, D, (int64_t)Lk * D))) return rc;
    TEAM_LAUNCH(mha_softmax_bwd_kernel, (p.Rq + 7) / 8, 256, 0, st, p.A, p.dA, p.Rq, Lk, 1.f / sqrtf((float)D), dr.on ? 1 : 0, dr.attn, dr.thr, dr.inv_keep);
    if ((rc = bgemm(st, false, false, batch, Lq, D, Lk, 1.f, p.dA, Lk, (int64_t)Lq * Lk, p.K, D, (int64_t)Lk * D, 0.f, p.dQ, D, (int64_t)Lq * D))) return rc;
    if ((rc = bgemm(st, true, false, batch, Lk, D, Lq, 1.f, p.dA, Lk, (int64_t)Lq * Lk, p.Q, D, (int64_t)Lq * D, 0.f, p.dK, D, (int64_t)Lk * D))) return rc;
    // projections: dW = dP^T x, dx = dP W
    if ((rc = dense(e, true, false, D, D, p.Rq, p.dQ, D, q_in, D, 0.f, g_w_q, D, nullptr))) return rc;
    if ((rc = dense(e, true, false, D, D, p.Rk, p.dK, D, k_in, D, 0.f, g_w_k, D, nullptr))) return rc;
    if ((rc = dense(e, true, false, D, D, p.Rk, p.dV, D, v_in, D, 0.f, g_w_v, D, nullptr))) return rc;
    if (g_q_in != nullptr) {          // residual + through w_q
        TEAM_CUDA_CHECK(cudaMemcpyAsync(g_q_in, p.dPre, (size_t)p.Rq * D * 4, cudaMemcpyDeviceToDevice, st));
        if ((rc = dense(e, false, false, p.Rq, D, D, p.dQ, D, w_q, D, 1.f, g_q_in, D, nullptr))) return rc;
    }
    if (g_k_in != nullptr && (rc = dense(e, false, false, p.Rk, D, D, p.dK, D, w_k, D, 0.f, g_k_in, D, nullptr))) return rc;
    if (g_v_in != nullptr && (rc = dense(e, false, false, p.Rk, D, D, p.dV, D, w_v, D, 0.f, g_v_in, D, nullptr))) return rc;
    return TEAM_OK;
}

// keep[i] = 1 / 0 for element i of the tensor masked with (seed, offset) - what the kernels above regenerate on the fly
// (attention probabilities: offset; fc output: offset + 1).  For the statistical tests of the stream.
__global__ void __launch_bounds__(256) philox_mask_kernel(unsigned char* __restrict__ keep, int64_t n, Philox rng, uint32_t thr) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    uint32_t c[4];
    philox4(rng, (uint64_t)i >> 2, c);
    keep[i] = c[i & 3] >= thr ? 1 : 0;
}
extern "C" int team_dropout_keep_mask(unsigned char* keep, int64_t n, float dropout_p, uint64_t seed, uint64_t offset, void* stream) {
    TEAM_REQUIRE(keep != nullptr && n >= 0 && dropout_p >= 0.f && dropout_p < 1.f, "dropout mask: bad arguments");
    if (n == 0) return TEAM_OK;
    const MhaDrop dr = mha_drop(dropout_p, seed, offset);
    philox_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(keep, n, dr.attn, dr.thr);
    TEAM_LAUNCH_CHECK("philox_mask_kernel");
    return TEAM_OK;
}

// mean over dimension `red` of x[outer][red][inner] (torch.mean(dim) of the PROOF / class-text forms) and its backward
extern "C" int team_mean_mid(const float* x, float* out, int64_t outer, int64_t red, int64_t inner, void* stream) {
    TEAM_REQUIRE(x && out && outer >= 1 && red >= 1 && inner >= 1, "mean_mid: bad arguments");
    TEAM_LAUNCH(mean_mid_kernel, (outer * inner + 255) / 256, 256, 0, (cudaStream_t)stream, x, out, outer, red, inner);
    return TEAM_OK;
}
extern "C" int team_mean_mid_bwd(const float* g, float* dx, int64_t outer, int64_t red, int64_t inner, void* stream) {
    TEAM_REQUIRE(g && dx && outer >= 1 && red >= 1 && inner >= 1, "mean_mid_bwd: bad arguments");
    TEAM_LAUNCH(mean_mid_bwd_kernel, (outer * red * inner + 255) / 256, 256, 0, (cudaStream_t)stream, g, dx, outer, red, inner);
    return TEAM_OK;
}
