// Internal GEMM layer: the fp32 FFMA engine (TEAM_MODE_F32), the tcgen05 / TMA / TMEM bf16 grouped engine
// (TEAM_MODE_BF16) and run_wave, which issues a set of products on the engine of a mode.
#pragma once
#include "common.cuh"

namespace team {

// fp32 SIMT GEMM: C = alpha*op(A)op(B) + beta*C (+bias[N]).  ta: A stored [K,M]; tb: B stored [N,K].
int gemm_f32(cudaStream_t st, bool ta, bool tb, int64_t M, int64_t N, int64_t K, float alpha, const float* A,
             int64_t lda, const float* B, int64_t ldb, float beta, float* C, int64_t ldc, const float* bias,
             void* ws, size_t ws_bytes);
size_t gemm_f32_workspace_bytes(int64_t M, int64_t N, int64_t K);

constexpr int TC_MAXP = 8;           // problems per tcgen05 launch (kernel parameter space: 8 * 768 B; CUDA >= 12.1 allows 32 KB)

// one K-segment of a problem: op(A)[M,K] op(B)[K,N]
struct TcSeg {
    bool a_mn, b_mn;          // false: operand stored [rows,K] (K-major); true: stored [K,rows] (MN-major)
    int64_t K;
    const void* A;            // bf16
    int64_t lda;
    const void* B;            // bf16
    int64_t ldb;
};

// C[M,N] = alpha * sum_s op(A_s) op(B_s) (+ bias[N]) (+ beta * C): up to two K-segments accumulate into the
// same tensor-memory tile (dW = dQo^T Xo + dQs^T S and friends need no second pass and no ordering).
struct TcGemm {
    int64_t M, N;
    int nseg;                 // 1 or 2
    TcSeg s[2];
    float alpha, beta;
    float* C;                 // fp32 [M,N] output (and beta input), may be null if Cb is set
    int64_t ldc;
    void* Cb;                 // bf16 [M,N] copy of the output, may be null
    int64_t ldcb;
    const float* bias;        // fp32 [N] or null
};

// one launch per TC_MAXP problems; ws holds the split-K partials of the persistent path
int gemm_bf16_group(cudaStream_t st, const TcGemm* ops, int n, void* ws, size_t ws_bytes);
// fp32 [rows,cols] (lds) -> bf16 hi (+ optional lo = bf16(x - hi)) with leading dimension ldd
int to_bf16(cudaStream_t st, const float* src, int64_t lds, int64_t rows, int cols, void* hi, void* lo, int64_t ldd);

// fp32 matrix + (mode BF16) its bf16 shadow with the same leading dimension.  Every operand of run_wave is a
// Mat: the fp32 side feeds the CUDA-core kernels and the F32 mode, the bf16 side feeds tcgen05.  The shadow
// is written by whoever produces the fp32 values (GEMM epilogue or row kernel) - there is no separate
// conversion pass except for the caller's inputs and weights (the head's prep_kernel, mha's staging).
struct Mat {
    float* f;
    __nv_bfloat16* h;
    int64_t ld;
};
inline Mat sub(const Mat& m, int64_t r0, int64_t c0) {
    Mat o;
    o.f = m.f ? m.f + r0 * m.ld + c0 : nullptr;
    o.h = m.h ? m.h + r0 * m.ld + c0 : nullptr;
    o.ld = m.ld;
    return o;
}

// GEMM waves.  The head is a short chain of WAVES; every wave is a set of independent products
//   C[M,N] = alpha * sum_{s<nseg} op(A_s) op(B_s) (+ bias) (+ beta C)
// BF16 mode: the whole wave is ONE launch of the grouped tcgen05 kernel (bf16 shadows of the operands,
// fp32 accumulation in tensor memory, fp32 output + optional bf16 shadow written by the epilogue).
// F32 mode: one fp32 FFMA GEMM per segment (parity mode, not the fast path).
struct GSeg {
    bool a_mn, b_mn;          // false: operand stored [rows,K] (K-major); true: stored [K,rows]
    int64_t K;
    Mat A, B;
};
struct GOp {
    int64_t M, N;
    int nseg;
    GSeg s[2];
    float alpha, beta;
    Mat C;                    // C.h (if any) receives the bf16 shadow of the result
    const float* bias;
};

struct Wave {
    GOp op[TC_MAXP];          // one launch of the grouped engine
    int n = 0;
    GOp& add(int64_t M, int64_t N, float beta, const Mat& C, const float* bias = nullptr) {
        GOp& o = op[n++];
        o.M = M; o.N = N; o.nseg = 0; o.alpha = 1.f; o.beta = beta; o.C = C; o.bias = bias;
        return o;
    }
};
// A [M,K] K-major / A stored [K,M] (a_mn) times B stored [N,K] (K-major) / B stored [K,N] (b_mn)
inline GOp& seg(GOp& o, bool a_mn, const Mat& A, bool b_mn, const Mat& B, int64_t K) {
    GSeg& g = o.s[o.nseg++];
    g.a_mn = a_mn; g.b_mn = b_mn; g.K = K; g.A = A; g.B = B;
    return o;
}

// Runs the non-empty products of `wv` on the engine of `mode` and empties it.  ws: split-K scratch of the engine.
int run_wave(cudaStream_t st, int mode, Wave& wv, void* ws, size_t ws_bytes);

}  // namespace team
