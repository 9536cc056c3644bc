// tcgen05 / TMA / TMEM bf16 grouped GEMM (mode BF16) - declarations.
#pragma once
#include "common.cuh"

namespace team {

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

}  // namespace team
