// K8 - fused L2-normalise + cosine logits + argmax against <= 32 class rows per pass.
//
// Replaces CosineLinear.forward (convs/linears.py:51-61) and the last stage of
// Learner.forward_for_classification (models/proof.py:526-535).
//
// HBM-bound for the class counts of the path (C <= 20): each feature row (2 KB fp32) is
// read once with 128-bit streaming loads; the normalised class matrix lives in shared
// memory.  A warp owns two rows at a time: lane l keeps columns {4(l+32j)..+3} of both rows
// in registers, accumulates one partial dot product per class, and a 31-shuffle
// transpose-reduce leaves the total for class l on lane l (instead of 5 shuffles per
// class).  Algorithmic bytes per row: 512*e + 4*C (logits) + 8 (argmax)   (SURVEY 8d).
#include "common.cuh"
#include "head.cuh"

namespace team {

constexpr int COS_WARPS = 8;
constexpr int COS_CCHUNK = 32;

template <typename T> struct XLoad;
template <> struct XLoad<float> {
    static __device__ __forceinline__ float4 load(const float* row, int c4) { return ld_stream_f4(row + 4 * c4); }
};
template <> struct XLoad<__nv_bfloat16> {
    static __device__ __forceinline__ float4 load(const __nv_bfloat16* row, int c4) {
        uint2 u = ld_stream_u2(row + 4 * c4);
        return make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
    }
};

__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
    return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
}

// v[0..31] partial sums per class on every lane -> returns the full sum of class `lane`.
__device__ __forceinline__ float transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
            const float send = upper ? v[i] : v[i + off];
            const float keep = upper ? v[i + off] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0];
}

template <typename T>
__global__ void __launch_bounds__(COS_WARPS * 32)
cosine_logits_kernel(const T* __restrict__ x, int64_t n_rows, const float* __restrict__ w, int num_classes,
                     const float* __restrict__ sigma_dev, float* __restrict__ logits,
                     int64_t* __restrict__ argmax_out, float* __restrict__ chunk_best, int n_chunks) {
    extern __shared__ __align__(16) float4 ws[];         // [min(C,32)][128] normalised class rows of this chunk
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c0 = blockIdx.y * COS_CCHUNK;
    const int nc = min(COS_CCHUNK, num_classes - c0);
    const int c_alloc = min(COS_CCHUNK, num_classes);
    // class rows of this warp (c = warp, warp + 8, ...: at most COS_CCHUNK / COS_WARPS = 4): ALL their loads first, then the
    // norms - one L2 round trip instead of one per class row (this prologue is most of the kernel at ~1 000 rows)
    {
        constexpr int CPW = (COS_CCHUNK + COS_WARPS - 1) / COS_WARPS;
        float4 r[CPW][4];
#pragma unroll
        for (int u = 0; u < CPW; ++u) {
            const int c = warp + u * COS_WARPS;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                r[u][j] = (c < nc) ? __ldg(reinterpret_cast<const float4*>(w + (size_t)(c0 + c) * D) + lane + 32 * j)
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < CPW; ++u) {
            const int c = warp + u * COS_WARPS;
            if (c >= c_alloc) continue;
            float ss = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) ss += dot4(r[u][j], r[u][j]);
            ss = warp_sum(ss);
            const float inv = 1.0f / fmaxf(sqrtf(ss), NORM_EPS);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                ws[c * (D / 4) + lane + 32 * j] = make_float4(r[u][j].x * inv, r[u][j].y * inv, r[u][j].z * inv, r[u][j].w * inv);
        }
    }
    __syncthreads();
    const float sigma = sigma_dev ? __ldg(sigma_dev) : 1.0f;
    const int64_t pair_stride = (int64_t)gridDim.x * COS_WARPS;
    const int64_t n_pairs = (n_rows + 1) / 2;
    for (int64_t pr = (int64_t)blockIdx.x * COS_WARPS + warp; pr < n_pairs; pr += pair_stride) {
        const int64_t ra = 2 * pr, rb = 2 * pr + 1;
        const bool has_b = rb < n_rows;
        float4 xa[4], xb[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            xa[j] = XLoad<T>::load(x + ra * D, lane + 32 * j);
            xb[j] = has_b ? XLoad<T>::load(x + rb * D, lane + 32 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float ssa = 0.f, ssb = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) { ssa += dot4(xa[j], xa[j]); ssb += dot4(xb[j], xb[j]); }
        ssa = warp_sum(ssa);
        ssb = warp_sum(ssb);
        float va[32], vb[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            float a = 0.f, b = 0.f;
            if (c < nc) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 w4 = ws[c * (D / 4) + lane + 32 * j];
                    a += dot4(xa[j], w4);
                    b += dot4(xb[j], w4);
                }
            }
            va[c] = a;
            vb[c] = b;
        }
        float ta = transpose_reduce32(va, lane);
        float tb = transpose_reduce32(vb, lane);
        ta *= sigma / fmaxf(sqrtf(ssa), NORM_EPS);
        tb *= sigma / fmaxf(sqrtf(ssb), NORM_EPS);
        if (logits != nullptr && lane < nc) {
            logits[ra * num_classes + c0 + lane] = ta;
            if (has_b) logits[rb * num_classes + c0 + lane] = tb;
        }
        if (argmax_out != nullptr) {
            // first maximal index (torch.max semantics): max value, ties -> lower index
            float ba = lane < nc ? ta : -INFINITY, bb = lane < nc ? tb : -INFINITY;
            int ia = lane, ib = lane;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float oa = __shfl_xor_sync(0xffffffffu, ba, o);
                const int oia = __shfl_xor_sync(0xffffffffu, ia, o);
                if (oa > ba || (oa == ba && oia < ia)) { ba = oa; ia = oia; }
                const float ob = __shfl_xor_sync(0xffffffffu, bb, o);
                const int oib = __shfl_xor_sync(0xffffffffu, ib, o);
                if (ob > bb || (ob == bb && oib < ib)) { bb = ob; ib = oib; }
            }
            if (lane == 0) {
                if (n_chunks == 1) {
                    argmax_out[ra] = c0 + ia;
                    if (has_b) argmax_out[rb] = c0 + ib;
                } else {   // multi-chunk: stash (value,index) per chunk, merged by cosine_argmax_merge
                    chunk_best[(ra * n_chunks + blockIdx.y) * 2 + 0] = ba;
                    chunk_best[(ra * n_chunks + blockIdx.y) * 2 + 1] = __int_as_float(c0 + ia);
                    if (has_b) {
                        chunk_best[(rb * n_chunks + blockIdx.y) * 2 + 0] = bb;
                        chunk_best[(rb * n_chunks + blockIdx.y) * 2 + 1] = __int_as_float(c0 + ib);
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------ second generation: the contraction on the tensor pipe
// The kernel above is issue-bound, not HBM-bound: 20 classes x 512 columns = 10 k FMAs per 2 KB row plus the shared-memory
// re-reads of the class rows and two 31-shuffle transposes per row pair (~535 warp instructions per row, 22 % of the HBM
// copy peak measured).  Here a warp owns 16 rows and computes their [16, 8 NTILES] logit tile with
// mma.sync.m16n8k8 TF32 in the 3xTF32 split (x = x_hi + x_lo, w = w_hi + w_lo; x_hi w_hi + x_hi w_lo + x_lo w_hi: error
// ~2^-21 per product, i.e. fp32-grade - a plain TF32 product would miss the 1e-5 bar) with fp32 accumulation, the
// row norms on CUDA cores, normalisation / sigma / first-index argmax in the epilogue on the accumulator fragments:
// ~85 warp instructions per row.  A operands come straight from global memory as 128-bit loads: the k index inside a
// 16-column chunk is permuted (the same permutation is baked into the B fragments in shared memory), so that the four
// consecutive columns a lane loads ARE its fragment elements of two k-steps - no staging, no shared-memory traffic for x.
// bf16 rows are exact in TF32, so their low part vanishes (two MMAs per tile instead of three).
// B fragments: Bf[chunk s][k-step j][n-tile][lane] = (b0_hi, b1_hi, b0_lo, b1_lo) of the NORMALISED class rows, where
//   b0 <-> W[8 nt + lane / 4][16 s + 4 (lane % 4) + 2 j],  b1 <-> the next column.
constexpr int COS2_WARPS = 8;

__device__ __forceinline__ uint32_t tf32_hi(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

template <typename T> struct XQuad;           // four consecutive columns of a row as fp32
template <> struct XQuad<float> {
    static constexpr bool EXACT = false;
    static __device__ __forceinline__ float4 load(const float* p) { return ld_stream_f4(p); }
};
template <> struct XQuad<__nv_bfloat16> {
    static constexpr bool EXACT = true;       // bf16 values are TF32 numbers: no low part
    static __device__ __forceinline__ float4 load(const __nv_bfloat16* p) {
        const uint2 u = ld_stream_u2(p);
        return make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
    }
};

template <typename T, int NTILES>
__global__ void __launch_bounds__(COS2_WARPS * 32)
cosine_mma_kernel(const T* __restrict__ x, int64_t n_rows, const float* __restrict__ w, int num_classes,
                  const float* __restrict__ sigma_dev, float* __restrict__ logits,
                  int64_t* __restrict__ argmax_out, float* __restrict__ chunk_best, int n_chunks) {
    extern __shared__ __align__(16) float4 bf[];          // [32 chunks][2 steps][NTILES][32 lanes]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c0 = blockIdx.y * COS_CCHUNK;
    const int nc = min(COS_CCHUNK, num_classes - c0);
    // ---- B fragments: normalise the class rows of this chunk, split hi / lo, scatter into fragment order
    for (int c = warp; c < NTILES * 8; c += COS2_WARPS) {
        float4 r[4];
        float ss = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            r[j] = (c < nc) ? reinterpret_cast<const float4*>(w + (size_t)(c0 + c) * D)[lane + 32 * j] : make_float4(0.f, 0.f, 0.f, 0.f);
            ss += dot4(r[j], r[j]);
        }
        ss = warp_sum(ss);
        const float inv = 1.0f / fmaxf(sqrtf(ss), NORM_EPS);
        const int nt = c >> 3, n = c & 7;
        float* bfl = reinterpret_cast<float*>(bf);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float e[4] = {r[j].x * inv, r[j].y * inv, r[j].z * inv, r[j].w * inv};
            const int col = 4 * (lane + 32 * j);          // columns col .. col + 3: chunk s, quad q, elements 0..3
            const int sidx = col >> 4, q = (col & 15) >> 2;
#pragma unroll
            for (int i = 0; i < 4; ++i) {                 // element i: k-step i / 2, b0 / b1 = i % 2
                const float hi = __uint_as_float(tf32_hi(e[i]));
                const float lo = e[i] - hi;
                const size_t base = ((((size_t)sidx * 2 + (i >> 1)) * NTILES + nt) * 32 + (n * 4 + q)) * 4;
                bfl[base + (i & 1)] = hi;
                bfl[base + 2 + (i & 1)] = lo;
            }
        }
    }
    __syncthreads();
    const float sigma = sigma_dev ? __ldg(sigma_dev) : 1.0f;
    const int rq = lane >> 2, q = lane & 3;               // fragment row (and row + 8), quad column
    const int64_t n_tiles = (n_rows + 15) / 16;
    for (int64_t tile = (int64_t)blockIdx.x * COS2_WARPS + warp; tile < n_tiles; tile += (int64_t)gridDim.x * COS2_WARPS) {
        const int64_t ra = tile * 16 + rq, rb = ra + 8;
        const bool va = ra < n_rows, vb = rb < n_rows;
        const T* pa = x + (va ? ra : 0) * D + 4 * q;
        const T* pb = x + (vb ? rb : 0) * D + 4 * q;
        float acc[NTILES][4];
#pragma unroll
        for (int nt = 0; nt < NTILES; ++nt) { acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f; }
        float ssa = 0.f, ssb = 0.f;
        // software pipeline over groups of 4 column chunks (64 columns): the next group's loads are in flight under this group's MMAs
        float4 xa[4], xb[4], ya[4], yb[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { xa[i] = XQuad<T>::load(pa + 16 * i); xb[i] = XQuad<T>::load(pb + 16 * i); }
#pragma unroll 1
        for (int g = 0; g < 8; ++g) {
            if (g < 7) {
#pragma unroll
                for (int i = 0; i < 4; ++i) { ya[i] = XQuad<T>::load(pa + 16 * (4 * g + 4 + i)); yb[i] = XQuad<T>::load(pb + 16 * (4 * g + 4 + i)); }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int sidx = 4 * g + i;
                const float ea[4] = {xa[i].x, xa[i].y, xa[i].z, xa[i].w}, eb[4] = {xb[i].x, xb[i].y, xb[i].z, xb[i].w};
                ssa = fmaf(ea[0], ea[0], fmaf(ea[1], ea[1], fmaf(ea[2], ea[2], fmaf(ea[3], ea[3], ssa))));
                ssb = fmaf(eb[0], eb[0], fmaf(eb[1], eb[1], fmaf(eb[2], eb[2], fmaf(eb[3], eb[3], ssb))));
#pragma unroll
                for (int j = 0; j < 2; ++j) {             // k-step j of the chunk: a0 / a2 = elements 2j, 2j + 1 of row a; a1 / a3 of row b
                    uint32_t h0, h1, h2, h3, l0 = 0, l1 = 0, l2 = 0, l3 = 0;
                    if (XQuad<T>::EXACT) {
                        h0 = __float_as_uint(ea[2 * j]); h1 = __float_as_uint(eb[2 * j]);
                        h2 = __float_as_uint(ea[2 * j + 1]); h3 = __float_as_uint(eb[2 * j + 1]);
                    } else {
                        h0 = tf32_hi(ea[2 * j]); h1 = tf32_hi(eb[2 * j]); h2 = tf32_hi(ea[2 * j + 1]); h3 = tf32_hi(eb[2 * j + 1]);
                        l0 = __float_as_uint(ea[2 * j] - __uint_as_float(h0)); l1 = __float_as_uint(eb[2 * j] - __uint_as_float(h1));
                        l2 = __float_as_uint(ea[2 * j + 1] - __uint_as_float(h2)); l3 = __float_as_uint(eb[2 * j + 1] - __uint_as_float(h3));
                    }
#pragma unroll
                    for (int nt = 0; nt < NTILES; ++nt) {
                        const float4 b = bf[(((size_t)sidx * 2 + j) * NTILES + nt) * 32 + lane];
                        if (!XQuad<T>::EXACT) mma_tf32(acc[nt], l0, l1, l2, l3, __float_as_uint(b.x), __float_as_uint(b.y));
                        mma_tf32(acc[nt], h0, h1, h2, h3, __float_as_uint(b.z), __float_as_uint(b.w));
                        mma_tf32(acc[nt], h0, h1, h2, h3, __float_as_uint(b.x), __float_as_uint(b.y));
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) { xa[i] = ya[i]; xb[i] = yb[i]; }
        }
        // row norms: the four lanes of a quad hold the four column quarters of rows ra / rb
        ssa += __shfl_xor_sync(0xffffffffu, ssa, 1); ssa += __shfl_xor_sync(0xffffffffu, ssa, 2);
        ssb += __shfl_xor_sync(0xffffffffu, ssb, 1); ssb += __shfl_xor_sync(0xffffffffu, ssb, 2);
        const float sa = sigma / fmaxf(sqrtf(ssa), NORM_EPS), sb = sigma / fmaxf(sqrtf(ssb), NORM_EPS);
        // accumulator fragment: acc[nt][0..1] = row ra, classes 8 nt + 2 q, + 1;  acc[nt][2..3] = row rb
        float ba = -INFINITY, bb = -INFINITY;
        int ia = 0x7fffffff, ib = 0x7fffffff;
#pragma unroll
        for (int nt = 0; nt < NTILES; ++nt) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = 8 * nt + 2 * q + e;
                const float la = acc[nt][e] * sa, lb = acc[nt][2 + e] * sb;
                if (c < nc) {
                    if (logits != nullptr) {
                        if (va) logits[ra * num_classes + c0 + c] = la;
                        if (vb) logits[rb * num_classes + c0 + c] = lb;
                    }
                    if (la > ba) { ba = la; ia = c; }     // ascending c: ties keep the lower index
                    if (lb > bb) { bb = lb; ib = c; }
                }
            }
        }
        if (argmax_out != nullptr) {
#pragma unroll
            for (int o = 1; o <= 2; o <<= 1) {            // over the quad: max value, ties -> lower index (torch.max)
                const float oa = __shfl_xor_sync(0xffffffffu, ba, o); const int oia = __shfl_xor_sync(0xffffffffu, ia, o);
                if (oa > ba || (oa == ba && oia < ia)) { ba = oa; ia = oia; }
                const float ob = __shfl_xor_sync(0xffffffffu, bb, o); const int oib = __shfl_xor_sync(0xffffffffu, ib, o);
                if (ob > bb || (ob == bb && oib < ib)) { bb = ob; ib = oib; }
            }
            if (q == 0) {
                if (n_chunks == 1) {
                    if (va) argmax_out[ra] = c0 + ia;
                    if (vb) argmax_out[rb] = c0 + ib;
                } else {
                    if (va) { chunk_best[(ra * n_chunks + blockIdx.y) * 2] = ba; chunk_best[(ra * n_chunks + blockIdx.y) * 2 + 1] = __int_as_float(c0 + ia); }
                    if (vb) { chunk_best[(rb * n_chunks + blockIdx.y) * 2] = bb; chunk_best[(rb * n_chunks + blockIdx.y) * 2 + 1] = __int_as_float(c0 + ib); }
                }
            }
        }
    }
}

template <typename T, int NTILES>
static int cosine_mma_launch(cudaStream_t st, dim3 grid, const void* x, int64_t n_rows, const float* w, int num_classes,
                             const float* sigma_dev, float* logits, int64_t* argmax, float* chunk_best, int n_chunks) {
    const size_t smem = (size_t)32 * 2 * NTILES * 32 * sizeof(float4);
    TEAM_CUDA_CHECK(cudaFuncSetAttribute(cosine_mma_kernel<T, NTILES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cosine_mma_kernel<T, NTILES><<<grid, COS2_WARPS * 32, smem, st>>>(reinterpret_cast<const T*>(x), n_rows, w, num_classes, sigma_dev, logits, argmax, chunk_best, n_chunks);
    count_launch();
    TEAM_LAUNCH_CHECK("cosine_mma_kernel");
    return TEAM_OK;
}

__global__ void cosine_argmax_merge(const float* __restrict__ chunk_best, int64_t n_rows, int n_chunks,
                                    int64_t* __restrict__ argmax_out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    float best = -INFINITY;
    int bi = 0;
    for (int q = 0; q < n_chunks; ++q) {
        const float v = chunk_best[(r * n_chunks + q) * 2];
        const int i = __float_as_int(chunk_best[(r * n_chunks + q) * 2 + 1]);
        if (q == 0 || v > best) { best = v; bi = i; }
    }
    argmax_out[r] = bi;
}

}  // namespace team

using namespace team;

int team::cosine_logits_launch(cudaStream_t st, const float* x, int64_t n_rows, const float* w, int64_t num_classes,
                               const float* sigma_dev, float* logits, int64_t* argmax) {
    return team_cosine_logits(x, TEAM_DTYPE_F32, n_rows, w, num_classes, sigma_dev, logits, argmax, (void*)st);
}

extern "C" int team_cosine_logits(const void* x, int x_dtype, int64_t n_rows, const float* w,
                                  int64_t num_classes, const float* sigma_dev, float* logits,
                                  int64_t* argmax, void* stream) {
    TEAM_REQUIRE(x != nullptr && w != nullptr && n_rows >= 0 && num_classes >= 1, "team_cosine_logits: bad args");
    TEAM_REQUIRE(x_dtype == TEAM_DTYPE_F32 || x_dtype == TEAM_DTYPE_BF16, "team_cosine_logits: bad dtype %d", x_dtype);
    if (n_rows == 0) return TEAM_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int n_chunks = (int)((num_classes + COS_CCHUNK - 1) / COS_CCHUNK);
    float* chunk_best = nullptr;
    if (n_chunks > 1 && argmax != nullptr) {
        // rare path (C > 32): scratch from the stream-ordered allocator
        TEAM_CUDA_CHECK(cudaMallocAsync((void**)&chunk_best, (size_t)n_rows * n_chunks * 2 * sizeof(float), st));
    }
    // Small inputs (the classification logits of a 1 024-sample step): the tensor-pipe kernel is its prologue there (every CTA
    // normalises and hi/lo-splits the whole class table: 19 us on 8 CTAs at 1 024 rows, on the forward's critical path beside
    // the table rows) - the CUDA-core kernel takes 8 us on 64 CTAs.  From 8 192 rows the streaming rate decides.
    if (n_rows > 8192) {          // tensor-pipe contraction (3xTF32), see cosine_mma_kernel
        const int nt = (int)((((num_classes < COS_CCHUNK ? num_classes : COS_CCHUNK)) + 7) / 8);
        const int64_t tiles = (n_rows + 15) / 16;
        int64_t gx2 = (tiles + COS2_WARPS - 1) / COS2_WARPS;
        const int64_t cap2 = (int64_t)NUM_SMS * (nt <= 2 ? 3 : (nt == 3 ? 2 : 1));     // CTAs per SM by shared memory (32 KB per n-tile)
        if (gx2 > cap2) gx2 = cap2;
        dim3 grid2((unsigned)gx2, (unsigned)n_chunks, 1);
        int rc;
#define COS_GO(T) (nt == 1 ? cosine_mma_launch<T, 1>(st, grid2, x, n_rows, w, (int)num_classes, sigma_dev, logits, argmax, chunk_best, n_chunks) \
                 : nt == 2 ? cosine_mma_launch<T, 2>(st, grid2, x, n_rows, w, (int)num_classes, sigma_dev, logits, argmax, chunk_best, n_chunks) \
                 : nt == 3 ? cosine_mma_launch<T, 3>(st, grid2, x, n_rows, w, (int)num_classes, sigma_dev, logits, argmax, chunk_best, n_chunks) \
                           : cosine_mma_launch<T, 4>(st, grid2, x, n_rows, w, (int)num_classes, sigma_dev, logits, argmax, chunk_best, n_chunks))
        rc = x_dtype == TEAM_DTYPE_F32 ? COS_GO(float) : COS_GO(__nv_bfloat16);
#undef COS_GO
        if (rc) return rc;
    } else {
    const int64_t n_pairs = (n_rows + 1) / 2;
    int64_t gx = (n_pairs + COS_WARPS - 1) / COS_WARPS;
    const int64_t cap = (int64_t)NUM_SMS * 2;          // persistent over row pairs (register-limited to 2 CTAs / SM)
    if (gx > cap) gx = cap;
    dim3 grid((unsigned)gx, (unsigned)n_chunks, 1);
    const size_t smem = (size_t)(num_classes < COS_CCHUNK ? num_classes : COS_CCHUNK) * D * sizeof(float);
    if (x_dtype == TEAM_DTYPE_F32) {
        TEAM_CUDA_CHECK(cudaFuncSetAttribute(cosine_logits_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cosine_logits_kernel<float><<<grid, COS_WARPS * 32, smem, st>>>(reinterpret_cast<const float*>(x), n_rows, w, (int)num_classes, sigma_dev, logits, argmax, chunk_best, n_chunks);
    } else {
        TEAM_CUDA_CHECK(cudaFuncSetAttribute(cosine_logits_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cosine_logits_kernel<__nv_bfloat16><<<grid, COS_WARPS * 32, smem, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), n_rows, w, (int)num_classes, sigma_dev, logits, argmax, chunk_best, n_chunks);
    }
    TEAM_LAUNCH_CHECK("cosine_logits_kernel");
    }
    if (chunk_best != nullptr) {
        cosine_argmax_merge<<<(unsigned)((n_rows + 255) / 256), 256, 0, st>>>(chunk_best, n_rows, n_chunks, argmax);
        TEAM_LAUNCH_CHECK("cosine_argmax_merge");
        TEAM_CUDA_CHECK(cudaFreeAsync(chunk_best, st));
    }
    return TEAM_OK;
}
