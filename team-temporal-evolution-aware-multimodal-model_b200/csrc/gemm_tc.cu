// tcgen05 / TMA / TMEM bf16 grouped GEMM for sm_100a (TEAM_MODE_BF16).
//
//   for every problem p of a group:  C_p[M,N] = alpha * op(A_p) op(B_p) (+ bias[N]) (+ beta * C_p)
//   written as fp32 and/or bf16 (the bf16 copy is what the next GEMM of the head consumes, so no
//   separate conversion pass exists); fp32 accumulation in tensor memory.
//
// ONE launch runs up to TC_MAXP independent problems (the head's many small GEMMs have <= 64 output
// tiles each and would leave most of the 148 SMs idle one at a time): the problem table - tensor
// maps included - travels as a __grid_constant__ kernel parameter, so a captured CUDA graph holds it
// by value.  CTA = one 128 x BN output tile of one problem (x one split of K).
//
//   operands : bf16 in global memory -> shared memory through TMA (cp.async.bulk.tensor.2d,
//              SWIZZLE_128B) into a 3-stage mbarrier ring; either operand K-major (row-major
//              [rows,K]) or MN-major (row-major [K,rows]) via the UMMA descriptor major bits, so
//              A^T B / A B products of the backward need no transposed copies.
//   math     : one elected thread issues tcgen05.mma (UMMA 128 x BN x 16, cta_group::1), BN runtime
//              (multiple of 16, <= 128); the accumulator lives in TMEM.
//   epilogue : tcgen05.ld (warp w owns TMEM lanes 32w..32w+31) -> padded shared-memory tile ->
//              row-contiguous 128-bit global stores (fp32) / 64-bit (bf16).
//   split-K  : the 2 / 4 / 8 CTAs that share an output tile form (part of) a thread-block CLUSTER; each keeps
//              its fp32 partial tile in its own shared memory and, after a cluster barrier, reduces one
//              row slice of the tile over all partials through distributed shared memory
//              (ld.shared::cluster) in split order - deterministic, no global-memory round trip, no
//              second kernel - and runs the epilogue for that slice.
//   PDL      : griddepcontrol.launch_dependents / .wait bracket the prologue (barrier init, TMEM
//              alloc, tensor-map prefetch) so it overlaps the previous kernel's tail when the launch
//              carries the programmatic-stream-serialization attribute.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <mutex>
#include <stdlib.h>
#include "gemm.cuh"
#include "prof.cuh"

namespace team {

constexpr int TC_BM = 128;           // UMMA_M
constexpr int TC_BK = 64;            // 64 bf16 = 128 B = one SWIZZLE_128B row
constexpr int TC_UMMA_K = 16;
constexpr int TC_THREADS = 128;
constexpr int TC_STAGES = 3;          // 2 CTAs / SM (multi-wave launches)
constexpr int TC_MAX_STAGES = 6;      // 1 CTA / SM: single-wave launches keep twice the bytes in flight per CTA
constexpr int TC_MAX_BN = 128;
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;          // 16 KB
constexpr int TC_B_BYTES = TC_MAX_BN * TC_BK * 2;      // 16 KB
constexpr int TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr int tc_smem_bytes(int stages) { return stages * TC_STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/; }   // 3 stages: 97.25 KB -> 2 CTAs / SM
constexpr uint32_t TC_TMEM_COLS = 128;
constexpr int TC_MAX_SPLITS = 8;     // = largest portable cluster size
constexpr int TC_TARGET_CTAS = 2 * NUM_SMS;

static_assert(TC_BM * (TC_MAX_BN + 4) * 4 <= TC_STAGES * TC_STAGE_BYTES, "epilogue staging must fit in the operand ring");

struct alignas(64) TcSegDev {
    CUtensorMap ma, mb;
    int K, nkb, a_mn, b_mn;
};
struct alignas(64) TcProb {
    TcSegDev s[2];            // K-segments accumulated into the same TMEM tile (s[1].nkb == 0: single segment)
    float* C;
    __nv_bfloat16* Cb;
    const float* bias;
    long long ldc, ldcb;
    float alpha, beta;
    int M, N;
    int bn, tiles_n, n_tiles, cta_begin, splits, kb_per_split;
};
struct TcGroup {
    TcProb p[TC_MAXP];
    int n;
    int stages;
    int cluster;                 // CTAs per cluster (1, 2, 4 or 8) = largest split count of the group
    unsigned long long* dbg;     // optional [cta][16] globaltimer stamps (tools/gemm_probe.py), else null
};
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define TC_STAMP(slot) do { if (g.dbg != nullptr && blockIdx.x < 1024) g.dbg[(size_t)blockIdx.x * 16 + (slot)] = gtime(); } while (0)

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a wrong descriptor / byte count traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t spin = 0; !mbar_try_wait(bar, parity); ++spin)
        if (spin > (1u << 24)) __trap();
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tcgen05_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ float4 ld_cluster_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// shared-memory matrix descriptors (SWIZZLE_128B, descriptor version 1)
//   K-major : rows of 128 B (64 bf16 along K); 8-row groups SBO = 1024 B apart.
//   MN-major: rows of 128 B (64 bf16 along M/N), one row per k; 8-k groups SBO = 1024 B apart;
//             64-element M/N chunks LBO bytes apart.
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor, kind::f16: D=f32, A / B format bf16 (1) @7 / @10, majors, N>>3 @17, M>>4 @24
__host__ __device__ inline uint32_t umma_idesc(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// grid = total CTAs of the group; 128 threads.
__global__ void __launch_bounds__(TC_THREADS)
gemm_bf16_tcgen05_kernel(const __grid_constant__ TcGroup g) {
    extern __shared__ unsigned char tc_smem_raw[];
    // pointer arithmetic on the __shared__ array (not an integer round trip) keeps the shared address space -> LDS/STS
    unsigned char* smem = tc_smem_raw + ((1024u - (smem_u32(tc_smem_raw) & 1023u)) & 1023u);
    const int nstages = g.stages;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + nstages * TC_STAGE_BYTES);
    uint64_t* empty_bar = full_bar + TC_MAX_STAGES;
    uint64_t* tmem_full_bar = empty_bar + TC_MAX_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    if (threadIdx.x == 0) TC_STAMP(0);

    int pi = 0;
    for (int i = 1; i < g.n; ++i)
        if ((int)blockIdx.x >= g.p[i].cta_begin) pi = i;
    const TcProb& P = g.p[pi];
    const int local = (int)blockIdx.x - P.cta_begin;
    const int split = local % P.splits, tile = local / P.splits;
    if (tile >= P.n_tiles) {           // padding CTA of a cluster: only keeps the cluster barriers balanced
        if (P.splits > 1) { cluster_sync_all(); cluster_sync_all(); }
        return;
    }
    const int m0 = (tile / P.tiles_n) * TC_BM, bn = P.bn, n0 = (tile % P.tiles_n) * bn;
    const int nkb0 = P.s[0].nkb;
    const int nkb = nkb0 + P.s[1].nkb;
    const int kb_begin = split * P.kb_per_split;
    const int kb_end = min(nkb, kb_begin + P.kb_per_split);

    if (threadIdx.x == 0) {
        for (int s = 0; s < nstages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&P.s[0].ma)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&P.s[0].mb)) : "memory");
        if (P.s[1].nkb > 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&P.s[1].ma)) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&P.s[1].mb)) : "memory");
        }
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TC_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    // PDL: let the next kernel start its own prologue; wait until everything before us has completed
    if (threadIdx.x == 0) TC_STAMP(1);
    pdl_wait();
    if (threadIdx.x == 0) TC_STAMP(2);

    if (threadIdx.x == 0) {
        // ===================== TMA producer =====================
        const uint32_t tx_bytes = (uint32_t)(TC_A_BYTES + bn * TC_BK * 2);
        int stage = 0; uint32_t phase = 0;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            unsigned char* sa = smem + stage * TC_STAGE_BYTES;
            unsigned char* sb = sa + TC_A_BYTES;
            mbar_expect_tx(&full_bar[stage], tx_bytes);
            const TcSegDev& sg = P.s[kb >= nkb0 ? 1 : 0];
            const int k0 = (kb >= nkb0 ? kb - nkb0 : kb) * TC_BK;
            if (!sg.a_mn) {
                tma_load_2d(sa, &sg.ma, &full_bar[stage], k0, m0);                     // box {64 k, 128 rows}
            } else {
#pragma unroll
                for (int c = 0; c < TC_BM / 64; ++c)                                    // box {64 m, 64 k} per chunk
                    tma_load_2d(sa + c * (TC_BK * 128), &sg.ma, &full_bar[stage], m0 + 64 * c, k0);
            }
            if (!sg.b_mn) {
                tma_load_2d(sb, &sg.mb, &full_bar[stage], k0, n0);                     // box {64 k, bn rows}
            } else {
                for (int c = 0; c < bn / 64; ++c)
                    tma_load_2d(sb + c * (TC_BK * 128), &sg.mb, &full_bar[stage], n0 + 64 * c, k0);
            }
            if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
        TC_STAMP(3);
    } else if (threadIdx.x == 32) {
        // ===================== MMA issuer (one thread) =====================
        const uint32_t idesc0 = umma_idesc(TC_BM, bn, P.s[0].a_mn, P.s[0].b_mn);
        const uint32_t idesc1 = umma_idesc(TC_BM, bn, P.s[1].a_mn, P.s[1].b_mn);
        int stage = 0; uint32_t phase = 0;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
            const int si = kb >= nkb0 ? 1 : 0;
            const int a_mn = P.s[si].a_mn, b_mn = P.s[si].b_mn;
            const uint32_t idesc = si ? idesc1 : idesc0;
            mbar_wait(&full_bar[stage], phase);
            if (kb == kb_begin) TC_STAMP(4);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t sa = smem_u32(smem + stage * TC_STAGE_BYTES);
            const uint32_t sb = sa + TC_A_BYTES;
#pragma unroll
            for (int k = 0; k < TC_BK / TC_UMMA_K; ++k) {
                const uint64_t ad = a_mn ? umma_desc(sa + k * 2048, TC_BK * 128, 1024) : umma_desc(sa + k * 32, 0, 1024);
                const uint64_t bd = b_mn ? umma_desc(sb + k * 2048, TC_BK * 128, 1024) : umma_desc(sb + k * 32, 0, 1024);
                tcgen05_mma_f16(tmem_base, ad, bd, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
            }
            tcgen05_commit(&empty_bar[stage]);          // smem slot free once these MMAs retire
            if (++stage == nstages) { stage = 0; phase ^= 1; }
        }
        tcgen05_commit(tmem_full_bar);                  // accumulator complete (and every smem read retired)
    }
    // ===================== epilogue: all 4 warps =====================
    __syncwarp();
    mbar_wait(tmem_full_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (threadIdx.x == 64) TC_STAMP(5);

    // TMEM -> padded smem tile (the operand ring is idle now); thread = one accumulator row
    float* stg = reinterpret_cast<float*>(smem);
    const int sld = bn + 4;
    float* my = stg + (size_t)(warp * 32 + lane) * sld;
    const uint32_t tbase = tmem_base + ((uint32_t)(warp * 32) << 16);
    int c = 0;
    for (; c + 32 <= bn; c += 32) {              // two 16-column loads in flight per wait
        uint32_t r[32];
        tmem_ld16_nowait(tbase + (uint32_t)c, r);
        tmem_ld16_nowait(tbase + (uint32_t)(c + 16), r + 16);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int i = 0; i < 32; i += 4)
            *reinterpret_cast<float4*>(my + c + i) = make_float4(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
    }
    if (c < bn) {
        uint32_t r[16];
        tmem_ld16_nowait(tbase + (uint32_t)c, r);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int i = 0; i < 16; i += 4)
            *reinterpret_cast<float4*>(my + c + i) = make_float4(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
    }
    if (threadIdx.x == 64) TC_STAMP(8);
    // split-K: every CTA of the tile publishes its partial (cluster barrier), then owns rows [row0, row0 + nrow)
    const int splits = P.splits;
    int row0 = 0, nrow = TC_BM;
    uint32_t rank0 = 0;
    if (splits > 1) {
        cluster_sync_all();
        nrow = TC_BM / splits;
        row0 = split * nrow;
        uint32_t myrank;
        asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(myrank));
        rank0 = myrank - (uint32_t)split;              // rank of split 0 of this tile
    } else {
        __syncthreads();
    }
    if (threadIdx.x == 64) TC_STAMP(9);
    const int M = P.M, N = P.N;
    float* const C = P.C;
    __nv_bfloat16* const Cb = P.Cb;
    const long long ldc = P.ldc, ldcb = P.ldcb;
    const bool vec_ok = (N % 4 == 0) && (C == nullptr || ((ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0))) &&
                        (Cb == nullptr || ((ldcb % 4 == 0) && ((reinterpret_cast<uintptr_t>(Cb) & 7) == 0)));
    const float alpha = P.alpha, beta = P.beta;
    const bool acc_c = beta != 0.f && C != nullptr;
    const float* bias = P.bias;
    // thread -> (row offset r_off, float4 column c4): lanes run along the columns, rpp rows per pass
    const int lpr = bn >> 2;                                   // float4 columns per row (4..32)
    const int rpp = TC_THREADS / lpr;                          // rows per pass (4..32)
    const int r_off = (int)threadIdx.x / lpr, c4 = (int)threadIdx.x - r_off * lpr;
    const int col = n0 + 4 * c4;
    if (r_off < rpp && col < N) {
        float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (bias != nullptr) {
            bv.x = __ldg(bias + col);
            if (col + 1 < N) bv.y = __ldg(bias + col + 1);
            if (col + 2 < N) bv.z = __ldg(bias + col + 2);
            if (col + 3 < N) bv.w = __ldg(bias + col + 3);
        }
        // rows of this thread: row0 + r_off + q * rpp, q = 0 .. nq-1, clipped to the slice and to M
        int nq = (nrow - r_off + rpp - 1) / rpp;
        {
            const int left = M - (m0 + row0 + r_off);
            const int cap = left <= 0 ? 0 : (left + rpp - 1) / rpp;
            if (cap < nq) nq = cap;
        }
        const uint32_t stg_addr = smem_u32(stg);
        const uint32_t off0 = (uint32_t)(((row0 + r_off) * sld + 4 * c4) * 4), ostep = (uint32_t)(rpp * sld * 4);
        const unsigned char* lp = reinterpret_cast<const unsigned char*>(stg) + off0;
        uint32_t rbase[TC_MAX_SPLITS];
#pragma unroll
        for (int z = 0; z < TC_MAX_SPLITS; ++z) rbase[z] = z < splits ? map_to_cta(stg_addr + off0, rank0 + (uint32_t)z) : 0u;
        float* cp = C != nullptr ? C + (long long)(m0 + row0 + r_off) * ldc + col : nullptr;
        __nv_bfloat16* bp = Cb != nullptr ? Cb + (long long)(m0 + row0 + r_off) * ldcb + col : nullptr;
        const long long cstep = (long long)rpp * ldc, bstep = (long long)rpp * ldcb;
        constexpr int UN = 8;                                  // rows in flight per thread
        for (int q0 = 0; q0 < nq; q0 += UN) {
            float4 v[UN], o[UN];
            if (splits == 1) {
#pragma unroll
                for (int j = 0; j < UN; ++j)
                    if (q0 + j < nq) v[j] = *reinterpret_cast<const float4*>(lp + (size_t)(q0 + j) * ostep);
            } else {
#pragma unroll
                for (int j = 0; j < UN; ++j)
                    if (q0 + j < nq) v[j] = ld_cluster_f4(rbase[0] + (uint32_t)(q0 + j) * ostep);
#pragma unroll
                for (int z = 1; z < TC_MAX_SPLITS; ++z) {      // fixed order: deterministic
                    if (z >= splits) break;
                    float4 a[UN];
#pragma unroll
                    for (int j = 0; j < UN; ++j)
                        if (q0 + j < nq) a[j] = ld_cluster_f4(rbase[z] + (uint32_t)(q0 + j) * ostep);
#pragma unroll
                    for (int j = 0; j < UN; ++j)
                        if (q0 + j < nq) { v[j].x += a[j].x; v[j].y += a[j].y; v[j].z += a[j].z; v[j].w += a[j].w; }
                }
            }
            if (acc_c && vec_ok) {
#pragma unroll
                for (int j = 0; j < UN; ++j)
                    if (q0 + j < nq) o[j] = *reinterpret_cast<const float4*>(cp + (q0 + j) * cstep);
            }
#pragma unroll
            for (int j = 0; j < UN; ++j) {
                if (q0 + j >= nq) continue;
                float4 x = make_float4(fmaf(alpha, v[j].x, bv.x), fmaf(alpha, v[j].y, bv.y), fmaf(alpha, v[j].z, bv.z), fmaf(alpha, v[j].w, bv.w));
                if (vec_ok) {
                    if (acc_c) { x.x = fmaf(beta, o[j].x, x.x); x.y = fmaf(beta, o[j].y, x.y); x.z = fmaf(beta, o[j].z, x.z); x.w = fmaf(beta, o[j].w, x.w); }
                    if (cp != nullptr) *reinterpret_cast<float4*>(cp + (q0 + j) * cstep) = x;
                    if (bp != nullptr) *reinterpret_cast<uint2*>(bp + (q0 + j) * bstep) = pack_bf16x4(x);
                } else {
                    // ragged N / unaligned outputs: element-wise with guards
                    const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (col + i >= N) continue;
                        float y = xs[i];
                        if (cp != nullptr) {
                            float* dst = cp + (q0 + j) * cstep + i;
                            if (acc_c) y = fmaf(beta, *dst, y);
                            *dst = y;
                        }
                        if (bp != nullptr) bp[(q0 + j) * bstep + i] = __float2bfloat16_rn(y);
                    }
                }
            }
        }
    }
    if (splits > 1) cluster_sync_all();        // peers may still be reading this CTA's partial
    if (threadIdx.x == 64) TC_STAMP(6);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) TC_STAMP(7);
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
    }
}

// =========================================================================================================
// Persistent variant for LARGE launches (many more tiles than SMs): one CTA per SM walks a static list of work
// items (problem, 128 x BN tile, K split), BN up to 256.
//   warp 0     : TMA producer - keeps a 3-stage ring of {A 128x64, B BNx64} k-blocks full ACROSS tiles
//   warp 1     : MMA issuer   - tcgen05.mma into one of TWO tensor-memory accumulators (2 x 256 columns)
//   warps 2..9 : epilogue     - tcgen05.ld of accumulator i while the tensor pipe already fills accumulator i+1;
//                warp (q, half) owns 32 accumulator rows and every other 32-column chunk, stages a chunk through
//                its own padded shared-memory patch (the next chunk's TMEM load already in flight) and stores
//                row-contiguous 128-byte segments (fp32) / 64-byte (bf16)
// so neither the prologue (barriers, TMEM allocation, tensor-map fetch) nor the epilogue of a tile is exposed,
// and a 128 x 256 tile needs 25 % less L2 -> SM operand traffic per flop than 128 x 128 (these K = 512 products
// are bound by that traffic, not by the tensor pipe).
//   split-K : long-K / few-tile problems (weight gradients, K = 2B) are cut into items of equal k-range; every
//             item stores its fp32 partial tile to the workspace and a small second kernel (pk_fixup_kernel, all SMs)
//             sums the partials in split order (deterministic) and runs the epilogue.  (A "last arriver reduces"
//             ticket scheme was measured first: one CTA pulling 16 x 128 KB of partials takes ~100 us and stalls
//             its remaining items.)
constexpr int PK_BN_MAX = 256;
constexpr int PK_STAGES = 3;
constexpr int PK_A_BYTES = TC_BM * TC_BK * 2;                 // 16 KB
constexpr int PK_B_BYTES = PK_BN_MAX * TC_BK * 2;             // 32 KB
constexpr int PK_STAGE_BYTES = PK_A_BYTES + PK_B_BYTES;       // 48 KB
constexpr int PK_EPI_LD = 36;                                 // floats per staged row: 32 + 4 (conflict-free both ways)
constexpr int PK_EPI_BYTES = 8 * 32 * PK_EPI_LD * 4;          // 8 epilogue warps x 32 rows
constexpr int PK_THREADS = 320;                               // producer warp, MMA warp, 8 epilogue warps
constexpr int PK_SMEM_BYTES = PK_STAGES * PK_STAGE_BYTES + PK_EPI_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
static_assert(PK_SMEM_BYTES <= 227 * 1024, "persistent GEMM: shared memory budget");

struct alignas(64) PkProb {
    TcSegDev s[2];
    float* C;
    __nv_bfloat16* Cb;
    const float* bias;
    long long ldc, ldcb;
    float alpha, beta;
    int M, N;
    int bn, tiles_n, n_tiles, item_begin, splits, kb_per_split;
    float* partials;              // [n_tiles][splits][128][bn] fp32 (splits > 1): summed by pk_fixup_kernel
};
struct PkGroup {
    PkProb p[TC_MAXP];
    int n;
    int total_items;
    unsigned long long* dbg;      // optional [cta < 148][item < 8][8] globaltimer stamps (tools/pk_stamps.py), else null
};
#define PK_STAMP(n_it, slot) do { if (g.dbg != nullptr && (n_it) < 8) g.dbg[((size_t)blockIdx.x * 8 + (n_it)) * 8 + (slot)] = gtime(); } while (0)
struct PkItem {
    int pi, tile, split, m0, n0, bn, kb_begin, kb_end, nkb0;
};
__device__ __forceinline__ PkItem pk_decode(const PkGroup& g, int item) {
    PkItem it;
    int pi = 0;
    for (int i = 1; i < g.n; ++i)
        if (item >= g.p[i].item_begin) pi = i;
    const PkProb& P = g.p[pi];
    const int local = item - P.item_begin;
    it.pi = pi;
    it.split = local % P.splits;
    it.tile = local / P.splits;
    it.bn = P.bn;
    it.m0 = (it.tile / P.tiles_n) * TC_BM;
    it.n0 = (it.tile % P.tiles_n) * P.bn;
    it.nkb0 = P.s[0].nkb;
    const int nkb = P.s[0].nkb + P.s[1].nkb;
    it.kb_begin = it.split * P.kb_per_split;
    it.kb_end = min(nkb, it.kb_begin + P.kb_per_split);
    return it;
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

__global__ void __launch_bounds__(PK_THREADS, 1)
gemm_bf16_persistent_kernel(const __grid_constant__ PkGroup g) {
    extern __shared__ unsigned char tc_smem_raw[];
    unsigned char* smem = tc_smem_raw + ((1024u - (smem_u32(tc_smem_raw) & 1023u)) & 1023u);
    float* epi_all = reinterpret_cast<float*>(smem + PK_STAGES * PK_STAGE_BYTES);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + PK_STAGES * PK_STAGE_BYTES + PK_EPI_BYTES);
    uint64_t* empty_bar = full_bar + PK_STAGES;
    uint64_t* acc_full = empty_bar + PK_STAGES;        // [2]
    uint64_t* acc_empty = acc_full + 2;                // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    if (threadIdx.x == 0) {
        for (int s = 0; s < PK_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int i = 0; i < g.n; ++i) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&g.p[i].s[0].ma)) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&g.p[i].s[0].mb)) : "memory");
        }
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();

    if (warp == 0) {
        if (lane == 0) {
            // ===================== TMA producer =====================
            int stage = 0; uint32_t phase = 0;
            int n_it = 0;
            for (int item = blockIdx.x; item < g.total_items; item += gridDim.x, ++n_it) {
                const PkItem it = pk_decode(g, item);
                const PkProb& P = g.p[it.pi];
                const uint32_t tx_bytes = (uint32_t)(PK_A_BYTES + it.bn * TC_BK * 2);
                PK_STAMP(n_it, 0);
                for (int kb = it.kb_begin; kb < it.kb_end; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    unsigned char* sa = smem + stage * PK_STAGE_BYTES;
                    unsigned char* sb = sa + PK_A_BYTES;
                    mbar_expect_tx(&full_bar[stage], tx_bytes);
                    const TcSegDev& sg = P.s[kb >= it.nkb0 ? 1 : 0];
                    const int k0 = (kb >= it.nkb0 ? kb - it.nkb0 : kb) * TC_BK;
                    if (!sg.a_mn) {
                        tma_load_2d(sa, &sg.ma, &full_bar[stage], k0, it.m0);
                    } else {
#pragma unroll
                        for (int c = 0; c < TC_BM / 64; ++c)
                            tma_load_2d(sa + c * (TC_BK * 128), &sg.ma, &full_bar[stage], it.m0 + 64 * c, k0);
                    }
                    if (!sg.b_mn) {
                        tma_load_2d(sb, &sg.mb, &full_bar[stage], k0, it.n0);
                    } else {
                        for (int c = 0; c < it.bn / 64; ++c)
                            tma_load_2d(sb + c * (TC_BK * 128), &sg.mb, &full_bar[stage], it.n0 + 64 * c, k0);
                    }
                    if (++stage == PK_STAGES) { stage = 0; phase ^= 1; }
                }
                PK_STAMP(n_it, 1);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ===================== MMA issuer =====================
            int stage = 0; uint32_t phase = 0;
            int n_it = 0;
            for (int item = blockIdx.x; item < g.total_items; item += gridDim.x, ++n_it) {
                const PkItem it = pk_decode(g, item);
                const PkProb& P = g.p[it.pi];
                const int buf = n_it & 1;
                const uint32_t accph = (uint32_t)(n_it >> 1) & 1u;
                mbar_wait(&acc_empty[buf], accph ^ 1);              // epilogue has drained this accumulator
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t d_tmem = tmem_base + (uint32_t)(buf * PK_BN_MAX);
                const uint32_t idesc0 = umma_idesc(TC_BM, it.bn, P.s[0].a_mn, P.s[0].b_mn);
                const uint32_t idesc1 = umma_idesc(TC_BM, it.bn, P.s[1].a_mn, P.s[1].b_mn);
                for (int kb = it.kb_begin; kb < it.kb_end; ++kb) {
                    const int si = kb >= it.nkb0 ? 1 : 0;
                    const int a_mn = P.s[si].a_mn, b_mn = P.s[si].b_mn;
                    const uint32_t idesc = si ? idesc1 : idesc0;
                    mbar_wait(&full_bar[stage], phase);
                    if (kb == it.kb_begin) PK_STAMP(n_it, 2);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t sa = smem_u32(smem + stage * PK_STAGE_BYTES);
                    const uint32_t sb = sa + PK_A_BYTES;
#pragma unroll
                    for (int k = 0; k < TC_BK / TC_UMMA_K; ++k) {
                        const uint64_t ad = a_mn ? umma_desc(sa + k * 2048, TC_BK * 128, 1024) : umma_desc(sa + k * 32, 0, 1024);
                        const uint64_t bd = b_mn ? umma_desc(sb + k * 2048, TC_BK * 128, 1024) : umma_desc(sb + k * 32, 0, 1024);
                        tcgen05_mma_f16(d_tmem, ad, bd, idesc, (kb > it.kb_begin || k > 0) ? 1u : 0u);
                    }
                    tcgen05_commit(&empty_bar[stage]);
                    if (++stage == PK_STAGES) { stage = 0; phase ^= 1; }
                }
                tcgen05_commit(&acc_full[buf]);
                PK_STAMP(n_it, 3);
            }
        }
    } else {
        // ===================== epilogue: 8 warps = 4 TMEM lane groups (q = warp % 4) x 2 column halves =====================
        // warp (q, half) owns accumulator rows 32q..32q+31 and the 32-column chunks ci with (ci & 1) == half.
        const int q = warp & 3, half = (warp - 2) >> 2;
        float* epi = epi_all + (size_t)(warp - 2) * 32 * PK_EPI_LD;
        int n_it = 0;
        for (int item = blockIdx.x; item < g.total_items; item += gridDim.x, ++n_it) {
            const PkItem it = pk_decode(g, item);
            const PkProb& P = g.p[it.pi];
            const int buf = n_it & 1;
            const uint32_t accph = (uint32_t)(n_it >> 1) & 1u;
            const int bn = it.bn, M = P.M, N = P.N, splits = P.splits;
            const float alpha = P.alpha, beta = P.beta;
            float* const C = P.C;
            __nv_bfloat16* const Cb = P.Cb;
            const float* const bias = P.bias;
            const long long ldc = P.ldc, ldcb = P.ldcb;
            const bool acc_c = beta != 0.f && C != nullptr;
            float* const part = splits > 1 ? P.partials + ((size_t)it.tile * splits + it.split) * (size_t)(TC_BM * bn) : nullptr;
            mbar_wait(&acc_full[buf], accph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (threadIdx.x == 64) { PK_STAMP(n_it, 4); if (g.dbg != nullptr && n_it < 8) g.dbg[((size_t)blockIdx.x * 8 + n_it) * 8 + 7] = (unsigned long long)(it.kb_end - it.kb_begin) | ((unsigned long long)it.pi << 32); }
            const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * PK_BN_MAX);
            const int nchunks = (bn + 31) >> 5;
            uint32_t r[32];
            int ci = half;
            if (ci < nchunks) {                              // first TMEM load of this warp
                if (bn - 32 * ci >= 32) tmem_ld32_nowait(tbase + (uint32_t)(32 * ci), r);
                else tmem_ld16_nowait(tbase + (uint32_t)(32 * ci), r);
            } else {                                         // nothing to read (bn <= 32 and half == 1): release at once
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[buf]);
            }
            for (; ci < nchunks; ci += 2) {
                const int c0 = 32 * ci;
                const int ncols = min(32, bn - c0);          // 32 or 16 (bn is a multiple of 16)
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                {
                    float* my = epi + lane * PK_EPI_LD;
#pragma unroll
                    for (int i = 0; i < 32; i += 4)
                        if (i < ncols) *reinterpret_cast<float4*>(my + i) = make_float4(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
                }
                if (ci + 2 < nchunks) {                      // next chunk's TMEM load flies under this chunk's stores
                    if (bn - (c0 + 64) >= 32) tmem_ld32_nowait(tbase + (uint32_t)(c0 + 64), r);
                    else tmem_ld16_nowait(tbase + (uint32_t)(c0 + 64), r);
                } else {                                     // accumulator fully read by this warp: hand it back
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[buf]);
                }
                __syncwarp();
                // row-contiguous phase: lpr lanes per row, rpi rows per instruction, lane rows r_off + j * rpi
                const int lpr = ncols == 32 ? 8 : 4, rpi = ncols == 32 ? 4 : 8;
                const int r_off = ncols == 32 ? (lane >> 3) : (lane >> 2), c4 = ncols == 32 ? (lane & 7) : (lane & 3);
                const int col = it.n0 + c0 + 4 * c4;
                if (col < N) {
                    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (bias != nullptr && part == nullptr) bv = __ldg(reinterpret_cast<const float4*>(bias + col));
                    const int row0 = it.m0 + q * 32 + r_off;
                    int nj = ncols == 32 ? 8 : 4;
                    {
                        const int left = M - row0;
                        const int cap = left <= 0 ? 0 : (left + rpi - 1) / rpi;
                        if (cap < nj) nj = cap;
                    }
                    (void)lpr;
                    const float* sp = epi + r_off * PK_EPI_LD + 4 * c4;
                    float4 v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (j < nj) v[j] = *reinterpret_cast<const float4*>(sp + j * rpi * PK_EPI_LD);
                    if (part != nullptr) {
                        float* dp = part + (size_t)(q * 32 + r_off) * bn + c0 + 4 * c4;
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (j < nj) *reinterpret_cast<float4*>(dp + (size_t)j * rpi * bn) = v[j];
                    } else {
                        float* cp = C != nullptr ? C + (long long)row0 * ldc + col : nullptr;
                        __nv_bfloat16* bp = Cb != nullptr ? Cb + (long long)row0 * ldcb + col : nullptr;
                        const long long cstep = (long long)rpi * ldc, bstep = (long long)rpi * ldcb;
                        if (acc_c) {                          // all C reads of the chunk in flight before the first store
                            float4 o[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                if (j < nj) o[j] = *reinterpret_cast<const float4*>(cp + j * cstep);
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                if (j < nj) { v[j].x = fmaf(alpha, v[j].x, fmaf(beta, o[j].x, bv.x)); v[j].y = fmaf(alpha, v[j].y, fmaf(beta, o[j].y, bv.y));
                                              v[j].z = fmaf(alpha, v[j].z, fmaf(beta, o[j].z, bv.z)); v[j].w = fmaf(alpha, v[j].w, fmaf(beta, o[j].w, bv.w)); }
                        } else {
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                if (j < nj) { v[j].x = fmaf(alpha, v[j].x, bv.x); v[j].y = fmaf(alpha, v[j].y, bv.y); v[j].z = fmaf(alpha, v[j].z, bv.z); v[j].w = fmaf(alpha, v[j].w, bv.w); }
                        }
                        if (cp != nullptr) {
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                if (j < nj) *reinterpret_cast<float4*>(cp + j * cstep) = v[j];
                        }
                        if (bp != nullptr) {
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                if (j < nj) *reinterpret_cast<uint2*>(bp + j * bstep) = pack_bf16x4(v[j]);
                        }
                    }
                }
                __syncwarp();                                 // staging patch is rewritten by the next chunk
            }
            if (threadIdx.x == 64) PK_STAMP(n_it, 5);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// Split-K fix-up of the persistent kernel: out = alpha * sum_s partial[s] (+ bias) (+ beta C), partials summed in
// split order.  Block = 8 rows of one tile (256 threads, row-contiguous float4 accesses): 16 blocks per tile keep
// all SMs busy even when a launch has only a handful of split tiles.
struct PkFixProb {
    const float* partials;
    float* C;
    __nv_bfloat16* Cb;
    const float* bias;
    long long ldc, ldcb;
    float alpha, beta;
    int M, N, bn, tiles_n, n_tiles, splits, blk_begin;
};
struct PkFix {
    PkFixProb p[TC_MAXP];
    int n;
};
__global__ void __launch_bounds__(256)
pk_fixup_kernel(const __grid_constant__ PkFix f) {
    pdl_trigger();
    pdl_wait();
    int pi = 0;
    for (int i = 1; i < f.n; ++i)
        if ((int)blockIdx.x >= f.p[i].blk_begin) pi = i;
    const PkFixProb& P = f.p[pi];
    const int local = (int)blockIdx.x - P.blk_begin;
    const int tile = local >> 4, rq = local & 15;
    const int bn = P.bn, lpr = bn >> 2, splits = P.splits;
    const int m0 = (tile / P.tiles_n) * TC_BM + rq * 8, n0 = (tile % P.tiles_n) * bn;
    const float* tile_part = P.partials + (size_t)tile * splits * (size_t)(TC_BM * bn) + (size_t)(rq * 8) * bn;
    const bool acc_c = P.beta != 0.f && P.C != nullptr;
    for (int idx = threadIdx.x; idx < 8 * lpr; idx += 256) {
        const int rr = idx / lpr, c4 = idx - rr * lpr;
        const int row = m0 + rr, col = n0 + 4 * c4;
        if (row >= P.M || col >= P.N) continue;
        const float* src = tile_part + (size_t)rr * bn + 4 * c4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int z0 = 0; z0 < splits; z0 += 8) {
            float4 a[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (z0 + u < splits) a[u] = __ldcg(reinterpret_cast<const float4*>(src + (size_t)(z0 + u) * (TC_BM * bn)));
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (z0 + u < splits) { v.x += a[u].x; v.y += a[u].y; v.z += a[u].z; v.w += a[u].w; }
        }
        float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (P.bias != nullptr) bv = __ldg(reinterpret_cast<const float4*>(P.bias + col));
        float4 x = make_float4(fmaf(P.alpha, v.x, bv.x), fmaf(P.alpha, v.y, bv.y), fmaf(P.alpha, v.z, bv.z), fmaf(P.alpha, v.w, bv.w));
        if (acc_c) {
            const float4 o = *reinterpret_cast<const float4*>(P.C + (long long)row * P.ldc + col);
            x.x = fmaf(P.beta, o.x, x.x); x.y = fmaf(P.beta, o.y, x.y); x.z = fmaf(P.beta, o.z, x.z); x.w = fmaf(P.beta, o.w, x.w);
        }
        if (P.C != nullptr) *reinterpret_cast<float4*>(P.C + (long long)row * P.ldc + col) = x;
        if (P.Cb != nullptr) *reinterpret_cast<uint2*>(P.Cb + (long long)row * P.ldcb + col) = pack_bf16x4(x);
    }
}

// fp32 -> bf16 (hi) and optional residual (lo = bf16(x - hi)); rows x cols with leading dims
__global__ void __launch_bounds__(256)
f32_to_bf16_kernel(const float* __restrict__ src, int64_t lds, int64_t rows, int cols,
                   __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, int64_t ldd) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;       // index over rows * cols/4
    const int c4 = cols / 4;
    if (i >= rows * c4) return;
    const int64_t r = i / c4;
    const int c = (int)(i % c4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(src + r * lds + c);
    const __nv_bfloat16 h0 = __float2bfloat16_rn(v.x), h1 = __float2bfloat16_rn(v.y), h2 = __float2bfloat16_rn(v.z), h3 = __float2bfloat16_rn(v.w);
    __nv_bfloat162 a = __halves2bfloat162(h0, h1), b = __halves2bfloat162(h2, h3);
    uint2 o;
    o.x = *reinterpret_cast<uint32_t*>(&a); o.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(hi + r * ldd + c) = o;
    if (lo != nullptr) {
        const __nv_bfloat16 l0 = __float2bfloat16_rn(v.x - __bfloat162float(h0)), l1 = __float2bfloat16_rn(v.y - __bfloat162float(h1));
        const __nv_bfloat16 l2 = __float2bfloat16_rn(v.z - __bfloat162float(h2)), l3 = __float2bfloat16_rn(v.w - __bfloat162float(h3));
        __nv_bfloat162 c0 = __halves2bfloat162(l0, l1), c1 = __halves2bfloat162(l2, l3);
        o.x = *reinterpret_cast<uint32_t*>(&c0); o.y = *reinterpret_cast<uint32_t*>(&c1);
        *reinterpret_cast<uint2*>(lo + r * ldd + c) = o;
    }
}

// ------------------------------------------------------------------ host side
static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
static std::once_flag g_encode_once;
static unsigned long long* g_dbg = nullptr;
static int g_dbg_launch = 0;      // launch slot inside the stamp buffer (32 slots x 1024 CTAs x 16 stamps)

static int get_encode() {
    std::call_once(g_encode_once, [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    });
    if (g_encode == nullptr) {
        set_error("cuTensorMapEncodeTiled not available from the driver");
        return TEAM_EUNSUPPORTED;
    }
    return TEAM_OK;
}

// 2-D bf16 tensor map over a row-major [outer, inner] matrix with leading dimension ld (elements).
static int make_map(CUtensorMap* map, const void* base, int64_t inner, int64_t outer, int64_t ld, int box_inner, int box_outer) {
    cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): base=%p inner=%lld outer=%lld ld=%lld box=%dx%d", (int)r, base,
                  (long long)inner, (long long)outer, (long long)ld, box_inner, box_outer);
        return TEAM_ECUDA;
    }
    return TEAM_OK;
}

// The device K-segments of problem g (sd[1] is left alone when g has one segment), with B's tensor map for an N tile
// of bn columns.  *ksum: the problem's K summed over its segments.
static int fill_segs(TcSegDev* sd, const TcGemm& g, int bn, double* ksum) {
    int rc;
    *ksum = 0;
    for (int q = 0; q < g.nseg; ++q) {
        const TcSeg& sg = g.s[q];
        TcSegDev& d = sd[q];
        d.K = (int)sg.K; d.a_mn = sg.a_mn ? 1 : 0; d.b_mn = sg.b_mn ? 1 : 0;
        d.nkb = (int)((sg.K + TC_BK - 1) / TC_BK);
        // K-major operand [rows,K]: inner = K, box {64, tile rows};  MN-major operand [K,rows]: inner = rows, box {64, 64}
        if (!sg.a_mn) rc = make_map(&d.ma, sg.A, sg.K, g.M, sg.lda, TC_BK, TC_BM); else rc = make_map(&d.ma, sg.A, g.M, sg.K, sg.lda, 64, TC_BK);
        if (rc) return rc;
        if (!sg.b_mn) rc = make_map(&d.mb, sg.B, sg.K, g.N, sg.ldb, TC_BK, bn); else rc = make_map(&d.mb, sg.B, g.N, sg.K, sg.ldb, 64, TC_BK);
        if (rc) return rc;
        *ksum += (double)sg.K;
    }
    return TEAM_OK;
}

// the profiler's estimate of one problem: 2 M N K flops; bf16 operands read once, fp32 / bf16 output written once
static void add_cost(double& flops, double& bytes, const TcGemm& g, double ksum) {
    const int M = (int)g.M, N = (int)g.N;
    flops += 2.0 * M * N * ksum;
    bytes += 2.0 * ((double)M + (double)N) * ksum + (g.C ? 4.0 : 0.0) * M * N + (g.Cb ? 2.0 : 0.0) * M * N;
}

// this launch's slot of the globaltimer stamp buffer (team_gemm_debug_stamps), or null
static unsigned long long* next_dbg() { return g_dbg != nullptr ? g_dbg + (size_t)(g_dbg_launch++ % 32) * 1024 * 16 : nullptr; }

// raises a kernel's dynamic shared memory limit once per device (a process may drive several GPUs); cheap enough
// to skip a lock: a racing second call only repeats it
static int set_smem_once(bool (&done)[64], const void* kernel, int bytes) {
    int dev = 0;
    TEAM_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !done[dev]) {
        TEAM_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        if (dev >= 0 && dev < 64) done[dev] = true;
    }
    return TEAM_OK;
}

// one profiler record (prof.cuh) from construction to the end of the scope
struct ProfScope {
    cudaStream_t st;
    int slot;
    ProfScope(cudaStream_t s, double flops, double bytes) : st(s), slot(prof_enabled() ? prof_begin(s, 1, flops, bytes) : -1) {}
    ~ProfScope() { if (slot >= 0) prof_end(st, slot); }
};

// launch with programmatic stream serialization and, for cluster > 1, a cluster dimension; counts the launch
template <typename Group>
static int tc_launch(cudaStream_t st, void (*kernel)(Group), const Group& g, const char* name, int grid, int threads,
                     int smem, int cluster) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3((unsigned)threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (cluster > 1) {
        at[na].id = cudaLaunchAttributeClusterDimension;
        at[na].val.clusterDim.x = (unsigned)cluster; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
        ++na;
    }
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
    cfg.attrs = at;
    cfg.numAttrs = na;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, g);
    count_launch();
    if (e != cudaSuccess) return cuda_fail(e, name);
    return TEAM_OK;
}

// ---- persistent path: planning + launch of one group (<= TC_MAXP problems).  ws holds the split-K partials.
static bool pk_eligible(const TcGemm& g) {
    if (g.N % 4 != 0) return false;
    if (g.C != nullptr && (g.ldc % 4 != 0 || (reinterpret_cast<uintptr_t>(g.C) & 15) != 0)) return false;
    if (g.Cb != nullptr && (g.ldcb % 4 != 0 || (reinterpret_cast<uintptr_t>(g.Cb) & 7) != 0)) return false;
    if (g.bias != nullptr && (reinterpret_cast<uintptr_t>(g.bias) & 15) != 0) return false;
    return true;
}

static int pk_launch_group(cudaStream_t st, const TcGemm* const* sel, int np, void* ws, size_t ws_bytes) {
    static bool smem_set[64] = {};
    int rc = set_smem_once(smem_set, (const void*)gemm_bf16_persistent_kernel, PK_SMEM_BYTES);
    if (rc) return rc;
    const bool have_ws = ws != nullptr && ws_bytes > 4096 && (reinterpret_cast<uintptr_t>(ws) & 15) == 0;
    char* part_base = have_ws ? reinterpret_cast<char*>(ws) : nullptr;
    size_t part_cap = have_ws ? ws_bytes : 0, part_off = 0;
    int order[TC_MAXP], bn_[TC_MAXP], tiles_n_[TC_MAXP], tiles_[TC_MAXP], splits_[TC_MAXP], kbps_[TC_MAXP];
    float* partials[TC_MAXP];
    bool any_split = false;
    for (int i = 0; i < np; ++i) {
        const TcGemm& g = *sel[i];
        bool any_b_mn = false;
        int nkb = 0;
        for (int q = 0; q < g.nseg; ++q) { any_b_mn = any_b_mn || g.s[q].b_mn; nkb += (int)((g.s[q].K + TC_BK - 1) / TC_BK); }
        int bn;
        if (g.N >= PK_BN_MAX) bn = PK_BN_MAX;
        else bn = any_b_mn ? (int)((g.N + 63) / 64 * 64) : (int)((g.N + 15) / 16 * 16);
        const int tiles_n = (int)((g.N + bn - 1) / bn), tiles = (int)((g.M + TC_BM - 1) / TC_BM) * tiles_n;
        int splits = 1;
        if (have_ws && tiles < NUM_SMS / 2 && nkb >= 64) {
            // a partial tile costs 2 x 128 x bn x 4 bytes of extra traffic: keep >= 32 k-blocks (1.5 MB of operands) per item
            splits = (NUM_SMS + tiles - 1) / tiles;
            if (splits > nkb / 32) splits = nkb / 32;
            if (splits > 32) splits = 32;
            while (splits > 1 && part_off + (size_t)tiles * splits * TC_BM * bn * 4 > part_cap) splits /= 2;
            if (splits < 1) splits = 1;
        }
        int kbps = (nkb + splits - 1) / splits;
        splits = (nkb + kbps - 1) / kbps;                 // every split owns at least one k-block
        bn_[i] = bn; tiles_n_[i] = tiles_n; tiles_[i] = tiles; splits_[i] = splits; kbps_[i] = kbps;
        order[i] = i;
        partials[i] = nullptr;
        if (splits > 1) {
            any_split = true;
            partials[i] = reinterpret_cast<float*>(part_base + part_off);
            part_off += align_up((size_t)tiles * splits * TC_BM * bn * 4, 256);
        }
    }
    // longest items first: the static round-robin over CTAs then balances to within one short item
    for (int a = 0; a < np; ++a)
        for (int b = a + 1; b < np; ++b)
            if (kbps_[order[b]] > kbps_[order[a]]) { const int t = order[a]; order[a] = order[b]; order[b] = t; }
    PkGroup out;
    memset(&out, 0, sizeof(out));
    int item = 0;
    double flops = 0, bytes = 0;
    for (int o = 0; o < np; ++o) {
        const int i = order[o];
        const TcGemm& g = *sel[i];
        PkProb& p = out.p[o];
        p.partials = partials[i];
        p.C = g.C; p.ldc = g.ldc; p.Cb = reinterpret_cast<__nv_bfloat16*>(g.Cb); p.ldcb = g.ldcb; p.bias = g.bias;
        p.alpha = g.alpha; p.beta = g.beta; p.M = (int)g.M; p.N = (int)g.N;
        p.bn = bn_[i]; p.tiles_n = tiles_n_[i]; p.n_tiles = tiles_[i]; p.splits = splits_[i]; p.kb_per_split = kbps_[i];
        p.item_begin = item;
        item += tiles_[i] * splits_[i];
        double ksum;
        if ((rc = fill_segs(p.s, g, p.bn, &ksum))) return rc;
        if (g.nseg == 1) { p.s[1] = p.s[0]; p.s[1].nkb = 0; p.s[1].K = 0; }   // valid (unused) maps
        add_cost(flops, bytes, g, ksum);
    }
    out.n = np;
    out.total_items = item;
    out.dbg = next_dbg();
    ProfScope prof(st, flops, bytes);    // the fix-up kernel is part of the timed GEMM
    if ((rc = tc_launch(st, gemm_bf16_persistent_kernel, out, "gemm_bf16_persistent_kernel", item < NUM_SMS ? item : NUM_SMS,
                        PK_THREADS, PK_SMEM_BYTES, 1)))
        return rc;
    if (any_split) {
        PkFix fx;
        memset(&fx, 0, sizeof(fx));
        int blocks = 0;
        for (int o = 0; o < np; ++o) {
            const PkProb& p = out.p[o];
            if (p.splits <= 1) continue;
            PkFixProb& q = fx.p[fx.n++];
            q.partials = p.partials; q.C = p.C; q.Cb = p.Cb; q.bias = p.bias; q.ldc = p.ldc; q.ldcb = p.ldcb;
            q.alpha = p.alpha; q.beta = p.beta; q.M = p.M; q.N = p.N; q.bn = p.bn; q.tiles_n = p.tiles_n;
            q.n_tiles = p.n_tiles; q.splits = p.splits; q.blk_begin = blocks;
            blocks += 16 * p.n_tiles;
        }
        TEAM_LAUNCH(pk_fixup_kernel, blocks, 256, 0, st, fx);
    }
    return TEAM_OK;
}

// co-resident CTA budget of a launch whose cluster size is `cluster`
static int tc_target_ctas(int cluster) {
    static constexpr int cap[4] = {TC_TARGET_CTAS, TC_TARGET_CTAS, 272, 240};      // measured at B = 1024: -2 % step time
    return cap[cluster >= 8 ? 3 : cluster >= 4 ? 2 : cluster >= 2 ? 1 : 0];
}

// Plans tiles / splits for ops[0..n) and launches them in chunks of TC_MAXP problems.
//   * N tile: 128 wide unless the whole launch would leave most SMs without a tile, then 64;
//   * split-K: while the launch stays within two CTAs per SM, the problem with the most k-blocks per CTA is
//     split further (2 / 4 / 8 ways), so that a [512,512] weight gradient over K = 2B rows does not run as 16 long CTAs
//     next to hundreds of short ones.  The largest split count is the cluster size of the launch.
int gemm_bf16_group(cudaStream_t st, const TcGemm* ops, int n, void* ws, size_t ws_bytes) {
    static bool smem_set[64] = {};
    int rc = get_encode();
    if (rc) return rc;
    for (int base = 0; base < n; base += TC_MAXP) {
        const int cnt = n - base < TC_MAXP ? n - base : TC_MAXP;
        TcGroup grp;
        memset(&grp, 0, sizeof(grp));
        const TcGemm* sel[TC_MAXP];
        int np = 0, tiles128 = 0;
        for (int i = 0; i < cnt; ++i) {
            const TcGemm& g = ops[base + i];
            if (g.M <= 0 || g.N <= 0) continue;
            TEAM_REQUIRE(g.nseg == 1 || g.nseg == 2, "gemm_bf16: nseg %d", g.nseg);
            TEAM_REQUIRE(g.C != nullptr || g.Cb != nullptr, "gemm_bf16: no output");
            for (int q = 0; q < g.nseg; ++q) {
                const TcSeg& sg = g.s[q];
                TEAM_REQUIRE(sg.K > 0 && sg.lda % 8 == 0 && sg.ldb % 8 == 0, "gemm_bf16: K=%lld lda=%lld ldb=%lld (leading dims must be multiples of 8)", (long long)sg.K, (long long)sg.lda, (long long)sg.ldb);
                TEAM_REQUIRE((reinterpret_cast<uintptr_t>(sg.A) & 15) == 0 && (reinterpret_cast<uintptr_t>(sg.B) & 15) == 0, "gemm_bf16: operands must be 16-byte aligned");
            }
            sel[np++] = &g;
            tiles128 += (int)((g.M + TC_BM - 1) / TC_BM) * (int)((g.N + TC_MAX_BN - 1) / TC_MAX_BN);
        }
        if (np == 0) continue;
        {   // large launches: persistent kernel (128 x 256 tiles, overlapped epilogue)
            bool ok = tiles128 >= 2 * NUM_SMS;
            for (int i = 0; i < np && ok; ++i) ok = pk_eligible(*sel[i]);
            if (ok) {
                if ((rc = pk_launch_group(st, sel, np, ws, ws_bytes))) return rc;
                continue;
            }
        }
        const bool narrow = tiles128 < NUM_SMS;
        int tiles[TC_MAXP], nkbs[TC_MAXP];
        double ksums[TC_MAXP];
        for (int i = 0; i < np; ++i) {
            const TcGemm& g = *sel[i];
            bool any_b_mn = false;
            for (int q = 0; q < g.nseg; ++q) any_b_mn = any_b_mn || g.s[q].b_mn;
            TcProb& p = grp.p[i];
            const int tiles_m = (int)((g.M + TC_BM - 1) / TC_BM);
            const int nt128 = (int)((g.N + TC_MAX_BN - 1) / TC_MAX_BN);
            int bn;
            if (any_b_mn) {
                bn = (g.N > 64 && !narrow) ? 128 : 64;
            } else {
                const int nt = (narrow && g.N > 64) ? (int)((g.N + 63) / 64) : nt128;
                bn = (int)(((g.N + nt - 1) / nt + 15) / 16 * 16);
            }
            p.bn = bn;
            p.tiles_n = (int)((g.N + bn - 1) / bn);
            p.M = (int)g.M; p.N = (int)g.N;
            p.alpha = g.alpha; p.beta = g.beta;
            p.C = g.C; p.ldc = g.ldc; p.Cb = reinterpret_cast<__nv_bfloat16*>(g.Cb); p.ldcb = g.ldcb; p.bias = g.bias;
            if ((rc = fill_segs(p.s, g, bn, &ksums[i]))) return rc;
            nkbs[i] = p.s[0].nkb + p.s[1].nkb;
            tiles[i] = tiles_m * p.tiles_n;
            p.n_tiles = tiles[i];
            p.splits = 1;
        }
        // split-K by doubling: always the problem with the most k-blocks per CTA, while two CTAs per SM can hold the launch
        int total = 0;
        for (int i = 0; i < np; ++i) total += tiles[i];
        for (;;) {
            int best = -1, best_kb = 10;
            for (int i = 0; i < np; ++i) {
                const int s = grp.p[i].splits;
                const int per = (nkbs[i] + s - 1) / s;
                const int per2 = (nkbs[i] + 2 * s - 1) / (2 * s);
                const bool valid = 2 * s <= TC_MAX_SPLITS && (2 * s - 1) * per2 < nkbs[i];     // every split keeps >= 1 k-block
                // the launch's cluster size is its largest split: clusters are placed GPC by GPC, so a launch of
                // 8-CTA clusters holds fewer co-resident CTAs than 2 per SM (a late second wave of clusters costs ~10 us)
                int cl = 2 * s;
                for (int q = 0; q < np; ++q) cl = grp.p[q].splits > cl ? grp.p[q].splits : cl;
                if (per > best_kb && valid && total + tiles[i] * s <= tc_target_ctas(cl)) { best = i; best_kb = per; }
            }
            if (best < 0) break;
            total += tiles[best] * grp.p[best].splits;
            grp.p[best].splits *= 2;
        }
        int cluster = 1;
        for (int i = 0; i < np; ++i) cluster = grp.p[i].splits > cluster ? grp.p[i].splits : cluster;
        int cta = 0;
        double flops = 0, bytes = 0;
        for (int i = 0; i < np; ++i) {
            TcProb& p = grp.p[i];
            p.kb_per_split = (nkbs[i] + p.splits - 1) / p.splits;
            p.cta_begin = cta;
            cta += (tiles[i] * p.splits + cluster - 1) / cluster * cluster;        // whole clusters per problem
            add_cost(flops, bytes, *sel[i], ksums[i]);
        }
        grp.n = np;
        grp.cluster = cluster;
        grp.stages = cta <= NUM_SMS ? TC_MAX_STAGES : TC_STAGES;
        grp.dbg = next_dbg();
        if ((rc = set_smem_once(smem_set, (const void*)gemm_bf16_tcgen05_kernel, tc_smem_bytes(TC_MAX_STAGES)))) return rc;
        ProfScope prof(st, flops, bytes);
        if ((rc = tc_launch(st, gemm_bf16_tcgen05_kernel, grp, "gemm_bf16_tcgen05_kernel", cta, TC_THREADS, tc_smem_bytes(grp.stages),
                            grp.cluster)))
            return rc;
    }
    return TEAM_OK;
}

int to_bf16(cudaStream_t st, const float* src, int64_t lds, int64_t rows, int cols, void* hi, void* lo, int64_t ldd) {
    TEAM_REQUIRE(cols % 4 == 0 && lds % 4 == 0 && ldd % 4 == 0, "to_bf16: cols/ld must be multiples of 4");
    const int64_t n = rows * (cols / 4);
    if (n == 0) return TEAM_OK;
    f32_to_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, lds, rows, cols, reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo), ldd);
    TEAM_LAUNCH_CHECK("f32_to_bf16_kernel");
    return TEAM_OK;
}

int run_wave(cudaStream_t st, int mode, Wave& wv, void* ws, size_t ws_bytes) {
    if (wv.n == 0) return TEAM_OK;
    int rc;
    if (mode == TEAM_MODE_BF16) {
        TcGemm t[TC_MAXP];
        int nt = 0;
        for (int i = 0; i < wv.n; ++i) {
            const GOp& o = wv.op[i];
            if (o.M <= 0 || o.N <= 0) continue;
            TcGemm& g = t[nt++];
            memset(&g, 0, sizeof(g));
            g.M = o.M; g.N = o.N; g.nseg = o.nseg; g.alpha = o.alpha; g.beta = o.beta;
            for (int q = 0; q < o.nseg; ++q) {
                TEAM_REQUIRE(o.s[q].A.h != nullptr && o.s[q].B.h != nullptr, "gemm: operand without bf16 shadow (wave op %d)", i);
                g.s[q].a_mn = o.s[q].a_mn; g.s[q].b_mn = o.s[q].b_mn; g.s[q].K = o.s[q].K;
                g.s[q].A = o.s[q].A.h; g.s[q].lda = o.s[q].A.ld; g.s[q].B = o.s[q].B.h; g.s[q].ldb = o.s[q].B.ld;
            }
            g.C = o.C.f; g.ldc = o.C.ld; g.Cb = o.C.h; g.ldcb = o.C.ld; g.bias = o.bias;
        }
        rc = gemm_bf16_group(st, t, nt, ws, ws_bytes);
        wv.n = 0;
        return rc;
    }
    // F32 mode: segment 0 applies beta and bias, later segments accumulate
    for (int i = 0; i < wv.n; ++i) {
        const GOp& o = wv.op[i];
        if (o.M <= 0 || o.N <= 0) continue;
        for (int q = 0; q < o.nseg; ++q) {
            const GSeg& g = o.s[q];
            rc = gemm_f32(st, g.a_mn, !g.b_mn, o.M, o.N, g.K, o.alpha, g.A.f, g.A.ld, g.B.f, g.B.ld, q == 0 ? o.beta : 1.f,
                          o.C.f, o.C.ld, q == 0 ? o.bias : nullptr, ws, ws_bytes);
            if (rc) return rc;
        }
    }
    wv.n = 0;
    return TEAM_OK;
}

}  // namespace team

using namespace team;

extern "C" int team_gemm_bf16(int a_mn, int b_mn, int64_t M, int64_t N, int64_t K, float alpha, const void* A,
                              const void* A_lo, int64_t lda, const void* B, int64_t ldb, float beta, float* C,
                              int64_t ldc, const float* bias, void* workspace, size_t workspace_bytes, void* stream) {
    TcGemm g;
    memset(&g, 0, sizeof(g));
    g.M = M; g.N = N; g.nseg = 1; g.alpha = alpha; g.beta = beta;
    g.s[0].a_mn = a_mn != 0; g.s[0].b_mn = b_mn != 0; g.s[0].K = K;
    g.s[0].A = A; g.s[0].lda = lda; g.s[0].B = B; g.s[0].ldb = ldb; g.C = C; g.ldc = ldc; g.bias = bias;
    const cudaStream_t st = (cudaStream_t)stream;
    int rc = gemm_bf16_group(st, &g, 1, workspace, workspace_bytes);
    if (rc || A_lo == nullptr) return rc;
    // two-term split of A: C = alpha (A_hi + A_lo) B + ... as two passes, the second accumulating into the fp32 output
    TEAM_REQUIRE(C != nullptr, "gemm_bf16: the two-term A split needs an fp32 output");
    g.s[0].A = A_lo; g.beta = 1.f; g.bias = nullptr;
    return gemm_bf16_group(st, &g, 1, workspace, workspace_bytes);
}

extern "C" int team_gemm_bf16_group(const team_gemm_desc* descs, int32_t n, void* workspace, size_t workspace_bytes,
                                    void* stream) {
    TEAM_REQUIRE(descs != nullptr && n >= 1 && n <= 64, "team_gemm_bf16_group: bad args");
    TcGemm ops[64];
    for (int i = 0; i < n; ++i) {
        const team_gemm_desc& d = descs[i];
        TcGemm& g = ops[i];
        memset(&g, 0, sizeof(g));
        g.M = d.M; g.N = d.N; g.alpha = d.alpha; g.beta = d.beta;
        g.nseg = d.K2 > 0 ? 2 : 1;
        g.s[0].a_mn = d.a_mn != 0; g.s[0].b_mn = d.b_mn != 0; g.s[0].K = d.K;
        g.s[0].A = d.A; g.s[0].lda = d.lda; g.s[0].B = d.B; g.s[0].ldb = d.ldb;
        g.s[1].a_mn = d.a_mn2 != 0; g.s[1].b_mn = d.b_mn2 != 0; g.s[1].K = d.K2;
        g.s[1].A = d.A2; g.s[1].lda = d.lda2; g.s[1].B = d.B2; g.s[1].ldb = d.ldb2;
        g.C = d.C; g.ldc = d.ldc; g.Cb = d.C_bf16; g.ldcb = d.ldc_bf16;
        g.bias = d.bias;
    }
    return gemm_bf16_group((cudaStream_t)stream, ops, n, workspace, workspace_bytes);
}

extern "C" int team_f32_to_bf16(const float* src, int64_t lds, int64_t rows, int64_t cols, void* hi, void* lo,
                                int64_t ldd, void* stream) {
    return to_bf16((cudaStream_t)stream, src, lds, rows, (int)cols, hi, lo, ldd);
}

extern "C" int team_gemm_debug_stamps(void* buf) {
    g_dbg = reinterpret_cast<unsigned long long*>(buf);
    g_dbg_launch = 0;
    return TEAM_OK;
}
