// In-place fp32 all-reduce (sum) of one buffer per GPU over NVLink peer memory - the gradient exchange of the
// data-parallel head step (SURVEY 8e: 1.85 M floats, far too small for a ring to reach wire speed).
//
// Every rank maps every peer's buffer and flag array (symmetric memory; the host hands in the W pointers).  ONE
// kernel per rank, two-shot:
//   barrier A  (per block: "my gradients are complete" flags written into every peer, wait for all peers)
//   reduce     rank r sums slice r of all W buffers in rank order 0..W-1 (=> bit-identical on every rank)
//   broadcast  and stores the result into slice r of every peer's buffer (and its own)
//              [with a multicast mapping: multimem.ld_reduce / multimem.st - the NVSwitch adds and replicates]
//   barrier B  (per block: "my slice is written everywhere")
// Flags carry a monotonically increasing epoch kept in the rank's own flag array, so nothing is ever reset and the
// launch can sit inside a replayed CUDA graph.  Block b of every rank works on the same float4 indices, so the
// barriers are per block (no grid-wide sync); the grid is small enough to be co-resident.
// The all-gather of the data-parallel losses (team_peer_allgather, below) uses the same barriers and flag layout.
#include <stdlib.h>
#include "common.cuh"

namespace team {

constexpr int AR_MAX_RANKS = 8;
constexpr int AR_BLOCKS = 64;
constexpr int AR_THREADS = 512;
// flag array layout (uint32): [0, AR_BLOCKS) own epoch per block | A flags [AR_BLOCKS][8] | B flags [AR_BLOCKS][8]
constexpr int AR_FLAG_WORDS = AR_BLOCKS + 2 * AR_BLOCKS * AR_MAX_RANKS;
// after the two channels: AR_STATUS_WORDS status words of the rank itself.  word 0: 0 = healthy, else
// 1 + (phase << 8) + (peer << 16) of the first wait that ran past its deadline (team_peer_allreduce_status)
constexpr int AR_STATUS_WORDS = 16;

struct ArArgs {
    float* buf[AR_MAX_RANKS];
    uint32_t* flag[AR_MAX_RANKS];
    float* mc;                 // multicast (NVLS) mapping of the same buffer on all ranks, or null
    int rank, world;
    long long n4;              // float4 count
    uint32_t* status;          // this rank's status words (after both flag channels)
    unsigned long long timeout_ns;   // 0: wait for ever
};
__device__ __forceinline__ unsigned long long ar_gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_volatile_f4(const float4* p) {
    float4 v;
    asm volatile("ld.volatile.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_volatile_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// All threads of the block call it; threads [0, world) of warp 0 each handle one peer.
//   START barrier (release_writes = false): what the peers are about to read was written by EARLIER kernels of
//   this rank (complete and at its home L2 when this kernel runs), so a plain volatile flag store suffices; the
//   poll is an ACQUIRE load (ld.acquire.sys - a strong load, not a MEMBAR.SYS), which orders the peer-data loads /
//   multimem.ld_reduce that follow behind the flag it observed, inside the PTX memory model.
//   END barrier (release_writes = true): this block's stores into the peers' buffers must be performed before the
//   flag - one system-scope release per polling thread (the CTA barrier in front makes the whole block's writes
//   part of it).  The readers of the result are LATER kernels (kernel boundary).
// MEMBAR.SYS, not the NVLink round trip, is the expensive part of such a barrier: 1 instead of 4 per call.
// A peer that does not show up (rank skew: evaluation / checkpointing on one rank, a stalled loader, lazy init) is
// waited for until a %globaltimer deadline (TEAM_PEER_TIMEOUT_S, default 1800 s, 0 = for ever); past it the wait
// gives up, records who / where in the rank's status word and the kernel finishes WITHOUT trapping - the CUDA
// context stays usable and the host reads the status (team_peer_allreduce_status) instead of a sticky error.
__device__ __forceinline__ void ar_barrier(const ArArgs& a, int phase, uint32_t epoch, bool release_writes) {
    __syncthreads();
    const int t = threadIdx.x;
    if (t < a.world) {
        const int slot = AR_BLOCKS + (phase * AR_BLOCKS + (int)blockIdx.x) * AR_MAX_RANKS;
        if (release_writes) st_release_sys(a.flag[t] + slot + a.rank, epoch);      // tell peer t
        else st_volatile_u32(a.flag[t] + slot + a.rank, epoch);
        const uint32_t* mine = a.flag[a.rank] + slot + t;                          // hear from peer t
        unsigned long long deadline = 0;
        uint32_t spins = 0;
        while ((int)(ld_acquire_sys(mine) - epoch) < 0) {
            if ((++spins & 1023u) == 0u && a.timeout_ns != 0ull) {
                const unsigned long long now = ar_gtime();
                if (deadline == 0) deadline = now + a.timeout_ns;
                else if (now > deadline) {
                    atomicCAS(a.status, 0u, 1u + ((uint32_t)phase << 8) + ((uint32_t)t << 16));
                    break;
                }
            }
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(AR_THREADS)
peer_allreduce_f32_kernel(const __grid_constant__ ArArgs a) {
    pdl_trigger();
    pdl_wait();
    __shared__ uint32_t s_epoch;
    if (threadIdx.x == 0) {
        uint32_t* e = a.flag[a.rank] + blockIdx.x;
        s_epoch = *e + 1;
        *e = s_epoch;
    }
    __syncthreads();
    const uint32_t epoch = s_epoch;
    ar_barrier(a, 0, epoch, false);
    const int W = a.world;
    const long long c0 = a.n4 * a.rank / W, c1 = a.n4 * (a.rank + 1) / W;
    if (a.mc != nullptr) {
        // NVLS: the switch sums the W copies on the way in (multimem.ld_reduce) and replicates the result on the way
        // out (multimem.st), so each rank moves 2/W of the buffer over its own links instead of 2 (W-1)/W
        float4* mc = reinterpret_cast<float4*>(a.mc);
        constexpr int U = 4;                                   // independent round trips in flight per thread
        const long long stride = (long long)gridDim.x * AR_THREADS;
        for (long long i0 = c0 + (long long)blockIdx.x * AR_THREADS + threadIdx.x; i0 < c1; i0 += U * stride) {
            float4 s[U];
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (i0 + u * stride < c1)
                    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                                 : "=f"(s[u].x), "=f"(s[u].y), "=f"(s[u].z), "=f"(s[u].w) : "l"(mc + i0 + u * stride) : "memory");
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (i0 + u * stride < c1)
                    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
                                 ::"l"(mc + i0 + u * stride), "f"(s[u].x), "f"(s[u].y), "f"(s[u].z), "f"(s[u].w) : "memory");
        }
    } else
    for (long long i = c0 + (long long)blockIdx.x * AR_THREADS + threadIdx.x; i < c1; i += (long long)gridDim.x * AR_THREADS) {
        float4 v[AR_MAX_RANKS];
#pragma unroll
        for (int r = 0; r < AR_MAX_RANKS; ++r)
            if (r < W) v[r] = ld_volatile_f4(reinterpret_cast<const float4*>(a.buf[r]) + i);
        float4 s = v[0];
#pragma unroll
        for (int r = 1; r < AR_MAX_RANKS; ++r)
            if (r < W) { s.x += v[r].x; s.y += v[r].y; s.z += v[r].z; s.w += v[r].w; }
#pragma unroll
        for (int r = 0; r < AR_MAX_RANKS; ++r)
            if (r < W) reinterpret_cast<float4*>(a.buf[r])[i] = s;
    }
    ar_barrier(a, 1, epoch, true);
}

// All-gather of one slice per rank (the exchanges between the phases of team_loss_shard_run): buf[r] is rank r's
// gathered buffer, world slices of n4 16-byte units in rank order, and this rank's slice is already in slot `rank` of
// its own buffer (the loss phase wrote it there).  No arithmetic, so every rank ends with the same bytes.
//   barrier A  "my slice is written and I no longer read my gathered buffer": earlier kernels of this rank did both
//              (complete when this kernel runs), so the peers may now overwrite the other slots.  This makes reusing
//              the buffers from step to step safe whatever runs between two calls.
//   store      the slice into slot `rank` of every peer's buffer [with a multicast mapping: ONE multimem.st of the
//              slice, which the switch replicates into every rank's buffer]
//   barrier B  (release) "my slice is in your buffer"; the readers are later kernels
__global__ void __launch_bounds__(AR_THREADS)
peer_allgather_kernel(const __grid_constant__ ArArgs a) {
    pdl_trigger();
    pdl_wait();
    __shared__ uint32_t s_epoch;
    if (threadIdx.x == 0) {
        uint32_t* e = a.flag[a.rank] + blockIdx.x;
        s_epoch = *e + 1;
        *e = s_epoch;
    }
    __syncthreads();
    const uint32_t epoch = s_epoch;
    ar_barrier(a, 0, epoch, false);
    const int W = a.world, me = a.rank;
    const long long n4 = a.n4, slot = n4 * me;
    const float4* src = reinterpret_cast<const float4*>(a.buf[me]) + slot;
    const long long stride = (long long)gridDim.x * AR_THREADS;
    if (a.mc != nullptr) {
        float4* mc = reinterpret_cast<float4*>(a.mc) + slot;
        for (long long i = (long long)blockIdx.x * AR_THREADS + threadIdx.x; i < n4; i += stride) {
            const float4 v = src[i];
            asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
                         ::"l"(mc + i), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
        }
    } else
    for (long long i = (long long)blockIdx.x * AR_THREADS + threadIdx.x; i < n4; i += stride) {
        const float4 v = src[i];
#pragma unroll
        for (int r = 0; r < AR_MAX_RANKS; ++r)
            if (r < W && r != me) (reinterpret_cast<float4*>(a.buf[r]) + slot)[i] = v;
    }
    ar_barrier(a, 1, epoch, true);
}

// Blocks per call: about two float4 per thread of a rank's slice, between 8 and AR_BLOCKS.  A small bucket that is
// exchanged UNDER compute kernels should not park 64 spinning blocks on the SMs those kernels need; every rank
// derives the same grid from the same n, and each block keeps its own epoch, so grids may differ between calls.
static unsigned long long ar_timeout_ns() {
    static long long v = -1;
    if (v < 0) {
        const char* e = getenv("TEAM_PEER_TIMEOUT_S");
        double sec = e != nullptr ? atof(e) : 1800.0;
        if (sec < 0) sec = 0;
        v = (long long)(sec * 1e9);
    }
    return (unsigned long long)v;
}
static int ar_grid(int64_t n4, int world) {
    const int64_t per_rank = (n4 + world - 1) / world;
    int64_t g = (per_rank + 2 * AR_THREADS - 1) / (2 * AR_THREADS);
    if (g < 8) g = 8;
    if (g > AR_BLOCKS) g = AR_BLOCKS;
    return (int)g;
}

// all-reduce of floats [offset, offset + n) of the buffers described by `c` (both multiples of 4)
int peer_allreduce_range(cudaStream_t st, const team_peer_comm* c, int64_t offset, int64_t n, int channel) {
    TEAM_REQUIRE(channel == 0 || channel == 1, "peer_allreduce: channel %d", channel);
    TEAM_REQUIRE(c != nullptr && c->world >= 1 && c->world <= AR_MAX_RANKS && c->rank >= 0 && c->rank < c->world, "peer_allreduce: bad comm");
    TEAM_REQUIRE(offset >= 0 && n >= 0 && offset % 4 == 0 && n % 4 == 0 && offset + n <= c->n_total, "peer_allreduce: range [%lld, +%lld) of %lld", (long long)offset, (long long)n, (long long)c->n_total);
    if (n == 0 || c->world == 1) return TEAM_OK;
    ArArgs a;
    memset(&a, 0, sizeof(a));
    for (int r = 0; r < c->world; ++r) {
        TEAM_REQUIRE(c->bufs[r] != nullptr && c->flags[r] != nullptr && (reinterpret_cast<uintptr_t>(c->bufs[r]) & 15) == 0, "peer_allreduce: bad pointer of rank %d", r);
        a.buf[r] = reinterpret_cast<float*>(c->bufs[r]) + offset;
        a.flag[r] = reinterpret_cast<uint32_t*>(c->flags[r]) + (size_t)channel * AR_FLAG_WORDS;
    }
    a.mc = c->multicast != nullptr ? reinterpret_cast<float*>(c->multicast) + offset : nullptr;
    a.rank = c->rank; a.world = c->world; a.n4 = n / 4;
    a.status = reinterpret_cast<uint32_t*>(c->flags[c->rank]) + (size_t)2 * AR_FLAG_WORDS;
    a.timeout_ns = ar_timeout_ns();
    TEAM_LAUNCH(peer_allreduce_f32_kernel, ar_grid(a.n4, a.world), AR_THREADS, 0, st, a);
    return TEAM_OK;
}

}  // namespace team

using namespace team;

// two independent flag channels: two exchanges may be in flight at once (team_head_grads.comm: the late bucket starts
// while the q/k/v bucket is still finishing)
extern "C" size_t team_peer_allreduce_flag_bytes(void) { return ((size_t)2 * AR_FLAG_WORDS + AR_STATUS_WORDS) * sizeof(uint32_t); }

// Health of the exchanges issued so far on this rank: synchronises `stream`, then reads the rank's status word.
// 0 = every wait completed; otherwise 1 + (phase << 8) + (peer << 16) of the first wait that ran past the deadline
// (the data of that exchange is then NOT the sum over the ranks).  `own_flags` = flags[rank] of the calls.
extern "C" int team_peer_allreduce_status(const void* own_flags, void* stream, uint32_t* status) {
    TEAM_REQUIRE(own_flags != nullptr && status != nullptr, "peer_allreduce_status: null pointer");
    TEAM_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    TEAM_CUDA_CHECK(cudaMemcpy(status, reinterpret_cast<const uint32_t*>(own_flags) + (size_t)2 * AR_FLAG_WORDS, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return TEAM_OK;
}

extern "C" int team_peer_allreduce_f32(void* const* bufs, void* const* flags, void* multicast, int32_t rank,
                                       int32_t world, int64_t n, void* stream) {
    TEAM_REQUIRE(bufs != nullptr && flags != nullptr, "peer_allreduce: null pointer table");
    TEAM_REQUIRE(world >= 1 && world <= AR_MAX_RANKS && rank >= 0 && rank < world, "peer_allreduce: rank %d / world %d", rank, world);
    TEAM_REQUIRE(n >= 0 && n % 4 == 0, "peer_allreduce: element count %lld must be a multiple of 4", (long long)n);
    if (n == 0 || world == 1) return TEAM_OK;
    ArArgs a;
    memset(&a, 0, sizeof(a));
    for (int r = 0; r < world; ++r) {
        TEAM_REQUIRE(bufs[r] != nullptr && flags[r] != nullptr && (reinterpret_cast<uintptr_t>(bufs[r]) & 15) == 0, "peer_allreduce: bad pointer of rank %d", r);
        a.buf[r] = reinterpret_cast<float*>(bufs[r]);
        a.flag[r] = reinterpret_cast<uint32_t*>(flags[r]);
    }
    a.mc = reinterpret_cast<float*>(multicast);
    a.rank = rank; a.world = world; a.n4 = n / 4;
    a.status = reinterpret_cast<uint32_t*>(flags[rank]) + (size_t)2 * AR_FLAG_WORDS;
    a.timeout_ns = ar_timeout_ns();
    TEAM_LAUNCH(peer_allreduce_f32_kernel, ar_grid(a.n4, a.world), AR_THREADS, 0, (cudaStream_t)stream, a);
    return TEAM_OK;
}

extern "C" int team_peer_allgather(void* const* bufs, void* const* flags, void* multicast, int32_t rank, int32_t world,
                                   int64_t slice_bytes, void* stream) {
    TEAM_REQUIRE(bufs != nullptr && flags != nullptr, "peer_allgather: null pointer table");
    TEAM_REQUIRE(world >= 1 && world <= AR_MAX_RANKS && rank >= 0 && rank < world, "peer_allgather: rank %d / world %d", rank, world);
    TEAM_REQUIRE(slice_bytes >= 0 && slice_bytes % 16 == 0, "peer_allgather: slice of %lld bytes must be a multiple of 16", (long long)slice_bytes);
    if (slice_bytes == 0 || world == 1) return TEAM_OK;
    ArArgs a;
    memset(&a, 0, sizeof(a));
    for (int r = 0; r < world; ++r) {
        TEAM_REQUIRE(bufs[r] != nullptr && flags[r] != nullptr && (reinterpret_cast<uintptr_t>(bufs[r]) & 15) == 0, "peer_allgather: bad pointer of rank %d", r);
        a.buf[r] = reinterpret_cast<float*>(bufs[r]);
        a.flag[r] = reinterpret_cast<uint32_t*>(flags[r]);
    }
    TEAM_REQUIRE((reinterpret_cast<uintptr_t>(multicast) & 15) == 0, "peer_allgather: misaligned multicast mapping");
    a.mc = reinterpret_cast<float*>(multicast);
    a.rank = rank; a.world = world; a.n4 = slice_bytes / 16;
    a.status = reinterpret_cast<uint32_t*>(flags[rank]) + (size_t)2 * AR_FLAG_WORDS;
    a.timeout_ns = ar_timeout_ns();
    // the grid is sized by the slice each rank sends (every rank derives the same one from the same slice_bytes)
    TEAM_LAUNCH(peer_allgather_kernel, ar_grid(a.n4, 1), AR_THREADS, 0, (cudaStream_t)stream, a);
    return TEAM_OK;
}
