// K9/K17 - deterministic, atomic-free keyed segmented sum over [N,512] feature rows.
//
// Replaces the Python class/state loops of models/proof.py:258-276 (cal_prototype),
// models/simplecil.py:48-55 (replace_fc) and utils/state_distance.py:98-103.
//
// HBM-bound: every feature row (2 KB fp32 / 1 KB bf16) is read exactly once with 128-bit
// (64-bit for bf16) streaming loads; algorithmic bytes = 512*e + 8 (label) [+ 8 (state)]
// per row (SURVEY 8d).  Layout of the reduction:
//   pass 1  grid = (8*n_clusters, n_slabs), 128 threads.  A CTA streams a contiguous chunk
//           of rows.  Thread t owns columns [4t,4t+4) of every key accumulator in shared
//           memory, so the per-key sums are built in row order with no atomics and no
//           inter-thread races -> bit-reproducible.  8 rows are in flight per thread.
//           The 8 CTAs of a thread-block cluster then fold their accumulators through
//           distributed shared memory in rank order (one partial per cluster instead of
//           per CTA: 8x less partial traffic).
//   pass 2  partials [n_clusters,K,512] are summed in cluster order (fixed tree).
// Counts are int64 and exact.
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;
namespace team {

constexpr int SEG_THREADS = 128;
constexpr int SEG_UNROLL = 8;
constexpr int SEG_CLUSTER = 8;
constexpr int SEG_SLAB_KEYS = 24;      // 24 keys * 2 KB = 48 KB smem -> 4 CTAs / SM
constexpr int SEG_MAX_SLAB_KEYS = 104; // 208 KB of accumulators: the most one CTA can hold

template <typename T> struct RowLoad;
template <> struct RowLoad<float> {
    static __device__ __forceinline__ float4 load(const float* row, int t) { return ld_stream_f4(row + 4 * t); }
};
template <> struct RowLoad<__nv_bfloat16> {
    static __device__ __forceinline__ float4 load(const __nv_bfloat16* row, int t) {
        uint2 u = ld_stream_u2(row + 4 * t);
        return make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
    }
};

template <typename T, bool NORM, bool DEEP>
__global__ void __launch_bounds__(SEG_THREADS)
segsum_partial_kernel(const T* __restrict__ x, const int64_t* __restrict__ labels,
                      const int64_t* __restrict__ states, int64_t n_rows, int64_t rows_per_cta,
                      int64_t class_base, int num_classes, int num_states, int K, int slab_keys,
                      float* __restrict__ part_sums, long long* __restrict__ part_counts) {
    extern __shared__ __align__(16) unsigned char seg_smem[];
    float4* acc = reinterpret_cast<float4*>(seg_smem);                       // [slab_keys][128] float4
    int* cnt = reinterpret_cast<int*>(seg_smem + (size_t)slab_keys * D * sizeof(float));   // [slab_keys]
    float* red = reinterpret_cast<float*>(cnt + slab_keys);                  // [2][4][SEG_UNROLL]
    const int t = threadIdx.x;
    const int k0 = blockIdx.y * slab_keys;
    const int nk = min(slab_keys, K - k0);
    for (int i = t; i < slab_keys * (D / 4); i += SEG_THREADS) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < slab_keys) cnt[t] = 0;
    __syncthreads();

    const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t r1 = min(n_rows, r0 + rows_per_cta);
    // Three-deep software pipeline over groups of SEG_UNROLL rows.  A group needs three dependent memory round
    // trips (label, then state, then the feature row of a row whose key falls into this slab) before its serial
    // shared-memory read-modify-write chain; issued back to back they cost ~3 us per group and the memory system idles
    // (measured: 52 % of the HBM peak for class keys, 4 % for class x state keys).  Here the labels AND states of
    // group g+2 are requested unconditionally while the feature rows of group g+1 are in flight and group g is
    // accumulated, so every wait is one round trip old when it is consumed.
    auto load_raw = [&](int64_t r, int64_t (&lab)[SEG_UNROLL], int64_t (&stt)[SEG_UNROLL]) {
#pragma unroll
        for (int u = 0; u < SEG_UNROLL; ++u) {
            const int64_t row = r + u;
            lab[u] = -1; stt[u] = 0;
            if (row < r1) {
                lab[u] = __ldg(labels + row);
                if (states != nullptr) stt[u] = __ldg(states + row);
            }
        }
    };
    auto make_keys = [&](int64_t r, const int64_t (&lab)[SEG_UNROLL], const int64_t (&stt)[SEG_UNROLL], int (&key)[SEG_UNROLL]) {
#pragma unroll
        for (int u = 0; u < SEG_UNROLL; ++u) {
            key[u] = -1;
            if (r + u < r1) {
                const int64_t c = lab[u] - class_base;
                int64_t k = -1;
                if (c >= 0 && c < num_classes) {
                    if (states != nullptr) {
                        if (stt[u] >= 0 && stt[u] < num_states) k = c * num_states + stt[u];
                    } else {
                        k = c;
                    }
                }
                k -= k0;
                if (k >= 0 && k < nk) key[u] = (int)k;
            }
        }
    };
    auto load_feats = [&](int64_t r, const int (&key)[SEG_UNROLL], float4 (&v)[SEG_UNROLL]) {
#pragma unroll
        for (int u = 0; u < SEG_UNROLL; ++u) {
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (key[u] >= 0) v[u] = RowLoad<T>::load(x + (r + u) * D, t);
        }
    };
    int buf = 0;
    int key[SEG_UNROLL], keyn[SEG_UNROLL];
    float4 v[SEG_UNROLL], vn[SEG_UNROLL];
    int64_t lab[SEG_UNROLL], stt[SEG_UNROLL];
    // DEEP (class x state keys): the three-deep pipeline above.  Otherwise (class keys only: one round trip less per
    // group, and measured no faster - for bf16 rows slower - with the deeper pipeline) a two-deep one: the next
    // group's labels and features are requested before this group is accumulated.
    load_raw(r0, lab, stt);
    make_keys(r0, lab, stt, key);
    load_feats(r0, key, v);
    if (DEEP) load_raw(r0 + SEG_UNROLL, lab, stt);
    for (int64_t r = r0; r < r1; r += SEG_UNROLL) {
        if (DEEP) {
            // group g+1: keys from the raw values requested one iteration ago, feature loads now in flight
            make_keys(r + SEG_UNROLL, lab, stt, keyn);
            load_feats(r + SEG_UNROLL, keyn, vn);
            // group g+2: labels / states
            load_raw(r + 2 * SEG_UNROLL, lab, stt);
        } else {
            load_raw(r + SEG_UNROLL, lab, stt);
            make_keys(r + SEG_UNROLL, lab, stt, keyn);
            load_feats(r + SEG_UNROLL, keyn, vn);
        }
        if (NORM) {
            float ss[SEG_UNROLL];
#pragma unroll
            for (int u = 0; u < SEG_UNROLL; ++u) {
                ss[u] = v[u].x * v[u].x + v[u].y * v[u].y + v[u].z * v[u].z + v[u].w * v[u].w;
                ss[u] = warp_sum(ss[u]);
            }
            if ((t & 31) == 0) {
#pragma unroll
                for (int u = 0; u < SEG_UNROLL; ++u) red[(buf * 4 + (t >> 5)) * SEG_UNROLL + u] = ss[u];
            }
            __syncthreads();
#pragma unroll
            for (int u = 0; u < SEG_UNROLL; ++u) {
                const float tot = red[(buf * 4 + 0) * SEG_UNROLL + u] + red[(buf * 4 + 1) * SEG_UNROLL + u] +
                                  red[(buf * 4 + 2) * SEG_UNROLL + u] + red[(buf * 4 + 3) * SEG_UNROLL + u];
                const float inv = 1.0f / fmaxf(sqrtf(tot), NORM_EPS);
                v[u].x *= inv; v[u].y *= inv; v[u].z *= inv; v[u].w *= inv;
            }
            buf ^= 1;
        }
#pragma unroll
        for (int u = 0; u < SEG_UNROLL; ++u) {
            if (key[u] >= 0) {
                float4 a = acc[key[u] * (D / 4) + t];
                a.x += v[u].x; a.y += v[u].y; a.z += v[u].z; a.w += v[u].w;
                acc[key[u] * (D / 4) + t] = a;
                if (t == 0) cnt[key[u]] += 1;
            }
        }
#pragma unroll
        for (int u = 0; u < SEG_UNROLL; ++u) { key[u] = keyn[u]; v[u] = vn[u]; }
    }
    // fold the 8 CTAs of the cluster in rank order through distributed shared memory
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();
    const unsigned rank = cluster.block_rank();
    const int cluster_id = blockIdx.x / SEG_CLUSTER;
    // rank r owns float4 columns [16r, 16r+16) of every key
    for (int i = t; i < nk * 16; i += SEG_THREADS) {
        const int k = i >> 4, c4 = (int)rank * 16 + (i & 15);
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < SEG_CLUSTER; ++q) {
            const float4* remote = cluster.map_shared_rank(acc, q);
            const float4 a = remote[k * (D / 4) + c4];
            s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
        }
        reinterpret_cast<float4*>(part_sums)[((size_t)cluster_id * K + k0 + k) * (D / 4) + c4] = s;
    }
    if (rank == 0 && t < nk) {
        long long c = 0;
        for (int q = 0; q < SEG_CLUSTER; ++q) c += cluster.map_shared_rank(cnt, q)[t];
        part_counts[(size_t)cluster_id * K + k0 + t] = c;
    }
    cluster.sync();     // keep smem alive until every peer has read it
}

// ------------------------------------------------------------------ second generation of pass 1 (K <= 400 keys)
// The first generation above reaches 55 % of the HBM copy peak with class keys and 8.5 % with class x state keys
// (profiles/r1j_*): a feature row is only requested once its label has arrived and says its key lies in the CTA's key
// slab - every group of rows costs dependent round trips, and with several slabs the loads are sparse.  Here
//   * the COLUMNS are split instead of the keys: a CTA owns 128 * VEC columns (VEC = 4 / 2 / 1 floats per thread ->
//     1 / 2 / 4 CTAs side by side per row chunk) of ALL keys (K * VEC * 512 bytes of accumulators), so every row is
//     read exactly once, densely and unconditionally - the loads never wait for a label;
//   * keys are computed once per CTA for a block of 128 rows (thread t: row t) into shared memory, one block ahead;
//   * 2 x U rows are in flight per thread (double-buffered register groups);
//   * no clusters: the per-CTA partials ([chunks][K][512]) are summed by pass 2 in chunk order (< 2 % extra traffic).
// Thread t still owns its columns of every key accumulator and adds rows in row order: no atomics, bit-reproducible.
constexpr int SEG2_KBLK = 128;

template <typename T, int VEC> struct VecLoad;
template <> struct VecLoad<float, 4> { static __device__ __forceinline__ void load(const float* p, float (&v)[4]) { const float4 a = ld_stream_f4(p); v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; } };
template <> struct VecLoad<float, 2> { static __device__ __forceinline__ void load(const float* p, float (&v)[2]) { const uint2 a = ld_stream_u2(p); v[0] = __uint_as_float(a.x); v[1] = __uint_as_float(a.y); } };
template <> struct VecLoad<float, 1> { static __device__ __forceinline__ void load(const float* p, float (&v)[1]) { v[0] = __ldg(p); } };
template <> struct VecLoad<__nv_bfloat16, 4> { static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[4]) { const uint2 u = ld_stream_u2(p); v[0] = bf16_lo(u.x); v[1] = bf16_hi(u.x); v[2] = bf16_lo(u.y); v[3] = bf16_hi(u.y); } };
template <> struct VecLoad<__nv_bfloat16, 2> { static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[2]) { const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(p)); v[0] = bf16_lo(u); v[1] = bf16_hi(u); } };
template <> struct VecLoad<__nv_bfloat16, 1> { static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[1]) { v[0] = __bfloat162float(*p); } };

template <typename T, int VEC, int U, bool NORM, int NT>
__global__ void __launch_bounds__(NT)
segsum2_partial_kernel(const T* __restrict__ x, const int64_t* __restrict__ labels, const int64_t* __restrict__ states,
                       int64_t n_rows, int64_t rows_per_cta, int64_t class_base, int num_classes, int num_states, int K,
                       float* __restrict__ part_sums, long long* __restrict__ part_counts) {
    static_assert(NT >= SEG2_KBLK && (!NORM || (VEC == 4 && NT == 128)), "row normalisation needs the whole row in one CTA");
    static_assert(SEG2_KBLK % (2 * U) == 0, "key block must hold whole group pairs");
    extern __shared__ __align__(16) unsigned char seg_smem[];
    constexpr int W = NT * VEC;                        // columns of this CTA
    constexpr int NCOL = D / W;
    float* acc = reinterpret_cast<float*>(seg_smem);            // [K][W]
    int* cnt = reinterpret_cast<int*>(acc + (size_t)K * W);     // [K]
    int* keys = cnt + K;                                        // [2][SEG2_KBLK]
    float* red = reinterpret_cast<float*>(keys + 2 * SEG2_KBLK);    // [2][NT / 32][U] (NORM)
    const int t = threadIdx.x;
    const int cs = blockIdx.x % NCOL;
    const int64_t chunk = blockIdx.x / NCOL;
    for (int i = t; i < K * W; i += NT) acc[i] = 0.f;
    for (int i = t; i < K; i += NT) cnt[i] = 0;
    const int64_t r0 = chunk * rows_per_cta;
    const int64_t r1 = min(n_rows, r0 + rows_per_cta);
    const T* xc = x + (size_t)cs * W + (size_t)t * VEC;         // this thread's columns of row 0
    auto key_of = [&](int64_t row) -> int {
        if (row >= r1) return -1;
        const int64_t c = __ldg(labels + row) - class_base;
        if (c < 0 || c >= num_classes) return -1;
        if (states == nullptr) return (int)c;
        const int64_t s = __ldg(states + row);
        return (s >= 0 && s < num_states) ? (int)(c * num_states + s) : -1;
    };
    auto load_group = [&](int64_t r, float (&v)[U][VEC]) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (r + u < r1) {
                VecLoad<T, VEC>::load(xc + (r + u) * D, v[u]);
            } else {
#pragma unroll
                for (int q = 0; q < VEC; ++q) v[u][q] = 0.f;
            }
        }
    };
    int nbuf = 0;
    auto add_group = [&](const int* kb, float (&v)[U][VEC]) {
        if (NORM) {
            float ss[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                ss[u] = 0.f;
#pragma unroll
                for (int q = 0; q < VEC; ++q) ss[u] = fmaf(v[u][q], v[u][q], ss[u]);
                ss[u] = warp_sum(ss[u]);
            }
            if ((t & 31) == 0) {
#pragma unroll
                for (int u = 0; u < U; ++u) red[(nbuf * 4 + (t >> 5)) * U + u] = ss[u];
            }
            __syncthreads();
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const float tot = red[(nbuf * 4 + 0) * U + u] + red[(nbuf * 4 + 1) * U + u] + red[(nbuf * 4 + 2) * U + u] + red[(nbuf * 4 + 3) * U + u];
                const float inv = 1.0f / fmaxf(sqrtf(tot), NORM_EPS);
#pragma unroll
                for (int q = 0; q < VEC; ++q) v[u][q] *= inv;
            }
            nbuf ^= 1;
        }
        // Four rows at a time.  The read-modify-write of a row depends on the previous one only when the keys collide, but
        // the compiler has to assume they always do: one serial shared-memory round trip per row (~180 cycles measured)
        // bounded the row rate of the whole CTA - every warp has to walk every row of the chunk.  With four DISTINCT valid
        // keys (a CTA-uniform test) the four updates are independent and issue back to back; otherwise in row order.
        auto rmw = [&](int k, const float (&x)[VEC]) {
            float* a = acc + (size_t)k * W + t * VEC;
            if (VEC == 4) {
                float4 o = *reinterpret_cast<float4*>(a);
                o.x += x[0]; o.y += x[1 % VEC]; o.z += x[2 % VEC]; o.w += x[3 % VEC];
                *reinterpret_cast<float4*>(a) = o;
            } else if (VEC == 2) {
                float2 o = *reinterpret_cast<float2*>(a);
                o.x += x[0]; o.y += x[1 % VEC];
                *reinterpret_cast<float2*>(a) = o;
            } else {
                a[0] += x[0];
            }
        };
#pragma unroll
        for (int u = 0; u < U; u += 4) {
            const int k0 = kb[u], k1 = kb[u + 1], k2 = kb[u + 2], k3 = kb[u + 3];
            const bool indep = (k0 | k1 | k2 | k3) >= 0 && k0 != k1 && k0 != k2 && k0 != k3 && k1 != k2 && k1 != k3 && k2 != k3;
            if (indep) {
                float* a0 = acc + (size_t)k0 * W + t * VEC; float* a1 = acc + (size_t)k1 * W + t * VEC;
                float* a2 = acc + (size_t)k2 * W + t * VEC; float* a3 = acc + (size_t)k3 * W + t * VEC;
                if (VEC == 4) {
                    float4 o0 = *reinterpret_cast<float4*>(a0), o1 = *reinterpret_cast<float4*>(a1);
                    float4 o2 = *reinterpret_cast<float4*>(a2), o3 = *reinterpret_cast<float4*>(a3);
                    o0.x += v[u][0]; o0.y += v[u][1 % VEC]; o0.z += v[u][2 % VEC]; o0.w += v[u][3 % VEC];
                    o1.x += v[u + 1][0]; o1.y += v[u + 1][1 % VEC]; o1.z += v[u + 1][2 % VEC]; o1.w += v[u + 1][3 % VEC];
                    o2.x += v[u + 2][0]; o2.y += v[u + 2][1 % VEC]; o2.z += v[u + 2][2 % VEC]; o2.w += v[u + 2][3 % VEC];
                    o3.x += v[u + 3][0]; o3.y += v[u + 3][1 % VEC]; o3.z += v[u + 3][2 % VEC]; o3.w += v[u + 3][3 % VEC];
                    *reinterpret_cast<float4*>(a0) = o0; *reinterpret_cast<float4*>(a1) = o1;
                    *reinterpret_cast<float4*>(a2) = o2; *reinterpret_cast<float4*>(a3) = o3;
                } else if (VEC == 2) {
                    float2 o0 = *reinterpret_cast<float2*>(a0), o1 = *reinterpret_cast<float2*>(a1);
                    float2 o2 = *reinterpret_cast<float2*>(a2), o3 = *reinterpret_cast<float2*>(a3);
                    o0.x += v[u][0]; o0.y += v[u][1 % VEC]; o1.x += v[u + 1][0]; o1.y += v[u + 1][1 % VEC];
                    o2.x += v[u + 2][0]; o2.y += v[u + 2][1 % VEC]; o3.x += v[u + 3][0]; o3.y += v[u + 3][1 % VEC];
                    *reinterpret_cast<float2*>(a0) = o0; *reinterpret_cast<float2*>(a1) = o1;
                    *reinterpret_cast<float2*>(a2) = o2; *reinterpret_cast<float2*>(a3) = o3;
                } else {
                    const float o0 = a0[0] + v[u][0], o1 = a1[0] + v[u + 1][0], o2 = a2[0] + v[u + 2][0], o3 = a3[0] + v[u + 3][0];
                    a0[0] = o0; a1[0] = o1; a2[0] = o2; a3[0] = o3;
                }
                if (t == 0 && cs == 0) { cnt[k0] += 1; cnt[k1] += 1; cnt[k2] += 1; cnt[k3] += 1; }
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int k = kb[u + e];
                    if (k >= 0) {
                        rmw(k, v[u + e]);
                        if (t == 0 && cs == 0) cnt[k] += 1;
                    }
                }
            }
        }
    };
    float va[U][VEC], vb[U][VEC];
    if (t < SEG2_KBLK) keys[t] = key_of(r0 + t);  // thread t < 128 computes the key of row t of a block
    load_group(r0, va);
    __syncthreads();
    int cur = 0;
    for (int64_t blk = r0; blk < r1; blk += SEG2_KBLK) {
        const int knext = t < SEG2_KBLK ? key_of(blk + SEG2_KBLK + t) : -1;      // next block's keys: in flight under this block
        const int* kb = keys + cur * SEG2_KBLK;
#pragma unroll 1
        for (int g = 0; g < SEG2_KBLK; g += 2 * U) {
            const int64_t r = blk + g;
            load_group(r + U, vb);
            add_group(kb + g, va);
            load_group(r + 2 * U, va);
            add_group(kb + g + U, vb);
        }
        if (t < SEG2_KBLK) keys[(cur ^ 1) * SEG2_KBLK + t] = knext;
        __syncthreads();
        cur ^= 1;
    }
    // per-CTA partial: [chunk][K][512], this CTA's columns
    float* out = part_sums + ((size_t)chunk * K) * D + (size_t)cs * W;
    for (int i = t; i < K * (W / VEC); i += NT) {
        const int k = i / (W / VEC), c = (i - k * (W / VEC)) * VEC;
#pragma unroll
        for (int q = 0; q < VEC; ++q) out[(size_t)k * D + c + q] = acc[(size_t)k * W + c + q];
    }
    if (cs == 0) for (int i = t; i < K; i += NT) part_counts[(size_t)chunk * K + i] = cnt[i];
}

// ------------------------------------------------------------------ third generation of pass 1 (many keys: K > 100)
// With K = 200 (class x state) keys the accumulators of all keys no longer fit beside each other at full row width:
// the second generation then gives every thread ONE column (4-byte loads, a shared-memory read-modify-write per 4 bytes)
// and measured 32 % of the HBM copy peak.  Here the rows are first PARTITIONED by key, which costs a few bytes per row,
// and then summed straight from HBM into registers - no shared-memory accumulators at all:
//   A  sg_rank_kernel     per block of 1024 rows: key of every row, its stable rank among the block's rows of that key
//                         (warp match + per-warp counts), per-block key counts                       reads 16 B / row
//   B  sg_scan_kernel     per key: exclusive scan of the block counts (a row's position = key start + blocks before +
//                         rank); sg_table_kernel: key starts and the segment table (runs of <= seg_len rows of one key)
//   C  sg_scatter_kernel  row index -> its position in the key-sorted order                            8 B / row
//   D  sg_gather_kernel   one warp per segment: streams its rows (whole 2 KB rows, 4 in flight, 128-bit loads) and adds
//                         them in index order in registers; one partial row per segment
//   E  sg_fold_kernel     per key: partials in segment order
// Everything is a pure function of the input: ranks come from ballots, not from atomics' arrival order - bit-reproducible.
constexpr int SG_BLK = 1024;           // rows per ranking block (one thread per row)
constexpr int SG_SEG_MAX = 512;        // rows per gather segment (fewer for small inputs: >= ~32 warps per SM wanted)
constexpr int SG_GW = 8;               // warps per gather CTA

__device__ __forceinline__ int sg_key(const int64_t* __restrict__ labels, const int64_t* __restrict__ states, int64_t row,
                                      int64_t n_rows, int64_t class_base, int num_classes, int num_states, int K) {
    if (row >= n_rows) return -1;
    const int64_t c = __ldg(labels + row) - class_base;
    if (c < 0 || c >= num_classes) return K;                       // bucket K = rows that belong to no key
    if (states == nullptr) return (int)c;
    const int64_t st = __ldg(states + row);
    return (st >= 0 && st < num_states) ? (int)(c * num_states + st) : K;
}

// packed[row] = key << 10 | rank within (block, key);  blk_counts[key][block]
__global__ void __launch_bounds__(SG_BLK)
sg_rank_kernel(const int64_t* __restrict__ labels, const int64_t* __restrict__ states, int64_t n_rows, int64_t class_base,
               int num_classes, int num_states, int K, int nblk, int* __restrict__ packed, int* __restrict__ blk_counts) {
    extern __shared__ int sg_cnt[];                                // [32 warps][K + 1]
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5, K1 = K + 1;
    for (int i = t; i < 32 * K1; i += SG_BLK) sg_cnt[i] = 0;
    __syncthreads();
    const int64_t row = (int64_t)blockIdx.x * SG_BLK + t;
    const int key = sg_key(labels, states, row, n_rows, class_base, num_classes, num_states, K);
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    const int wrank = __popc(peers & ((1u << lane) - 1u));
    if (key >= 0 && wrank == 0) sg_cnt[warp * K1 + key] = __popc(peers);      // one writer per (warp, key)
    __syncthreads();
    for (int k = t; k < K1; k += SG_BLK) {                         // exclusive scan over the warps, per key
        int run = 0;
        for (int w = 0; w < 32; ++w) { const int c = sg_cnt[w * K1 + k]; sg_cnt[w * K1 + k] = run; run += c; }
        blk_counts[(size_t)k * nblk + blockIdx.x] = run;
    }
    __syncthreads();
    if (key >= 0) packed[row] = (key << 10) | (sg_cnt[warp * K1 + key] + wrank);
}

// one CTA per key: blk_counts[key][:] -> exclusive scan in place, totals[key]
__global__ void __launch_bounds__(1024)
sg_scan_kernel(int* __restrict__ blk_counts, int nblk, long long* __restrict__ totals) {
    __shared__ long long part[1024];
    const int t = threadIdx.x;
    int* c = blk_counts + (size_t)blockIdx.x * nblk;
    const int per = (nblk + 1023) / 1024;
    const int b0 = t * per, b1 = min(nblk, b0 + per);
    long long s = 0;
    for (int b = b0; b < b1; ++b) s += c[b];
    part[t] = s;
    __syncthreads();
    if (t == 0) {
        long long run = 0;
        for (int i = 0; i < 1024; ++i) { const long long v = part[i]; part[i] = run; run += v; }
        totals[blockIdx.x] = run;
    }
    __syncthreads();
    long long run = part[t];
    for (int b = b0; b < b1; ++b) { const int v = c[b]; c[b] = (int)run; run += v; }
}

// key_start[k] (exclusive scan of the totals) and seg_base[k] (segments before key k); single CTA
__global__ void __launch_bounds__(32)
sg_table_kernel(const long long* __restrict__ totals, int K, int seg_len, long long* __restrict__ key_start, int* __restrict__ seg_base) {
    if (threadIdx.x != 0) return;
    long long run = 0;
    int segs = 0;
    for (int k = 0; k <= K; ++k) {
        key_start[k] = run;
        seg_base[k] = segs;
        run += totals[k];
        if (k < K) segs += (int)((totals[k] + seg_len - 1) / seg_len);
    }
    seg_base[K] = segs;            // total number of segments (bucket K is never gathered)
}

__global__ void __launch_bounds__(256)
sg_scatter_kernel(const int* __restrict__ packed, const int* __restrict__ blk_excl, const long long* __restrict__ key_start,
                  int64_t n_rows, int nblk, int* __restrict__ order) {
    const int64_t row = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (row >= n_rows) return;
    const int p = packed[row];
    const int key = p >> 10, rank = p & 1023;
    const int blk = (int)(row / SG_BLK);
    order[key_start[key] + blk_excl[(size_t)key * nblk + blk] + rank] = (int)row;
}

template <typename T, bool NORM>
__global__ void __launch_bounds__(SG_GW * 32)
sg_gather_kernel(const T* __restrict__ x, const int* __restrict__ order, const long long* __restrict__ key_start,
                 const long long* __restrict__ totals, const int* __restrict__ seg_base, int K, int seg_len, float* __restrict__ partials) {
    const int lane = threadIdx.x & 31;
    const int seg = blockIdx.x * SG_GW + (threadIdx.x >> 5);
    if (seg >= seg_base[K]) return;
    int lo = 0, hi = K;                                            // last key with seg_base[key] <= seg
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (seg_base[mid] <= seg) lo = mid; else hi = mid; }
    const int key = lo;
    const long long first = key_start[key] + (long long)(seg - seg_base[key]) * seg_len;
    const long long last = min(key_start[key] + totals[key], first + seg_len);
    float4 acc[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    constexpr int U = 4;
    for (long long p = first; p < last; p += U) {
        int r[U];
        float4 v[U][4];
#pragma unroll
        for (int u = 0; u < U; ++u) r[u] = p + u < last ? __ldg(order + p + u) : -1;
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                v[u][j] = r[u] >= 0 ? RowLoad<T>::load(x + (size_t)r[u] * D, lane + 32 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            float inv = 1.f;
            if (NORM) {
                float ss = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) ss += v[u][j].x * v[u][j].x + v[u][j].y * v[u][j].y + v[u][j].z * v[u][j].z + v[u][j].w * v[u][j].w;
                inv = 1.0f / fmaxf(sqrtf(warp_sum(ss)), NORM_EPS);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[j].x = fmaf(v[u][j].x, inv, acc[j].x); acc[j].y = fmaf(v[u][j].y, inv, acc[j].y);
                acc[j].z = fmaf(v[u][j].z, inv, acc[j].z); acc[j].w = fmaf(v[u][j].w, inv, acc[j].w);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) reinterpret_cast<float4*>(partials + (size_t)seg * D)[lane + 32 * j] = acc[j];
}

__global__ void __launch_bounds__(128)
sg_fold_kernel(const float* __restrict__ partials, const int* __restrict__ seg_base, const long long* __restrict__ totals,
               float* __restrict__ sums, int64_t* __restrict__ counts) {
    const int k = blockIdx.x, c4 = threadIdx.x;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    const int s0 = seg_base[k], s1 = seg_base[k + 1];
    int q = s0;
    for (; q + 4 <= s1; q += 4) {
        float4 a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] = reinterpret_cast<const float4*>(partials + (size_t)(q + u) * D)[c4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { s.x += a[u].x; s.y += a[u].y; s.z += a[u].z; s.w += a[u].w; }
    }
    for (; q < s1; ++q) {
        const float4 a = reinterpret_cast<const float4*>(partials + (size_t)q * D)[c4];
        s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
    }
    reinterpret_cast<float4*>(sums)[(size_t)k * (D / 4) + c4] = s;
    if (c4 == 0) counts[k] = totals[k];
}

struct SgPlan {
    int nblk, seg_len;
    int64_t max_segs;
    size_t off_packed, off_order, off_blk, off_totals, off_kstart, off_segbase, off_partials, total;
};
static SgPlan sg_plan(int64_t n_rows, int64_t K) {
    SgPlan p;
    p.nblk = (int)((n_rows + SG_BLK - 1) / SG_BLK);
    if (p.nblk < 1) p.nblk = 1;
    p.seg_len = SG_SEG_MAX;                                        // ~4 700 warp-segments fill the machine (148 SMs x 32 warps)
    while (p.seg_len > 64 && n_rows / p.seg_len < 4736) p.seg_len >>= 1;
    p.max_segs = n_rows / p.seg_len + K + 1;
    size_t off = 0;
    auto take = [&](size_t b) { const size_t r = off; off += align_up(b, 256); return r; };
    p.off_packed = take((size_t)p.nblk * SG_BLK * sizeof(int));
    p.off_order = take((size_t)(n_rows > 0 ? n_rows : 1) * sizeof(int));
    p.off_blk = take((size_t)(K + 1) * p.nblk * sizeof(int));
    p.off_totals = take((size_t)(K + 2) * sizeof(long long));
    p.off_kstart = take((size_t)(K + 2) * sizeof(long long));
    p.off_segbase = take((size_t)(K + 2) * sizeof(int));
    p.off_partials = take((size_t)p.max_segs * D * sizeof(float));
    p.total = off;
    return p;
}
// the sorted path serves many-key problems (K > 100) of any size up to 2^31 rows and K < 2^20
// ... and bf16 rows with few keys from 64 K rows on: the shared-memory kernel is issue-bound on 1 KB rows (45 % of the copy peak
// at 4 M rows), the gather is not
static bool sg_wanted(int64_t n_rows, int64_t K, bool bf16_rows = false) {
    const bool many_keys = K > 100 && n_rows >= 4096;
    const bool narrow_rows = bf16_rows && n_rows >= 65536;
    return (many_keys || narrow_rows) && K < (1 << 20) && n_rows < (1ll << 31) && (size_t)(K + 1) * 32 * sizeof(int) <= 200 * 1024;
}

template <typename T>
static int sg_run(const void* x, const int64_t* labels, const int64_t* states, int64_t n_rows, int64_t class_base, int num_classes,
                  int num_states, int K, bool norm, float* sums, int64_t* counts, void* ws, cudaStream_t st) {
    const SgPlan p = sg_plan(n_rows, K);
    char* b = reinterpret_cast<char*>(ws);
    int* packed = reinterpret_cast<int*>(b + p.off_packed);
    int* order = reinterpret_cast<int*>(b + p.off_order);
    int* blk = reinterpret_cast<int*>(b + p.off_blk);
    long long* totals = reinterpret_cast<long long*>(b + p.off_totals);
    long long* kstart = reinterpret_cast<long long*>(b + p.off_kstart);
    int* segbase = reinterpret_cast<int*>(b + p.off_segbase);
    float* partials = reinterpret_cast<float*>(b + p.off_partials);
    const size_t smem = (size_t)32 * (K + 1) * sizeof(int);
    TEAM_CUDA_CHECK(cudaFuncSetAttribute(sg_rank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sg_rank_kernel<<<p.nblk, SG_BLK, smem, st>>>(labels, states, n_rows, class_base, num_classes, num_states, K, p.nblk, packed, blk);
    TEAM_LAUNCH_CHECK("sg_rank_kernel");
    sg_scan_kernel<<<K + 1, 1024, 0, st>>>(blk, p.nblk, totals);
    TEAM_LAUNCH_CHECK("sg_scan_kernel");
    sg_table_kernel<<<1, 32, 0, st>>>(totals, K, p.seg_len, kstart, segbase);
    TEAM_LAUNCH_CHECK("sg_table_kernel");
    sg_scatter_kernel<<<(unsigned)((n_rows + 255) / 256), 256, 0, st>>>(packed, blk, kstart, n_rows, p.nblk, order);
    TEAM_LAUNCH_CHECK("sg_scatter_kernel");
    const unsigned gblocks = (unsigned)((p.max_segs + SG_GW - 1) / SG_GW);
    const T* xp = reinterpret_cast<const T*>(x);
    if (norm) sg_gather_kernel<T, true><<<gblocks, SG_GW * 32, 0, st>>>(xp, order, kstart, totals, segbase, K, p.seg_len, partials);
    else sg_gather_kernel<T, false><<<gblocks, SG_GW * 32, 0, st>>>(xp, order, kstart, totals, segbase, K, p.seg_len, partials);
    TEAM_LAUNCH_CHECK("sg_gather_kernel");
    sg_fold_kernel<<<K, 128, 0, st>>>(partials, segbase, totals, sums, counts);
    TEAM_LAUNCH_CHECK("sg_fold_kernel");
    return TEAM_OK;
}

// pass 2: fixed-order sum over clusters.  grid = K, 512 threads = 128 float4 columns x 4 lanes
// of cluster partials; lane g sums clusters g, g+4, ... then the 4 lanes fold in order.
__global__ void __launch_bounds__(512)
segsum_final_kernel(const float* __restrict__ part_sums, const long long* __restrict__ part_counts,
                    int n_clusters, int K, float* __restrict__ sums, int64_t* __restrict__ counts) {
    __shared__ float4 fold[4][128];
    const int k = blockIdx.x, c4 = threadIdx.x & 127, g = threadIdx.x >> 7;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int q = g; q < n_clusters; q += 4) {
        const float4 a = reinterpret_cast<const float4*>(part_sums)[((size_t)q * K + k) * (D / 4) + c4];
        s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
    }
    fold[g][c4] = s;
    __syncthreads();
    if (g == 0) {
        float4 r = fold[0][c4];
#pragma unroll
        for (int q = 1; q < 4; ++q) { r.x += fold[q][c4].x; r.y += fold[q][c4].y; r.z += fold[q][c4].z; r.w += fold[q][c4].w; }
        reinterpret_cast<float4*>(sums)[(size_t)k * (D / 4) + c4] = r;
    }
    if (threadIdx.x == 0) {
        long long c = 0;
        for (int q = 0; q < n_clusters; ++q) c += part_counts[(size_t)q * K + k];
        counts[k] = c;
    }
}

// means[k] = sums[k]/counts[k] (count>0 only); optional per-group (class) totals over `group` keys.
__global__ void __launch_bounds__(128)
segmean_kernel(const float* __restrict__ sums, const int64_t* __restrict__ counts, int K,
               float* __restrict__ means, int group, float* __restrict__ class_means,
               int64_t* __restrict__ class_counts) {
    const int c4 = threadIdx.x;
    if (class_means == nullptr && class_counts == nullptr) {
        const int k = blockIdx.x;
        const int64_t n = counts[k];
        if (n > 0 && means != nullptr) {
            float4 s = reinterpret_cast<const float4*>(sums)[(size_t)k * (D / 4) + c4];
            const float fn = (float)n;
            reinterpret_cast<float4*>(means)[(size_t)k * (D / 4) + c4] = make_float4(s.x / fn, s.y / fn, s.z / fn, s.w / fn);
        }
        return;
    }
    const int gidx = blockIdx.x;            // one CTA per group (class)
    float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
    int64_t ntot = 0;
    for (int j = 0; j < group; ++j) {
        const int k = gidx * group + j;
        const int64_t n = counts[k];
        if (n > 0) {
            const float4 s = reinterpret_cast<const float4*>(sums)[(size_t)k * (D / 4) + c4];
            tot.x += s.x; tot.y += s.y; tot.z += s.z; tot.w += s.w;
            ntot += n;
            if (means != nullptr) {
                const float fn = (float)n;
                reinterpret_cast<float4*>(means)[(size_t)k * (D / 4) + c4] = make_float4(s.x / fn, s.y / fn, s.z / fn, s.w / fn);
            }
        }
    }
    if (ntot > 0 && class_means != nullptr) {
        const float fn = (float)ntot;
        reinterpret_cast<float4*>(class_means)[(size_t)gidx * (D / 4) + c4] = make_float4(tot.x / fn, tot.y / fn, tot.z / fn, tot.w / fn);
    }
    if (c4 == 0 && class_counts != nullptr) class_counts[gidx] = ntot;
}

static void seg_plan(int64_t n_rows, int64_t K, int* n_clusters, int* n_slabs, int* slab_keys, int64_t* rows_per_cta) {
    // Few keys (class-only, K <= 24): 48 KB of accumulators, 4 CTAs per SM.  Many keys (class x state): a CTA only
    // loads the rows whose key falls into its slab, so small slabs mean sparse loads and an idle memory system
    // (measured: 24-key slabs at K = 200 ran at 4 % of the HBM peak) - use the largest slabs shared memory allows
    // (<= 104 keys = 208 KB, one CTA per SM), i.e. the fewest passes over the label stream.
    if (K <= SEG_SLAB_KEYS) {
        *slab_keys = (int)K;
        *n_slabs = 1;
    } else {
        *n_slabs = (int)((K + SEG_MAX_SLAB_KEYS - 1) / SEG_MAX_SLAB_KEYS);
        *slab_keys = (int)((K + *n_slabs - 1) / *n_slabs);
    }
    const int occ = *slab_keys <= SEG_SLAB_KEYS ? 4 : (*slab_keys <= 52 ? 2 : 1);       // CTAs per SM by shared memory
    // aim for >= 256 rows per CTA, at most one resident wave across all slabs
    int64_t max_ctas = (int64_t)NUM_SMS * occ / *n_slabs;
    if (max_ctas < SEG_CLUSTER) max_ctas = SEG_CLUSTER;
    int64_t ctas = (n_rows + 255) / 256;
    if (ctas > max_ctas) ctas = max_ctas;
    int64_t ncl = (ctas + SEG_CLUSTER - 1) / SEG_CLUSTER;
    if (ncl < 1) ncl = 1;
    *n_clusters = (int)ncl;
    int64_t total = ncl * SEG_CLUSTER;
    int64_t rpc = (n_rows + total - 1) / total;
    rpc = (rpc + SEG_UNROLL - 1) / SEG_UNROLL * SEG_UNROLL;
    if (rpc < SEG_UNROLL) rpc = SEG_UNROLL;
    *rows_per_cta = rpc;
}

// second generation: columns per CTA (128 x 4 floats for K <= 100, 256 x 1 for K <= 200, 128 x 1 for K <= 400), n_chunks row
// chunks; returns false when the first generation must run
static bool seg2_plan(int64_t n_rows, int64_t K, bool norm, int* width, int* n_chunks, int64_t* rows_per_cta) {
    if (K > 400 || (norm && K > 100)) return false;
    const int w = K <= 100 ? 512 : (K <= 200 ? 256 : 128);
    const size_t smem = (size_t)K * w * sizeof(float) + 8192;
    int occ = (int)((size_t)(220 * 1024) / smem);
    if (occ < 1) occ = 1;
    if (occ > 4) occ = 4;                                // ~100 registers x 128 threads per CTA
    const int ncol = 512 / w;
    int64_t chunks = (int64_t)NUM_SMS * occ / ncol;
    const int64_t by_rows = (n_rows + 4 * SEG2_KBLK - 1) / (4 * SEG2_KBLK);      // at least 512 rows per chunk
    if (chunks > by_rows) chunks = by_rows;
    if (chunks < 1) chunks = 1;
    int64_t rpc = (n_rows + chunks - 1) / chunks;
    rpc = (rpc + SEG2_KBLK - 1) / SEG2_KBLK * SEG2_KBLK;
    if (rpc < SEG2_KBLK) rpc = SEG2_KBLK;
    chunks = n_rows > 0 ? (n_rows + rpc - 1) / rpc : 1;
    *width = w; *n_chunks = (int)chunks; *rows_per_cta = rpc;
    return true;
}

template <typename T, int VEC, int U, bool NORM, int NT>
static int seg2_launch(const void* x, const int64_t* labels, const int64_t* states, int64_t n_rows, int64_t class_base,
                       int num_classes, int num_states, int K, int n_chunks, int64_t rows_per_cta, float* part_sums,
                       long long* part_counts, cudaStream_t st) {
    const size_t smem = (size_t)K * VEC * NT * sizeof(float) + (size_t)K * sizeof(int) + 2 * SEG2_KBLK * sizeof(int) +
                        2 * (NT / 32) * U * sizeof(float);
    auto kern = segsum2_partial_kernel<T, VEC, U, NORM, NT>;
    TEAM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<n_chunks * (D / (VEC * NT)), NT, smem, st>>>(reinterpret_cast<const T*>(x), labels, states, n_rows, rows_per_cta,
                                                        class_base, num_classes, num_states, K, part_sums, part_counts);
    count_launch();
    TEAM_LAUNCH_CHECK("segsum2_partial_kernel");
    return TEAM_OK;
}

template <typename T, bool NORM, bool DEEP>
static int seg_launch(const void* x, const int64_t* labels, const int64_t* states, int64_t n_rows,
                      int64_t class_base, int num_classes, int num_states, int K, int n_clusters,
                      int n_slabs, int slab_keys, int64_t rows_per_cta, float* part_sums,
                      long long* part_counts, cudaStream_t st) {
    const size_t smem = (size_t)slab_keys * D * sizeof(float) + (size_t)slab_keys * sizeof(int) +
                        2 * 4 * SEG_UNROLL * sizeof(float);
    auto kern = segsum_partial_kernel<T, NORM, DEEP>;
    TEAM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_clusters * SEG_CLUSTER, n_slabs, 1);
    cfg.blockDim = dim3(SEG_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = SEG_CLUSTER;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const T* xp = reinterpret_cast<const T*>(x);
    TEAM_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, xp, labels, states, n_rows, rows_per_cta, class_base,
                                       num_classes, num_states, K, slab_keys, part_sums, part_counts));
    return TEAM_OK;
}

}  // namespace team

using namespace team;

extern "C" size_t team_segsum_workspace_bytes(int64_t n_rows, int64_t num_keys) {
    int ncl, nsl, sk;
    int64_t rpc;
    if (num_keys < 1) num_keys = 1;
    seg_plan(n_rows, num_keys, &ncl, &nsl, &sk, &rpc);
    int vec, chunks;
    if (seg2_plan(n_rows, num_keys, false, &vec, &chunks, &rpc) && chunks > ncl) ncl = chunks;      // partial records of either generation
    size_t need = align_up((size_t)ncl * num_keys * D * sizeof(float), 256) + align_up((size_t)ncl * num_keys * sizeof(long long), 256);
    if (sg_wanted(n_rows, num_keys, true)) { const size_t s3 = sg_plan(n_rows, num_keys).total; if (s3 > need) need = s3; }
    return need;
}

extern "C" int team_segsum(const void* x, int x_dtype, const int64_t* labels, const int64_t* states,
                           int64_t n_rows, int64_t class_base, int64_t num_classes, int64_t num_states,
                           int normalize_rows, float* sums, int64_t* counts, void* workspace,
                           size_t workspace_bytes, void* stream) {
    TEAM_REQUIRE(n_rows >= 0 && num_classes >= 1, "team_segsum: n_rows=%lld num_classes=%lld", (long long)n_rows, (long long)num_classes);
    TEAM_REQUIRE(x_dtype == TEAM_DTYPE_F32 || x_dtype == TEAM_DTYPE_BF16, "team_segsum: bad dtype %d", x_dtype);
    TEAM_REQUIRE(sums != nullptr && counts != nullptr && (labels != nullptr || n_rows == 0), "team_segsum: null output/labels");
    if (states == nullptr) num_states = 1;
    TEAM_REQUIRE(num_states >= 1 && num_classes * num_states <= (1 << 20), "team_segsum: too many keys");
    const int K = (int)(num_classes * num_states);
    int ncl, nsl, sk;
    int64_t rpc;
    seg_plan(n_rows, K, &ncl, &nsl, &sk, &rpc);
    const size_t need = team_segsum_workspace_bytes(n_rows, K);
    if (workspace == nullptr || workspace_bytes < need) {
        set_error("team_segsum: workspace %zu < %zu", workspace_bytes, need);
        return TEAM_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (sg_wanted(n_rows, K, x_dtype == TEAM_DTYPE_BF16)) {            // many keys (or narrow rows): partition the rows by key, then sum them straight from HBM
        TEAM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "team_segsum: workspace must be 256-byte aligned");
        return x_dtype == TEAM_DTYPE_F32
                   ? sg_run<float>(x, labels, states, n_rows, class_base, (int)num_classes, (int)num_states, K, normalize_rows != 0, sums, counts, workspace, st)
                   : sg_run<__nv_bfloat16>(x, labels, states, n_rows, class_base, (int)num_classes, (int)num_states, K, normalize_rows != 0, sums, counts, workspace, st);
    }
    float* part_sums = reinterpret_cast<float*>(workspace);
    int vec2 = 0, chunks2 = 0;
    int64_t rpc2 = 0;
    if (seg2_plan(n_rows, K, normalize_rows != 0, &vec2, &chunks2, &rpc2)) {       // column-partitioned pass 1 (K <= 400)
        long long* pc = reinterpret_cast<long long*>(reinterpret_cast<char*>(workspace) + align_up((size_t)chunks2 * K * D * sizeof(float), 256));
        TEAM_REQUIRE(align_up((size_t)chunks2 * K * D * sizeof(float), 256) + (size_t)chunks2 * K * sizeof(long long) <= workspace_bytes, "team_segsum: workspace too small");
        int rc2;
#define SEG2_GO(T, VEC, U, NORM, NT) seg2_launch<T, VEC, U, NORM, NT>(x, labels, states, n_rows, class_base, (int)num_classes, (int)num_states, K, chunks2, rpc2, part_sums, pc, st)
        if (x_dtype == TEAM_DTYPE_F32) {
            rc2 = vec2 == 512 ? (normalize_rows ? SEG2_GO(float, 4, 8, true, 128) : SEG2_GO(float, 4, 8, false, 128))
                              : (vec2 == 256 ? SEG2_GO(float, 1, 32, false, 256) : SEG2_GO(float, 1, 32, false, 128));
        } else {
            rc2 = vec2 == 512 ? (normalize_rows ? SEG2_GO(__nv_bfloat16, 4, 8, true, 128) : SEG2_GO(__nv_bfloat16, 4, 8, false, 128))
                              : (vec2 == 256 ? SEG2_GO(__nv_bfloat16, 1, 32, false, 256) : SEG2_GO(__nv_bfloat16, 1, 32, false, 128));
        }
#undef SEG2_GO
        if (rc2 != TEAM_OK) return rc2;
        segsum_final_kernel<<<K, 512, 0, st>>>(part_sums, pc, chunks2, K, sums, counts);
        count_launch();
        TEAM_LAUNCH_CHECK("segsum_final_kernel");
        return TEAM_OK;
    }
    long long* part_counts = reinterpret_cast<long long*>(reinterpret_cast<char*>(workspace) +
                                                          align_up((size_t)ncl * K * D * sizeof(float), 256));
    int rc;
#define SEG_GO(T, NORM, DEEP) seg_launch<T, NORM, DEEP>(x, labels, states, n_rows, class_base, (int)num_classes, (int)num_states, K, ncl, nsl, sk, rpc, part_sums, part_counts, st)
    const bool deep = states != nullptr;
    if (x_dtype == TEAM_DTYPE_F32) {
        rc = normalize_rows ? (deep ? SEG_GO(float, true, true) : SEG_GO(float, true, false))
                            : (deep ? SEG_GO(float, false, true) : SEG_GO(float, false, false));
    } else {
        rc = normalize_rows ? (deep ? SEG_GO(__nv_bfloat16, true, true) : SEG_GO(__nv_bfloat16, true, false))
                            : (deep ? SEG_GO(__nv_bfloat16, false, true) : SEG_GO(__nv_bfloat16, false, false));
    }
#undef SEG_GO
    if (rc != TEAM_OK) return rc;
    segsum_final_kernel<<<K, 512, 0, st>>>(part_sums, part_counts, ncl, K, sums, counts);
    TEAM_LAUNCH_CHECK("segsum_final_kernel");
    return TEAM_OK;
}

extern "C" int team_segmean_finalize(const float* sums, const int64_t* counts, int64_t num_keys,
                                     float* means, int64_t group, float* class_means,
                                     int64_t* class_counts, void* stream) {
    TEAM_REQUIRE(num_keys >= 1 && sums && counts, "team_segmean_finalize: bad args");
    cudaStream_t st = (cudaStream_t)stream;
    if (class_means == nullptr && class_counts == nullptr) {
        segmean_kernel<<<(int)num_keys, 128, 0, st>>>(sums, counts, (int)num_keys, means, 1, nullptr, nullptr);
    } else {
        TEAM_REQUIRE(group >= 1 && num_keys % group == 0, "team_segmean_finalize: group %lld does not divide %lld", (long long)group, (long long)num_keys);
        segmean_kernel<<<(int)(num_keys / group), 128, 0, st>>>(sums, counts, (int)num_keys, means, (int)group, class_means, class_counts);
    }
    TEAM_LAUNCH_CHECK("segmean_kernel");
    return TEAM_OK;
}
