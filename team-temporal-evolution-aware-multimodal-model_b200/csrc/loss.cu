// Contrastive losses of the training step, forward + gradient in one call (SURVEY 8f "next" rows):
//   team_unicl_loss : unicl_loss (models/proof.py:21-191, evolution_features = None) - the three-way contrastive
//                     loss on the head outputs; its gradients ARE the cotangents of team_head_tri_bwd
//   team_clip_loss  : ClipLoss.forward (utils/toolkit.py:128-141, world_size 1) on the encode_image / encode_text rows
// The B x B similarity matrices and the two "coefficient x rows" gradient products are grouped tensor-core GEMMs
// (fp32 FFMA GEMMs in TEAM_MODE_F32); the softmax statistics, the per-sample 3 x 3 instance term and the
// normalise-backward are warp-per-row kernels; every batch reduction is a fixed-order fold (deterministic).
#include "head_kernels.cuh"

namespace team {

constexpr int64_t LOSS_MAX_BATCH = 16384;        // the losses are O(B^2) by definition (B x B similarities)

struct LossWS {
    Mat X[3];                 // normalised image / text / state rows [B][D]
    float* inv[3];            // 1 / max(|x|, eps)
    float* sim;               // [B][B]
    float* simT;              // [B][B] (clip only)
    Mat G;                    // [B][B] gradient coefficients
    float* rmax; float* rpos; float* rall; float* rloss;     // [2B]
    float* dcat;              // [B][D]
    float* part;              // [1024] fold scratch
    float* scal;              // [8] device scalars: 0 valid count, 1 category loss, 2 instance sum
    void* gemm_ws; size_t gemm_ws_bytes;
    size_t total;
};

static void loss_plan(int64_t B, void* base, LossWS* w) {
    size_t off = 0;
    auto take = [&](size_t bytes) -> char* {
        char* p = base ? reinterpret_cast<char*>(base) + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    for (int i = 0; i < 3; ++i) {
        w->X[i].f = reinterpret_cast<float*>(take((size_t)B * D * 4));
        w->X[i].h = reinterpret_cast<__nv_bfloat16*>(take((size_t)B * D * 2));
        w->X[i].ld = D;
        w->inv[i] = reinterpret_cast<float*>(take((size_t)B * 4));
    }
    const int64_t Bp = (B + 7) / 8 * 8;                      // leading dimension of the B x B matrices
    w->sim = reinterpret_cast<float*>(take((size_t)B * Bp * 4));
    w->simT = reinterpret_cast<float*>(take((size_t)B * Bp * 4));
    w->G.f = reinterpret_cast<float*>(take((size_t)B * Bp * 4));
    w->G.h = reinterpret_cast<__nv_bfloat16*>(take((size_t)B * Bp * 2));
    w->G.ld = Bp;
    w->rmax = reinterpret_cast<float*>(take((size_t)2 * B * 4));
    w->rpos = reinterpret_cast<float*>(take((size_t)2 * B * 4));
    w->rall = reinterpret_cast<float*>(take((size_t)2 * B * 4));
    w->rloss = reinterpret_cast<float*>(take((size_t)2 * B * 4));
    w->dcat = reinterpret_cast<float*>(take((size_t)B * D * 4));
    w->part = reinterpret_cast<float*>(take(1024 * 4));
    w->scal = reinterpret_cast<float*>(take(8 * 4));
    w->gemm_ws_bytes = 64u << 20;
    w->gemm_ws = take(w->gemm_ws_bytes);
    w->total = off;
}

// ------------------------------------------------------------------ kernels
// rows [0,B): image, [B,2B): text, [2B,3B): state -> normalised copies (+ bf16 shadow) and inverse norms
__global__ void __launch_bounds__(256)
loss_normalize_kernel(int64_t B, const float* __restrict__ x0, const float* __restrict__ x1, const float* __restrict__ x2,
                      float* y0, float* y1, float* y2, __nv_bfloat16* h0, __nv_bfloat16* h1, __nv_bfloat16* h2,
                      float* i0, float* i1, float* i2, int n_sets, int do_normalize) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= (int64_t)n_sets * B) return;
    const int k = (int)(r / B);
    const int64_t b = r - (int64_t)k * B;
    const float* x = (k == 0 ? x0 : k == 1 ? x1 : x2) + b * D;
    float* y = (k == 0 ? y0 : k == 1 ? y1 : y2) + b * D;
    __nv_bfloat16* h = k == 0 ? h0 : k == 1 ? h1 : h2;
    float* iv = k == 0 ? i0 : k == 1 ? i1 : i2;
    float4 v[4];
    ld_row(x, lane, v);
    float s = 1.f;
    if (do_normalize) {
        s = 1.0f / fmaxf(sqrtf(warp_sum(dot_part(v, v))), NORM_EPS);
        scale_row(v, s);
    }
    st_row(y, lane, v);
    st_row_h(h != nullptr ? h + b * D : nullptr, lane, v);
    if (lane == 0 && iv != nullptr) iv[b] = s;
}

// category term, per row i of sim / tau: max over ALL j, pos = sum_{j != i, y_j == y_i} e_j, all = sum_{j != i} e_j.
// Rows are the B samples starting at global row r0, columns the ncols samples of the (global) batch: the diagonal is
// column r0 + i.  Single GPU: r0 = 0, ncols = B.
__global__ void __launch_bounds__(256)
unicl_cat_stats_kernel(int B, int ncols, int r0, int ld, const float* __restrict__ sim, const int64_t* __restrict__ labels,
                       float inv_tau, float* __restrict__ rmax, float* __restrict__ rpos, float* __restrict__ rall,
                       float* __restrict__ rloss, float* __restrict__ rvalid) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= B) return;
    // 128-bit loads, four of them in flight per lane (ld is a multiple of 4; columns >= B are masked): with scalar loads and
    // the compiler's own unrolling the two passes were chains of L2 round trips (16 us at B = 1 024, tools/timeline_train.py)
    const float4* row4 = reinterpret_cast<const float4*>(sim + (size_t)i * ld);
    const longlong2* lab2 = reinterpret_cast<const longlong2*>(labels);
    const int64_t yi = labels[r0 + i];
    const int n4 = (ncols + 3) >> 2;
    float mx = -INFINITY;
#pragma unroll 4
    for (int q = lane; q < n4; q += 32) {
        const float4 v = row4[q];
        const int j = 4 * q;
        mx = fmaxf(mx, v.x * inv_tau);
        if (j + 1 < ncols) mx = fmaxf(mx, v.y * inv_tau);
        if (j + 2 < ncols) mx = fmaxf(mx, v.z * inv_tau);
        if (j + 3 < ncols) mx = fmaxf(mx, v.w * inv_tau);
    }
    mx = warp_max(mx);
    float pos = 0.f, all = 0.f;
#pragma unroll 4
    for (int q = lane; q < n4; q += 32) {
        const float4 v = row4[q];
        const int j = 4 * q;
        long long y[4];
        if (j + 3 < ncols) {
            const longlong2 la = lab2[2 * q], lb = lab2[2 * q + 1];
            y[0] = la.x; y[1] = la.y; y[2] = lb.x; y[3] = lb.y;
        } else {
#pragma unroll
            for (int u = 0; u < 4; ++u) y[u] = j + u < ncols ? labels[j + u] : -1;
        }
        const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (j + u >= ncols || j + u == r0 + i) continue;
            const float e = expf(x[u] * inv_tau - mx);
            all += e;
            if (y[u] == yi) pos += e;
        }
    }
    pos = warp_sum(pos); all = warp_sum(all);
    if (lane == 0) {
        const bool valid = pos > 0.f && all > 0.f;
        rmax[i] = mx; rpos[i] = pos; rall[i] = all;
        rloss[i] = valid ? -logf(pos / (all + 1e-8f)) : 0.f;
        rvalid[i] = valid ? 1.f : 0.f;
    }
}

// single block: fixed-order sums of n values of a and (optionally) b -> out[0], out[1]
__global__ void __launch_bounds__(1024)
loss_fold2_kernel(int n, const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                  int finish = 0, float c = 0.f, const float* __restrict__ scal = nullptr, float* __restrict__ losses = nullptr) {
    pdl_trigger();
    pdl_wait();
    __shared__ float sa[1024], sb[1024];
    float x = 0.f, y = 0.f;
    for (int i = threadIdx.x; i < n; i += 1024) { x += a[i]; if (b != nullptr) y += b[i]; }
    sa[threadIdx.x] = x; sb[threadIdx.x] = y;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { sa[threadIdx.x] += sa[threadIdx.x + o]; sb[threadIdx.x] += sb[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = sa[0]; out[1] = sb[0];
        // the loss value(s) right here instead of in a one-thread kernel of their own (one launch less on the chain):
        if (finish == 1) {                      // ClipLoss: sum of the 2B row losses / 2B
            losses[0] = sa[0] * c;
        } else if (finish == 2) {               // unicl: scal = {valid count, category sum}, this fold = instance sum; c = 1 / 3B
            const float cat = scal[0] > 0.f ? scal[1] / scal[0] : 0.f;
            const float inst = sa[0] * c;
            losses[0] = inst + 0.5f * cat; losses[1] = inst; losses[2] = cat;
        }
    }
}

// G[i][j] = d(0.5 * grad_scale * category_loss) / d(sim_ij)   (scal[0] = valid count); rows r0 + [0, B), ncols columns.
// With column statistics (cmax != null, indexed by column) the kernel also writes the transposed half
// H[i][j] = G[j][r0 + i] (sim is symmetric) into H: dcat of the rows is then G X + H X over all columns, one GEMM of two
// K-segments, and H is rounded to bf16 entry by entry like the single-GPU G^T.
__global__ void __launch_bounds__(256)
unicl_cat_grad_kernel(int B, int ncols, int r0, int ld, const float* __restrict__ sim, const int64_t* __restrict__ labels,
                      float inv_tau, float weight, const float* __restrict__ rmax, const float* __restrict__ rpos,
                      const float* __restrict__ rall, const float* __restrict__ rvalid, const float* __restrict__ cmax,
                      const float* __restrict__ cpos, const float* __restrict__ call, const float* __restrict__ cvalid,
                      const float* __restrict__ scal, float* __restrict__ G, __nv_bfloat16* __restrict__ Gh,
                      float* __restrict__ H, __nv_bfloat16* __restrict__ Hh) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= B) return;
    const float nvalid = scal[0];
    const bool valid = rvalid[i] != 0.f && nvalid > 0.f;
    const float kk = nvalid > 0.f ? weight * inv_tau / nvalid : 0.f;
    const float k = valid ? kk : 0.f;
    const float mx = rmax[i], ip = valid ? 1.0f / rpos[i] : 0.f, ia = valid ? 1.0f / (rall[i] + 1e-8f) : 0.f;
    const int64_t yi = labels[r0 + i];
    const float4* row4 = reinterpret_cast<const float4*>(sim + (size_t)i * ld);
    const longlong2* lab2 = reinterpret_cast<const longlong2*>(labels);
    float4* g4 = reinterpret_cast<float4*>(G + (size_t)i * ld);
    uint2* h4 = Gh != nullptr ? reinterpret_cast<uint2*>(Gh + (size_t)i * ld) : nullptr;
    float4* t4 = H != nullptr ? reinterpret_cast<float4*>(H + (size_t)i * ld) : nullptr;
    uint2* th4 = Hh != nullptr ? reinterpret_cast<uint2*>(Hh + (size_t)i * ld) : nullptr;
#pragma unroll 4
    for (int q = lane; q < ld / 4; q += 32) {
        const int j = 4 * q;
        float g[4] = {0.f, 0.f, 0.f, 0.f}, t[4] = {0.f, 0.f, 0.f, 0.f};
        if ((valid || cmax != nullptr) && j < ncols) {
            const float4 v = row4[q];
            long long y[4];
            if (j + 3 < ncols) {
                const longlong2 la = lab2[2 * q], lb = lab2[2 * q + 1];
                y[0] = la.x; y[1] = la.y; y[2] = lb.x; y[3] = lb.y;
            } else {
#pragma unroll
                for (int u = 0; u < 4; ++u) y[u] = j + u < ncols ? labels[j + u] : -1;
            }
            const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = j + u;
                if (c >= ncols || c == r0 + i) continue;
                if (valid) g[u] = k * expf(x[u] * inv_tau - mx) * (ia - (y[u] == yi ? ip : 0.f));
                if (cmax != nullptr && cvalid[c] != 0.f)
                    t[u] = kk * expf(x[u] * inv_tau - cmax[c]) * (1.0f / (call[c] + 1e-8f) - (y[u] == yi ? 1.0f / cpos[c] : 0.f));
            }
        }
        const float4 o = make_float4(g[0], g[1], g[2], g[3]);
        g4[q] = o;
        if (h4 != nullptr) h4[q] = pack_bf16x4(o);
        if (t4 != nullptr) {
            const float4 ot = make_float4(t[0], t[1], t[2], t[3]);
            t4[q] = ot;
            if (th4 != nullptr) th4[q] = pack_bf16x4(ot);
        }
    }
}

// instance term + assembly of the three cotangents (warp per sample; rloss may be null, g_image null = loss only):
//   3 x 3 similarities of (image, text, state) / tau; row r: pos = 1 + sum_{c != r} e_rc, all = sum_c e_rc,
//   loss -= log(pos / (all + 1e-8));  then d total / d xhat = instance part + dcat (image only), normalise-backward.
__global__ void __launch_bounds__(256)
unicl_instance_kernel(int B, const float* __restrict__ Xi, const float* __restrict__ Xt, const float* __restrict__ Xs,
                      const float* __restrict__ inv_i, const float* __restrict__ inv_t, const float* __restrict__ inv_s,
                      const float* __restrict__ dcat, float inv_tau, float inst_weight, float* __restrict__ g_image,
                      float* __restrict__ g_text, float* __restrict__ g_state, float* __restrict__ rloss,
                      float* __restrict__ d_state_hat) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    float4 v[3][4];
    ld_row(Xi + (size_t)b * D, lane, v[0]);
    ld_row(Xt + (size_t)b * D, lane, v[1]);
    ld_row(Xs + (size_t)b * D, lane, v[2]);
    float s[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = r; c < 3; ++c) {
            const float d = warp_sum(dot_part(v[r], v[c])) * inv_tau;
            s[r][c] = d; s[c][r] = d;
        }
    float loss = 0.f, wgt[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        float e[3], pos = 1.f, all = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) { e[c] = expf(s[r][c]); all += e[c]; if (c != r) pos += e[c]; }
        loss -= logf(pos / (all + 1e-8f));
        const float ia = 1.0f / (all + 1e-8f), ip = 1.0f / pos;
#pragma unroll
        for (int c = 0; c < 3; ++c) wgt[r][c] = c == r ? e[c] * ia : e[c] * (ia - ip);
    }
    if (lane == 0 && rloss != nullptr) rloss[b] = loss;
    if (g_image == nullptr) return;                      // loss only (data-parallel form: the value is exchanged first)
    const float k = inst_weight * inv_tau;
    const float* invs[3] = {inv_i, inv_t, inv_s};
    float* outs[3] = {g_image, g_text, g_state};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        // d/d v_r = sum_{c != r} (w_rc + w_cr) v_c + 2 w_rr v_r
        float4 dv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) dv[i] = mul4s(2.f * k * wgt[r][r], v[r][i]);
#pragma unroll
        for (int c = 0; c < 3; ++c)
            if (c != r) axpy_row(dv, k * (wgt[r][c] + wgt[c][r]), v[c]);
        if (r == 0) {
            float4 t[4];
            ld_row(dcat + (size_t)b * D, lane, t);
            add_row(dv, t);
        }
        if (r == 2 && d_state_hat != nullptr) {      // evolution branch: the state rows went through evo_fwd_kernel first;
            st_row(d_state_hat + (size_t)b * D, lane, dv);   // its backward (evo_bwd*_kernel) finishes g_state
            continue;
        }
        const float proj = warp_sum(dot_part(dv, v[r]));
        const float iv = invs[r][b];
#pragma unroll
        for (int i = 0; i < 4; ++i) dv[i] = mul4s(iv, fma4s(-proj, v[r][i], dv[i]));
        st_row(outs[r] + (size_t)b * D, lane, dv);
    }
}

// ------------------------------------------------------------------ evolution_features branch of unicl_loss
// models/proof.py:51-106 (restated in oracle/team_oracle.py:enhance_state_features).  With s_j the normalised state
// rows, c the class and st the state id of sample i, and `evo_c` the class's evolution feature:
//   class seen once in the batch          : out_i = N(0.8 s_i + 0.2 N(evo_c))
//   class seen >= 2x with >= 2 states     : t(st) = rank of st among the class's states / (n_states - 1),
//                                           w(i,j) = 1 - |t_i - t_j| (only if > 0.3),
//                                           mix_i = evo_c + 0.2 sum_{j != i in class} w(i,j) s_j,  out_i = N(0.7 s_i + 0.3 N(mix_i))
//   otherwise                             : out_i = s_i
// The weights depend on (state_i, state_j) only, so with the keyed sums SS[c][st] = sum_{j in class c, state st} s_j
//   mix_i = evo_c + 0.2 (sum_st w(st_i, st) SS[c][st] - s_i)
// and the backward needs the same keyed sum of dL/dmix: no O(B^2) loops, no host round trips (the reference reads
// every label and state id on the host).  Keyed sums are one CTA per key scanning the batch in index order
// (deterministic).  State ids must lie in [0, 10) (they index the 10-row state embedding).
constexpr int EVO_NS = 10;

// One CTA per key.  Phase 1: all threads test 128 samples at a time and leave one ballot word per warp in shared memory
// (the label / state loads of all chunks are independent); phase 2: every thread walks the set bits in index order and
// adds its float4 column of each matching row - the same deterministic order as a serial scan, without its B dependent
// iterations (the serial form took 64 us per call at B = 1 024: a quarter of the whole training step, tools/timeline_train.py).
__global__ void __launch_bounds__(128)
evo_keysum_kernel(int B, const float* __restrict__ rows, const unsigned char* __restrict__ rowmask,
                  const int64_t* __restrict__ labels, const int64_t* __restrict__ states, int num_evo,
                  const unsigned char* __restrict__ evo_mask, float* __restrict__ out, int* __restrict__ cnt) {
    extern __shared__ unsigned int evo_bits[];               // [ceil(B / 32)]
    pdl_trigger();
    pdl_wait();
    const int key = blockIdx.x, c = key / EVO_NS, st = key - c * EVO_NS;
    const int t = threadIdx.x, lane = t & 31;
    if (!evo_mask[c]) {                  // defined zeros (the data-parallel form exchanges every key)
        reinterpret_cast<float4*>(out + (size_t)key * D)[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (cnt != nullptr && t == 0) cnt[key] = 0;
        return;
    }
    const int nwords = (B + 31) / 32;
#pragma unroll 4
    for (int base = 0; base < nwords * 32; base += 128) {
        const int j = base + t;
        const bool hit = j < B && labels[j] == c && clamp_state(states[j]) == st;
        const unsigned int m = __ballot_sync(0xffffffffu, hit);
        if (lane == 0 && (j >> 5) < nwords) evo_bits[j >> 5] = m;
    }
    __syncthreads();
    // phase 2: the matching rows in index order, four loads in flight (the bit walk itself is register arithmetic; a row
    // load per set bit, one after the other, was a chain of dependent L2 round trips)
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int n = 0, pend = 0;
    int idx[4];
    auto flush = [&]() {
        float4 v[4];
        bool use[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            use[q] = q < pend && (rowmask == nullptr || rowmask[idx[q]] != 0);
            if (use[q]) v[q] = reinterpret_cast<const float4*>(rows + (size_t)idx[q] * D)[t];
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (use[q]) { acc.x += v[q].x; acc.y += v[q].y; acc.z += v[q].z; acc.w += v[q].w; }
        pend = 0;
    };
    for (int w = 0; w < nwords; ++w) {
        unsigned int m = evo_bits[w];
        n += __popc(m);
        while (m) {
            idx[pend++] = w * 32 + __ffs(m) - 1;
            m &= m - 1;
            if (pend == 4) flush();
        }
    }
    if (pend > 0) flush();
    reinterpret_cast<float4*>(out + (size_t)key * D)[t] = acc;
    if (cnt != nullptr && t == 0) cnt[key] = n;
    (void)num_evo;
}

// time weights of sample i's state against the ten states of its class (0 for absent states / weights <= 0.3);
// returns the enhancement mode: 0 = unchanged, 1 = single sample, 2 = temporal mixture
__device__ __forceinline__ int evo_class_weights(const int* __restrict__ cnt_c, int st_i, float (&w)[EVO_NS]) {
    int n = 0, uniq = 0, rank_i = 0;
#pragma unroll
    for (int s = 0; s < EVO_NS; ++s) {
        const int k = cnt_c[s];
        n += k;
        if (k > 0) { if (s < st_i) ++rank_i; ++uniq; }
        w[s] = 0.f;
    }
    if (n <= 1) return 1;
    if (uniq < 2) return 0;
    const float inv = 1.0f / (float)(uniq - 1);
    const float t_i = (float)rank_i * inv;
    int rank = 0;
#pragma unroll
    for (int s = 0; s < EVO_NS; ++s) {
        if (cnt_c[s] <= 0) continue;
        const float ws = 1.0f - fabsf(t_i - (float)rank * inv);
        if (ws > 0.3f) w[s] = ws;
        ++rank;
    }
    return 2;
}

// forward: enhanced rows Xe, normalised mixtures Mh, per-row scalars sc[b] = {mode, 1/|e|, 1/|mix|, -}
__global__ void __launch_bounds__(256)
evo_fwd_kernel(int B, const float* __restrict__ Xs, const int64_t* __restrict__ labels, const int64_t* __restrict__ states,
               int num_evo, const float* __restrict__ evo, const unsigned char* __restrict__ evo_mask,
               const float* __restrict__ SS, const int* __restrict__ cnt, float* __restrict__ Xe, float* __restrict__ Mh,
               float* __restrict__ sc, unsigned char* __restrict__ rowmask) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    float4 s[4];
    ld_row(Xs + (size_t)b * D, lane, s);
    const int64_t c = labels[b];
    int mode = 0;
    float w[EVO_NS];
    const int st_i = clamp_state(states[b]);
    if (c >= 0 && c < num_evo && evo_mask[c]) mode = evo_class_weights(cnt + (size_t)c * EVO_NS, st_i, w);
    float inv_e = 1.f, inv_m = 1.f;
    if (mode != 0) {
        float4 m[4];
        ld_row(evo + (size_t)c * D, lane, m);
        if (mode == 2) {
            axpy_row(m, -0.2f, s);
#pragma unroll
            for (int q = 0; q < EVO_NS; ++q) {
                if (w[q] == 0.f) continue;                 // warp-uniform
                float4 t[4];
                ld_row(SS + ((size_t)c * EVO_NS + q) * D, lane, t);
                axpy_row(m, 0.2f * w[q], t);
            }
        }
        inv_m = 1.0f / fmaxf(sqrtf(warp_sum(dot_part(m, m))), NORM_EPS);
        scale_row(m, inv_m);
        st_row(Mh + (size_t)b * D, lane, m);
        const float ks = mode == 2 ? 0.7f : 0.8f, km = mode == 2 ? 0.3f : 0.2f;
#pragma unroll
        for (int i = 0; i < 4; ++i) s[i] = fma4s(km, m[i], mul4s(ks, s[i]));
        inv_e = 1.0f / fmaxf(sqrtf(warp_sum(dot_part(s, s))), NORM_EPS);
        scale_row(s, inv_e);
    }
    st_row(Xe + (size_t)b * D, lane, s);
    if (lane == 0) {
        sc[(size_t)b * 4] = (float)mode; sc[(size_t)b * 4 + 1] = inv_e; sc[(size_t)b * 4 + 2] = inv_m;
        rowmask[b] = mode == 2 ? 1 : 0;
    }
}

// backward 1: g = dL/dXe (in dXe) -> dXe := direct part of dL/ds, dMix := dL/dmix (rows of mode 2 only)
__global__ void __launch_bounds__(256)
evo_bwd1_kernel(int B, const float* __restrict__ Xe, const float* __restrict__ Mh, const float* __restrict__ sc,
                float* __restrict__ dXe, float* __restrict__ dMix) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    const int mode = (int)sc[(size_t)b * 4];
    if (mode == 0) return;
    const float inv_e = sc[(size_t)b * 4 + 1], inv_m = sc[(size_t)b * 4 + 2];
    float4 g[4], o[4];
    ld_row(dXe + (size_t)b * D, lane, g);
    ld_row(Xe + (size_t)b * D, lane, o);
    const float pg = warp_sum(dot_part(g, o));
#pragma unroll
    for (int i = 0; i < 4; ++i) g[i] = mul4s(inv_e, fma4s(-pg, o[i], g[i]));        // dL/de
    if (mode == 2) {
        float4 m[4], dm[4];
        ld_row(Mh + (size_t)b * D, lane, m);
        const float pm = warp_sum(dot_part(g, m));
#pragma unroll
        for (int i = 0; i < 4; ++i) dm[i] = mul4s(0.3f * inv_m, fma4s(-pm, m[i], g[i]));   // dL/dmix
        st_row(dMix + (size_t)b * D, lane, dm);
#pragma unroll
        for (int i = 0; i < 4; ++i) g[i] = fma4s(-0.2f, dm[i], mul4s(0.7f, g[i]));          // own row is excluded from its mixture
    } else {
        scale_row(g, 0.8f);
    }
    st_row(dXe + (size_t)b * D, lane, g);
}

// backward 2: add the mixture part 0.2 sum_st w(st_j, st) DM[c][st], then the normalise-backward of the raw state rows
__global__ void __launch_bounds__(256)
evo_bwd2_kernel(int B, const float* __restrict__ Xs, const float* __restrict__ inv_s, const int64_t* __restrict__ labels,
                const int64_t* __restrict__ states, const float* __restrict__ sc, const float* __restrict__ DM,
                const int* __restrict__ cnt, const float* __restrict__ dXe, float* __restrict__ g_state) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    float4 d[4], s[4];
    ld_row(dXe + (size_t)b * D, lane, d);
    ld_row(Xs + (size_t)b * D, lane, s);
    if ((int)sc[(size_t)b * 4] == 2) {
        const int64_t c = labels[b];
        float w[EVO_NS];
        evo_class_weights(cnt + (size_t)c * EVO_NS, clamp_state(states[b]), w);
#pragma unroll
        for (int q = 0; q < EVO_NS; ++q) {
            if (w[q] == 0.f) continue;
            float4 t[4];
            ld_row(DM + ((size_t)c * EVO_NS + q) * D, lane, t);
            axpy_row(d, 0.2f * w[q], t);
        }
    }
    const float proj = warp_sum(dot_part(d, s));
    const float iv = inv_s[b];
#pragma unroll
    for (int i = 0; i < 4; ++i) d[i] = mul4s(iv, fma4s(-proj, s[i], d[i]));
    st_row(g_state + (size_t)b * D, lane, d);
}

// ---- ClipLoss: per row of s * L (rows [0,B): image->text from L, rows [B,2B): text->image from L^T): lse and loss.
// The rows are the samples r0 + [0, B) against ncols columns (single GPU: r0 = 0, ncols = B).
__global__ void __launch_bounds__(256)
clip_stats_kernel(int B, int ncols, int r0, int ld, const float* __restrict__ L, const float* __restrict__ LT, float scale,
                  float* __restrict__ lse, float* __restrict__ rloss) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= 2 * B) return;
    const int i = r < B ? r : r - B;
    const float* row = (r < B ? L : LT) + (size_t)i * ld;
    const float4* row4 = reinterpret_cast<const float4*>(row);
    const int n4 = (ncols + 3) >> 2;
    float mx = -INFINITY;
#pragma unroll 4
    for (int q = lane; q < n4; q += 32) {
        const float4 v = row4[q];
        const int j = 4 * q;
        mx = fmaxf(mx, v.x * scale);
        if (j + 1 < ncols) mx = fmaxf(mx, v.y * scale);
        if (j + 2 < ncols) mx = fmaxf(mx, v.z * scale);
        if (j + 3 < ncols) mx = fmaxf(mx, v.w * scale);
    }
    mx = warp_max(mx);
    float z = 0.f;
#pragma unroll 4
    for (int q = lane; q < n4; q += 32) {
        const float4 v = row4[q];
        const int j = 4 * q;
        z += expf(v.x * scale - mx);
        if (j + 1 < ncols) z += expf(v.y * scale - mx);
        if (j + 2 < ncols) z += expf(v.z * scale - mx);
        if (j + 3 < ncols) z += expf(v.w * scale - mx);
    }
    z = warp_sum(z);
    if (lane == 0) {
        const float l = logf(z) + mx;
        lse[r] = l;
        rloss[r] = l - row[r0 + i] * scale;
    }
}
// G[i][j] = d(grad_scale * loss) / d(L_ij) = k * (softmax_i2t[i][j] + softmax_t2i[j][i] - 2 delta_ij),  k = scale*grad_scale/(2B)
// lse_row: the logsumexps of the B rows (row r0 + i of the global L), lse_col: those of the ncols columns' other direction.
// Fed L^T's rows with the two vectors swapped it gives the rows of G^T (data-parallel form).
__global__ void __launch_bounds__(256)
clip_grad_kernel(int B, int ncols, int r0, int ld, const float* __restrict__ L, float scale, float k,
                 const float* __restrict__ lse_row, const float* __restrict__ lse_col, float* __restrict__ G,
                 __nv_bfloat16* __restrict__ Gh) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= B) return;
    const float li = lse_row[i];
    const float4* row4 = reinterpret_cast<const float4*>(L + (size_t)i * ld);
    float4* g4 = reinterpret_cast<float4*>(G + (size_t)i * ld);
    uint2* h4 = Gh != nullptr ? reinterpret_cast<uint2*>(Gh + (size_t)i * ld) : nullptr;
#pragma unroll 4
    for (int q = lane; q < ld / 4; q += 32) {
        const int j = 4 * q;
        float g[4] = {0.f, 0.f, 0.f, 0.f};
        if (j < ncols) {
            const float4 v = row4[q];
            const float x[4] = {v.x * scale, v.y * scale, v.z * scale, v.w * scale};
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (j + u < ncols) g[u] = k * (expf(x[u] - li) + expf(x[u] - lse_col[j + u]) - (j + u == r0 + i ? 2.f : 0.f));
        }
        const float4 o = make_float4(g[0], g[1], g[2], g[3]);
        g4[q] = o;
        if (h4 != nullptr) h4[q] = pack_bf16x4(o);
    }
}
static int loss_setup(LossWS& w, int64_t batch, void* workspace, size_t workspace_bytes, const char* who) {
    TEAM_REQUIRE(batch >= 1 && batch <= LOSS_MAX_BATCH, "%s: batch %lld out of [1, %lld]", who, (long long)batch, (long long)LOSS_MAX_BATCH);
    loss_plan(batch, workspace, &w);
    if (workspace == nullptr || workspace_bytes < w.total) {
        set_error("%s: workspace %zu < %zu bytes", who, workspace_bytes, w.total);
        return TEAM_EWORKSPACE;
    }
    TEAM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "%s: workspace must be 256-byte aligned", who);
    return TEAM_OK;
}

}  // namespace team

using namespace team;

extern "C" size_t team_loss_workspace_bytes(int64_t batch) {
    if (batch < 1 || batch > LOSS_MAX_BATCH) return 0;
    LossWS w;
    loss_plan(batch, nullptr, &w);
    return w.total;
}

struct EvoArgs {
    const int64_t* state_ids;
    const float* evo;                 // [num_evo][D]
    const unsigned char* evo_mask;    // [num_evo]
    int num_evo;
};
static size_t evo_plan(int64_t B, int num_evo, char* base, float** Xe, float** Mh, float** dXe, float** dMix, float** SS,
                       float** DM, int** cnt, float** sc, unsigned char** rowmask) {
    size_t off = 0;
    auto take = [&](size_t bytes) -> char* { char* p = base ? base + off : nullptr; off += align_up(bytes, 256); return p; };
    const size_t keys = (size_t)num_evo * EVO_NS;
    *Xe = reinterpret_cast<float*>(take((size_t)B * D * 4)); *Mh = reinterpret_cast<float*>(take((size_t)B * D * 4));
    *dXe = reinterpret_cast<float*>(take((size_t)B * D * 4)); *dMix = reinterpret_cast<float*>(take((size_t)B * D * 4));
    *SS = reinterpret_cast<float*>(take(keys * D * 4)); *DM = reinterpret_cast<float*>(take(keys * D * 4));
    *cnt = reinterpret_cast<int*>(take(keys * 4)); *sc = reinterpret_cast<float*>(take((size_t)B * 16));
    *rowmask = reinterpret_cast<unsigned char*>(take((size_t)B));
    return off;
}

static int unicl_impl(int mode, const float* image, const float* text, const float* state, const int64_t* labels,
                      const EvoArgs* ev, int64_t batch, float temperature, float grad_scale, float* losses, float* g_image,
                      float* g_text, float* g_state, void* workspace, size_t workspace_bytes, void* stream) {
    TEAM_REQUIRE(mode == TEAM_MODE_F32 || mode == TEAM_MODE_BF16, "unicl_loss: bad mode %d", mode);
    TEAM_REQUIRE(image && text && state && labels && losses && g_image && g_text && g_state, "unicl_loss: null pointer");
    TEAM_REQUIRE(temperature > 0.f, "unicl_loss: temperature must be positive");
    LossWS w;
    int rc = loss_setup(w, batch, workspace, workspace_bytes, "unicl_loss");
    if (rc) return rc;
    float *Xe = nullptr, *Mh = nullptr, *dXe = nullptr, *dMix = nullptr, *SS = nullptr, *DM = nullptr, *sc = nullptr;
    int* cnt = nullptr;
    unsigned char* rowmask = nullptr;
    if (ev != nullptr) {
        TEAM_REQUIRE(ev->state_ids && ev->evo && ev->evo_mask && ev->num_evo >= 1 && ev->num_evo <= 4096, "unicl_loss: bad evolution arguments");
        const size_t extra = evo_plan(batch, ev->num_evo, reinterpret_cast<char*>(workspace) + w.total, &Xe, &Mh, &dXe, &dMix, &SS, &DM, &cnt, &sc, &rowmask);
        if (workspace_bytes < w.total + extra) {
            set_error("unicl_loss: workspace %zu < %zu bytes", workspace_bytes, w.total + extra);
            return TEAM_EWORKSPACE;
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int B = (int)batch, ld = (int)w.G.ld;
    const bool bf = mode == TEAM_MODE_BF16;
    const float inv_tau = 1.0f / temperature;
    TEAM_LAUNCH(loss_normalize_kernel, (3 * B + 7) / 8, 256, 0, st, batch, image, text, state, w.X[0].f, w.X[1].f, w.X[2].f,
                bf ? w.X[0].h : nullptr, (__nv_bfloat16*)nullptr, (__nv_bfloat16*)nullptr, w.inv[0], w.inv[1], w.inv[2], 3, 1);
    if (ev != nullptr) {          // enhanced state rows (models/proof.py:51-106) replace the normalised ones in the instance term
        const int keys = ev->num_evo * EVO_NS;
        TEAM_LAUNCH(evo_keysum_kernel, keys, 128, (size_t)((B + 31) / 32) * sizeof(unsigned int), st, B, w.X[2].f, (const unsigned char*)nullptr, labels, ev->state_ids, ev->num_evo, ev->evo_mask, SS, cnt);
        TEAM_LAUNCH(evo_fwd_kernel, (B + 7) / 8, 256, 0, st, B, w.X[2].f, labels, ev->state_ids, ev->num_evo, ev->evo, ev->evo_mask, SS, cnt, Xe, Mh, sc, rowmask);
    }
    {   // sim = Xi Xi^T
        Wave wv;
        seg(wv.add(B, B, 0.f, Mat{w.sim, nullptr, ld}), false, w.X[0], false, w.X[0], D);
        if ((rc = run_wave(st, mode, wv, w.gemm_ws, w.gemm_ws_bytes))) return rc;
    }
    TEAM_LAUNCH(unicl_cat_stats_kernel, (B + 7) / 8, 256, 0, st, B, B, 0, ld, w.sim, labels, inv_tau, w.rmax, w.rpos, w.rall, w.rloss, w.rmax + B);
    TEAM_LAUNCH(loss_fold2_kernel, 1, 1024, 0, st, B, w.rmax + B, w.rloss, w.scal, 0, 0.f, (const float*)nullptr, (float*)nullptr);   // valid count, category sum
    TEAM_LAUNCH(unicl_cat_grad_kernel, (B + 7) / 8, 256, 0, st, B, B, 0, ld, w.sim, labels, inv_tau, 0.5f * grad_scale, w.rmax, w.rpos, w.rall, w.rmax + B,
                (const float*)nullptr, (const float*)nullptr, (const float*)nullptr, (const float*)nullptr, w.scal, w.G.f, bf ? w.G.h : nullptr,
                (float*)nullptr, (__nv_bfloat16*)nullptr);
    {   // dcat = G Xi + G^T Xi
        Wave wv;
        seg(seg(wv.add(B, D, 0.f, Mat{w.dcat, nullptr, D}), false, w.G, true, w.X[0], B), true, w.G, true, w.X[0], B);
        if ((rc = run_wave(st, mode, wv, w.gemm_ws, w.gemm_ws_bytes))) return rc;
    }
    TEAM_LAUNCH(unicl_instance_kernel, (B + 7) / 8, 256, 0, st, B, w.X[0].f, w.X[1].f, ev != nullptr ? Xe : w.X[2].f, w.inv[0], w.inv[1], w.inv[2], w.dcat, inv_tau, grad_scale / (3.0f * (float)B), g_image, g_text, g_state, w.rloss + B, dXe);
    if (ev != nullptr) {
        const int keys = ev->num_evo * EVO_NS;
        TEAM_LAUNCH(evo_bwd1_kernel, (B + 7) / 8, 256, 0, st, B, Xe, Mh, sc, dXe, dMix);
        TEAM_LAUNCH(evo_keysum_kernel, keys, 128, (size_t)((B + 31) / 32) * sizeof(unsigned int), st, B, dMix, rowmask, labels, ev->state_ids, ev->num_evo, ev->evo_mask, DM, (int*)nullptr);
        TEAM_LAUNCH(evo_bwd2_kernel, (B + 7) / 8, 256, 0, st, B, w.X[2].f, w.inv[2], labels, ev->state_ids, sc, DM, cnt, dXe, g_state);
    }
    TEAM_LAUNCH(loss_fold2_kernel, 1, 1024, 0, st, B, w.rloss + B, (const float*)nullptr, w.scal + 2, 2, 1.0f / (3.0f * (float)B), w.scal, losses);
    return TEAM_OK;
}

extern "C" int team_unicl_loss(int mode, const float* image, const float* text, const float* state, const int64_t* labels,
                               int64_t batch, float temperature, float grad_scale, float* losses, float* g_image,
                               float* g_text, float* g_state, void* workspace, size_t workspace_bytes, void* stream) {
    return unicl_impl(mode, image, text, state, labels, nullptr, batch, temperature, grad_scale, losses, g_image, g_text,
                      g_state, workspace, workspace_bytes, stream);
}

// ---- cross-entropy VALUE of the classification logits (models/proof.py:417: the logits are computed under no_grad, so the
// term carries no gradient) and the learner's total (:442), in one launch: losses6 = [total, ce, clip, unicl, unicl
// instance, unicl category]; entries 2..5 must already hold the ClipLoss / unicl_loss values (their `losses` outputs).
// One CTA, rows strided over the threads, block fold in a fixed order (deterministic).
__global__ void __launch_bounds__(1024)
ce_total_kernel(int B, int C, const float* __restrict__ logits, const int64_t* __restrict__ labels, float w_clip, float w_unicl,
                float* __restrict__ losses6, float* __restrict__ partial) {
    __shared__ float part[1024];
    pdl_trigger();
    pdl_wait();
    float s = 0.f;
    for (int b = threadIdx.x; b < B; b += 1024) {
        const float* r = logits + (size_t)b * C;
        float m = -INFINITY;
        for (int c = 0; c < C; ++c) m = fmaxf(m, r[c]);
        float z = 0.f;
        for (int c = 0; c < C; ++c) z += expf(r[c] - m);
        const int64_t y = labels[b];
        s += (m + logf(z)) - ((y >= 0 && y < C) ? r[y] : 0.f);
    }
    part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0 && partial != nullptr) {      // data-parallel form: the shard's sum; mean and total after the exchange
        partial[0] = part[0];
    } else if (threadIdx.x == 0) {
        const float ce = part[0] / (float)B;
        losses6[1] = ce;
        losses6[0] = ce + w_clip * losses6[2] + w_unicl * losses6[3];
    }
}

extern "C" int team_ce_total(const float* logits, const int64_t* labels, int64_t batch, int64_t num_classes, float w_clip,
                             float w_unicl, float* losses6, void* stream) {
    TEAM_REQUIRE(logits && labels && losses6 && batch >= 1 && batch < (1ll << 31) && num_classes >= 1 && num_classes < (1 << 20),
                 "ce_total: bad arguments");
    TEAM_LAUNCH(ce_total_kernel, 1, 1024, 0, (cudaStream_t)stream, (int)batch, (int)num_classes, logits, labels, w_clip, w_unicl, losses6, (float*)nullptr);
    return TEAM_OK;
}

extern "C" size_t team_loss_evo_workspace_bytes(int64_t batch, int num_evo) {
    if (batch < 1 || batch > LOSS_MAX_BATCH || num_evo < 1 || num_evo > 4096) return 0;
    LossWS w;
    loss_plan(batch, nullptr, &w);
    float *a, *b, *c, *d, *e, *f, *g; int* n; unsigned char* m;
    return w.total + evo_plan(batch, num_evo, nullptr, &a, &b, &c, &d, &e, &f, &n, &g, &m);
}

extern "C" int team_unicl_loss_evo(int mode, const float* image, const float* text, const float* state, const int64_t* labels,
                                   const int64_t* state_ids, const float* evo, const unsigned char* evo_mask, int num_evo,
                                   int64_t batch, float temperature, float grad_scale, float* losses, float* g_image,
                                   float* g_text, float* g_state, void* workspace, size_t workspace_bytes, void* stream) {
    EvoArgs ev{state_ids, evo, evo_mask, num_evo};
    return unicl_impl(mode, image, text, state, labels, &ev, batch, temperature, grad_scale, losses, g_image, g_text,
                      g_state, workspace, workspace_bytes, stream);
}

extern "C" int team_clip_loss(int mode, const float* image, const float* text, int64_t batch, float logit_scale,
                              float grad_scale, float* loss, float* g_image, float* g_text, void* workspace,
                              size_t workspace_bytes, void* stream) {
    TEAM_REQUIRE(mode == TEAM_MODE_F32 || mode == TEAM_MODE_BF16, "clip_loss: bad mode %d", mode);
    TEAM_REQUIRE(image && text && loss && g_image && g_text, "clip_loss: null pointer");
    LossWS w;
    int rc = loss_setup(w, batch, workspace, workspace_bytes, "clip_loss");
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int B = (int)batch, ld = (int)w.G.ld;
    const bool bf = mode == TEAM_MODE_BF16;
    // staged copies (bf16 shadows for the tensor-core path); ClipLoss does not normalise (the caller did)
    TEAM_LAUNCH(loss_normalize_kernel, (2 * B + 7) / 8, 256, 0, st, batch, image, text, (const float*)nullptr, w.X[0].f, w.X[1].f, (float*)nullptr,
                bf ? w.X[0].h : nullptr, bf ? w.X[1].h : nullptr, (__nv_bfloat16*)nullptr, (float*)nullptr, (float*)nullptr, (float*)nullptr, 2, 0);
    Wave wv;       // one product per wave: a wave of two would plan its split-K, and so its summation order, as a group
    seg(wv.add(B, B, 0.f, Mat{w.sim, nullptr, ld}), false, w.X[0], false, w.X[1], D);               // L = I T^T
    if ((rc = run_wave(st, mode, wv, w.gemm_ws, w.gemm_ws_bytes))) return rc;
    seg(wv.add(B, B, 0.f, Mat{w.simT, nullptr, ld}), false, w.X[1], false, w.X[0], D);              // L^T = T I^T
    if ((rc = run_wave(st, mode, wv, w.gemm_ws, w.gemm_ws_bytes))) return rc;
    TEAM_LAUNCH(clip_stats_kernel, (2 * B + 7) / 8, 256, 0, st, B, B, 0, ld, w.sim, w.simT, logit_scale, w.rmax, w.rloss);
    TEAM_LAUNCH(loss_fold2_kernel, 1, 1024, 0, st, 2 * B, w.rloss, (const float*)nullptr, w.scal, 1, 1.0f / (2.0f * (float)B), (const float*)nullptr, loss);
    TEAM_LAUNCH(clip_grad_kernel, (B + 7) / 8, 256, 0, st, B, B, 0, ld, w.sim, logit_scale, logit_scale * grad_scale / (2.0f * (float)B), w.rmax, w.rmax + B, w.G.f, bf ? w.G.h : nullptr);
    seg(wv.add(B, D, 0.f, Mat{g_image, nullptr, D}), false, w.G, true, w.X[1], B);                  // dI = G T
    if ((rc = run_wave(st, mode, wv, w.gemm_ws, w.gemm_ws_bytes))) return rc;
    seg(wv.add(B, D, 0.f, Mat{g_text, nullptr, D}), true, w.G, true, w.X[0], B);                    // dT = G^T I
    if ((rc = run_wave(st, mode, wv, w.gemm_ws, w.gemm_ws_bytes))) return rc;
    return TEAM_OK;
}

// ------------------------------------------------------------------ data-parallel form (team_loss_shard_*)
// Rank r owns the global rows r0 + [0, B), r0 = r B.  The similarity blocks are B x Bg (own rows against every column)
// and the kernels above run on them with (r0, ncols = Bg); the exchanges only move slices, every sum over ranks is a
// rank-order fold in the next phase.  See include/team_b200.h for the phases and the exchanges.
namespace team {

constexpr int64_t SHARD_MAX_GLOBAL = 65536;
constexpr int SHARD_MAX_WORLD = 64;

// exchange 0 row: [normalised image | own image | own text | label (int64), 0 (int64)] in the GEMM operand format
static int64_t shard_row_ld(int mode) { return 3 * D + (mode == TEAM_MODE_BF16 ? 8 : 4); }
static int shard_elem(int mode) { return mode == TEAM_MODE_BF16 ? 2 : 4; }

// float offsets inside one rank's slice of exchanges 1 and 2
struct ShardX {
    int64_t keys;
    int64_t x1_scal, x1_ss, x1_cnt;       // exchange 1: columns [6][B] at 0 (lse i2t, lse t2i, max, pos, all, valid)
    int64_t x2_scal;                      // exchange 2: DM [keys][D] at 0
    size_t bytes[3];
};
// scalar slots of an exchange: 0 valid count, 1 category sum, 2 clip sum, 4 ce sum, 5 instance sum (3, 6, 7: zero)
static void shard_xplan(int mode, int64_t B, int num_evo, ShardX* x) {
    const int64_t a = 64;                             // 256 bytes in floats
    auto up = [&](int64_t n) { return (n + a - 1) / a * a; };
    x->keys = (int64_t)num_evo * EVO_NS;
    x->bytes[0] = (size_t)(B * shard_row_ld(mode) * shard_elem(mode));     // no padding: the gathered rows are one matrix
    x->x1_scal = up(6 * B);
    int64_t n1 = x->x1_scal + a;
    x->x1_ss = n1;
    x->x1_cnt = num_evo ? x->x1_ss + up(x->keys * D) : n1;
    if (num_evo) n1 = x->x1_cnt + up(x->keys);
    x->bytes[1] = (size_t)n1 * 4;
    x->x2_scal = up(x->keys * D);
    x->bytes[2] = num_evo ? (size_t)(x->x2_scal + a) * 4 : 0;
}

struct ShardWS {
    float* X[3]; float* inv[3];
    int64_t* labels_g;        // [Bg]
    Mat S[3];                 // [B][Bgp] fp32: 0 unicl X_loc X_g^T, 1 ClipLoss I_loc T_g^T, 2 T_loc I_g^T
    Mat G[4];                 // [B][Bgp] coefficients (+ bf16 shadow in BF16 mode): 0 unicl G, 1 ClipLoss G, 2 G^T, 3 unicl H
    float* rloss;             // [3B]: ClipLoss rows [2B], unicl category rows [B]
    float* rinst;             // [B]
    float* cols;              // [6][Bg] gathered per-row statistics, column-contiguous
    float* scal;              // [8] global sums (slots as in the exchange)
    float* dcat;              // [B][D]
    void* gemm_ws; size_t gemm_ws_bytes;
    float *Xe, *Mh, *dXe, *dMix, *SS, *DM, *sc; int* cnt; unsigned char* rowmask;
    size_t total;
};
static void shard_plan(int mode, int64_t B, int world, int num_evo, void* base, ShardWS* w) {
    size_t off = 0;
    auto take = [&](size_t bytes) -> char* {
        char* p = base ? reinterpret_cast<char*>(base) + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    const int64_t Bg = B * world, Bgp = (Bg + 7) / 8 * 8;
    for (int i = 0; i < 3; ++i) {
        w->X[i] = reinterpret_cast<float*>(take((size_t)B * D * 4));
        w->inv[i] = reinterpret_cast<float*>(take((size_t)B * 4));
    }
    w->labels_g = reinterpret_cast<int64_t*>(take((size_t)Bg * 8));
    for (int i = 0; i < 3; ++i) w->S[i] = Mat{reinterpret_cast<float*>(take((size_t)B * Bgp * 4)), nullptr, Bgp};
    for (int i = 0; i < 4; ++i) {
        w->G[i].f = reinterpret_cast<float*>(take((size_t)B * Bgp * 4));
        w->G[i].h = mode == TEAM_MODE_BF16 ? reinterpret_cast<__nv_bfloat16*>(take((size_t)B * Bgp * 2)) : nullptr;
        w->G[i].ld = Bgp;
    }
    w->rloss = reinterpret_cast<float*>(take((size_t)3 * B * 4));
    w->rinst = reinterpret_cast<float*>(take((size_t)B * 4));
    w->cols = reinterpret_cast<float*>(take((size_t)6 * Bg * 4));
    w->scal = reinterpret_cast<float*>(take(8 * 4));
    w->dcat = reinterpret_cast<float*>(take((size_t)B * D * 4));
    w->gemm_ws_bytes = 64u << 20;
    w->gemm_ws = take(w->gemm_ws_bytes);
    w->Xe = w->Mh = w->dXe = w->dMix = w->SS = w->DM = w->sc = nullptr;
    w->cnt = nullptr; w->rowmask = nullptr;
    if (num_evo) off += evo_plan(B, num_evo, base ? reinterpret_cast<char*>(base) + off : nullptr, &w->Xe, &w->Mh, &w->dXe,
                                 &w->dMix, &w->SS, &w->DM, &w->cnt, &w->sc, &w->rowmask);
    w->total = off;
}

// exchange 0 rows of this rank (warp per row segment: image xhat, own image, own text)
__global__ void __launch_bounds__(256)
shard_pack_rows_kernel(int B, const float* __restrict__ Xi, const float* __restrict__ own, const int64_t* __restrict__ labels,
                       int bf, int64_t ld, void* __restrict__ rows) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= 3 * B) return;
    const int k = r / B, b = r - k * B;
    float4 v[4];
    ld_row(k == 0 ? Xi + (size_t)b * D : own + ((size_t)(k - 1) * B + b) * D, lane, v);
    char* row = reinterpret_cast<char*>(rows) + (size_t)b * ld * (bf ? 2 : 4);
    if (bf) st_row_h(reinterpret_cast<__nv_bfloat16*>(row) + k * D, lane, v);
    else st_row(reinterpret_cast<float*>(row) + k * D, lane, v);
    if (k == 0 && lane == 0) {
        int64_t* meta = reinterpret_cast<int64_t*>(row + (size_t)3 * D * (bf ? 2 : 4));
        meta[0] = labels[b]; meta[1] = 0;
    }
}

__global__ void __launch_bounds__(256)
shard_labels_kernel(int Bg, const void* __restrict__ rows, int64_t row_bytes, int64_t meta_off, int64_t* __restrict__ labels) {
    pdl_trigger();
    pdl_wait();
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j < Bg) labels[j] = *reinterpret_cast<const int64_t*>(reinterpret_cast<const char*>(rows) + (size_t)j * row_bytes + meta_off);
}

// gathered per-row vectors [world][nvec][B] (+ slice stride) -> [nvec][Bg], column j = rank * B + i
__global__ void __launch_bounds__(256)
shard_cols_kernel(int B, int Bg, int nvec, const float* __restrict__ g, int64_t slice, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= (int64_t)nvec * Bg) return;
    const int v = (int)(e / Bg), j = (int)(e - (int64_t)v * Bg), w = j / B, i = j - w * B;
    out[e] = g[(size_t)w * slice + (size_t)v * B + i];
}

// out[e] = sum over ranks of g[w * slice + e], in rank order
template <typename T>
__global__ void __launch_bounds__(256)
shard_sum_kernel(int world, int64_t n, const T* __restrict__ g, int64_t slice, T* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= n) return;
    T s = g[e];
    for (int w = 1; w < world; ++w) s += g[(size_t)w * slice + e];
    out[e] = s;
}

// global sums of the scalar slots (exchange 1; the instance sum from exchange 2 when given) and, when losses6 is given,
// the six loss values
__global__ void __launch_bounds__(32)
shard_losses_kernel(int world, const float* __restrict__ g1, int64_t slice1, const float* __restrict__ g2, int64_t slice2,
                    int64_t Bg, float w_clip, float w_unicl, float* __restrict__ scal, float* __restrict__ losses6) {
    pdl_trigger();
    pdl_wait();
    if (threadIdx.x != 0) return;
    float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int w = 0; w < world; ++w)
        for (int s = 0; s < 6; ++s) v[s] += g1[(size_t)w * slice1 + s];
    if (g2 != nullptr) {
        v[5] = 0.f;
        for (int w = 0; w < world; ++w) v[5] += g2[(size_t)w * slice2 + 5];
    }
    for (int s = 0; s < 6; ++s) scal[s] = v[s];
    if (losses6 == nullptr) return;
    const float n = (float)Bg;
    const float cat = v[0] > 0.f ? v[1] / v[0] : 0.f, inst = v[5] / (3.0f * n), clip = v[2] / (2.0f * n), ce = v[4] / n;
    const float unicl = inst + 0.5f * cat;
    losses6[0] = ce + w_clip * clip + w_unicl * unicl;
    losses6[1] = ce; losses6[2] = clip; losses6[3] = unicl; losses6[4] = inst; losses6[5] = cat;
}

static int shard_check(int32_t phase, const team_loss_shard* s, ShardWS& w, ShardX& x) {
    TEAM_REQUIRE(s != nullptr, "loss_shard: null struct");
    TEAM_REQUIRE(s->mode == TEAM_MODE_F32 || s->mode == TEAM_MODE_BF16, "loss_shard: bad mode %d", s->mode);
    TEAM_REQUIRE(s->world >= 1 && s->world <= SHARD_MAX_WORLD && s->rank >= 0 && s->rank < s->world,
                 "loss_shard: rank %d / world %d", s->rank, s->world);
    const int64_t Bg = s->batch * s->world;
    TEAM_REQUIRE(s->batch >= 1 && s->batch <= LOSS_MAX_BATCH && Bg >= 2 && Bg <= SHARD_MAX_GLOBAL,
                 "loss_shard: batch %lld x world %d out of range (batch <= %lld, 2 <= global batch <= %lld)",
                 (long long)s->batch, s->world, (long long)LOSS_MAX_BATCH, (long long)SHARD_MAX_GLOBAL);
    TEAM_REQUIRE(s->num_evo >= 0 && s->num_evo <= 4096, "loss_shard: num_evo %d", s->num_evo);
    TEAM_REQUIRE(s->num_classes >= 1 && s->num_classes < (1 << 20), "loss_shard: num_classes %lld", (long long)s->num_classes);
    TEAM_REQUIRE(s->temperature > 0.f, "loss_shard: temperature must be positive");
    const int P = s->num_evo ? 4 : 3;
    TEAM_REQUIRE(phase >= 0 && phase < P, "loss_shard: phase %d of %d", phase, P);
    TEAM_REQUIRE(s->image && s->text && s->state && s->own_rows && s->logits && s->labels && s->g_image && s->g_text &&
                 s->g_state && s->g_own_rows && s->losses6, "loss_shard: null pointer");
    TEAM_REQUIRE(!s->num_evo || (s->state_ids && s->evo && s->evo_mask), "loss_shard: null evolution pointer");
    for (int p = 0; p < P - 1; ++p) {
        if (phase == p) TEAM_REQUIRE(s->send[p] && (reinterpret_cast<uintptr_t>(s->send[p]) & 15) == 0, "loss_shard: send[%d] null or not 16-byte aligned", p);
        if (phase > p) TEAM_REQUIRE(s->gathered[p] && (reinterpret_cast<uintptr_t>(s->gathered[p]) & 15) == 0, "loss_shard: gathered[%d] null or not 16-byte aligned", p);
    }
    shard_plan(s->mode, s->batch, s->world, s->num_evo, s->workspace, &w);
    if (s->workspace == nullptr || s->workspace_bytes < w.total) {
        set_error("loss_shard: workspace %zu < %zu bytes", s->workspace_bytes, w.total);
        return TEAM_EWORKSPACE;
    }
    TEAM_REQUIRE((reinterpret_cast<uintptr_t>(s->workspace) & 255) == 0, "loss_shard: workspace must be 256-byte aligned");
    shard_xplan(s->mode, s->batch, s->num_evo, &x);
    return TEAM_OK;
}

}  // namespace team

extern "C" int team_loss_shard_phases(int32_t num_evo) { return num_evo > 0 ? 4 : 3; }

extern "C" size_t team_loss_shard_workspace_bytes(int32_t mode, int64_t batch, int32_t world, int32_t num_evo) {
    if ((mode != TEAM_MODE_F32 && mode != TEAM_MODE_BF16) || batch < 1 || batch > LOSS_MAX_BATCH || world < 1 ||
        world > SHARD_MAX_WORLD || batch * world < 2 || batch * world > SHARD_MAX_GLOBAL || num_evo < 0 || num_evo > 4096)
        return 0;
    ShardWS w;
    shard_plan(mode, batch, world, num_evo, nullptr, &w);
    return w.total;
}

extern "C" size_t team_loss_shard_xchg_bytes(int32_t mode, int64_t batch, int32_t num_evo, int32_t exchange) {
    if ((mode != TEAM_MODE_F32 && mode != TEAM_MODE_BF16) || batch < 1 || batch > LOSS_MAX_BATCH || num_evo < 0 ||
        num_evo > 4096 || exchange < 0 || exchange > 2)
        return 0;
    ShardX x;
    shard_xplan(mode, batch, num_evo, &x);
    return x.bytes[exchange];
}

extern "C" int team_loss_shard_run(int32_t phase, const team_loss_shard* s, void* stream) {
    ShardWS w;
    ShardX x;
    int rc = shard_check(phase, s, w, x);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int mode = s->mode, B = (int)s->batch, W = s->world, Bg = B * W, r0 = s->rank * B, ld = (int)w.S[0].ld;
    const bool bf = mode == TEAM_MODE_BF16, evo = s->num_evo > 0;
    const int keys = s->num_evo * EVO_NS;
    const float inv_tau = 1.0f / s->temperature;
    const int64_t rld = shard_row_ld(mode);
    // the gathered rows as GEMM operands: X_g (normalised image rows), I_g, T_g (own rows), [Bg][rld]
    auto rows = [&](int k) {
        char* p = const_cast<char*>(reinterpret_cast<const char*>(s->gathered[0])) + (size_t)k * D * shard_elem(mode);
        return bf ? Mat{nullptr, reinterpret_cast<__nv_bfloat16*>(p), rld} : Mat{reinterpret_cast<float*>(p), nullptr, rld};
    };
    const int64_t slice1 = (int64_t)(x.bytes[1] / 4), slice2 = (int64_t)(x.bytes[2] / 4);
    const float* g1 = reinterpret_cast<const float*>(s->gathered[1]);
    if (phase == 0) {
        TEAM_LAUNCH(loss_normalize_kernel, (3 * B + 7) / 8, 256, 0, st, s->batch, s->image, s->text, s->state, w.X[0], w.X[1], w.X[2],
                    (__nv_bfloat16*)nullptr, (__nv_bfloat16*)nullptr, (__nv_bfloat16*)nullptr, w.inv[0], w.inv[1], w.inv[2], 3, 1);
        TEAM_LAUNCH(shard_pack_rows_kernel, (3 * B + 7) / 8, 256, 0, st, B, (const float*)w.X[0], s->own_rows, s->labels, bf ? 1 : 0, rld, s->send[0]);
    } else if (phase == 1) {
        TEAM_LAUNCH(shard_labels_kernel, (Bg + 255) / 256, 256, 0, st, Bg, s->gathered[0], rld * shard_elem(mode),
                    (int64_t)3 * D * shard_elem(mode), w.labels_g);
        const Mat Xg = rows(0), Ig = rows(1), Tg = rows(2);
        Wave wv;
        seg(wv.add(B, Bg, 0.f, w.S[0]), false, sub(Xg, r0, 0), false, Xg, D);        // X_loc X_g^T
        seg(wv.add(B, Bg, 0.f, w.S[1]), false, sub(Ig, r0, 0), false, Tg, D);        // I_loc T_g^T: rows of L
        seg(wv.add(B, Bg, 0.f, w.S[2]), false, sub(Tg, r0, 0), false, Ig, D);        // T_loc I_g^T: rows of L^T
        if ((rc = run_wave(st, mode, wv, w.gemm_ws, w.gemm_ws_bytes))) return rc;
        float* o = reinterpret_cast<float*>(s->send[1]);
        float* sc = o + x.x1_scal;
        TEAM_CUDA_CHECK(cudaMemsetAsync(sc, 0, 8 * sizeof(float), st));     // slots no fold of this configuration writes stay 0
        TEAM_LAUNCH(unicl_cat_stats_kernel, (B + 7) / 8, 256, 0, st, B, Bg, r0, ld, (const float*)w.S[0].f, (const int64_t*)w.labels_g, inv_tau,
                    o + 2 * B, o + 3 * B, o + 4 * B, w.rloss + 2 * B, o + 5 * B);
        TEAM_LAUNCH(clip_stats_kernel, (2 * B + 7) / 8, 256, 0, st, B, Bg, r0, ld, (const float*)w.S[1].f, (const float*)w.S[2].f, s->logit_scale, o, w.rloss);
        TEAM_LAUNCH(loss_fold2_kernel, 1, 1024, 0, st, B, (const float*)(o + 5 * B), (const float*)(w.rloss + 2 * B), sc, 0, 0.f, (const float*)nullptr, (float*)nullptr);
        TEAM_LAUNCH(loss_fold2_kernel, 1, 1024, 0, st, 2 * B, (const float*)w.rloss, (const float*)nullptr, sc + 2, 0, 0.f, (const float*)nullptr, (float*)nullptr);
        TEAM_LAUNCH(ce_total_kernel, 1, 1024, 0, st, B, (int)s->num_classes, s->logits, s->labels, 0.f, 0.f, (float*)nullptr, sc + 4);
        if (!evo) {       // the instance term is per sample: its value goes into this exchange, its gradient waits for dcat
            TEAM_LAUNCH(unicl_instance_kernel, (B + 7) / 8, 256, 0, st, B, (const float*)w.X[0], (const float*)w.X[1], (const float*)w.X[2],
                        (const float*)w.inv[0], (const float*)w.inv[1], (const float*)w.inv[2], (const float*)nullptr, inv_tau, 0.f,
                        (float*)nullptr, (float*)nullptr, (float*)nullptr, w.rinst, (float*)nullptr);
            TEAM_LAUNCH(loss_fold2_kernel, 1, 1024, 0, st, B, (const float*)w.rinst, (const float*)nullptr, sc + 5, 0, 0.f, (const float*)nullptr, (float*)nullptr);
        } else {          // local (class, state) keyed sums and counts of the normalised state rows
            TEAM_LAUNCH(evo_keysum_kernel, keys, 128, (size_t)((B + 31) / 32) * sizeof(unsigned int), st, B, (const float*)w.X[2], (const unsigned char*)nullptr,
                        s->labels, s->state_ids, s->num_evo, s->evo_mask, o + x.x1_ss, reinterpret_cast<int*>(o + x.x1_cnt));
        }
    } else if (phase == 2) {
        TEAM_LAUNCH(shard_cols_kernel, (6 * Bg + 255) / 256, 256, 0, st, B, Bg, 6, g1, slice1, w.cols);
        TEAM_LAUNCH(shard_losses_kernel, 1, 32, 0, st, W, g1 + x.x1_scal, slice1, (const float*)nullptr, (int64_t)0, (int64_t)Bg,
                    s->w_clip, s->w_unicl, w.scal, evo ? (float*)nullptr : s->losses6);
        if (evo) {
            TEAM_LAUNCH(shard_sum_kernel<float>, (keys * D + 255) / 256, 256, 0, st, W, (int64_t)keys * D, g1 + x.x1_ss, slice1, w.SS);
            TEAM_LAUNCH(shard_sum_kernel<int>, (keys + 255) / 256, 256, 0, st, W, (int64_t)keys, reinterpret_cast<const int*>(g1 + x.x1_cnt), slice1, w.cnt);
            TEAM_LAUNCH(evo_fwd_kernel, (B + 7) / 8, 256, 0, st, B, (const float*)w.X[2], s->labels, s->state_ids, s->num_evo, s->evo, s->evo_mask,
                        (const float*)w.SS, (const int*)w.cnt, w.Xe, w.Mh, w.sc, w.rowmask);
        }
        const float* c = w.cols;     // [0] lse i2t, [1] lse t2i, [2] max, [3] pos, [4] all, [5] valid; each [Bg]
        TEAM_LAUNCH(unicl_cat_grad_kernel, (B + 7) / 8, 256, 0, st, B, Bg, r0, ld, (const float*)w.S[0].f, (const int64_t*)w.labels_g, inv_tau,
                    0.5f * s->w_unicl, c + 2 * Bg + r0, c + 3 * Bg + r0, c + 4 * Bg + r0, c + 5 * Bg + r0, c + 2 * Bg, c + 3 * Bg, c + 4 * Bg,
                    c + 5 * Bg, (const float*)w.scal, w.G[0].f, w.G[0].h, w.G[3].f, w.G[3].h);
        const float kc = s->logit_scale * s->w_clip / (2.0f * (float)Bg);
        TEAM_LAUNCH(clip_grad_kernel, (B + 7) / 8, 256, 0, st, B, Bg, r0, ld, (const float*)w.S[1].f, s->logit_scale, kc, c + r0, c + Bg, w.G[1].f, w.G[1].h);
        TEAM_LAUNCH(clip_grad_kernel, (B + 7) / 8, 256, 0, st, B, Bg, r0, ld, (const float*)w.S[2].f, s->logit_scale, kc, c + Bg + r0, c, w.G[2].f, w.G[2].h);
        const Mat Xg = rows(0), Ig = rows(1), Tg = rows(2);
        Wave wv;
        seg(seg(wv.add(B, D, 0.f, Mat{w.dcat, nullptr, D}), false, w.G[0], true, Xg, Bg), false, w.G[3], true, Xg, Bg);   // dcat = G X_g + H X_g
        seg(wv.add(B, D, 0.f, Mat{s->g_own_rows, nullptr, D}), false, w.G[1], true, Tg, Bg);             // dI = G T_g
        seg(wv.add(B, D, 0.f, Mat{s->g_own_rows + (size_t)B * D, nullptr, D}), false, w.G[2], true, Ig, Bg);   // dT = (G^T)_loc I_g
        if ((rc = run_wave(st, mode, wv, w.gemm_ws, w.gemm_ws_bytes))) return rc;
        TEAM_LAUNCH(unicl_instance_kernel, (B + 7) / 8, 256, 0, st, B, (const float*)w.X[0], (const float*)w.X[1], (const float*)(evo ? w.Xe : w.X[2]),
                    (const float*)w.inv[0], (const float*)w.inv[1], (const float*)w.inv[2], (const float*)w.dcat, inv_tau,
                    s->w_unicl / (3.0f * (float)Bg), s->g_image, s->g_text, s->g_state, evo ? w.rinst : (float*)nullptr, evo ? w.dXe : (float*)nullptr);
        if (evo) {
            float* o = reinterpret_cast<float*>(s->send[2]);
            TEAM_CUDA_CHECK(cudaMemsetAsync(o + x.x2_scal, 0, 8 * sizeof(float), st));
            TEAM_LAUNCH(evo_bwd1_kernel, (B + 7) / 8, 256, 0, st, B, (const float*)w.Xe, (const float*)w.Mh, (const float*)w.sc, w.dXe, w.dMix);
            TEAM_LAUNCH(evo_keysum_kernel, keys, 128, (size_t)((B + 31) / 32) * sizeof(unsigned int), st, B, (const float*)w.dMix, (const unsigned char*)w.rowmask,
                        s->labels, s->state_ids, s->num_evo, s->evo_mask, o, (int*)nullptr);
            TEAM_LAUNCH(loss_fold2_kernel, 1, 1024, 0, st, B, (const float*)w.rinst, (const float*)nullptr, o + x.x2_scal + 5, 0, 0.f, (const float*)nullptr, (float*)nullptr);
        }
    } else {              // phase 3: evolution features only
        const float* g2 = reinterpret_cast<const float*>(s->gathered[2]);
        TEAM_LAUNCH(shard_sum_kernel<float>, (keys * D + 255) / 256, 256, 0, st, W, (int64_t)keys * D, g2, slice2, w.DM);
        TEAM_LAUNCH(shard_losses_kernel, 1, 32, 0, st, W, g1 + x.x1_scal, slice1, g2 + x.x2_scal, slice2, (int64_t)Bg,
                    s->w_clip, s->w_unicl, w.scal, s->losses6);
        TEAM_LAUNCH(evo_bwd2_kernel, (B + 7) / 8, 256, 0, st, B, (const float*)w.X[2], (const float*)w.inv[2], s->labels, s->state_ids,
                    (const float*)w.sc, (const float*)w.DM, (const int*)w.cnt, (const float*)w.dXe, s->g_state);
    }
    return TEAM_OK;
}
