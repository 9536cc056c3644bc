// Host orchestration + C ABI of the fusion head (include/team_b200.h): the tri-modal forward and backward
// (team_head_tri_fwd / team_head_tri_bwd), the two forwards whose text rows are shared by the whole batch
// (team_head_tri_classtext_fwd, team_head_proof_fwd: shared_rows_fwd), the projections alone and their backward
// (team_head_encode, team_head_encode_bwd, team_head_encode_rows_bwd) and the workspace queries.  Every launch goes to
// the caller's stream or a side lane joined before the call returns; there is no synchronisation and no allocation,
// so a whole step can be captured into a CUDA graph.
#include "head_proof_kernels.cuh"
#include "head_table_kernels.cuh"
#include "head_table_gram.cuh"
#include "head_dropout_kernels.cuh"

namespace team {

HeadDims head_dims(int64_t B, int C, int P, int Tc) {
    HeadDims d;
    d.B = (int)B; d.B2 = 2 * (int)B; d.C = C; d.P = P; d.M = C + P; d.Ns = d.M + 10;
    d.Nsp = (d.Ns + 15) / 16 * 16; d.Rt = C + 10; d.Tc = Tc; d.nctas = 3 * NUM_SMS;
    return d;
}

void head_plan(const HeadDims& d, int mode, void* base, HeadWS* w) {
    size_t off = 0;
    const bool bf = mode == TEAM_MODE_BF16;
    auto take_bytes = [&](size_t bytes) -> char* {
        char* p = base ? reinterpret_cast<char*>(base) + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    auto take = [&](size_t n_floats) -> float* { return reinterpret_cast<float*>(take_bytes(n_floats * sizeof(float))); };
    // fp32 matrix [rows, cols] and, in BF16 mode, its bf16 shadow
    auto mat = [&](size_t rows, size_t cols, bool want_f = true) -> Mat {
        Mat m;
        m.f = want_f ? take(rows * cols) : nullptr;
        m.h = bf ? reinterpret_cast<__nv_bfloat16*>(take_bytes(rows * cols * 2)) : nullptr;
        m.ld = (int64_t)cols;
        return m;
    };
    const size_t B2 = d.B2, Nsp = d.Nsp, Rt = d.Rt, Bn = d.B;
    for (int i = 0; i < 3; ++i) { w->Wsum[i] = mat(D, D); w->bsum[i] = take(D); }
    w->Wqkv = mat(3 * D, D);
    w->Wfc = mat(D, D, false);
    w->protos = mat(d.C, D, false); w->E = mat(10, D, false);
    w->img = mat(Bn, D, false); w->txt = mat(Bn, D, false);
    w->Ztab = take(Rt * D);
    w->S = mat(Nsp, D); w->invS = take(Nsp);
    w->QKVs = mat(Nsp, 3 * D);
    w->VFs = mat(Nsp + 2 * TG_RP, D);    // + the table rows (s, n) of the Gram GEMM (head_table_gram.cuh)
    w->TT = take(Nsp * Nsp); w->mt = take(Nsp); w->Zt = take(Nsp); w->Pt = mat(Nsp, Nsp); w->NFt = take(Nsp * D);
    w->Xo = mat(B2, D); w->invo = take(B2);
    w->QKVo = mat(B2, 3 * D); w->VFo = mat(B2, D);
    w->SQ = mat(B2, Nsp); w->SK = take(B2 * Nsp);
    w->Aext = mat(B2, Nsp); w->aown = take(B2 * 2);
    w->Ybo = take(B2 * D);
    w->dYo = mat(B2, D); w->rowdot = take(B2); w->dsown = take(B2 * 2);
    w->dSK = mat(B2, Nsp); w->dVFo = mat(B2, D); w->dVFo_own = take(B2 * D);
    w->dQKVo = mat(B2, 3 * D); w->dXo = mat(B2, D);
    w->Rfull = take(Nsp * D); w->Gfull = mat(Nsp, D); w->hfull = take(Nsp);
    w->dTT = mat(Nsp, Nsp); w->tmpNN = take(Nsp * Nsp); w->dVFs = mat(Nsp, D);
    w->dQKVs = mat(Nsp, 3 * D); w->dZtab = mat(Rt, D);
    w->ldA = 2 * ((d.Rt + 63) / 64 * 64);
    w->GG = mat(B2, D); w->A1 = mat(B2, w->ldA); w->A23 = mat(B2, w->ldA);
    w->RG = take((size_t)w->ldA * D);
    w->dVFs_a = take(Nsp * D); w->dbfc_parts = take((size_t)EXP_SUM_BLOCKS * D);
    const TabOff to = tab_offsets(d);
    w->tab_partials = take((size_t)d.nctas * to.len); w->tab_reduced = take(to.len);
    w->own_partials = take((size_t)d.nctas * OWN_PARTIAL_LEN); w->own_reduced = take(OWN_PARTIAL_LEN);
    w->nrm_partials = take((size_t)4 * NRM_MAX_PARTIALS * D);
    w->W0 = take(B2 * (size_t)tg_ldw(d)); w->xs = take(Bn * D); w->xst = take(Bn * D); w->RS = take(Bn * (size_t)TG_NRS * 32); w->GT = take(TG_GT_LEN);
    // split-K scratch: largest user is a [512,512] weight gradient reduced over 2B rows
    size_t g = gemm_f32_workspace_bytes(D, D, B2);
    const size_t g2 = gemm_f32_workspace_bytes(Nsp, D, B2);
    if (g2 > g) g = g2;
    if (g < (size_t)96 * D * D * sizeof(float)) g = (size_t)96 * D * D * sizeof(float);
    w->gemm_ws_bytes = g;
    w->gemm_ws = take(g / sizeof(float));
    // last, so that the layout of everything above does not depend on the number of text-class rows
    w->tcls = mat((size_t)(d.Tc > 0 ? d.Tc : 1), D, false);
    w->Zc = take((size_t)(d.Tc > 0 ? d.Tc : 1) * D);
    w->total_bytes = off;
}

// Workspace of the dropout route (team_head_dropout_workspace_bytes), NT = B (C + 1) table-query rows.
struct DropWS {
    Mat Ad;              // [B2][Nsp]  masked own-row probabilities
    float* aownd;        // [B2][2]    masked own-key probabilities
    Mat Wd;              // [NT][Nsp]  masked table-row probabilities
    float* tsc;          // [NT][DROP_NSC] row scalars
    float* Yt;           // [NT][D]    Wd VFs, then Ybar of the table rows
    Mat dYt;             // [NT][D]    gradient of the fc output of the table rows
    float* dU;           // [NT][D]    residual gradient of the table rows
    float* dWd;          // [NT][Nsp]  dYt VFs^T
    float* tpart;        // [NUM_SMS][OWN_PARTIAL_LEN] per-CTA partials of drop_table_bwd_kernel
    size_t total_bytes;
};
static void drop_plan(const HeadDims& d, int mode, void* base, DropWS* w) {
    size_t off = 0;
    const bool bf = mode == TEAM_MODE_BF16;
    auto take_bytes = [&](size_t bytes) -> char* {
        char* p = base ? reinterpret_cast<char*>(base) + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    auto take = [&](size_t n) -> float* { return reinterpret_cast<float*>(take_bytes(n * sizeof(float))); };
    auto mat = [&](size_t rows, size_t cols) -> Mat {
        Mat m;
        m.f = take(rows * cols);
        m.h = bf ? reinterpret_cast<__nv_bfloat16*>(take_bytes(rows * cols * 2)) : nullptr;
        m.ld = (int64_t)cols;
        return m;
    };
    const size_t NT = (size_t)d.B * (d.C + 1);
    w->Ad = mat(d.B2, d.Nsp); w->aownd = take((size_t)d.B2 * 2);
    w->Wd = mat(NT, d.Nsp); w->tsc = take(NT * DROP_NSC);
    w->Yt = take(NT * D); w->dYt = mat(NT, D); w->dU = take(NT * D); w->dWd = take(NT * d.Nsp);
    w->tpart = take((size_t)NUM_SMS * OWN_PARTIAL_LEN);
    w->total_bytes = off;
}

// A team_dropout with p > 0, checked, and its workspace laid out; on = false: the undropped head.
struct DropCfg {
    bool on = false;
    DropArgs a;
    DropWS w;
};
static int drop_setup(const HeadDims& d, int mode, const team_dropout* dr, DropCfg* c) {
    c->on = false;
    if (dr == nullptr || dr->p == 0.f) return TEAM_OK;
    TEAM_REQUIRE(dr->p > 0.f && dr->p < 1.f, "head dropout: p = %g out of [0, 1)", (double)dr->p);
    drop_plan(d, mode, dr->workspace, &c->w);
    if (dr->workspace == nullptr || dr->workspace_bytes < c->w.total_bytes) {
        set_error("head dropout: workspace %zu < %zu bytes", dr->workspace_bytes, c->w.total_bytes);
        return TEAM_EWORKSPACE;
    }
    TEAM_REQUIRE((reinterpret_cast<uintptr_t>(dr->workspace) & 255) == 0, "head dropout: workspace must be 256-byte aligned");
    c->on = true;
    c->a.attn = Philox{(uint32_t)dr->seed, (uint32_t)(dr->seed >> 32), dr->offset};
    const double t = (double)dr->p * 4294967296.0;
    c->a.thr = t >= 4294967295.0 ? 4294967295u : (uint32_t)t;
    c->a.inv_keep = 1.f / (1.f - dr->p);
    c->a.offset_dev = dr->offset_dev;
    c->a.L = 3 + d.M;
    return TEAM_OK;
}

struct HeadCtx {
    cudaStream_t st;
    int mode;
    HeadDims d;
    HeadWS w;
};

// ---------------------------------------------------------------------------------------------------------
// GEMM waves (gemm.cuh): BF16 mode runs a wave as one grouped tcgen05 launch, F32 mode as fp32 FFMA GEMMs.
static Mat fonly(float* p, int64_t ld) { return Mat{p, nullptr, ld}; }
// outputs that are only ever GEMM operands: in BF16 mode the fp32 copy is not written at all
static Mat honly(const Mat& m, int mode) { return mode == TEAM_MODE_BF16 ? Mat{nullptr, m.h, m.ld} : m; }

#define RUN(wave)                                                                  \
    do {                                                                           \
        int _rc = run_wave(cx.st, cx.mode, wave, cx.w.gemm_ws, cx.w.gemm_ws_bytes); \
        if (_rc != TEAM_OK) return _rc;                                            \
    } while (0)

static int validate(const team_head_weights* hw, int mode, int64_t batch) {
    TEAM_REQUIRE(hw != nullptr, "head: null weights");
    TEAM_REQUIRE(mode == TEAM_MODE_F32 || mode == TEAM_MODE_BF16, "head: bad mode %d", mode);
    TEAM_REQUIRE(hw->num_tasks >= 1 && hw->num_tasks <= TEAM_MAX_TASKS, "head: num_tasks %d out of [1,%d]", hw->num_tasks, TEAM_MAX_TASKS);
    TEAM_REQUIRE(hw->prompts_per_task >= 0 && hw->num_classes >= 1, "head: bad prompts_per_task/num_classes");
    TEAM_REQUIRE(batch >= 1 && batch < (1 << 22), "head: batch %lld out of range", (long long)batch);
    TEAM_REQUIRE(hw->num_classes + hw->num_tasks * hw->prompts_per_task <= 4096, "head: too many shared rows");
    return TEAM_OK;
}

static PtrList plist(const float* const* p, int n) {
    PtrList l;
    memset(&l, 0, sizeof(l));
    for (int i = 0; i < n; ++i) l.p[i] = p[i];
    l.n = n;
    return l;
}

static void conv_add(ConvList& cl, int& blocks, const float* src, float* dstf, __nv_bfloat16* dsth, int64_t n_floats) {
    if (n_floats <= 0 || (dstf == nullptr && dsth == nullptr)) return;
    ConvSeg& s = cl.s[cl.n++];
    s.src = src; s.dstf = dstf; s.dsth = dsth; s.n4 = n_floats / 4; s.blk0 = blocks;
    blocks += (int)((s.n4 + 255) / 256);
}

// step prologue (one launch): summed projections, packed {Wq;Wk;Wv}, bf16 shadows of weights and inputs
static int prologue(HeadCtx& cx, const team_head_weights* hw, int nsum, const float* image, const float* text,
                    const float* text_cls, int64_t batch) {
    HeadWS& w = cx.w;
    const HeadDims& d = cx.d;
    const int T = hw->num_tasks;
    PrepSum ps;
    memset(&ps, 0, sizeof(ps));
    const float* const* Ws[3] = {hw->w_img, hw->w_text, hw->w_state};
    const float* const* Bs[3] = {hw->b_img, hw->b_text, hw->b_state};
    const int nf = hw->num_frozen;
    for (int k = 0; k < 3; ++k) {
        if (nf > 0 && nf <= T && hw->w_frozen[k] != nullptr && hw->b_frozen[k] != nullptr) {
            // frozen tasks enter as ONE precomputed term (team_head_frozen_sums): ((W_0 + W_1) + ...) + W_nf + ... as before
            PtrList lw, lb;
            memset(&lw, 0, sizeof(lw)); memset(&lb, 0, sizeof(lb));
            lw.p[0] = hw->w_frozen[k]; lb.p[0] = hw->b_frozen[k];
            for (int t = nf; t < T; ++t) { lw.p[1 + t - nf] = Ws[k][t]; lb.p[1 + t - nf] = Bs[k][t]; }
            lw.n = lb.n = 1 + T - nf;
            ps.W[k] = lw; ps.Bv[k] = lb;
        } else {
            ps.W[k] = plist(Ws[k], T); ps.Bv[k] = plist(Bs[k], T);
        }
        ps.Wout[k] = w.Wsum[k].f; ps.Wh[k] = w.Wsum[k].h; ps.bout[k] = w.bsum[k];
    }
    ps.n = nsum;
    ConvList cl;
    memset(&cl, 0, sizeof(cl));
    cl.sum_blocks = nsum * PREP_SUM_BLOCKS_PER_W;
    int blocks = 0;
    if (hw->w_q) conv_add(cl, blocks, hw->w_q, w.Wqkv.f, w.Wqkv.h, (int64_t)D * D);
    if (hw->w_k) conv_add(cl, blocks, hw->w_k, w.Wqkv.f + (size_t)D * D, w.Wqkv.h ? w.Wqkv.h + (size_t)D * D : nullptr, (int64_t)D * D);
    if (hw->w_v) conv_add(cl, blocks, hw->w_v, w.Wqkv.f + (size_t)2 * D * D, w.Wqkv.h ? w.Wqkv.h + (size_t)2 * D * D : nullptr, (int64_t)D * D);
    if (hw->w_fc) conv_add(cl, blocks, hw->w_fc, nullptr, w.Wfc.h, (int64_t)D * D);
    if (hw->prototypes) conv_add(cl, blocks, hw->prototypes, nullptr, w.protos.h, (int64_t)hw->num_classes * D);
    if (hw->state_emb) conv_add(cl, blocks, hw->state_emb, nullptr, w.E.h, (int64_t)10 * D);
    if (image) conv_add(cl, blocks, image, nullptr, w.img.h, batch * D);
    if (text) conv_add(cl, blocks, text, nullptr, w.txt.h, batch * D);
    if (text_cls && d.Tc > 0) conv_add(cl, blocks, text_cls, nullptr, w.tcls.h, (int64_t)d.Tc * D);
    TEAM_LAUNCH(prep_kernel, cl.sum_blocks + blocks, 256, 0, cx.st, ps, cl);
    return TEAM_OK;
}

static void bind_inputs(HeadCtx& cx, const team_head_weights* hw, const float* image, const float* text, const float* text_cls) {
    HeadWS& w = cx.w;
    w.Wfc.f = const_cast<float*>(hw->w_fc);
    w.protos.f = const_cast<float*>(hw->prototypes);
    w.E.f = const_cast<float*>(hw->state_emb);
    w.img.f = const_cast<float*>(image);
    w.txt.f = const_cast<float*>(text);
    w.tcls.f = const_cast<float*>(text_cls);
}

// Checks the weights and the workspace and lays the workspace out.  The "class" block of the step rows is the
// text_rows class-text rows followed by the C prototype rows (text_rows = 0 outside shared_rows_fwd); Tc is the
// number of class-text rows staged by the prologue.  who names the caller in the workspace error.
static int setup(HeadCtx& cx, const char* who, const team_head_weights* hw, int mode, int64_t batch, int text_rows, int Tc,
                 void* workspace, size_t workspace_bytes, void* stream) {
    int rc = validate(hw, mode, batch);
    if (rc) return rc;
    cx.st = (cudaStream_t)stream;
    cx.mode = mode;
    cx.d = head_dims(batch, text_rows + hw->num_classes, hw->num_tasks * hw->prompts_per_task, Tc);
    head_plan(cx.d, mode, workspace, &cx.w);
    if (workspace == nullptr || workspace_bytes < cx.w.total_bytes) {
        set_error("%s: workspace %zu < %zu bytes", who, workspace_bytes, cx.w.total_bytes);
        return TEAM_EWORKSPACE;
    }
    TEAM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "head: workspace must be 256-byte aligned");
    return TEAM_OK;
}

// gradient-ready event (team_head_grads.ev_*): an external record node under capture, a plain record otherwise
static int record_ready(cudaStream_t st, void* ev) {
    if (ev == nullptr) return TEAM_OK;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    TEAM_CUDA_CHECK(cudaStreamIsCapturing(st, &cs));
    TEAM_CUDA_CHECK(cudaEventRecordWithFlags((cudaEvent_t)ev, st, cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault));
    return TEAM_OK;
}

// ---- fork / join onto a per-thread side stream, so that independent kernels of one call run concurrently (under
// stream capture the side stream joins the capture and the kernels become parallel branches of the graph).
// Resources are created lazily per host thread and device; if that fails (e.g. creation refused during a capture)
// the call simply stays on the caller's stream.
struct SideStream {                 // one lane: a stream and its fork / join events
    cudaStream_t st = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
struct SideLanes {
    SideStream lane[3];             // 0: independent compute kernels, 1: the gradient exchange, 2: classification logits
    bool tried = false, ok = false;
};
static SideStream* side_stream(int lane) {
    static thread_local SideLanes tab[16];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
    SideLanes& t = tab[dev];
    if (!t.tried) {
        t.tried = true;
        t.ok = true;
        for (int i = 0; i < 3; ++i) {
            SideStream& s = t.lane[i];
            if (cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking) != cudaSuccess ||
                cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                t.ok = false;
            }
        }
    }
    return t.ok ? &t.lane[lane] : nullptr;
}
// make the lane wait for everything enqueued on `main` so far; returns the stream to launch the forked work on
// (the caller's own stream when forking is unavailable).  May be called again on an already forked lane to add a
// later dependency (the second gradient bucket).
static cudaStream_t fork_side(cudaStream_t main, SideStream** out, int lane = 0) {
    *out = nullptr;
    SideStream* s = side_stream(lane);
    if (s == nullptr) return main;
    if (cudaEventRecord(s->fork, main) != cudaSuccess || cudaStreamWaitEvent(s->st, s->fork, 0) != cudaSuccess) {
        cudaGetLastError();
        return main;
    }
    *out = s;
    return s->st;
}
static int join_side(cudaStream_t main, SideStream* s) {
    if (s == nullptr) return TEAM_OK;
    TEAM_CUDA_CHECK(cudaEventRecord(s->join, s->st));
    TEAM_CUDA_CHECK(cudaStreamWaitEvent(main, s->join, 0));
    return TEAM_OK;
}

// second-generation table-row kernels unless the head is too large for them
static bool use_table2(const HeadDims& d) {
    return table2_supported(d) && table2_bwd_smem_floats(d) * sizeof(float) <= 227 * 1024;
}

// Gram formulation of the table-query rows (head_table_gram.cuh) for batches of at least TABLE_GRAM_MIN_B samples.
// Measured (profiles/EXPERIMENTS.md round 2): its kernels are 1.5 - 1.9x faster than the second generation in isolation
// at 65 536 samples, but the step gains only 2 % there (both generations fill the register file, so the side-lane kernels
// no longer overlap) and loses below ~16 384 samples, where its two extra step-level launches sit on the critical path.
constexpr int TABLE_GRAM_MIN_B = 16384;
static bool use_table_gram(const HeadDims& d) {
    return d.B >= TABLE_GRAM_MIN_B && table_gram_supported(d);
}

static void norm_add(NormList& nl, int& blocks, const float* Z, float* X, __nv_bfloat16* Xh, float* inv, int64_t rows) {
    if (rows <= 0) return;
    NormSeg& s = nl.s[nl.n++];
    s.Z = Z; s.X = X; s.Xh = Xh; s.inv = inv; s.rows = rows; s.blk0 = blocks;
    blocks += (int)((rows + 7) / 8);
}

// GEMM waves 2 and 3 of every forward: q/k/v of the step rows and of the `own` own rows, then fc folded into V and
// every score matrix.  VFo: the own-row fc values, with the bf16 shadow only where a later kernel reads it.
static int qkv_score_waves(HeadCtx& cx, int64_t own, const Mat& VFo) {
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    Wave wv;
    // ---- wave 2: q/k/v of the step rows and of the own rows against the packed [3D, D] weight
    seg(wv.add(d.Nsp, 3 * D, 0.f, honly(w.QKVs, cx.mode)), false, w.S, false, w.Wqkv, D);
    seg(wv.add(own, 3 * D, 0.f, honly(w.QKVo, cx.mode)), false, w.Xo, false, w.Wqkv, D);
    RUN(wv);
    // ---- wave 3: fc folded into V, and every score matrix
    const Mat Qs = sub(w.QKVs, 0, 0), Ks = sub(w.QKVs, 0, D), Vs = sub(w.QKVs, 0, 2 * D);
    const Mat Qo = sub(w.QKVo, 0, 0), Ko = sub(w.QKVo, 0, D), Vo = sub(w.QKVo, 0, 2 * D);
    seg(wv.add(d.Nsp, D, 0.f, w.VFs), false, Vs, false, w.Wfc, D);
    seg(wv.add(own, D, 0.f, VFo), false, Vo, false, w.Wfc, D);
    seg(wv.add(d.Nsp, d.Nsp, 0.f, fonly(w.TT, d.Nsp)), false, Qs, false, Ks, D);
    seg(wv.add(own, d.Nsp, 0.f, fonly(w.SQ.f, d.Nsp)), false, Qo, false, Ks, D);
    seg(wv.add(own, d.Nsp, 0.f, fonly(w.SK, d.Nsp)), false, Ko, false, Qs, D);
    RUN(wv);
    return TEAM_OK;
}

// Forward of the two layouts whose Tn text rows are shared by the whole batch, up to the image-row outputs: step rows
// [Tn text | C prototypes | P prompts | 10 state rows], own rows = the B image rows (head_proof_kernels.cuh).
// Class-text form of forward_tri_modal: state_ids given, the state table fills the 10 state rows and the sample's
// state row is one more key of its image query.  PROOF: state_ids = nullptr, the state rows stay zero and unseen;
// with inputs_encoded the image / text rows arrive projected and normalised.  cx comes from setup(text_rows = Tn).
static int shared_rows_fwd(HeadCtx& cx, const team_head_weights* hw, const float* image_feat, const float* text_feat,
                           int Tn, const int64_t* state_ids, int inputs_encoded, float* out_image) {
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    const bool states = state_ids != nullptr;
    const int C = hw->num_classes, R = Tn + C, M = d.M, B = d.B;
    int rc;
    bind_inputs(cx, hw, image_feat, nullptr, text_feat);
    {
        team_head_weights staged = *hw;
        if (!states) staged.state_emb = nullptr;
        if ((rc = prologue(cx, &staged, states ? 3 : 2, inputs_encoded ? nullptr : image_feat, nullptr,
                           inputs_encoded ? nullptr : text_feat, B))) return rc;
    }
    if (inputs_encoded) {                                  // rows arrive projected + normalised: straight into Xo / S
        PrepSum ps;
        memset(&ps, 0, sizeof(ps));
        ConvList cl;
        memset(&cl, 0, sizeof(cl));
        int blocks = 0;
        conv_add(cl, blocks, image_feat, w.Xo.f, w.Xo.h, (int64_t)B * D);
        conv_add(cl, blocks, text_feat, w.S.f, w.S.h, (int64_t)Tn * D);
        TEAM_LAUNCH(prep_kernel, blocks, 256, 0, cx.st, ps, cl);
    }
    // prompt rows [R, M), then zeros up to Nsp: from Ns with a state table, from M without (the state rows are zero)
    const int zero_from = states ? d.Ns : M;
    const int fill_rows = d.P + (d.Nsp - zero_from);
    if (fill_rows > 0)
        TEAM_LAUNCH(fill_prompt_rows_kernel, fill_rows, 128, 0, cx.st, plist(hw->prompts, hw->num_tasks), hw->prompts_per_task > 0 ? hw->prompts_per_task : 1, R, zero_from, d.Nsp, w.S.f, w.S.h);
    Wave wv;
    // ---- wave 1: projections (class-text rows, prototype rows, state table, image rows)
    if (!inputs_encoded) seg(wv.add(Tn, D, 0.f, fonly(w.Ztab, D), w.bsum[1]), false, w.tcls, false, w.Wsum[1], D);
    seg(wv.add(C, D, 0.f, fonly(w.Ztab + (size_t)Tn * D, D), w.bsum[0]), false, w.protos, false, w.Wsum[0], D);
    if (states) seg(wv.add(10, D, 0.f, fonly(w.Ztab + (size_t)R * D, D), w.bsum[2]), false, w.E, false, w.Wsum[2], D);
    if (!inputs_encoded) seg(wv.add(B, D, 0.f, fonly(w.Xo.f, D), w.bsum[0]), false, w.img, false, w.Wsum[0], D);
    RUN(wv);
    {   // L2-normalise: projected text and prototype rows -> S[0,R), state table -> S[M,M+10), image rows in place
        NormList nl;
        memset(&nl, 0, sizeof(nl));
        nl.do_normalize = 1;
        int blocks = 0;
        const int r0 = inputs_encoded ? Tn : 0;
        norm_add(nl, blocks, w.Ztab + (size_t)r0 * D, w.S.f + (size_t)r0 * D, w.S.h ? w.S.h + (size_t)r0 * D : nullptr, w.invS + r0, R - r0);
        if (states) norm_add(nl, blocks, w.Ztab + (size_t)R * D, w.S.f + (size_t)M * D, w.S.h ? w.S.h + (size_t)M * D : nullptr, w.invS + M, 10);
        if (!inputs_encoded) norm_add(nl, blocks, w.Xo.f, w.Xo.f, w.Xo.h, w.invo, B);
        TEAM_LAUNCH(rows_normalize_kernel, blocks, 256, 0, cx.st, nl);
    }
    if ((rc = qkv_score_waves(cx, B, fonly(w.VFo.f, D)))) return rc;
    TEAM_LAUNCH(table_prep_kernel, (d.Nsp + 7) / 8, 256, 0, cx.st, w.TT, M, d.Nsp, w.mt, w.Zt, w.Pt.f, w.Pt.h, (const float*)nullptr, (const float*)nullptr, (const float*)nullptr, (const __nv_bfloat16*)nullptr, 0, 0, (float*)nullptr, (__nv_bfloat16*)nullptr);
    TEAM_LAUNCH(image_attn_own_kernel, (B + 7) / 8, 256, 0, cx.st, B, M, d.Nsp, w.SQ.f, w.QKVo.f, cx.mode == TEAM_MODE_BF16 ? w.QKVo.h : nullptr, state_ids, w.Aext.f, w.Aext.h, w.aown);
    // ---- wave 4: probabilities x (fc-space) values
    seg(wv.add(d.Nsp, D, 0.f, fonly(w.NFt, D)), false, w.Pt, true, w.VFs, d.Nsp);
    seg(wv.add(B, D, 0.f, fonly(w.Ybo, D)), false, w.Aext, true, w.VFs, d.Nsp);
    RUN(wv);
    TEAM_LAUNCH(proof_ln_own_fwd_kernel, (B + 7) / 8, 256, 0, cx.st, B, w.Ybo, w.aown, w.VFo.f, w.Xo.f, hw->b_fc, hw->ln_g, hw->ln_b, out_image);
    return TEAM_OK;
}

// Forward of the dropout route from the score matrices on (after GEMM wave 3): the two softmax kernels as in the undropped
// forward, the masked probability rows, GEMM wave 4 with one product per probability set, and the fc / LayerNorm rows.
static int drop_fwd(HeadCtx& cx, const team_head_weights* hw, const DropCfg& dc, const int64_t* state_ids, bool want_cls,
                    float* cls_logits, int64_t* cls_argmax, float* out_image, float* out_text, float* out_state, float* out_proto) {
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    const DropWS& dw = dc.w;
    int rc;
    SideStream* side = nullptr;
    {
        const cudaStream_t tst = fork_side(cx.st, &side);
        TEAM_LAUNCH(table_prep_kernel, (d.Nsp + 7) / 8, 256, 0, tst, w.TT, d.M, d.Nsp, w.mt, w.Zt, w.Pt.f, (__nv_bfloat16*)nullptr, (const float*)nullptr, (const float*)nullptr, (const float*)nullptr, (const __nv_bfloat16*)nullptr, 0, 0, (float*)nullptr, (__nv_bfloat16*)nullptr);
        TEAM_LAUNCH(attn_own_kernel, (d.B2 + 7) / 8, 256, 0, cx.st, d, w.SQ.f, w.QKVo.f, cx.mode == TEAM_MODE_BF16 ? w.QKVo.h : nullptr, state_ids, w.Aext.f, (__nv_bfloat16*)nullptr, w.aown);
        if ((rc = join_side(cx.st, side))) return rc;
    }
    const int64_t NT = (int64_t)d.B * (d.C + 1);
    const int own_blocks = (d.B2 + 7) / 8;
    TEAM_LAUNCH(drop_probs_kernel, own_blocks + (NT + 7) / 8, 256, 0, cx.st, d, dc.a, own_blocks, (const float*)w.Aext.f, (const float*)w.aown, state_ids, (const float*)w.SK, (const float*)w.TT, (const float*)w.mt, (const float*)w.Zt, (const float*)w.Pt.f, dw.Ad.f, dw.Ad.h, dw.aownd, dw.Wd.f, dw.Wd.h, dw.tsc);
    // ---- wave 4: masked probabilities x (fc-space) values
    Wave wv;
    seg(wv.add(d.B2, D, 0.f, fonly(w.Ybo, D)), false, dw.Ad, true, w.VFs, d.Nsp);
    seg(wv.add(NT, D, 0.f, fonly(dw.Yt, D)), false, dw.Wd, true, w.VFs, d.Nsp);
    RUN(wv);
    SideStream* cls_side = nullptr;
    if (want_cls) {
        const cudaStream_t cst = fork_side(cx.st, &cls_side, 2);
        if ((rc = cosine_logits_launch(cst, w.Xo.f, d.B, w.Zc, d.Tc, nullptr, cls_logits, cls_argmax))) return rc;
    }
    TEAM_LAUNCH(drop_ln_fwd_kernel, own_blocks + (d.B + 7) / 8, 256, 0, cx.st, d, dc.a, own_blocks, w.Ybo, (const float*)dw.aownd, dw.Yt, (const float*)dw.tsc, (const float*)w.VFo.f, (const float*)w.Xo.f, (const float*)w.S.f, hw->b_fc, hw->ln_g, hw->ln_b, state_ids, out_image, out_text, out_state, out_proto);
    return join_side(cx.st, cls_side);
}

// The backward from GEMM wave 7 on (score gradients dS / dSK / dTT, dVFo, dVFs, Rfull and the LayerNorm / bias partials are
// complete): shared by the undropped head and the dropout route.
static int bwd_tail(HeadCtx& cx, const team_head_grads* gr) {
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    int rc;
    const Mat Qs = sub(w.QKVs, 0, 0), Ks = sub(w.QKVs, 0, D), Vs = sub(w.QKVs, 0, 2 * D);
    const Mat Qo = sub(w.QKVo, 0, 0), Ko = sub(w.QKVo, 0, D), Vo = sub(w.QKVo, 0, 2 * D);
    const Mat dQo = sub(w.dQKVo, 0, 0), dVo = sub(w.dQKVo, 0, 2 * D);
    const Mat dQs = sub(w.dQKVs, 0, 0), dKs = sub(w.dQKVs, 0, D), dVs = sub(w.dQKVs, 0, 2 * D);
    Wave wv;
    const Mat& dS = w.SQ;
    // ---- wave 7: score gradients -> dQ/dK, fc folded into V, dWfc
    seg(wv.add(d.B2, D, 1.f, dQo), false, dS, true, Ks, d.Nsp);                                                                     // dQo = dS Ks + the own x own part
    seg(seg(wv.add(d.Nsp, D, 0.f, honly(dKs, cx.mode)), true, dS, true, Qo, d.B2), true, w.dTT, true, Qs, d.Nsp);                  // dKs = dS^T Qo + dTT^T Qs
    seg(seg(wv.add(d.Nsp, D, 0.f, honly(dQs, cx.mode)), true, w.dSK, true, Ko, d.B2), false, w.dTT, true, Ks, d.Nsp);              // dQs = dSK^T Ko + dTT Ks
    seg(wv.add(d.B2, D, 0.f, honly(dVo, cx.mode)), false, w.dVFo, true, w.Wfc, D);                                                 // dVo = dVFo Wfc
    seg(wv.add(d.Nsp, D, 0.f, honly(dVs, cx.mode)), false, w.dVFs, true, w.Wfc, D);
    seg(seg(wv.add(D, D, 0.f, fonly(gr->w_fc, D)), true, w.dVFo, true, Vo, d.B2), true, w.dVFs, true, Vs, d.Nsp);  // dWfc = dVFo^T Vo + dVFs^T Vs
    RUN(wv);
    if ((rc = record_ready(cx.st, gr->ev_w_fc))) return rc;
    // data-parallel: gradient buckets are summed over the ranks on the comm lane as soon as they are final, under
    // the remaining kernels of this call: w_fc now, w_q / w_k / w_v after wave 8, everything else at the end
    SideStream* comm_side = nullptr;
    const team_peer_comm* comm = gr->comm != nullptr && gr->comm->world > 1 ? gr->comm : nullptr;
    const int64_t DD = (int64_t)D * D;
    if (comm != nullptr) {
        const float* base = reinterpret_cast<const float*>(comm->bufs[comm->rank]);
        auto inside = [&](const float* p, int64_t lo, int64_t hi) { return p >= base + lo && p + 1 <= base + hi; };
        TEAM_REQUIRE(comm->split_at >= DD && gr->w_fc == base && inside(gr->w_q, DD, comm->split_at) && inside(gr->w_k, DD, comm->split_at) &&
                     inside(gr->w_v, DD, comm->split_at) && inside(gr->w_img, comm->split_at, comm->n_total) &&
                     inside(gr->w_text, comm->split_at, comm->n_total) && inside(gr->w_state, comm->split_at, comm->n_total) &&
                     inside(gr->state_emb, comm->split_at, comm->n_total) && inside(gr->b_fc, comm->split_at, comm->n_total),
                     "head bwd: gradient pointers do not match the peer-comm buckets");
        const cudaStream_t cst = fork_side(cx.st, &comm_side, 1);
        if (comm_side != nullptr && (rc = peer_allreduce_range(cst, comm, 0, DD, 0))) return rc;
    }
    // ---- wave 8: through the packed q/k/v projection
    seg(wv.add(d.B2, D, 1.f, fonly(w.dXo.f, D)), false, w.dQKVo, true, w.Wqkv, 3 * D);                             // dXo += dQKVo Wqkv
    seg(wv.add(d.Nsp, D, 1.f, fonly(w.Rfull, D)), false, w.dQKVs, true, w.Wqkv, 3 * D);                            // dS_rows (in Rfull)
    {
        float* dW[3] = {gr->w_q, gr->w_k, gr->w_v};
        for (int i = 0; i < 3; ++i)
            seg(seg(wv.add(D, D, 0.f, fonly(dW[i], D)), true, sub(w.dQKVo, 0, i * D), true, w.Xo, d.B2), true, sub(w.dQKVs, 0, i * D), true, w.S, d.Nsp);
    }
    RUN(wv);
    if ((rc = record_ready(cx.st, gr->ev_w_qkv))) return rc;
    if (comm != nullptr && comm_side != nullptr) {
        SideStream* again = nullptr;
        const cudaStream_t cst = fork_side(cx.st, &again, 1);            // second dependency of the same lane
        if (again != nullptr) {
            if ((rc = peer_allreduce_range(cst, comm, DD, comm->split_at - DD, 0))) return rc;
        } else {
            comm_side = nullptr;      // cannot happen once the lane exists; keep the end-of-call fallback consistent
        }
    }
    // ---- normalisation backward of own rows, prototype rows and state-table rows (+ bias-gradient partials)
    NrmList nl;
    memset(&nl, 0, sizeof(nl));
    int nblk[4];
    {
        int blocks = 0;
        auto add = [&](const float* src, const float* X, const float* inv, float* dZ, __nv_bfloat16* dZh, int64_t rows, int64_t src_off) {
            NrmSeg& s = nl.s[nl.n];
            int rpb = (int)((rows + NRM_MAX_PARTIALS - 1) / NRM_MAX_PARTIALS);
            rpb = (rpb + 7) / 8 * 8;
            if (rpb < 8) rpb = 8;
            s.dXsrc = src; s.X = X; s.inv = inv; s.dZ = dZ; s.dZh = dZh; s.rows = rows; s.src_off = src_off;
            s.rows_per_block = rpb; s.blk0 = blocks;
            s.partial = w.nrm_partials + (size_t)nl.n * NRM_MAX_PARTIALS * D;
            nblk[nl.n] = (int)((rows + rpb - 1) / rpb);
            blocks += nblk[nl.n];
            ++nl.n;
        };
        add(w.dXo.f, w.Xo.f, w.invo, w.dXo.f, w.dXo.h, d.B, 0);                                                    // dz0 (in place)
        add(w.dXo.f, w.Xo.f, w.invo, w.dXo.f + (size_t)d.B * D, w.dXo.h ? w.dXo.h + (size_t)d.B * D : nullptr, d.B, d.B);   // dz1
        add(w.Rfull, w.S.f, w.invS, w.dZtab.f, w.dZtab.h, d.C, 0);                                                 // dzp
        add(w.Rfull, w.S.f, w.invS, w.dZtab.f + (size_t)d.C * D, w.dZtab.h ? w.dZtab.h + (size_t)d.C * D : nullptr, 10, d.M);   // dzs
        TEAM_LAUNCH(nrm_bwd_kernel, blocks, 256, 0, cx.st, nl);
    }
    // the bias / prompt gradients (finish_bwd) only need the partials of nrm_bwd: side lane, beside wave 9
    SideStream* fin_side = nullptr;
    {
        const cudaStream_t fst = fork_side(cx.st, &fin_side);
        FinishArgs fa;
        memset(&fa, 0, sizeof(fa));
        for (int i = 0; i < 4; ++i) { fa.part[i] = nl.s[i].partial; fa.nblk[i] = nblk[i]; }
        fa.b_img = gr->b_img; fa.b_text = gr->b_text; fa.b_state = gr->b_state;
        fa.Rfull = w.Rfull; fa.prompts = d.P > 0 ? gr->prompts : nullptr; fa.C = d.C; fa.P = d.P;
        fa.dbfc_parts = w.dbfc_parts; fa.dbfc = gr->b_fc;
        TEAM_LAUNCH(finish_bwd_kernel, 4 + (fa.prompts ? (d.P + 3) / 4 : 0), 512, 0, fst, fa);
    }
    // ---- wave 9: gradients of the newest projections and of the state embedding
    const Mat dz0 = sub(w.dXo, 0, 0), dz1 = sub(w.dXo, d.B, 0), dzp = sub(w.dZtab, 0, 0), dzs = sub(w.dZtab, d.C, 0);
    seg(seg(wv.add(D, D, 0.f, fonly(gr->w_img, D)), true, dz0, true, w.img, d.B), true, dzp, true, w.protos, d.C);  // dWi = dz0^T x + dzp^T protos
    seg(wv.add(D, D, 0.f, fonly(gr->w_text, D)), true, dz1, true, w.txt, d.B);
    seg(wv.add(D, D, 0.f, fonly(gr->w_state, D)), true, dzs, true, w.E, 10);
    seg(wv.add(10, D, 0.f, fonly(gr->state_emb, D)), false, dzs, true, w.Wsum[2], D);                              // dE = dzs Ws
    RUN(wv);
    if ((rc = join_side(cx.st, fin_side))) return rc;
    if (comm != nullptr) {
        // Late bucket: on the second flag channel, so it starts as soon as the last kernel is done even if the q/k/v
        // bucket on the comm lane is still finishing.  Measured against "join the comm lane first" with the same
        // kernels: N = 2 0.229 vs 0.236 ms per step, N = 8 0.233 vs 0.235 ms.
        const bool overlap_late = comm_side != nullptr;
        if (comm_side == nullptr) {
            if ((rc = peer_allreduce_range(cx.st, comm, 0, comm->split_at, 0))) return rc;       // no side lanes: everything at the end
        } else if (!overlap_late) {
            if ((rc = join_side(cx.st, comm_side))) return rc;
        }
        if ((rc = peer_allreduce_range(cx.st, comm, comm->split_at, comm->n_total - comm->split_at, overlap_late ? 1 : 0))) return rc;
        if (overlap_late && (rc = join_side(cx.st, comm_side))) return rc;
    }
    return TEAM_OK;
}

// Backward of the dropout route up to GEMM wave 7: own rows (side lane) beside the table-query rows, then one wave with
// dA = dYo VFs^T, dKo += dSK Qs, dVFs = Ad^T dYo + Wd^T dYt and dWd = dYt VFs^T, the own-query softmax backward and the
// fixed-order batch folds of the table rows (dTT, Rfull, LayerNorm and fc-bias gradients).
static int drop_bwd(HeadCtx& cx, const team_head_weights* hw, const DropCfg& dc, const int64_t* state_ids, const float* g_image,
                    const float* g_text, const float* g_state, const float* g_proto, const team_head_grads* gr) {
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    const DropWS& dw = dc.w;
    const bool bf = cx.mode == TEAM_MODE_BF16;
    int rc;
    int ogrid = (d.B + 7) / 8;
    if (ogrid > NUM_SMS) ogrid = NUM_SMS;
    SideStream* own_side = nullptr;
    const cudaStream_t ost = fork_side(cx.st, &own_side);
    TEAM_LAUNCH(drop_ln_own_bwd_kernel, ogrid, 256, 0, ost, d, dc.a, (const float*)w.Ybo, (const float*)w.Xo.f, (const float*)w.VFo.f, (const float*)w.aown, (const float*)dw.aownd, hw->b_fc, hw->ln_g, hw->ln_b, g_image, g_text, w.dYo.f, w.dYo.h, w.dXo.f, w.rowdot, w.dsown, w.dVFo_own, w.own_partials, gr->g_own_rows);
    TEAM_LAUNCH(own_own_bwd_kernel, (d.B + 7) / 8, 256, 0, ost, d, w.QKVo.f, bf ? w.QKVo.h : nullptr, w.dsown, w.dQKVo.f, (__nv_bfloat16*)nullptr);
    TEAM_LAUNCH(drop_table_bwd_kernel, ogrid, 256, 0, cx.st, d, dc.a, (const float*)dw.Yt, dw.tsc, (const float*)w.VFo.f, (const float*)w.S.f, hw->b_fc, hw->ln_g, hw->ln_b, state_ids, g_proto, g_state, dw.dYt.f, dw.dYt.h, dw.dU, w.dSK.f, w.dSK.h, w.dVFo.f, dw.tpart);
    if ((rc = join_side(cx.st, own_side))) return rc;
    {
        const int64_t n4 = (int64_t)d.B2 * D / 4;
        TEAM_LAUNCH(add_rows_kernel, (unsigned)((n4 + 255) / 256), 256, 0, cx.st, n4, w.dVFo.f, (const float*)w.dVFo_own, w.dVFo.h);
    }
    const int64_t NT = (int64_t)d.B * (d.C + 1);
    const Mat Qs = sub(w.QKVs, 0, 0), dKo = sub(w.dQKVo, 0, D);
    Wave wv;
    seg(wv.add(d.B2, d.Nsp, 0.f, fonly(w.SQ.f, d.Nsp)), false, w.dYo, false, w.VFs, D);                            // dA = dYo VFs^T
    seg(wv.add(d.B2, D, 1.f, dKo), false, w.dSK, true, Qs, d.Nsp);                                                 // dKo += dSK Qs
    seg(seg(wv.add(d.Nsp, D, 0.f, w.dVFs), true, dw.Ad, true, w.dYo, d.B2), true, dw.Wd, true, dw.dYt, NT);       // dVFs
    seg(wv.add(NT, d.Nsp, 0.f, fonly(dw.dWd, d.Nsp)), false, dw.dYt, false, w.VFs, D);                            // dWd = dYt VFs^T
    RUN(wv);
    {
        const int64_t n4 = (int64_t)d.B2 * d.Nsp / 4;
        TEAM_LAUNCH(drop_ds_kernel, (unsigned)((n4 + 255) / 256), 256, 0, cx.st, n4, d.Nsp / 4, (const float*)w.Aext.f, (const float*)dw.Ad.f, (const float*)w.rowdot, w.SQ.f, w.SQ.h, bf ? 0 : 1);
        const int tt_blocks = (d.Nsp * d.Nsp + 255) / 256;
        TEAM_LAUNCH(drop_fold_kernel, tt_blocks + d.Nsp + 1, 256, 0, cx.st, d, tt_blocks, (const float*)dw.Wd.f, (const float*)dw.dWd, (const float*)w.Pt.f, (const float*)dw.tsc, state_ids, (const float*)dw.dU, (const float*)dw.tpart, ogrid, (const float*)w.own_partials, ogrid, w.dTT.f, w.dTT.h, w.Rfull, gr->ln_g, gr->ln_b, w.dbfc_parts);
    }
    return bwd_tail(cx, gr);
}

}  // namespace team

using namespace team;

extern "C" size_t team_head_workspace_bytes(int64_t batch, int32_t num_classes, int32_t num_prompts,
                                            int32_t num_text_cls, int mode) {
    HeadDims d = head_dims(batch, num_classes, num_prompts, num_text_cls);
    HeadWS w;
    head_plan(d, mode, nullptr, &w);
    return w.total_bytes;
}

// *p += v on the device (one thread): the per-step advance of team_dropout.offset_dev, capturable, no host sync
static __global__ void u64_add_kernel(uint64_t* p, uint64_t v) {
    pdl_trigger();
    pdl_wait();
    *p += v;
}
extern "C" int team_u64_add(uint64_t* p, uint64_t v, void* stream) {
    TEAM_REQUIRE(p != nullptr, "u64 add: null pointer");
    TEAM_LAUNCH(u64_add_kernel, 1, 1, 0, (cudaStream_t)stream, p, v);
    return TEAM_OK;
}

extern "C" size_t team_head_dropout_workspace_bytes(int64_t batch, int32_t num_classes, int32_t num_prompts, int mode) {
    DropWS w;
    drop_plan(head_dims(batch, num_classes, num_prompts, 0), mode, nullptr, &w);
    return w.total_bytes;
}

extern "C" int team_head_frozen_sums(const team_head_weights* hw, int32_t num_frozen, float* w_sums, float* b_sums, void* stream) {
    TEAM_REQUIRE(hw != nullptr && w_sums != nullptr && b_sums != nullptr, "head frozen sums: null pointer");
    TEAM_REQUIRE(num_frozen >= 1 && num_frozen <= hw->num_tasks && hw->num_tasks <= TEAM_MAX_TASKS, "head frozen sums: num_frozen %d out of [1, %d]", num_frozen, hw->num_tasks);
    PrepSum ps;
    memset(&ps, 0, sizeof(ps));
    const float* const* Ws[3] = {hw->w_img, hw->w_text, hw->w_state};
    const float* const* Bs[3] = {hw->b_img, hw->b_text, hw->b_state};
    for (int k = 0; k < 3; ++k) {
        for (int t = 0; t < num_frozen; ++t) TEAM_REQUIRE(Ws[k][t] != nullptr && Bs[k][t] != nullptr, "head frozen sums: null projection %d of task %d", k, t);
        ps.W[k] = plist(Ws[k], num_frozen); ps.Bv[k] = plist(Bs[k], num_frozen);
        ps.Wout[k] = w_sums + (size_t)k * D * D; ps.Wh[k] = nullptr; ps.bout[k] = b_sums + (size_t)k * D;
    }
    ps.n = 3;
    ConvList cl;
    memset(&cl, 0, sizeof(cl));
    cl.sum_blocks = 3 * PREP_SUM_BLOCKS_PER_W;
    TEAM_LAUNCH(prep_kernel, cl.sum_blocks, 256, 0, (cudaStream_t)stream, ps, cl);
    return TEAM_OK;
}

// byte offset of the normalised projected own rows Xo ([2B,512] fp32: image rows, then text rows) inside the workspace
extern "C" size_t team_head_own_rows_offset(int64_t batch, int32_t num_classes, int32_t num_prompts, int32_t num_text_cls, int mode) {
    HeadDims d = head_dims(batch, num_classes, num_prompts, num_text_cls);
    HeadWS w;
    head_plan(d, mode, reinterpret_cast<void*>(uintptr_t(256)), &w);          // a non-null fake base: only the offsets are used
    return (size_t)(reinterpret_cast<uintptr_t>(w.Xo.f) - 256);
}

// Forward: 13 launches (prologue, prompt rows, 4 GEMM waves, 7 row kernels; three short side-lane branches) - see
// DESIGN.md section 4.
extern "C" int team_head_tri_fwd(const team_head_weights* hw, int mode, int64_t batch, const float* image_feat,
                                 const float* text_feat, const int64_t* state_ids, const float* text_cls,
                                 int64_t num_text_cls, float* out_image, float* out_text, float* out_state,
                                 float* out_proto, float* cls_logits, int64_t* cls_argmax, void* workspace,
                                 size_t workspace_bytes, void* stream, const team_dropout* dropout) {
    HeadCtx cx;
    int rc = setup(cx, "head", hw, mode, batch, 0, (int)(text_cls ? num_text_cls : 0), workspace, workspace_bytes, stream);
    if (rc) return rc;
    DropCfg dc;
    if ((rc = drop_setup(cx.d, mode, dropout, &dc))) return rc;
    TEAM_REQUIRE(image_feat && text_feat && state_ids && out_image && out_text && out_state && out_proto, "head fwd: null pointer");
    TEAM_REQUIRE(hw->w_q && hw->w_k && hw->w_v && hw->w_fc && hw->b_fc && hw->ln_g && hw->ln_b && hw->state_emb && hw->prototypes, "head fwd: null weight");
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    const bool want_cls = d.Tc > 0 && (cls_logits != nullptr || cls_argmax != nullptr);
    bind_inputs(cx, hw, image_feat, text_feat, text_cls);
    SideStream* side = nullptr;
    const int fill_rows = d.P + (d.Nsp - d.Ns);
    if (fill_rows > 0) {          // prompt rows of S: independent of the prologue -> side lane
        const cudaStream_t fst = fork_side(cx.st, &side);
        TEAM_LAUNCH(fill_prompt_rows_kernel, fill_rows, 128, 0, fst, plist(hw->prompts, hw->num_tasks), hw->prompts_per_task > 0 ? hw->prompts_per_task : 1, d.C, d.Ns, d.Nsp, w.S.f, w.S.h);
    }
    if ((rc = prologue(cx, hw, 3, image_feat, text_feat, want_cls ? text_cls : nullptr, batch))) return rc;
    SideStream* fill_side = side;        // joined before wave 2 (the first reader of the prompt rows): wave 1 chains straight behind the prologue
    Wave wv;
    // ---- wave 1: every projection of the step (prototype rows, state table, image rows, text rows, class text)
    seg(wv.add(d.C, D, 0.f, fonly(w.Ztab, D), w.bsum[0]), false, w.protos, false, w.Wsum[0], D);
    seg(wv.add(10, D, 0.f, fonly(w.Ztab + (size_t)d.C * D, D), w.bsum[2]), false, w.E, false, w.Wsum[2], D);
    seg(wv.add(d.B, D, 0.f, fonly(w.Xo.f, D), w.bsum[0]), false, w.img, false, w.Wsum[0], D);
    seg(wv.add(d.B, D, 0.f, fonly(w.Xo.f + (size_t)d.B * D, D), w.bsum[1]), false, w.txt, false, w.Wsum[1], D);
    if (want_cls) seg(wv.add(d.Tc, D, 0.f, fonly(w.Zc, D), w.bsum[1]), false, w.tcls, false, w.Wsum[1], D);
    RUN(wv);
    {   // L2-normalise: prototype rows -> S[0,C), state table -> S[M,M+10), own rows in place
        NormList nl;
        memset(&nl, 0, sizeof(nl));
        nl.do_normalize = 1;
        int blocks = 0;
        norm_add(nl, blocks, w.Ztab, w.S.f, w.S.h, w.invS, d.C);
        norm_add(nl, blocks, w.Ztab + (size_t)d.C * D, w.S.f + (size_t)d.M * D, w.S.h ? w.S.h + (size_t)d.M * D : nullptr, w.invS + d.M, 10);
        norm_add(nl, blocks, w.Xo.f, w.Xo.f, w.Xo.h, w.invo, d.B2);
        TEAM_LAUNCH(rows_normalize_kernel, blocks, 256, 0, cx.st, nl);
    }
    if ((rc = join_side(cx.st, fill_side))) return rc;
    // waves 2 and 3; VFo keeps its bf16 shadow (GEMM operand of the backward and of the Gram table rows)
    if ((rc = qkv_score_waves(cx, d.B2, w.VFo))) return rc;
    if (dc.on) return drop_fwd(cx, hw, dc, state_ids, want_cls, cls_logits, cls_argmax, out_image, out_text, out_state, out_proto);
    SideStream* gram_side = nullptr;
    {   // the two softmax kernels (step-row table, own rows) are independent
        const cudaStream_t tst = fork_side(cx.st, &side);
        const bool gram = use_table_gram(d);
        const int xwarps = TG_RP;                            // + the s rows S_r + b_fc (bulk-copy source of the table-row kernels; Gram operand)
        TEAM_LAUNCH(table_prep_kernel, (d.Nsp + xwarps + 7) / 8, 256, 0, tst, w.TT, d.M, d.Nsp, w.mt, w.Zt, w.Pt.f, w.Pt.h, w.S.f, hw->b_fc,
                    w.VFs.f, (const __nv_bfloat16*)w.VFs.h, d.C, TG_RP,
                    w.VFs.f + (size_t)d.Nsp * D, w.VFs.h ? w.VFs.h + (size_t)d.Nsp * D : (__nv_bfloat16*)nullptr);
        if (gram)             // ... and its n rows
            TEAM_LAUNCH(table_nf_kernel, d.Rt, 256, ((d.M + 3) / 4 * 4 + 512) * sizeof(float), tst, w.TT, d.M, d.Nsp, d.C, w.VFs.f, (const __nv_bfloat16*)w.VFs.h,
                        w.VFs.f + (size_t)(d.Nsp + TG_RP) * D, w.VFs.h ? w.VFs.h + (size_t)(d.Nsp + TG_RP) * D : (__nv_bfloat16*)nullptr);
        TEAM_LAUNCH(attn_own_kernel, (d.B2 + 7) / 8, 256, 0, cx.st, d, w.SQ.f, w.QKVo.f, cx.mode == TEAM_MODE_BF16 ? w.QKVo.h : nullptr, state_ids, w.Aext.f, w.Aext.h, w.aown);
        if ((rc = join_side(cx.st, side))) return rc;
        // step-level dot products of the table rows: beside GEMM wave 4 (joined before the table-row kernel)
        if (gram) TEAM_LAUNCH(table_gram_prep_kernel, (d.Rt + 10 + 7) / 8, 256, 0, side != nullptr ? side->st : cx.st, d.Rt, w.VFs.f + (size_t)d.Nsp * D, w.VFs.f + (size_t)d.M * D, w.GT);
        gram_side = gram ? side : nullptr;
    }
    // ---- wave 4: probabilities x (fc-space) values
    seg(wv.add(d.Nsp, D, 0.f, fonly(w.NFt, D)), false, w.Pt, true, w.VFs, d.Nsp);
    seg(wv.add(d.B2, D, 0.f, fonly(w.Ybo, D)), false, w.Aext, true, w.VFs, d.Nsp);
    // sample x table dot products of the table-query rows (head_table_gram.cuh): W0 = VFo x [VFs ; S_table + b_fc]^T
    if (use_table_gram(d)) seg(wv.add(d.B2, tg_ldw(d), 0.f, fonly(w.W0, tg_ldw(d))), false, w.VFo, false, w.VFs, D);
    RUN(wv);
    // the own-row outputs and the classification logits do not depend on the table-query rows: side stream
    const cudaStream_t sst = fork_side(cx.st, &side);
    TEAM_LAUNCH(ln_own_fwd_kernel, (d.B2 + 7) / 8, 256, 0, sst, d, w.Ybo, w.aown, w.VFo.f, w.Xo.f, hw->b_fc, hw->ln_g, hw->ln_b, out_image, out_text);
    // forward_for_classification (models/proof.py:519-536; image rows are already normalised in Xo): a third lane beside the
    // own-row LayerNorm and the table rows.  Measured alternatives (tools/timeline.py, profiles/r2z_timeline_*): behind
    // ln_own_fwd on the same lane the pair outlasts the table rows by 5 us; forked right after the normalisation (its inputs
    // are ready there, 45 us of slack) it slows GEMM waves 2 and 3 by more than it saves (0.194 vs 0.189 ms per step), at the
    // lowest stream priority as well - the kernels of one step compete for the same SMs and L2 bandwidth.
    SideStream* cls_side = nullptr;
    if (want_cls) {
        const cudaStream_t cst = fork_side(cx.st, &cls_side, 2);
        if ((rc = cosine_logits_launch(cst, w.Xo.f, d.B, w.Zc, d.Tc, nullptr, cls_logits, cls_argmax))) return rc;
    }
    if (use_table_gram(d)) {      // Gram formulation: scalar LayerNorm algebra per (sample, row), vector outputs as coefficient sums
        if ((rc = join_side(cx.st, gram_side))) return rc;          // table_gram_prep_kernel
        const int nw = tg_warps(d), groups = (d.B + nw - 1) / nw;
        const size_t tsm = tg_fwd_smem_floats(d) * sizeof(float);
        TEAM_CUDA_CHECK(cudaFuncSetAttribute(table_gram_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm));
        TEAM_LAUNCH(table_gram_fwd_kernel, groups < NUM_SMS ? groups : NUM_SMS, nw * 32, tsm, cx.st, d, w.SK, w.TT, w.mt, w.Zt, w.VFs.f + (size_t)d.Nsp * D, w.GT, w.W0, w.VFo.f, w.VFs.f, hw->ln_g, hw->ln_b, state_ids, out_proto, out_state, w.xs, w.xst, w.RS);
    } else if (use_table2(d)) {   // warp per sample, table rows resident in shared memory (head_table_kernels.cuh)
        const int groups = (d.B + TW - 1) / TW;
        const size_t tsm = table2_fwd_smem_floats(d) * sizeof(float);
        TEAM_CUDA_CHECK(cudaFuncSetAttribute(table_rows_fwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm));
        TEAM_LAUNCH(table_rows_fwd2_kernel, groups < NUM_SMS ? groups : NUM_SMS, TW * 32, tsm, cx.st, d, w.SK, w.TT, w.mt, w.Zt, w.NFt, w.VFo.f, w.VFs.f, w.S.f, hw->b_fc, hw->ln_g, hw->ln_b, state_ids, out_proto, out_state, w.VFs.f + (size_t)d.Nsp * D);
    } else {
        const int tgrid = d.B < 6 * NUM_SMS ? d.B : 6 * NUM_SMS;
        TEAM_LAUNCH(table_rows_fwd_kernel, tgrid, TQ_WARPS * 32, 0, cx.st, d, w.SK, w.TT, w.mt, w.Zt, w.NFt, w.VFo.f, w.VFs.f, w.S.f, hw->b_fc, hw->ln_g, hw->ln_b, state_ids, out_proto, out_state);
    }
    if ((rc = join_side(cx.st, side))) return rc;
    if ((rc = join_side(cx.st, cls_side))) return rc;
    return TEAM_OK;
}

// Backward: 13 launches at the headline size (5 GEMM waves, 8 row kernels; more when split-K runs through the fix-up
// kernel or the gradient exchange is folded in); needs the workspace of the matching forward call.
extern "C" int team_head_tri_bwd(const team_head_weights* hw, int mode, int64_t batch, const float* image_feat,
                                 const float* text_feat, const int64_t* state_ids, const float* g_image,
                                 const float* g_text, const float* g_state, const float* g_proto,
                                 const team_head_grads* gr, void* workspace, size_t workspace_bytes, void* stream,
                                 const team_dropout* dropout) {
    HeadCtx cx;
    int rc = setup(cx, "head", hw, mode, batch, 0, 0, workspace, workspace_bytes, stream);
    if (rc) return rc;
    DropCfg dc;
    if ((rc = drop_setup(cx.d, mode, dropout, &dc))) return rc;
    TEAM_REQUIRE(gr && g_image && g_text && g_state && image_feat && text_feat && state_ids, "head bwd: null pointer");
    TEAM_REQUIRE(gr->w_img && gr->b_img && gr->w_text && gr->b_text && gr->w_state && gr->b_state && gr->state_emb &&
                 gr->w_q && gr->w_k && gr->w_v && gr->w_fc && gr->b_fc && gr->ln_g && gr->ln_b, "head bwd: null gradient buffer");
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    bind_inputs(cx, hw, image_feat, text_feat, nullptr);
    if (dc.on) return drop_bwd(cx, hw, dc, state_ids, g_image, g_text, g_state, g_proto, gr);
    const TabOff to = tab_offsets(d);
    const bool bf = cx.mode == TEAM_MODE_BF16;
    // ---- own query rows: independent of the table-query rows -> side lane, beside them (its dVF part goes to dVFo_own)
    int ogrid = (d.B + 7) / 8;
    if (ogrid > NUM_SMS) ogrid = NUM_SMS;
    SideStream* own_side = nullptr;
    // (Enqueueing the table-row kernel first - it needs a whole register file per CTA and cannot share an SM with these two -
    // was measured: it then runs alone in 26 us, but the own-row kernels are squeezed onto the 20 remaining SMs and finish
    // later than before: 0.1948 vs 0.1885 ms per step, tools/timeline.py.)
    const cudaStream_t ost = fork_side(cx.st, &own_side);
    TEAM_LAUNCH(ln_own_bwd_kernel, ogrid, 256, 0, ost, d, w.Ybo, w.Xo.f, w.VFo.f, w.aown, hw->b_fc, hw->ln_g, hw->ln_b, g_image, g_text, w.dYo.f, w.dYo.h, w.dXo.f, w.rowdot, w.dsown, w.dVFo_own, (__nv_bfloat16*)nullptr, w.own_partials, gr->g_own_rows);
    // own x own score gradients: initial values of the dQ / dK rows (the GEMMs of waves 5 and 7 accumulate on top)
    TEAM_LAUNCH(own_own_bwd_kernel, (d.B + 7) / 8, 256, 0, ost, d, w.QKVo.f, bf ? w.QKVo.h : nullptr, w.dsown, w.dQKVo.f, (__nv_bfloat16*)nullptr);
    // ---- table-query rows (prototype / state outputs)
    int tgrid;
    if (use_table_gram(d)) {      // Gram formulation (head_table_gram.cuh); needs W0 / GT / xs / xst / RS of the matching forward
        const int nw = 8, groups = (d.B + nw - 1) / nw;
        tgrid = groups < NUM_SMS ? groups : NUM_SMS;
        // LayerNorm gamma / beta gradients of the table rows: own kernel on the side lane (fields dgam / dbet of the records)
        TEAM_LAUNCH(table_dgamma_kernel, tgrid, 256, 0, own_side != nullptr ? own_side->st : cx.st, d, g_proto, g_state, w.xs, w.xst, w.tab_partials);
        const size_t tsm = tg_bwd_smem_floats(d, nw) * sizeof(float);
        TEAM_CUDA_CHECK(cudaFuncSetAttribute(table_gram_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm));
        TEAM_LAUNCH(table_gram_bwd_kernel, tgrid, nw * 32, tsm, cx.st, d, w.SK, w.TT, w.mt, w.Zt, w.VFs.f + (size_t)d.Nsp * D, w.GT, w.VFo.f, w.VFs.f, hw->ln_g, state_ids, g_proto, g_state, w.RS, w.dSK.f, w.dSK.h, w.dVFo.f, w.GG.f, w.GG.h, w.A1.f, w.A1.h, w.A23.f, w.A23.h, w.ldA, w.tab_partials);
    } else if (use_table2(d)) {   // warp per sample, table rows resident in shared memory (head_table_kernels.cuh)
        const int groups = (d.B + TW - 1) / TW;
        tgrid = groups < NUM_SMS ? groups : NUM_SMS;
        const size_t tsm = table2_bwd_smem_floats(d) * sizeof(float);
        TEAM_CUDA_CHECK(cudaFuncSetAttribute(table_rows_bwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm));
        TEAM_LAUNCH(table_rows_bwd2_kernel, tgrid, TW * 32, tsm, cx.st, d, w.SK, w.TT, w.mt, w.Zt, w.NFt, w.VFo.f, w.VFs.f, w.S.f, hw->b_fc, hw->ln_g, state_ids, g_proto, g_state, w.dSK.f, w.dSK.h, w.dVFo.f, w.GG.f, w.GG.h, w.A1.f, w.A1.h, w.A23.f, w.A23.h, w.ldA, w.tab_partials, w.VFs.f + (size_t)d.Nsp * D);
    } else {
        tgrid = d.B < d.nctas ? d.B : d.nctas;
        const size_t tsm = table_bwd_smem_floats(d) * sizeof(float);
        TEAM_REQUIRE(tsm <= 200 * 1024, "head bwd: too many classes for the table-row kernel (%d)", d.C);
        TEAM_CUDA_CHECK(cudaFuncSetAttribute(table_rows_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm));
        TEAM_LAUNCH(table_rows_bwd_kernel, tgrid, TQ_WARPS * 32, tsm, cx.st, d, w.SK, w.TT, w.mt, w.Zt, w.NFt, w.VFo.f, w.VFs.f, w.S.f, hw->b_fc, hw->ln_g, state_ids, g_proto, g_state, w.dSK.f, w.dSK.h, w.dVFo.f, w.GG.f, w.GG.h, w.A1.f, w.A1.h, w.A23.f, w.A23.h, w.ldA, w.tab_partials);
    }
    if ((rc = join_side(cx.st, own_side))) return rc;
    // the fixed-order fold of the per-CTA partials and dVFo += dVFo_own are not needed before expand_table / wave 7:
    // side lane, beside GEMM wave 5
    SideStream* red_side = nullptr;
    {
        const cudaStream_t rst = fork_side(cx.st, &red_side);
        ReduceJobs rj;
        rj.j[0] = ReduceJob{w.tab_partials, w.tab_reduced, to.len / 4, tgrid};
        rj.j[1] = ReduceJob{w.own_partials, w.own_reduced, OWN_PARTIAL_LEN / 4, ogrid};
        rj.blocks0 = (int)((to.len / 4 + RP_COLS - 1) / RP_COLS);
        TEAM_LAUNCH(reduce_partials_kernel, rj.blocks0 + (OWN_PARTIAL_LEN / 4 + RP_COLS - 1) / RP_COLS, RP_COLS * RP_GROUPS, 0, rst, rj);
        const int64_t n4 = (int64_t)d.B2 * D / 4;
        TEAM_LAUNCH(add_rows_kernel, (unsigned)((n4 + 255) / 256), 256, 0, rst, n4, w.dVFo.f, w.dVFo_own, w.dVFo.h);
    }
    const Mat Qs = sub(w.QKVs, 0, 0), dKo = sub(w.dQKVo, 0, D);
    Wave wv;
    // ---- wave 5: R/G coefficient GEMM (A1^T GG + A23^T VFo), dA = dYo VFs^T (into SQ), dKo = dSK Qs
    seg(seg(wv.add(w.ldA, D, 0.f, fonly(w.RG, D)), true, w.A1, true, w.GG, d.B2), true, w.A23, true, w.VFo, d.B2);
    seg(wv.add(d.B2, d.Nsp, 0.f, fonly(w.SQ.f, d.Nsp)), false, w.dYo, false, w.VFs, D);
    seg(wv.add(d.B2, D, 1.f, dKo), false, w.dSK, true, Qs, d.Nsp);                       // += the own x own part (own_own_bwd_kernel)
    seg(wv.add(d.Nsp, D, 0.f, fonly(w.dVFs_a, D)), true, w.Aext, true, w.dYo, d.B2);
    RUN(wv);
    if ((rc = join_side(cx.st, red_side))) return rc;
    TEAM_LAUNCH(expand_table_kernel, d.Nsp + EXP_SUM_BLOCKS, 128, 0, cx.st, d, w.tab_reduced, w.own_reduced, w.RG, w.ldA / 2, w.NFt, w.S.f, w.VFs.f, hw->b_fc, w.Rfull, w.Gfull.f, w.Gfull.h, w.hfull, w.dTT.f, w.dVFs.f, w.dVFs_a, gr->ln_g, gr->ln_b, w.dbfc_parts);
    // ---- wave 6: G VFs^T, dVFs += Pt^T G
    seg(wv.add(d.Nsp, d.Nsp, 0.f, fonly(w.tmpNN, d.Nsp)), false, w.Gfull, false, w.VFs, D);
    seg(wv.add(d.Nsp, D, 1.f, w.dVFs), true, w.Pt, true, w.Gfull, d.Nsp);
    RUN(wv);
    {   // dS = Aext .* (dA - rowdot) / tau (in place);  dTT += Pt .* (G VFs^T - h) / tau
        const int64_t n4 = (int64_t)d.B2 * d.Nsp / 4;
        SideStream* sd = nullptr;
        const cudaStream_t dst = fork_side(cx.st, &sd);
        TEAM_LAUNCH(dtt_kernel, (d.Nsp * d.Nsp + 255) / 256, 256, 0, dst, d.Nsp, d.M, w.Pt.f, w.tmpNN, w.hfull, w.dTT.f, w.dTT.h);
        TEAM_LAUNCH(ds_kernel, (unsigned)((n4 + 255) / 256), 256, 0, cx.st, n4, d.Nsp / 4, w.Aext.f, w.rowdot, w.SQ.f, w.SQ.h, bf ? 0 : 1);
        if ((rc = join_side(cx.st, sd))) return rc;
    }
    return bwd_tail(cx, gr);
}

// PROOF fusion forward (Proof_Net.forward, utils/inc_net.py:436-463; forward_transformer with transformer=True,
// :465-492, when inputs_encoded != 0: image_feat / text_feat are then the already projected + normalised rows).
// 14 launches.  workspace: team_head_workspace_bytes(batch, num_text + C, P, num_text, mode).
extern "C" int team_head_proof_fwd(const team_head_weights* hw, int mode, int64_t batch, const float* image_feat,
                                   const float* text_feat, int64_t num_text, int inputs_encoded, float* out_image,
                                   float* out_text, float* out_proto, void* workspace, size_t workspace_bytes,
                                   void* stream) {
    TEAM_REQUIRE(image_feat && text_feat && out_image && out_text && out_proto, "head proof fwd: null pointer");
    TEAM_REQUIRE(num_text >= 1 && num_text <= 2048, "head proof fwd: num_text %lld out of range", (long long)num_text);
    const int Tn = (int)num_text;
    HeadCtx cx;
    int rc = setup(cx, "head proof fwd", hw, mode, batch, Tn, Tn, workspace, workspace_bytes, stream);
    if (rc) return rc;
    TEAM_REQUIRE(hw->w_q && hw->w_k && hw->w_v && hw->w_fc && hw->b_fc && hw->ln_g && hw->ln_b && hw->prototypes, "head proof fwd: null weight");
    if ((rc = shared_rows_fwd(cx, hw, image_feat, text_feat, Tn, nullptr, inputs_encoded, out_image))) return rc;
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    const int R = Tn + hw->num_classes, B = d.B;           // shared rows whose outputs are returned (batch means)
    // ---- shared-row queries: per-CTA sums over a contiguous sample block, then the fixed-order batch mean
    int per_cta = (B + 2 * NUM_SMS - 1) / (2 * NUM_SMS);
    if (per_cta < 4) per_cta = 4;
    const int nparts = (B + per_cta - 1) / per_cta;
    TEAM_REQUIRE((size_t)nparts * R * D * sizeof(float) <= w.gemm_ws_bytes, "head proof fwd: partial buffer too small");
    float* partials = reinterpret_cast<float*>(w.gemm_ws);
    TEAM_LAUNCH(proof_table_rows_fwd_kernel, nparts, PT_WARPS * 32, 0, cx.st, B, R, d.Nsp, per_cta, w.SK, w.mt, w.Zt, w.NFt, w.VFo.f, w.S.f, hw->b_fc, partials);
    TEAM_LAUNCH(proof_finalize_kernel, R, 512, 0, cx.st, partials, nparts, R, Tn, 1.0f / (float)B, hw->ln_g, hw->ln_b, out_text, out_proto);
    return TEAM_OK;
}

// Class-text form of forward_tri_modal (utils/inc_net.py:528-580 with num_text != batch): forward only.
// workspace: team_head_workspace_bytes(batch, num_text + C, P, num_text, mode).
extern "C" int team_head_tri_classtext_fwd(const team_head_weights* hw, int mode, int64_t batch, const float* image_feat,
                                           const float* text_feat, int64_t num_text, const int64_t* state_ids,
                                           float* out_image, float* out_text, float* out_state, float* out_proto,
                                           void* workspace, size_t workspace_bytes, void* stream) {
    TEAM_REQUIRE(image_feat && text_feat && state_ids && out_image && out_text && out_state && out_proto, "head classtext fwd: null pointer");
    TEAM_REQUIRE(num_text >= 1 && num_text <= 2048, "head classtext fwd: num_text %lld out of range", (long long)num_text);
    const int Tn = (int)num_text;
    HeadCtx cx;
    int rc = setup(cx, "head classtext fwd", hw, mode, batch, Tn, Tn, workspace, workspace_bytes, stream);
    if (rc) return rc;
    TEAM_REQUIRE(hw->w_q && hw->w_k && hw->w_v && hw->w_fc && hw->b_fc && hw->ln_g && hw->ln_b && hw->prototypes && hw->state_emb, "head classtext fwd: null weight");
    if ((rc = shared_rows_fwd(cx, hw, image_feat, text_feat, Tn, state_ids, 0, out_image))) return rc;
    const HeadDims& d = cx.d;
    HeadWS& w = cx.w;
    TEAM_LAUNCH(ct_table_rows_fwd_kernel, (d.B + 7) / 8, 256, 0, cx.st, d.B, Tn, hw->num_classes, d.M, d.Nsp, w.SK, w.TT, w.mt, w.Zt, w.NFt, w.VFo.f, w.VFs.f, w.S.f, hw->b_fc, hw->ln_g, hw->ln_b, state_ids, out_text, out_state, out_proto);
    return TEAM_OK;
}

// workspace: team_head_workspace_bytes(which <= 1 ? n_rows : 1, C, P, 0, mode)
extern "C" int team_head_encode(const team_head_weights* hw, int mode, int which, const void* x, int64_t n_rows,
                                int normalize, float* out, void* workspace, size_t workspace_bytes, void* stream) {
    HeadCtx cx;
    TEAM_REQUIRE(which >= 0 && which <= 3 && out != nullptr && n_rows >= 0, "head encode: bad args");
    if (which == 3 && hw != nullptr) n_rows = hw->num_classes;
    if (n_rows == 0) return TEAM_OK;
    int rc = setup(cx, "head", hw, mode, which <= 1 ? n_rows : 1, 0, 0, workspace, workspace_bytes, stream);
    if (rc) return rc;
    HeadWS& w = cx.w;
    const float* xf = which <= 1 ? reinterpret_cast<const float*>(x) : nullptr;
    TEAM_REQUIRE(which > 1 || xf != nullptr, "head encode: null input");
    TEAM_REQUIRE(which != 2 || (x != nullptr && hw->state_emb != nullptr), "head encode: null state ids / embedding");
    TEAM_REQUIRE(which != 3 || hw->prototypes != nullptr, "head encode: null prototypes");
    bind_inputs(cx, hw, xf, nullptr, nullptr);
    {
        team_head_weights tmp = *hw;            // only the projections (and the rows being encoded) are staged
        tmp.w_q = tmp.w_k = tmp.w_v = tmp.w_fc = nullptr;
        if (which != 3) tmp.prototypes = nullptr;
        if (which != 2) tmp.state_emb = nullptr;
        if ((rc = prologue(cx, &tmp, 3, xf, nullptr, nullptr, which <= 1 ? n_rows : 0))) return rc;
    }
    const int k = which == 3 ? 0 : which;
    Wave wv;
    NormList nl;
    memset(&nl, 0, sizeof(nl));
    nl.do_normalize = normalize;
    int blocks = 0;
    if (which == 2) {
        // 10-row table first, then gather by state id
        seg(wv.add(10, D, 0.f, fonly(w.Ztab, D), w.bsum[2]), false, w.E, false, w.Wsum[2], D);
        RUN(wv);
        norm_add(nl, blocks, w.Ztab, w.Ztab, nullptr, nullptr, 10);
        TEAM_LAUNCH(rows_normalize_kernel, blocks, 256, 0, cx.st, nl);
        TEAM_LAUNCH(gather_rows_kernel, (unsigned)((n_rows + 7) / 8), 256, 0, cx.st, w.Ztab, reinterpret_cast<const int64_t*>(x), n_rows, out);
        return TEAM_OK;
    }
    seg(wv.add(n_rows, D, 0.f, fonly(out, D), w.bsum[k]), false, which == 3 ? w.protos : w.img, false, w.Wsum[k], D);
    RUN(wv);
    if (normalize) {
        norm_add(nl, blocks, out, out, nullptr, nullptr, n_rows);
        TEAM_LAUNCH(rows_normalize_kernel, blocks, 256, 0, cx.st, nl);
    }
    return TEAM_OK;
}

// Gradient of encode_image / encode_text (which = 0 | 1) with respect to the newest projection of that
// modality (older ones are frozen and share the same gradient, utils/inc_net.py:494-507):
//   y = [normalize](x Wsum^T + bsum);  g_w = dz^T x,  g_b = colsum(dz),  dz = g_out or its normalise-backward.
// The forward is recomputed (one GEMM + one row kernel) instead of being kept alive by the caller.
// workspace: team_head_workspace_bytes(n_rows, C, P, 0, mode)
extern "C" int team_head_encode_bwd(const team_head_weights* hw, int mode, int which, const float* x, int64_t n_rows,
                                    int normalize, const float* g_out, float* g_w, float* g_b, void* workspace,
                                    size_t workspace_bytes, void* stream) {
    TEAM_REQUIRE(which == 0 || which == 1, "head encode bwd: which must be 0 (image) or 1 (text)");
    return team_head_encode_rows_bwd(hw, mode, which, x, n_rows, normalize, g_out, g_w, g_b, nullptr, workspace, workspace_bytes, stream);
}

// The same with the state modality (which = 2: x = the gathered embedding rows E[state_ids], fp32) and an optional
// gradient w.r.t. the input rows g_x = dz Wsum (state embedding table: the caller sums g_x by state id; prototype rows
// pushed through projs_img: which = 0, g_x unused).
extern "C" int team_head_encode_rows_bwd(const team_head_weights* hw, int mode, int which, const float* x, int64_t n_rows,
                                         int normalize, const float* g_out, float* g_w, float* g_b, float* g_x,
                                         void* workspace, size_t workspace_bytes, void* stream) {
    HeadCtx cx;
    TEAM_REQUIRE(which >= 0 && which <= 2 && x != nullptr && g_out != nullptr && g_w != nullptr && g_b != nullptr && n_rows >= 1,
                 "head encode bwd: bad args");
    int rc = setup(cx, "head", hw, mode, n_rows, 0, 0, workspace, workspace_bytes, stream);
    if (rc) return rc;
    HeadWS& w = cx.w;
    bind_inputs(cx, hw, x, nullptr, nullptr);
    {
        team_head_weights tmp = *hw;
        tmp.w_q = tmp.w_k = tmp.w_v = tmp.w_fc = nullptr;
        tmp.prototypes = nullptr; tmp.state_emb = nullptr;
        if ((rc = prologue(cx, &tmp, 3, x, nullptr, nullptr, n_rows))) return rc;
    }
    Wave wv;
    if (normalize) {
        seg(wv.add(n_rows, D, 0.f, fonly(w.Xo.f, D), w.bsum[which]), false, w.img, false, w.Wsum[which], D);
        RUN(wv);
        NormList nl;
        memset(&nl, 0, sizeof(nl));
        nl.do_normalize = 1;
        int blocks = 0;
        norm_add(nl, blocks, w.Xo.f, w.Xo.f, nullptr, w.invo, n_rows);
        TEAM_LAUNCH(rows_normalize_kernel, blocks, 256, 0, cx.st, nl);
    }
    NrmList nl;
    memset(&nl, 0, sizeof(nl));
    nl.identity = normalize ? 0 : 1;
    int rpb = (int)((n_rows + NRM_MAX_PARTIALS - 1) / NRM_MAX_PARTIALS);
    rpb = (rpb + 7) / 8 * 8;
    NrmSeg& sg = nl.s[0];
    sg.dXsrc = g_out; sg.X = w.Xo.f; sg.inv = w.invo; sg.dZ = w.dXo.f; sg.dZh = w.dXo.h; sg.rows = n_rows; sg.src_off = 0;
    sg.rows_per_block = rpb; sg.blk0 = 0; sg.partial = w.nrm_partials;
    nl.n = 1;
    const int nblk = (int)((n_rows + rpb - 1) / rpb);
    TEAM_LAUNCH(nrm_bwd_kernel, nblk, 256, 0, cx.st, nl);
    seg(wv.add(D, D, 0.f, fonly(g_w, D)), true, sub(w.dXo, 0, 0), true, w.img, n_rows);
    if (g_x != nullptr) seg(wv.add(n_rows, D, 0.f, fonly(g_x, D)), false, sub(w.dXo, 0, 0), true, w.Wsum[which], D);
    RUN(wv);
    FinishArgs fa;
    memset(&fa, 0, sizeof(fa));
    fa.part[0] = w.nrm_partials; fa.nblk[0] = nblk;
    fa.b_img = g_b;
    TEAM_LAUNCH(finish_bwd_kernel, 3, 512, 0, cx.st, fa);
    return TEAM_OK;
}
