/*
 * team_b200.h - C ABI of the B200-native TEAM head (libteam_b200.so).
 *
 * The reference (ericzhengz/TEAM-Temporal-Evolution-Aware-Multimodal-model) is pure
 * Python/torch and has no FFI of its own; every entry point below replaces the tensor
 * math of the reference method cited next to it (file:line relative to the reference
 * root) and is what a ctypes binding inside that method would call (INTEGRATION.md).
 *
 * Conventions
 *   - return 0 on success, a negative TEAM_E* code otherwise; team_last_error() gives a
 *     thread-local message for the last failure.
 *   - all pointers are DEVICE pointers unless the name ends in _host; row-major,
 *     contiguous, 16-byte aligned.  The caller owns all memory (outputs + workspace);
 *     team_*_workspace_bytes() sizes the workspace.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); no hidden
 *     synchronisation, no global mutable state, re-entrant across streams.
 *   - feature width is fixed to TEAM_D = 512 (CLIP ViT-B/16, utils/inc_net.py:21).
 */
#ifndef TEAM_B200_H
#define TEAM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TEAM_D 512
#define TEAM_NUM_STATES 10          /* utils/inc_net.py:361 */
#define TEAM_MAX_TASKS 64

#define TEAM_OK 0
#define TEAM_EINVAL (-1)            /* bad argument / unsupported shape */
#define TEAM_ECUDA (-2)             /* CUDA runtime error (message in team_last_error) */
#define TEAM_EWORKSPACE (-3)        /* workspace too small */
#define TEAM_EUNSUPPORTED (-4)      /* needs an sm_100 device */

#define TEAM_DTYPE_F32 0
#define TEAM_DTYPE_BF16 1

/* precision modes of the head */
#define TEAM_MODE_F32 0             /* all GEMMs in fp32 FFMA (parity mode, 1e-5) */
#define TEAM_MODE_BF16 1            /* large GEMMs on tcgen05 with bf16 operands, fp32 accumulate */

const char* team_last_error(void);
int team_version(void);
/* 0 if the current device is sm_100 (B200), TEAM_EUNSUPPORTED otherwise */
int team_device_check(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
long long team_launch_count(void);
/* optional per-launch CUDA-event timing of the GEMM kernels (kind 0 = fp32 FFMA GEMM, 1 = tcgen05 bf16 GEMM);
 * team_prof_collect synchronises, sums and clears.  Not for use under stream capture. */
int team_prof_enable(int on);
int team_prof_collect(int kind, double* total_ms, double* total_flops, double* total_bytes, long long* launches);
/* per-launch records in launch order (ms, flops, kind) for up to cap launches; returns the count; clears. */
long long team_prof_dump(double* ms, double* flops, int* kind, long long cap);

/* ------------------------------------------------------------------ prototype build
 * Deterministic, atomic-free keyed segmented sum (K9/K17).
 * Replaces: Learner.cal_prototype reduction loop   models/proof.py:258-276
 *           simplecil.Learner.replace_fc loop      models/simplecil.py:48-55
 *           per-state batch centres                utils/state_distance.py:98-103
 * key(i) = (labels[i]-class_base)*num_states + states[i]   if states != NULL
 *        =  labels[i]-class_base                            otherwise
 * Rows whose label is outside [class_base, class_base+num_classes) or whose state is
 * outside [0,num_states) are skipped.  If normalize_rows != 0 every row is L2-normalised
 * (F.normalize, eps 1e-12) before accumulation (convnet.encode_image(normalize=True),
 * models/proof.py:248).  sums[K,512] fp32 and counts[K] int64 are OVERWRITTEN
 * (K = num_classes * max(num_states,1)).  Result is bit-reproducible run to run.
 */
size_t team_segsum_workspace_bytes(int64_t n_rows, int64_t num_keys);
int team_segsum(const void* x, int x_dtype, const int64_t* labels, const int64_t* states,
                int64_t n_rows, int64_t class_base, int64_t num_classes, int64_t num_states,
                int normalize_rows, float* sums, int64_t* counts,
                void* workspace, size_t workspace_bytes, void* stream);
/* means[k,:] = sums[k,:]/counts[k] for counts[k]>0; rows with counts==0 are left untouched
 * (empty classes keep their previous prototype, models/proof.py:261).  If class_sums /
 * class_counts are non-NULL they receive the per-class totals over states
 * (num_groups = num_keys/group) and class_means the per-class means. */
int team_segmean_finalize(const float* sums, const int64_t* counts, int64_t num_keys,
                          float* means, int64_t group, float* class_means,
                          int64_t* class_counts, void* stream);

/* ------------------------------------------------------------------ cosine classifier
 * logits[n,c] = sigma * <x_n/|x_n|, w_c/|w_c|>    (K8)
 * Replaces: CosineLinear.forward                    convs/linears.py:51-61
 *           final stage of forward_for_classification models/proof.py:526-535 (sigma = 1)
 * logits (fp32 [N,C]) and argmax (int64 [N], first maximal index like torch.max) are
 * each optional (NULL to skip).  sigma_dev may be NULL (= 1).
 */
int team_cosine_logits(const void* x, int x_dtype, int64_t n_rows, const float* w,
                       int64_t num_classes, const float* sigma_dev, float* logits,
                       int64_t* argmax, void* stream);

/* ------------------------------------------------------------------ the fusion head
 * forward_tri_modal + forward_for_classification, fwd and bwd.
 * Replaces: Proof_Net.encode_image/encode_text/encode_state/encode_prototpyes
 *               utils/inc_net.py:401-422, :518-526
 *           Proof_Net.forward_tri_modal               utils/inc_net.py:528-580
 *           MultiHeadAttention.forward (sel_attn)      convs/projections.py:64-87
 *           Learner.forward_for_classification         models/proof.py:519-536
 *           and their autograd backward (models/proof.py:444).
 */
typedef struct team_head_weights {
    int32_t num_tasks;                       /* T */
    int32_t prompts_per_task;                /* context_prompt_length_per_task */
    const float* w_img[TEAM_MAX_TASKS];      /* projs_img[t].MLP[0].weight [512,512] */
    const float* b_img[TEAM_MAX_TASKS];      /* projs_img[t].MLP[0].bias   [512] */
    const float* w_text[TEAM_MAX_TASKS];
    const float* b_text[TEAM_MAX_TASKS];
    const float* w_state[TEAM_MAX_TASKS];
    const float* b_state[TEAM_MAX_TASKS];
    const float* prompts[TEAM_MAX_TASKS];    /* context_prompts[t] [prompts_per_task,512] */
    const float* state_emb;                  /* state_embedder.state_embeddings.weight [10,512] */
    const float* w_q;                        /* sel_attn.w_qs.weight [512,512] */
    const float* w_k;
    const float* w_v;
    const float* w_fc;                       /* sel_attn.fc.weight */
    const float* b_fc;
    const float* ln_g;                       /* sel_attn.layer_norm.weight */
    const float* ln_b;
    const float* prototypes;                 /* img_prototypes [C,512] */
    int32_t num_classes;                     /* C */
    /* Optional: the projections of the first num_frozen tasks are frozen (utils/inc_net.py:392-393, :494-502), so their
     * sums are constants of the task: w_frozen[k] [512,512] / b_frozen[k] [512] (k = 0 image, 1 text, 2 state) hold
     * sum_{t < num_frozen} W_t as written by team_head_frozen_sums, and the step prologue adds only the remaining tasks
     * (same left-to-right order, bit-identical to summing all T).  num_frozen = 0: every task is summed per call. */
    int32_t num_frozen;
    const float* w_frozen[3];
    const float* b_frozen[3];
} team_head_weights;

/* w_sums [3][512*512], b_sums [3][512]: sum over tasks t < num_frozen of the image / text / state projections
 * (1 <= num_frozen <= T), for team_head_weights.w_frozen / b_frozen.  Call again whenever those parameters change. */
int team_head_frozen_sums(const team_head_weights* w, int32_t num_frozen, float* w_sums, float* b_sums, void* stream);

/* Peer-memory gradient exchange folded into the backward (optional, see team_peer_allreduce_f32 for the meaning of
 * the pointer tables): the gradient pointers of team_head_grads must then lie inside bufs[rank][0, n_total) with
 * w_fc, w_q, w_k, w_v inside [0, split_at) and everything else at or beyond split_at.  The backward sums the early
 * bucket over the ranks on a side stream as soon as it is final (after the q/k/v weight gradients), under its
 * remaining kernels, and the late bucket after its last kernel. */
typedef struct team_peer_comm {
    void* bufs[8];
    void* flags[8];
    void* multicast;                         /* NVLS mapping of the buffers or NULL */
    int32_t rank, world;
    int64_t n_total;                         /* floats in the gradient buffer (multiple of 4) */
    int64_t split_at;                        /* first float of the late bucket (multiple of 4) */
} team_peer_comm;

typedef struct team_head_grads {            /* all OVERWRITTEN by team_head_tri_bwd */
    float* w_img;  float* b_img;             /* newest task only (utils/inc_net.py:494-507) */
    float* w_text; float* b_text;
    float* w_state; float* b_state;
    float* prompts;                          /* all prompt rows [T*prompts_per_task,512]; may be NULL */
    float* state_emb;                        /* [10,512] */
    float* w_q; float* w_k; float* w_v;
    float* w_fc; float* b_fc;
    float* ln_g; float* ln_b;
    /* Optional cudaEvent_t handles (NULL = none) recorded on the call's stream as soon as a group of gradients is
     * final, so a data-parallel caller can start their all-reduce on another stream while the rest of the backward
     * still runs: ev_w_fc after w_fc, ev_w_qkv after w_q / w_k / w_v (everything else is final when the call's last
     * kernel ends).  Under stream capture they become external event-record nodes (cudaEventRecordExternal). */
    void* ev_w_fc;
    void* ev_w_qkv;
    const team_peer_comm* comm;              /* NULL: no exchange inside the call */
    /* Optional INPUT: an extra cotangent [2B,512] on the normalised projected own rows themselves (image rows, then text
     * rows: what encode_image / encode_text(normalize=True) return and team_head_own_rows_offset exposes).  The
     * learner's ClipLoss branch (models/proof.py:428-431) consumes exactly these rows, so its gradient joins the
     * head's backward here instead of running the two projections and their backward a second time.  NULL = none. */
    const float* g_own_rows;
} team_head_grads;

size_t team_head_workspace_bytes(int64_t batch, int32_t num_classes, int32_t num_prompts,
                                 int32_t num_text_cls, int mode);

/* Train-mode dropout of sel_attn inside team_head_tri_fwd / team_head_tri_bwd (convs/projections.py:28, :62, :84): the
 * attention probabilities and the fc output are masked exactly as team_mha_fwd masks the token tensor
 * [image | text | state | C prototypes | P prompts] (L = 3 + C + P) of every sample: probability (b L + i) L + j with the
 * Philox stream (seed, offset), fc element (b L + i) 512 + c with (seed, offset + 1); kept iff the output is >= p 2^32,
 * kept values scaled by 1 / (1 - p).  Only the query tokens i < 3 + C are computed (the prompt outputs are discarded).
 * offset_dev, if not NULL, is read on the device and overrides offset (a replayed CUDA graph then draws the masks of
 * whatever offset the device holds).  workspace: team_head_dropout_workspace_bytes, untouched between the forward and
 * the backward of one step, 256-byte aligned.  p = 0 (or a NULL team_dropout*) runs the undropped head. */
typedef struct team_dropout {
    float p;
    uint64_t seed;
    uint64_t offset;
    const uint64_t* offset_dev;
    void* workspace;
    size_t workspace_bytes;
} team_dropout;
/* Bytes of the dropout workspace, linear in the batch: about (C + 1) B (10 Nsp + 7 200) + 12 B Nsp in BF16 mode and
 * (C + 1) B (8 Nsp + 6 176) + 8 B Nsp in F32 mode (Nsp = C + P + 10 rounded up to 16): 188 MB at B = 1024, C = 20, P = 100. */
size_t team_head_dropout_workspace_bytes(int64_t batch, int32_t num_classes, int32_t num_prompts, int mode);
/* *p += v on the device, on `stream` (one thread, no host sync; capturable): advances team_dropout.offset_dev by 2 per
 * step, so the replays of a captured step draw fresh masks. */
int team_u64_add(uint64_t* p, uint64_t v, void* stream);
/* Byte offset, inside the workspace of team_head_tri_fwd (same arguments as team_head_workspace_bytes), of the
 * [2B,512] fp32 rows normalize(encode_image(x)) | normalize(encode_text(t)) the forward leaves there (valid until the
 * matching team_head_tri_bwd): the inputs of the ClipLoss branch, models/proof.py:428-430. */
size_t team_head_own_rows_offset(int64_t batch, int32_t num_classes, int32_t num_prompts,
                                 int32_t num_text_cls, int mode);

/* image_feat/text_feat [B,512] fp32 (post-CLIP features; per-sample text), state_ids [B] int64.
 * Outputs (fp32): out_image [B,512], out_text [B,512] (the [B,1,512] view is the caller's),
 * out_state [B,512], out_proto [B,512].
 * If text_cls != NULL (fp32 [num_text_cls,512]) also computes the no-grad classification
 * logits cls_logits [B,num_text_cls] = normalize(encode_image(x)) @ normalize(encode_text(t)).T
 * and, if cls_argmax != NULL, their row argmax.
 * The workspace keeps the intermediates team_head_tri_bwd needs and must stay untouched
 * between the two calls. */
int team_head_tri_fwd(const team_head_weights* w, int mode, int64_t batch,
                      const float* image_feat, const float* text_feat, const int64_t* state_ids,
                      const float* text_cls, int64_t num_text_cls,
                      float* out_image, float* out_text, float* out_state, float* out_proto,
                      float* cls_logits, int64_t* cls_argmax,
                      void* workspace, size_t workspace_bytes, void* stream, const team_dropout* dropout);

/* g_proto may be NULL = a zero cotangent for the prototype output (what the learner's losses produce: neither
 * unicl_loss nor ClipLoss reads proto_feats, models/proof.py:434-442); heads of up to 22 classes then skip the C
 * prototype query rows of every sample in the backward, larger heads run them with a zero cotangent.
 * dropout: the team_dropout of the matching forward (same p, seed, offset and workspace). */
int team_head_tri_bwd(const team_head_weights* w, int mode, int64_t batch,
                      const float* image_feat, const float* text_feat, const int64_t* state_ids,
                      const float* g_image, const float* g_text, const float* g_state,
                      const float* g_proto, const team_head_grads* grads,
                      void* workspace, size_t workspace_bytes, void* stream, const team_dropout* dropout);

/* encode_* alone (utils/inc_net.py:401-422, :518-526): out = [normalize](sum_t x W_t^T + b_t).
 * which: 0 image, 1 text, 2 state (x = state_ids int64, embedding gather fused), 3 prototypes
 * (x ignored, rows = img_prototypes). */
int team_head_encode(const team_head_weights* w, int mode, int which, const void* x,
                     int64_t n_rows, int normalize, float* out,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Gradient of encode_image / encode_text (which = 0 | 1) w.r.t. the newest projection of that modality:
 * y = [normalize](x Wsum^T + bsum); g_w[512,512] = dz^T x, g_b[512] = colsum(dz) with dz = g_out or its
 * normalise-backward.  This is the autograd path of the ClipLoss branch (models/proof.py:428-431).
 * workspace: team_head_workspace_bytes(n_rows, C, P, 0, mode); team_head_encode takes the same size
 * (which <= 1) or the batch-1 size (which >= 2). */
int team_head_encode_bwd(const team_head_weights* w, int mode, int which, const float* x, int64_t n_rows,
                         int normalize, const float* g_out, float* g_w, float* g_b,
                         void* workspace, size_t workspace_bytes, void* stream);
/* The same for which = 0 | 1 | 2 (2 = state: x = the gathered embedding rows E[state_ids], fp32) with the optional
 * gradient w.r.t. the input rows g_x[n_rows,512] = dz Wsum (NULL = not needed): autograd of encode_state
 * (utils/inc_net.py:518-526; the caller folds g_x by state id into the embedding table, models/state_evolution.py:45-47)
 * and of encode_prototpyes (:417-422) in the differentiable PROOF / class-text forms. */
int team_head_encode_rows_bwd(const team_head_weights* w, int mode, int which, const float* x, int64_t n_rows,
                              int normalize, const float* g_out, float* g_w, float* g_b, float* g_x,
                              void* workspace, size_t workspace_bytes, void* stream);

/* PROOF fusion forward.
 * Replaces: Proof_Net.forward                     utils/inc_net.py:436-463
 *           Proof_Net.forward_transformer         utils/inc_net.py:465-492 (transformer=True; inputs_encoded = 1:
 *           image_feat / text_feat are then rows already produced by encode_image / encode_text(normalize=True))
 * tokens of sample b = [image_b | num_text class-text rows | C prototype rows | P prompt rows].
 * image_feat [B,512], text_feat [num_text,512] fp32.  Outputs (fp32): out_image [B,512],
 * out_text [num_text,512] and out_proto [C,512] = means over the batch of the text / prototype rows.
 * Forward only (the TEAM learner never calls this path, SURVEY 8a row a8).
 * workspace: team_head_workspace_bytes(batch, num_text + C, P, num_text, mode). */
int team_head_proof_fwd(const team_head_weights* w, int mode, int64_t batch, const float* image_feat,
                        const float* text_feat, int64_t num_text, int inputs_encoded,
                        float* out_image, float* out_text, float* out_proto,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Class-text form of forward_tri_modal (utils/inc_net.py:528-580 when text has num_text != batch rows: the text
 * rows are shared by all samples and the text output is the per-sample MEAN over them, :573-574).
 * image_feat [B,512], text_feat [num_text,512], state_ids [B] int64; outputs [B,512] each.  Forward only (the learner
 * always passes one text per sample, models/proof.py:421-425).
 * workspace: team_head_workspace_bytes(batch, num_text + C, P, num_text, mode). */
int team_head_tri_classtext_fwd(const team_head_weights* w, int mode, int64_t batch, const float* image_feat,
                                const float* text_feat, int64_t num_text, const int64_t* state_ids,
                                float* out_image, float* out_text, float* out_state, float* out_proto,
                                void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ exemplar herding (SURVEY 8f row 4)
 * Replaces: the selection loop of BaseLearner._construct_exemplar   models/base.py:284-311 and the exemplar mean :335-341.
 * feats [n_rows,512] fp32 = extract_vector outputs, rows grouped by class: group g owns rows [group_ptr[g], group_ptr[g+1])
 * (group_ptr: n_groups + 1 int64 on the device).  For every group: rows are L2-normalised (v / (||v|| + 1e-8)), the class mean
 * taken, and m exemplars picked greedily so that the running exemplar mean stays closest to the class mean (first index
 * on ties).  out_idx [n_groups,m] int64 = picked rows, relative to the group's first row, in pick order (-1 where a group has
 * fewer than m rows); out_mean [n_groups,512] = normalised mean of the picked normalised rows (the _class_means row);
 * out_class_mean (optional) [n_groups,512] = mean of all normalised rows.  One CTA per group. */
size_t team_herding_workspace_bytes(int64_t n_rows);
int team_herding_select(const float* feats, const int64_t* group_ptr, int32_t n_groups, int32_t m, int64_t n_rows,
                        int64_t* out_idx, float* out_mean, float* out_class_mean, void* workspace,
                        size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ standalone MultiHeadAttention (SURVEY 8a row a6)
 * Replaces: MultiHeadAttention.forward (+ ScaledDotProductAttention)   convs/projections.py:64-87, :31-38
 *           (n_head = 1, d_model = d_k = d_v = 512; eval mode and train mode with dropout) and its autograd backward.
 * out[B,Lq,512] = LayerNorm(fc(softmax(Q K^T / sqrt(512)) V) + q_in), Q = q_in Wq^T, K = k_in Wk^T, V = v_in Wv^T.
 * q_in [B,Lq,512], k_in / v_in [B,Lk,512] fp32 row-major; weights as nn.Linear stores them ([out,in]).
 * The forward saves what the backward needs in `workspace` (team_mha_workspace_bytes), which must be handed to
 * the matching team_mha_bwd unchanged.  The dense projections run on the mode's GEMM engine (tcgen05 in
 * TEAM_MODE_BF16), the per-sample attention core in fp32.  team_mha_bwd: g_q_in / g_k_in / g_v_in may be NULL; when
 * q_in, k_in, v_in are one tensor (self-attention) the caller adds the three input gradients.
 * Used by the differentiable PROOF fusion (utils/inc_net.py:436-492) and the class-text form of forward_tri_modal
 * (:544-547, :573-576); the learner's per-batch path runs the factorised kernels of team_head_tri_fwd instead. */
size_t team_mha_workspace_bytes(int64_t batch, int64_t len_q, int64_t len_k);
/* Train mode: dropout_p > 0 applies the block's two dropouts (attention probabilities, fc output; nn.Dropout(0.1) in the
 * reference, convs/projections.py:28, :62, :84) with counter-based Philox4x32-10 masks: element i of the probabilities is
 * kept iff philox(key = seed, counter = (i / 4, offset))[i % 4] >= p * 2^32, the fc output uses offset + 1; kept values are
 * scaled by 1 / (1 - p).  The backward regenerates the masks from the same (dropout_p, seed, offset).  A caller advances
 * `offset` by 2 per forward call.  dropout_p = 0: eval mode.  team_dropout_keep_mask writes the 0 / 1 mask of n elements. */
int team_mha_fwd(int mode, int64_t batch, int64_t len_q, int64_t len_k, const float* q_in, const float* k_in,
                 const float* v_in, const float* w_q, const float* w_k, const float* w_v, const float* w_fc,
                 const float* b_fc, const float* ln_g, const float* ln_b, float dropout_p, uint64_t seed,
                 uint64_t offset, float* out, void* workspace, size_t workspace_bytes, void* stream);
int team_mha_bwd(int mode, int64_t batch, int64_t len_q, int64_t len_k, const float* q_in, const float* k_in,
                 const float* v_in, const float* w_q, const float* w_k, const float* w_v, const float* w_fc,
                 const float* ln_g, float dropout_p, uint64_t seed, uint64_t offset, const float* g_out,
                 float* g_q_in, float* g_k_in, float* g_v_in, float* g_w_q, float* g_w_k, float* g_w_v,
                 float* g_w_fc, float* g_b_fc, float* g_ln_g, float* g_ln_b, void* workspace,
                 size_t workspace_bytes, void* stream);
int team_dropout_keep_mask(unsigned char* keep, int64_t n, float dropout_p, uint64_t seed, uint64_t offset, void* stream);
/* torch.mean over the middle dimension of x[outer][red][inner] -> out[outer][inner] (serial fixed-order sums: the batch
 * means of Proof_Net.forward, utils/inc_net.py:458-459, and the row means of forward_tri_modal, :573-576) and its
 * backward dx[o][r][i] = g[o][i] / red. */
int team_mean_mid(const float* x, float* out, int64_t outer, int64_t red, int64_t inner, void* stream);
int team_mean_mid_bwd(const float* g, float* dx, int64_t outer, int64_t red, int64_t inner, void* stream);

/* ------------------------------------------------------------------ losses of the training step (SURVEY 8f "next")
 * Replaces: unicl_loss                                     models/proof.py:21-191, called at :434-441
 *           ClipLoss.forward (world_size 1)               utils/toolkit.py:128-141, called at :431
 * Both return the loss value(s) on the device AND the gradient w.r.t. their feature inputs times grad_scale (the
 * learner's weights: total = ce + clip + 0.3 unicl, models/proof.py:442), i.e. the cotangents of team_head_tri_bwd /
 * team_head_encode_bwd - loss forward and backward are one call.  batch <= 16384 (B x B similarities).
 * team_unicl_loss: image/text/state [B,512] fp32 as returned by forward_tri_modal (un-normalised), labels [B] int64,
 *   temperature = the dynamic temperature of :111-116 (host scalar); losses[3] = {total, instance, category}.
 * team_clip_loss: image/text [B,512] as handed to ClipLoss (the learner normalises them first), logit_scale host scalar. */
size_t team_loss_workspace_bytes(int64_t batch);
/* Value of the classification cross-entropy (models/proof.py:417; mean over the batch of lse(logits) - logits[label]; no
 * gradient: the logits are computed under no_grad, :411-416) and the learner's total loss (:442) in one launch:
 * losses6 = [total, ce, clip, unicl, unicl_instance, unicl_category]; entries 2..5 are INPUTS (written before by
 * team_clip_loss -> losses6 + 2 and team_unicl_loss(_evo) -> losses6 + 3); total = ce + w_clip * clip + w_unicl * unicl. */
int team_ce_total(const float* logits, const int64_t* labels, int64_t batch, int64_t num_classes, float w_clip,
                  float w_unicl, float* losses6, void* stream);
int team_unicl_loss(int mode, const float* image, const float* text, const float* state, const int64_t* labels,
                    int64_t batch, float temperature, float grad_scale, float* losses,
                    float* g_image, float* g_text, float* g_state,
                    void* workspace, size_t workspace_bytes, void* stream);
/* unicl_loss with evolution_features (models/proof.py:51-106 - what the learner always passes once
 * evolve_state_prototypes() has run, :435-441): the normalised state rows are first enhanced per class with the
 * class's evolution feature and, when the class occurs with >= 2 life stages in the batch, a time-weighted mixture of
 * the class's other state rows; the gradient flows back through the enhancement into every contributing state row.
 * state_ids [B] int64 in [0,10); evo [num_evo,512] fp32 (row c = evolution_features[c]); evo_mask [num_evo] bytes
 * (0 = evolution_features[c] is None).  Classes >= num_evo are left alone like in the reference.  Everything runs on
 * the device (keyed sums over (class, state) instead of the reference's host loops).
 * workspace: team_loss_evo_workspace_bytes(batch, num_evo). */
size_t team_loss_evo_workspace_bytes(int64_t batch, int num_evo);
int team_unicl_loss_evo(int mode, const float* image, const float* text, const float* state, const int64_t* labels,
                        const int64_t* state_ids, const float* evo, const unsigned char* evo_mask, int num_evo,
                        int64_t batch, float temperature, float grad_scale, float* losses,
                        float* g_image, float* g_text, float* g_state,
                        void* workspace, size_t workspace_bytes, void* stream);
int team_clip_loss(int mode, const float* image, const float* text, int64_t batch, float logit_scale, float grad_scale,
                   float* loss, float* g_image, float* g_text,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ the same losses under data parallelism
 * `world` ranks hold `batch` samples each; the global batch is their concatenation in rank order (Bg = world * batch).
 * Every rank computes the rows of its own samples against the columns of the whole global batch, so together the
 * ranks compute what team_clip_loss + team_unicl_loss(_evo) + team_ce_total compute on one GPU at batch Bg:
 *   - losses6 = [total, ce, clip, unicl, unicl_instance, unicl_category], the same values on every rank,
 *     total = ce + w_clip * clip + w_unicl * unicl;
 *   - the gradient of that total w.r.t. this rank's rows: g_image / g_text / g_state (the cotangents of the head's three
 *     feature outputs, unicl) and g_own_rows [2B,512] (image rows, then text rows: ClipLoss on the normalised own rows,
 *     team_head_grads.g_own_rows).  The head's parameter gradient is then the SUM over ranks of each rank's backward.
 * The call is split into phases with an exchange between consecutive ones: phase p writes this rank's slice of exchange
 * p into send[p] (team_loss_shard_xchg_bytes(.., p) bytes), the caller all-gathers the slices of all ranks in rank order
 * into gathered[p] (world * that many bytes), and phase p + 1 reads it.  Nothing is reduced by the exchange: every sum
 * over ranks is folded in rank order by the next phase, so the results are deterministic and identical on all ranks.
 *   exchange 0: per sample [normalised image row | own image row | own text row | label]: the GEMM operands of the B x Bg
 *               blocks, bf16 in TEAM_MODE_BF16 and fp32 in TEAM_MODE_F32
 *   exchange 1: per-row statistics (ClipLoss logsumexps, unicl category max / positive / all / valid), the loss partial
 *               sums and, with evolution features, the (class, state) keyed sums and counts of the state rows
 *   exchange 2: (evolution features only) the keyed sums of the mixture gradients and the unicl instance loss partial
 * Phases: team_loss_shard_phases(num_evo) = 3 without evolution features, 4 with them.  All gathered buffers must stay
 * intact until the last phase; the workspace carries state from phase to phase (same struct, same workspace).
 * Limits: 1 <= batch <= 16384, 2 <= Bg <= 65536 (the B x Bg similarity and coefficient blocks live in the workspace),
 * world <= 64.  Equal shards only.  world = 1 is the single-GPU computation.  Pointers: see the fields. */
typedef struct team_loss_shard {
    int32_t mode;                  /* TEAM_MODE_F32 / TEAM_MODE_BF16 */
    int32_t rank, world;
    int32_t num_evo;               /* rows of evo; 0 = no evolution features */
    int64_t batch;                 /* samples per rank */
    int64_t num_classes;           /* columns of logits */
    const float* image;            /* [B,512] head outputs (un-normalised), as team_unicl_loss */
    const float* text;
    const float* state;
    const float* own_rows;         /* [2B,512] normalised own rows (image, then text), as team_clip_loss's inputs */
    const float* logits;           /* [B,num_classes] classification logits (value only) */
    const int64_t* labels;         /* [B] */
    const int64_t* state_ids;      /* [B] in [0,10); read only with evolution features */
    const float* evo;              /* [num_evo,512] */
    const unsigned char* evo_mask; /* [num_evo] */
    float temperature, logit_scale, w_clip, w_unicl;
    void* send[3];                 /* this rank's slice of exchange p (written by phase p) */
    const void* gathered[3];       /* all ranks' slices of exchange p in rank order (read by phases > p) */
    float* g_image;                /* [B,512] outputs, OVERWRITTEN */
    float* g_text;
    float* g_state;
    float* g_own_rows;             /* [2B,512] */
    float* losses6;                /* [6], written by the last phase */
    void* workspace;               /* 256-byte aligned */
    size_t workspace_bytes;
} team_loss_shard;
int team_loss_shard_phases(int32_t num_evo);
size_t team_loss_shard_workspace_bytes(int32_t mode, int64_t batch, int32_t world, int32_t num_evo);
/* bytes of ONE rank's slice of exchange `exchange` (0 = no such exchange) */
size_t team_loss_shard_xchg_bytes(int32_t mode, int64_t batch, int32_t num_evo, int32_t exchange);
int team_loss_shard_run(int32_t phase, const team_loss_shard* s, void* stream);

/* Fused multi-tensor AdamW step (SURVEY 8f "next").
 * Replaces: torch.optim.AdamW(...).step()    models/proof.py:361, :445  (decoupled weight decay, bias correction,
 * amsgrad off).  params / grads / exp_avg / exp_avg_sq: HOST arrays of n_tensors device pointers (fp32, numel[i]
 * elements each, at most 48 per call); step = 1 for the first update.  One launch, element-wise, capturable. */
int team_adamw_step(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                    float* const* exp_avg_sq, const int64_t* numel, float lr, float beta1, float beta2, float eps,
                    float weight_decay, int64_t step, void* stream);
/* The same update for a CUDA graph that is replayed every step: the step count t lives in device memory (*step_dev =
 * number of updates done so far, int64), the bias corrections are computed from it on the device; with advance != 0 a
 * one-thread kernel increments it behind the update (pass 0 for all but the last call of a step with > 48 tensors). */
int team_adamw_step_graph(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                          float* const* exp_avg_sq, const int64_t* numel, float lr, float beta1, float beta2, float eps,
                          float weight_decay, int64_t* step_dev, int32_t advance, void* stream);

/* ------------------------------------------------------------------ gradient all-reduce over NVLink peer memory
 * The reference has no working multi-GPU path (its nn.DataParallel wrap crashes, models/proof.py:312-313 vs :248);
 * this is the exchange step of the data-parallel training step (the sum autograd would produce on one big batch,
 * models/proof.py:444).  In-place sum of n fp32 values: bufs[r] / flags[r] (r < world, HOST arrays of device
 * pointers) are every rank's buffer and flag array as mapped on THIS device (symmetric memory); flags are
 * team_peer_allreduce_flag_bytes() bytes each (two channels), zeroed once before the first call.  One kernel, two-shot, summed in
 * rank order (bit-identical on all ranks); every rank must make the matching call.  n % 4 == 0.
 * multicast: NVLS multicast mapping of the same buffers (NULL = none): the switch then adds (multimem.ld_reduce)
 * and replicates (multimem.st); the sum order is the switch's, still identical on all ranks. */
size_t team_peer_allreduce_flag_bytes(void);
int team_peer_allreduce_f32(void* const* bufs, void* const* flags, void* multicast, int32_t rank, int32_t world,
                            int64_t n, void* stream);
/* A peer that never arrives is waited for until a device-clock deadline (environment TEAM_PEER_TIMEOUT_S, default
 * 1800 s, 0 = for ever); the kernel then gives up WITHOUT trapping (the context stays usable).  This call
 * synchronises `stream` and returns this rank's status word: 0 = all exchanges completed, otherwise
 * 1 + (phase << 8) + (peer << 16) of the first wait that timed out.  own_flags = flags[rank]. */
int team_peer_allreduce_status(const void* own_flags, void* stream, uint32_t* status);
/* All-gather of one slice of slice_bytes bytes per rank over NVLink peer memory: the exchanges between the phases of
 * team_loss_shard_run inside a captured training step.  bufs[r] / flags[r] (r < world, HOST arrays of device pointers)
 * are every rank's gathered buffer (world * slice_bytes bytes, rank-major) and flag array as mapped on THIS device
 * (symmetric memory); flags are team_peer_allreduce_flag_bytes() bytes each, zeroed once before the first call, and
 * must not be the arrays of an all-reduce.  Rank r's own slice must already be in slot r of bufs[rank] (bytes
 * [rank * slice_bytes, (rank + 1) * slice_bytes)): the kernel stores it into slot r of every peer's buffer and never
 * copies locally.  One kernel, bit-exact (no arithmetic), safe to call again on the same buffers (the kernel waits
 * until every rank has finished reading before any slot is overwritten); every rank must make the matching call.
 * slice_bytes % 16 == 0 (every team_loss_shard_xchg_bytes size is), world <= 8; world == 1 is a no-op.
 * multicast: NVLS multicast mapping of the same buffers (NULL = none): each rank then sends its slice once and the
 * switch replicates it.  Health: team_peer_allreduce_status on flags[rank]. */
int team_peer_allgather(void* const* bufs, void* const* flags, void* multicast, int32_t rank, int32_t world,
                        int64_t slice_bytes, void* stream);

/* ------------------------------------------------------------------ temporal GCN + state distances
 * Replaces: TemporalStateGCN.forward / TemporalGCNBlock.forward   models/dynamic_modal_graph.py:239-337
 *           (called under no_grad from InsectLifecycleModel.evolve_and_update, models/state_evolution.py:326-327).
 * Edges arrive as a destination-sorted CSR (rowptr[N+1], src[E], edge_w[E]) that keeps the reference's
 * edge order inside every destination (intra-class edges first, then inter-class, each by source index).
 * out[N,512] = L2-normalised evolved node features. */
typedef struct team_tgcn_block {
    const float* msg_w;  const float* msg_b;  const float* msg_ln_g;  const float* msg_ln_b;   /* message_net: [320,640],[320],[320],[320] */
    const float* upd_w;  const float* upd_b;  const float* upd_ln_g;  const float* upd_ln_b;   /* update_net */
    const float* gate_w; const float* gate_b;                                                   /* temporal_gate: [1,320],[1] */
} team_tgcn_block;
typedef struct team_tgcn_weights {
    const float* node_w; const float* node_b; const float* node_ln_g; const float* node_ln_b;  /* node_encoder: [256,512],[256],[256],[256] */
    const float* time_w; const float* time_b; const float* time_ln_g; const float* time_ln_b;  /* time_encoder: [64,1],[64],[64],[64] */
    team_tgcn_block blocks[8];
    int32_t num_blocks;
    int32_t reserved;
    const float* out_w;  const float* out_b;                                                     /* output_proj: [512,320],[512] */
} team_tgcn_weights;
size_t team_tgcn_workspace_bytes(int64_t n_nodes);
int team_tgcn_forward(const team_tgcn_weights* w, const float* node_feat, const float* time_steps,
                      int64_t n_nodes, const int32_t* rowptr, const int32_t* src, const float* edge_w,
                      float* out, void* workspace, size_t workspace_bytes, void* stream);
/* d_ij = 1 - cosine(u_i,u_j) for every ordered pair i != j, summed per (state_i,state_j) in double
 * (models/state_evolution.py:345-364).  sums[100] double, counts[100] int64, row-major [state_i][state_j].
 * workspace >= n_nodes*10*12 + 256 bytes. */
int team_pairwise_state_dist(const float* node_feat, const int32_t* node_states, int64_t n_nodes,
                             double* sums, int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);
/* Proof_Net._sync_class_prototypes (utils/inc_net.py:600-617): nodes grouped by class (group_ptr CSR);
 * img_prototypes[group_class[g]] = normalize(sum_i w_i p_i / sum w), w = 1.5 for state 4 else 1. */
int team_sync_prototypes(const float* nodes, const int32_t* group_ptr, const int32_t* node_states,
                         const int32_t* group_class, int64_t n_groups, float* img_prototypes, void* stream);
int team_rows_normalize(float* x, int64_t n_rows, void* stream);
/* out[g] = mean of nodes[member[i]] over i in [group_ptr[g], group_ptr[g+1]) (member NULL = identity):
 * class embeddings / lifecycle features of evolve_and_update (models/state_evolution.py:256-258, :334-343). */
int team_group_mean(const float* nodes, const int32_t* group_ptr, const int32_t* member, int64_t n_groups,
                    float* out, void* stream);
/* AdaptiveStateDistanceMatrix.get_distance_matrix (utils/state_distance.py:65-71) */
int team_dist_matrix(const float* factors, int32_t n, float* out, void* stream);
/* Learner.update_state_distance_matrix EMA (models/proof.py:666-675), sequential over (keys[e], vals[e]) */
int team_dist_ema(float* factors, int32_t n, const int32_t* keys, const double* vals, int32_t m, double weight,
                  void* stream);
/* AdaptiveStateDistanceMatrix.forward update branch (utils/state_distance.py:96-134): per-state sums/counts
 * (from team_segsum with key = state id) -> centres -> 2 - cosine -> sequential EMA into factors[10,10];
 * pre_update_matrix (optional) receives get_distance_matrix() of the factors BEFORE the update. */
int team_state_dist_forward(const float* state_sums, const int64_t* state_counts, float* factors, double decay,
                            float* pre_update_matrix, void* stream);
/* DynamicGCN.forward, eval mode (models/dynamic_modal_graph.py:131-163) */
typedef struct team_dgcn_layer {
    const float* w; const float* b; const float* ln_g; const float* ln_b;
    int32_t in_dim; int32_t out_dim;
} team_dgcn_layer;
size_t team_dgcn_workspace_bytes(int64_t n_nodes, int32_t max_dim);
int team_dgcn_forward(const team_dgcn_layer* layers, int32_t n_layers, const float* x, int64_t n_nodes,
                      const int32_t* rowptr, const int32_t* src, const float* edge_w, float* out,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ generic GEMM (tests/bench)
 * C[M,N] = alpha * op(A) op(B) + beta * C (+ bias[N]);  fp32 SIMT path.
 * ta: 0 -> A is [M,K] row-major (lda), 1 -> A is [K,M] row-major.
 * tb: 0 -> B is [K,N] row-major (ldb), 1 -> B is [N,K] row-major. */
int team_gemm_f32(int ta, int tb, int64_t M, int64_t N, int64_t K, float alpha,
                  const float* A, int64_t lda, const float* B, int64_t ldb, float beta,
                  float* C, int64_t ldc, const float* bias, void* workspace,
                  size_t workspace_bytes, void* stream);
/* tcgen05 + TMA + TMEM GEMM: C[M,N] fp32 = alpha * op(A) op(B) (+bias[N]) (+beta*C), bf16 operands.
 * a_mn = 0: A stored [M,K] row-major (K-major); a_mn = 1: A stored [K,M] row-major (M-major).
 * b_mn = 0: B stored [N,K] row-major (K-major); b_mn = 1: B stored [K,N] row-major (N-major).
 * A_lo (optional) is the low half of a two-term bf16 split of an fp32 A: C = (A + A_lo) B. */
int team_gemm_bf16(int a_mn, int b_mn, int64_t M, int64_t N, int64_t K, float alpha, const void* A,
                   const void* A_lo, int64_t lda, const void* B, int64_t ldb, float beta, float* C,
                   int64_t ldc, const float* bias, void* workspace, size_t workspace_bytes, void* stream);
/* Grouped form: n independent problems in as few launches as possible (8 problems per launch), each
 * C = alpha op(A) op(B) (+bias) (+beta C) written as fp32 (C) and/or bf16 (C_bf16); split-K is folded
 * inside the kernel in a fixed order (deterministic).  workspace: >= 16 KiB + room for split-K partials
 * (without it long-K problems simply run unsplit). */
typedef struct team_gemm_desc {
    int32_t a_mn, b_mn;
    int64_t M, N, K;
    float alpha, beta;
    const void* A; int64_t lda;
    const void* B; int64_t ldb;
    float* C; int64_t ldc;
    void* C_bf16; int64_t ldc_bf16;
    const float* bias;
    /* optional second K-segment accumulated into the same output tile: C = alpha (op(A) op(B) + op(A2) op(B2)) ...
     * (K2 = 0: none).  Lets dW = dQo^T Xo + dQs^T S run as one problem. */
    int32_t a_mn2, b_mn2;
    int64_t K2;
    const void* A2; int64_t lda2;
    const void* B2; int64_t ldb2;
} team_gemm_desc;
int team_gemm_bf16_group(const team_gemm_desc* descs, int32_t n, void* workspace, size_t workspace_bytes, void* stream);
/* One launch that copies a device-resident batch (image / text rows [B,512] fp32, state ids / labels [B] int64) into the static
 * input buffers of a captured step (train.TrainStep.load): replaces four device-to-device copies between graph replays. */
int team_copy_batch(const float* image, const float* text, const int64_t* state_ids, const int64_t* labels, int64_t batch,
                    float* d_image, float* d_text, int64_t* d_state_ids, int64_t* d_labels, void* stream);
/* debugging aid: if buf != NULL (32 x 1024 x 16 uint64) every GEMM CTA writes globaltimer stamps of its phases into the slot of its launch (tools/wave_stamps.py) */
int team_gemm_debug_stamps(void* buf);
/* fp32 [rows,cols] -> bf16 hi (and optional lo residual) */
int team_f32_to_bf16(const float* src, int64_t lds, int64_t rows, int64_t cols, void* hi, void* lo,
                     int64_t ldd, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TEAM_B200_H */
