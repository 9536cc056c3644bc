"""CPU oracle for the TEAM head hot path (TEST INFRASTRUCTURE - not the product).

A plain-PyTorch (CPU, fp32 or fp64) restatement of the reference algorithm for the
path named by BASELINE.json:north_star, written *as the reference computes it*
(replicated shared rows, full L x L attention, Python loops over edges / node pairs),
so it doubles as the "port" CPU baseline of ``bench.py``.  Every function cites the
reference file:line it follows.  The reference is 100 % Python/torch, its arithmetic
lives in the third-party dependency ``torch`` (unpinned by the reference; this image
ships 2.11 CPU kernels).

Parity pin: the reference has no tests or golden vectors (SURVEY.md 8c).  The oracle
is pinned against *outputs of the reference itself run in the build container*:
``oracle/gen_golden.py`` imports ``/root/reference`` (with timm / matplotlib /
open_clip stubbed), feeds it the seeded tensors of ``oracle/synth.py`` and commits the
results under ``tests/golden``; ``tests/test_oracle_golden.py`` checks every oracle
function against them.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` legs may import this module.  The product path
(``team_b200``) never does.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Params = Dict[str, torch.Tensor]

LN_EPS = 1e-5          # nn.LayerNorm default (convs/projections.py:58)
NORM_EPS = 1e-12       # F.normalize default
COS_EPS = 1e-8         # F.cosine_similarity default


def num_tasks(p: Params) -> int:
    t = 0
    while f"projs_img.{t}.MLP.0.weight" in p:
        t += 1
    return t


def cast_params(p: Params, dtype) -> Params:
    return {k: v.to(dtype) if v.is_floating_point() else v for k, v in p.items()}


# --------------------------------------------------------------------------- a1-a5
def proj_sum(x: torch.Tensor, p: Params, kind: str) -> torch.Tensor:
    """sum_t proj_t(x): utils/inc_net.py:404-406, :412-414, :419-421, :521-523
    (list of Proj_Pure_MLP = nn.Linear, convs/projections.py:7-18; stack dim=1; sum)."""
    feats = [F.linear(x, p[f"projs_{kind}.{t}.MLP.0.weight"], p[f"projs_{kind}.{t}.MLP.0.bias"])
             for t in range(num_tasks(p))]
    return torch.sum(torch.stack(feats, dim=1), dim=1)


def encode_image(x, p: Params, normalize=False):
    """utils/inc_net.py:401-407 (the frozen CLIP tower is the identity on features)."""
    f = proj_sum(x, p, "img")
    return F.normalize(f, dim=-1) if normalize else f


def encode_text(x, p: Params, normalize=False):
    """utils/inc_net.py:409-415."""
    f = proj_sum(x, p, "text")
    return F.normalize(f, dim=-1) if normalize else f


def encode_prototypes(protos, p: Params, normalize=False):
    """utils/inc_net.py:417-422 (uses the *image* projections)."""
    f = proj_sum(protos, p, "img")
    return F.normalize(f, dim=-1) if normalize else f


def encode_state(state_ids, p: Params, normalize=False):
    """utils/inc_net.py:518-526 + models/state_evolution.py:45-47 (nn.Embedding lookup)."""
    e = F.embedding(state_ids, p["state_embedder.state_embeddings.weight"])
    f = proj_sum(e, p, "state")
    return F.normalize(f, dim=1) if normalize else f


def context_prompts(p: Params) -> torch.Tensor:
    """utils/inc_net.py:398-399."""
    return torch.cat([p[f"context_prompts.{t}"] for t in range(num_tasks(p))], dim=0)


# --------------------------------------------------------------------------- a6
def philox4x32_10(c0, c1, c2, c3, k0: int, k1: int):
    """Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11; Random123):
    multipliers 0xD2511F53 / 0xCD9E8D57, Weyl key increments 0x9E3779B9 / 0xBB67AE85, ten rounds.  Counter words as numpy
    uint64 arrays holding 32-bit values; returns the four output words.  Pinned by the Random123 known-answer vectors
    (tests/test_oracle_golden.py)."""
    import numpy as np
    M32 = np.uint64(0xFFFFFFFF)
    c = [np.asarray(x, dtype=np.uint64) for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0 & 0xFFFFFFFF), np.uint64(k1 & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c


def philox_keep_mask(n: int, dropout_p: float, seed: int, offset: int):
    """0 / 1 keep mask of n elements as the library defines it (include/team_b200.h: team_mha_fwd): element i is kept iff
    philox4x32_10(counter = (i // 4 low, i // 4 high, offset low, offset high), key = (seed low, seed high))[i % 4]
    >= dropout_p * 2**32."""
    import numpy as np
    nb = (n + 3) // 4
    blk = np.arange(nb, dtype=np.uint64)
    c = philox4x32_10(blk & np.uint64(0xFFFFFFFF), blk >> np.uint64(32), np.full(nb, offset & 0xFFFFFFFF, np.uint64),
                      np.full(nb, (offset >> 32) & 0xFFFFFFFF, np.uint64), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    out = np.stack(c, axis=1).reshape(-1)[:n]
    thr = min(int(dropout_p * 4294967296.0), 4294967295)
    return torch.from_numpy((out >= np.uint64(thr)).astype(np.float64))


def mha(q_in: torch.Tensor, k_in: torch.Tensor, v_in: torch.Tensor, p: Params, drop=None) -> torch.Tensor:
    """MultiHeadAttention(n_head=1).forward(q, k, v): convs/projections.py:64-87 with ScaledDotProductAttention :31-38
    (temperature sqrt(512) :57; the discarded log_softmax :34 is omitted).  ``drop`` = None: eval mode (both nn.Dropout
    are the identity); ``drop`` = (p, seed, offset): train mode - the reference's two dropouts (attention probabilities
    :35, fc output :84) with EXPLICIT masks (philox_keep_mask; torch's own mask stream is not reproducible)."""
    d = q_in.shape[-1]
    q = F.linear(q_in, p["sel_attn.w_qs.weight"])
    k = F.linear(k_in, p["sel_attn.w_ks.weight"])
    v = F.linear(v_in, p["sel_attn.w_vs.weight"])
    attn = torch.bmm(q, k.transpose(1, 2)) / float(d ** 0.5)
    attn = torch.softmax(attn, dim=2)
    if drop is not None:
        pd, seed, offset = drop
        attn = attn * philox_keep_mask(attn.numel(), pd, seed, offset).reshape(attn.shape).to(attn.dtype) / (1.0 - pd)
    out = torch.bmm(attn, v)
    out = F.linear(out, p["sel_attn.fc.weight"], p["sel_attn.fc.bias"])
    if drop is not None:
        out = out * philox_keep_mask(out.numel(), pd, seed, offset + 1).reshape(out.shape).to(out.dtype) / (1.0 - pd)
    return F.layer_norm(out + q_in, (d,), p["sel_attn.layer_norm.weight"],
                        p["sel_attn.layer_norm.bias"], LN_EPS)


def sel_attn(x: torch.Tensor, p: Params) -> torch.Tensor:
    """sel_attn(features, features, features) as Proof_Net calls it (utils/inc_net.py:453, :559)."""
    return mha(x, x, x, p)


# --------------------------------------------------------------------------- a7
def forward_tri_modal(p: Params, image, text, state_ids, img_prototypes):
    """Proof_Net.forward_tri_modal: utils/inc_net.py:528-580.
    Returns (image[B,D], text[B,1,D] or [B,D], state[B,D], proto[B,D], exp(logit_scale))."""
    d = image.shape[-1]
    imf = encode_image(image, p, True)
    txf = encode_text(text, p, True)
    stf = encode_state(state_ids, p, True)
    prf = encode_prototypes(img_prototypes, p, True)
    cp = context_prompts(p)
    len_texts, len_protos = txf.shape[0], prf.shape[0]
    B = imf.shape[0]
    imf = imf.view(B, 1, d)
    stf = stf.view(B, 1, d)
    if txf.shape[0] == B:
        txf = txf.unsqueeze(1)
    else:
        txf = txf.view(txf.shape[0], d).expand(B, txf.shape[0], d)
    prf = prf.view(len_protos, d).expand(B, len_protos, d)
    cp = cp.view(cp.shape[0], d).expand(B, cp.shape[0], d)
    feats = torch.cat([imf, txf, stf, prf, cp], dim=1)
    feats = sel_attn(feats, p)
    if txf.shape[1] == 1:
        t_end = 2
    else:
        t_end = 1 + len_texts
    s_idx = t_end
    img_o = feats[:, 0]
    txt_o = feats[:, 1:t_end]
    st_o = feats[:, s_idx]
    pr_o = feats[:, s_idx + 1:s_idx + 1 + len_protos]
    if txt_o.shape[1] > 1:
        txt_o = torch.mean(txt_o, dim=1)
    if pr_o.shape[1] > 1:
        pr_o = torch.mean(pr_o, dim=1)
    return img_o, txt_o, st_o, pr_o, p["convnet.logit_scale"].exp()


# --------------------------------------------------------------------------- a8
def forward_proof(p: Params, image, text, img_prototypes):
    """Proof_Net.forward (PROOF fusion): utils/inc_net.py:436-463.
    Returns (image[B,D], text[C,D] batch-mean, exp(ls), proto[C,D] batch-mean)."""
    d = image.shape[-1]
    imf = encode_image(image, p, True)
    txf = encode_text(text, p, True)
    prf = encode_prototypes(img_prototypes, p, True)
    cp = context_prompts(p)
    nt, npr = txf.shape[0], prf.shape[0]
    B = imf.shape[0]
    feats = torch.cat([imf.view(B, -1, d), txf.view(nt, d).expand(B, nt, d),
                       prf.view(npr, d).expand(B, npr, d),
                       cp.view(cp.shape[0], d).expand(B, cp.shape[0], d)], dim=1)
    feats = sel_attn(feats, p)
    img_o = feats[:, 0, :]
    txt_o = torch.mean(feats[:, 1:nt + 1, :], dim=0)
    pr_o = torch.mean(feats[:, nt + 1:nt + 1 + npr, :], dim=0)
    return img_o.view(B, -1), txt_o.view(nt, -1), p["convnet.logit_scale"].exp(), pr_o.view(npr, -1)


# --------------------------------------------------------------------------- 8f: exemplar herding
def herding_select(features, m: int):
    """Selection loop and exemplar mean of BaseLearner._construct_exemplar for ONE class: models/base.py:284-311 (normalise
    with EPSILON = 1e-8 :12, class mean, greedy argmin with np.delete) and :335-341 (exemplar mean).  ``features`` =
    extract_vector outputs [n,512] (numpy float32, as tensor2numpy returns them).  Returns (indices into the ORIGINAL rows
    in pick order, normalised exemplar mean, class mean)."""
    import numpy as np
    vectors = np.asarray(features, dtype=np.float32)
    vectors = (vectors.T / (np.linalg.norm(vectors.T, axis=0) + 1e-8)).T
    all_vectors = vectors
    class_mean = np.mean(vectors, axis=0)
    alive = np.arange(vectors.shape[0])
    picked, exemplar_vectors = [], []
    for k in range(1, m + 1):
        S = np.sum(exemplar_vectors, axis=0)
        mu_p = (vectors + S) / k
        i = int(np.argmin(np.sqrt(np.sum((class_mean - mu_p) ** 2, axis=1))))
        picked.append(int(alive[i]))
        exemplar_vectors.append(np.array(vectors[i]))
        vectors = np.delete(vectors, i, axis=0)
        alive = np.delete(alive, i)
    sel = all_vectors[picked]
    mean = np.mean(sel, axis=0)
    mean = mean / np.linalg.norm(mean)
    return np.asarray(picked, dtype=np.int64), mean, class_mean


# --------------------------------------------------------------------------- 8f: losses of the training step
def unicl_loss(image_features, text_features, state_features, labels, temperature=0.07, epoch=None, max_epoch=None,
               state_ids=None, evolution_features=None):
    """unicl_loss: models/proof.py:21-191 (evolution_features branch: enhance_state_features) (normalise :44-46, dynamic temperature
    :111-116, instance term :126-149 incl. the exp(row_sim * mask) quirk (the masked self entry counts as
    exp(0) = 1), category term :151-174, weights :177-179).  Returns (total, instance, category) as tensors."""
    B = image_features.shape[0]
    im = F.normalize(image_features.reshape(B, -1), dim=1)
    tx = F.normalize(text_features.reshape(B, -1), dim=1)
    st = F.normalize(state_features.reshape(B, -1), dim=1)
    if evolution_features is not None and len(evolution_features) > 0:
        st = enhance_state_features(st, labels, state_ids, evolution_features)
    if epoch is not None and max_epoch is not None:
        progress = float(epoch) / float(max_epoch)
        tau = temperature * (0.5 + 0.5 * 0.5 * (1.0 + math.cos(math.pi * progress)))
    else:
        tau = temperature
    tri = torch.stack([im, tx, st], dim=1)                       # [B,3,D]
    sim = torch.matmul(tri, tri.transpose(1, 2)) / tau           # [B,3,3]
    eye = torch.eye(3, dtype=sim.dtype, device=sim.device)
    pos = torch.exp(sim * (1 - eye)).sum(-1)                     # self entry -> exp(0)
    allv = torch.exp(sim).sum(-1)
    instance = -(torch.log(pos / (allv + 1e-8))).sum() / (3 * B)
    lm = (labels.unsqueeze(1) == labels.unsqueeze(0)).to(sim.dtype)
    sm = 1 - torch.eye(B, dtype=sim.dtype, device=sim.device)
    lm = lm * sm
    ii = im @ im.t() / tau
    ex = torch.exp(ii - ii.max(dim=1, keepdim=True).values)
    p = (ex * lm).sum(1)
    a = (ex * sm).sum(1)
    valid = (p > 0) & (a > 0)
    if bool(valid.any()):
        category = -(torch.log(p[valid] / (a[valid] + 1e-8))).sum() / int(valid.sum())
    else:
        category = torch.zeros((), dtype=sim.dtype)
    return instance + 0.5 * category, instance, category


def enhance_state_features(state_features, labels, state_ids, evolution_features):
    """The `evolution_features` branch of unicl_loss: models/proof.py:51-106.  `state_features` are the NORMALISED state
    rows; returns the enhanced rows (differentiable).  Per class present in the batch with an evolution feature:
      one sample  -> normalize(0.8 s + 0.2 normalize(evo))                                               (:100-103)
      >= 2 samples with >= 2 distinct states -> time position of a state = its rank / (n_states - 1);
          mixture_i = evo + sum_{j != i, w_ij > 0.3} 0.2 w_ij s_j,  w_ij = 1 - |t_i - t_j|;
          row_i = normalize(0.7 s_i + 0.3 normalize(mixture_i))                                           (:79-98)
      >= 2 samples, one distinct state -> unchanged                                                        (:76 guard)
    Mixtures read the ORIGINAL rows (state_features), never rows already enhanced in this call (:92)."""
    out = state_features.clone()
    by_class = {}
    for i, c in enumerate(labels.tolist()):
        by_class.setdefault(c, []).append(i)
    for c, idx in by_class.items():
        if c >= len(evolution_features) or evolution_features[c] is None:
            continue
        evo = evolution_features[c].to(state_features.dtype)
        if len(idx) >= 2:
            states = [int(state_ids[i]) for i in idx]
            uniq = sorted(set(states))
            if len(uniq) < 2:
                continue
            tpos = {s: k / (len(uniq) - 1) for k, s in enumerate(uniq)}
            for a, i in enumerate(idx):
                mix = evo.clone()
                for b2, j in enumerate(idx):
                    if a == b2:
                        continue
                    w = 1.0 - abs(tpos[states[a]] - tpos[states[b2]])
                    if w > 0.3:
                        mix = mix + w * 0.2 * state_features[j]
                out[i] = F.normalize(0.7 * state_features[i] + 0.3 * F.normalize(mix, dim=0), dim=0)
        else:
            i = idx[0]
            out[i] = F.normalize(0.8 * state_features[i] + 0.2 * F.normalize(evo, dim=0), dim=0)
    return out


def clip_loss(image_features, text_features, logit_scale):
    """ClipLoss.forward, world_size 1: utils/toolkit.py:110-141."""
    li = logit_scale * image_features @ text_features.t()
    lt = logit_scale * text_features @ image_features.t()
    y = torch.arange(li.shape[0], device=li.device)
    return (F.cross_entropy(li, y) + F.cross_entropy(lt, y)) / 2


# --------------------------------------------------------------------------- a9/a10
def forward_for_classification(p: Params, image, text_cls):
    """Learner.forward_for_classification: models/proof.py:519-536."""
    imf = F.normalize(encode_image(image, p), dim=1)
    txf = F.normalize(encode_text(text_cls, p), dim=1)
    return imf @ txf.t()


def cosine_linear(x, weight, sigma=None):
    """CosineLinear.forward (nb_proxy=1): convs/linears.py:51-61."""
    out = F.linear(F.normalize(x, p=2, dim=1), F.normalize(weight, p=2, dim=1))
    if sigma is not None:
        out = sigma * out
    return out


# --------------------------------------------------------------------------- a11/a12
def cal_prototype(emb, labels, states, known: int, total: int, img_prototypes,
                  by_state: Dict[int, Dict[int, torch.Tensor]]):
    """Learner.cal_prototype, the reduction part: models/proof.py:258-276.
    ``emb`` is already the L2-normalised CLIP feature (:248).  Mutates
    ``img_prototypes`` rows and ``by_state`` exactly like the reference; also returns
    the integer per-class / per-(class,state) counts the loop implies."""
    counts, counts_cs = {}, {}
    for c in range(known, total):
        idx = (labels == c).nonzero().squeeze(-1)
        counts[c] = int(len(idx))
        if len(idx) > 0:
            e = emb[idx]
            img_prototypes[c] = e.mean(0)
            st = states[idx]
            if c not in by_state:
                by_state[c] = {}
            for s in torch.unique(st):
                m = (st == s)
                if m.sum() > 0:
                    by_state[c][s.item()] = e[m].mean(0)
                    counts_cs[(c, s.item())] = int(m.sum())
    return counts, counts_cs


def simplecil_prototypes(emb, labels, fc_weight):
    """simplecil.Learner.replace_fc, the reduction part: models/simplecil.py:48-55
    (un-normalised features; class list = unique labels)."""
    for c in torch.unique(labels).tolist():
        idx = (labels == c).nonzero().squeeze(-1)
        fc_weight[c] = emb[idx].mean(0)
    return fc_weight


# --------------------------------------------------------------------------- a13/a14
def detect_evolution_type(state_ids: Sequence[int]) -> str:
    """InsectLifecycleModel._detect_evolution_type: models/state_evolution.py:53-66."""
    if 1 in state_ids and 4 in state_ids:
        return "larvae_to_adult"
    elif 3 in state_ids and 4 in state_ids:
        return "nymph_to_adult"
    elif 1 in state_ids:
        return "larvae_to_adult"
    elif 3 in state_ids:
        return "nymph_to_adult"
    elif 4 in state_ids:
        return "adult_only"
    return "unknown"


def build_evolution_graph(by_state: Dict[int, Dict[int, torch.Tensor]],
                          lifecycle_types: Optional[Dict[int, str]] = None):
    """Node / edge enumeration of evolve_and_update: models/state_evolution.py:260-316.
    Returns (node_classes, node_states, node_times, edges[(i,j)], weights,
    lifecycle_types) with the reference's ordering (SURVEY App. A-7)."""
    if lifecycle_types is None:
        lifecycle_types = {}
    ncls, nst, ntime = [], [], []
    for c, sd in by_state.items():
        if len(sd) < 2:
            continue
        sids = sorted(list(sd.keys()))
        lifecycle_types[c] = detect_evolution_type(sids)
        s2t = {s: i / max(1, len(sids) - 1) for i, s in enumerate(sids)}
        for s in sd.keys():
            ncls.append(c)
            nst.append(s)
            ntime.append(s2t[s])
    n = len(ncls)
    edges, w = [], []
    for i in range(n):
        for j in range(n):
            if i != j and ncls[i] == ncls[j] and ntime[i] < ntime[j]:
                edges.append((i, j))
                w.append(1.0 - abs(ntime[i] - ntime[j]))
    for i in range(n):
        for j in range(n):
            if i != j and ncls[i] != ncls[j] and nst[i] == nst[j]:
                if lifecycle_types.get(ncls[i]) == lifecycle_types.get(ncls[j]):
                    edges.append((i, j))
                    w.append(0.5)
    return ncls, nst, ntime, edges, w, lifecycle_types


def _seq_linear_ln_relu(x, p: Params, prefix: str):
    h = F.linear(x, p[prefix + ".0.weight"], p[prefix + ".0.bias"])
    h = F.layer_norm(h, (h.shape[-1],), p[prefix + ".1.weight"], p[prefix + ".1.bias"], LN_EPS)
    return F.relu(h)


def temporal_gcn_block(x, edge_index, edge_weights, p: Params, prefix: str):
    """TemporalGCNBlock.forward: models/dynamic_modal_graph.py:294-337 (edge loop as written)."""
    src, dst = edge_index
    n, h = x.shape
    messages = torch.zeros(n, h, dtype=x.dtype)
    counts = torch.zeros(n, 1, dtype=x.dtype)
    for i in range(src.shape[0]):
        s, d = src[i], dst[i]
        m = torch.cat([x[s], x[d]], dim=-1)
        m = _seq_linear_ln_relu(m, p, prefix + ".message_net") * edge_weights[i]
        messages[d] += m
        counts[d] += 1
    valid = (counts > 0).to(x.dtype)
    messages = messages / (counts + 1e-8) * valid
    gate = torch.sigmoid(F.linear(x, p[prefix + ".temporal_gate.0.weight"],
                                  p[prefix + ".temporal_gate.0.bias"]))
    h_new = _seq_linear_ln_relu(torch.cat([x, messages], dim=-1), p, prefix + ".update_net")
    return gate * h_new + (1 - gate) * x


def temporal_state_gcn(node_features, edge_index, edge_weights, time_steps, p: Params,
                       prefix: str = "state_embedder.temporal_gcn"):
    """TemporalStateGCN.forward: models/dynamic_modal_graph.py:239-266."""
    h = _seq_linear_ln_relu(node_features, p, prefix + ".node_encoder")
    t = _seq_linear_ln_relu(time_steps, p, prefix + ".time_encoder")
    h_t = torch.cat([h, t], dim=-1)
    blk = 0
    while f"{prefix}.temporal_blocks.{blk}.message_net.0.weight" in p:
        h_t = temporal_gcn_block(h_t, edge_index, edge_weights, p, f"{prefix}.temporal_blocks.{blk}")
        blk += 1
    out = F.linear(h_t, p[prefix + ".output_proj.weight"], p[prefix + ".output_proj.bias"])
    return F.normalize(out, dim=-1)


def evolve_and_update(p: Params, by_state: Dict[int, Dict[int, torch.Tensor]],
                      lifecycle_types: Optional[Dict[int, str]] = None):
    """InsectLifecycleModel.evolve_and_update: models/state_evolution.py:239-367.
    Reproduces the aliasing quirk (SURVEY App. C-2): ``result['prototypes']`` is a
    shallow copy, so the inner dicts of ``by_state`` are mutated in place."""
    result = {"prototypes": by_state.copy(), "embeddings": [], "lifecycle_features": {},
              "distances": {}}
    if len(by_state) < 1:
        return result
    if lifecycle_types is None:
        lifecycle_types = {}
    nodes = []
    for c, sd in by_state.items():
        if len(sd) < 2:
            continue
        sids = sorted(list(sd.keys()))
        for s in sd.keys():
            nodes.append(sd[s])
        result["lifecycle_features"][c] = torch.cat([sd[s].unsqueeze(0) for s in sids], dim=0).mean(0)
    ncls, nst, ntime, edges, w, lifecycle_types = build_evolution_graph(by_state, lifecycle_types)
    if not nodes:
        return result
    if not edges:
        return result
    x = torch.stack(nodes)
    ei = torch.tensor(edges, dtype=torch.int64).t()
    ew = torch.tensor(w, dtype=torch.float32).to(x.dtype)   # python floats -> float32 tensor (:320)
    ts = torch.tensor([[t] for t in ntime], dtype=torch.float32).to(x.dtype)
    with torch.no_grad():
        upd = temporal_state_gcn(x, ei, ew, ts, p)
    for i, (c, s) in enumerate(zip(ncls, nst)):
        result["prototypes"][c][s] = upd[i]
    for c in result["lifecycle_features"].keys():
        if c in result["prototypes"]:
            sd = result["prototypes"][c]
            if len(sd) >= 2:
                emb = torch.stack(list(sd.values())).mean(0)
                while len(result["embeddings"]) <= c:
                    result["embeddings"].append(None)
                result["embeddings"][c] = emb
    dist: Dict[int, Dict[int, list]] = {}
    for i, s1 in enumerate(nst):
        if s1 not in dist:
            dist[s1] = {}
        for j, s2 in enumerate(nst):
            if i != j:
                sim = F.cosine_similarity(upd[i].unsqueeze(0), upd[j].unsqueeze(0))
                dval = 1.0 - sim.item()
                dist[s1].setdefault(s2, []).append(dval)
    for s1 in dist:
        for s2 in dist[s1]:
            dist[s1][s2] = sum(dist[s1][s2]) / len(dist[s1][s2])
    result["distances"] = dist
    return result


# --------------------------------------------------------------------------- a15
def sync_class_prototypes(img_prototypes, by_state):
    """Proof_Net._sync_class_prototypes: utils/inc_net.py:600-617."""
    for c in range(len(img_prototypes)):
        if c in by_state and by_state[c]:
            protos, weights = [], []
            for s, pr in by_state[c].items():
                protos.append(pr)
                weights.append(1.5 if s == 4 else 1.0)
            wt = torch.tensor(weights).to(protos[0].dtype)
            wt = wt / wt.sum()
            acc = torch.zeros_like(protos[0])
            for i, pr in enumerate(protos):
                acc += wt[i] * pr
            img_prototypes[c] = F.normalize(acc, dim=0)
    return img_prototypes


def evolve_state_prototypes(p: Params, img_prototypes, by_state, lifecycle_types=None):
    """Proof_Net.evolve_state_prototypes: utils/inc_net.py:582-598 (alpha blend is a
    no-op by aliasing, then re-normalise, then sync)."""
    res = evolve_and_update(p, by_state, lifecycle_types)
    alpha = 0.6
    for c, sp in res["prototypes"].items():
        for s, ev in sp.items():
            if c in by_state and s in by_state[c]:
                orig = by_state[c][s]
                by_state[c][s] = F.normalize(alpha * orig + (1 - alpha) * ev, dim=0)
    sync_class_prototypes(img_prototypes, by_state)
    return res["embeddings"]


# --------------------------------------------------------------------------- a16-a18
def prior_distance_factors(num_states=10) -> torch.Tensor:
    """AdaptiveStateDistanceMatrix.__init__ prior: utils/state_distance.py:20-37."""
    m = torch.ones(num_states, num_states)
    m[1, 4] = m[4, 1] = 2.0
    m[3, 4] = m[4, 3] = 0.7
    m[1, 2] = m[2, 1] = 1.5
    m[0, :] = 1.8
    m[:, 0] = 1.8
    m[0, 0] = 1.0
    return m


def get_distance_matrix(factors: torch.Tensor) -> torch.Tensor:
    """utils/state_distance.py:65-71."""
    sym = (factors + factors.t()) / 2
    eye = torch.eye(factors.shape[0], dtype=factors.dtype)
    return sym * (1 - eye) + eye


def state_distance_forward(factors: torch.Tensor, state_features, state_ids,
                           update_counter: int, training=True, update_interval=10,
                           decay=0.9):
    """AdaptiveStateDistanceMatrix.forward: utils/state_distance.py:79-144.
    Mutates ``factors`` in place; returns (pre-update matrix, new counter)."""
    cur = get_distance_matrix(factors)
    n = factors.shape[0]
    if training and update_counter % update_interval == 0:
        centers = {}
        for s in range(1, n):
            m = (state_ids == s)
            if m.sum() > 0:
                centers[s] = state_features[m].mean(0)
        if len(centers) > 1:
            ids = sorted(centers.keys())
            ct = torch.stack([centers[i] for i in ids])
            sim = torch.mm(F.normalize(ct, dim=1), F.normalize(ct, dim=1).t())
            dm = 2.0 - sim
            for i, si in enumerate(ids):
                for j, sj in enumerate(ids):
                    if i != j:
                        old = factors[si, sj].item()
                        new = decay * old + (1 - decay) * dm[i, j].item()
                        factors[si, sj] = new
                        factors[sj, si] = new
    return cur, update_counter + 1


def update_state_distance_matrix(factors: torch.Tensor, distances: Dict[int, Dict[int, float]]):
    """Learner.update_state_distance_matrix EMA: models/proof.py:666-675."""
    for s1 in distances:
        for s2 in distances[s1]:
            d = distances[s1][s2]
            old = factors[s1, s2].item()
            weight = 0.3
            new = (1 - weight) * old + weight * d
            factors[s1, s2] = new
            factors[s2, s1] = new
    return factors


# --------------------------------------------------------------------------- a19
def dynamic_gcn(x, edge_index, edge_weights, layers: List[Tuple[torch.Tensor, ...]]):
    """DynamicGCN.forward (eval, with edges): models/dynamic_modal_graph.py:131-163.
    ``layers`` = [(W, b, ln_w, ln_b), ...]."""
    for (W, b, g, be) in layers:
        h = F.relu(F.linear(x, W, b))
        if edge_index is not None and edge_weights is not None:
            src, dst = edge_index
            hu = h.clone()
            for i in range(src.shape[0]):
                hu[dst[i]] = hu[dst[i]] + edge_weights[i] * h[src[i]]
            h = hu
        x = F.layer_norm(h, (h.shape[-1],), g, be, LN_EPS)
    return x


# --------------------------------------------------------------------------- step used by bench
def head_step_fwd_bwd(p: Params, batch, img_prototypes, cots, trainable: Sequence[str]):
    """One 'head fwd+bwd' step as BASELINE.md section 4.4 defines it: no-grad cosine
    logits (models/proof.py:415-418) + forward_tri_modal (:424-425) + VJP with fixed
    cotangents on the four feature outputs (stands for :444).  Returns (logits, outs, grads)."""
    with torch.no_grad():
        logits = forward_for_classification(p, batch["image"], batch["text_cls"])
    outs = forward_tri_modal(p, batch["image"], batch["text"], batch["state"], img_prototypes)
    wrt = [p[k] for k in trainable]
    grads = torch.autograd.grad(outs[:4], wrt, grad_outputs=list(cots), allow_unused=True)
    return logits, outs, dict(zip(trainable, grads))


def trainable_names(p: Params) -> List[str]:
    """Parameters that receive a gradient in the reference loop (SURVEY 8a tail;
    utils/inc_net.py:392-393, :494-513): newest projections, embedding table,
    sel_attn, newest prompts (logit_scale handled by the caller)."""
    t = num_tasks(p) - 1
    names = []
    for kind in ("img", "text", "state"):
        names += [f"projs_{kind}.{t}.MLP.0.weight", f"projs_{kind}.{t}.MLP.0.bias"]
    names += ["state_embedder.state_embeddings.weight",
              "sel_attn.w_qs.weight", "sel_attn.w_ks.weight", "sel_attn.w_vs.weight",
              "sel_attn.fc.weight", "sel_attn.fc.bias",
              "sel_attn.layer_norm.weight", "sel_attn.layer_norm.bias",
              f"context_prompts.{t}"]
    return names
