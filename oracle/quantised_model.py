"""Factorised head with the 16-bit rounding points of the CUDA kernels (TEST INFRASTRUCTURE).

The same algebra as ``tests/factorised_model.py`` (fp64, hand-written backward, checked against the
reference-pinned oracle), plus a rounding ``q*()`` at exactly the places where ``csrc/head.cu`` hands a
tensor to the tensor cores in TEAM_MODE_BF16:

  qw  inputs and weights (image, text, prototypes, state table, summed projections, Wq/Wk/Wv/Wfc) -> bf16
  qa  forward activations (S, Xo, q/k/v - stored ONLY as 16 bit -, VF, softmax probabilities)       -> bf16 (act="f16": IEEE half, an
      experiment the hardware rules out - tcgen05 kind::f16 cannot mix f16 and bf16 operands)
  qg  everything the backward feeds to a GEMM (dY, dS, dSK, dTT, G, dVF, dQ/dK/dV, dz)               -> bf16

Accumulation and all row-wise math (normalise, softmax, LayerNorm, their backward) stay exact here and fp32 in
the kernels.  With ``operands_only=True`` only ``qw`` is applied: that is "the reference evaluated on the
identically quantised operands" (SURVEY 7.3 (i)), the oracle of the 1e-3 claim on the forward outputs.  With every
rounding point on, kernel and model differ only by accumulation order, so the comparison pins the kernels'
arithmetic itself (the coefficient-GEMM form of the table-row gradients R / G is the one place evaluated exactly
here - see quantised points in DESIGN.md section 2).  Follows convs/projections.py:64-87 and
utils/inc_net.py:528-580 through tests/factorised_model.py.
"""
from __future__ import annotations

import math

import torch

LN_EPS = 1e-5
NORM_EPS = 1e-12


def q_bf16(x):
    return x.float().to(torch.bfloat16).to(x.dtype)


def q_f16(x):
    return x.float().to(torch.float16).to(x.dtype)


def _id(x):
    return x

def _nrm(z):
    n = z.norm(dim=-1, keepdim=True).clamp_min(NORM_EPS)
    return z / n, 1.0 / n


def _nrm_bwd(dx, x, inv):
    # x = z*inv ; dz = inv*(dx - x*(x.dx))   (norm above eps)
    return inv * (dx - x * (x * dx).sum(-1, keepdim=True))


def _ln(u, g, b):
    mu = u.mean(-1, keepdim=True)
    var = ((u - mu) ** 2).mean(-1, keepdim=True)
    rstd = (var + LN_EPS).rsqrt()
    xh = (u - mu) * rstd
    return xh * g + b, xh, rstd


def _ln_bwd(go, xh, rstd, g):
    gg = go * g
    du = rstd * (gg - gg.mean(-1, keepdim=True) - xh * (gg * xh).mean(-1, keepdim=True))
    return du


def head_fwd_bwd(p, image, text, sid, protos, cots, text_cls=None, operands_only=False, act="bf16", grad="bf16"):
    """Returns (outs, grads[, cls_logits]) where outs=(image,text[B,1,D],state,proto) and grads is a dict over
    oracle.trainable_names.  fp64 tensors in."""
    qw = q_bf16
    qa = _id if operands_only or act is None else (q_f16 if act == "f16" else q_bf16)
    qg = _id if operands_only or grad is None else q_bf16
    T = 0
    while f"projs_img.{T}.MLP.0.weight" in p:
        T += 1
    D = image.shape[1]
    B = image.shape[0]
    tau = math.sqrt(D)
    Wi = qw(sum(p[f"projs_img.{t}.MLP.0.weight"] for t in range(T))); bi = sum(p[f"projs_img.{t}.MLP.0.bias"] for t in range(T))
    Wt = qw(sum(p[f"projs_text.{t}.MLP.0.weight"] for t in range(T))); bt = sum(p[f"projs_text.{t}.MLP.0.bias"] for t in range(T))
    Ws = qw(sum(p[f"projs_state.{t}.MLP.0.weight"] for t in range(T))); bs = sum(p[f"projs_state.{t}.MLP.0.bias"] for t in range(T))
    E = qw(p["state_embedder.state_embeddings.weight"])
    Wq, Wk, Wv = qw(p["sel_attn.w_qs.weight"]), qw(p["sel_attn.w_ks.weight"]), qw(p["sel_attn.w_vs.weight"])
    Wfc, bfc = qw(p["sel_attn.fc.weight"]), p["sel_attn.fc.bias"]
    image, text, protos = qw(image), qw(text), qw(protos)
    gam, bet = p["sel_attn.layer_norm.weight"], p["sel_attn.layer_norm.bias"]
    Xc = torch.cat([p[f"context_prompts.{t}"] for t in range(T)], 0)
    C, P = protos.shape[0], Xc.shape[0]
    M = C + P
    Ns = M + 10
    # ---- step rows
    Xp, invp = _nrm(protos @ Wi.t() + bi)
    Xst, invs = _nrm(E @ Ws.t() + bs)
    S = torch.cat([Xp, Xc, Xst], 0)
    Sh = qa(S)
    Qs, Ks, Vs = qa(Sh @ Wq.t()), qa(Sh @ Wk.t()), qa(Sh @ Wv.t())      # q/k/v exist only as 16-bit values
    VFs = Vs @ Wfc.t()
    VFsh = qa(VFs)
    TT = Qs @ Ks.t()                                   # [Ns, Ns] raw dots
    tq = list(range(C)) + list(range(M, Ns))           # table query rows
    m_t = (TT[:, :M] / tau).max(dim=1, keepdim=True).values
    Pt = torch.exp(TT[:, :M] / tau - m_t)              # [Ns, M] (only tq rows used)
    Zt = Pt.sum(1)
    Pth = qa(Pt)
    NFt = Pth @ VFsh[:M]
    # ---- own rows
    X0, inv0 = _nrm(image @ Wi.t() + bi)
    X1, inv1 = _nrm(text @ Wt.t() + bt)
    Xo = torch.cat([X0, X1], 0)
    Xoh = qa(Xo)
    Qo, Ko, Vo = qa(Xoh @ Wq.t()), qa(Xoh @ Wk.t()), qa(Xoh @ Wv.t())
    VFo = Vo @ Wfc.t()
    VFoh = qa(VFo)
    SQ = Qo @ Ks.t()                                   # own queries vs step keys   [2B, Ns]
    SK = Ko @ Qs.t()                                   # own keys vs step queries   [2B, Ns]
    dev = image.device
    bidx = torch.arange(B, device=dev)
    rows_b = torch.cat([bidx, bidx])                   # sample of each own row
    scol = M + sid                                     # state column per sample
    # own query rows
    mask = torch.zeros(2 * B, Ns, dtype=torch.bool, device=dev)
    mask[:, :M] = True
    mask[torch.arange(2 * B, device=dev), scol[rows_b]] = True
    s_ext = torch.where(mask, SQ / tau, torch.full_like(SQ, -float("inf")))
    s_own = torch.stack([(Qo * Ko[rows_b]).sum(-1), (Qo * Ko[rows_b + B]).sum(-1)], 1) / tau   # vs img key, text key
    mx = torch.maximum(s_ext.max(1).values, s_own.max(1).values).unsqueeze(1)
    pe, po = torch.exp(s_ext - mx), torch.exp(s_own - mx)
    den = pe.sum(1, keepdim=True) + po.sum(1, keepdim=True)
    Aext, aown = pe / den, po / den
    Aexth = qa(Aext)
    Ybar_o = Aexth @ VFsh + aown[:, :1] * VFo[rows_b] + aown[:, 1:] * VFo[rows_b + B]
    out_o, xh_o, rstd_o = _ln(Ybar_o + bfc + Xo, gam, bet)
    out_img, out_txt = out_o[:B], out_o[B:]
    # table query rows, per sample: rows r in [0,C) and the state row
    rt = torch.cat([torch.arange(C, device=dev).unsqueeze(0).expand(B, C), scol.unsqueeze(1)], 1)      # [B, C+1] step-row ids
    s_i = SK[:B].gather(1, rt) / tau                   # vs own image key
    s_t = SK[B:].gather(1, rt) / tau                   # vs own text key
    s_s = TT[rt, scol.unsqueeze(1).expand(B, C + 1)] / tau   # vs own state key
    mr = m_t[rt, 0]
    m2 = torch.maximum(torch.maximum(mr, s_i), torch.maximum(s_t, s_s))
    c = torch.exp(mr - m2)
    p_i, p_t, p_s = torch.exp(s_i - m2), torch.exp(s_t - m2), torch.exp(s_s - m2)
    den_t = c * Zt[rt] + p_i + p_t + p_s
    VFst = VFs[scol]                                   # [B, D]
    Num = c.unsqueeze(-1) * NFt[rt] + p_i.unsqueeze(-1) * VFo[:B].unsqueeze(1) \
        + p_t.unsqueeze(-1) * VFo[B:].unsqueeze(1) + p_s.unsqueeze(-1) * VFst.unsqueeze(1)
    Ybar_t = Num / den_t.unsqueeze(-1)                 # [B, C+1, D]
    out_t, xh_t, rstd_t = _ln(Ybar_t + bfc + S[rt], gam, bet)
    out_proto = out_t[:, :C].mean(1) if C > 1 else out_t[:, 0]
    out_state = out_t[:, C]
    outs = (out_img, out_txt.unsqueeze(1), out_state, out_proto)
    cls_logits = None
    if text_cls is not None:        # forward_for_classification (models/proof.py:519-536): X0 is already normalised
        zc, _ = _nrm(qw(text_cls) @ Wt.t() + bt)
        x0n, _ = _nrm(X0)
        cls_logits = x0n @ zc.t()

    # =============================== backward ===============================
    g_img, g_txt, g_st, g_pr = cots[0], cots[1].reshape(B, D), cots[2], cots[3]
    dgam = torch.zeros_like(gam); dbet = torch.zeros_like(bet); dbfc = torch.zeros_like(bfc)
    # -- table rows
    go_t = torch.cat([(g_pr / C).unsqueeze(1).expand(B, C, D), g_st.unsqueeze(1)], 1)
    dgam += (go_t * xh_t).sum((0, 1)); dbet += go_t.sum((0, 1))
    du_t = _ln_bwd(go_t, xh_t, rstd_t, gam)            # [B, C+1, D] = dY = residual grad
    dbfc += du_t.sum((0, 1))
    R = torch.zeros(Ns, D, dtype=S.dtype, device=dev).index_add_(0, rt.reshape(-1), du_t.reshape(-1, D))
    w = 1.0 / den_t
    dot_yy = (du_t * Ybar_t).sum(-1)                   # dY . Ybar
    G = torch.zeros(Ns, D, dtype=S.dtype, device=dev).index_add_(0, rt.reshape(-1), ((c * w).unsqueeze(-1) * du_t).reshape(-1, D))
    h = torch.zeros(Ns, dtype=S.dtype, device=dev).index_add_(0, rt.reshape(-1), (c * w * dot_yy).reshape(-1))
    a_i, a_t, a_s = p_i * w, p_t * w, p_s * w
    ds_i = a_i * ((du_t * VFo[:B].unsqueeze(1)).sum(-1) - dot_yy) / tau
    ds_t = a_t * ((du_t * VFo[B:].unsqueeze(1)).sum(-1) - dot_yy) / tau
    ds_s = a_s * ((du_t * VFst.unsqueeze(1)).sum(-1) - dot_yy) / tau
    dSK = torch.zeros(2 * B, Ns, dtype=S.dtype, device=dev)
    dSK[:B].scatter_(1, rt, ds_i); dSK[B:].scatter_(1, rt, ds_t)
    dTT = torch.zeros(Ns, Ns, dtype=S.dtype, device=dev)
    dTT.index_put_((rt.reshape(-1), scol.unsqueeze(1).expand(B, C + 1).reshape(-1)), ds_s.reshape(-1), accumulate=True)
    dVFo = torch.zeros_like(VFo)
    dVFo[:B] += (a_i.unsqueeze(-1) * du_t).sum(1); dVFo[B:] += (a_t.unsqueeze(-1) * du_t).sum(1)
    dVFs = torch.zeros_like(VFs).index_add_(0, scol, (a_s.unsqueeze(-1) * du_t).sum(1))
    # shared part of the table queries (per step)
    Gh = qg(G)
    dTT[:, :M] += Pt * (Gh @ VFsh[:M].t() - h.unsqueeze(1)) / tau
    dVFs[:M] += Pth.t() @ Gh
    # -- own query rows
    go_o = torch.cat([g_img, g_txt], 0)
    dgam += (go_o * xh_o).sum(0); dbet += go_o.sum(0)
    du_o = _ln_bwd(go_o, xh_o, rstd_o, gam)
    dbfc += du_o.sum(0)
    dXo = du_o.clone()
    rowdot = (du_o * Ybar_o).sum(-1, keepdim=True)
    dYoh = qg(du_o)
    dA = dYoh @ VFsh.t()
    dS = qg(Aext * (dA - rowdot) / tau)                # [2B, Ns]; stored only as 16-bit
    da_own = torch.stack([(du_o * VFo[rows_b]).sum(-1), (du_o * VFo[rows_b + B]).sum(-1)], 1)
    ds_own = aown * (da_own - rowdot) / tau            # [2B, 2]
    dVFs += Aexth.t() @ dYoh
    dVFo.index_add_(0, rows_b, aown[:, :1] * du_o); dVFo.index_add_(0, rows_b + B, aown[:, 1:] * du_o)
    dSKh, dTTh = qg(dSK), None
    dQo = dS @ Ks + ds_own[:, :1] * Ko[rows_b] + ds_own[:, 1:] * Ko[rows_b + B]
    dKs = dS.t() @ Qo
    dKo = dSKh @ Qs
    dKo.index_add_(0, rows_b, ds_own[:, :1] * Qo); dKo.index_add_(0, rows_b + B, ds_own[:, 1:] * Qo)
    dQs = dSKh.t() @ Ko
    # step-level score grads
    dTTh = qg(dTT)
    dQs += dTTh @ Ks
    dKs += dTTh.t() @ Qs
    dQo, dKo, dQs, dKs = qg(dQo), qg(dKo), qg(dQs), qg(dKs)
    # fc / V
    dVFoh, dVFsh = qg(dVFo), qg(dVFs)
    dVo = qg(dVFoh @ Wfc)
    dVs = qg(dVFsh @ Wfc)
    dWfc = dVFoh.t() @ Vo + dVFsh.t() @ Vs
    # qkv projections
    dXo += dQo @ Wq + dKo @ Wk + dVo @ Wv
    dS_rows = dQs @ Wq + dKs @ Wk + dVs @ Wv + R
    dWq = dQo.t() @ Xoh + dQs.t() @ Sh
    dWk = dKo.t() @ Xoh + dKs.t() @ Sh
    dWv = dVo.t() @ Xoh + dVs.t() @ Sh
    # normalisations and the newest projections
    dz0 = _nrm_bwd(dXo[:B], X0, inv0); dz1 = _nrm_bwd(dXo[B:], X1, inv1)
    dzp = _nrm_bwd(dS_rows[:C], Xp, invp); dzs = _nrm_bwd(dS_rows[M:], Xst, invs)
    dWi = qg(dz0).t() @ image + qg(dzp).t() @ protos; dbi = dz0.sum(0) + dzp.sum(0)
    dWt = qg(dz1).t() @ text; dbt = dz1.sum(0)
    dWs = qg(dzs).t() @ E; dbs = dzs.sum(0)
    dE = qg(dzs) @ Ws
    ppt = Xc.shape[0] // T
    grads = {
        f"projs_img.{T-1}.MLP.0.weight": dWi, f"projs_img.{T-1}.MLP.0.bias": dbi,
        f"projs_text.{T-1}.MLP.0.weight": dWt, f"projs_text.{T-1}.MLP.0.bias": dbt,
        f"projs_state.{T-1}.MLP.0.weight": dWs, f"projs_state.{T-1}.MLP.0.bias": dbs,
        "state_embedder.state_embeddings.weight": dE,
        "sel_attn.w_qs.weight": dWq, "sel_attn.w_ks.weight": dWk, "sel_attn.w_vs.weight": dWv,
        "sel_attn.fc.weight": dWfc, "sel_attn.fc.bias": dbfc,
        "sel_attn.layer_norm.weight": dgam, "sel_attn.layer_norm.bias": dbet,
        f"context_prompts.{T-1}": dS_rows[M - ppt:M],
    }
    return (outs, grads) if text_cls is None else (outs, grads, cls_logits)
