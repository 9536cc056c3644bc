"""Executable specification of the factorised head algorithm the CUDA kernels implement
(DESIGN.md section 3).  Pure torch on the inputs' device, fp64-capable, hand-written backward - no
autograd - so that the algebra (shared-row dedup, fc folded into V, table-query
factorisation, batch-reduced shared gradients) is verified against the oracle before and
independently of any CUDA code.  Lives in tests/: it is a test helper, not the product.

Row sets (tri-modal, per-sample text):
  step rows  S = [Xp (C proto rows) ; Xc (P prompt rows) ; Xst (10 state-table rows)]   Ns = C+P+10
  own rows   Xown = [X0 (B image rows) ; X1 (B text rows)]
  shared keys = S rows [0, M), M = C+P ; state key of sample b = S row M+sid_b
  table queries = S rows [0, C) (proto outputs) and S row M+sid_b (state output)
"""
from __future__ import annotations

import math

import torch

LN_EPS = 1e-5
NORM_EPS = 1e-12


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


def head_fwd_bwd(p, image, text, sid, protos, cots):
    """Returns (outs, grads) where outs=(image,text[B,1,D],state,proto) and grads is a dict
    over oracle.trainable_names."""
    T = 0
    while f"projs_img.{T}.MLP.0.weight" in p:
        T += 1
    D = image.shape[1]
    B = image.shape[0]
    tau = math.sqrt(D)
    Wi = sum(p[f"projs_img.{t}.MLP.0.weight"] for t in range(T)); bi = sum(p[f"projs_img.{t}.MLP.0.bias"] for t in range(T))
    Wt = sum(p[f"projs_text.{t}.MLP.0.weight"] for t in range(T)); bt = sum(p[f"projs_text.{t}.MLP.0.bias"] for t in range(T))
    Ws = sum(p[f"projs_state.{t}.MLP.0.weight"] for t in range(T)); bs = sum(p[f"projs_state.{t}.MLP.0.bias"] for t in range(T))
    E = p["state_embedder.state_embeddings.weight"]
    Wq, Wk, Wv = p["sel_attn.w_qs.weight"], p["sel_attn.w_ks.weight"], p["sel_attn.w_vs.weight"]
    Wfc, bfc = p["sel_attn.fc.weight"], p["sel_attn.fc.bias"]
    gam, bet = p["sel_attn.layer_norm.weight"], p["sel_attn.layer_norm.bias"]
    Xc = torch.cat([p[f"context_prompts.{t}"] for t in range(T)], 0)
    C, P = protos.shape[0], Xc.shape[0]
    M = C + P
    Ns = M + 10
    # ---- step rows
    Xp, invp = _nrm(protos @ Wi.t() + bi)
    Xst, invs = _nrm(E @ Ws.t() + bs)
    S = torch.cat([Xp, Xc, Xst], 0)
    Qs, Ks, Vs = S @ Wq.t(), S @ Wk.t(), S @ Wv.t()
    VFs = Vs @ Wfc.t()
    TT = Qs @ Ks.t()                                   # [Ns, Ns] raw dots
    tq = list(range(C)) + list(range(M, Ns))           # table query rows
    m_t = (TT[:, :M] / tau).max(dim=1, keepdim=True).values
    Pt = torch.exp(TT[:, :M] / tau - m_t)              # [Ns, M] (only tq rows used)
    Zt = Pt.sum(1)
    NFt = Pt @ VFs[:M]
    # ---- own rows
    X0, inv0 = _nrm(image @ Wi.t() + bi)
    X1, inv1 = _nrm(text @ Wt.t() + bt)
    Xo = torch.cat([X0, X1], 0)
    Qo, Ko, Vo = Xo @ Wq.t(), Xo @ Wk.t(), Xo @ Wv.t()
    VFo = Vo @ Wfc.t()
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
    Ybar_o = Aext @ VFs + aown[:, :1] * VFo[rows_b] + aown[:, 1:] * VFo[rows_b + B]
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
    dTT[:, :M] += Pt * (G @ VFs[:M].t() - h.unsqueeze(1)) / tau
    dVFs[:M] += Pt.t() @ G
    # -- own query rows
    go_o = torch.cat([g_img, g_txt], 0)
    dgam += (go_o * xh_o).sum(0); dbet += go_o.sum(0)
    du_o = _ln_bwd(go_o, xh_o, rstd_o, gam)
    dbfc += du_o.sum(0)
    dXo = du_o.clone()
    rowdot = (du_o * Ybar_o).sum(-1, keepdim=True)
    dA = du_o @ VFs.t()
    dS = Aext * (dA - rowdot) / tau                    # [2B, Ns]
    da_own = torch.stack([(du_o * VFo[rows_b]).sum(-1), (du_o * VFo[rows_b + B]).sum(-1)], 1)
    ds_own = aown * (da_own - rowdot) / tau            # [2B, 2]
    dVFs += Aext.t() @ du_o
    dVFo.index_add_(0, rows_b, aown[:, :1] * du_o); dVFo.index_add_(0, rows_b + B, aown[:, 1:] * du_o)
    dQo = dS @ Ks + ds_own[:, :1] * Ko[rows_b] + ds_own[:, 1:] * Ko[rows_b + B]
    dKs = dS.t() @ Qo
    dKo = dSK @ Qs
    dKo.index_add_(0, rows_b, ds_own[:, :1] * Qo); dKo.index_add_(0, rows_b + B, ds_own[:, 1:] * Qo)
    dQs = dSK.t() @ Ko
    # step-level score grads
    dQs += dTT @ Ks
    dKs += dTT.t() @ Qs
    # fc / V
    dVo = dVFo @ Wfc
    dVs = dVFs @ Wfc
    dWfc = dVFo.t() @ Vo + dVFs.t() @ Vs
    # qkv projections
    dXo += dQo @ Wq + dKo @ Wk + dVo @ Wv
    dS_rows = dQs @ Wq + dKs @ Wk + dVs @ Wv + R
    dWq = dQo.t() @ Xo + dQs.t() @ S
    dWk = dKo.t() @ Xo + dKs.t() @ S
    dWv = dVo.t() @ Xo + dVs.t() @ S
    # normalisations and the newest projections
    dz0 = _nrm_bwd(dXo[:B], X0, inv0); dz1 = _nrm_bwd(dXo[B:], X1, inv1)
    dzp = _nrm_bwd(dS_rows[:C], Xp, invp); dzs = _nrm_bwd(dS_rows[M:], Xst, invs)
    dWi = dz0.t() @ image + dzp.t() @ protos; dbi = dz0.sum(0) + dzp.sum(0)
    dWt = dz1.t() @ text; dbt = dz1.sum(0)
    dWs = dzs.t() @ E; dbs = dzs.sum(0)
    dE = dzs @ Ws
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
    return outs, grads
