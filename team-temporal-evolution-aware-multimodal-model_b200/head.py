"""Host side of the fusion head: ``torch.autograd.Function`` over ``team_head_tri_fwd`` /
``team_head_tri_bwd`` (the C ABI in include/team_b200.h).

Mirrors what ``Proof_Net.forward_tri_modal`` (utils/inc_net.py:528-580) and
``Learner.forward_for_classification`` (models/proof.py:519-536) compute, with the same
parameter tensors.  torch only provides device memory, the stream and the autograd tape.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import torch

from . import capi

MODE_F32, MODE_BF16 = capi.MODE_F32, capi.MODE_BF16


def _stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def _check_state_ids(sid: torch.Tensor, num_states: int = capi.NUM_STATES) -> torch.Tensor:
    """nn.Embedding(10, 512) raises on an id outside [0, 10) (models/state_evolution.py:16, :45-47); the kernels
    would clamp it silently.  Device-side assert, no host synchronisation."""
    torch._assert_async(((sid >= 0) & (sid < num_states)).all(), "state id outside [0, num_states)")
    return sid


def _f32c(t: torch.Tensor, dev) -> torch.Tensor:
    t = t.detach()
    if t.device != dev or t.dtype != torch.float32 or not t.is_contiguous():
        t = t.to(device=dev, dtype=torch.float32).contiguous()
    return t


class HeadParamPack:
    """Flat, ordered view of the head parameters (reference state_dict names, SURVEY App. B)."""

    def __init__(self, w_img: Sequence[torch.Tensor], b_img, w_text, b_text, w_state, b_state,
                 prompts: Sequence[torch.Tensor], state_emb, w_q, w_k, w_v, w_fc, b_fc, ln_g, ln_b):
        self.T = len(w_img)
        if not (1 <= self.T <= capi.MAX_TASKS):
            raise ValueError(f"number of tasks {self.T} out of [1,{capi.MAX_TASKS}]")
        for lst in (b_img, w_text, b_text, w_state, b_state, prompts):
            if len(lst) != self.T:
                raise ValueError("per-task parameter lists must have equal length")
        self.ppt = int(prompts[0].shape[0])
        self.flat: List[torch.Tensor] = (list(w_img) + list(b_img) + list(w_text) + list(b_text) +
                                         list(w_state) + list(b_state) + list(prompts) +
                                         [state_emb, w_q, w_k, w_v, w_fc, b_fc, ln_g, ln_b])

    @staticmethod
    def from_state_dict(p: Dict[str, torch.Tensor]) -> "HeadParamPack":
        T = 0
        while f"projs_img.{T}.MLP.0.weight" in p:
            T += 1
        g = lambda fmt: [p[fmt.format(t)] for t in range(T)]
        return HeadParamPack(
            g("projs_img.{}.MLP.0.weight"), g("projs_img.{}.MLP.0.bias"),
            g("projs_text.{}.MLP.0.weight"), g("projs_text.{}.MLP.0.bias"),
            g("projs_state.{}.MLP.0.weight"), g("projs_state.{}.MLP.0.bias"),
            g("context_prompts.{}"), p["state_embedder.state_embeddings.weight"],
            p["sel_attn.w_qs.weight"], p["sel_attn.w_ks.weight"], p["sel_attn.w_vs.weight"],
            p["sel_attn.fc.weight"], p["sel_attn.fc.bias"],
            p["sel_attn.layer_norm.weight"], p["sel_attn.layer_norm.bias"])


def _fill_weights(T: int, ppt: int, flat: Sequence[torch.Tensor], protos: torch.Tensor) -> capi.HeadWeights:
    hw = capi.HeadWeights()
    hw.num_tasks, hw.prompts_per_task = T, ppt
    names = ("w_img", "b_img", "w_text", "b_text", "w_state", "b_state", "prompts")
    for k, n in enumerate(names):
        arr = getattr(hw, n)
        for t in range(T):
            arr[t] = flat[k * T + t].data_ptr()
    tail = flat[7 * T:]
    for n, t in zip(("state_emb", "w_q", "w_k", "w_v", "w_fc", "b_fc", "ln_g", "ln_b"), tail):
        setattr(hw, n, t.data_ptr())
    hw.prototypes = protos.data_ptr()
    hw.num_classes = int(protos.shape[0])
    return hw


class _TriModalFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, image, text, state_ids, protos, text_cls, mode, T, ppt, dropout, *params):
        capi.require_device()
        dev = image.device
        if not image.is_cuda:
            raise capi.TeamB200Error("forward_tri_modal needs CUDA tensors (no CPU fallback)")
        B = image.shape[0]
        image = _f32c(image, dev); text = _f32c(text, dev); protos = _f32c(protos, dev)
        sid = _check_state_ids(state_ids.detach().to(device=dev, dtype=torch.int64).contiguous())
        if image.shape != (B, capi.D) or text.shape != (B, capi.D) or sid.shape != (B,):
            raise ValueError("image/text must be [B,512] with per-sample text, state_ids [B]")
        flat = [_f32c(p, dev) for p in params]
        hw = _fill_weights(T, ppt, flat, protos)
        n_cls = 0 if text_cls is None else int(text_cls.shape[0])
        if text_cls is not None:
            text_cls = _f32c(text_cls, dev)
        L = capi.lib()
        nbytes = L.team_head_workspace_bytes(B, hw.num_classes, T * ppt, n_cls, mode)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        dr, dws = _dropout_arg(dropout, B, hw.num_classes, T * ppt, mode, dev)
        outs = torch.empty((4, B, capi.D), dtype=torch.float32, device=dev)
        logits = torch.empty((B, n_cls), dtype=torch.float32, device=dev) if n_cls else None
        amax = torch.empty((B,), dtype=torch.int64, device=dev) if n_cls else None
        capi.check(L.team_head_tri_fwd(
            C.byref(hw), mode, B, image.data_ptr(), text.data_ptr(), sid.data_ptr(),
            text_cls.data_ptr() if n_cls else None, n_cls,
            outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), outs[3].data_ptr(),
            logits.data_ptr() if n_cls else None, amax.data_ptr() if n_cls else None,
            ws.data_ptr(), nbytes, _stream_ptr(), dr), "team_head_tri_fwd")
        ctx.hold = (image, text, sid, protos, flat, ws, dr, dws)
        ctx.meta = (mode, T, ppt, B, nbytes)
        ctx.set_materialize_grads(False)        # an unused output arrives as None: a None g_proto skips the prototype rows
        res = (outs[0], outs[1].view(B, 1, capi.D), outs[2], outs[3])
        if n_cls:
            ctx.mark_non_differentiable(logits, amax)
            return res + (logits, amax)
        return res

    @staticmethod
    def backward(ctx, g_img, g_txt, g_st, g_pr, *unused):
        image, text, sid, protos, flat, ws, dr, dws = ctx.hold
        mode, T, ppt, B, nbytes = ctx.meta
        dev = image.device
        hw = _fill_weights(T, ppt, flat, protos)
        P = T * ppt
        mk = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
        g = {"w_img": mk(capi.D, capi.D), "b_img": mk(capi.D), "w_text": mk(capi.D, capi.D), "b_text": mk(capi.D),
             "w_state": mk(capi.D, capi.D), "b_state": mk(capi.D), "prompts": mk(max(P, 1), capi.D),
             "state_emb": mk(capi.NUM_STATES, capi.D), "w_q": mk(capi.D, capi.D), "w_k": mk(capi.D, capi.D),
             "w_v": mk(capi.D, capi.D), "w_fc": mk(capi.D, capi.D), "b_fc": mk(capi.D),
             "ln_g": mk(capi.D), "ln_b": mk(capi.D)}
        hg = capi.HeadGrads()
        for k, v in g.items():
            setattr(hg, k, v.data_ptr())
        zeros = None
        cots = []
        for k, x in enumerate((g_img, g_txt, g_st, g_pr)):
            if x is None:
                if k == 3:
                    cots.append(None)
                    continue
                zeros = zeros if zeros is not None else torch.zeros((B, capi.D), dtype=torch.float32, device=dev)
                x = zeros
            cots.append(_f32c(x.reshape(B, capi.D), dev))
        capi.check(capi.lib().team_head_tri_bwd(
            C.byref(hw), mode, B, image.data_ptr(), text.data_ptr(), sid.data_ptr(),
            cots[0].data_ptr(), cots[1].data_ptr(), cots[2].data_ptr(), cots[3].data_ptr() if cots[3] is not None else None,
            C.byref(hg), ws.data_ptr(), nbytes, _stream_ptr(), dr), "team_head_tri_bwd")
        need = ctx.needs_input_grad[9:]
        out: List[Optional[torch.Tensor]] = []
        names = ("w_img", "b_img", "w_text", "b_text", "w_state", "b_state")
        for k, n in enumerate(names):           # W = sum_t W_t  =>  dW_t = dW for every unfrozen t
            for t in range(T):
                out.append(g[n] if need[k * T + t] else None)
        for t in range(T):
            out.append(g["prompts"][t * ppt:(t + 1) * ppt] if need[6 * T + t] else None)
        for i, n in enumerate(("state_emb", "w_q", "w_k", "w_v", "w_fc", "b_fc", "ln_g", "ln_b")):
            out.append(g[n] if need[7 * T + i] else None)
        return (None,) * 9 + tuple(out)


def _dropout_arg(dropout, B: int, C_: int, P: int, mode: int, dev):
    """(team_dropout or None, its workspace) for ``dropout`` = None or (p, seed, offset)."""
    if dropout is None or float(dropout[0]) == 0.0:
        return None, None
    p, seed, offset = float(dropout[0]), int(dropout[1]), int(dropout[2])
    if not 0.0 < p < 1.0:
        raise ValueError(f"dropout p = {p} out of [0, 1)")
    n = capi.lib().team_head_dropout_workspace_bytes(B, C_, P, mode)
    dws = torch.empty((n,), dtype=torch.uint8, device=dev)
    dr = capi.Dropout(p, seed & 0xFFFFFFFFFFFFFFFF, offset & 0xFFFFFFFFFFFFFFFF, None, dws.data_ptr(), n)
    return C.pointer(dr), dws


def forward_tri_modal(pack: HeadParamPack, image: torch.Tensor, text: torch.Tensor,
                      state_ids: torch.Tensor, img_prototypes: torch.Tensor, *,
                      text_cls: Optional[torch.Tensor] = None, mode: int = MODE_F32, dropout=None):
    """(image[B,512], text[B,1,512], state[B,512], proto[B,512]) [+ (cls_logits[B,Tc], argmax[B])].
    ``image``/``text`` are post-CLIP 512-d features (per-sample text).  ``dropout`` = (p, seed, offset): sel_attn in train
    mode, with the masks ``mha(..., dropout_p=p, seed=seed, offset=offset)`` draws on the token tensor
    [image | text | state | C prototypes | P prompts]; the backward reuses the same masks.  None or p = 0: eval mode."""
    return _TriModalFn.apply(image, text, state_ids, img_prototypes, text_cls, mode, pack.T, pack.ppt, dropout,
                             *pack.flat)


def encode(pack: HeadParamPack, which: str, x: Optional[torch.Tensor], img_prototypes: Optional[torch.Tensor] = None,
           normalize: bool = False, mode: int = MODE_F32) -> torch.Tensor:
    """encode_image / encode_text / encode_state / encode_prototpyes without autograd
    (utils/inc_net.py:401-422, :518-526)."""
    capi.require_device()
    idx = {"image": 0, "text": 1, "state": 2, "prototypes": 3}[which]
    dev = pack.flat[0].device
    flat = [_f32c(p, dev) for p in pack.flat]
    protos = _f32c(img_prototypes, dev) if img_prototypes is not None else torch.zeros((1, capi.D), device=dev)
    hw = _fill_weights(pack.T, pack.ppt, flat, protos)
    if idx == 3:
        n, xp = protos.shape[0], None
    elif idx == 2:
        x = _check_state_ids(x.detach().to(device=dev, dtype=torch.int64).contiguous()); n, xp = x.shape[0], x.data_ptr()
    else:
        x = _f32c(x, dev); n, xp = x.shape[0], x.data_ptr()
    L = capi.lib()
    nbytes = L.team_head_workspace_bytes(n if idx <= 1 else 1, hw.num_classes, pack.T * pack.ppt, 0, mode)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    out = torch.empty((n, capi.D), dtype=torch.float32, device=dev)
    capi.check(L.team_head_encode(C.byref(hw), mode, idx, xp, n, int(normalize), out.data_ptr(),
                                  ws.data_ptr(), nbytes, _stream_ptr()), "team_head_encode")
    return out


def forward_proof(pack: HeadParamPack, image: torch.Tensor, text: torch.Tensor, img_prototypes: torch.Tensor, *,
                  inputs_encoded: bool = False, mode: int = MODE_F32):
    """PROOF fusion forward - ``Proof_Net.forward`` (utils/inc_net.py:436-463) on post-CLIP features, or
    ``forward_transformer(..., transformer=True)`` (:465-492) when ``inputs_encoded`` (rows already projected +
    normalised).  Returns (image [B,512], text [Tn,512] batch mean, proto [C,512] batch mean).  No autograd."""
    capi.require_device()
    if not image.is_cuda:
        raise capi.TeamB200Error("forward_proof needs CUDA tensors (no CPU fallback)")
    dev = image.device
    image, text, protos = _f32c(image, dev), _f32c(text, dev), _f32c(img_prototypes, dev)
    B, Tn = image.shape[0], text.shape[0]
    if image.shape != (B, capi.D) or text.shape != (Tn, capi.D) or B < 1 or Tn < 1:
        raise ValueError("image must be [B,512] and text [num_text,512]")
    flat = [_f32c(p, dev) for p in pack.flat]
    hw = _fill_weights(pack.T, pack.ppt, flat, protos)
    L = capi.lib()
    nbytes = L.team_head_workspace_bytes(B, Tn + hw.num_classes, pack.T * pack.ppt, Tn, mode)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    o_img = torch.empty((B, capi.D), dtype=torch.float32, device=dev)
    o_txt = torch.empty((Tn, capi.D), dtype=torch.float32, device=dev)
    o_pro = torch.empty((hw.num_classes, capi.D), dtype=torch.float32, device=dev)
    capi.check(L.team_head_proof_fwd(C.byref(hw), mode, B, image.data_ptr(), text.data_ptr(), Tn, int(inputs_encoded),
                                     o_img.data_ptr(), o_txt.data_ptr(), o_pro.data_ptr(), ws.data_ptr(), nbytes,
                                     _stream_ptr()), "team_head_proof_fwd")
    return o_img, o_txt, o_pro


def forward_tri_modal_class_text(pack: HeadParamPack, image: torch.Tensor, text: torch.Tensor, state_ids: torch.Tensor,
                                 img_prototypes: torch.Tensor, *, mode: int = MODE_F32):
    """``forward_tri_modal`` when ``text`` holds class texts ([Tn,512], Tn != batch; utils/inc_net.py:544-547,
    :573-574): (image [B,512], text [B,512] = mean over the Tn text rows, state [B,512], proto [B,512]).  No autograd."""
    capi.require_device()
    if not image.is_cuda:
        raise capi.TeamB200Error("forward_tri_modal needs CUDA tensors (no CPU fallback)")
    dev = image.device
    image, text, protos = _f32c(image, dev), _f32c(text, dev), _f32c(img_prototypes, dev)
    sid = _check_state_ids(state_ids.detach().to(device=dev, dtype=torch.int64).contiguous())
    B, Tn = image.shape[0], text.shape[0]
    if image.shape != (B, capi.D) or text.shape != (Tn, capi.D) or sid.shape != (B,) or B < 1 or Tn < 1:
        raise ValueError("image must be [B,512], text [num_text,512], state_ids [B]")
    flat = [_f32c(p, dev) for p in pack.flat]
    hw = _fill_weights(pack.T, pack.ppt, flat, protos)
    L = capi.lib()
    nbytes = L.team_head_workspace_bytes(B, Tn + hw.num_classes, pack.T * pack.ppt, Tn, mode)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    outs = torch.empty((4, B, capi.D), dtype=torch.float32, device=dev)
    capi.check(L.team_head_tri_classtext_fwd(C.byref(hw), mode, B, image.data_ptr(), text.data_ptr(), Tn, sid.data_ptr(),
                                             outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), outs[3].data_ptr(),
                                             ws.data_ptr(), nbytes, _stream_ptr()), "team_head_tri_classtext_fwd")
    # a single text row is not averaged away by the reference: it comes back as [B,1,512] (utils/inc_net.py:573-574)
    return outs[0], (outs[1].view(B, 1, capi.D) if Tn == 1 else outs[1]), outs[2], outs[3]


class _EncodeFn(torch.autograd.Function):
    """encode_image / encode_text / encode_state / encode_prototpyes with autograd to the projections (and, for the
    state modality, to the embedding table): the ClipLoss branch of the training step (models/proof.py:428-431) and the
    differentiable PROOF / class-text forms.  idx: 0 image (also prototype rows, which go through projs_img), 1 text,
    2 state (x = int64 state ids).  No gradient flows into the (frozen-backbone) features."""

    @staticmethod
    def forward(ctx, x, idx, normalize, mode, T, ppt, *params):
        capi.require_device()
        if not x.is_cuda:
            raise capi.TeamB200Error("encode needs CUDA tensors (no CPU fallback)")
        dev = x.device
        flat = [_f32c(p, dev) for p in params]
        hw = _fill_weights(T, ppt, flat, torch.zeros((1, capi.D), device=dev))
        if idx == 2:
            x = _check_state_ids(x.detach().to(device=dev, dtype=torch.int64).contiguous())
        else:
            x = _f32c(x, dev)
        n = x.shape[0]
        L = capi.lib()
        nbytes = L.team_head_workspace_bytes(max(n, 1), 1, T * ppt, 0, mode)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        out = torch.empty((n, capi.D), dtype=torch.float32, device=dev)
        capi.check(L.team_head_encode(C.byref(hw), mode, idx, x.data_ptr(), n, int(normalize), out.data_ptr(),
                                      ws.data_ptr(), nbytes, _stream_ptr()), "team_head_encode")
        ctx.hold = (x, flat)
        ctx.meta = (idx, int(normalize), mode, T, ppt, n, nbytes)
        return out

    @staticmethod
    def backward(ctx, g_out):
        x, flat = ctx.hold
        idx, normalize, mode, T, ppt, n, nbytes = ctx.meta
        dev = x.device
        hw = _fill_weights(T, ppt, flat, torch.zeros((1, capi.D), device=dev))
        gw = torch.empty((capi.D, capi.D), dtype=torch.float32, device=dev)
        gb = torch.empty((capi.D,), dtype=torch.float32, device=dev)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        g = _f32c(g_out, dev)
        need = ctx.needs_input_grad[6:]
        out: List[Optional[torch.Tensor]] = [None] * len(need)
        if idx == 2:
            # rows = E[state_ids] (a gather: data movement); dE = the input-row gradients summed by state id
            # (the library's deterministic keyed sum)
            from . import ops
            rows = flat[7 * T].index_select(0, x).contiguous()
            gx = torch.empty((n, capi.D), dtype=torch.float32, device=dev) if need[7 * T] else None
            capi.check(capi.lib().team_head_encode_rows_bwd(C.byref(hw), mode, 2, rows.data_ptr(), n, normalize, g.data_ptr(),
                                                            gw.data_ptr(), gb.data_ptr(), gx.data_ptr() if gx is not None else None,
                                                            ws.data_ptr(), nbytes, _stream_ptr()), "team_head_encode_rows_bwd")
            if gx is not None:
                out[7 * T] = ops.keyed_sums(gx, x, num_classes=capi.NUM_STATES)[0]
        else:
            capi.check(capi.lib().team_head_encode_bwd(C.byref(hw), mode, idx, x.data_ptr(), n, normalize, g.data_ptr(),
                                                       gw.data_ptr(), gb.data_ptr(), ws.data_ptr(), nbytes, _stream_ptr()),
                       "team_head_encode_bwd")
        for t in range(T):                       # W = sum_t W_t  =>  dW_t = dW for every unfrozen t
            if need[2 * idx * T + t]:
                out[2 * idx * T + t] = gw
            if need[(2 * idx + 1) * T + t]:
                out[(2 * idx + 1) * T + t] = gb
        return (None,) * 6 + tuple(out)


def encode_grad(pack: HeadParamPack, which: str, x: torch.Tensor, normalize: bool = False, mode: int = MODE_F32):
    """Differentiable encode_image / encode_text / encode_state / encode_prototpyes (utils/inc_net.py:401-422, :518-526;
    ``which='prototypes'``: ``x`` = img_prototypes, pushed through projs_img)."""
    idx = {"image": 0, "text": 1, "state": 2, "prototypes": 0}[which]
    if x.shape[0] == 0:
        return torch.empty((0, capi.D), dtype=torch.float32, device=x.device)
    return _EncodeFn.apply(x, idx, normalize, mode, pack.T, pack.ppt, *pack.flat)


class _MhaFn(torch.autograd.Function):
    """MultiHeadAttention.forward (convs/projections.py:64-87) on arbitrary [B, L, 512] tokens: team_mha_fwd / team_mha_bwd."""

    @staticmethod
    def forward(ctx, q, k, v, mode, w_q, w_k, w_v, w_fc, b_fc, ln_g, ln_b, dropout_p=0.0, seed=0, offset=0):
        capi.require_device()
        if not q.is_cuda:
            raise capi.TeamB200Error("sel_attn needs CUDA tensors (no CPU fallback)")
        dev = q.device
        same = (k is q, v is q)
        q = _f32c(q, dev)
        k = q if same[0] else _f32c(k, dev)
        v = q if same[1] else _f32c(v, dev)
        if q.dim() != 3 or k.dim() != 3 or q.shape[2] != capi.D or k.shape[2] != capi.D or k.shape != v.shape or k.shape[0] != q.shape[0]:
            raise ValueError("sel_attn: q [B,Lq,512], k / v [B,Lk,512]")
        B, Lq, Lk = q.shape[0], q.shape[1], k.shape[1]
        par = [_f32c(p, dev) for p in (w_q, w_k, w_v, w_fc, b_fc, ln_g, ln_b)]
        L = capi.lib()
        nbytes = L.team_mha_workspace_bytes(B, Lq, Lk)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        out = torch.empty((B, Lq, capi.D), dtype=torch.float32, device=dev)
        drop = (float(dropout_p), int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset) & 0xFFFFFFFFFFFFFFFF)
        capi.check(L.team_mha_fwd(mode, B, Lq, Lk, q.data_ptr(), k.data_ptr(), v.data_ptr(), *[p.data_ptr() for p in par],
                                  *drop, out.data_ptr(), ws.data_ptr(), nbytes, _stream_ptr()), "team_mha_fwd")
        ctx.hold = (q, k, v, par, ws)
        ctx.meta = (mode, B, Lq, Lk, nbytes, drop)
        return out

    @staticmethod
    def backward(ctx, g_out):
        q, k, v, par, ws = ctx.hold
        mode, B, Lq, Lk, nbytes, drop = ctx.meta
        dev = q.device
        g = _f32c(g_out, dev)
        need = ctx.needs_input_grad
        mk = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
        gq = mk(B, Lq, capi.D) if need[0] else None
        gk = mk(B, Lk, capi.D) if need[1] else None
        gv = mk(B, Lk, capi.D) if need[2] else None
        gw = [mk(capi.D, capi.D) for _ in range(4)] + [mk(capi.D) for _ in range(3)]
        ptr = lambda t: t.data_ptr() if t is not None else None
        w_q, w_k, w_v, w_fc, b_fc, ln_g, ln_b = par
        capi.check(capi.lib().team_mha_bwd(mode, B, Lq, Lk, q.data_ptr(), k.data_ptr(), v.data_ptr(), w_q.data_ptr(), w_k.data_ptr(),
                                           w_v.data_ptr(), w_fc.data_ptr(), ln_g.data_ptr(), *drop, g.data_ptr(), ptr(gq), ptr(gk), ptr(gv),
                                           *[t.data_ptr() for t in gw], ws.data_ptr(), nbytes, _stream_ptr()), "team_mha_bwd")
        return (gq, gk, gv, None) + tuple(t if need[4 + i] else None for i, t in enumerate(gw)) + (None, None, None)


def mha(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, w_q, w_k, w_v, w_fc, b_fc, ln_g, ln_b, mode: int = MODE_F32,
        dropout_p: float = 0.0, seed: int = 0, offset: int = 0):
    """Standalone ``sel_attn(q, k, v)`` (convs/projections.py:64-87), differentiable.  ``dropout_p`` > 0: train mode, the
    two dropouts of the block with counter-based masks keyed by ``(seed, offset)`` (``offset`` and ``offset + 1`` are used)."""
    return _MhaFn.apply(q, k, v, mode, w_q, w_k, w_v, w_fc, b_fc, ln_g, ln_b, dropout_p, seed, offset)


def dropout_keep_mask(n: int, dropout_p: float, seed: int, offset: int, device="cuda") -> torch.Tensor:
    """The 0 / 1 keep mask ``team_mha_fwd`` applies to a tensor of ``n`` elements under ``(dropout_p, seed, offset)``."""
    capi.require_device()
    keep = torch.empty((n,), dtype=torch.uint8, device=device)
    capi.check(capi.lib().team_dropout_keep_mask(keep.data_ptr(), n, float(dropout_p), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                                 int(offset) & 0xFFFFFFFFFFFFFFFF, _stream_ptr()), "team_dropout_keep_mask")
    return keep


class _MeanFn(torch.autograd.Function):
    """torch.mean(x, dim) for the batch / row means of the PROOF and class-text forms (utils/inc_net.py:458-459, :573-576)."""

    @staticmethod
    def forward(ctx, x, dim):
        capi.require_device()
        x = _f32c(x, x.device)
        dim = dim % x.dim()
        outer = int(torch.tensor(x.shape[:dim]).prod()) if dim > 0 else 1
        red = x.shape[dim]
        inner = int(torch.tensor(x.shape[dim + 1:]).prod()) if dim + 1 < x.dim() else 1
        out = torch.empty(x.shape[:dim] + x.shape[dim + 1:], dtype=torch.float32, device=x.device)
        capi.check(capi.lib().team_mean_mid(x.data_ptr(), out.data_ptr(), outer, red, inner, _stream_ptr()), "team_mean_mid")
        ctx.meta = (tuple(x.shape), outer, red, inner)
        return out

    @staticmethod
    def backward(ctx, g):
        shape, outer, red, inner = ctx.meta
        g = _f32c(g, g.device)
        dx = torch.empty(shape, dtype=torch.float32, device=g.device)
        capi.check(capi.lib().team_mean_mid_bwd(g.data_ptr(), dx.data_ptr(), outer, red, inner, _stream_ptr()), "team_mean_mid_bwd")
        return dx, None


def mean_dim(x: torch.Tensor, dim: int) -> torch.Tensor:
    return _MeanFn.apply(x, dim)


class _EmbeddingFn(torch.autograd.Function):
    """nn.Embedding lookup of InsectLifecycleModel.get_state_embeddings (models/state_evolution.py:45-47): the forward is
    a row gather, the backward the library's deterministic keyed sum of the row gradients by state id."""

    @staticmethod
    def forward(ctx, weight, ids):
        ids = _check_state_ids(ids.detach().to(device=weight.device, dtype=torch.int64).contiguous().reshape(-1), weight.shape[0])
        ctx.hold = (ids,)
        ctx.meta = (weight.shape[0],)
        return weight.detach().index_select(0, ids)

    @staticmethod
    def backward(ctx, g):
        from . import ops
        (ids,) = ctx.hold
        return ops.keyed_sums(_f32c(g, g.device), ids, num_classes=ctx.meta[0])[0], None


def embedding(weight: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
    shape = tuple(ids.shape)
    return _EmbeddingFn.apply(weight, ids).reshape(shape + (weight.shape[1],))


def linear(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """Proj_Pure_MLP.forward (convs/projections.py:7-18) on its own: x W^T + b for [*,512] inputs (no autograd)."""
    capi.require_device()
    if not x.is_cuda:
        raise capi.TeamB200Error("linear needs CUDA tensors (no CPU fallback)")
    dev = x.device
    shape = x.shape
    x2 = _f32c(x.reshape(-1, capi.D), dev)
    w, b = _f32c(weight, dev), _f32c(bias, dev)
    hw = capi.HeadWeights()
    hw.num_tasks, hw.prompts_per_task, hw.num_classes = 1, 0, 1
    hw.w_img[0], hw.b_img[0] = w.data_ptr(), b.data_ptr()
    hw.w_text[0], hw.b_text[0] = w.data_ptr(), b.data_ptr()
    hw.w_state[0], hw.b_state[0] = w.data_ptr(), b.data_ptr()
    n = x2.shape[0]
    out = torch.empty((n, capi.D), dtype=torch.float32, device=dev)
    if n == 0:
        return out.reshape(shape)
    L = capi.lib()
    nbytes = L.team_head_workspace_bytes(n, 1, 0, 0, MODE_F32)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    capi.check(L.team_head_encode(C.byref(hw), MODE_F32, 0, x2.data_ptr(), n, 0, out.data_ptr(), ws.data_ptr(), nbytes,
                                  _stream_ptr()), "team_head_encode")
    return out.reshape(shape)


# order of the flat gradient buffer = order in which the backward finishes its groups (w_fc first, then
# w_q / w_k / w_v, then everything else), so each all-reduce bucket is one contiguous slice
GRAD_LAYOUT = (("w_fc", capi.D * capi.D),
               ("w_q", capi.D * capi.D), ("w_k", capi.D * capi.D), ("w_v", capi.D * capi.D),
               ("w_img", capi.D * capi.D), ("b_img", capi.D), ("w_text", capi.D * capi.D), ("b_text", capi.D),
               ("w_state", capi.D * capi.D), ("b_state", capi.D), ("state_emb", capi.NUM_STATES * capi.D),
               ("b_fc", capi.D), ("ln_g", capi.D), ("ln_b", capi.D))


class HeadStepRunner:
    """Pre-allocated fwd+bwd step over the C ABI (no autograd tape, no allocation per step), the
    form a training loop or a CUDA graph replays.  All trainable-parameter gradients land in ONE
    flat fp32 buffer (``flat_grads``: the 1.85 M-element bucket that is all-reduced under data
    parallelism, SURVEY 8e)."""

    def __init__(self, pack: HeadParamPack, img_prototypes: torch.Tensor, batch: int, num_text_cls: int,
                 mode: int = MODE_F32, grad_events: bool = False, grad_buffer: Optional[torch.Tensor] = None,
                 peer=None, dropout_p: float = 0.0, seed: Optional[int] = None):
        """``peer``: a ``parallel.PeerAllReduce`` whose ``buffer`` becomes the gradient buffer; the backward then
        sums the gradients over the ranks itself (early bucket under its last kernels, late bucket at its end).
        ``dropout_p`` > 0: sel_attn in train mode (the masks of ``forward_tri_modal(dropout=(p, seed, offset))``).  The
        runner owns the dropout workspace and a device-resident offset (``offset_dev``, initially 2 randint(0, 2^62) from
        torch's CPU generator, as MultiHeadAttention.forward draws it; ``seed`` defaults to ``torch.initial_seed()``);
        ``advance_offset`` moves it to the next step's masks on the device, so a captured step draws fresh masks on
        every replay."""
        capi.require_device()
        dev = pack.flat[0].device
        self.dev, self.B, self.mode, self.n_cls = dev, batch, mode, num_text_cls
        if peer is not None:
            grad_buffer = peer.buffer
        self.pack = pack
        self.flat = [_f32c(p, dev) for p in pack.flat]
        self.protos = _f32c(img_prototypes, dev)
        self.hw = _fill_weights(pack.T, pack.ppt, self.flat, self.protos)
        L = capi.lib()
        self._frozen = None
        self.refresh_frozen()
        self.nbytes = L.team_head_workspace_bytes(batch, self.hw.num_classes, pack.T * pack.ppt, num_text_cls, mode)
        self.ws = torch.empty((self.nbytes,), dtype=torch.uint8, device=dev)
        self.outs = torch.empty((4, batch, capi.D), dtype=torch.float32, device=dev)
        self.dropout_p = float(dropout_p)
        self._drop = None
        if self.dropout_p != 0.0:
            if not 0.0 < self.dropout_p < 1.0:
                raise ValueError(f"dropout_p = {dropout_p} out of [0, 1)")
            self.seed = int(torch.initial_seed() if seed is None else seed) & 0xFFFFFFFFFFFFFFFF
            base = int(torch.randint(0, 2 ** 62, (1,)).item()) * 2
            self.offset_dev = torch.tensor([base], dtype=torch.int64, device=dev)      # read as uint64 by the kernels
            n = L.team_head_dropout_workspace_bytes(batch, self.hw.num_classes, pack.T * pack.ppt, mode)
            self.drop_ws = torch.empty((n,), dtype=torch.uint8, device=dev)
            self._drop = C.pointer(capi.Dropout(self.dropout_p, self.seed, base, self.offset_dev.data_ptr(), self.drop_ws.data_ptr(), n))
        self.logits = torch.empty((batch, max(num_text_cls, 1)), dtype=torch.float32, device=dev)
        self.argmax = torch.empty((batch,), dtype=torch.int64, device=dev)
        P = pack.T * pack.ppt
        n = self.grad_numel(pack)
        if grad_buffer is not None:              # e.g. parallel.PeerAllReduce.buffer (symmetric memory)
            if grad_buffer.numel() != n or grad_buffer.dtype != torch.float32 or not grad_buffer.is_contiguous():
                raise ValueError(f"grad_buffer must be a contiguous fp32 tensor of {n} elements")
            self.flat_grads = grad_buffer
        else:
            self.flat_grads = torch.zeros((n,), dtype=torch.float32, device=dev)
        self.hg = capi.HeadGrads()
        self.grad_views: Dict[str, torch.Tensor] = {}
        off = 0
        for name, sz in GRAD_LAYOUT + (("prompts", max(P, 1) * capi.D),):
            v = self.flat_grads[off:off + sz]
            self.grad_views[name] = v
            setattr(self.hg, name, v.data_ptr())
            off += sz
        self._comm = None
        if peer is not None:
            self._comm = peer.comm_struct(4 * capi.D * capi.D)       # early bucket = w_fc, w_q, w_k, w_v
            self.hg.comm = C.pointer(self._comm)
        # all-reduce buckets in the order the backward completes them (see team_head_grads.ev_*)
        d2 = capi.D * capi.D
        self.buckets = (self.flat_grads[:d2], self.flat_grads[d2:4 * d2], self.flat_grads[4 * d2:])
        self.ready_events = None
        self.comm_stream = None
        if grad_events:
            # external=True: recorded from inside a captured graph, waited on by a stream outside it
            self.ready_events = [torch.cuda.Event(external=True) for _ in range(2)]
            for ev in self.ready_events:
                ev.record()                       # materialises the handle
            torch.cuda.current_stream().synchronize()
            self.hg.ev_w_fc = self.ready_events[0].cuda_event
            self.hg.ev_w_qkv = self.ready_events[1].cuda_event
            self.comm_stream = torch.cuda.Stream(device=dev)

    def refresh_frozen(self):
        """The projections of the old tasks are frozen (utils/inc_net.py:392-393, :494-502; requires_grad False on every
        one of them): their sums are computed ONCE here (``team_head_frozen_sums``) and the step prologue adds only the
        newest task (``team_head_weights.num_frozen``).  Call again after loading other values into those parameters."""
        T = self.pack.T
        old = [p for k in range(6) for p in self.pack.flat[k * T:k * T + T - 1]]
        self._frozen_src = old
        self._frozen_ver = [p._version for p in old]
        if T < 2 or any(p.requires_grad for p in old):
            self.hw.num_frozen = 0
            return
        if self._frozen is None:
            self._frozen = (torch.empty((3, capi.D, capi.D), dtype=torch.float32, device=self.dev),
                            torch.empty((3, capi.D), dtype=torch.float32, device=self.dev))
        fw, fb = self._frozen
        self.hw.num_frozen = 0
        capi.check(capi.lib().team_head_frozen_sums(C.byref(self.hw), T - 1, fw.data_ptr(), fb.data_ptr(), _stream_ptr()),
                   "team_head_frozen_sums")
        for k in range(3):
            self.hw.w_frozen[k] = fw[k].data_ptr()
            self.hw.b_frozen[k] = fb[k].data_ptr()
        self.hw.num_frozen = T - 1
        # the sums are consumed by steps that may run on OTHER streams (a capture stream, a pipeline's compute stream): make
        # them visible now (once per task; not possible - and not needed, same stream - while that stream is being captured)
        if not torch.cuda.is_current_stream_capturing():
            torch.cuda.current_stream().synchronize()

    @staticmethod
    def grad_numel(pack: HeadParamPack) -> int:
        return sum(sz for _, sz in GRAD_LAYOUT) + max(pack.T * pack.ppt, 1) * capi.D

    def allreduce_grads(self, group=None):
        """Sum ``flat_grads`` over the ranks.  Call right after the step (eager call or graph replay) has been
        enqueued on the current stream.  With ``grad_events`` the three buckets are reduced on a side stream as
        soon as the backward has finished each of them (w_fc, then w_q/w_k/w_v, then the rest), overlapping the
        remaining kernels of the step; the current stream then waits for the side stream."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return
        if self.ready_events is None:
            dist.all_reduce(self.flat_grads, group=group)
            return
        cur = torch.cuda.current_stream()
        done = torch.cuda.Event()
        done.record(cur)                           # end of the step as enqueued so far
        with torch.cuda.stream(self.comm_stream):
            self.comm_stream.wait_event(self.ready_events[0])
            dist.all_reduce(self.buckets[0], group=group)
            self.comm_stream.wait_event(self.ready_events[1])
            dist.all_reduce(self.buckets[1], group=group)
            self.comm_stream.wait_event(done)
            dist.all_reduce(self.buckets[2], group=group)
        cur.wait_stream(self.comm_stream)

    def forward(self, image, text, sid, text_cls=None):
        if self.hw.num_frozen and any(p._version != v for p, v in zip(self._frozen_src, self._frozen_ver)):
            self.refresh_frozen()              # an old task's projection was written to (load_state_dict, ...): re-sum
        n_cls = self.n_cls if text_cls is not None else 0
        capi.check(capi.lib().team_head_tri_fwd(
            C.byref(self.hw), self.mode, self.B, image.data_ptr(), text.data_ptr(), sid.data_ptr(),
            text_cls.data_ptr() if n_cls else None, n_cls,
            self.outs[0].data_ptr(), self.outs[1].data_ptr(), self.outs[2].data_ptr(), self.outs[3].data_ptr(),
            self.logits.data_ptr() if n_cls else None, self.argmax.data_ptr() if n_cls else None,
            self.ws.data_ptr(), self.nbytes, _stream_ptr(), self._drop), "team_head_tri_fwd")

    def own_rows(self) -> torch.Tensor:
        """[2B,512] view of normalize(encode_image(x)) | normalize(encode_text(t)) as the last ``forward`` left them in the
        workspace (``team_head_own_rows_offset``): the inputs of the ClipLoss branch (models/proof.py:428-430)."""
        off = capi.lib().team_head_own_rows_offset(self.B, self.hw.num_classes, self.pack.T * self.pack.ppt, self.n_cls, self.mode)
        return self.ws[off:off + 2 * self.B * capi.D * 4].view(torch.float32).view(2 * self.B, capi.D)

    def backward(self, image, text, sid, cots, g_own_rows: Optional[torch.Tensor] = None):
        """``cots[3]`` (cotangent of the prototype output) may be None, a zero cotangent (team_head_tri_bwd).
        ``g_own_rows``: optional extra cotangent [2B,512] (or [2,B,512]) on ``own_rows()`` (``team_head_grads.g_own_rows``)."""
        if g_own_rows is not None and (g_own_rows.numel() != 2 * self.B * capi.D or g_own_rows.dtype != torch.float32
                                       or not g_own_rows.is_contiguous()):
            raise ValueError("g_own_rows must be a contiguous fp32 [2B,512] tensor")
        self.hg.g_own_rows = g_own_rows.data_ptr() if g_own_rows is not None else None
        capi.check(capi.lib().team_head_tri_bwd(
            C.byref(self.hw), self.mode, self.B, image.data_ptr(), text.data_ptr(), sid.data_ptr(),
            cots[0].data_ptr(), cots[1].data_ptr(), cots[2].data_ptr(), cots[3].data_ptr() if cots[3] is not None else None,
            C.byref(self.hg), self.ws.data_ptr(), self.nbytes, _stream_ptr(), self._drop), "team_head_tri_bwd")

    def advance_offset(self):
        """Next step's dropout masks: offset_dev += 2 (the attention and fc streams of one step use offset and offset + 1),
        on the device and on the current stream - no host sync, so it can be captured with the step.  No-op at p = 0."""
        if self._drop is not None:
            capi.check(capi.lib().team_u64_add(self.offset_dev.data_ptr(), 2, _stream_ptr()), "team_u64_add")

    @property
    def offset(self) -> int:
        """The dropout offset the next forward uses (host read: synchronises)."""
        return int(self.offset_dev.item()) if self._drop is not None else 0

    def step(self, image, text, sid, text_cls, cots):
        self.forward(image, text, sid, text_cls)
        self.backward(image, text, sid, cots)


class HostBatchPipeline:
    """Training-loop form of the step for batches that live in (pinned) HOST memory - what a DataLoader
    hands to ``Learner._train_proj_with_replay`` (models/proof.py:403-451): every ``submit`` copies the
    batch host->device on a copy stream, replays the captured fwd+bwd step (one CUDA graph per input
    slot) on the compute stream and copies the step's predictions (``argmax`` of the classification
    logits, models/proof.py:415-418) device->host.  ``depth`` input slots let the copy of step i+1 run
    under the kernels of step i; ``submit`` returns the predictions of the step submitted ``depth - 1``
    calls earlier (None while the pipeline fills), ``drain`` returns the outstanding ones.

    The gradients of the most recent replay are in ``runner.flat_grads`` (the bucket a data-parallel
    caller all-reduces); ``after_step`` - if given - is called on the compute stream right after each
    replay (optimizer step / all-reduce), before the next replay can overwrite them."""

    def __init__(self, pack: HeadParamPack, img_prototypes: torch.Tensor, batch: int, text_cls: torch.Tensor,
                 mode: int = MODE_F32, depth: int = 2, after_step=None, grad_events: bool = False,
                 grad_buffer: Optional[torch.Tensor] = None, in_graph=None, peer=None):
        capi.require_device()
        if depth < 1:
            raise ValueError("depth must be >= 1")
        dev = pack.flat[0].device
        self.dev, self.B, self.depth, self.after_step = dev, batch, depth, after_step
        self.text_cls = _f32c(text_cls, dev)
        self.runner = HeadStepRunner(pack, img_prototypes, batch, int(self.text_cls.shape[0]), mode,
                                     grad_events=grad_events, grad_buffer=grad_buffer, peer=peer)
        self.in_graph = in_graph                 # optional callable captured right after the step (e.g. PeerAllReduce)
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.compute_stream = torch.cuda.Stream(device=dev)
        mk = lambda *s, dt=torch.float32: torch.empty(s, dtype=dt, device=dev)
        self.slots = []
        for _ in range(depth):
            self.slots.append({
                "image": mk(batch, capi.D), "text": mk(batch, capi.D), "state": mk(batch, dt=torch.int64),
                "cots": [mk(batch, capi.D) for _ in range(4)],
                "pred": torch.empty((batch,), dtype=torch.int64).pin_memory(),
                "loaded": torch.cuda.Event(), "free": torch.cuda.Event(), "done": torch.cuda.Event(),
                "graph": None, "busy": False})
        self._n = 0
        self.h2d_bytes_per_step = 0              # set by submit: bytes of the arguments that were host tensors
        self.d2h_bytes_per_step = batch * 8

    def _capture(self, sl):
        r = self.runner
        with torch.cuda.stream(self.compute_stream):
            r.step(sl["image"], sl["text"], sl["state"], self.text_cls, sl["cots"])       # warm (lazy init outside capture)
            self.compute_stream.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.compute_stream):
                r.step(sl["image"], sl["text"], sl["state"], self.text_cls, sl["cots"])
                if self.in_graph is not None:
                    self.in_graph()
        sl["graph"] = g

    def submit(self, image: torch.Tensor, text: torch.Tensor, state_ids: torch.Tensor, cotangents: Sequence[torch.Tensor]):
        """Host tensors in (pinned for real overlap): image/text [B,512] fp32, state_ids [B] int64, four
        cotangents [B,512] (the loss gradients w.r.t. the four feature outputs; the loss itself is the caller's -
        cotangents that are already device tensors are copied device-to-device)."""
        sl = self.slots[self._n % self.depth]
        self.h2d_bytes_per_step = sum(t.numel() * t.element_size() for t in (image, text, state_ids, *cotangents)
                                      if not t.is_cuda)
        out = None
        if sl["busy"]:
            sl["done"].synchronize()
            out = sl["pred"].clone()
            sl["busy"] = False
        with torch.cuda.stream(self.copy_stream):
            if sl["graph"] is not None:
                self.copy_stream.wait_event(sl["free"])          # the replay that last read this slot has finished
            sl["image"].copy_(image, non_blocking=True)
            sl["text"].copy_(text, non_blocking=True)
            sl["state"].copy_(state_ids, non_blocking=True)
            for d, s in zip(sl["cots"], cotangents):
                d.copy_(s.reshape(self.B, capi.D), non_blocking=True)
            sl["loaded"].record(self.copy_stream)
        if sl["graph"] is None:
            self.copy_stream.synchronize()
            self._capture(sl)
        with torch.cuda.stream(self.compute_stream):
            self.compute_stream.wait_event(sl["loaded"])
            sl["graph"].replay()
            sl["free"].record(self.compute_stream)
            if self.after_step is not None:
                self.after_step(self.runner)
            sl["pred"].copy_(self.runner.argmax, non_blocking=True)
            sl["done"].record(self.compute_stream)
        sl["busy"] = True
        self._n += 1
        return out

    def drain(self) -> List[torch.Tensor]:
        outs = []
        for k in range(self.depth):
            sl = self.slots[(self._n + k) % self.depth]
            if sl["busy"]:
                sl["done"].synchronize()
                outs.append(sl["pred"].clone())
                sl["busy"] = False
        return outs
