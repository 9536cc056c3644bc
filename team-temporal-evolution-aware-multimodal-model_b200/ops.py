"""Thin torch-tensor wrappers over the C ABI for the bandwidth-bound ops of the path:
the keyed segmented sum (prototype build) and the cosine classifier.

torch is used only for device memory and the current stream; all arithmetic happens in
``libteam_b200.so``.  Inputs must be CUDA tensors - there is no CPU fallback."""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import capi


def _stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def _chk_rows(x: torch.Tensor, name: str):
    if not x.is_cuda:
        raise capi.TeamB200Error(f"{name} must be a CUDA tensor (no CPU fallback)")
    if x.dim() != 2 or x.shape[1] != capi.D:
        raise ValueError(f"{name} must be [N,{capi.D}], got {tuple(x.shape)}")
    if x.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError(f"{name} must be float32 or bfloat16, got {x.dtype}")
    return x.contiguous()


def _dt(x):
    return capi.DTYPE_F32 if x.dtype == torch.float32 else capi.DTYPE_BF16


def keyed_sums(x: torch.Tensor, labels: torch.Tensor, states: Optional[torch.Tensor] = None, *,
               class_base: int = 0, num_classes: int, num_states: int = capi.NUM_STATES,
               normalize_rows: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """Deterministic keyed segmented sum.  Returns (sums [K,512] fp32, counts [K] int64) with
    K = num_classes * (num_states if states is given else 1); key = (label-class_base)*S + state.
    Reference: models/proof.py:258-276, models/simplecil.py:48-55, utils/state_distance.py:98-103."""
    capi.require_device()
    x = _chk_rows(x, "x")
    n = x.shape[0]
    labels = labels.to(device=x.device, dtype=torch.int64).contiguous()
    if labels.shape != (n,):
        raise ValueError("labels must be [N]")
    if states is not None:
        states = states.to(device=x.device, dtype=torch.int64).contiguous()
        if states.shape != (n,):
            raise ValueError("states must be [N]")
    S = num_states if states is not None else 1
    K = num_classes * S
    sums = torch.empty((K, capi.D), dtype=torch.float32, device=x.device)
    counts = torch.empty((K,), dtype=torch.int64, device=x.device)
    L = capi.lib()
    ws_bytes = L.team_segsum_workspace_bytes(n, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=x.device)
    capi.check(L.team_segsum(x.data_ptr(), _dt(x), labels.data_ptr(),
                             states.data_ptr() if states is not None else None,
                             n, class_base, num_classes, S, int(normalize_rows),
                             sums.data_ptr(), counts.data_ptr(), ws.data_ptr(), ws_bytes, _stream_ptr()),
               "team_segsum")
    return sums, counts


def keyed_means(sums: torch.Tensor, counts: torch.Tensor, out: Optional[torch.Tensor] = None,
                group: int = 0, class_out: Optional[torch.Tensor] = None):
    """means[k] = sums[k]/counts[k] where counts[k] > 0 (other rows of ``out`` untouched).
    With ``group`` > 0 also folds every ``group`` consecutive keys into per-class means
    (written into ``class_out`` rows with a non-zero total) and returns the class counts."""
    capi.require_device()
    K = sums.shape[0]
    if out is None:
        out = torch.zeros_like(sums)
    L = capi.lib()
    if group:
        ng = K // group
        if class_out is None:
            class_out = torch.zeros((ng, capi.D), dtype=torch.float32, device=sums.device)
        ccounts = torch.empty((ng,), dtype=torch.int64, device=sums.device)
        capi.check(L.team_segmean_finalize(sums.data_ptr(), counts.data_ptr(), K, out.data_ptr(), group,
                                           class_out.data_ptr(), ccounts.data_ptr(), _stream_ptr()),
                   "team_segmean_finalize")
        return out, class_out, ccounts
    capi.check(L.team_segmean_finalize(sums.data_ptr(), counts.data_ptr(), K, out.data_ptr(), 1,
                                       None, None, _stream_ptr()), "team_segmean_finalize")
    return out


def cosine_logits(x: torch.Tensor, weight: torch.Tensor, sigma: Optional[torch.Tensor] = None, *,
                  want_logits: bool = True, want_argmax: bool = False):
    """sigma * normalize(x) @ normalize(weight).T (+ first-index argmax), one pass over x.
    Reference: convs/linears.py:51-61; models/proof.py:526-535."""
    capi.require_device()
    x = _chk_rows(x, "x")
    w = weight.detach().to(device=x.device, dtype=torch.float32).contiguous()
    if w.dim() != 2 or w.shape[1] != capi.D:
        raise ValueError("weight must be [C,512]")
    n, c = x.shape[0], w.shape[0]
    logits = torch.empty((n, c), dtype=torch.float32, device=x.device) if want_logits else None
    amax = torch.empty((n,), dtype=torch.int64, device=x.device) if want_argmax else None
    sg = None
    if sigma is not None:
        sg = sigma.detach().to(device=x.device, dtype=torch.float32).reshape(-1)[:1].contiguous()
    capi.check(capi.lib().team_cosine_logits(
        x.data_ptr(), _dt(x), n, w.data_ptr(), c, sg.data_ptr() if sg is not None else None,
        logits.data_ptr() if logits is not None else None,
        amax.data_ptr() if amax is not None else None, _stream_ptr()), "team_cosine_logits")
    if want_logits and want_argmax:
        return logits, amax
    return logits if want_logits else amax


def herding_select(features: torch.Tensor, m: int, group_sizes: Optional[Sequence[int]] = None):
    """Exemplar herding of ``BaseLearner._construct_exemplar`` (models/base.py:284-311, :335-341) for one class
    (``features`` [n,512]) or several (rows grouped by class, ``group_sizes`` = rows per class).  Returns
    (picked row indices within each class [G,m] int64 in pick order, exemplar means [G,512], class means [G,512]);
    G = 1 for a single class.  Every class needs at least ``m`` rows (the reference raises on fewer)."""
    capi.require_device()
    _chk_rows(features, "features")
    if features.dtype != torch.float32:
        raise TypeError("herding_select: fp32 features")
    n = features.shape[0]
    sizes = [n] if group_sizes is None else [int(v) for v in group_sizes]
    if sum(sizes) != n or any(v < m for v in sizes) or m < 1:
        raise ValueError(f"herding_select: every class needs >= m = {m} rows and the sizes must add up to {n} (got {sizes})")
    dev = features.device
    ptr = torch.tensor([0] + list(np.cumsum(sizes)), dtype=torch.int64).to(dev)
    G = len(sizes)
    L = capi.lib()
    nbytes = L.team_herding_workspace_bytes(n)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    idx = torch.empty((G, m), dtype=torch.int64, device=dev)
    emean = torch.empty((G, capi.D), dtype=torch.float32, device=dev)
    cmean = torch.empty((G, capi.D), dtype=torch.float32, device=dev)
    capi.check(L.team_herding_select(features.data_ptr(), ptr.data_ptr(), G, m, n, idx.data_ptr(), emean.data_ptr(),
                                     cmean.data_ptr(), ws.data_ptr(), nbytes, _stream_ptr()), "team_herding_select")
    return idx, emean, cmean


def dynamic_temperature(temperature: float = 0.07, epoch=None, max_epoch=None) -> float:
    """models/proof.py:111-116."""
    import math
    if epoch is None or max_epoch is None:
        return float(temperature)
    progress = float(epoch) / float(max_epoch)
    return float(temperature * (0.5 + 0.5 * 0.5 * (1.0 + math.cos(math.pi * progress))))


def pack_evolution_features(evolution_features, device):
    """``evolution_features`` as the reference passes it (a list indexed by class id, entries None or a 512-vector;
    Proof_Net.evolution_embeddings, utils/inc_net.py:594-617) -> (table [E,512] fp32, mask [E] uint8) on ``device``."""
    E = len(evolution_features)
    table = torch.zeros((E, capi.D), dtype=torch.float32, device=device)
    mask = torch.zeros((E,), dtype=torch.uint8, device=device)
    rows = [i for i, e in enumerate(evolution_features) if e is not None]
    if rows:
        table[rows] = torch.stack([evolution_features[i].detach().reshape(-1).to(device=device, dtype=torch.float32) for i in rows])
        mask[rows] = 1
    return table, mask


def unicl_loss(image: torch.Tensor, text: torch.Tensor, state: torch.Tensor, labels: torch.Tensor, *,
               state_ids: Optional[torch.Tensor] = None, evolution_features=None,
               temperature: float = 0.07, epoch=None, max_epoch=None, grad_scale: float = 1.0, mode: int = capi.MODE_F32,
               losses_out: Optional[torch.Tensor] = None):
    """unicl_loss (models/proof.py:21-191) forward + gradient in one call, including the ``evolution_features``
    branch (:51-106; pass the list the learner passes, or a ``(table, mask)`` pair from ``pack_evolution_features``).
    Returns (losses [3] = total / instance / category on the device, (g_image, g_text, g_state) [B,512] =
    grad_scale * d total / d input) - the gradients are the cotangents of the head's backward."""
    capi.require_device()
    B = image.shape[0]
    xs = [_chk_rows(t.detach().reshape(B, -1).float(), n) for t, n in ((image, "image"), (text, "text"), (state, "state"))]
    if B == 1:        # models/proof.py:41-45: a batch of one returns a zero loss (and therefore zero gradients)
        return (torch.zeros((3,), dtype=torch.float32, device=xs[0].device),
                tuple(torch.zeros((1, capi.D), dtype=torch.float32, device=xs[0].device) for _ in range(3)))
    dev = xs[0].device
    y = labels.detach().to(device=dev, dtype=torch.int64).contiguous()
    L = capi.lib()
    evo = None
    if evolution_features is not None and len(evolution_features) > 0:          # models/proof.py:52
        if state_ids is None:
            raise ValueError("unicl_loss: evolution_features needs state_ids")
        evo = evolution_features if isinstance(evolution_features, tuple) else pack_evolution_features(evolution_features, dev)
        sid = state_ids.detach().to(device=dev, dtype=torch.int64).contiguous()
        if sid.shape != (B,):
            raise ValueError("state_ids must be [B]")
        nbytes = L.team_loss_evo_workspace_bytes(B, evo[0].shape[0])
    else:
        nbytes = L.team_loss_workspace_bytes(B)
    if nbytes == 0:
        raise ValueError(f"unicl_loss: batch {B} out of range")
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    losses = losses_out if losses_out is not None else torch.empty((3,), dtype=torch.float32, device=dev)
    if losses.shape != (3,) or losses.dtype != torch.float32 or not losses.is_contiguous() or losses.device != dev:
        raise ValueError("unicl_loss: losses_out must be a contiguous fp32 [3] tensor on the inputs' device")
    grads = torch.empty((3, B, capi.D), dtype=torch.float32, device=dev)
    tau = dynamic_temperature(temperature, epoch, max_epoch)
    if evo is None:
        capi.check(L.team_unicl_loss(mode, xs[0].data_ptr(), xs[1].data_ptr(), xs[2].data_ptr(), y.data_ptr(), B,
                                     tau, float(grad_scale), losses.data_ptr(),
                                     grads[0].data_ptr(), grads[1].data_ptr(), grads[2].data_ptr(), ws.data_ptr(), nbytes,
                                     _stream_ptr()), "team_unicl_loss")
    else:
        capi.check(L.team_unicl_loss_evo(mode, xs[0].data_ptr(), xs[1].data_ptr(), xs[2].data_ptr(), y.data_ptr(),
                                         sid.data_ptr(), evo[0].data_ptr(), evo[1].data_ptr(), evo[0].shape[0], B,
                                         tau, float(grad_scale), losses.data_ptr(),
                                         grads[0].data_ptr(), grads[1].data_ptr(), grads[2].data_ptr(), ws.data_ptr(), nbytes,
                                         _stream_ptr()), "team_unicl_loss_evo")
    return losses, (grads[0], grads[1], grads[2])


def clip_loss(image: torch.Tensor, text: torch.Tensor, logit_scale: float, *, grad_scale: float = 1.0,
              mode: int = capi.MODE_F32, grads_out: Optional[torch.Tensor] = None, loss_out: Optional[torch.Tensor] = None):
    """ClipLoss.forward (utils/toolkit.py:128-141, world_size 1) forward + gradient: (loss [1], (g_image, g_text)).
    ``grads_out``: optional contiguous fp32 [2,B,512] buffer the two gradients are written to (image rows, then text rows -
    the layout of ``team_head_grads.g_own_rows``)."""
    capi.require_device()
    B = image.shape[0]
    xi, xt = _chk_rows(image.detach().float(), "image"), _chk_rows(text.detach().float(), "text")
    L = capi.lib()
    nbytes = L.team_loss_workspace_bytes(B)
    if nbytes == 0:
        raise ValueError(f"clip_loss: batch {B} out of range")
    dev = xi.device
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    loss = loss_out if loss_out is not None else torch.empty((1,), dtype=torch.float32, device=dev)
    if loss.shape != (1,) or loss.dtype != torch.float32 or loss.device != dev:
        raise ValueError("clip_loss: loss_out must be an fp32 [1] tensor on the inputs' device")
    grads = grads_out if grads_out is not None else torch.empty((2, B, capi.D), dtype=torch.float32, device=dev)
    if grads.shape != (2, B, capi.D) or grads.dtype != torch.float32 or not grads.is_contiguous() or grads.device != dev:
        raise ValueError("clip_loss: grads_out must be a contiguous fp32 [2,B,512] tensor on the inputs' device")
    capi.check(L.team_clip_loss(mode, xi.data_ptr(), xt.data_ptr(), B, float(logit_scale), float(grad_scale),
                                loss.data_ptr(), grads[0].data_ptr(), grads[1].data_ptr(), ws.data_ptr(), nbytes,
                                _stream_ptr()), "team_clip_loss")
    return loss, (grads[0], grads[1])


def ce_total(logits: torch.Tensor, labels: torch.Tensor, losses6: torch.Tensor, w_clip: float = 1.0, w_unicl: float = 0.3):
    """Cross-entropy VALUE of the no-grad classification logits (models/proof.py:417) and the learner's total (:442) written
    into ``losses6`` = [total, ce, clip, unicl, unicl_instance, unicl_category] (entries 2.. are read): ``team_ce_total``."""
    capi.require_device()
    if losses6.shape != (6,) or losses6.dtype != torch.float32 or not losses6.is_contiguous():
        raise ValueError("ce_total: losses6 must be a contiguous fp32 [6] tensor")
    lg = logits.detach().float().contiguous()
    y = labels.detach().to(device=lg.device, dtype=torch.int64).contiguous()
    capi.check(capi.lib().team_ce_total(lg.data_ptr(), y.data_ptr(), lg.shape[0], lg.shape[1], float(w_clip), float(w_unicl),
                                        losses6.data_ptr(), _stream_ptr()), "team_ce_total")
    return losses6


class FusedAdamW:
    """torch.optim.AdamW(params, lr, betas, eps, weight_decay).step() (models/proof.py:361, :445) as ONE kernel over
    all tensors (``team_adamw_step``).  ``step(grads)`` takes the gradients as a list aligned with ``params`` (e.g.
    views of ``HeadStepRunner.flat_grads``) or uses ``p.grad``; tensors whose gradient is None are skipped.
    ``lr`` may be changed between steps (the learner's cosine schedule, models/proof.py:363)."""

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1e-2):
        capi.require_device()
        self.params = [p for p in params if p.requires_grad]
        for p in self.params:
            if not p.is_cuda or p.dtype != torch.float32 or not p.is_contiguous():
                raise capi.TeamB200Error("FusedAdamW needs contiguous fp32 CUDA parameters (no CPU fallback)")
        self.lr, self.betas, self.eps, self.weight_decay = lr, betas, eps, weight_decay
        self.exp_avg = [torch.zeros_like(p) for p in self.params]
        self.exp_avg_sq = [torch.zeros_like(p) for p in self.params]
        self.steps = [0] * len(self.params)      # per tensor, like torch: a tensor without gradient does not advance
        # step count of step_graph, created here rather than on first use: a first use inside a CUDA graph capture would
        # allocate it from the graph's pool and capture its zero fill, so every replay would restart the count at 1
        self.step_dev = torch.zeros((1,), dtype=torch.int64, device=self.params[0].device) if self.params else None

    @torch.no_grad()
    def step(self, grads=None):
        import ctypes as C
        if grads is None:
            grads = [p.grad for p in self.params]
        by_step = {}
        for i, g in enumerate(grads):
            if g is None:
                continue
            self.steps[i] += 1
            by_step.setdefault(self.steps[i], []).append(i)
        L = capi.lib()
        for t, idx in by_step.items():           # normally one group: every tensor has seen the same number of steps
            for lo in range(0, len(idx), 48):
                chunk = idx[lo:lo + 48]
                n = len(chunk)
                vp = C.c_void_p * n
                gs = [grads[i].detach().to(torch.float32).contiguous() for i in chunk]
                capi.check(L.team_adamw_step(n, vp(*[self.params[i].data_ptr() for i in chunk]), vp(*[g.data_ptr() for g in gs]),
                                             vp(*[self.exp_avg[i].data_ptr() for i in chunk]),
                                             vp(*[self.exp_avg_sq[i].data_ptr() for i in chunk]),
                                             (C.c_int64 * n)(*[self.params[i].numel() for i in chunk]), float(self.lr),
                                             float(self.betas[0]), float(self.betas[1]), float(self.eps),
                                             float(self.weight_decay), t, _stream_ptr()), "team_adamw_step")

    @torch.no_grad()
    def step_graph(self, grads):
        """The same update in a form a CUDA graph can replay every step: the step count lives on the device
        (``self.step_dev``; every tensor must receive a gradient at every step).  ``lr`` is baked into the captured
        launch - re-capture when the schedule changes it (once per epoch for the learner's cosine schedule)."""
        import ctypes as C
        if any(g is None for g in grads) or len(grads) != len(self.params):
            raise ValueError("step_graph needs one gradient per parameter")
        L = capi.lib()
        idx = list(range(len(self.params)))
        for lo in range(0, len(idx), 48):
            chunk = idx[lo:lo + 48]
            n = len(chunk)
            vp = C.c_void_p * n
            capi.check(L.team_adamw_step_graph(n, vp(*[self.params[i].data_ptr() for i in chunk]), vp(*[grads[i].data_ptr() for i in chunk]),
                                               vp(*[self.exp_avg[i].data_ptr() for i in chunk]),
                                               vp(*[self.exp_avg_sq[i].data_ptr() for i in chunk]),
                                               (C.c_int64 * n)(*[self.params[i].numel() for i in chunk]), float(self.lr),
                                               float(self.betas[0]), float(self.betas[1]), float(self.eps),
                                               float(self.weight_decay), self.step_dev.data_ptr(),
                                               1 if lo + 48 >= len(idx) else 0, _stream_ptr()), "team_adamw_step_graph")

