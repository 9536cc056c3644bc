"""The learner's inner-loop body (models/proof.py:403-451) after the frozen CLIP towers as ONE replayable CUDA graph.

    cls logits (no grad, :411-416) -> forward_tri_modal (:421-422) -> ClipLoss on the projected rows (:425-431)
    -> unicl_loss with evolution features (:434-441) -> total = ce + clip + 0.3 unicl (:442) -> backward (:444)
    -> AdamW step (:445)

`Learner._train_proj_with_replay` keeps working unchanged on `inc_net.Proof_Net` (tests/test_gpu_learner_dropin.py);
`TrainStep` is the fast form of the same loop body for callers that can hand over pre-extracted features: every
launch of the step - 50-odd library kernels - is captured once per epoch (the learner's cosine learning-rate schedule
and unicl's dynamic temperature change per epoch, :111-116, :363) and replayed per batch.  The Adam step count lives
on the device (`team_adamw_step_graph`).  Not captured (and not trained here): `convnet.logit_scale` - the captured
ClipLoss launch bakes its value in; pass the current value when an epoch's graph is captured.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch

from . import capi, head, ops


class TrainStep:
    def __init__(self, params: Dict[str, torch.Tensor], img_prototypes: torch.Tensor, batch: int, text_cls: torch.Tensor,
                 mode: int = head.MODE_BF16, init_lr: float = 0.004, min_lr: float = 1e-8, weight_decay: float = 0.05,
                 tuned_epoch: int = 20, logit_scale: float = math.exp(2.6592600369327783),
                 evolution_features=None, dropout_p: float = 0.0, seed: Optional[int] = None):
        """``params``: the network's parameters under their state_dict names (updated IN PLACE by ``step``).
        ``dropout_p`` > 0: sel_attn in train mode, as the learner trains it (models/proof.py:398).  Every replay draws
        fresh masks: step k (counted over all epochs) uses offset ``dropout_offset(k)`` = base + 2 k, advanced on the
        device inside the graph."""
        capi.require_device()
        self.params, self.mode, self.B = params, mode, batch
        self.pack = head.HeadParamPack.from_state_dict(params)
        pack = self.pack
        T = pack.T
        dev = pack.flat[0].device
        self.dev = dev
        self.text_cls = text_cls.to(device=dev, dtype=torch.float32).contiguous()
        self.runner = head.HeadStepRunner(pack, img_prototypes, batch, int(self.text_cls.shape[0]), mode,
                                          dropout_p=dropout_p, seed=seed)
        self.dropout_base = self.runner.offset
        gv = self.runner.grad_views
        P = pack.T * pack.ppt
        D = capi.D
        # trainable tensors (utils/inc_net.py:494-516: newest projections, sel_attn, state embedder) with their slices
        # of the flat gradient buffer
        self.pairs = [(params[f"projs_img.{T - 1}.MLP.0.weight"], gv["w_img"].view(D, D)), (params[f"projs_img.{T - 1}.MLP.0.bias"], gv["b_img"]),
                      (params[f"projs_text.{T - 1}.MLP.0.weight"], gv["w_text"].view(D, D)), (params[f"projs_text.{T - 1}.MLP.0.bias"], gv["b_text"]),
                      (params[f"projs_state.{T - 1}.MLP.0.weight"], gv["w_state"].view(D, D)), (params[f"projs_state.{T - 1}.MLP.0.bias"], gv["b_state"]),
                      (params[f"context_prompts.{T - 1}"], gv["prompts"].view(P, D)[(T - 1) * pack.ppt:]),
                      (params["state_embedder.state_embeddings.weight"], gv["state_emb"].view(10, D)),
                      (params["sel_attn.w_qs.weight"], gv["w_q"].view(D, D)), (params["sel_attn.w_ks.weight"], gv["w_k"].view(D, D)),
                      (params["sel_attn.w_vs.weight"], gv["w_v"].view(D, D)), (params["sel_attn.fc.weight"], gv["w_fc"].view(D, D)),
                      (params["sel_attn.fc.bias"], gv["b_fc"]), (params["sel_attn.layer_norm.weight"], gv["ln_g"]),
                      (params["sel_attn.layer_norm.bias"], gv["ln_b"])]
        for p, _ in self.pairs:
            p.requires_grad_(True)
        self.opt = ops.FusedAdamW([p for p, _ in self.pairs], lr=init_lr, weight_decay=weight_decay)
        self.init_lr, self.min_lr, self.tuned_epoch, self.logit_scale = init_lr, min_lr, tuned_epoch, float(logit_scale)
        self.evo = None
        if evolution_features is not None and len(evolution_features) > 0:
            self.evo = evolution_features if isinstance(evolution_features, tuple) else ops.pack_evolution_features(evolution_features, dev)
        mk = lambda *s, dt=torch.float32: torch.empty(s, dtype=dt, device=dev)
        # static inputs of the captured step
        self.image, self.text = mk(batch, D), mk(batch, D)
        self.state, self.labels = mk(batch, dt=torch.int64), mk(batch, dt=torch.int64)
        self._inputs = [self.image, self.text, self.state, self.labels]
        self.losses6 = torch.zeros((6,), dtype=torch.float32, device=dev)    # total, ce, clip, unicl total, unicl instance, unicl category
        self.losses = self.losses6[:5]
        self.g_own = torch.zeros((2, batch, D), dtype=torch.float32, device=dev)   # ClipLoss gradient w.r.t. the normalised own rows
        self._graphs: Dict[int, torch.cuda.CUDAGraph] = {}
        self._stream = torch.cuda.Stream(device=dev)
        self._side = torch.cuda.Stream(device=dev)

    def lr_at(self, epoch: int) -> float:
        """CosineAnnealingLR(T_max=tuned_epoch, eta_min=min_lr) stepped once per epoch (models/proof.py:363, :447)."""
        return self.min_lr + 0.5 * (self.init_lr - self.min_lr) * (1.0 + math.cos(math.pi * epoch / self.tuned_epoch))

    def _body(self, epoch: int):
        r, mode = self.runner, self.mode
        img, txt, sid, y = self.image, self.text, self.state, self.labels
        r.forward(img, txt, sid, self.text_cls)                                   # cls logits + the four feature outputs
        un, cots = ops.unicl_loss(r.outs[0], r.outs[1], r.outs[2], y, state_ids=sid, evolution_features=self.evo,
                                  epoch=epoch, max_epoch=self.tuned_epoch, grad_scale=0.3, mode=mode, losses_out=self.losses6[3:6])
        # ClipLoss branch (:428-431): its inputs normalize(encode_text(..)) / normalize(encode_image(..)) ARE the normalised
        # own rows the head's forward just produced, so the loss reads them in place and its gradient joins the head's
        # backward as an extra cotangent on those rows (team_head_grads.g_own_rows) - no second pass through the projections
        xo = r.own_rows()
        ops.clip_loss(xo[:self.B], xo[self.B:], self.logit_scale, mode=mode, grads_out=self.g_own, loss_out=self.losses6[2:3])
        # ce VALUE (the logits carry no gradient, :411-417) and total = ce + clip + 0.3 unicl (:442): one single-CTA launch on a
        # side stream beside the backward (a parallel branch of the captured graph), no host sync
        cur = torch.cuda.current_stream()
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            ops.ce_total(r.logits, y, self.losses6, w_clip=1.0, w_unicl=0.3)
        r.backward(img, txt, sid, [cots[0], cots[1], cots[2], None], g_own_rows=self.g_own)   # the losses never touch the prototype output
        r.advance_offset()                                                        # next step's dropout masks (no-op at p = 0)
        self.opt.lr = self.lr_at(epoch)
        self.opt.step_graph([g for _, g in self.pairs])
        cur.wait_stream(self._side)

    def _capture(self, epoch: int):
        st = self._stream
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            # warm-up outside the capture (lazy initialisation, autograd buffers) on a snapshot of the trainable state
            snap = [(p.detach().clone(), m.clone(), v.clone()) for p, m, v in zip(self.opt.params, self.opt.exp_avg, self.opt.exp_avg_sq)]
            step0 = self.opt.step_dev.clone()
            off0 = self.runner.offset_dev.clone() if self.runner.dropout_p else None
            self._body(epoch)
            st.synchronize()
            with torch.no_grad():
                for p, m, v, (p0, m0, v0) in zip(self.opt.params, self.opt.exp_avg, self.opt.exp_avg_sq, snap):
                    p.copy_(p0); m.copy_(m0); v.copy_(v0)
                self.opt.step_dev.copy_(step0)
                if off0 is not None:
                    self.runner.offset_dev.copy_(off0)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                self._body(epoch)
        torch.cuda.current_stream().wait_stream(st)
        self._graphs[epoch] = g

    def dropout_offset(self, k: int) -> int:
        """The dropout offset of optimisation step k (0-based, counted over all epochs): base + 2 k."""
        return self.dropout_base + 2 * k

    def load(self, image, text, state_ids, labels):
        """Copy one batch (host or device tensors) into the step's static input buffers on the current stream."""
        src = [image, text.reshape(self.B, capi.D), state_ids, labels]
        if all(t.is_cuda and t.dtype == d.dtype and t.is_contiguous() and t.shape == d.shape for t, d in zip(src, self._inputs)):
            # device-resident batch: one launch (team_copy_batch) instead of four device-to-device copies
            capi.check(capi.lib().team_copy_batch(*[t.data_ptr() for t in src], self.B, *[d.data_ptr() for d in self._inputs],
                                                  torch.cuda.current_stream().cuda_stream), "team_copy_batch")
        else:
            for d, t in zip(self._inputs, src):
                d.copy_(t, non_blocking=True)

    def step(self, epoch: int = 0):
        """One optimisation step on the loaded batch; returns the device tensor [total, ce, clip, unicl, unicl_instance]."""
        if epoch not in self._graphs:
            self._capture(epoch)
        self._graphs[epoch].replay()
        return self.losses
