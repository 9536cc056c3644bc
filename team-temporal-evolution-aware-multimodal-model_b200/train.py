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
`DataParallelTrainStep` is the same loop body on N GPUs of one box over a global batch (losses over the whole batch,
gradient summed over the ranks inside the graph).
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
        self.runner = self._make_runner(pack, img_prototypes, batch, int(self.text_cls.shape[0]), mode, dropout_p, seed)
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

    def _make_runner(self, pack, img_prototypes, batch, n_cls, mode, dropout_p, seed):
        return head.HeadStepRunner(pack, img_prototypes, batch, n_cls, mode, dropout_p=dropout_p, seed=seed)

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


class DataParallelTrainStep(TrainStep):
    """``TrainStep`` over a GLOBAL batch of ``world * batch`` samples, one rank per GPU: every rank loads its own
    ``batch`` samples (contiguous shards in rank order) and replays one CUDA graph per epoch holding

        head forward -> loss phase 0 -> all-gather 0 -> phase 1 -> all-gather 1 -> ... -> last phase
        -> head backward (its parameter gradients summed over the ranks inside it) -> AdamW step

    The loss phases (``ops.ShardedLosses``) give every rank the same ``losses6`` and the gradient of the global-batch
    total for its own rows, so the rank sum of the backwards is the gradient one GPU computes on the whole batch: it is
    applied as is (no averaging), by every rank, and the parameters stay bit-identical across ranks without a
    broadcast.  The all-gathers run on ``parallel.PeerAllGather`` and the gradient sum on ``parallel.PeerAllReduce``
    (both peer-memory kernels, capturable); by default both are built from the process group (``group``).

    Every exchange is a matching call on all ranks, and capturing an epoch's graph first runs the step once eagerly:
    all ranks must call ``step(epoch)`` the same number of times with the same epochs in the same order.

    The step is also written as stages (``bind``, ``stage_forward``, ``stage_loss``, ``stage_exchange``,
    ``stage_backward``, ``stage_update``).  With explicit ``rank`` / ``world`` and ``build_exchanges=False`` no exchange
    object is built, and a caller that holds all ranks in one process drives the stages itself: it concatenates the
    ranks' ``sl.send[p]`` into every ``sl.gathered[p]`` and sums the ranks' ``runner.flat_grads`` in rank order.

    Not supported: ``dropout_p`` > 0 (the masks are keyed by the LOCAL sample index, so every rank would draw rank 0's
    masks), more than 8 ranks, and batches beyond the ``team_loss_shard`` limits (batch <= 16384, world * batch <=
    65536)."""

    def __init__(self, params: Dict[str, torch.Tensor], img_prototypes: torch.Tensor, batch: int, text_cls: torch.Tensor,
                 mode: int = head.MODE_BF16, init_lr: float = 0.004, min_lr: float = 1e-8, weight_decay: float = 0.05,
                 tuned_epoch: int = 20, logit_scale: float = math.exp(2.6592600369327783),
                 evolution_features=None, dropout_p: float = 0.0, seed: Optional[int] = None, *,
                 rank: Optional[int] = None, world: Optional[int] = None, group=None, gather=None, peer=None,
                 build_exchanges: bool = True):
        from . import parallel
        r0, w0 = parallel.world(group)
        rank = r0 if rank is None else int(rank)
        world = w0 if world is None else int(world)
        if dropout_p != 0.0:
            raise ValueError("DataParallelTrainStep: dropout_p > 0 is not supported (the dropout masks are keyed by the "
                             "local sample index, so every rank would draw rank 0's masks)")
        if not 1 <= world <= 8 or not 0 <= rank < world:
            raise ValueError(f"DataParallelTrainStep: rank {rank} / world {world} (one NVSwitch box: at most 8 ranks)")
        if not 1 <= batch <= 16384 or not 2 <= world * batch <= 65536:
            raise ValueError(f"DataParallelTrainStep: {batch} samples per rank x {world} ranks out of range "
                             "(batch <= 16384, 2 <= world * batch <= 65536)")
        for obj in (gather, peer):
            if obj is not None and (obj.rank, obj.world) != (rank, world):
                raise ValueError(f"DataParallelTrainStep: exchange of rank {obj.rank} / world {obj.world} for rank {rank} / world {world}")
        self.rank, self.world, self.group = rank, world, group
        self._build = build_exchanges and world > 1
        self.peer = peer
        super().__init__(params, img_prototypes, batch, text_cls, mode=mode, init_lr=init_lr, min_lr=min_lr,
                         weight_decay=weight_decay, tuned_epoch=tuned_epoch, logit_scale=logit_scale,
                         evolution_features=evolution_features, seed=seed)
        L = capi.lib()
        ne = self.evo[0].shape[0] if self.evo is not None else 0
        sizes = [L.team_loss_shard_xchg_bytes(mode, batch, ne, k) for k in range(L.team_loss_shard_phases(ne) - 1)]
        if gather is None and self._build:
            gather = parallel.PeerAllGather(sizes, self.dev, group)
        self.gather = gather
        # without an all-gather object the step still owns rank-major gathered buffers, so send[p] is the rank's slot:
        # at world 1 the exchange is then nothing at all
        gathered = gather.gathered if gather is not None else [torch.empty((world * n,), dtype=torch.uint8, device=self.dev)
                                                               for n in sizes]
        self.sl = ops.ShardedLosses(rank, world, batch, int(self.text_cls.shape[0]), evolution_features=self.evo, mode=mode,
                                    device=self.dev, gathered=gathered)
        self.losses6 = self.sl.losses6          # total, ce, clip, unicl total, unicl instance, unicl category
        self.losses = self.losses6[:5]
        self.g_own = self.sl.g_own

    def _make_runner(self, pack, img_prototypes, batch, n_cls, mode, dropout_p, seed):
        from . import parallel
        if self.peer is None and self._build:
            self.peer = parallel.PeerAllReduce(head.HeadStepRunner.grad_numel(pack), pack.flat[0].device, self.group)
        return head.HeadStepRunner(pack, img_prototypes, batch, n_cls, mode, peer=self.peer)

    def bind(self, epoch: int):
        """Point the loss phases at the head's outputs and this epoch's temperature / logit scale (host only: the values
        are passed by value when the phases are enqueued, so a captured graph keeps them)."""
        r = self.runner
        self.sl.bind(r.outs[0], r.outs[1], r.outs[2], r.own_rows(), r.logits, self.labels, self.state, epoch=epoch,
                     max_epoch=self.tuned_epoch, logit_scale=self.logit_scale, w_clip=1.0, w_unicl=0.3)

    def stage_forward(self):
        self.runner.forward(self.image, self.text, self.state, self.text_cls)      # cls logits + the four feature outputs

    def stage_loss(self, p: int):
        self.sl.run(p)

    def stage_exchange(self, p: int):
        """All-gather ``sl.send[p]`` of every rank into ``sl.gathered[p]`` (nothing to do at world 1)."""
        if self.world == 1:
            return
        if self.gather is None:
            raise RuntimeError("DataParallelTrainStep built without exchanges: the caller performs them")
        self.gather(p)

    def stage_backward(self):
        # the losses never touch the prototype output; with a PeerAllReduce the backward sums the gradients over the ranks
        self.runner.backward(self.image, self.text, self.state, [self.sl.g_image, self.sl.g_text, self.sl.g_state, None],
                             g_own_rows=self.sl.g_own)

    def stage_update(self, epoch: int):
        self.runner.advance_offset()
        self.opt.lr = self.lr_at(epoch)
        self.opt.step_graph([g for _, g in self.pairs])

    def _body(self, epoch: int):
        self.bind(epoch)
        self.stage_forward()
        n = self.sl.phases
        for p in range(n):
            self.stage_loss(p)
            if p < n - 1:
                self.stage_exchange(p)
        self.stage_backward()
        self.stage_update(epoch)

    def step(self, epoch: int = 0):
        """One optimisation step on the loaded shard of the global batch; returns the device tensor [total, ce, clip, unicl,
        unicl_instance] of the GLOBAL batch (the same on every rank).  Every rank must make the same calls."""
        if self.world > 1 and (self.gather is None or self.peer is None):
            raise RuntimeError("DataParallelTrainStep built without exchanges: drive the stages instead of step()")
        return super().step(epoch)

    def check(self):
        """Raise if an exchange of this rank waited past its deadline (``TEAM_PEER_TIMEOUT_S``); synchronises."""
        for x in (self.gather, self.peer):
            if x is not None:
                x.check()
