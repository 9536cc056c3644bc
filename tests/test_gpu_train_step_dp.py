"""team_b200.train.DataParallelTrainStep on ONE B200: W virtual ranks in one process drive the step's stages eagerly
(forward, loss phase p, exchange p, backward, update); each all-gather is the concatenation of the ranks' send slices
in rank order and the gradient all-reduce is the rank-ordered sum of the ranks' flat gradient buffers, which is what
the peer kernels compute.  Three optimisation steps over two epochs, with and without evolution features.

f32 mode (T = 3, B = 48 per rank, C = 6): against the fp64 oracle loop on the global batch of W * B samples with the
bars of test_gpu_train_step.py (losses <= 2e-5 relative, parameters <= 2e-3 of their movement), and against the
single-GPU TrainStep at W * B (losses <= 1e-5, parameters <= 1e-3 of their movement).
bf16 mode (T = 10, B = 1024 per rank, C = 20, P = 100: the benchmark's training step; W = 1, 2, 3, 4 and 8): against
the single-GPU TrainStep at W * B: losses <= 1e-4 relative, the bar of the bf16 sharded losses in
test_gpu_losses_sharded.py.  Gradients of the first step (both sides start from the same parameters), block by block
for every trainable parameter: <= 5e-3 relative, the bf16 gradient bar of smoke().  Both sides round the same operands
to bf16, but the head runs at B instead of W * B (other kernels and GEMM tilings; the weight gradients summed per rank,
then over ranks).  Parameters after three steps: < 0.1 of their movement each, and at most the largest distance of the
bf16 TrainStep from the f32 TrainStep on the same batches.  These bars are looser because AdamW divides every entry by
its own running RMS: an entry whose gradient is near zero moves by up to lr whatever the gradient's size, so a
last-bit difference in it is a full-size difference in the update.
Measured on an NVIDIA B200 (1 000 W power limit): f32 against TrainStep losses <= 2.0e-7, parameters <= 6.0e-5 of their
movement (against the oracle <= 8.7e-5); bf16 losses <= 3.5e-5, first-step gradients <= 1.4e-4 at W = 1 and
<= 2.6e-3 at W = 2-8 (largest in the blocks behind the attention: w_q / w_k / w_v / w_fc, w_state, prompts,
state_emb), parameters <= 6.8e-2 of their movement, where the bf16 TrainStep is 7.6e-2 to 1.4e-1 of the movement away
from the f32 TrainStep.  The differences are printed (-s).
W = 1 at world 1 through step() (captured graphs) is the single-GPU step: the loss values agree within 1e-6
(measured 9.3e-8: the loss phases sum in another order) and the parameters are bit-identical to TrainStep at B."""
import math

import pytest
import torch

from oracle import synth
from oracle import team_oracle as O

pytestmark = pytest.mark.gpu

LS = math.exp(2.6592600369327783)
LR0, WD, TUNED = 0.004, 0.05, 20
EPOCHS = [0, 0, 1]


def rel(a, b):
    a = a.detach().double().cpu(); b = b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _setup(T, C, evo_on, seed):
    params = synth.make_params(T, seed=seed, perturb_ln=T < 10)
    protos = synth.make_prototypes(C, seed=5)
    text_cls = synth.make_text_class_features(20)[:C].contiguous()
    g = torch.Generator().manual_seed(9)
    evo = [torch.randn(512, generator=g) if c != 2 else None for c in range(C)] if evo_on else None
    return params, protos, text_cls, evo


def _oracle(params, protos, text_cls, evo, batches):
    """fp64 CPU loop body of the learner (as test_gpu_train_step.py): losses per step, parameters after the last."""
    p64 = {k: v.double().clone() for k, v in params.items()}
    names = O.trainable_names(params)
    for n in names:
        p64[n].requires_grad_(True)
    opt = torch.optim.AdamW([p64[n] for n in names], lr=LR0, weight_decay=WD)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=TUNED, eta_min=1e-8)
    out, last = [], 0
    evo64 = None if evo is None else [None if e is None else e.double() for e in evo]
    for b, ep in zip(batches, EPOCHS):
        if ep != last:
            sched.step(); last = ep
        img, txt, sid, y = b["image"].double(), b["text"].double(), b["state"], b["label"]
        with torch.no_grad():
            ce = torch.nn.functional.cross_entropy(O.forward_for_classification(p64, img, text_cls.double()), y)
        o = O.forward_tri_modal(p64, img, txt, sid, protos.double())
        un, inst, _ = O.unicl_loss(o[0], o[1], o[2], y, epoch=ep, max_epoch=TUNED, state_ids=sid, evolution_features=evo64)
        ei = torch.nn.functional.normalize(O.encode_image(img, p64, normalize=True), dim=1)
        et = torch.nn.functional.normalize(O.encode_text(txt, p64, normalize=True), dim=1)
        cl = O.clip_loss(ei, et, LS)
        total = ce + cl + 0.3 * un
        opt.zero_grad()
        total.backward()
        opt.step()
        out.append([float(total), float(ce), float(cl), float(un), float(inst)])
    return out, {n: p64[n].detach() for n in names}


# the trainable blocks in the order of TrainStep.pairs
PAIR_NAMES = ["w_img", "b_img", "w_text", "b_text", "w_state", "b_state", "prompts", "state_emb", "w_q", "w_k", "w_v",
              "w_fc", "b_fc", "ln_g", "ln_b"]


def _single(params, protos, text_cls, evo, batches, batch, mode, grads=None):
    """The single-GPU TrainStep (captured graph) on the whole batch.  ``grads``: a list that receives the gradient of
    every trainable block at every step."""
    from team_b200 import train
    dev = torch.device("cuda")
    pg = {k: v.clone().to(dev) for k, v in params.items()}
    ts = train.TrainStep(pg, protos.to(dev), batch, text_cls.to(dev), mode=mode, init_lr=LR0, min_lr=1e-8, weight_decay=WD,
                         tuned_epoch=TUNED, logit_scale=LS, evolution_features=evo)
    out = []
    for b, ep in zip(batches, EPOCHS):
        ts.load(b["image"], b["text"], b["state"], b["label"])
        out.append(ts.step(epoch=ep).clone())
        if grads is not None:
            grads.append([g.detach().cpu().double() for _, g in ts.pairs])
    torch.cuda.synchronize()
    return [o.cpu().double().tolist() for o in out], pg


def _virtual(params, protos, text_cls, evo, batches, W, B, mode, grads=None):
    """W ranks of DataParallelTrainStep in this process, stages driven eagerly with substituted exchanges.  ``grads``:
    a list that receives the rank-summed gradient of every trainable block at every step."""
    from team_b200 import train
    dev = torch.device("cuda")
    ranks = []
    for r in range(W):
        pg = {k: v.clone().to(dev) for k, v in params.items()}
        ranks.append(train.DataParallelTrainStep(pg, protos.to(dev), B, text_cls.to(dev), mode=mode, init_lr=LR0, min_lr=1e-8,
                                                 weight_decay=WD, tuned_epoch=TUNED, logit_scale=LS, evolution_features=evo,
                                                 rank=r, world=W, build_exchanges=False))
    for s in ranks:              # all-ones bytes: every entry a phase reads must have been written by this step
        for t in s.sl.gathered:
            t.fill_(255)
    out = []
    for b, ep in zip(batches, EPOCHS):
        for r, s in enumerate(ranks):
            sh = slice(r * B, (r + 1) * B)
            s.load(b["image"][sh], b["text"][sh], b["state"][sh], b["label"][sh])
            s.bind(ep)
            s.stage_forward()
        n = ranks[0].sl.phases
        for p in range(n):
            for s in ranks:
                s.stage_loss(p)
            if p < n - 1:
                cat = torch.cat([s.sl.send[p] for s in ranks])
                for s in ranks:
                    s.sl.gathered[p].copy_(cat)
        for s in ranks:
            s.stage_backward()
        gsum = ranks[0].runner.flat_grads.clone()
        for s in ranks[1:]:
            gsum += s.runner.flat_grads
        for s in ranks:
            s.runner.flat_grads.copy_(gsum)
        if grads is not None:
            grads.append([g.detach().cpu().double() for _, g in ranks[0].pairs])
        for s in ranks:
            s.stage_update(ep)
        torch.cuda.synchronize()
        for s in ranks[1:]:
            assert torch.equal(s.losses6, ranks[0].losses6), "losses6 differ between ranks"
        out.append(ranks[0].losses.cpu().double().tolist())
    for s in ranks[1:]:
        for (p, _), (p0, _) in zip(s.pairs, ranks[0].pairs):
            assert torch.equal(p, p0), "parameters differ between ranks"
    assert all(int(s.opt.step_dev.cpu()) == 3 for s in ranks)
    return out, ranks[0].params


def _param_errs(got, want, start, names):
    errs = {}
    for n in names:
        moved = float((want[n].double().cpu() - start[n].double()).norm())
        errs[n] = float((got[n].detach().double().cpu() - want[n].double().cpu()).norm()) / max(moved, 1e-30)
    return errs


def _loss_err(got, want):
    return max(abs(a - r) / max(1.0, abs(r)) for g, w in zip(got, want) for a, r in zip(g, w))


@pytest.mark.parametrize("W", [1, 2, 3, 4])
@pytest.mark.parametrize("evo_on", [False, True])
def test_dp_stages_f32_match_the_oracle_and_train_step(W, evo_on):
    from team_b200 import head
    T, B, C = 3, 48, 6
    params, protos, text_cls, evo = _setup(T, C, evo_on, seed=77)
    batches = [synth.make_batch(W * B, C, step=s) for s in range(3)]
    names = O.trainable_names(params)
    got_l, got_p = _virtual(params, protos, text_cls, evo, batches, W, B, head.MODE_F32)
    ref_l, ref_p = _oracle(params, protos, text_cls, evo, batches)
    one_l, one_p = _single(params, protos, text_cls, evo, batches, W * B, head.MODE_F32)
    for g, r in zip(got_l, ref_l):
        for a, b in zip(g, r):
            assert abs(a - b) < 2e-5 * max(1.0, abs(b)), (got_l, ref_l)
    e_or = _param_errs(got_p, ref_p, params, names)
    e_one = _param_errs(got_p, {n: one_p[n].detach() for n in names}, params, names)
    l_one = _loss_err(got_l, one_l)
    print(f"dp f32 W={W} evo={evo_on}: losses vs TrainStep {l_one:.1e}; params vs oracle {max(e_or.values()):.1e}, "
          f"vs TrainStep {max(e_one.values()):.1e} of their movement")
    for n in names:
        assert e_or[n] < 2e-3 + 1e-7, (n, e_or[n])
        assert e_one[n] < 1e-3, (n, e_one[n])
    assert l_one < 1e-5, (got_l, one_l)


@pytest.mark.parametrize("W", [1, 2, 3, 4, 8])
def test_dp_stages_bf16_match_train_step(W):
    from team_b200 import head
    T, B, C = 10, 1024, 20
    for evo_on in (False, True):
        params, protos, text_cls, evo = _setup(T, C, evo_on, seed=42)
        batches = [synth.make_batch(W * B, C, step=s) for s in range(3)]
        names = O.trainable_names(params)
        g_dp, g_one = [], []
        got_l, got_p = _virtual(params, protos, text_cls, evo, batches, W, B, head.MODE_BF16, grads=g_dp)
        one_l, one_p = _single(params, protos, text_cls, evo, batches, W * B, head.MODE_BF16, grads=g_one)
        _, f32_p = _single(params, protos, text_cls, evo, batches, W * B, head.MODE_F32)
        e = _param_errs(got_p, {n: one_p[n].detach() for n in names}, params, names)
        e_prec = _param_errs({n: one_p[n].detach() for n in names}, {n: f32_p[n].detach() for n in names}, params, names)
        # step 1 starts from the same parameters on both sides: its gradients compare block by block without AdamW
        eg = {k: float((a - b).norm() / b.norm().clamp_min(1e-30)) for k, a, b in zip(PAIR_NAMES, g_dp[0], g_one[0])}
        lerr = max(abs(a - r) / max(abs(r), 1e-30) for g, w in zip(got_l, one_l) for a, r in zip(g, w))
        print(f"dp bf16 W={W} evo={evo_on}: losses vs TrainStep {lerr:.1e}; step-1 gradients {max(eg.values()):.1e} "
              f"({' '.join(f'{k}={v:.1e}' for k, v in eg.items())}); params {max(e.values()):.1e} of their movement, "
              f"TrainStep bf16 vs f32 {max(e_prec.values()):.1e}")
        assert lerr <= 1e-4, (got_l, one_l)
        for k, v in eg.items():
            assert v <= 5e-3, (k, v, eg)
        assert max(e.values()) <= max(e_prec.values()), (e, e_prec)
        for n in names:
            assert e[n] < 0.1, (n, e[n], e_prec[n])


@pytest.mark.parametrize("mode", [0, 1])
def test_dp_world_one_is_train_step(mode):
    """world = 1 through step() (captured graphs): the single-GPU TrainStep at the same batch."""
    from team_b200 import train
    T, B, C = 3, 64, 6
    params, protos, text_cls, evo = _setup(T, C, True, seed=78)
    batches = [synth.make_batch(B, C, step=s) for s in range(3)]
    names = O.trainable_names(params)
    dev = torch.device("cuda")
    pg = {k: v.clone().to(dev) for k, v in params.items()}
    dp = train.DataParallelTrainStep(pg, protos.to(dev), B, text_cls.to(dev), mode=mode, init_lr=LR0, min_lr=1e-8, weight_decay=WD,
                                     tuned_epoch=TUNED, logit_scale=LS, evolution_features=evo, rank=0, world=1)
    assert dp.gather is None and dp.peer is None
    got = []
    for b, ep in zip(batches, EPOCHS):
        dp.load(b["image"], b["text"], b["state"], b["label"])
        got.append(dp.step(epoch=ep).clone())
    torch.cuda.synchronize()
    assert len(dp._graphs) == 2 and int(dp.opt.step_dev.cpu()) == 3
    got = [g.cpu().double().tolist() for g in got]
    one_l, one_p = _single(params, protos, text_cls, evo, batches, B, mode)
    e = _param_errs(pg, {n: one_p[n].detach() for n in names}, params, names)
    lerr = _loss_err(got, one_l)
    print(f"dp world 1 mode={mode}: losses vs TrainStep {lerr:.1e}; params {max(e.values()):.1e} of their movement")
    assert lerr < 1e-6, (got, one_l)
    for n in names:
        assert torch.equal(pg[n].cpu(), one_p[n].cpu()), (n, e[n])


def test_dp_rejects_bad_arguments():
    from team_b200 import train
    T, C = 2, 4
    params, protos, text_cls, _ = _setup(T, C, False, seed=1)
    dev = torch.device("cuda")
    pg = {k: v.to(dev) for k, v in params.items()}
    mk = lambda B, **kw: train.DataParallelTrainStep(pg, protos.to(dev), B, text_cls.to(dev), build_exchanges=False, **kw)
    with pytest.raises(ValueError, match="dropout"):
        mk(8, rank=0, world=2, dropout_p=0.1)
    with pytest.raises(ValueError):
        mk(8, rank=0, world=9)
    with pytest.raises(ValueError):
        mk(8, rank=2, world=2)
    with pytest.raises(ValueError):
        mk(16385, rank=0, world=1)                            # more than 16 384 samples per rank
    with pytest.raises(ValueError):
        mk(16384, rank=0, world=5)                            # more than 65 536 in the global batch
    with pytest.raises(ValueError):
        mk(1, rank=0, world=1)                                # a global batch of one
    s = mk(8, rank=1, world=2)
    with pytest.raises(RuntimeError):                         # no exchange objects: the caller drives the stages
        s.step(0)
