"""The training step the benchmark times - team_b200.train.TrainStep in bf16 mode at T = 10 tasks, C = 20 classes,
B = 1024, an evolution feature for every class, device-resident batches - and the kernels only that step runs:
team_ce_total, team_copy_batch, team_adamw_step_graph, team_unicl_loss_evo in bf16 mode, and the losses up to
LOSS_MAX_BATCH = 16384 samples.  Every kernel is compared with a plain fp64 reference of the same operation.
Bars are norm-wise relative errors unless a docstring says otherwise; the errors quoted were measured on a B200."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import synth
from oracle import team_oracle as O

pytestmark = pytest.mark.gpu

W_CLIP, W_UNICL = 0.7, 1.9          # weights of team_ce_total's total other than the learner's (1, 0.3)


def rel(a, b):
    a = torch.as_tensor(a).detach().double()
    b = torch.as_tensor(b).detach().double().to(a.device)
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def bits(t):
    """The raw bits of a tensor, so that torch.equal compares NaN payloads and signed zeros too."""
    t = t.detach().contiguous()
    return t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int64)


def _feats(B, seed, noise):
    """Three correlated [B,512] feature sets with norms far from 1 (the losses normalise them themselves)."""
    g = torch.Generator().manual_seed(seed)
    base = torch.randn((B, 512), generator=g)
    return [base + noise * torch.randn((B, 512), generator=g) for _ in range(3)], g


# --------------------------------------------------------------------------------------------------- 1. team_ce_total
def _ce_inputs(kind, B, C, seed):
    g = torch.Generator().manual_seed(seed)
    y = torch.randint(0, C, (B,), generator=g, dtype=torch.int64)
    if kind == "ordinary":
        x = 3.0 * torch.randn((B, C), generator=g)
    elif kind == "ties":
        x = torch.randint(-2, 3, (B, C), generator=g).float()          # integers: many exact ties, the max included
        x[0] = 0.5                                                      # one row all equal
        y[::2] = x[::2].argmax(1)                                       # labels on a tied maximum
    else:
        x = torch.rand((B, C), generator=g) * 180.0 - 90.0             # about +-90: exp() overflows fp32 above 88.7
        x[torch.arange(B), torch.randint(0, C, (B,), generator=g)] = 90.0
    return x.contiguous(), y


@pytest.mark.parametrize("kind", ["ordinary", "ties", "large"])
@pytest.mark.parametrize("C", [1, 2, 20, 1000])
@pytest.mark.parametrize("B", [1, 7, 1024, 1025, 3000, 16384])
def test_ce_total_vs_fp64(B, C, kind):
    """team_ce_total (one CTA of 1024 threads striding over the rows) against F.cross_entropy in fp64: B up to 16384
    (the multi-row path starts at B = 1025), C up to 1000, tied rows and logits of about +-90, where a log-sum-exp
    without the max subtraction overflows.  Bar: |ce - ref| <= 1e-5 max(1, |ref|) (measured <= 3.5e-7).  The total
    ce + w_clip l[2] + w_unicl l[3] with weights 0.7 / 1.9 and random preset l[2:6] agrees with its fp64 evaluation
    from the kernel's ce to 1e-6 of the summed magnitudes (fp32 rounding); l[2:6] come back bit for bit and a second
    call is bitwise the same.  The contract is labels in [0, C): for others the kernel counts the row's log-sum-exp
    only, where torch raises."""
    from team_b200 import ops
    x, y = _ce_inputs(kind, B, C, seed=B * 7 + C)
    xd, yd = x.cuda(), y.cuda()
    ref = float(F.cross_entropy(xd.double(), yd))
    pre = torch.randn((4,), generator=torch.Generator().manual_seed(C))
    out = []
    for _ in range(2):
        l6 = torch.cat([torch.full((2,), float("nan")), pre]).cuda()
        ops.ce_total(xd, yd, l6, w_clip=W_CLIP, w_unicl=W_UNICL)
        out.append(l6.cpu())
    got = out[0]
    ce = float(got[1])
    assert math.isfinite(ce) and abs(ce - ref) <= 1e-5 * max(1.0, abs(ref)), (ce, ref)
    l2, l3 = float(pre[0]), float(pre[1])
    total = ce + float(torch.tensor(W_CLIP)) * l2 + float(torch.tensor(W_UNICL)) * l3
    assert abs(float(got[0]) - total) <= 1e-6 * (abs(ce) + abs(W_CLIP * l2) + abs(W_UNICL * l3)), (float(got[0]), total)
    assert torch.equal(bits(got[2:]), bits(pre))
    assert torch.equal(bits(out[1]), bits(got))
    print(f"measured ce_total B={B} C={C} {kind}: {abs(ce - ref) / max(1.0, abs(ref)):.2e}")


# ------------------------------------------------------------------------------------------------- 2. team_copy_batch
def _copy_batch(src, dst, B):
    from team_b200 import capi
    return capi.lib().team_copy_batch(*[t.data_ptr() if torch.is_tensor(t) else t for t in src], B,
                                      *[t.data_ptr() if torch.is_tensor(t) else t for t in dst],
                                      torch.cuda.current_stream().cuda_stream)


def _copy_operands(B, seed):
    g = torch.Generator().manual_seed(seed)
    img, txt = torch.randn((B, 512), generator=g), torch.randn((B, 512), generator=g)
    img[0, 0], img[0, 1], txt[-1, -1] = -0.0, float("nan"), float("inf")
    sid = torch.randint(0, 10, (B,), generator=g, dtype=torch.int64)
    lab = torch.randint(-5, 1 << 40, (B,), generator=g, dtype=torch.int64)
    src = [t.cuda() for t in (img, txt, sid, lab)]
    # one guard row past the end of each destination
    dst = [torch.full((B + 1, 512), float("nan"), device="cuda"), torch.full((B + 1, 512), float("nan"), device="cuda"),
           torch.full((B + 1,), -1, dtype=torch.int64, device="cuda"), torch.full((B + 1,), -1, dtype=torch.int64, device="cuda")]
    return src, dst


@pytest.mark.parametrize("B", [1, 3, 1024, 4097])
def test_copy_batch_is_a_bitwise_copy(B):
    """team_copy_batch (TrainStep.load of a device-resident batch): the destination is a bitwise copy of all four
    inputs (NaN, -0 and inf included), and the guard row after each destination is untouched."""
    src, dst = _copy_operands(B, seed=B)
    guard = [bits(d[B]).clone() for d in dst]
    assert _copy_batch(src, dst, B) == 0
    torch.cuda.synchronize()
    for s, d, g0 in zip(src, dst, guard):
        assert torch.equal(bits(d[:B]), bits(s))
        assert torch.equal(bits(d[B]), g0)


def test_copy_batch_rejects_misaligned_rows():
    """A feature pointer 4 bytes off a 16-byte boundary is refused on the host, before any launch, with a message;
    nothing is written."""
    from team_b200 import capi
    B = 4
    src, dst = _copy_operands(B, seed=11)
    base = torch.zeros((B * 512 + 4,), device="cuda")
    before = [bits(d).clone() for d in dst]
    for which in (0, 1):                               # source image rows, then destination image rows
        s, d = list(src), list(dst)
        if which == 0:
            s[0] = base.data_ptr() + 4
        else:
            d[0] = base.data_ptr() + 4
        rc = _copy_batch(s, d, B)
        assert rc != 0
        assert "16-byte aligned" in capi.lib().team_last_error().decode()
    torch.cuda.synchronize()
    for d, b0 in zip(dst, before):
        assert torch.equal(bits(d), b0)


# ----------------------------------------------------------------------------------------- 3. team_adamw_step_graph
def _adamw_shapes():
    """60 tensors of ragged sizes, so that FusedAdamW makes two launches of at most 48 tensors; zero-element tensors
    first, last, in the middle and on both sides of the chunk boundary."""
    g = torch.Generator().manual_seed(17)
    shapes = [(0,), (1,), (1023,), (1025,), (512, 512), (1024,), (0, 512), (3, 7), (2049,), (10, 512)]
    while len(shapes) < 60:
        shapes.append((int(torch.randint(1, 5000, (1,), generator=g)),))
    shapes[47], shapes[48], shapes[-1] = (0,), (0,), (0,)
    shapes[30] = (512, 512)
    return shapes


def test_adamw_step_graph_replays_match_torch():
    """FusedAdamW.step_graph captured once in a CUDA graph and replayed 5 times, new gradients written into the static
    gradient buffers before each replay, against torch.optim.AdamW in fp64 on the same values (same lr and weight
    decay).  Per tensor after every replay: parameters, exp_avg and exp_avg_sq <= 1e-6 (measured <= 1.7e-7).  The device
    step count is 5 at the end: only the last of the two launches advances it."""
    from team_b200 import ops
    shapes = _adamw_shapes()
    g = torch.Generator().manual_seed(5)
    init = [torch.randn(s, generator=g) for s in shapes]
    lr, wd = 3e-3, 0.05
    ref = [torch.nn.Parameter(t.double().cuda()) for t in init]
    mine = [t.clone().cuda() for t in init]
    # the kernel receives the hyper-parameters as fp32: the reference uses the same values (1 - fl32(0.999) is 1.3e-5
    # away from 0.001, which exp_avg_sq would show)
    f32 = lambda v: float(torch.tensor(v, dtype=torch.float32))
    opt = torch.optim.AdamW(ref, lr=f32(lr), betas=(f32(0.9), f32(0.999)), eps=f32(1e-8), weight_decay=f32(wd))
    fused = ops.FusedAdamW([p.requires_grad_(True) for p in mine], lr=lr, weight_decay=wd)
    gbuf = [torch.zeros(s, device="cuda") for s in shapes]
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fused.step_graph(gbuf)
    worst = 0.0
    for it in range(5):
        new = [torch.randn(s, generator=g) * (10.0 ** (i % 5 - 3)) for i, s in enumerate(shapes)]
        for b, n, p in zip(gbuf, new, ref):
            b.copy_(n)
            p.grad = n.double().cuda()
        graph.replay()
        opt.step()
        torch.cuda.synchronize()
        step = int(fused.step_dev.cpu())
        for i, (p, r) in enumerate(zip(mine, ref)):
            st = opt.state[r]
            errs = (rel(p, r), rel(fused.exp_avg[i], st["exp_avg"]), rel(fused.exp_avg_sq[i], st["exp_avg_sq"]))
            worst = max(worst, *errs)
            assert step == it + 1 and max(errs) <= 1e-6, (it, step, i, shapes[i], errs)
    assert int(fused.step_dev.cpu()) == 5
    print(f"measured adamw graph replays vs fp64 torch: {worst:.2e}")


def test_adamw_step_graph_eager_matches_step():
    """FusedAdamW.step_graph called eagerly (the step count read on the device) against FusedAdamW.step (the step count
    passed from the host), the same 60 tensors, three steps: <= 1e-7 per tensor (the same arithmetic)."""
    from team_b200 import ops
    shapes = _adamw_shapes()
    g = torch.Generator().manual_seed(6)
    init = [torch.randn(s, generator=g).cuda() for s in shapes]
    a = [t.clone().requires_grad_(True) for t in init]
    b = [t.clone().requires_grad_(True) for t in init]
    fa = ops.FusedAdamW(a, lr=2e-3, weight_decay=0.01)
    fb = ops.FusedAdamW(b, lr=2e-3, weight_decay=0.01)
    for _ in range(3):
        grads = [torch.randn(s, generator=g).cuda() for s in shapes]
        fa.step(grads)
        fb.step_graph(grads)
    torch.cuda.synchronize()
    assert int(fb.step_dev.cpu()) == 3
    for x, y in zip(a, b):
        assert rel(y, x) <= 1e-7, rel(y, x)


# ----------------------------------------------------------------------------- 4. evolution loss in bf16, large batches
def _unicl_check(got_losses, grads, ref, xs, tv, tg):
    total, inst, cat = ref
    got = got_losses.detach().double().cpu()
    ev = (rel(got[0], total), abs(float(got[1]) - float(inst)) / max(1.0, abs(float(inst))),
          abs(float(got[2]) - float(cat)) / max(1.0, abs(float(cat))))
    eg = [rel(t, x.grad) for t, x in zip(grads, xs)]
    assert max(ev) <= tv and max(eg) <= tg, (ev, eg)
    return max(ev), max(eg)


def _evo_case(B, C, nstates, holes, seed):
    feats, g = _feats(B, seed, 0.7)
    labels = torch.randint(0, C, (B,), generator=g, dtype=torch.int64)
    states = torch.randint(0, nstates, (B,), generator=g, dtype=torch.int64)
    n_evo = C - 2 if holes else C
    evo = [torch.randn(512, generator=g) for _ in range(n_evo)]
    if holes:
        evo[1] = None
    return feats, labels, states, evo


@pytest.mark.parametrize("B,C,nstates,holes,bench", [(64, 6, 4, True, False), (257, 20, 10, True, False),
                                                     (1024, 20, 5, False, False), (40, 30, 10, False, False),
                                                     (1024, 20, 0, False, True)])
def test_unicl_evolution_bf16_vs_oracle(B, C, nstates, holes, bench):
    """team_unicl_loss_evo in bf16 mode (the bf16 shadow of the normalised image rows feeds the similarity and the
    category-gradient products; the evolution kernels work on the fp32 rows) against the fp64 oracle, on the four
    configurations of the fp32 test and the benchmarked one (B = 1024, C = 20, a feature for every class, states and
    labels from synth.make_batch, epoch 0 of 20, grad_scale 0.3).  Bars at about 3x the measured error, inside those
    of the bf16 loss tests (1e-2 / 2e-2): values <= 7e-4 (measured <= 2.2e-4, B = 40), gradients <= 7e-3 (measured
    <= 2.1e-3)."""
    from team_b200 import ops, capi
    if bench:
        b = synth.make_batch(B, C, step=0)
        feats, _ = _feats(B, 900, 0.7)
        labels, states = b["label"], b["state"]
        evo = [torch.randn(512, generator=torch.Generator().manual_seed(5)) for _ in range(C)]
        epoch = 0
    else:
        feats, labels, states, evo = _evo_case(B, C, nstates, holes, 300 + B)
        epoch = 3
    x = [f.clone().double().requires_grad_(True) for f in feats]
    ref = O.unicl_loss(x[0], x[1], x[2], labels, epoch=epoch, max_epoch=20, state_ids=states,
                       evolution_features=[None if e is None else e.double() for e in evo])
    (0.3 * ref[0]).backward()
    losses, grads = ops.unicl_loss(*[f.cuda() for f in feats], labels.cuda(), state_ids=states.cuda(), evolution_features=evo,
                                   epoch=epoch, max_epoch=20, grad_scale=0.3, mode=capi.MODE_BF16)
    ev, eg = _unicl_check(losses, grads, ref, x, 7e-4, 7e-3)
    print(f"measured unicl evo bf16 B={B} C={C}: values {ev:.2e} gradients {eg:.2e}")


@pytest.fixture(scope="module")
def b4096_reference():
    """B = 4096, C = 200, an evolution feature for every class, ten states: the fp64 oracle once for both modes."""
    B, C = 4096, 200
    feats, labels, states, evo = _evo_case(B, C, 10, False, 4096)
    x = [f.clone().double().requires_grad_(True) for f in feats]
    ref = O.unicl_loss(x[0], x[1], x[2], labels, epoch=5, max_epoch=20, state_ids=states,
                       evolution_features=[e.double() for e in evo])
    (0.3 * ref[0]).backward()
    ci, ct = F.normalize(feats[0], dim=1), F.normalize(feats[1], dim=1)
    y = [ci.double().requires_grad_(True), ct.double().requires_grad_(True)]
    cl = O.clip_loss(y[0], y[1], 14.285714)
    cl.backward()
    return dict(feats=feats, labels=labels, states=states, evo=evo, x=x, ref=[r.detach() for r in ref], clip=(ci, ct, y, cl.detach()))


# mode -> (values, gradients) at about 3x the errors measured at B = 4096 and 16384, inside the bars of the existing loss
# tests (fp32 1e-5 / 3e-5, bf16 1e-2 / 2e-2)
BARS = {0: (4e-7, 8e-6), 1: (2e-4, 9e-3)}


@pytest.mark.parametrize("mode", [0, 1], ids=["f32", "bf16"])
def test_losses_b4096_vs_oracle(mode, b4096_reference):
    """unicl_loss with evolution features (C = 200 classes, num_evo = 200) and clip_loss at B = 4096, where the B x B
    products and the K = B gradient products (dcat, dI, dT) may take other tile and split-K plans than at 1024, against
    the fp64 oracle.  fp32: values <= 4e-7 (measured 1.2e-7), gradients <= 8e-6 (measured 2.7e-6, the ClipLoss
    gradient); bf16: values <= 2e-4 (measured 3.5e-6), gradients <= 9e-3 (measured 2.7e-3)."""
    from team_b200 import ops
    r = b4096_reference
    tv, tg = BARS[mode]
    losses, grads = ops.unicl_loss(*[f.cuda() for f in r["feats"]], r["labels"].cuda(), state_ids=r["states"].cuda(),
                                   evolution_features=r["evo"], epoch=5, max_epoch=20, grad_scale=0.3, mode=mode)
    ev, eg = _unicl_check(losses, grads, r["ref"], r["x"], tv, tg)
    ci, ct, y, cl = r["clip"]
    loss, cg = ops.clip_loss(ci.cuda(), ct.cuda(), 14.285714, mode=mode)
    cv = abs(float(loss.cpu()[0]) - float(cl)) / max(1.0, abs(float(cl)))
    cgr = max(rel(cg[0], y[0].grad), rel(cg[1], y[1].grad))
    assert cv <= tv and cgr <= tg, (cv, cgr)
    print(f"measured B=4096 mode={mode}: unicl values {ev:.2e} gradients {eg:.2e}; clip value {cv:.2e} gradients {cgr:.2e}")


@pytest.mark.parametrize("mode", [0, 1], ids=["f32", "bf16"])
def test_losses_at_max_batch_vs_fp64(mode):
    """unicl_loss and clip_loss at LOSS_MAX_BATCH = 16384: [B,Bp] workspaces of 268 M elements indexed with an int
    leading dimension, K = 16384 in the gradient products.  The reference is the fp64 oracle evaluated on the GPU.
    fp32: values <= 4e-7 (measured 1.0e-7), gradients <= 8e-6 (measured 2.7e-6, the ClipLoss gradient); bf16: values
    <= 2e-4 (measured 4.7e-5, the ClipLoss value), gradients <= 9e-3 (measured 2.6e-3)."""
    from team_b200 import ops
    B, C = 16384, 20
    tv, tg = BARS[mode]
    feats, g = _feats(B, 16384, 0.7)
    labels = torch.randint(0, C, (B,), generator=g, dtype=torch.int64).cuda()
    feats = [f.cuda() for f in feats]
    x = [f.double().requires_grad_(True) for f in feats]
    ref = O.unicl_loss(x[0], x[1], x[2], labels, epoch=7, max_epoch=20)
    (0.3 * ref[0]).backward()
    ref = [r.detach() for r in ref]
    losses, grads = ops.unicl_loss(feats[0], feats[1], feats[2], labels, epoch=7, max_epoch=20, grad_scale=0.3, mode=mode)
    ev, eg = _unicl_check(losses, grads, ref, x, tv, tg)
    del x, grads
    ci, ct = F.normalize(feats[0], dim=1), F.normalize(feats[1], dim=1)
    y = [ci.double().requires_grad_(True), ct.double().requires_grad_(True)]
    cl = O.clip_loss(y[0], y[1], 14.285714)
    cl.backward()
    loss, cg = ops.clip_loss(ci, ct, 14.285714, mode=mode)
    cv = abs(float(loss.cpu()[0]) - float(cl)) / max(1.0, abs(float(cl)))
    cgr = max(rel(cg[0], y[0].grad), rel(cg[1], y[1].grad))
    assert cv <= tv and cgr <= tg, (cv, cgr)
    print(f"measured B=16384 mode={mode}: unicl values {ev:.2e} gradients {eg:.2e}; clip value {cv:.2e} gradients {cgr:.2e}")
    torch.cuda.empty_cache()


def test_losses_reject_batches_above_the_maximum():
    """B = 16385 is one past LOSS_MAX_BATCH: no workspace size, and both losses raise ValueError before any launch."""
    from team_b200 import ops, capi
    L = capi.lib()
    assert L.team_loss_workspace_bytes(16384) > 0 and L.team_loss_workspace_bytes(16385) == 0
    assert L.team_loss_evo_workspace_bytes(16385, 20) == 0
    B = 16385
    x = torch.randn((B, 512), device="cuda")
    y = torch.zeros((B,), dtype=torch.int64, device="cuda")
    with pytest.raises(ValueError):
        ops.unicl_loss(x, x, x, y)
    with pytest.raises(ValueError):
        ops.unicl_loss(x, x, x, y, state_ids=y, evolution_features=[torch.ones(512)])
    with pytest.raises(ValueError):
        ops.clip_loss(x, x, 14.285714)


# ------------------------------------------------------------------------------ 5. TrainStep as the benchmark runs it
EPOCHS = [0, 0, 1]


def _step_config(T, B):
    """Parameters, prototypes, class text features, evolution features and three batches: T = 10, B = 1024 is the
    benchmark's configuration (reference initialisers, a feature for every class); T = 1 is the first task (no
    frozen projections; the second class has no evolution feature)."""
    C = 2 * T
    params = synth.make_params(T, seed=42, perturb_ln=T == 1)
    protos = synth.make_prototypes(C)
    text_cls = synth.make_text_class_features(20)[:C].contiguous()
    gen = torch.Generator().manual_seed(5)
    evo = [torch.randn(512, generator=gen) for _ in range(C)]
    if T == 1:
        evo[1] = None
    batches = [synth.make_batch(B, C, step=s) for s in range(3)]
    return params, protos, text_cls, evo, batches


def _make_step(params, protos, text_cls, evo, B, mode):
    from team_b200 import train
    pg = {k: v.clone().cuda() for k, v in params.items()}
    ts = train.TrainStep(pg, protos.cuda(), B, text_cls.cuda(), mode=mode, evolution_features=evo)
    return pg, ts


def _reference_step(p64, params, protos, text_cls, evo, batch, epoch, ts, names):
    """fp64 losses [total, ce, clip, unicl, unicl instance] and d total / d trainable at the parameters ``p64``."""
    from factorised_model import head_fwd_bwd
    img, txt, sid, y = batch["image"].double(), batch["text"].double(), batch["state"], batch["label"]
    pr = protos.double()
    evo64 = [None if e is None else e.double() for e in evo]
    B = img.shape[0]
    with torch.no_grad():
        ce = F.cross_entropy(O.forward_for_classification(p64, img, text_cls.double()), y)
    ls = ts.logit_scale
    if O.num_tasks(params) == 1:
        # the oracle directly: autograd through forward_tri_modal
        p = {k: v.clone().requires_grad_(k in names) for k, v in p64.items()}
        o = O.forward_tri_modal(p, img, txt, sid, pr)
        un, inst, _ = O.unicl_loss(o[0], o[1], o[2], y, epoch=epoch, max_epoch=ts.tuned_epoch, state_ids=sid,
                                   evolution_features=evo64)
        ei = F.normalize(O.encode_image(img, p, normalize=True), dim=1)
        et = F.normalize(O.encode_text(txt, p, normalize=True), dim=1)
        cl = O.clip_loss(ei, et, ls)
        total = ce + cl + 0.3 * un
        grads = dict(zip(names, torch.autograd.grad(total, [p[n] for n in names])))
        return [float(v.detach()) for v in (total, ce, cl, un, inst)], grads, _clip_conditioning(ei, et, ls)
    # T = 10, B = 1024: the factorised head (pinned to the oracle by tests/test_quantised_model.py) with cotangents
    # from autograd through the oracle's unicl_loss, plus the ClipLoss gradient through the projections
    z = dict(dtype=torch.float64, device=img.device)
    zeros = [torch.zeros(B, 512, **z), torch.zeros(B, 1, 512, **z), torch.zeros(B, 512, **z), torch.zeros(B, 512, **z)]
    outs, _ = head_fwd_bwd(p64, img, txt, sid, pr, zeros)
    o = [t.detach().clone().requires_grad_(True) for t in outs[:3]]
    un, inst, _ = O.unicl_loss(o[0], o[1], o[2], y, epoch=epoch, max_epoch=ts.tuned_epoch, state_ids=sid,
                               evolution_features=evo64)
    cots = torch.autograd.grad(0.3 * un, o)
    _, grads = head_fwd_bwd(p64, img, txt, sid, pr, [cots[0], cots[1], cots[2], zeros[3]])
    T = O.num_tasks(params)
    clip_names = [f"projs_img.{T - 1}.MLP.0.weight", f"projs_img.{T - 1}.MLP.0.bias",
                  f"projs_text.{T - 1}.MLP.0.weight", f"projs_text.{T - 1}.MLP.0.bias"]
    p = {k: v.clone().requires_grad_(k in clip_names) for k, v in p64.items()}
    ei = F.normalize(O.encode_image(img, p, normalize=True), dim=1)
    et = F.normalize(O.encode_text(txt, p, normalize=True), dim=1)
    cl = O.clip_loss(ei, et, ls)
    for n, gc in zip(clip_names, torch.autograd.grad(cl, [p[n] for n in clip_names])):
        grads[n] = grads[n] + gc
    total = ce + cl + 0.3 * un
    return [float(v.detach()) for v in (total, ce, cl, un, inst)], grads, _clip_conditioning(ei, et, ls)


def _clip_conditioning(ei, et, ls):
    """How much the ClipLoss row gradients dI = G T and dT = G^T I cancel, |G| |T| / |G T| norm-wise (the larger of the
    two), G = softmax_i2t + softmax_t2i^T - 2 I.  The bf16 mode rounds G and the rows to bf16 for these products, so
    their relative error is about this factor times the bf16 rounding."""
    with torch.no_grad():
        L = ls * ei @ et.t()
        G = torch.softmax(L, 1) + torch.softmax(L.t(), 1).t() - 2 * torch.eye(L.shape[0], dtype=L.dtype, device=L.device)
        return max(float((G.abs() @ et.abs()).norm() / (G @ et).norm()),
                   float((G.abs().t() @ ei.abs()).norm() / (G.t() @ ei).norm()))


# mode -> (losses, gradients, amplified gradients).  The loss gradients reach the newest projections and the state
# embedding table as sums over rows that nearly cancel: the contrastive losses' row gradients sum to about zero over the
# batch (their norms add up to 20-30x the norm of the sum, measured on the oracle for the image and text projection
# biases at T = 1, B = 64 and T = 10, B = 256), the text rows are the C class-text features and the state rows the ten
# table rows, so those weight gradients are a few such sums too.  The query and key weights receive the loss gradients
# through the softmax backward A (dA - sum A dA), a difference of nearly equal terms.  The rows' own rounding error
# reaches these gradients amplified by up to that factor.
STEP_BARS = {0: (2e-5, 2e-5, 3e-4), 1: (1e-2, 1.5e-2, 8e-2)}


def _summed(name):
    return name.startswith(("projs_", "state_embedder.", "sel_attn.w_qs.", "sel_attn.w_ks."))


# As a step trains the image rows towards their class text, the ClipLoss gradient becomes a difference of nearly equal
# terms: every text row is one of the C class-text features, and a row's gradient is the small remainder of (softmax - 1)
# on its own row plus the softmax mass on the other copies of its class text.  At T = 1, B = 64 the cancellation factor
# of dI = G T grows from 4 at the first step to 31 and 54 at the next two, and evaluating the products in fp64 from
# bf16-rounded operands - what the bf16 mode does by design - already gives them 2.6e-2 and 6.3e-2 relative error;
# the projections' gradients are batch sums of these rows and cancel further.  There the bf16 mode does not determine
# the gradients of the image and text projections to a bar that could catch a fault, so in bf16 they are compared only
# at steps whose ClipLoss products are conditioned at most this well (every configuration's first step is).
CLIP_KAPPA_MAX = 10.0


def _clip_fed(name):
    return name.startswith(("projs_img.", "projs_text."))


@pytest.mark.parametrize("mode", [0, 1], ids=["f32", "bf16"])
@pytest.mark.parametrize("T,B", [(10, 1024), (1, 64)], ids=["bench_T10_B1024", "first_task_T1_B64"])
def test_train_step_vs_fp64(T, B, mode):
    """TrainStep, 3 steps over epochs [0, 0, 1] (the second epoch re-captures with a new learning rate and unicl
    temperature), batches loaded from device tensors (team_copy_batch).  Checked in two parts per step:
      a. optimizer chain: the step's gradients, read through TrainStep.pairs, drive an fp64 torch.optim.AdamW over a
         mirror of the trainable parameters at lr = lr_at(epoch); the GPU parameters match the mirror to <= 1e-6 per
         tensor after every step (measured <= 8.7e-8) and the device step count equals the number of steps;
      b. the five loss values and the gradient of the total with respect to every trainable tensor against fp64 at the
         parameters the step began with (the mirror's).  fp32: losses <= 2e-5 max(1, |r|), gradients <= 2e-5, the bars
         of test_gpu_train_step.py (measured <= 1.0e-7 / 9.7e-7); bf16: losses <= 1e-2 max(1, |r|), gradients
         <= 1.5e-2, the operand-level bars of test_head_bf16_mode (measured <= 5.5e-4 / 7.4e-3).  The newest
         projections, the state table and the query / key weights have wider bars (STEP_BARS: fp32 3e-4, measured
         1.0e-4; bf16 8e-2, measured 3.0e-2), and in bf16 the image and text projections are compared only at steps
         whose ClipLoss products are well conditioned (CLIP_KAPPA_MAX; measured factors 2.5 / 4.3 / 15 at T = 10 and
         3.9 / 31 / 54 at T = 1) - the reasons are written beside those constants.
    The final parameters of the bf16 step are not compared with an fp64 training loop: Adam's first steps are close to
    sign(g), so the bf16 error of gradient components near zero becomes an error of order lr in those elements."""
    params, protos, text_cls, evo, batches = _step_config(T, B)
    pg, ts = _make_step(params, protos, text_cls, evo, B, mode)
    names = O.trainable_names(params)
    by_id = {id(pg[n]): n for n in names}
    views = {by_id[id(p)]: g for p, g in ts.pairs}
    assert sorted(views) == sorted(names)
    mirror = {n: pg[n].detach().double().cpu().clone().requires_grad_(True) for n in names}
    opt = torch.optim.AdamW([mirror[n] for n in names], lr=ts.init_lr, weight_decay=0.05)
    p64 = {k: v.double() for k, v in params.items()}
    tl, tg, tb = STEP_BARS[mode]
    worst = [0.0, 0.0, 0.0, 0.0]
    checked, kappas = set(), []
    for i, (b, ep) in enumerate(zip(batches, EPOCHS)):
        ts.load(b["image"].cuda(), b["text"].cuda(), b["state"].cuda(), b["label"].cuda())
        got = ts.step(epoch=ep).double().cpu().tolist()
        grads = {n: views[n].detach().double().cpu().reshape(mirror[n].shape) for n in names}
        start = dict(p64, **{n: mirror[n].detach().clone() for n in names})
        ref_l, ref_g, kappa = _reference_step(start, params, protos, text_cls, evo, b, ep, ts, names)
        el = max(abs(a - r) / max(1.0, abs(r)) for a, r in zip(got, ref_l))
        eg = {n: rel(grads[n], ref_g[n]) for n in names
              if mode == 0 or kappa <= CLIP_KAPPA_MAX or not _clip_fed(n)}
        checked |= set(eg)
        kappas.append(round(kappa, 1))
        assert el <= tl, (i, got, ref_l)
        bad = {n: e for n, e in eg.items() if e > (tb if _summed(n) else tg)}
        assert not bad, (i, bad)
        for grp in opt.param_groups:
            grp["lr"] = ts.lr_at(ep)
        for n in names:
            mirror[n].grad = grads[n]
        opt.step()
        ep_ = {n: rel(pg[n].cpu(), mirror[n]) for n in names}
        assert max(ep_.values()) <= 1e-6, (i, ep_)
        assert int(ts.opt.step_dev.cpu()) == i + 1
        wb = max(e for n, e in eg.items() if _summed(n))
        wg = max(e for n, e in eg.items() if not _summed(n))
        worst = [max(worst[0], el), max(worst[1], wg), max(worst[2], wb), max(worst[3], max(ep_.values()))]
    assert sorted(ts._graphs) == [0, 1]
    assert checked == set(names)                          # every gradient was compared at one step at least
    print(f"measured train step T={T} B={B} mode={mode}: losses {worst[0]:.2e} gradients {worst[1]:.2e} "
          f"projection / state table gradients {worst[2]:.2e} parameters vs mirror {worst[3]:.2e} "
          f"ClipLoss cancellation per step {kappas}")


def test_train_step_capture_and_loading_are_bitwise_neutral():
    """Three TrainSteps on the same parameters and batches in the benchmarked configuration (bf16, T = 10, B = 1024):
    loaded from device tensors (team_copy_batch) and replayed, loaded from pinned host tensors (copy_) and replayed, and
    loaded from device tensors and run eagerly through _body without a graph.  After three steps over two epochs the
    losses, the gradients and the parameters are bitwise equal: the kernels are run-to-run deterministic."""
    T, B = 10, 1024
    params, protos, text_cls, evo, batches = _step_config(T, B)
    runs = [_make_step(params, protos, text_cls, evo, B, 1) for _ in range(3)]
    for b, ep in zip(batches, EPOCHS):
        dev = [b["image"].cuda(), b["text"].cuda(), b["state"].cuda(), b["label"].cuda()]
        host = [t.clone().pin_memory() for t in (b["image"], b["text"], b["state"], b["label"])]
        runs[0][1].load(*dev)
        runs[0][1].step(epoch=ep)
        runs[1][1].load(*host)
        runs[1][1].step(epoch=ep)
        runs[2][1].load(*dev)
        runs[2][1]._body(ep)
        torch.cuda.synchronize()
    (p0, t0) = runs[0]
    for pg, ts in runs[1:]:
        assert torch.equal(bits(ts.losses6), bits(t0.losses6))
        assert torch.equal(bits(ts.runner.flat_grads), bits(t0.runner.flat_grads))
        for (a, _), (c, _) in zip(ts.pairs, t0.pairs):
            assert torch.equal(bits(a), bits(c))
        assert int(ts.opt.step_dev.cpu()) == 3
