"""Train-mode sel_attn dropout in the fused tri-modal head (team_dropout): the fused route must compute the same function
on the same masks as the token route (the [B, L, 512] tokens [image | text | state | C prototypes | P prompts] through
head.mha with the same (p, seed, offset)), in fp32 mode at the fp32 parity bar, in bf16 mode within twice the error of
the undropped bf16 step; both routes must equal the fp64 oracle on explicit masks; the masks must move with the offset and
be reproducible; HeadStepRunner replays and TrainStep steps must draw fresh masks from the device-resident offset;
Proof_Net in train mode must take the fused route and equal its token route after the same torch.manual_seed.  Plus a
CPU check of the ABI struct."""
import ctypes
import os
import subprocess
import tempfile

import pytest
import torch

from oracle import synth
from oracle import team_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P_DROP = 0.1


def rel(a, b):
    a = torch.as_tensor(a).detach().double()
    b = torch.as_tensor(b).detach().double().to(a.device)
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def test_dropout_struct_matches_the_c_header():
    from team_b200 import capi
    fields = ["p", "seed", "offset", "offset_dev", "workspace", "workspace_bytes"]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "team_b200.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(team_dropout));']
    lines += [f'  printf("{f} %zu\\n", offsetof(team_dropout, {f}));' for f in fields]
    lines += ["  return 0;", "}"]
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "abi.c"), os.path.join(td, "abi")
        open(src, "w").write("\n".join(lines))
        subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        got = dict((ln.split()[0], int(ln.split()[1])) for ln in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines())
    assert ctypes.sizeof(capi.Dropout) == got["size"]
    for f in fields:
        assert getattr(capi.Dropout, f).offset == got[f], f


def _case(C, T, ppt, B, seed, five_state=False):
    params = {k: v.cuda().requires_grad_(True) for k, v in synth.make_params(T, seed=seed, prompts_per_task=ppt).items()}
    protos = synth.make_prototypes(C, seed=seed + 1).cuda()
    batch = {k: v.cuda() for k, v in synth.make_batch(B, C, step=seed % 97, five_state=five_state, num_classes_total=max(C, 20)).items()}
    cots = [c.reshape(B, 512).cuda() for c in synth.make_cotangents(B, step=seed % 97)]
    return params, protos, batch, cots


def _fused(params, protos, batch, mode, dropout):
    from team_b200 import head
    pack = head.HeadParamPack.from_state_dict(params)
    return head.forward_tri_modal(pack, batch["image"], batch["text"], batch["state"], protos, mode=mode, dropout=dropout)[:4]


def _tokens(params, protos, batch, mode, dropout):
    from team_b200 import head
    pack = head.HeadParamPack.from_state_dict(params)
    img, txt, sid = batch["image"], batch["text"], batch["state"]
    B, C = img.shape[0], protos.shape[0]
    xi = head.encode_grad(pack, "image", img, normalize=True, mode=mode)
    xt = head.encode_grad(pack, "text", txt, normalize=True, mode=mode)
    xs = head.encode_grad(pack, "state", sid, normalize=True, mode=mode)
    xp = head.encode_grad(pack, "prototypes", protos, normalize=True, mode=mode)
    T = pack.T
    prompts = torch.cat([params[f"context_prompts.{t}"] for t in range(T)], 0)
    toks = torch.cat([xi.view(B, 1, 512), xt.view(B, 1, 512), xs.view(B, 1, 512), xp.view(1, C, 512).expand(B, C, 512),
                      prompts.view(1, -1, 512).expand(B, -1, 512)], 1).contiguous()
    p, s, o = dropout
    f = head.mha(toks, toks, toks, params["sel_attn.w_qs.weight"], params["sel_attn.w_ks.weight"], params["sel_attn.w_vs.weight"],
                 params["sel_attn.fc.weight"], params["sel_attn.fc.bias"], params["sel_attn.layer_norm.weight"],
                 params["sel_attn.layer_norm.bias"], mode=mode, dropout_p=p, seed=s, offset=o)
    return f[:, 0], f[:, 1:2], f[:, 2], f[:, 3:3 + C].mean(1)


def _with_grads(fn, params, protos, batch, cots, mode, dropout):
    outs = fn(params, protos, batch, mode, dropout)
    loss = sum((o.reshape(c.shape) * c).sum() for o, c in zip(outs, cots))
    names = [k for k, v in params.items()]
    gs = torch.autograd.grad(loss, [params[k] for k in names], allow_unused=True)
    return [o.detach() for o in outs], {k: g for k, g in zip(names, gs) if g is not None}


CASES = [  # (C, T, prompts per task, B, seed, five_state)
    (20, 1, 10, 6, 11, False),
    (20, 3, 10, 5, 12, True),
    (20, 2, 10, 7, 13, False),
    (24, 2, 10, 6, 14, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("C,T,ppt,B,seed,five", CASES)
def test_fused_route_equals_the_token_route_f32(C, T, ppt, B, seed, five):
    from team_b200 import head
    params, protos, batch, cots = _case(C, T, ppt, B, seed, five)
    drop = (P_DROP, 1234 + seed, 2 * seed + 6)
    fo, fg = _with_grads(_fused, params, protos, batch, cots, head.MODE_F32, drop)
    to, tg = _with_grads(_tokens, params, protos, batch, cots, head.MODE_F32, drop)
    for a, b in zip(fo, to):
        assert rel(a.reshape(b.shape), b) <= 1e-5, [rel(x.reshape(y.shape), y) for x, y in zip(fo, to)]
    for k in tg:
        assert k in fg, k
        assert rel(fg[k], tg[k]) <= 2e-5, (k, rel(fg[k], tg[k]))
    # the undropped head differs: the masks took effect
    ev = _fused(params, protos, batch, head.MODE_F32, None)
    assert rel(fo[0], ev[0].detach()) > 1e-3
    # both against the fp64 oracle: the reference's token tensor with EXPLICIT masks (team_oracle.mha(drop=...))
    oo, og = _oracle(params, protos, batch, cots, drop)
    for a, b, c in zip(fo, to, oo):
        assert rel(a.reshape(c.shape), c) <= 1e-5 and rel(b.reshape(c.shape), c) <= 1e-5
    for k in og:
        if k in fg:
            assert rel(fg[k], og[k]) <= 2e-5 and rel(tg[k], og[k]) <= 2e-5, (k, rel(fg[k], og[k]), rel(tg[k], og[k]))


def _oracle(params, protos, batch, cots, drop):
    """fp64 CPU: oracle.forward_tri_modal with sel_attn in train mode on the masks of ``drop``; outputs and gradients."""
    p64 = {k: v.detach().double().cpu().requires_grad_(True) for k, v in params.items()}
    old = O.sel_attn
    O.sel_attn = lambda x, p: O.mha(x, x, x, p, drop=drop)
    try:
        o = O.forward_tri_modal(p64, batch["image"].double().cpu(), batch["text"].double().cpu(), batch["state"].cpu(),
                                protos.double().cpu())[:4]
    finally:
        O.sel_attn = old
    loss = sum((x.reshape(c.shape) * c.double().cpu()).sum() for x, c in zip(o, cots))
    names = O.trainable_names(params)
    gs = torch.autograd.grad(loss, [p64[n] for n in names], allow_unused=True)
    return [x.detach() for x in o], {n: g for n, g in zip(names, gs) if g is not None}


@pytest.mark.gpu
def test_masks_move_with_the_offset_and_reproduce():
    from team_b200 import head
    params, protos, batch, cots = _case(20, 2, 10, 7, 21)
    with torch.no_grad():
        a = _fused(params, protos, batch, head.MODE_F32, (P_DROP, 99, 10))
        b = _fused(params, protos, batch, head.MODE_F32, (P_DROP, 99, 10))
        c = _fused(params, protos, batch, head.MODE_F32, (P_DROP, 99, 12))
        z = _fused(params, protos, batch, head.MODE_F32, (0.0, 99, 10))
        n = _fused(params, protos, batch, head.MODE_F32, None)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert all(rel(x, y) > 1e-3 for x, y in zip(a, c))
    for x, y in zip(z, n):
        assert torch.equal(x, y)
    # a real team_dropout with p = 0 (not a NULL pointer) runs the undropped head as well
    import ctypes as C
    from team_b200 import capi
    keep = []

    def p0_struct(dropout, B, C_, P, mode, dev):
        dws = torch.empty((256,), dtype=torch.uint8, device=dev)
        keep.append(dws)
        return C.pointer(capi.Dropout(0.0, 99, 10, None, dws.data_ptr(), 256)), dws
    orig = head._dropout_arg
    head._dropout_arg = p0_struct
    try:
        with torch.no_grad():
            z2 = _fused(params, protos, batch, head.MODE_F32, (0.0, 99, 10))
    finally:
        head._dropout_arg = orig
    assert keep
    for x, y in zip(z2, n):
        assert torch.equal(x, y)
    # gradients are reproducible bit for bit (fixed-order folds)
    _, g1 = _with_grads(_fused, params, protos, batch, cots, head.MODE_F32, (P_DROP, 99, 10))
    _, g2 = _with_grads(_fused, params, protos, batch, cots, head.MODE_F32, (P_DROP, 99, 10))
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1024, 4096])
def test_bf16_dropout_within_twice_the_undropped_bf16_error(B):
    """bench shape (T = 10, C = 20, P = 100); B = 4096 takes the persistent GEMM path."""
    from team_b200 import head
    params, protos, batch, cots = _case(20, 10, 10, B, 31)
    drop = (P_DROP, 555, 40)
    err = {}
    for name, dr in (("drop", drop), ("plain", None)):
        ref_o, ref_g = _with_grads(_fused if dr is None else _tokens, params, protos, batch, cots, head.MODE_F32,
                                   dr if dr is not None else None)
        o, g = _with_grads(_fused, params, protos, batch, cots, head.MODE_BF16, dr)
        err[name] = (max(rel(a.reshape(b.shape), b) for a, b in zip(o, ref_o)), max(rel(g[k], ref_g[k]) for k in ref_g))
    assert err["drop"][0] <= 2 * err["plain"][0], err
    assert err["drop"][1] <= 2 * err["plain"][1], err


@pytest.mark.gpu
def test_proof_net_train_mode_takes_the_fused_route():
    from team_b200 import inc_net, head
    from oracle.ref_loader import FakeCLIP
    dev = torch.device("cuda:0")
    args = {"device": [dev], "projection_type": "pure_mlp", "context_prompt_length_per_task": 10}
    net = inc_net.Proof_Net(args, False, convnet=FakeCLIP().to(dev), tokenizer=lambda t: t)
    net.update_prototype(4); net.update_context_prompt(); net.extend_task()
    net.to(dev)
    net.train()
    batch = synth.make_batch(5, 4, step=3)
    a = (batch["image"].to(dev), batch["text"].to(dev), batch["state"].to(dev))
    cots = [c.to(dev) for c in synth.make_cotangents(5, step=3)]
    params = [p for p in net.parameters() if p.requires_grad]

    def run(fn):
        torch.manual_seed(77)
        outs = fn()
        loss = sum((o.reshape(c.shape) * c).sum() for o, c in zip(outs[:4], cots))
        gs = torch.autograd.grad(loss, params, allow_unused=True)
        return [o.detach() for o in outs[:4]], gs, torch.randint(0, 2 ** 62, (1,)).item()

    fo, fg, fr = run(lambda: net.forward_tri_modal(*a))
    to, tg, tr = run(lambda: net._tri_modal_tokens(net._img_feats(a[0]), net._txt_feats(a[1]), a[2]))
    assert fr == tr                                          # same consumption of torch's generator
    for x, y in zip(fo, to):
        assert rel(x.reshape(y.shape), y) <= 1e-5
    for x, y in zip(fg, tg):
        if y is not None and float(y.norm()) > 0:
            assert x is not None and rel(x, y) <= 2e-5


@pytest.mark.gpu
def test_head_step_runner_graph_replays_draw_fresh_masks():
    """A captured HeadStepRunner step (forward, backward, advance_offset): replay k uses offset base + 2 k, read on the
    device, and equals the eager call with that offset."""
    from team_b200 import head
    params, protos, batch, cots = _case(20, 1, 10, 6, 41)
    pack = head.HeadParamPack.from_state_dict(params)
    run = head.HeadStepRunner(pack, protos, 6, 0, head.MODE_F32, dropout_p=P_DROP, seed=4242)
    base = run.offset
    assert base % 2 == 0
    img, txt, sid = batch["image"], batch["text"], batch["state"]
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            run.forward(img, txt, sid)
            run.backward(img, txt, sid, cots)
            run.advance_offset()
    torch.cuda.current_stream().wait_stream(st)
    assert run.offset == base                       # capture runs nothing
    got = []
    for k in range(2):
        g.replay()
        torch.cuda.synchronize()
        got.append((run.outs.clone(), {n: v.clone() for n, v in run.grad_views.items()}))
    assert run.offset == base + 4
    for k in range(2):
        eo, eg = _with_grads(_fused, params, protos, batch, cots, head.MODE_F32, (P_DROP, 4242, base + 2 * k))
        outs, gv = got[k]
        for i in range(4):
            assert rel(outs[i], eo[i].reshape(6, 512)) <= 1e-6, (k, i)
        for n, pn in (("w_q", "sel_attn.w_qs.weight"), ("w_fc", "sel_attn.fc.weight"), ("ln_g", "sel_attn.layer_norm.weight"),
                      ("b_fc", "sel_attn.fc.bias"), ("state_emb", "state_embedder.state_embeddings.weight")):
            assert rel(gv[n].view_as(eg[pn]), eg[pn]) <= 1e-6, (k, n)
    assert rel(got[0][0], got[1][0]) > 1e-3            # two replays, two sets of masks


@pytest.mark.gpu
def test_train_step_with_dropout_matches_the_oracle_loop():
    """TrainStep(dropout_p = 0.1) against the fp64 oracle loop of tests/test_gpu_train_step.py whose head forward is the
    reference's token tensor through team_oracle.mha(drop=(p, seed, base + 2 k)) at step k: 3 steps over 2 epochs."""
    import math
    from team_b200 import train, head
    T, B, C = 3, 48, 6
    params = synth.make_params(T, seed=77)
    protos = synth.make_prototypes(C, seed=5)
    text_cls = synth.make_text_class_features(20)[:C].contiguous()
    gen = torch.Generator().manual_seed(9)
    evo = [torch.randn(512, generator=gen) if c != 2 else None for c in range(C)]
    batches = [synth.make_batch(B, C, step=s) for s in range(3)]
    epochs = [0, 0, 1]
    lr0, wd, tuned = 0.004, 0.05, 20
    ls = math.exp(2.6592600369327783)
    dev = torch.device("cuda")
    pg = {k: v.clone().to(dev) for k, v in params.items()}
    ts = train.TrainStep(pg, protos.to(dev), B, text_cls.to(dev), mode=head.MODE_F32, init_lr=lr0, min_lr=1e-8,
                         weight_decay=wd, tuned_epoch=tuned, logit_scale=ls, evolution_features=evo, dropout_p=P_DROP, seed=31337)
    got = []
    for b, ep in zip(batches, epochs):
        ts.load(b["image"], b["text"], b["state"], b["label"])
        got.append(ts.step(epoch=ep).cpu().double().tolist())
    assert int(ts.runner.offset) == ts.dropout_offset(3)
    # ---- oracle loop (fp64, CPU)
    p64 = {k: v.double().clone() for k, v in params.items()}
    names = O.trainable_names(params)
    for n in names:
        p64[n].requires_grad_(True)
    opt = torch.optim.AdamW([p64[n] for n in names], lr=lr0, weight_decay=wd)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=tuned, eta_min=1e-8)
    old = O.sel_attn
    last_epoch = 0
    try:
        for k, (b, ep) in enumerate(zip(batches, epochs)):
            if ep != last_epoch:
                sched.step(); last_epoch = ep
            O.sel_attn = lambda x, p, k=k: O.mha(x, x, x, p, drop=(P_DROP, 31337, ts.dropout_offset(k)))
            img, txt, sid, y = b["image"].double(), b["text"].double(), b["state"], b["label"]
            with torch.no_grad():
                ce = torch.nn.functional.cross_entropy(O.forward_for_classification(p64, img, text_cls.double()), y)
            o = O.forward_tri_modal(p64, img, txt, sid, protos.double())
            un, inst, _ = O.unicl_loss(o[0], o[1], o[2], y, epoch=ep, max_epoch=tuned, state_ids=sid,
                                       evolution_features=[None if e is None else e.double() for e in evo])
            ei = torch.nn.functional.normalize(O.encode_image(img, p64, normalize=True), dim=1)
            et = torch.nn.functional.normalize(O.encode_text(txt, p64, normalize=True), dim=1)
            cl = O.clip_loss(ei, et, ls)
            total = ce + cl + 0.3 * un
            opt.zero_grad()
            total.backward()
            opt.step()
            ref = [float(total), float(ce), float(cl), float(un), float(inst)]
            for a, r in zip(got[k], ref):
                assert abs(a - r) < 2e-5 * max(1.0, abs(r)), (k, got[k], ref)
    finally:
        O.sel_attn = old
    for n in names:
        moved = (p64[n].detach() - params[n].double()).norm()
        err = (pg[n].detach().double().cpu() - p64[n].detach()).norm()
        assert float(err) < 2e-3 * float(moved) + 1e-7, (n, float(err), float(moved))
