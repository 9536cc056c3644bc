"""Launches every kernel family of libteam_b200.so once (after a warm-up pass) between cudaProfilerStart/Stop, for
    ncu --set full --profile-from-start off ... python tools/all_kernels.py
Sizes: the headline head step (B = 1024, T = 10, bf16), a 16384-sample step for the persistent GEMM + Gram table-row
kernels (the smallest batch that selects them), 512 K rows (1 GB) for the HBM kernels, the 200-class graph.  Kept small on purpose: ncu saves
and restores device memory around every replay pass.  Peer all-reduce needs > 1 GPU and is not covered here."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from team_b200 import capi, graph, head, ops, train   # noqa: E402
from oracle import synth                              # noqa: E402

capi.require_device()
dev = torch.device("cuda")
T, C, B = 10, 20, 1024
params = {k: v.to(dev) for k, v in synth.make_params(T, seed=42, perturb_ln=False).items()}
pack = head.HeadParamPack.from_state_dict(params)
protos = synth.make_prototypes(C).to(dev)
text_cls = synth.make_text_class_features(20)[:C].contiguous().to(dev)
b = {k: v.to(dev) for k, v in synth.make_batch(B, C, step=0).items()}
cots = [c.to(dev).reshape(B, 512) for c in synth.make_cotangents(B, step=0)]
ONLY = os.environ.get("ALLK_ONLY", "")            # "graph": only the graph / state-distance kernels (a short second capture)
gen = torch.Generator(device=dev).manual_seed(0)
big = 8 if ONLY == "graph" else int(os.environ.get('ALLK_BIG', '16384'))   # >= 16384 samples select the Gram table-row kernels
bigx = [torch.nn.functional.normalize(torch.randn(big, 512, generator=gen, device=dev), dim=-1) for _ in range(2)]
bigs = torch.randint(1, 5, (big,), generator=gen, device=dev)
bigc = [torch.randn(big, 512, generator=gen, device=dev) for _ in range(4)]
N = 1024 if ONLY == "graph" else 1 << 19
xr = torch.randn(N, 512, generator=gen, device=dev)
yr = torch.randint(0, 20, (N,), generator=gen, device=dev)
sr = torch.randint(0, 10, (N,), generator=gen, device=dev)
Wr = torch.randn(20, 512, generator=gen, device=dev)
gp = {k: v.to(dev) for k, v in synth.make_params(2, seed=77).items()}
bs = {c: {s_: v.to(dev) for s_, v in sd.items()} for c, sd in synth.make_state_prototype_dict(200, seed=9).items()}
evo = [torch.randn(512) for _ in range(C)]
runner = head.HeadStepRunner(pack, protos, B, C, head.MODE_BF16)
runner32 = head.HeadStepRunner(pack, protos, B, C, head.MODE_F32)
runner_big = head.HeadStepRunner(pack, protos, big, C, head.MODE_BF16)
ts = train.TrainStep({k: v.clone() for k, v in params.items()}, protos, B, text_cls, mode=head.MODE_BF16, evolution_features=evo)
mp = [params["sel_attn." + n].clone().requires_grad_(True) for n in
      ("w_qs.weight", "w_ks.weight", "w_vs.weight", "fc.weight", "fc.bias", "layer_norm.weight", "layer_norm.bias")]
tok = torch.randn(64, 141, 512, generator=gen, device=dev).requires_grad_(True)
hx = torch.randn(4096, 512, generator=gen, device=dev)
f = graph.prior_distance_factors(device=dev)


def graph_part():
    r = graph.evolve_and_update(gp, bs, {})
    graph.evolve_state_prototypes(gp, torch.zeros(200, 512, device=dev), bs, {})
    graph.update_state_distance_matrix(f, r["distances"])
    graph.state_distance_forward(f, b["image"], b["state"], 0, training=True)
    graph.get_distance_matrix(f)
    g12 = torch.Generator().manual_seed(1)
    x12 = torch.randn(12, 512, generator=g12).to(dev)
    layers = [tuple(t.to(dev) for t in (torch.randn(o, i, generator=g12) * 0.05, torch.zeros(o), torch.ones(o), torch.zeros(o)))
              for i, o in ((512, 256), (256, 512))]
    graph.dynamic_gcn(x12, torch.randint(0, 12, (2, 30), generator=g12).to(dev), torch.rand(30, generator=g12).to(dev), layers)


def everything():
    if ONLY == "graph":
        return graph_part()
    runner.step(b["image"], b["text"], b["state"], text_cls, cots)                      # head fwd + bwd, bf16 (tcgen05)
    runner32.step(b["image"], b["text"], b["state"], text_cls, cots)                    # fp32 parity mode (FFMA GEMM)
    runner_big.step(bigx[0], bigx[1], bigs, text_cls, bigc)                             # persistent GEMM, Gram table rows
    ts.load(b["image"], b["text"], b["state"], b["label"]); ts._body(0)                 # losses, encode fwd/bwd, AdamW
    head.forward_proof(pack, b["image"], text_cls, protos, mode=head.MODE_BF16)
    head.forward_tri_modal_class_text(pack, b["image"], text_cls, b["state"], protos, mode=head.MODE_BF16)
    out = head.mha(tok, tok, tok, *mp, mode=head.MODE_BF16)
    out.sum().backward()
    head.mean_dim(tok.detach(), 0)
    sums, counts = ops.keyed_sums(xr, yr, num_classes=20); ops.keyed_means(sums, counts)
    ops.keyed_sums(xr, yr, sr, num_classes=20)
    ops.keyed_sums(xr.bfloat16(), yr, num_classes=20)
    ops.cosine_logits(xr, Wr, want_argmax=True)
    ops.cosine_logits(xr[:300], Wr, want_argmax=True)
    ops.herding_select(hx, 20, [1024] * 4)
    graph_part()


everything()
torch.cuda.synchronize()
torch.cuda.profiler.start()
c0 = capi.lib().team_launch_count()
everything()
torch.cuda.synchronize()
torch.cuda.profiler.stop()
print("library launches in the profiled pass:", capi.lib().team_launch_count() - c0)
