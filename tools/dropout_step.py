"""Cost of train-mode sel_attn dropout at the bench shape (B = 1024, T = 10, C = 20, P = 100, bf16): the head's forward +
backward (HeadStepRunner, one captured graph replayed) at p = 0 and p = 0.1, the complete training step (TrainStep graph)
at p = 0 and p = 0.1, and Proof_Net.forward_tri_modal + backward in train mode (autograd, eager) on the token route and on
the fused route.  Pairs are run alternately in one process; CUDA events, median of the rounds.  Prints the card name and
power limit beside the numbers.

    python tools/dropout_step.py [--batch 1024] [--rounds 5] [--iters 20]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import synth  # noqa: E402
from team_b200 import head  # noqa: E402


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    B, T, ppt, C = a.batch, 10, 10, 20
    params = {k: v.cuda().requires_grad_(True) for k, v in synth.make_params(T, seed=5, prompts_per_task=ppt).items()}
    protos = synth.make_prototypes(C, seed=6).cuda()
    batch = {k: v.cuda() for k, v in synth.make_batch(B, C, step=1).items()}
    cots = [c.reshape(B, 512).cuda() for c in synth.make_cotangents(B, step=1)]
    pack = head.HeadParamPack.from_state_dict(params)
    img, txt, sid = batch["image"], batch["text"], batch["state"]

    def head_graph(p):
        """HeadStepRunner forward + backward (+ the offset advance) captured once, timed as graph replays."""
        run = head.HeadStepRunner(pack, protos, B, 0, head.MODE_BF16, dropout_p=p, seed=7)
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            run.forward(img, txt, sid); run.backward(img, txt, sid, cots); run.advance_offset()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                run.forward(img, txt, sid); run.backward(img, txt, sid, cots); run.advance_offset()
        torch.cuda.current_stream().wait_stream(st)
        return g.replay

    def train_graph(p):
        from team_b200 import train
        pg = {k: v.detach().clone() for k, v in params.items()}
        text_cls = synth.make_text_class_features(20)[:C].contiguous().cuda()
        ts = train.TrainStep(pg, protos, B, text_cls, mode=head.MODE_BF16, dropout_p=p, seed=7)
        ts.load(img, txt, sid, batch["label"])
        return lambda: ts.step(epoch=0)

    from team_b200 import inc_net
    from oracle.ref_loader import FakeCLIP
    args = {"device": [torch.device("cuda:0")], "projection_type": "pure_mlp", "context_prompt_length_per_task": ppt}
    net = inc_net.Proof_Net(args, False, convnet=FakeCLIP().cuda(), tokenizer=lambda t: t)
    net.update_prototype(C)
    for _ in range(T):
        net.update_context_prompt(); net.extend_task()
    net.cuda().train()
    net.team_mode = head.MODE_BF16
    nparams = [p for p in net.parameters() if p.requires_grad]

    def net_step(tokens):
        def f():
            o = net._tri_modal_tokens(net._img_feats(img), net._txt_feats(txt), sid) if tokens else net.forward_tri_modal(img, txt, sid)
            torch.autograd.grad(sum((x.reshape(c.shape) * c).sum() for x, c in zip(o[:4], cots)), nparams, allow_unused=True)
        return f

    pairs = {"head_fwd_bwd_graph": (head_graph(0.0), head_graph(0.1)),
             "train_step_graph": (train_graph(0.0), train_graph(0.1)),
             "proof_net_train_mode": (net_step(True), net_step(False))}
    res = {k: ([], []) for k in pairs}
    for _ in range(a.rounds):
        for k, (f0, f1) in pairs.items():
            res[k][0].append(timed(f0, a.iters))
            res[k][1].append(timed(f1, a.iters))
    med = lambda v: sorted(v)[len(v) // 2]
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    out = {"card": card, "batch": B, "T": T, "C": C, "P": T * ppt, "mode": "bf16", "timing": "CUDA events, median of rounds",
           "head_fwd_bwd_graph_ms": {"p0": med(res["head_fwd_bwd_graph"][0]), "p0.1": med(res["head_fwd_bwd_graph"][1])},
           "train_step_graph_ms": {"p0": med(res["train_step_graph"][0]), "p0.1": med(res["train_step_graph"][1])},
           "proof_net_train_mode_eager_ms": {"token_route": med(res["proof_net_train_mode"][0]), "fused_route": med(res["proof_net_train_mode"][1])}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
