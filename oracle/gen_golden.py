"""Generate golden vectors from the REAL reference (run in the build container only).

    python oracle/gen_golden.py            # writes tests/golden/*.npz

Imports the original project (``$TEAM_REFERENCE_ROOT`` or ``oracle/_ref``) through ``oracle/ref_loader.py`` (stubbed timm / matplotlib /
open_clip), feeds it the seeded tensors of ``oracle/synth.py`` and stores the reference's
outputs.  Inputs and parameters are NOT stored: tests rebuild them from the seeds in
``CASES`` (``oracle/cases.py``).  Large gradients are stored as a row subsample
(``GRAD_ROW_STRIDE``).  TEST INFRASTRUCTURE - never imported by the product.
"""
from __future__ import annotations

import contextlib
import copy
import io
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import ref_loader, synth  # noqa: E402
from oracle.cases import (CASES, GRAD_ROW_STRIDE, case_inputs, grad_subsample)  # noqa: E402
from oracle import team_oracle as O  # noqa: E402

OUT_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _np(t):
    return t.detach().cpu().clone().numpy()


def gen_head(case):
    ci = case_inputs(case)
    net = ref_loader.build_reference_net(ci["params"], ci["protos"])
    b = ci["batch"]
    text = b["text_cls"] if case.get("class_text") else b["text"]
    outs = net.forward_tri_modal(b["image"], text, b["state"])
    res = {"image": _np(outs[0]), "text": _np(outs[1]), "state": _np(outs[2]),
           "proto": _np(outs[3]), "logit_scale_exp": _np(outs[4])}
    names = O.trainable_names(ci["params"])
    sd = dict(net.named_parameters())
    cots = list(ci["cots"])
    if case.get("class_text"):
        cots[1] = cots[1].view(cots[1].shape[0], -1)
    grads = torch.autograd.grad(outs[:4], [sd[n] for n in names], grad_outputs=cots,
                                allow_unused=True)
    for n, g in zip(names, grads):
        res["grad:" + n] = _np(grad_subsample(g))
    with torch.no_grad():
        from models.proof import Learner
        fake = types.SimpleNamespace(_network=net, _device=torch.device("cpu"))
        logits = Learner.forward_for_classification(fake, b["image"], b["text_cls"])
    res["cls_logits"] = _np(logits)
    return res


def gen_proof_forward(case):
    ci = case_inputs(case)
    net = ref_loader.build_reference_net(ci["params"], ci["protos"])
    b = ci["batch"]
    with torch.no_grad():
        img, txt, ls, pr = net.forward(b["image"], b["text_cls"])
    return {"image": _np(img), "text": _np(txt), "proto": _np(pr), "logit_scale_exp": _np(ls)}


def gen_proof_grad(case):
    """Proof_Net.forward with autograd: cotangents = the first C rows of the synthetic cotangent set."""
    ci = case_inputs(case)
    net = ref_loader.build_reference_net(ci["params"], ci["protos"])
    b = ci["batch"]
    img, txt, ls, pr = net.forward(b["image"], b["text_cls"])
    C = ci["C"]
    cots = [ci["cots"][0], ci["cots"][2][:txt.shape[0]], ci["cots"][3][:C]]
    names = O.trainable_names(ci["params"])
    sd = dict(net.named_parameters())
    grads = torch.autograd.grad([img, txt, pr], [sd[n] for n in names], grad_outputs=cots, allow_unused=True)
    res = {"image": _np(img), "text": _np(txt), "proto": _np(pr)}
    for n, g in zip(names, grads):
        res["grad:" + n] = _np(grad_subsample(g))
    return res


def gen_mha(case):
    """The reference MultiHeadAttention module itself (convs/projections.py:41-87), eval mode, q != k != v."""
    ref_loader.install_stubs()
    from convs.projections import MultiHeadAttention
    ci = case_inputs(case)
    m = MultiHeadAttention(1, 512, 512, 512, dropout=0.1)
    p = ci["params"]
    with torch.no_grad():
        m.w_qs.weight.copy_(p["sel_attn.w_qs.weight"]); m.w_ks.weight.copy_(p["sel_attn.w_ks.weight"])
        m.w_vs.weight.copy_(p["sel_attn.w_vs.weight"]); m.fc.weight.copy_(p["sel_attn.fc.weight"])
        m.fc.bias.copy_(p["sel_attn.fc.bias"]); m.layer_norm.weight.copy_(p["sel_attn.layer_norm.weight"])
        m.layer_norm.bias.copy_(p["sel_attn.layer_norm.bias"])
    m.eval()
    q, k, v = (ci[n].clone().requires_grad_(True) for n in ("q", "k", "v"))
    out = m(q, k, v)
    par = [m.w_qs.weight, m.w_ks.weight, m.w_vs.weight, m.fc.weight, m.fc.bias, m.layer_norm.weight, m.layer_norm.bias]
    grads = torch.autograd.grad(out, [q, k, v] + par, grad_outputs=ci["cot"])
    res = {"out": _np(out)}
    for n, g in zip(("q", "k", "v", "w_q", "w_k", "w_v", "w_fc", "b_fc", "ln_g", "ln_b"), grads):
        res["grad:" + n] = _np(grad_subsample(g))
    return res


def gen_herding(case):
    """The real BaseLearner._construct_exemplar (models/base.py:274-343) on the synthetic DataManager (features ARE the
    vectors: extract_vector = identity): picked rows per class and the exemplar class means."""
    ref_loader.install_stubs()
    from oracle import learner_harness
    import models.base as ref_base
    from torch.utils.data import DataLoader as _DL
    ref_base.DataLoader = lambda *a, **k: _DL(*a, **{**k, "num_workers": 0})
    ci = case_inputs(case)
    dm = learner_harness.FakeDataManager(ci["data"])
    nc = case["n_classes"]
    net = types.SimpleNamespace(eval=lambda: None, extract_vector=lambda x: x)
    fake = types.SimpleNamespace(_network=net, _device=torch.device("cpu"), _known_classes=0, _total_classes=nc,
                                 _data_memory=np.array([]), _targets_memory=np.array([]), feature_dim=512,
                                 _class_means=np.zeros((nc, 512)))
    fake._extract_vectors = types.MethodType(ref_base.BaseLearner._extract_vectors, fake)
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        ref_base.BaseLearner._construct_exemplar(fake, dm, case["m"])
    mem = np.asarray(fake._data_memory, dtype=np.int64).reshape(nc, case["m"], 2)      # (split, row in the train split)
    first = np.array([np.where(ci["data"].y["train"] == c)[0][0] for c in range(nc)])
    return {"picked": mem[:, :, 1] - first[:, None], "class_means": np.asarray(fake._class_means, dtype=np.float64)}


def gen_cosine_linear(case):
    ref_loader.install_stubs()
    from convs.linears import CosineLinear
    ci = case_inputs(case)
    fc = CosineLinear(512, ci["weight"].shape[0])
    with torch.no_grad():
        fc.weight.copy_(ci["weight"])
        fc.sigma.fill_(case["sigma"])
        out = fc(ci["x"])["logits"]
    return {"logits": _np(out), "argmax": _np(out.argmax(1))}


def gen_cal_prototype(case):
    ref_loader.install_stubs()
    from models.proof import Learner
    ci = case_inputs(case)
    x, y, s = ci["x"], ci["y"], ci["s"]
    net = ref_loader.build_reference_net(synth.make_params(1, seed=7), None)
    C = case["num_classes"]
    with contextlib.redirect_stdout(io.StringIO()):
        net.update_prototype(C)
    bs = case["loader_batch"]
    loader = [(None, {"image": x[i:i + bs], "stage_id": s[i:i + bs]}, y[i:i + bs])
              for i in range(0, x.shape[0], bs)]
    fake = types.SimpleNamespace(_network=net, _device=torch.device("cpu"),
                                 _known_classes=case["known"], _total_classes=C)
    Learner.cal_prototype(fake, loader, net)
    res = {"img_prototypes": _np(net.img_prototypes)}
    keys, vals = [], []
    for c, sd in net.img_prototypes_by_state.items():
        for st, pr in sd.items():
            keys.append((c, st))
            vals.append(_np(pr))
    res["by_state_keys"] = np.array(keys, dtype=np.int64).reshape(-1, 2)
    res["by_state_vals"] = np.stack(vals) if vals else np.zeros((0, 512), np.float32)
    return res


def gen_simplecil(case):
    ref_loader.install_stubs()
    from models.simplecil import Learner as SLearner
    from convs.linears import CosineLinear
    ci = case_inputs(case)
    x, y = ci["x"], ci["y"]
    C = case["num_classes"]
    fcnet = types.SimpleNamespace(fc=CosineLinear(512, C))
    with torch.no_grad():
        fcnet.fc.weight.zero_()
    model = types.SimpleNamespace(convnet=ref_loader.FakeCLIP())
    model.eval = lambda: model
    bs = case["loader_batch"]
    loader = [(None, x[i:i + bs], y[i:i + bs]) for i in range(0, x.shape[0], bs)]
    fake = types.SimpleNamespace(_device=torch.device("cpu"), _network=fcnet,
                                 train_dataset=types.SimpleNamespace(labels=y.numpy()))
    with contextlib.redirect_stdout(io.StringIO()):
        SLearner.replace_fc(fake, loader, model, None)
    W = fcnet.fc.weight.data
    with torch.no_grad():
        logits = fcnet.fc(x[:64])["logits"]
    return {"fc_weight": _np(W), "logits64": _np(logits)}


def gen_evolve(case):
    ci = case_inputs(case)
    net = ref_loader.build_reference_net(ci["params"], ci["protos"])
    by_state = {c: {s: v.clone() for s, v in sd.items()} for c, sd in ci["by_state"].items()}
    net.img_prototypes_by_state = by_state
    captured = {}
    gcn = net.state_embedder.temporal_gcn
    orig_forward = gcn.forward

    def spy(node_features, edge_index, edge_weights, time_steps):
        captured["edge_index"] = edge_index.clone()
        captured["edge_weights"] = edge_weights.clone()
        captured["time_steps"] = time_steps.clone()
        return orig_forward(node_features, edge_index, edge_weights, time_steps)

    gcn.forward = spy
    res_ref = net.state_evolution_graph.evolve_and_update(net.img_prototypes_by_state)
    res = {"edge_index": _np(captured["edge_index"]), "edge_weights": _np(captured["edge_weights"]),
           "time_steps": _np(captured["time_steps"])}
    keys, vals = [], []
    for c, sd in res_ref["prototypes"].items():
        for st, pr in sd.items():
            keys.append((c, st))
            vals.append(_np(pr))
    res["proto_keys"] = np.array(keys, dtype=np.int64).reshape(-1, 2)
    res["proto_vals"] = np.stack(vals)
    emb_idx = [i for i, e in enumerate(res_ref["embeddings"]) if e is not None]
    res["emb_idx"] = np.array(emb_idx, dtype=np.int64)
    res["emb_vals"] = np.stack([_np(res_ref["embeddings"][i]) for i in emb_idx])
    lf = res_ref["lifecycle_features"]
    res["lifecycle_idx"] = np.array(list(lf.keys()), dtype=np.int64)
    res["lifecycle_vals"] = np.stack([_np(v) for v in lf.values()])
    dk, dv = [], []
    for s1, dd in res_ref["distances"].items():
        for s2, v in dd.items():
            dk.append((s1, s2))
            dv.append(v)
    res["dist_keys"] = np.array(dk, dtype=np.int64).reshape(-1, 2)
    res["dist_vals"] = np.array(dv, dtype=np.float64)
    # second phase: evolve_state_prototypes (second GCN pass on the mutated dict) + sync,
    # then the Learner's EMA into the distance matrix (models/proof.py:643-682)
    gcn.forward = orig_forward
    with contextlib.redirect_stdout(io.StringIO()):
        net.evolve_state_prototypes()
    res["img_prototypes_after_sync"] = _np(net.img_prototypes)
    from models.proof import Learner
    from utils.state_distance import AdaptiveStateDistanceMatrix
    sdm = AdaptiveStateDistanceMatrix(num_states=10, feature_dim=512, init_with_prior=True)
    res["prior_matrix"] = _np(sdm.get_distance_matrix())
    res["prior_factors"] = _np(sdm.distance_factors)
    fake = types.SimpleNamespace(_network=net, state_distance=sdm)
    Learner.update_state_distance_matrix(fake, None)
    res["factors_after_update"] = _np(sdm.distance_factors)
    res["matrix_after_update"] = _np(sdm.get_distance_matrix())
    return res


def gen_state_distance_forward(case):
    ref_loader.install_stubs()
    from utils.state_distance import AdaptiveStateDistanceMatrix
    ci = case_inputs(case)
    sdm = AdaptiveStateDistanceMatrix(num_states=10, feature_dim=512, init_with_prior=True)
    sdm.train()
    with torch.no_grad():
        ret0 = sdm(ci["feat"], ci["sid"])
        f1 = sdm.distance_factors.detach().clone()
        ret1 = sdm(ci["feat"], ci["sid"])      # counter=1: no update
        f2 = sdm.distance_factors.detach().clone()
    return {"ret0": _np(ret0), "factors1": _np(f1), "ret1": _np(ret1), "factors2": _np(f2),
            "counter": np.array(sdm.update_counter)}


def gen_dynamic_gcn(case):
    ref_loader.install_stubs()
    from models.dynamic_modal_graph import DynamicGCN
    ci = case_inputs(case)
    net = DynamicGCN(512, 256, 512, num_layers=2)
    with torch.no_grad():
        for i, (W, b, g, be) in enumerate(ci["layers"]):
            net.layers[i].weight.copy_(W)
            net.layers[i].bias.copy_(b)
            net.norms[i].weight.copy_(g)
            net.norms[i].bias.copy_(be)
    net.eval()
    with torch.no_grad():
        out = net(ci["x"], ci["edge_index"], ci["edge_weights"])
    return {"out": _np(out)}


def gen_unicl(case):
    ref_loader.install_stubs()
    from models.proof import unicl_loss
    ci = case_inputs(case)
    x = [ci[k].clone().requires_grad_(True) for k in ("image", "text", "state")]
    total, info = unicl_loss(x[0], x[1], x[2], ci["labels"], ci["states"], state_distance=None,
                             epoch=case["epoch"], max_epoch=case["max_epoch"], evolution_features=ci.get("evolution"))
    total.backward()
    return {"total": _np(total.detach()), "instance": np.float64(info["instance_loss"]), "category": np.float64(info["category_loss"]),
            "temperature": np.float64(info["temperature"]), "g_image": _np(x[0].grad), "g_text": _np(x[1].grad.reshape(-1, 512)),
            "g_state": _np(x[2].grad)}


def gen_clip(case):
    ref_loader.install_stubs()
    from utils.toolkit import ClipLoss
    ci = case_inputs(case)
    x = [ci[k].clone().requires_grad_(True) for k in ("image", "text")]
    loss = ClipLoss()(x[0], x[1], torch.tensor(case["logit_scale"]))
    loss.backward()
    return {"loss": _np(loss.detach()), "g_image": _np(x[0].grad), "g_text": _np(x[1].grad)}


def gen_learner(case):
    """The unmodified reference learner (models/proof.py Learner.incremental_train) on the synthetic DataManager of
    oracle/learner_harness.py, CPU, dropout p = 0: accuracy curve, prototypes, per-state prototypes, distance factors,
    exemplar memory and trained parameters after `tasks` tasks."""
    from oracle import learner_harness
    import contextlib, io
    with contextlib.redirect_stderr(io.StringIO()):
        return learner_harness.run(torch.device("cpu"), swap=False, tasks=case["tasks"], epochs=case["epochs"], seed=case["seed"])


GENERATORS = {"head": gen_head, "learner": gen_learner, "unicl": gen_unicl, "clip": gen_clip, "proof_forward": gen_proof_forward, "proof_grad": gen_proof_grad, "mha": gen_mha, "herding": gen_herding,
              "cosine_linear": gen_cosine_linear, "cal_prototype": gen_cal_prototype,
              "simplecil": gen_simplecil, "evolve": gen_evolve,
              "state_distance_forward": gen_state_distance_forward,
              "dynamic_gcn": gen_dynamic_gcn}


def main():
    assert ref_loader.available(), "reference not mounted; golden vectors can only be generated in the build container"
    os.makedirs(OUT_DIR, exist_ok=True)
    torch.set_num_threads(1)           # deterministic reduction order on the generating box
    only = sys.argv[1:]
    for name, case in CASES.items():
        if only and name not in only:
            continue
        res = GENERATORS[case["kind"]](case)
        path = os.path.join(OUT_DIR, name + ".npz")
        np.savez_compressed(path, **res)
        print(f"{name}: {len(res)} arrays -> {path} ({os.path.getsize(path) / 1024:.0f} KiB)")


if __name__ == "__main__":
    main()
