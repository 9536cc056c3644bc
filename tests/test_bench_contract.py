"""The bench contract on the CPU: the reference arm runs without a GPU and prints ONE JSON line with the keys its readers
use; the argument parser defaults finish within minutes; the workload description is the one BASELINE.json names.
On the GPU: --dump-outputs writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert rec["impl"] == "reference" and rec["n_gpus"] == 1 and rec["steps"] == 1
    assert rec["metric"] == "team_head_fwd_bwd_samples_per_sec" and rec["unit"] == "samples/s" and rec["higher_is_better"] is True
    assert "samples/sec" in base["metric"] and not base["published"]                 # vs_baseline stays null: nothing published
    assert rec["value"] > 0 and abs(rec["value"] - 1024 / (rec["ms_per_step"] * 1e-3)) < 1e-6 * rec["value"]
    assert rec["vs_baseline"] is None and rec["gpu_launches"] == 0
    cb = rec["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == rec["value"] and cb["sample"]
    e2e = rec["e2e"]
    assert e2e["value"] == rec["value"] and e2e["unit"] == rec["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert rec["config"]["tasks"] == 10 and rec["config"]["batch_per_gpu"] == 1024 and "model" not in rec["config"]


def test_reference_arm_other_ranks_exit_without_work():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_defaults_and_workload_description():
    import bench
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        a = bench.parse()
    finally:
        sys.argv = argv
    assert a.gpus == 1 and a.warmup >= 3 and a.steps >= 1 and a.impl != "reference"
    cfg = bench.workload_config(10, 1024, 8)
    assert cfg["global_batch"] == 8192 and cfg["parallelism"] == "dp8" and "T=10" in cfg["workload"]


def test_dump_outputs_keep_a_fixed_row_sample_within_the_budget():
    import types
    import torch
    import bench
    B = 1000
    g = torch.Generator().manual_seed(1)
    runner = types.SimpleNamespace(B=B, outs=torch.randn(4, B, 512, generator=g), logits=torch.randn(B, 20, generator=g),
                                   argmax=torch.randint(0, 20, (B,), generator=g),
                                   grad_views={"w_fc": torch.randn(512 * 512, generator=g), "b_fc": torch.randn(512, generator=g)})
    full = bench.last_step_outputs(runner)
    assert "sample_rows" not in full and torch.equal(full["out_text"], runner.outs[1])
    assert torch.equal(full["cls_argmax"], runner.argmax.double()) and torch.equal(full["grad_b_fc"], runner.grad_views["b_fc"])
    budget = 2 << 20
    a, b = bench.last_step_outputs(runner, budget), bench.last_step_outputs(runner, budget)
    assert all(v.dtype in (torch.float32, torch.float64) for v in a.values())
    assert sum(v.numel() * v.element_size() for v in a.values()) <= budget
    rows = a["sample_rows"].long()
    assert 0 < len(rows) < B and torch.equal(rows, rows.unique())
    assert torch.equal(a["out_state"], runner.outs[2][rows]) and torch.equal(a["cls_logits"], runner.logits[rows])
    assert torch.equal(a["cls_argmax"], runner.argmax[rows].double())
    assert torch.equal(a["grad_w_fc"], runner.grad_views["w_fc"])
    assert set(a) == set(b) and all(torch.equal(a[k], b[k]) for k in a)
    with pytest.raises(ValueError):
        bench.last_step_outputs(runner, 1 << 20)                      # the gradients alone are 1 MiB + 2 KiB


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """The dumped arrays equal a direct HeadStepRunner step on the inputs of the last timed step.  With 3 warm-up and 3
    timed steps bench.py rotates over 8 input sets, so step 5 (the last) reads set 5; set 4 must not match."""
    import torch
    from oracle import synth
    from team_b200 import head
    T, B, warmup, steps = 2, 64, 3, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                          "--tasks", str(T), "--batch", str(B), "--mode", "f32", "--no-scale", "--no-e2e", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert sum(v.nbytes for v in got.values()) <= 64 << 20
    C, dev = 2 * T, torch.device("cuda")
    pack = head.HeadParamPack.from_state_dict({k: v.to(dev) for k, v in synth.make_params(T, seed=42, perturb_ln=False).items()})
    r = head.HeadStepRunner(pack, synth.make_prototypes(C).to(dev), B, C, head.MODE_F32)
    text_cls = synth.make_text_class_features(20)[:C].contiguous().to(dev)

    def step(j):
        b = synth.make_batch(B, C, step=j)
        cots = [c.reshape(B, 512).to(dev) for c in synth.make_cotangents(B, step=j)]
        r.step(b["image"].to(dev), b["text"].to(dev), b["state"].to(dev), text_cls, cots)
        torch.cuda.synchronize()
        want = {"out_image": r.outs[0], "out_text": r.outs[1], "out_state": r.outs[2], "out_proto": r.outs[3],
                "cls_logits": r.logits, "cls_argmax": r.argmax.double()}
        want.update({"grad_" + k: v for k, v in r.grad_views.items()})
        return {k: v.cpu().numpy() for k, v in want.items()}

    last = step(warmup + steps - 1)
    assert set(got) == set(last), sorted(set(got) ^ set(last))
    for k in last:
        assert got[k].shape == last[k].shape and rel(got[k], last[k]) < 1e-6, k
    assert rel(got["out_image"], step(warmup + steps - 2)["out_image"]) > 1e-3
