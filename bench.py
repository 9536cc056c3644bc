#!/usr/bin/env python
"""bench.py - TEAM head fwd+bwd throughput on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the reference algorithm (oracle port) on the host CPU
    python bench.py ... --dump-outputs DIR      # also write the last timed step's outputs as DIR/<name>.npy

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): PROOF/TEAM
head fwd+bwd, 10 incremental tasks (C=20 classes, P=100 prompts, L=123 tokens), batch 1024
per GPU, synthetic IIMinsects202-shaped 512-d features, reference-initialised weights.
One step = no-grad classification logits (models/proof.py:415-418) + forward_tri_modal
(:424-425) + VJP with fixed N(0,1) cotangents on the four feature outputs (stands for :444),
plus, for N>1, the NCCL all-reduce of the flat 1.85 M-element head-gradient buffer in three buckets
(w_fc | w_q,w_k,w_v | rest) started on a side stream as the backward finishes each of them.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "team_head_fwd_bwd_samples_per_sec"
UNIT = "samples/s"
NUM_TASKS = 10
ROT = 64                         # rotating input slots: 64 x (2 x 2 MiB + cotangents 8 MiB) >> 126 MB L2
DUMP_BYTES = 64 << 20            # --dump-outputs: size of all written arrays together


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="team", choices=["team", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="samples per GPU per step")
    ap.add_argument("--tasks", type=int, default=NUM_TASKS)
    ap.add_argument("--mode", default=os.environ.get("TEAM_BENCH_MODE", "bf16"), choices=["bf16", "f32"])
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-scale", action="store_true", help="skip the larger-batch points (at_scale)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch samples per GPU (headline); strong: --global-batch samples in total, split over the GPUs "
                         "(BASELINE configs[3]: 4096 over 8 GPUs).  For N > 1 the weak line also carries the strong point "
                         "(`strong_scaling`) and an untimed check of the gradient exchange (`grad_exchange_check`).")
    ap.add_argument("--global-batch", type=int, default=4096)
    ap.add_argument("--comm", default="peer", choices=["peer", "nccl", "nccl-buckets"],
                    help="N>1 gradient exchange: own NVLink peer-memory kernel inside the step graph (default), one NCCL "
                         "all-reduce after the step, or three NCCL buckets overlapped with the backward")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed on rank 0 (feature outputs, "
                         "classification logits and argmax, parameter gradients) as DIR/<name>.npy, so that two builds "
                         "can be compared on the same seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "team":
        ap.error("--dump-outputs needs --impl team")
    return a


def ncu_dram_bytes_per_launch(kernel_prefix: str):
    """Average DRAM bytes (read + write) per launch of a kernel from the committed `ncu --set full` summary of this
    workload (profiles/, written by tools/ncu_summary.py); None if the file is missing."""
    import csv
    path = os.path.join(ROOT, "profiles", "r2s_ncu_full_gemm_waves_B1024_T10_summary.csv")
    if not os.path.exists(path):
        return None, None
    rows = list(csv.reader(open(path)))
    hdr = rows[0]
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    cols = [(i, scale.get(h[h.index("[") + 1:h.index("]")], None)) for i, h in enumerate(hdr) if h.startswith("dram__bytes_")]
    vals = [sum(float(r[i]) * sc for i, sc in cols if sc) for r in rows[1:] if r[1].startswith(kernel_prefix)]
    if not vals:
        return None, None
    return sum(vals) / len(vals), os.path.relpath(path, ROOT)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm": d["hbm_gbs"], "tensor_burst": d["bf16_tflops"], "tensor_sustained": d["bf16_tflops_sustained"],
                "src": "measured"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Index of the next sample line: only lines read after mark() are reported."""
        self.first = len(self.lines)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.lines = self.lines[getattr(self, "first", 0):]
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def workload_config(tasks: int, batch: int, world: int) -> dict:
    """The `config` object of BOTH arms (the driver compares them): only what names the workload."""
    C = 2 * tasks
    return {"workload": f"TEAM/PROOF head fwd+bwd (BASELINE configs[2]): T={tasks} tasks, C={C} classes, "
                        f"P={10 * tasks} prompts, L={3 + 12 * tasks} tokens, batch {batch} per GPU",
            "tasks": tasks, "batch_per_gpu": batch, "global_batch": batch * world, "parallelism": f"dp{world}",
            "l2": "rotating input + cotangent sets, together larger than L2 (count and MiB under `run`)",
            "alg_flops_per_sample_survey": 55.07e6 if tasks == 10 else None}


def last_step_outputs(runner, budget: int = DUMP_BYTES) -> dict:
    """Device copies of what the caller of `runner.step` receives from its last step: the four [B,512] feature outputs,
    the classification logits and argmax (as float64) and the gradient of every trainable parameter.  When all of it would
    exceed `budget` bytes, the per-sample arrays keep the same fixed, seeded sample of rows, listed in `sample_rows`.
    Enqueued on the current stream, so later steps on that stream cannot overwrite them."""
    import torch
    rows = {"out_image": runner.outs[0], "out_text": runner.outs[1], "out_state": runner.outs[2],
            "out_proto": runner.outs[3], "cls_logits": runner.logits, "cls_argmax": runner.argmax.double()}
    grads = {"grad_" + k: v for k, v in runner.grad_views.items()}
    fixed = sum(v.numel() * v.element_size() for v in grads.values())
    per_row = sum(v[0].numel() * v.element_size() for v in rows.values())
    if fixed + runner.B * per_row > budget:
        k = (budget - fixed) // (per_row + 8)
        if k < 1:
            raise ValueError(f"--dump-outputs: the gradients alone ({fixed / 2**20:.1f} MiB) leave no room for a sample of "
                             f"rows within {budget / 2**20:.0f} MiB")
        idx = torch.randperm(runner.B, generator=torch.Generator().manual_seed(0))[:k].sort().values
        rows = {n: v.index_select(0, idx.to(v.device)) for n, v in rows.items()}
        rows["sample_rows"] = idx.double()
    return {n: v.detach().clone() for n, v in {**rows, **grads}.items()}


def write_outputs(arrays: dict, out_dir: str):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        v = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), v)
        total += v.nbytes
    print(f"[bench] wrote {len(arrays)} arrays of the last timed step ({total / 2**20:.1f} MiB) to {out_dir}",
          file=sys.stderr, flush=True)


def cpu_reference_step_fn(tasks: int, batch: int, nsets: int = 4):
    """One head step on the host CPU, same step definition as the GPU arm (no-grad classification logits +
    forward_tri_modal + VJP with fixed cotangents).  kind "reference": the UNMODIFIED reference modules
    (utils/inc_net.py Proof_Net, models/proof.py Learner.forward_for_classification) loaded from $TEAM_REFERENCE_ROOT
    or oracle/_ref through oracle/ref_loader.py, fake CLIP = identity on the 512-d features, eval mode.
    kind "port": the oracle restatement (only when the reference tree is not there)."""
    import types
    import torch
    from oracle import ref_loader, synth
    from oracle import team_oracle as O
    C = synth.CLASSES_PER_TASK * tasks
    params = synth.make_params(tasks, seed=42, perturb_ln=False)
    names = O.trainable_names(params)
    protos = synth.make_prototypes(C)
    sets = [(synth.make_batch(batch, C, step=i), synth.make_cotangents(batch, step=i)) for i in range(nsets)]
    if ref_loader.available():
        net = ref_loader.build_reference_net(params, protos)
        from models.proof import Learner                     # reference module (oracle/ref_loader.py)
        fake = types.SimpleNamespace(_network=net, _device=torch.device("cpu"))
        sd = dict(net.named_parameters())
        train = [sd[n] for n in names]
        it = [0]

        def step():
            b, cots = sets[it[0] % nsets]
            it[0] += 1
            for q in train:
                q.grad = None
            with torch.no_grad():
                logits = Learner.forward_for_classification(fake, b["image"], b["text_cls"])
            outs = net.forward_tri_modal(b["image"], b["text"], b["state"])
            torch.autograd.backward(list(outs[:4]), [c.reshape(o.shape) for c, o in zip(cots, outs[:4])])
            return logits
        return step, "reference"
    p = {k: (v.clone().requires_grad_(k in names)) for k, v in params.items()}
    it = [0]

    def step():
        b, cots = sets[it[0] % nsets]
        it[0] += 1
        return O.head_step_fwd_bwd(p, b, protos, cots, names)
    return step, "port"


def time_cpu(tasks: int, batch: int, steps: int, warmup: int, budget_s: float = 0.0):
    """Times `steps` CPU steps (fewer if `budget_s` > 0 would be exceeded - the count actually timed is returned)."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    fn, kind = cpu_reference_step_fn(tasks, batch)
    for _ in range(warmup):
        fn()
    done = 0
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
        done += 1
        if budget_s > 0 and time.perf_counter() - t0 > budget_s:
            break
    dt = (time.perf_counter() - t0) / max(done, 1)
    what = ("the unmodified reference (utils/inc_net.py Proof_Net.forward_tri_modal + models/proof.py "
            "forward_for_classification + autograd), fake CLIP = identity" if kind == "reference"
            else "oracle port of the reference head")
    return {"value": batch / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{done} steps of a {batch}-sample batch (T={tasks}, C={2 * tasks}, L={3 + 12 * tasks}), "
                      f"{what}, torch-CPU fp32 eval mode, {cores} threads, {dt * 1e3:.1f} ms/step"}, dt, done


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warm = max(1, a.warmup)
    # the same batch as the GPU arm (B per GPU), exactly --steps timed steps
    cb, dt, done = time_cpu(a.tasks, a.batch, a.steps, warm)
    # BASELINE configs[0], exactly: B=64, T=1, CPU fp32 (the reference's own CPU-runnable case)
    c1, dt1, n1 = time_cpu(1, 64, 10, 2, budget_s=30.0)
    line = {"metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": workload_config(a.tasks, a.batch, world),
            "run": {"steps_timed": done, "host_threads": cb["cores"], "note": "rank 0 only; one per-GPU batch per step"},
            "cpu_baseline": cb,
            "c1": {"workload": "BASELINE configs[0]: B=64, T=1 (C=2, P=10, L=15), CPU fp32", "samples_per_s": c1["value"],
                   "ms_per_step": dt1 * 1e3, "steps": n1, "kind": c1["kind"], "cores": c1["cores"]},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_team(a):
    import torch
    import torch.distributed as dist
    from oracle import synth                    # input generation only
    from team_b200 import capi, head

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    capi.require_device()
    L = capi.lib()
    mode = head.MODE_BF16 if a.mode == "bf16" else head.MODE_F32
    T, B = a.tasks, a.batch
    if a.scaling == "strong":
        if a.global_batch % world:
            raise SystemExit(f"--global-batch {a.global_batch} is not a multiple of {world} GPUs")
        B = a.global_batch // world
    C = synth.CLASSES_PER_TASK * T
    warmup = max(a.warmup, 3)

    params = synth.make_params(T, seed=42, perturb_ln=False)      # reference initialisers, same on every rank
    pdev = {k: v.to(dev) for k, v in params.items()}
    pack = head.HeadParamPack.from_state_dict(pdev)
    protos = synth.make_prototypes(C).to(dev)
    # rotating inputs (distinct per rank), resident in HBM, total >> L2
    rot = min(ROT, max(8, a.steps + warmup))
    imgs, txts, sids, cots = [], [], [], []
    for i in range(rot):
        b = synth.make_batch(B, C, step=rank * 1000 + i)
        imgs.append(b["image"].to(dev)); txts.append(b["text"].to(dev)); sids.append(b["state"].to(dev))
        c = synth.make_cotangents(B, step=rank * 1000 + i)
        cots.append([c[0].to(dev), c[1].reshape(B, 512).to(dev), c[2].to(dev), c[3].to(dev)])
    text_cls = synth.make_text_class_features(20)[:C].contiguous().to(dev)
    # N > 1: the gradient buffer lives in symmetric memory and is summed over the ranks by ONE kernel over NVLink
    # peer memory, captured at the end of the step's graph (--comm nccl: torch.distributed all-reduce after the replay)
    peer, comm = None, (a.comm if world > 1 else None)
    if world > 1 and a.comm == "peer":
        from team_b200 import parallel
        try:
            peer = parallel.PeerAllReduce(head.HeadStepRunner.grad_numel(pack), dev)
        except Exception as e:                    # no symmetric memory on this box: every rank falls back together
            print(f"[bench] rank {rank}: peer all-reduce unavailable ({e}); using NCCL", file=sys.stderr, flush=True)
        ok = torch.tensor([0 if peer is None else 1], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            peer, comm = None, "nccl (peer-memory all-reduce unavailable)"
    runner = head.HeadStepRunner(pack, protos, B, C, mode, grad_events=comm == "nccl-buckets", peer=peer)
    stream = torch.cuda.Stream(device=dev)

    def eager_step(i):
        j = i % rot
        runner.step(imgs[j], txts[j], sids[j], text_cls, cots[j])

    # launches per step (counted by the library itself)
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        eager_step(0)
        c0 = L.team_launch_count()
        eager_step(1)
        launches_per_step = L.team_launch_count() - c0
    torch.cuda.synchronize()

    graphs = None
    if not a.no_graph:
        graphs = []
        with torch.cuda.stream(stream):
            for j in range(rot):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream):
                    runner.step(imgs[j], txts[j], sids[j], text_cls, cots[j])      # N > 1: the exchange is inside the backward
                graphs.append(g)
        torch.cuda.synchronize()

    def step(i):
        if graphs is not None:
            graphs[i % rot].replay()
        else:
            eager_step(i)
        if world > 1 and peer is None:
            runner.allreduce_grads()                  # NCCL: the only per-step collective

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        for i in range(warmup):
            step(i)
        barrier()
        # nvidia-smi needs a few hundred ms before its first sample: keep the same load running (extra
        # untimed warm-up steps) so that the samples are taken under load
        def load(seconds):            # keep the GPU under the step's load; the SAME replay count on every rank
            t_w = time.perf_counter()         # (the peer all-reduce inside the graphs is a collective)
            for j in range(20):
                step(j)
            torch.cuda.synchronize()
            n = torch.tensor([max(1, int(seconds / max((time.perf_counter() - t_w) / 20, 2e-5)))], device=dev)
            if world > 1:
                dist.broadcast(n, 0)
            for j in range(int(n.item())):
                step(j)
            torch.cuda.synchronize()
        load(1.0)
        if rank == 0:
            sampler.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for i in range(a.steps):
            step(warmup + i)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        dump = last_step_outputs(runner) if a.dump_outputs and rank == 0 else None
        # the timed region of K steps can be shorter than one nvidia-smi period: keep replaying the same
        # steps (untimed) for 0.3 s so that the sampler sees the load the timed region ran under
        load(0.3)
        clocks = sampler.stop() if rank == 0 else None
        if clocks is not None:
            clocks["window"] = "timed region + 0.3 s of the same replayed steps (25 ms nvidia-smi period)"
    if dump is not None:
        write_outputs(dump, a.dump_outputs)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / a.steps
    value = world * B * a.steps / (ms / 1e3)

    # ---- roofline of the dominant kernel: CUDA events around every launch of the GEMM kernels, K extra eager steps
    pk = peaks()
    roof = None
    kind = 1 if mode == head.MODE_BF16 else 0
    nprof = min(a.steps, 10)
    tms, tfl, tby, nl = ctypes.c_double(), ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
    with torch.cuda.stream(stream):
        stats = {}
        for k in (1, 0):
            L.team_prof_enable(1)
            for i in range(nprof):
                eager_step(warmup + a.steps + i)
            L.team_prof_enable(0)
            capi.check(L.team_prof_collect(k, ctypes.byref(tms), ctypes.byref(tfl), ctypes.byref(tby), ctypes.byref(nl)),
                       "team_prof_collect")
            stats[k] = (tms.value, tfl.value, tby.value, nl.value)
    dom = kind if stats[kind][3] > 0 else 0
    dms, dfl, dby, dn = stats[dom]
    if dn > 0 and dms > 0:
        ach = dfl / (dms * 1e-3) / 1e12
        peak = pk["tensor_sustained"]
        traffic, traffic_src = ncu_dram_bytes_per_launch("gemm_bf16_tcgen05") if dom == 1 else (None, None)
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": dby / dn,
                "kernel": "gemm_bf16_tcgen05_kernel" if dom == 1 else "gemm_f32_kernel (fp32 FFMA; no tensor pipe)",
                "launches_timed": dn, "avg_launch_us": dms * 1e3 / dn,
                "share_of_step": (dms / nprof) / ms_per_step,
                "algorithmic_flops_per_launch": dfl / dn,
                "peak_source": f"bf16 dense sustained, {pk['src']}",
                "how": f"CUDA events around each launch of the kernel on the launching stream, {nprof} extra eager steps "
                       "after the timed region"}

    # ---- the same kernel INSIDE a graph replay: in-kernel globaltimer stamps (team_gemm_debug_stamps) of a graph captured
    # with the stamp buffer attached.  Span of a launch = first CTA past its dependency wait -> last CTA done, i.e. without the
    # launch latency and the broken PDL overlap that the event pair around an eager launch adds.  These are the `roofline`
    # numbers; the event-pair numbers stay beside them (`eager_events`).
    if roof is not None and dom == 1 and graphs is not None:
        try:
            L.team_gemm_debug_stamps.argtypes = [ctypes.c_void_p]
            dbg = torch.zeros((32, 1024, 16), dtype=torch.int64, device=dev)
            with torch.cuda.stream(stream):
                L.team_gemm_debug_stamps(dbg.data_ptr())
                gs = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gs, stream=stream):
                    runner.step(imgs[0], txts[0], sids[0], text_cls, cots[0])
                L.team_gemm_debug_stamps(None)
                spans = []
                for rep in range(5):
                    for j in range(3):
                        step(j + 1)                     # ordinary replays around it, as in the timed region
                    dbg.zero_()
                    gs.replay()
                    torch.cuda.synchronize()
                    dcpu = dbg.cpu()
                    for l in range(32):
                        x = dcpu[l]
                        x = x[(x[:, 7] > 0) & (x[:, 2] > 0)]          # CTAs that ran a tile (cluster padding CTAs leave no end stamp)
                        if x.shape[0]:
                            spans.append(float(int(x[:, 7].max()) - int(x[:, 2].min())) * 1e-3)
                del gs
            if spans:
                us = sum(spans) / len(spans)
                fl = roof["algorithmic_flops_per_launch"]
                # The launch duration INSIDE the timed graph is the roofline's denominator.  The event pair around an eager launch
                # (kept under `eager_events`) also times the launch latency and loses the PDL overlap: its share of the step (0.8)
                # contradicts the ncu launch list (GEMM launches = 0.47 of the summed launch durations), the in-graph share agrees.
                roof["eager_events"] = {k: roof[k] for k in ("achieved", "frac", "avg_launch_us", "share_of_step", "launches_timed", "how")}
                roof.update({"avg_launch_us": us, "launches_timed": len(spans), "achieved": fl / us / 1e6, "frac": fl / us / 1e6 / roof["peak"],
                             "share_of_step": us * (len(spans) / 5) / 1e3 / ms_per_step,
                             "how": "launch duration inside the replayed step graph (the timed region's own graphs): in-kernel globaltimer "
                                    "stamps, first CTA past griddepcontrol.wait -> last CTA done, mean over the GEMM launches of 5 replays "
                                    "among ordinary replays; `eager_events` = CUDA events around each eager launch of the same kernel"})
        except Exception as exc:
            roof["in_graph_error"] = str(exc)[:200]

    # ---- end to end through the public API (head.HostBatchPipeline): every step copies its batch from pinned
    # host memory (copy stream, double-buffered), replays the fwd+bwd graph, all-reduces the gradient bucket
    # (N > 1) and copies the step's predictions back to the host, where they are compared with the labels
    e2e = None
    if not a.no_e2e:
        nrot = min(rot, 16)
        h_img = [imgs[j].cpu().pin_memory() for j in range(nrot)]
        h_txt = [txts[j].cpu().pin_memory() for j in range(nrot)]
        h_sid = [sids[j].cpu().pin_memory() for j in range(nrot)]
        h_lab = [synth.make_batch(B, C, step=rank * 1000 + j)["label"] for j in range(nrot)]
        after = (lambda r: r.allreduce_grads()) if world > 1 and peer is None else None
        peer2 = parallel.PeerAllReduce(head.HeadStepRunner.grad_numel(pack), dev) if peer is not None else None
        pipe = head.HostBatchPipeline(pack, protos, B, text_cls, mode=mode, depth=2, after_step=after,
                                      grad_events=comm == "nccl-buckets",
                                      peer=peer2)
        correct = [0]

        def e2e_step(i):
            j = i % nrot
            pred = pipe.submit(h_img[j], h_txt[j], h_sid[j], cots[j])
            if pred is not None:
                correct[0] += int((pred == h_lab[(i - 1) % nrot]).sum())      # host-side metric on the D2H result

        for i in range(4):
            e2e_step(i)
        pipe.drain()
        barrier()
        ksteps = a.steps
        t0 = time.perf_counter()
        for i in range(ksteps):
            e2e_step(4 + i)
        pipe.drain()
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        e2e = {"value": world * B * ksteps / dt, "unit": UNIT,
               "h2d_bytes_per_step": pipe.h2d_bytes_per_step, "d2h_bytes_per_step": pipe.d2h_bytes_per_step,
               "steps": ksteps, "ms_per_step": dt / ksteps * 1e3,
               "api": "team_b200.head.HostBatchPipeline.submit: pinned host image/text/state batch -> H2D on a copy "
                      "stream (2 slots) -> graph replay of fwd+bwd -> D2H of the predictions; wall clock over all steps "
                      "incl. drain; cotangents device-resident (the loss is the caller's)"}

    # ---- N > 1: (i) untimed check that the in-graph peer exchange leaves the SUM of the per-rank gradients in every
    # rank's buffer (against an NCCL all-reduce of gradients computed without the exchange); (ii) the strong-scaling
    # point of BASELINE configs[3]: 4096 samples in total, split over the GPUs, same graph-replayed step.
    grad_check, strong = None, None
    if world > 1:
        try:
            with torch.cuda.stream(stream):
                local = head.HeadStepRunner(pack, protos, B, C, mode)
                local.step(imgs[0], txts[0], sids[0], text_cls, cots[0])
                want = local.flat_grads.clone()
                dist.all_reduce(want)
                mine = local.flat_grads.clone()
                eager_step(0)                                   # the runner of the timed region (exchange inside the backward)
                if peer is None:
                    runner.allreduce_grads()
                torch.cuda.synchronize()
                got = runner.flat_grads
                err = float((got.double() - want.double()).norm() / want.double().norm().clamp_min(1e-30))
                changed = float((got.double() - mine.double()).norm() / want.double().norm().clamp_min(1e-30))
                worst = torch.tensor([err], device=dev)
                dist.all_reduce(worst, op=dist.ReduceOp.MAX)
                same = got.clone()
                dist.broadcast(same, 0)
                ident = torch.tensor([1 if torch.equal(same, got) else 0], device=dev)
                dist.all_reduce(ident, op=dist.ReduceOp.MIN)
                grad_check = {"ok": bool(float(worst.item()) <= 1e-5), "max_rel_err_over_ranks": float(worst.item()), "tolerance": 1e-5,
                              "bit_identical_on_all_ranks": bool(int(ident.item())),
                              "rel_change_vs_local_gradient": changed,
                              "what": "flat gradient buffer after one step with the exchange vs NCCL all-reduce(sum) of the per-rank "
                                      "gradients of the same step computed without it (norm-wise relative, fp32)"}
                del local
        except Exception as exc:
            grad_check = {"ok": False, "error": str(exc)[:300]}
        try:
            if a.scaling == "weak" and a.global_batch % world == 0 and a.global_batch // world >= 8:
                Bs = a.global_batch // world
                peer_s = parallel.PeerAllReduce(head.HeadStepRunner.grad_numel(pack), dev) if peer is not None else None
                rs = head.HeadStepRunner(pack, protos, Bs, C, mode, peer=peer_s)
                nset = min(rot, 32)
                sets = []
                for i in range(nset):
                    bb = synth.make_batch(Bs, C, step=5000 + rank * 1000 + i)
                    cc = synth.make_cotangents(Bs, step=5000 + rank * 1000 + i)
                    sets.append((bb["image"].to(dev), bb["text"].to(dev), bb["state"].to(dev),
                                 [cc[0].to(dev), cc[1].reshape(Bs, 512).to(dev), cc[2].to(dev), cc[3].to(dev)]))
                with torch.cuda.stream(stream):
                    rs.step(sets[0][0], sets[0][1], sets[0][2], text_cls, sets[0][3])
                    torch.cuda.synchronize()
                    gs = []
                    for q in sets:
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g, stream=stream):
                            rs.step(q[0], q[1], q[2], text_cls, q[3])
                        gs.append(g)

                    def sstep(i):
                        gs[i % nset].replay()
                        if peer_s is None:
                            rs.allreduce_grads()
                    for i in range(warmup):
                        sstep(i)
                    barrier()
                    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s0.record(stream)
                    for i in range(a.steps):
                        sstep(warmup + i)
                    s1.record(stream)
                    barrier()
                    sms = torch.tensor([s0.elapsed_time(s1)], device=dev)
                    dist.all_reduce(sms, op=dist.ReduceOp.MAX)
                sms = float(sms.item()) / a.steps
                strong = {"scaling": "strong", "global_batch": a.global_batch, "batch_per_gpu": Bs, "ms_per_step": sms,
                          "samples_per_s": a.global_batch / sms * 1e3,
                          "timing": f"CUDA events, {a.steps} graph replays, max over ranks, {nset} rotating input sets"}
                del rs, gs, sets
        except Exception as exc:
            strong = {"error": str(exc)[:300]}

    # ---- the same step at larger per-GPU batches (BASELINE configs[4] sweep), N = 1 only: where the launch-latency
    # floor of the 26-launch chain no longer hides the kernels, i.e. what the kernels themselves sustain
    at_scale = None
    if world == 1 and not a.no_scale:
        at_scale = []
        for Bs in (256, 4096, 16384, 65536):         # BASELINE configs[4]: 256 ... 65 536 (1 024 is the headline itself)
            try:
                gen = torch.Generator(device="cpu").manual_seed(Bs)
                sets = []
                for i in range(2 if Bs > 4096 else (8 if Bs >= 4096 else 64)):
                    si = torch.nn.functional.normalize(torch.randn(Bs, 512, generator=gen), dim=-1).to(dev)
                    stx = torch.nn.functional.normalize(torch.randn(Bs, 512, generator=gen), dim=-1).to(dev)
                    ss = torch.tensor([1, 3, 4])[torch.randint(0, 3, (Bs,), generator=gen)].to(dev)
                    sets.append((si, stx, ss, [torch.randn(Bs, 512, generator=gen).to(dev) for _ in range(4)]))
                rs = head.HeadStepRunner(pack, protos, Bs, C, mode)
                with torch.cuda.stream(stream):
                    for i in range(3):
                        q = sets[i % len(sets)]
                        rs.step(q[0], q[1], q[2], text_cls, q[3])
                    torch.cuda.synchronize()
                    k = 10
                    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    ev0.record(stream)
                    for i in range(k):
                        q = sets[i % len(sets)]
                        rs.step(q[0], q[1], q[2], text_cls, q[3])
                    ev1.record(stream)
                    torch.cuda.synchronize()
                    msb = ev0.elapsed_time(ev1) / k
                    L.team_prof_enable(1)
                    for i in range(2):
                        q = sets[i % len(sets)]
                        rs.step(q[0], q[1], q[2], text_cls, q[3])
                    L.team_prof_enable(0)
                    capi.check(L.team_prof_collect(kind, ctypes.byref(tms), ctypes.byref(tfl), ctypes.byref(tby), ctypes.byref(nl)), "team_prof_collect")
                falg = 55.07e6 * Bs + 0.47e9
                at_scale.append({"batch_per_gpu": Bs, "ms_per_step": msb, "samples_per_s": Bs / msb * 1e3,
                                 "alg_tflops": falg / msb / 1e9, "frac_of_tensor_peak": falg / msb / 1e9 / pk["tensor_sustained"],
                                 "gemm_tflops": tfl.value / max(tms.value, 1e-9) / 1e9,
                                 "gemm_frac_of_tensor_peak": tfl.value / max(tms.value, 1e-9) / 1e9 / pk["tensor_sustained"],
                                 "gemm_share_of_step": tms.value / 2 / msb, "timing": f"CUDA events, {k} eager steps, "
                                 f"{len(sets)} rotating input sets ({len(sets) * Bs * 512 * 4 * 6 / 2**20:.0f} MiB)"})
                del rs, sets
                torch.cuda.empty_cache()
            except Exception as exc:      # an extra point must never cost the headline line
                at_scale.append({"batch_per_gpu": Bs, "error": str(exc)[:200]})
                torch.cuda.empty_cache()

    # ---- the COMPLETE training step of the learner's loop body (models/proof.py:403-451 after the frozen towers):
    # logits + forward_tri_modal + ClipLoss branch + unicl_loss with evolution features + backward + fused AdamW,
    # captured as one CUDA graph (team_b200.train.TrainStep), N = 1.  Device-resident batches (value) and host
    # batches through load() with the losses read back every step (e2e).
    train_step = None
    if world == 1 and not a.no_e2e:
        try:
            from team_b200 import train
            ptrain = {k: v.clone() for k, v in pdev.items()}
            gen = torch.Generator().manual_seed(5)
            evo = [torch.randn(512, generator=gen) for _ in range(C)]
            ts = train.TrainStep(ptrain, protos, B, text_cls, mode=mode, evolution_features=evo)
            nrot = min(rot, 16)
            labs = [synth.make_batch(B, C, step=rank * 1000 + j)["label"].to(dev) for j in range(nrot)]
            with torch.cuda.stream(stream):
                for i in range(3):
                    ts.load(imgs[i], txts[i], sids[i], labs[i]); ts.step(epoch=0)
                torch.cuda.synchronize()
                c0 = L.team_launch_count()
                ts._body(0)                                   # one eager pass only to count the library launches
                tl = L.team_launch_count() - c0
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record(stream)
                for i in range(a.steps):
                    j = i % nrot
                    ts.load(imgs[j], txts[j], sids[j], labs[j]); ts.step(epoch=0)
                ev1.record(stream)
                torch.cuda.synchronize()
                tms_dev = ev0.elapsed_time(ev1) / a.steps
                h = [(imgs[j].cpu().pin_memory(), txts[j].cpu().pin_memory(), sids[j].cpu().pin_memory(), labs[j].cpu().pin_memory())
                     for j in range(nrot)]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                last = None
                for i in range(a.steps):
                    ts.load(*h[i % nrot])
                    lossv = ts.step(epoch=0).cpu()            # D2H of the step's losses (and the sync a logging loop has)
                    last = lossv
                dt = time.perf_counter() - t0
            train_step = {"what": "cls logits + forward_tri_modal + ClipLoss on the head's own normalised rows (gradient joins the head "
                                  "backward: team_head_grads.g_own_rows) + unicl_loss (evolution features) + backward + fused AdamW "
                                  "as one CUDA graph (team_b200.train.TrainStep)",
                          "batch": B, "ms_per_step": tms_dev, "samples_per_s": B / tms_dev * 1e3, "library_launches_per_step": int(tl),
                          "e2e": {"ms_per_step": dt / a.steps * 1e3, "samples_per_s": B * a.steps / dt,
                                  "h2d_bytes_per_step": B * (512 * 4 * 2 + 16), "d2h_bytes_per_step": 20,
                                  "api": "TrainStep.load(pinned host batch) + step() + losses.cpu() every step"},
                          "last_losses": [float(v) for v in last]}
            del ts
        except Exception as exc:
            train_step = {"error": str(exc)[:300]}

    # ---- BASELINE configs[1]: SimpleCIL prototype build (keyed segmented sum) + cosine classifier at 4 M rows (8.6 GB of
    # fp32 features, far beyond L2) against the measured HBM copy peak; N = 1.  Algorithmic bytes per row: 512 e + 8 (label)
    # [+ 8 (state)] for the build, 512 e + 4 C + 8 for logits + argmax (SURVEY 8d).
    proto_build = None
    if world == 1 and not a.no_scale:
        try:
            from team_b200 import ops
            Np = 4 * 1024 * 1024
            gdev = torch.Generator(device=dev).manual_seed(0)
            proto_build = {"rows": Np, "hbm_peak_gbs": pk["hbm"], "peak_source": pk["src"], "timing": "CUDA events, 5 launches after a warm-up launch"}
            for name, dt, e in (("fp32", torch.float32, 4), ("bf16", torch.bfloat16, 2)):
                xr = torch.randn((Np, 512), generator=gdev, device=dev, dtype=torch.float32).to(dt)
                yr = torch.randint(0, 20, (Np,), generator=gdev, device=dev)
                sr = torch.randint(0, 10, (Np,), generator=gdev, device=dev)
                Wr = torch.randn((20, 512), generator=gdev, device=dev)

                def timed(fn, iters=5):
                    fn(); torch.cuda.synchronize()
                    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    q0.record()
                    for _ in range(iters):
                        fn()
                    q1.record(); torch.cuda.synchronize()
                    return q0.elapsed_time(q1) / iters

                for key, fn, by in ((f"segsum_class_{name}", lambda: ops.keyed_sums(xr, yr, num_classes=20), 512 * e + 8),
                                    (f"segsum_class_state_{name}", lambda: ops.keyed_sums(xr, yr, sr, num_classes=20), 512 * e + 16),
                                    (f"cosine_logits_argmax_{name}", lambda: ops.cosine_logits(xr, Wr, want_argmax=True), 512 * e + 88)):
                    msq = timed(fn)
                    proto_build[key] = {"ms": msq, "rows_per_s": Np / msq * 1e3, "gbs": Np * by / msq / 1e6,
                                        "frac_of_hbm_peak": Np * by / msq / 1e6 / pk["hbm"], "bytes_per_row": by}
                del xr
                torch.cuda.empty_cache()
        except Exception as exc:
            proto_build = {"error": str(exc)[:300]}
            torch.cuda.empty_cache()

    # ---- N > 1 (BASELINE configs[4]): the prototype build data-parallel - every rank sums its own shard of rows (4 M fp32 rows
    # per GPU: weak scaling), then the two collectives of the path on it: NCCL all-reduce of the [K,512] sums and the int64 counts
    # (parallel.allreduce_prototype_sums), then the means.  Max over ranks of the CUDA-event time, aggregate rows/s; counts checked.
    proto_dp = None
    if world > 1 and not a.no_scale:
        try:
            from team_b200 import ops, parallel
            Np = 4 * 1024 * 1024
            gdev = torch.Generator(device=dev).manual_seed(100 + rank)
            xr = torch.randn((Np, 512), generator=gdev, device=dev, dtype=torch.float32)
            yr = torch.randint(0, 20, (Np,), generator=gdev, device=dev)
            sr = torch.randint(0, 10, (Np,), generator=gdev, device=dev)
            proto_dp = {"rows_per_gpu": Np, "rows_total": Np * world, "hbm_peak_gbs_per_gpu": pk["hbm"]}
            for key, st_, K_ in (("class_keys", None, 20), ("class_state_keys", sr, 200)):
                def build():
                    sums, counts = ops.keyed_sums(xr, yr, st_, num_classes=20)
                    parallel.allreduce_prototype_sums(sums, counts)
                    return ops.keyed_means(sums, counts), counts
                _, counts = build()
                torch.cuda.synchronize(); dist.barrier()
                q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                q0.record()
                for _ in range(5):
                    build()
                q1.record(); torch.cuda.synchronize()
                tm = torch.tensor([q0.elapsed_time(q1) / 5], device=dev)
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                msq = float(tm.item())
                by = 2048 + (16 if st_ is not None else 8)
                proto_dp[key] = {"ms": msq, "rows_per_s": Np * world / msq * 1e3, "gbs_per_gpu": Np * by / msq / 1e6,
                                 "frac_of_hbm_peak": Np * by / msq / 1e6 / pk["hbm"], "keys": K_,
                                 "counts_exact": bool(int(counts.sum().item()) == Np * world)}
            del xr
            torch.cuda.empty_cache()
        except Exception as exc:
            proto_dp = {"error": str(exc)[:300]}
            torch.cuda.empty_cache()

    # ---- BASELINE configs[3] graph path: evolve_and_update (graph build on the host + temporal GCN + pairwise state
    # distances), evolve_state_prototypes (second GCN pass + prototype sync) and the state-distance EMA, wall clock with a
    # device sync per call (the learner calls them once per epoch, models/proof.py:463-513); native size (20 classes,
    # 46 nodes; the reference takes 1.24 s per evolve_and_update call on 8 host threads, SURVEY section 6) and scaled graphs.
    graph_path = None
    if world == 1 and not a.no_scale:
        try:
            from team_b200 import graph
            gp = {k: v.to(dev) for k, v in synth.make_params(2, seed=77).items()}
            graph_path = []
            for ncls in (20, 200, 2000):       # 46 / 466 / 4 666 nodes (the pairwise state distances are O(nodes^2): 57 s at 46 666)
                bs = synth.make_state_prototype_dict(ncls, seed=9)
                bs = {c: {s_: v.to(dev) for s_, v in sd.items()} for c, sd in bs.items()}
                protos_g = torch.zeros(ncls, 512, device=dev)
                nodes = sum(len(sd) for sd in bs.values())
                f = graph.prior_distance_factors(device=dev)

                def wall(fn, iters):
                    fn(); torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(iters):
                        fn()
                    torch.cuda.synchronize()
                    return (time.perf_counter() - t0) / iters * 1e3

                iters = 10 if ncls <= 200 else 2
                res_box = {}

                def ev():
                    res_box["r"] = graph.evolve_and_update(gp, bs, {})
                ms_ev = wall(ev, iters)
                ms_sync = wall(lambda: graph.evolve_state_prototypes(gp, protos_g, bs, {}), iters)
                ms_ema = wall(lambda: graph.update_state_distance_matrix(f, res_box["r"]["distances"]), iters)
                c0 = L.team_launch_count(); ev(); nl_ev = L.team_launch_count() - c0
                graph_path.append({"classes": ncls, "nodes": nodes, "evolve_and_update_ms": ms_ev, "evolve_state_prototypes_ms": ms_sync,
                                   "update_state_distance_matrix_ms": ms_ema, "library_launches_evolve_and_update": int(nl_ev)})
                del bs
        except Exception as exc:
            graph_path = {"error": str(exc)[:300]}

    cb = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cb, _, _ = time_cpu(T, B, 3, 1, budget_s=25.0)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
                "dtype": a.mode, "data": "synthetic",
                "config": workload_config(T, B, world),
                "run": {"grad_exchange": comm, "cuda_graphs": graphs is not None,
                        "l2": f"{rot} rotating input+cotangent sets ({rot * B * 512 * 4 * 6 / 2**20:.0f} MiB) larger than L2"},
                "roofline": roof, "at_scale": at_scale, "train_step": train_step, "proto_build": proto_build, "graph": graph_path, "cpu_baseline": cb, "clocks": clocks, "e2e": e2e,
                "grad_exchange_check": grad_check, "strong_scaling": strong, "proto_build_dp": proto_dp,
                "gpu_launches": int(launches_per_step) * a.steps,
                "survey_falg_tflops": value * 55.07e6 / 1e12 / world}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_team(a)


if __name__ == "__main__":
    main()
