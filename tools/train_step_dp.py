"""Data-parallel training step (team_b200.train.DataParallelTrainStep) on N GPUs of one box, one JSON line:

    torchrun --nproc-per-node N tools/train_step_dp.py [--steps 200] [--out profiles/train_step_dp_nN.json]

Configuration of bench.py's train_step: B = 1 024 samples per GPU, bf16, T = 10 tasks, C = 20 classes, P = 100 prompts,
evolution features for the 20 classes.  Reported:
  * step: ms per replay of the captured step (CUDA events around >= 200 replays, each after a device-to-device load of
    one of 40 rotating device-resident batches per rank, 160 MiB > the 126 MB L2), the max over ranks and the global
    samples/s;
  * single_gpu: TrainStep at 1 024 samples, same timing, on every rank in the same call (max over ranks);
  * exchanges (N > 1): each of the step's all-gathers alone, team_peer_allgather (a captured graph of 20 calls) against
    NCCL all_gather_into_tensor (20 eager calls) at the same sizes, max over ranks;
  * the GPU's name and power limit, read in the same call."""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from team_b200 import capi, head, parallel, train   # noqa: E402
from oracle import synth                             # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--warmup", type=int, default=20)
ap.add_argument("--out", default=None)
a = ap.parse_args()

local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
rank, world = dist.get_rank(), dist.get_world_size()
capi.require_device()
B, T, C, NROT = 1024, 10, 20, 40
mode = head.MODE_BF16
params = synth.make_params(T, seed=42, perturb_ln=False)
protos = synth.make_prototypes(C).to(dev)
text_cls = synth.make_text_class_features(20)[:C].contiguous().to(dev)
gen = torch.Generator().manual_seed(5)
evo = [torch.randn(512, generator=gen) for _ in range(C)]
sets = []
for j in range(NROT):
    b = synth.make_batch(B, C, step=rank * 1000 + j)
    sets.append([b["image"].to(dev), b["text"].to(dev), b["state"].to(dev), b["label"].to(dev)])


def time_step(ts, steps):
    st = torch.cuda.Stream(device=dev)
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        for i in range(a.warmup):
            ts.load(*sets[i % NROT]); ts.step(epoch=0)
        st.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for i in range(steps):
            ts.load(*sets[i % NROT]); ts.step(epoch=0)
        e1.record(st)
        st.synchronize()
    return e0.elapsed_time(e1) / steps


def max_over_ranks(x):
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


dp = train.DataParallelTrainStep({k: v.clone().to(dev) for k, v in params.items()}, protos, B, text_cls, mode=mode,
                                 evolution_features=evo)
ms = max_over_ranks(time_step(dp, a.steps))
dp.check()
losses = [float(v) for v in dp.losses.cpu()]
xchg = list(dp.sl.xchg_bytes)
multicast = bool(dp.gather is not None and any(dp.gather.multicast_ptrs))
del dp
torch.cuda.empty_cache()

# every rank times its own single-GPU TrainStep, so all ranks issue the same collectives in the same order
ts = train.TrainStep({k: v.clone().to(dev) for k, v in params.items()}, protos, B, text_cls, mode=mode,
                     evolution_features=evo)
ms1 = max_over_ranks(time_step(ts, a.steps))
single = {"batch": B, "ms_per_step": ms1, "samples_per_s": B / ms1 * 1e3}
del ts
torch.cuda.empty_cache()

exchanges = None
if world > 1:
    ag = parallel.PeerAllGather(xchg, dev)
    exchanges = []
    st = torch.cuda.Stream(device=dev)
    for p, n in enumerate(xchg):
        with torch.cuda.stream(st):
            ag(p); st.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                for _ in range(20):
                    ag(p)
            g.replay(); st.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st); g.replay(); e1.record(st); st.synchronize()
            t_peer = e0.elapsed_time(e1) / 20 * 1e3
            send = torch.zeros(n, dtype=torch.uint8, device=dev)
            out = torch.empty(world * n, dtype=torch.uint8, device=dev)
            for _ in range(3):
                dist.all_gather_into_tensor(out, send)
            torch.cuda.synchronize(); dist.barrier()
            e0.record(st)
            for _ in range(20):
                dist.all_gather_into_tensor(out, send)
            e1.record(st); st.synchronize()
            t_nccl = e0.elapsed_time(e1) / 20 * 1e3
        exchanges.append({"exchange": p, "slice_bytes": n, "peer_us": max_over_ranks(t_peer), "nccl_us": max_over_ranks(t_nccl)})
    ag.check()
    del ag

gpu = torch.cuda.get_device_name(dev)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", f"--id={local}"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as exc:
    power = f"unavailable ({exc.__class__.__name__})"
if rank == 0:
    res = {"what": "DataParallelTrainStep: cls logits + forward_tri_modal + sharded ClipLoss / unicl_loss (evolution features) "
                   "with peer all-gathers + backward with the peer gradient all-reduce + fused AdamW, one CUDA graph per rank",
           "gpus": world, "gpu": gpu, "power_limit": power, "mode": "bf16", "batch_per_gpu": B, "tasks": T, "classes": C,
           "prompts": T * 10, "global_batch": world * B, "ms_per_step": ms, "samples_per_s": world * B / ms * 1e3,
           "multicast": multicast, "xchg_bytes": xchg, "exchanges": exchanges, "single_gpu": single,
           "speedup_vs_single_gpu": (world * B / ms) / single["samples_per_s"] * 1e3 if single else None,
           "timing": f"CUDA events around {a.steps} replays after {a.warmup} warm-up replays, {NROT} rotating device-resident "
                     f"batches per rank ({NROT * B * 512 * 4 * 2 / 2**20:.0f} MiB); max over ranks",
           "last_losses": losses}
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
dist.destroy_process_group()
