"""The data-parallel training step on several GPUs of one box: one process per GPU (torch.multiprocessing.spawn, NCCL),
with W = 2 and with every GPU of the box up to 8.  Skipped with fewer than two GPUs.

  * team_peer_allgather (parallel.PeerAllGather): slices of 16 B, 24 KiB, 425 KiB and 3 088 x 1 024 B (exchange 0 at
    1 024 bf16 samples per rank) with NaN / infinity / -0 float patterns among random bytes equal
    dist.all_gather_into_tensor byte for byte on every rank, eagerly and inside one captured graph replayed three times
    with fresh slices; on the multicast path as well when the box maps it; status() is 0 after every run.
  * DataParallelTrainStep (captured graphs, three steps over two epochs, with and without evolution features): the bars
    of test_gpu_train_step_dp.py against the fp64 oracle (f32) and the single-GPU TrainStep at W * B (bf16: losses, the
    first step's gradients block by block, parameters), and
    losses6 and every trainable parameter bit-identical on all ranks after every step.
The workers use a 120 s peer deadline (TEAM_PEER_TIMEOUT_S) and destroy their process group."""
import os
import socket

import pytest
import torch

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more GPUs")]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, fn, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["TEAM_PEER_TIMEOUT_S"] = "120"
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        ret[rank] = fn(rank, world, dev)
    finally:
        dist.destroy_process_group()


def _run(fn, world):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    mgr = ctx.Manager()
    try:
        ret = mgr.dict()
        mp.spawn(_worker, args=(world, _free_port(), fn, ret), nprocs=world, join=True)
        return [ret[r] for r in range(world)]
    finally:
        mgr.shutdown()


def _worlds():
    n = min(torch.cuda.device_count(), 8)
    return sorted({2, n}) if n >= 2 else [2]


SIZES = [16, 24 * 1024, 425 * 1024, 3088 * 1024]


def _slice(n, rank, it):
    g = torch.Generator().manual_seed(7919 * it + 101 * rank + n)
    x = torch.randint(0, 256, (n,), generator=g, dtype=torch.uint8)
    f = x[:16].view(torch.float32)
    f.copy_(torch.tensor([float("nan"), float("inf"), float("-inf"), -0.0]))
    if n >= 4096:                                          # special floats further in as well
        x[1024:1040].view(torch.float32).copy_(torch.tensor([float("-inf"), float("nan"), 0.0, float("inf")]))
    return x


def _allgather_job(rank, world, dev):
    import torch.distributed as dist
    from team_b200 import parallel
    paths = []
    for mc in (False, True):
        ag = parallel.PeerAllGather(SIZES, dev, multicast=mc)
        if mc and not any(ag.multicast_ptrs):
            del ag
            continue
        paths.append(bool(any(ag.multicast_ptrs)))

        def check(it):
            for p, n in enumerate(SIZES):
                want = torch.empty(world * n, dtype=torch.uint8, device=dev)
                dist.all_gather_into_tensor(want, _slice(n, rank, it).to(dev))
                assert torch.equal(ag.gathered[p], want), (rank, p, n, it, mc)
        # eager
        for p, n in enumerate(SIZES):
            ag.send[p].copy_(_slice(n, rank, 0))
            ag(p)
        assert ag.status() == 0
        check(0)
        # one captured graph of the three exchanges, replayed with fresh slices
        st = torch.cuda.Stream(device=dev)
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                for p in range(len(SIZES)):
                    ag(p)
        torch.cuda.current_stream().wait_stream(st)
        for it in (1, 2, 3):
            for p, n in enumerate(SIZES):
                ag.send[p].copy_(_slice(n, rank, it))
            g.replay()
            assert ag.status() == 0
            check(it)
        del g, ag
        torch.cuda.synchronize()
    return paths


@pytest.mark.parametrize("world", _worlds())
def test_peer_allgather_equals_nccl(world):
    if world > torch.cuda.device_count():
        pytest.skip(f"needs {world} GPUs")
    paths = _run(_allgather_job, world)
    print(f"peer all-gather world={world}: paths {paths[0]} (True = multicast) byte-equal to NCCL on every rank")
    assert all(p == paths[0] for p in paths)


def _same_on_all_ranks(t):
    import torch.distributed as dist
    flat = t.detach().reshape(-1).contiguous()
    allv = torch.empty((dist.get_world_size(), flat.numel()), dtype=flat.dtype, device=flat.device)
    dist.all_gather_into_tensor(allv, flat)
    return all(torch.equal(allv[r], allv[0]) for r in range(allv.shape[0]))


def _dp_job(rank, world, dev):
    import test_gpu_train_step_dp as S
    from oracle import synth
    from oracle import team_oracle as O
    from team_b200 import head, train
    out = []
    for mode, T, B, C in ((head.MODE_F32, 3, 48, 6), (head.MODE_BF16, 10, 1024, 20)):
        for evo_on in (False, True):
            params, protos, text_cls, evo = S._setup(T, C, evo_on, seed=77 if mode == head.MODE_F32 else 42)
            names = O.trainable_names(params)
            batches = [synth.make_batch(world * B, C, step=s) for s in range(3)]
            pg = {k: v.clone().to(dev) for k, v in params.items()}
            dp = train.DataParallelTrainStep(pg, protos.to(dev), B, text_cls.to(dev), mode=mode, init_lr=S.LR0, min_lr=1e-8,
                                             weight_decay=S.WD, tuned_epoch=S.TUNED, logit_scale=S.LS, evolution_features=evo)
            assert (dp.rank, dp.world) == (rank, world)
            got, g_dp = [], None
            sh = slice(rank * B, (rank + 1) * B)
            for b, ep in zip(batches, S.EPOCHS):
                dp.load(b["image"][sh], b["text"][sh], b["state"][sh], b["label"][sh])
                got.append(dp.step(epoch=ep).clone())
                dp.check()
                if g_dp is None:                # the first step's gradients, summed over the ranks in the backward
                    g_dp = [g.detach().cpu().double() for _, g in dp.pairs]
                assert _same_on_all_ranks(dp.losses6), "losses6 differ between ranks"
                assert _same_on_all_ranks(torch.cat([p.detach().reshape(-1) for p, _ in dp.pairs])), "parameters differ between ranks"
            assert len(dp._graphs) == 2 and int(dp.opt.step_dev.cpu()) == 3
            got = [g.cpu().double().tolist() for g in got]
            res = None
            if rank == 0:
                if mode == head.MODE_F32:
                    ref_l, ref_p = S._oracle(params, protos, text_cls, evo, batches)
                    for g, r in zip(got, ref_l):
                        for a, b in zip(g, r):
                            assert abs(a - b) < 2e-5 * max(1.0, abs(b)), (got, ref_l)
                    e = S._param_errs(pg, ref_p, params, names)
                    assert max(e.values()) < 2e-3 + 1e-7, e
                    res = ("f32 vs oracle", evo_on, max(e.values()))
                else:
                    g_one = []
                    one_l, one_p = S._single(params, protos, text_cls, evo, batches, world * B, mode, grads=g_one)
                    eg = {k: float((a - b).norm() / b.norm().clamp_min(1e-30)) for k, a, b in zip(S.PAIR_NAMES, g_dp, g_one[0])}
                    assert max(eg.values()) <= 5e-3, eg
                    _, f32_p = S._single(params, protos, text_cls, evo, batches, world * B, head.MODE_F32)
                    lerr = max(abs(a - r) / max(abs(r), 1e-30) for g, w in zip(got, one_l) for a, r in zip(g, w))
                    e = S._param_errs(pg, {n: one_p[n].detach() for n in names}, params, names)
                    e_prec = S._param_errs({n: one_p[n].detach() for n in names}, {n: f32_p[n].detach() for n in names},
                                           params, names)
                    assert lerr <= 1e-4, (got, one_l)
                    assert max(e.values()) <= max(e_prec.values()) and max(e.values()) < 0.1, (e, e_prec)
                    res = ("bf16 vs TrainStep", evo_on, lerr, max(eg.values()), max(e.values()))
            out.append(res)
            del dp
            torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("world", _worlds())
def test_dp_train_step_on_several_gpus(world):
    if world > torch.cuda.device_count():
        pytest.skip(f"needs {world} GPUs")
    res = _run(_dp_job, world)
    print(f"DataParallelTrainStep world={world}: {res[0]}")
