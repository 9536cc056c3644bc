"""GPU parity of the data-parallel losses (team_loss_shard_*, ops.ShardedLosses) on ONE B200: W virtual ranks run the
phases in one process, each exchange is the concatenation of the ranks' send slices in rank order.  Every rank's
losses6 and the concatenation of the ranks' cotangents must equal one call of ops.unicl_loss / ops.clip_loss /
ops.ce_total on the global batch (the single-GPU entry points, same mode).
fp32 mode: <= 1e-5 relative, norm-wise.  bf16 mode: <= 1e-4 (values) / 5e-3 (cotangents), tighter than the bars of the bf16
losses against fp64 in test_gpu_losses.py (1e-2 / 2e-2): both sides round the same operands to bf16, only the summation
order differs.  Measured on a B200: fp32 values <= 1.2e-7,
cotangents <= 1.2e-6; bf16 values <= 7e-8, cotangents <= 5e-7.  The differences are printed (run with -s)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

SCALE = 14.285714


def rel(a, b):
    a = a.detach().double().cpu(); b = b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _inputs(W, B, seed):
    """Global batch of W * B samples.  Labels: random classes 0..5 spread over all ranks, sample 0 is the only one of
    class 9 (seen once in the global batch: no positives, single-sample evolution), samples 1 and 2 of rank 0 are the
    only ones of class 10 (a class on one rank only), the last sample is class 11 (beyond the evolution list)."""
    Bg = W * B
    g = torch.Generator().manual_seed(seed)
    base = torch.randn((Bg, 512), generator=g)
    feats = [base + 0.7 * torch.randn((Bg, 512), generator=g) for _ in range(3)]
    own = torch.nn.functional.normalize(torch.randn((2, Bg, 512), generator=g) + base, dim=2)
    labels = torch.randint(0, 6, (Bg,), generator=g, dtype=torch.int64)
    states = torch.randint(0, 4, (Bg,), generator=g, dtype=torch.int64)
    labels[0] = 9
    if B >= 4:
        labels[1] = labels[2] = 10
        labels[-1] = 11
    logits = 3.0 * torch.randn((Bg, 12), generator=g)
    evo = [torch.randn(512, generator=g) for _ in range(11)]
    evo[1] = None
    dev = torch.device("cuda")
    return dict(image=feats[0].to(dev), text=feats[1].to(dev), state=feats[2].to(dev), own=own.to(dev),
                labels=labels.to(dev), states=states.to(dev), logits=logits.to(dev)), evo


def _global(x, evo, mode):
    from team_b200 import ops
    un, cots = ops.unicl_loss(x["image"], x["text"], x["state"], x["labels"], state_ids=x["states"], evolution_features=evo,
                              epoch=3, max_epoch=20, grad_scale=0.3, mode=mode)
    losses6 = torch.zeros(6, dtype=torch.float32, device=x["image"].device)
    losses6[3:6] = un
    _, g_own = ops.clip_loss(x["own"][0], x["own"][1], SCALE, mode=mode, loss_out=losses6[2:3])
    ops.ce_total(x["logits"], x["labels"], losses6, w_clip=1.0, w_unicl=0.3)
    return losses6, cots, g_own


def _sharded(x, evo, mode, W, B):
    from team_b200 import ops
    ranks = [ops.ShardedLosses(r, W, B, 12, evolution_features=evo, mode=mode) for r in range(W)]
    for s in ranks:          # all-ones bytes (NaN floats, -1 ints): every entry the next phase reads must be written
        for t in s.send + s.gathered:
            t.fill_(255)
    for r, s in enumerate(ranks):
        sh = slice(r * B, (r + 1) * B)
        s.bind(x["image"][sh].contiguous(), x["text"][sh].contiguous(), x["state"][sh].contiguous(),
               x["own"][:, sh].reshape(2 * B, 512).contiguous(), x["logits"][sh].contiguous(), x["labels"][sh].contiguous(),
               x["states"][sh].contiguous(), epoch=3, max_epoch=20, logit_scale=SCALE, w_clip=1.0, w_unicl=0.3)
    P = ranks[0].phases
    assert P == (4 if evo else 3)
    for p in range(P):
        for s in ranks:
            s.run(p)
        if p < P - 1:
            cat = torch.cat([s.send[p] for s in ranks])
            for s in ranks:
                s.gathered[p].copy_(cat)
    return ranks


def _compare(W, B, mode, evo_on, seed):
    from team_b200 import capi
    x, evo = _inputs(W, B, seed)
    evo = evo if evo_on else None
    ref6, cots, g_own = _global(x, evo, mode)
    ranks = _sharded(x, evo, mode, W, B)
    torch.cuda.synchronize()
    for s in ranks[1:]:
        assert torch.equal(s.losses6, ranks[0].losses6), "losses6 differ between ranks"
    got = {"losses6": ranks[0].losses6,
           "g_image": torch.cat([s.g_image for s in ranks]), "g_text": torch.cat([s.g_text for s in ranks]),
           "g_state": torch.cat([s.g_state for s in ranks]),
           "g_own_image": torch.cat([s.g_own[0] for s in ranks]), "g_own_text": torch.cat([s.g_own[1] for s in ranks])}
    want = {"losses6": ref6, "g_image": cots[0], "g_text": cots[1], "g_state": cots[2], "g_own_image": g_own[0],
            "g_own_text": g_own[1]}
    errs = {k: rel(got[k], want[k]) for k in got}
    tv, tg = (1e-5, 1e-5) if mode == capi.MODE_F32 else (1e-4, 5e-3)
    print(f"sharded losses W={W} B={B} mode={'f32' if mode == capi.MODE_F32 else 'bf16'} evo={evo_on}: "
          + " ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    for k, v in errs.items():
        assert v <= (tv if k == "losses6" else tg), (k, v, errs)
    return x


@pytest.mark.parametrize("W", [1, 2, 3, 4])
@pytest.mark.parametrize("B", [2, 37, 256, 1024])
def test_sharded_losses_equal_the_global_batch_f32(W, B):
    from team_b200 import capi
    for evo_on in (False, True):
        x = _compare(W, B, capi.MODE_F32, evo_on, seed=1000 + 10 * W + B)
    if W >= 2 and B >= 37:
        # a class with samples on several ranks in >= 2 life stages: its evolution mixture needs the global keyed sums
        y, st = x["labels"].cpu(), x["states"].cpu()
        split = [c for c in range(6) if len({int(v) // B for v in torch.nonzero(y == c)}) > 1 and len(set(st[y == c].tolist())) > 1]
        assert split


@pytest.mark.parametrize("W,B", [(1, 256), (2, 37), (3, 256), (4, 1024)])
def test_sharded_losses_equal_the_global_batch_bf16(W, B):
    from team_b200 import capi
    for evo_on in (False, True):
        _compare(W, B, capi.MODE_BF16, evo_on, seed=2000 + 10 * W + B)


def test_sharded_losses_reject_bad_shapes():
    from team_b200 import capi, ops
    with pytest.raises(ValueError):
        ops.ShardedLosses(0, 1, 1, 12)                     # a global batch of one
    s = ops.ShardedLosses(0, 2, 8, 12)
    z = torch.zeros((8, 512), device="cuda")
    with pytest.raises(ValueError):
        s.bind(z, z, z, torch.zeros((15, 512), device="cuda"), torch.zeros((8, 12), device="cuda"),
               torch.zeros(8, dtype=torch.int64, device="cuda"), logit_scale=SCALE)
    with pytest.raises(ValueError):                          # logits on the host
        s.bind(z, z, z, torch.zeros((16, 512), device="cuda"), torch.zeros((8, 12)),
               torch.zeros(8, dtype=torch.int64, device="cuda"), logit_scale=SCALE)
    with pytest.raises(capi.TeamB200Error):
        s.bind(z, z, z, torch.zeros((16, 512), device="cuda"), torch.zeros((8, 12), device="cuda"),
               torch.zeros(8, dtype=torch.int64, device="cuda"), logit_scale=SCALE)
        s.run(3)                                             # three phases without evolution features
