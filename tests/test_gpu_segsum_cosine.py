"""GPU parity: prototype build (keyed segmented sum) and cosine classifier through the C ABI
against the CPU oracle and the reference-generated golden vectors.
Bar: counts and argmax exact; sums/means/logits <= 1e-5 relative (fp32)."""
import numpy as np
import pytest
import torch

from oracle import synth
from oracle import team_oracle as O
from oracle.cases import CASES, case_inputs

pytestmark = pytest.mark.gpu


def rel(a, b):
    a = a.detach().double().cpu(); b = torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def test_cal_prototype_vs_golden(golden):
    from team_b200 import ops
    case, g = CASES["cal_prototype"], golden("cal_prototype")
    ci = case_inputs(case)
    C, known = case["num_classes"], case["known"]
    x = ci["x"].cuda()      # raw features; normalisation fused (encode_image(normalize=True))
    sums, counts = ops.keyed_sums(x, ci["y"].cuda(), ci["s"].cuda(), class_base=known,
                                  num_classes=C - known, num_states=10, normalize_rows=True)
    protos = torch.zeros(C, 512, device="cuda")
    by_state = torch.zeros((C - known) * 10, 512, device="cuda")
    _, _, ccounts = ops.keyed_means(sums, counts, out=by_state, group=10, class_out=protos[known:])
    assert rel(protos, g["img_prototypes"]) < 1e-5
    y, s = ci["y"], ci["s"]
    for c in range(known, C):
        assert int(ccounts[c - known]) == int((y == c).sum())
        for st in range(10):
            assert int(counts[(c - known) * 10 + st]) == int(((y == c) & (s == st)).sum())
    keys = [tuple(k) for k in g["by_state_keys"].tolist()]
    got = torch.stack([by_state[(c - known) * 10 + st] for c, st in keys])
    assert rel(got, g["by_state_vals"]) < 1e-5
    nz = {(c, st) for c in range(known, C) for st in range(10) if int(counts[(c - known) * 10 + st]) > 0}
    assert nz == set(keys)
    assert float(protos[case["empty_class"]].abs().sum()) == 0.0


def test_simplecil_vs_golden(golden):
    from team_b200 import ops
    case, g = CASES["simplecil"], golden("simplecil")
    ci = case_inputs(case)
    x = ci["x"].cuda()
    sums, counts = ops.keyed_sums(x, ci["y"].cuda(), num_classes=case["num_classes"])
    W = ops.keyed_means(sums, counts)
    assert rel(W, g["fc_weight"]) < 1e-5
    logits, am = ops.cosine_logits(x[:64], W, torch.ones(1), want_argmax=True)
    assert rel(logits, g["logits64"]) < 1e-5
    assert np.array_equal(am.cpu().numpy(), g["logits64"].argmax(1))


def test_cosine_linear_vs_golden(golden):
    from team_b200 import ops
    case, g = CASES["cosine_linear"], golden("cosine_linear")
    ci = case_inputs(case)
    logits, am = ops.cosine_logits(ci["x"].cuda(), ci["weight"].cuda(), torch.tensor([case["sigma"]]),
                                   want_argmax=True)
    assert rel(logits, g["logits"]) < 1e-5
    assert np.array_equal(am.cpu().numpy(), g["argmax"])


@pytest.mark.parametrize("n,C,zipf,norm,dtype", [
    (1, 3, False, False, torch.float32), (7, 2, False, True, torch.float32),
    (4099, 20, True, False, torch.float32), (65536, 20, False, True, torch.float32),
    (30001, 20, True, False, torch.bfloat16), (5000, 70, False, False, torch.float32),
    (70001, 20, True, False, torch.bfloat16), (66000, 6, False, True, torch.bfloat16),      # bf16 rows, few keys: key-partitioned path
    (3000, 50, False, False, torch.float32), (2500, 30, True, True, torch.float32),          # first generation below 4 096 rows: K > 400; K > 100 normalised
    (20000, 170, True, False, torch.bfloat16),                                               # first generation: K >= 1 600 keys
])
def test_keyed_sums_vs_oracle(n, C, zipf, norm, dtype):
    from team_b200 import ops
    x, y, s = synth.make_prototype_build_inputs(n, C, seed=77 + n, normalize=False, zipf=zipf,
                                                empty_class=1 if C > 2 else None)
    xq = x.to(dtype)
    sums, counts = ops.keyed_sums(xq.cuda(), y.cuda(), s.cuda(), num_classes=C, num_states=10,
                                  normalize_rows=norm)
    xe = xq.double()
    if norm:
        xe = torch.nn.functional.normalize(xq.float(), dim=-1).double()
    key = y * 10 + s
    ref = torch.zeros(C * 10, 512, dtype=torch.float64).index_add_(0, key, xe)
    cref = torch.bincount(key, minlength=C * 10)
    assert torch.equal(counts.cpu(), cref)
    assert rel(sums, ref) < 1e-5
    # class-only keys + oracle means (reference loop)
    sums_c, counts_c = ops.keyed_sums(xq.cuda(), y.cuda(), num_classes=C, normalize_rows=norm)
    W = ops.keyed_means(sums_c, counts_c)
    Wref = O.simplecil_prototypes(xe.float(), y, torch.zeros(C, 512))
    assert torch.equal(counts_c.cpu(), torch.bincount(y, minlength=C))
    assert rel(W, Wref) < 1e-5
    # bit-reproducible run to run (deterministic, atomic-free)
    sums2, _ = ops.keyed_sums(xq.cuda(), y.cuda(), s.cuda(), num_classes=C, num_states=10,
                              normalize_rows=norm)
    assert torch.equal(sums, sums2)


def test_keyed_sums_empty_and_out_of_range():
    from team_b200 import ops
    x = torch.randn(64, 512)
    y = torch.arange(64) % 8
    sums, counts = ops.keyed_sums(x.cuda(), y.cuda(), class_base=2, num_classes=3)   # keeps labels 2,3,4
    assert counts.cpu().tolist() == [8, 8, 8]
    ref = torch.stack([x[y == c].double().sum(0) for c in (2, 3, 4)])
    assert rel(sums, ref) < 1e-5
    sums0, counts0 = ops.keyed_sums(torch.zeros(0, 512).cuda(), torch.zeros(0, dtype=torch.int64).cuda(), num_classes=4)
    assert counts0.cpu().tolist() == [0, 0, 0, 0] and float(sums0.abs().sum()) == 0.0


@pytest.mark.parametrize("n", [3000, 4096, 10007, 300000])
def test_keyed_sums_many_keys_foreign_rows(n):
    """Labels outside the class window, states outside [0, 10), keys that own no row, a key that owns nearly every row, on
    the key-partitioned path (K > 100 from 4 096 rows: rows sorted by key, then summed from HBM) and below 4 096 rows on the
    column-partitioned shared-memory path: exact counts, sums to round-off."""
    from team_b200 import ops
    g = torch.Generator().manual_seed(n)
    x = torch.randn(n, 512, generator=g)
    y = torch.randint(-2, 26, (n,), generator=g)
    s = torch.randint(-1, 12, (n,), generator=g)
    y[: n // 2] = 7; s[: n // 2] = 4                        # one heavy key
    y[y == 11] = 12                                          # class 11 owns nothing
    sums, counts = ops.keyed_sums(x.cuda(), y.cuda(), s.cuda(), class_base=3, num_classes=20, num_states=10)
    ok = (y >= 3) & (y < 23) & (s >= 0) & (s < 10)
    key = ((y - 3) * 10 + s)[ok]
    ref = torch.zeros(200, 512, dtype=torch.float64).index_add_(0, key, x[ok].double())
    assert torch.equal(counts.cpu(), torch.bincount(key, minlength=200))
    assert rel(sums, ref) < 1e-5
    assert int(counts[80:90].sum()) == 0 and float(sums[80:90].abs().sum()) == 0.0
    again, _ = ops.keyed_sums(x.cuda(), y.cuda(), s.cuda(), class_base=3, num_classes=20, num_states=10)
    assert torch.equal(sums, again)


@pytest.mark.parametrize("n,C,dtype", [(1, 2, torch.float32), (1025, 20, torch.float32),
                                       (4096, 32, torch.float32), (999, 50, torch.float32),
                                       (2048, 20, torch.bfloat16),
                                       # more than 8 192 rows: the tensor-pipe kernel (C = 50: two class chunks)
                                       (8193, 20, torch.float32), (70001, 50, torch.float32),
                                       (8193, 50, torch.bfloat16), (70001, 20, torch.bfloat16)])
def test_cosine_logits_vs_oracle(n, C, dtype):
    from team_b200 import ops
    x, y, _ = synth.make_prototype_build_inputs(n, max(C, 2), seed=5 + n, normalize=False)
    g = torch.Generator().manual_seed(9)
    w = torch.randn(C, 512, generator=g)
    sig = torch.tensor([1.7])
    xq = x.to(dtype)
    logits, am = ops.cosine_logits(xq.cuda(), w.cuda(), sig, want_argmax=True)
    ref = O.cosine_linear(xq.double(), w.double(), sig.double())
    assert rel(logits, ref) < 1e-5
    # argmax exact wherever the fp64 margin exceeds 10x the fp32 error bound
    top2 = ref.topk(2, dim=1).values
    safe = (top2[:, 0] - top2[:, 1]) > 1e-5
    assert torch.equal(am.cpu()[safe], ref.argmax(1)[safe])
    assert int(safe.sum()) >= int(0.99 * n)
    am_only = ops.cosine_logits(xq.cuda(), w.cuda(), sig, want_logits=False, want_argmax=True)
    assert torch.equal(am_only, am)


def test_peer_allreduce_single_rank_and_argument_checks():
    """team_peer_allreduce_f32: world = 1 is a no-op; bad arguments are rejected before any launch.  (The W > 1
    path needs one GPU per rank: tools/peer_allreduce_check.py under torchrun, profiles/r1g_peer_allreduce_check.txt.)"""
    import ctypes as C
    from team_b200 import capi
    L = capi.lib()
    x = torch.arange(16, dtype=torch.float32, device="cuda")
    flags = torch.zeros(L.team_peer_allreduce_flag_bytes() // 4, dtype=torch.int32, device="cuda")
    bufs, flgs = (C.c_void_p * 1)(x.data_ptr()), (C.c_void_p * 1)(flags.data_ptr())
    st = torch.cuda.current_stream().cuda_stream
    assert L.team_peer_allreduce_f32(bufs, flgs, None, 0, 1, 16, st) == 0
    torch.cuda.synchronize()
    assert torch.equal(x.cpu(), torch.arange(16, dtype=torch.float32))
    assert L.team_peer_allreduce_f32(bufs, flgs, None, 0, 1, 15, st) != 0        # n % 4
    assert L.team_peer_allreduce_f32(bufs, flgs, None, 3, 2, 16, st) != 0        # rank >= world
    assert L.team_peer_allreduce_f32(bufs, flgs, None, 0, 9, 16, st) != 0        # more than one box
