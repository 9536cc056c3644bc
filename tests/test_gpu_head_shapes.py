"""Head shapes that the benchmarked configuration (T = 10, C = 20, B = 1 024) does not reach, each on the kernel that
serves it: class counts around the switch between the table-row kernels (C <= 22: warp per sample, C >= 23: the first
generation with its 32-row chunks), ragged and benchmarked batches of the Gram formulation (B >= 16 384), the cosine
classifier's tensor-pipe tiles, its chunk merge and its ties, and TrainStep above 22 classes.  Every case asserts from a
torch.profiler trace that it ran the kernels it names, so that a moved threshold cannot move it off its path unnoticed,
and compares with a plain fp64 reference evaluated on the GPU: the oracle or the factorised model in fp32 mode,
oracle/quantised_model.py in bf16 mode.  Errors are norm-wise relative; the errors quoted were measured on a B200."""
import re

import pytest
import torch

from oracle import synth
from oracle import team_oracle as O
from oracle import quantised_model as Q
import factorised_model as FM
from test_gpu_training_path import (CLIP_KAPPA_MAX, EPOCHS, STEP_BARS, _clip_fed, _make_step, _reference_step,
                                    _summed, bits)

pytestmark = pytest.mark.gpu

BARS = {"f32": (1e-5, 2e-5), "bf16": (1e-3, 5e-3)}      # outputs, gradients
LOGIT_BAR = {"f32": 1e-5, "bf16": 1e-3}                 # bf16: against the logits of the bf16-rounded operands
MARGIN = {"f32": 1e-5, "bf16": 2e-3}                    # argmax must match the reference where its top-2 gap exceeds this


def rel(a, b):
    a = torch.as_tensor(a).detach().double()
    b = torch.as_tensor(b).detach().double().to(a.device)
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def kernels_run(fn):
    """fn() under torch.profiler with CUDA activities: (its result, the names of the kernels it launched)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def assert_ran(names, want=(), absent=()):
    """Every kernel of ``want`` and none of ``absent`` is among ``names`` (whole identifiers: table_rows_fwd_kernel does
    not match table_rows_fwd2_kernel or ct_table_rows_fwd_kernel)."""
    has = lambda k: any(re.search(r"(?<![\w])" + re.escape(k) + r"(?![\w])", n) for n in names)
    kernels = sorted(n for n in names if "team::" in n)
    for k in want:
        assert has(k), (k, kernels)
    for k in absent:
        assert not has(k), (k, kernels)


def table_kernels(C, B):
    """The table-row kernels the head selects for C classes and B samples (csrc/head.cu: use_table_gram, use_table2)."""
    if C + 10 > 32:
        return ("table_rows_fwd_kernel", "table_rows_bwd_kernel")
    if B >= 16384:
        return ("table_gram_fwd_kernel", "table_gram_bwd_kernel")
    return ("table_rows_fwd2_kernel", "table_rows_bwd2_kernel")


def cosine_kernel(C, n, tname="float"):
    """The classification-logit kernel for n rows and C classes (csrc/cosine.cu: team_cosine_logits)."""
    if n > 8192:
        return f"cosine_mma_kernel<{tname}, {(min(C, 32) + 7) // 8}>"
    return f"cosine_logits_kernel<{tname}>"


ALL_TABLE = ("table_rows_fwd_kernel", "table_rows_bwd_kernel", "table_rows_fwd2_kernel", "table_rows_bwd2_kernel",
             "table_gram_fwd_kernel", "table_gram_bwd_kernel")


def _inputs(C, T, ppt, B, seed):
    params = synth.make_params(T, seed=seed, prompts_per_task=ppt)
    protos = synth.make_prototypes(C, seed=seed + 1)
    batch = synth.make_batch(B, C, step=seed % 97, five_state=C % 2 == 1, num_classes_total=max(C, 20))
    cots = [c.reshape(B, 512) for c in synth.make_cotangents(B, step=seed % 97)]
    return params, protos, {k: v.cuda() for k, v in batch.items()}, [c.cuda() for c in cots]


def run_head(params, batch, protos, cots, mode):
    """The library through autograd: ([image, text, state, proto] as [B,512], logits, argmax, {name: gradient})."""
    from team_b200 import head
    B = batch["image"].shape[0]
    p = {k: v.cuda().requires_grad_(v.is_floating_point() and v.dim() > 0) for k, v in params.items()}
    outs = head.forward_tri_modal(head.HeadParamPack.from_state_dict(p), batch["image"], batch["text"], batch["state"],
                                  protos.cuda(), text_cls=batch["text_cls"], mode=mode)
    names = O.trainable_names(params)
    grads = torch.autograd.grad([o.reshape(B, 512) for o in outs[:4]], [p[n] for n in names], grad_outputs=cots)
    return [o.detach().reshape(B, 512) for o in outs[:4]], outs[4], outs[5], dict(zip(names, grads))


def reference(params, batch, protos, cots, mode_name, oracle=True):
    """fp64 on the GPU: outputs [B,512] x 4, logits [B,C] and {name: gradient}.  fp32 mode: the oracle with autograd
    (``oracle``) or the factorised model; bf16 mode: the model that rounds where the kernels round, whose logits are
    those of the bf16-rounded operands."""
    B = batch["image"].shape[0]
    names = O.trainable_names(params)
    img, txt, sid = batch["image"].double(), batch["text"].double(), batch["state"]
    pr, c64, tc = protos.double().cuda(), [c.double() for c in cots], batch["text_cls"].double()
    if mode_name == "bf16":
        p64 = {k: v.double().cuda() for k, v in params.items()}
        outs, grads, logits = Q.head_fwd_bwd(p64, img, txt, sid, pr, c64, text_cls=tc)
        return [o.reshape(B, 512) for o in outs], logits, grads
    p64 = {k: v.double().cuda().requires_grad_(k in names) for k, v in params.items()}
    with torch.no_grad():
        logits = O.forward_for_classification(p64, img, tc)
    if oracle:
        outs = [o.reshape(B, 512) for o in O.forward_tri_modal(p64, img, txt, sid, pr)[:4]]
        grads = dict(zip(names, torch.autograd.grad(outs, [p64[n] for n in names], grad_outputs=c64)))
        return [o.detach() for o in outs], logits, grads
    outs, grads = FM.head_fwd_bwd({k: v.detach() for k, v in p64.items()}, img, txt, sid, pr, c64)
    return [o.reshape(B, 512) for o in outs], logits, grads


def check_logits(logits, am, ref, mode_name):
    """Logits within the bar, argmax = torch.argmax of the returned logits exactly (first index on ties), and = the
    reference's argmax wherever its top-2 margin exceeds MARGIN.  Returns the logits error."""
    el = rel(logits, ref)
    assert el < LOGIT_BAR[mode_name], el
    assert torch.equal(am, logits.argmax(1))
    if ref.shape[1] == 1:
        assert bool((am == 0).all())
    else:
        top2 = ref.topk(2, dim=1).values
        safe = (top2[:, 0] - top2[:, 1]) > MARGIN[mode_name]
        assert torch.equal(am[safe], ref.argmax(1)[safe])
        if mode_name == "f32":              # the check is not vacuous
            assert int(safe.sum()) >= int(0.95 * ref.shape[0]), int(safe.sum())
    return el


def null_proto_cotangent_error(params, protos, batch, cots, mode):
    """HeadStepRunner backward with g_proto = NULL against an explicit all-zero prototype cotangent."""
    from team_b200 import head
    B, C = batch["image"].shape[0], protos.shape[0]
    pack = head.HeadParamPack.from_state_dict({k: v.cuda() for k, v in params.items()})
    r = head.HeadStepRunner(pack, protos.cuda(), B, C, mode)
    img, txt, sid = batch["image"], batch["text"], batch["state"]
    r.forward(img, txt, sid, batch["text_cls"])
    r.backward(img, txt, sid, [cots[0], cots[1], cots[2], torch.zeros_like(cots[3])])
    torch.cuda.synchronize()
    want = r.flat_grads.clone()
    r.forward(img, txt, sid, batch["text_cls"])
    r.backward(img, txt, sid, [cots[0], cots[1], cots[2], None])
    torch.cuda.synchronize()
    return rel(r.flat_grads, want)


# ------------------------------------------------------------------------------------------ 1. class-count boundaries
# (C, T, prompts per task, B): Ns = C + T * ppt + 10 step rows, padded to Nsp, a multiple of 16
CLASS_CASES = [(1, 1, 10, 37),       # one prototype row: the prototype output is that row's output
               (7, 1, 15, 333),      # odd C; Ns = 32
               (7, 1, 16, 37),       # Ns = 33, padded to 48
               (21, 3, 10, 333),     # 31 table rows
               (22, 2, 0, 37),       # 32 table rows, 220 KB of shared memory in the backward; no prompt rows, Ns = 32
               (23, 2, 10, 333),     # the smallest head on the first-generation kernels
               (127, 1, 10, 37),     # C + 1 = 128 table-query rows: one full 32-row chunk per warp
               (128, 1, 10, 333),    # warp 0 gets a second chunk of one row
               (200, 1, 10, 1000)]   # Rt = 210, two chunks per warp; B > 6 x 148: the forward's grid-stride loop goes round twice


@pytest.mark.parametrize("mode_name", ["f32", "bf16"])
@pytest.mark.parametrize("C,T,ppt,B", CLASS_CASES, ids=[f"C{c[0]}_T{c[1]}_ppt{c[2]}_B{c[3]}" for c in CLASS_CASES])
def test_class_counts_vs_fp64(C, T, ppt, B, mode_name):
    """forward_tri_modal (outputs, gradients, classification logits over the C class texts) with C decoupled from T and
    the prompt count, against the fp64 oracle with autograd (fp32) or the bf16-rounding model (bf16) at the bars of
    test_gpu_head.py: fp32 outputs <= 1e-5, gradients <= 2e-5, logits <= 1e-5 (measured <= 3.2e-7 / 7.2e-7 / 3.0e-7);
    bf16 outputs <= 1e-3, gradients <= 5e-3, logits <= 1e-3 against the rounded operands (measured <= 4.9e-4 / 4.8e-3,
    C = 128, / 9.7e-6).  A NULL prototype cotangent gives the gradients of an explicit zero cotangent within 1e-6 on
    both table-row generations (measured: bitwise equal)."""
    from team_b200 import head
    mode = head.MODE_F32 if mode_name == "f32" else head.MODE_BF16
    params, protos, batch, cots = _inputs(C, T, ppt, B, seed=500 + C + ppt)
    (outs, logits, am, grads), names = kernels_run(lambda: run_head(params, batch, protos, cots, mode))
    assert_ran(names, table_kernels(C, B) + (cosine_kernel(C, B),) + (("cosine_argmax_merge",) if C > 32 else ()),
               absent=tuple(k for k in ALL_TABLE if k not in table_kernels(C, B)))
    ref_o, ref_l, ref_g = reference(params, batch, protos, cots, mode_name)
    tol_o, tol_g = BARS[mode_name]
    eo = {k: rel(o, r) for k, o, r in zip(("image", "text", "state", "proto"), outs, ref_o)}
    eg = {n: rel(grads[n], g) for n, g in ref_g.items()}
    print(f"measured C={C} T={T} ppt={ppt} B={B} {mode_name}: outputs {max(eo.values()):.2e} gradients "
          f"{max(eg.values()):.2e} ({max(eg, key=eg.get)}) logits {rel(logits, ref_l):.2e}")
    assert max(eo.values()) < tol_o, eo
    assert max(eg.values()) < tol_g, eg
    check_logits(logits, am, ref_l, mode_name)
    en = null_proto_cotangent_error(params, protos, batch, cots, mode)
    print(f"measured C={C} B={B} {mode_name}: null vs zero prototype cotangent {en:.2e}")
    assert en < 1e-6, en


# -------------------------------------------------------------------------------- 2. Gram formulation, ragged batches
GRAM_CASES = [(22, 2), (1, 1), (20, 10)]        # (C, T); (20, 10) is the benchmarked head


@pytest.mark.parametrize("mode_name", ["f32", "bf16"])
@pytest.mark.parametrize("C,T", GRAM_CASES, ids=[f"C{c}_T{t}" for c, t in GRAM_CASES])
def test_gram_ragged_batch_vs_fp64_and_chunks(C, T, mode_name):
    """B = 16 397 = 16 384 + 13: the Gram table-row kernels with a ragged last group of every warp count and GEMM tile,
    the tensor-pipe cosine kernel for the logits.  Against the fp64 factorised model (fp32) or the bf16-rounding model at
    the bars of test_gram_table_rows_match_the_oracle, and against the second-generation kernels on the same batch in
    2 048-sample chunks (the last one 13 samples): outputs chunk by chunk <= 2e-5 / 2e-3, gradients as the sum over the
    chunks <= 5e-5 / 5e-3 (measured fp32 <= 2.2e-7 / 1.5e-6, bf16 <= 2.0e-6 / 3.9e-3); against fp64, fp32 <= 3.4e-7 /
    1.4e-6, bf16 <= 4.1e-4 / 4.4e-3; logits <= 9.5e-6.  NULL vs zero prototype cotangent within 1e-6 (measured: bitwise
    equal)."""
    from team_b200 import head
    mode = head.MODE_F32 if mode_name == "f32" else head.MODE_BF16
    B, n = 16397, 2048
    params, protos, batch, cots = _inputs(C, T, 10, B, seed=600 + C)
    (outs, logits, am, grads), names = kernels_run(lambda: run_head(params, batch, protos, cots, mode))
    assert_ran(names, table_kernels(C, B) + (cosine_kernel(C, B),), absent=ALL_TABLE[:4])
    tol_co, tol_cg = (2e-5, 5e-5) if mode_name == "f32" else (2e-3, 5e-3)
    grad_sum = {k: torch.zeros_like(g, dtype=torch.float64) for k, g in grads.items()}
    worst_c = 0.0
    for c0 in range(0, B, n):
        sl = slice(c0, c0 + n)
        part = {k: (v if k == "text_cls" else v[sl]) for k, v in batch.items()}
        run = lambda: run_head(params, part, protos, [x[sl] for x in cots], mode)
        if c0 + n >= B:
            (outs_c, _, _, grads_c), names_c = kernels_run(run)
            assert_ran(names_c, table_kernels(C, B - c0))
        else:
            outs_c, _, _, grads_c = run()
        for k in range(4):
            worst_c = max(worst_c, rel(outs[k][sl], outs_c[k]))
        for k, g in grads_c.items():
            grad_sum[k] += g.double()
    ec = {k: rel(g, grad_sum[k]) for k, g in grads.items()}
    ref_o, ref_l, ref_g = reference(params, batch, protos, cots, mode_name, oracle=False)
    tol_o, tol_g = BARS[mode_name]
    eo = max(rel(o, r) for o, r in zip(outs, ref_o))
    eg = {k: rel(grads[k], g) for k, g in ref_g.items()}
    en = null_proto_cotangent_error(params, protos, batch, cots, mode)
    print(f"measured gram B={B} C={C} T={T} {mode_name}: vs chunks outputs {worst_c:.2e} gradients {max(ec.values()):.2e}; "
          f"vs fp64 outputs {eo:.2e} gradients {max(eg.values()):.2e}; null vs zero prototype cotangent {en:.2e}")
    assert worst_c < tol_co and max(ec.values()) < tol_cg, (worst_c, ec)
    assert eo < tol_o and max(eg.values()) < tol_g, (eo, eg)
    el = check_logits(logits, am, ref_l, mode_name)
    print(f"measured gram B={B} C={C} {mode_name}: logits {el:.2e}")
    assert en < 1e-6, en


@pytest.mark.parametrize("mode_name", ["f32", "bf16"])
def test_gram_at_65536_vs_fp64(mode_name):
    """The benchmarked head (T = 10, C = 20) at B = 65 536, the largest batch of the benchmark's at-scale sweep.  The
    outputs of a sample depend on that sample and the step rows only, and every gradient is a sum of per-sample terms,
    so the fp64 references run in 8 192-sample chunks on the GPU.  fp32: outputs <= 1e-5 and gradients (the sum over
    the chunks of the factorised model) <= 2e-5.  bf16: outputs <= 1e-3 against the bf16-rounding model chunk by chunk;
    that model rounds summed operands, so its gradients do not add up over chunks, and the gradients are compared
    with the sum of eight 8 192-sample runs of the library (second-generation kernels) at the bar of
    test_large_batch_equals_its_chunks, 4e-3.  Logits as everywhere.  Measured: fp32 outputs 3.3e-7, gradients 2.4e-6;
    bf16 outputs 1.2e-4, gradients 3.6e-3; logits <= 5.2e-6."""
    from team_b200 import head
    mode = head.MODE_F32 if mode_name == "f32" else head.MODE_BF16
    T, C, B, n = 10, 20, 65536, 8192
    params, protos, batch, cots = _inputs(C, T, 10, B, seed=65)
    (outs, logits, am, grads), names = kernels_run(lambda: run_head(params, batch, protos, cots, mode))
    assert_ran(names, table_kernels(C, B) + (cosine_kernel(C, B),), absent=ALL_TABLE[:4])
    names_t = O.trainable_names(params)
    err2, ref2 = [0.0] * 4, [0.0] * 4
    ref_l = []
    grad_sum = {k: torch.zeros_like(g, dtype=torch.float64) for k, g in grads.items()}
    for c0 in range(0, B, n):
        sl = slice(c0, c0 + n)
        part = {k: (v if k == "text_cls" else v[sl]) for k, v in batch.items()}
        ro, rl, rg = reference(params, part, protos, [x[sl] for x in cots], mode_name, oracle=False)
        for k in range(4):
            err2[k] += float((outs[k][sl].double() - ro[k]).norm() ** 2)
            ref2[k] += float(ro[k].norm() ** 2)
        ref_l.append(rl)
        if mode_name == "bf16":
            _, _, _, rg = run_head(params, part, protos, [x[sl] for x in cots], mode)
        for k in names_t:
            grad_sum[k] += rg[k].double()
        del ro, rg
    eo = max((e / r) ** 0.5 for e, r in zip(err2, ref2))
    eg = {k: rel(grads[k], g) for k, g in grad_sum.items()}
    tol_o, tol_g = (1e-5, 2e-5) if mode_name == "f32" else (1e-3, 4e-3)
    print(f"measured B={B} {mode_name}: outputs {eo:.2e} gradients {max(eg.values()):.2e} ({max(eg, key=eg.get)})")
    assert eo < tol_o and max(eg.values()) < tol_g, (eo, eg)
    el = check_logits(logits, am, torch.cat(ref_l), mode_name)
    print(f"measured B={B} {mode_name}: logits {el:.2e}")
    torch.cuda.empty_cache()


# ----------------------------------------------------------------------------- 3. cosine classifier: tiles, merge, ties
COS_CASES = [(8193, 1), (20011, 2), (20011, 8), (8193, 9), (20011, 16), (8193, 17), (20011, 32), (8193, 33),
             (20011, 200), (4097, 200)]
DTYPES = {"f32": (torch.float32, "float"), "bf16": (torch.bfloat16, "__nv_bfloat16")}


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("n,C", COS_CASES, ids=[f"n{n}_C{c}" for n, c in COS_CASES])
def test_cosine_tiles_and_chunks_vs_fp64(n, C, dt):
    """team_cosine_logits above 8 192 rows (8 193 is one past the switch) at every tile count of the tensor-pipe kernel
    (nt = ceil(min(C, 32) / 8) = 1..4), across the 32-class chunk boundary (C = 32 / 33) and with seven chunks, the last
    one ragged (C = 200, above and below 8 192 rows).  Against sigma normalize(x) normalize(W)^T in fp64 on the same
    (bf16-rounded) x: logits <= 1e-5; argmax = torch.argmax of the returned logits exactly; = the fp64 argmax where
    the fp64 top-2 margin exceeds 1e-5.  Measured logits: <= 3.7e-6 on the tensor pipe (3xTF32), 1.1e-7 below 8 192 rows."""
    from team_b200 import ops
    dtype, tname = DTYPES[dt]
    x, _, _ = synth.make_prototype_build_inputs(n, max(C, 2), seed=7 + n + C, normalize=False)
    w = torch.randn(C, 512, generator=torch.Generator().manual_seed(C)).cuda()
    sig = torch.tensor([1.7])
    xq = x.to(dtype).cuda()
    (logits, am), names = kernels_run(lambda: ops.cosine_logits(xq, w, sig, want_argmax=True))
    assert_ran(names, (cosine_kernel(C, n, tname),) + (("cosine_argmax_merge",) if C > 32 else ()),
               absent=("cosine_logits_kernel" if n > 8192 else "cosine_mma_kernel",) + (() if C > 32 else ("cosine_argmax_merge",)))
    ref = O.cosine_linear(xq.double(), w.double(), sig.double().cuda())
    el = check_logits(logits, am, ref, "f32")
    print(f"measured cosine n={n} C={C} {dt}: logits {el:.2e}")


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("n,C", [(1000, 16), (9001, 16), (1000, 72), (9001, 72)])
def test_cosine_ties_and_empty_classes(n, C, dt):
    """Ties built on purpose, on both kernels (1 000 and 9 001 rows), with one class chunk (C = 16) and three (C = 72):
    two equal class rows inside a chunk (5 and 6), two in different chunks (3 and 40; 3 and 9 at C = 16), and
    all-zero class rows (their logits are 0, not NaN).  Samples parallel to class 3 or 5 must pick the lower index of
    the tie; samples whose every non-zero class logit is negative must pick the first empty class, whose 0 they share
    with the other empty classes.  Equal class rows give bitwise-equal logits, and the argmax is torch.argmax of the
    returned logits (first maximal index) for every row."""
    from team_b200 import ops
    dtype, tname = DTYPES[dt]
    g = torch.Generator().manual_seed(n + C)
    w = torch.randn(C, 512, generator=g)
    w[:, 0] = w[:, 0].abs() + 4.0                # every non-empty class row leans towards +e0
    twin = 40 if C > 32 else 9
    empty = [10, 50, 70] if C > 32 else [10, 12]
    w[6], w[twin] = w[5], w[3]
    w[empty] = 0.0
    x = torch.randn(n, 512, generator=g)
    q = n // 4
    x[:q] = w[3] * (0.5 + torch.rand(q, 1, generator=g))
    x[q:2 * q] = w[5] * (0.5 + torch.rand(q, 1, generator=g))
    x[2 * q:3 * q] = 0.1 * x[2 * q:3 * q]
    x[2 * q:3 * q, 0] = -10.0                    # negative against every non-empty class, 0 against the empty ones
    xq, wd = x.to(dtype).cuda(), w.cuda()
    (logits, am), names = kernels_run(lambda: ops.cosine_logits(xq, wd, want_argmax=True))
    assert_ran(names, (cosine_kernel(C, n, tname),) + (("cosine_argmax_merge",) if C > 32 else ()))
    assert not bool(logits.isnan().any())
    assert bool((logits[:, empty] == 0).all())
    assert torch.equal(bits(logits[:, 3]), bits(logits[:, twin])) and torch.equal(bits(logits[:, 5]), bits(logits[:, 6]))
    assert torch.equal(am, logits.argmax(1))
    assert bool((am[:q] == 3).all()) and bool((am[q:2 * q] == 5).all()) and bool((am[2 * q:3 * q] == empty[0]).all())
    assert rel(logits, O.cosine_linear(xq.double(), wd.double())) < 1e-5


# ------------------------------------------------------------------------------- 4. TrainStep above 22 classes
def _step_config(T, C, B):
    """Parameters, prototypes, class text, an evolution feature for every class and three batches with C decoupled from
    T: C = 40 runs the first-generation table-row kernels and two cosine chunks."""
    params = synth.make_params(T, seed=42)
    protos = synth.make_prototypes(C)
    text_cls = synth.make_text_class_features(C)
    gen = torch.Generator().manual_seed(5)
    evo = [torch.randn(512, generator=gen) for _ in range(C)]
    batches = [synth.make_batch(B, C, step=s, num_classes_total=C) for s in range(3)]
    return params, protos, text_cls, evo, batches


@pytest.mark.parametrize("mode", [0, 1], ids=["f32", "bf16"])
def test_train_step_40_classes_vs_fp64(mode):
    """TrainStep (its backward passes g_proto = NULL) at T = 10, C = 40, B = 1 024, three steps over epochs [0, 0, 1],
    checked as test_train_step_vs_fp64 checks the benchmarked step and with its bars (STEP_BARS, CLIP_KAPPA_MAX): the
    five losses and every gradient against the fp64 step reference, and the parameters against an fp64 AdamW mirror
    driven by the step's own gradients (<= 1e-6).  Measured: fp32 losses 9.5e-8, gradients 1.1e-6, projection / state
    table gradients 2.4e-6; bf16 5.0e-4, 7.0e-3, 2.3e-2; parameters vs mirror <= 8.4e-8; ClipLoss cancellation factors
    2.5 / 2.8 / 4.6, so every gradient is compared at every step in both modes."""
    T, C, B = 10, 40, 1024
    params, protos, text_cls, evo, batches = _step_config(T, C, B)
    pg, ts = _make_step(params, protos, text_cls, evo, B, mode)
    names = O.trainable_names(params)
    by_id = {id(pg[n]): n for n in names}
    views = {by_id[id(p)]: g for p, g in ts.pairs}
    mirror = {n: pg[n].detach().double().clone().requires_grad_(True) for n in names}
    opt = torch.optim.AdamW([mirror[n] for n in names], lr=ts.init_lr, weight_decay=0.05)
    p64 = {k: v.double().cuda() for k, v in params.items()}
    pr, tc, evo64 = protos.cuda(), text_cls.cuda(), [e.double().cuda() for e in evo]
    tl, tg, tb = STEP_BARS[mode]
    worst, checked, kappas = [0.0, 0.0, 0.0, 0.0], set(), []
    for i, (b, ep) in enumerate(zip(batches, EPOCHS)):
        bd = {k: v.cuda() for k, v in b.items()}
        ts.load(bd["image"], bd["text"], bd["state"], bd["label"])
        got = ts.step(epoch=ep).double().cpu().tolist()
        grads = {n: views[n].detach().double().reshape(mirror[n].shape) for n in names}
        start = dict(p64, **{n: mirror[n].detach().clone() for n in names})
        ref_l, ref_g, kappa = _reference_step(start, params, pr, tc, evo64, bd, ep, ts, names)
        el = max(abs(a - r) / max(1.0, abs(r)) for a, r in zip(got, ref_l))
        eg = {n: rel(grads[n], ref_g[n]) for n in names if mode == 0 or kappa <= CLIP_KAPPA_MAX or not _clip_fed(n)}
        checked |= set(eg)
        kappas.append(round(kappa, 1))
        for grp in opt.param_groups:
            grp["lr"] = ts.lr_at(ep)
        for n in names:
            mirror[n].grad = grads[n]
        opt.step()
        ep_ = {n: rel(pg[n], mirror[n]) for n in names}
        wb = max(e for n, e in eg.items() if _summed(n))
        wg = max(e for n, e in eg.items() if not _summed(n))
        worst = [max(worst[0], el), max(worst[1], wg), max(worst[2], wb), max(worst[3], max(ep_.values()))]
        assert el <= tl, (i, got, ref_l)
        bad = {n: e for n, e in eg.items() if e > (tb if _summed(n) else tg)}
        assert not bad, (i, bad)
        assert max(ep_.values()) <= 1e-6, (i, ep_)
        assert int(ts.opt.step_dev.cpu()) == i + 1
    assert checked == set(names)
    print(f"measured train step C={C} B={B} mode={mode}: losses {worst[0]:.2e} gradients {worst[1]:.2e} "
          f"projection / state table gradients {worst[2]:.2e} parameters vs mirror {worst[3]:.2e} "
          f"ClipLoss cancellation per step {kappas}")


@pytest.mark.parametrize("mode", [0, 1], ids=["f32", "bf16"])
def test_train_step_40_classes_replays_match_eager(mode):
    """Two TrainSteps at C = 40 on the same parameters and batches: one replays its captured graph twice (the argmax
    scratch of the two cosine chunks is allocated inside the graph, from cudaMallocAsync on the classification side
    stream), the other runs the same body eagerly.  After each step the losses, the gradients, the classification
    logits and argmax and the parameters are bitwise equal; the eager run launched the first-generation backward and
    the argmax merge."""
    T, C, B = 10, 40, 1024
    params, protos, text_cls, evo, batches = _step_config(T, C, B)
    (p0, t0), (p1, t1) = [_make_step(params, protos, text_cls, evo, B, mode) for _ in range(2)]
    for s, b in enumerate(batches[:2]):
        dev = [b["image"].cuda(), b["text"].cuda(), b["state"].cuda(), b["label"].cuda()]
        t0.load(*dev)
        t0.step(epoch=0)
        t1.load(*dev)
        _, names = kernels_run(lambda: t1._body(0))
        if s == 0:
            assert_ran(names, table_kernels(C, B) + ("cosine_logits_kernel<float>", "cosine_argmax_merge"))
        torch.cuda.synchronize()
        assert sorted(t0._graphs) == [0]
        assert torch.equal(bits(t0.losses6), bits(t1.losses6))
        assert torch.equal(bits(t0.runner.flat_grads), bits(t1.runner.flat_grads))
        assert torch.equal(bits(t0.runner.logits), bits(t1.runner.logits))
        assert torch.equal(t0.runner.argmax, t1.runner.argmax)
        for (a, _), (c, _) in zip(t0.pairs, t1.pairs):
            assert torch.equal(bits(a), bits(c))
