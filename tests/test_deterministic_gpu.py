"""Bitwise-reproducible training step under torch.use_deterministic_algorithms(True) (DESIGN.md §5 (ix)).

With the switch on, the backward's fp32 reductions run their ordered variants (split-K weight gradients, LayerNorm dgamma /
dbeta, bias column sums, the token-embedding scatter and the position / rating-embedding sums): equal inputs, parameters and
seed give equal bits — loss, every gradient, every parameter after the optimizer — run after run, in another process, with
plain launches or graph replay, whatever the allocator cache and on-chip memory held before.  With the switch off nothing
changes.  Every test here turns the switch on through its own context and restores it, so no other test sees it."""
import contextlib
import hashlib
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

D = 1024


@contextlib.contextmanager
def deterministic(on=True):
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


@pytest.fixture
def det():
    with deterministic(True):
        yield


def _poison():
    """NaN patterns into the allocator's free blocks and every SM's shared / tensor memory."""
    from multimodalsum_b200 import ops
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    junk = [torch.full((n,), float("nan"), device="cuda") for n in (1 << 28, 1 << 26, 1 << 26, 1 << 24, 1 << 22, 1 << 20)]
    junk += [torch.full((1 << 16,), float("nan"), device="cuda") for _ in range(32)]
    del junk
    ops.debug_poison()
    torch.cuda.synchronize()


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t.contiguous()


def _same_bits(a, b):
    return torch.equal(_bits(a), _bits(b))


def _rel(a, b):
    return (a.double() - b.double()).norm().item() / max(b.double().norm().item(), 1e-30)


# ============================================================================================================ kernel level
# the split-K weight-gradient shapes of the training step (profiles/r02_gemm_shapes_in_step.txt: M N K, fp32 accumulate)
WGRAD_SHAPES = [(1024, 1024, 18432), (1024, 4096, 18432), (4096, 1024, 18432), (3072, 1024, 18432), (2048, 1024, 50544),
                (1024, 1024, 55296), (50265, 1024, 18432), (1024, 1024, 31360), (1024, 2048, 752), (1024, 1024, 752)]


def test_ordered_gemm_splits_the_step_shapes():
    """The ordered path is exercised: most wgrad shapes of the step run with several splits on this GPU."""
    from multimodalsum_b200 import ops
    split = [s for s in WGRAD_SHAPES if ops.gemm_workspace_elems(*s) > 0]
    assert len(split) >= 4, split


@pytest.mark.parametrize("M,N,K", WGRAD_SHAPES)
def test_ordered_splitk_gemm_is_bitwise_reproducible(M, N, K):
    from multimodalsum_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    ldm = (M + 7) // 8 * 8                                                      # 16-byte row pitch, as the step's logits have
    A = torch.randn(K, ldm, device="cuda", generator=g).to(torch.bfloat16)[:, :M]   # dy [T, N_out]
    B = torch.randn(K, N, device="cuda", generator=g).to(torch.bfloat16)        # x  [T, K_in]
    D0 = torch.randn(M, N, device="cuda", generator=g)                           # accumulate onto a non-zero gradient
    need = ops.gemm_workspace_elems(M, N, K)
    outs = []
    for _ in range(2):
        _poison()
        ws = torch.empty(max(need, 1), device="cuda")
        Dd = D0.clone()
        n0 = ops.ORDERED_CALLS["gemm"]
        ops.gemm(A, B, Dd, a_t=True, b_t=True, accumulate=True, workspace=ws)
        assert ops.ORDERED_CALLS["gemm"] == n0 + 1
        torch.cuda.synchronize()
        outs.append(Dd)
    assert _same_bits(outs[0], outs[1])
    Df = D0.clone()
    ops.gemm(A, B, Df, a_t=True, b_t=True, accumulate=True)
    assert torch.isfinite(outs[0]).all()
    assert _rel(outs[0] - D0, Df - D0) <= 2e-6, _rel(outs[0] - D0, Df - D0)
    if M * N <= 1024 * 1024:                                                    # and against an fp64 product
        ref = D0.double() + A.double().t() @ B.double()
        assert _rel(outs[0] - D0, ref - D0.double()) <= 1e-5


def test_ordered_gemm_rejects_a_short_workspace():
    from multimodalsum_b200 import _lib, ops
    M, N, K = 1024, 1024, 18432
    need = ops.gemm_workspace_elems(M, N, K)
    assert need > 0
    A = torch.zeros(K, M, device="cuda", dtype=torch.bfloat16)
    B = torch.zeros(K, N, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(_lib.MmsumError, match="rc=-1"):
        ops.gemm(A, B, torch.zeros(M, N, device="cuda"), a_t=True, b_t=True, accumulate=True,
                 workspace=torch.empty(need - 1, device="cuda"))


def _ln_inputs(rows, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    bf = lambda *s: torch.randn(*s, device="cuda", generator=g).to(torch.bfloat16)
    res, y, d1, d2 = bf(rows, D), bf(rows, D), bf(rows, D), bf(rows, D)
    z = res.float() + y.float()
    mean, rstd = z.mean(1), torch.rsqrt(z.var(1, unbiased=False) + 1e-5)
    gamma = torch.rand(D, device="cuda", generator=g) + 0.5
    return res, y, d1, d2, gamma, mean, rstd, torch.randn(D, device="cuda", generator=g), torch.randn(D, device="cuda", generator=g)


@pytest.mark.parametrize("rows,p_drop", [(18432, 0.1), (18432, 0.0), (5376, 0.1), (752, 0.0)])
def test_ordered_add_ln_bwd_is_bitwise_reproducible(rows, p_drop):
    from multimodalsum_b200 import ops
    res, y, d1, d2, gamma, mean, rstd, dg0, db0 = _ln_inputs(rows, rows)
    step = torch.tensor([3], device="cuda", dtype=torch.int32)

    def run(ws):
        dres, dy = torch.empty_like(res), torch.empty_like(res)
        dg, db = dg0.clone(), db0.clone()
        ops.add_ln_bwd(d1, d2, res, y, gamma, mean, rstd, dres, dy, dg, db, p_drop, 7, 11, step_dev=step, workspace=ws)
        torch.cuda.synchronize()
        return dres, dy, dg, db

    outs = []
    for _ in range(2):
        _poison()
        outs.append(run(torch.empty(ops.ADD_LN_BWD_WORKSPACE, device="cuda")))
    fast = run(None)
    for a, b, f in zip(outs[0], outs[1], fast):
        assert _same_bits(a, b)
    assert torch.equal(outs[0][0], fast[0]) and torch.equal(outs[0][1], fast[1])     # per-row outputs: the same kernel code
    for i in (2, 3):
        assert _rel(outs[0][i] - (dg0, db0)[i - 2], fast[i] - (dg0, db0)[i - 2]) <= 1e-5


@pytest.mark.parametrize("rows,N,ld", [(18432, 1024, 1024), (18432, 3072, 3072), (18432, 4096, 4096), (55296, 1024, 1024),
                                       (18432, 1024, 2048), (752, 2048, 2048)])
def test_ordered_colsum_is_bitwise_reproducible(rows, N, ld):
    from multimodalsum_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(rows + N)
    base = torch.randn(rows, ld, device="cuda", generator=g).to(torch.bfloat16)
    x = base[:, :N]
    o0 = torch.randn(N, device="cuda", generator=g)
    outs = []
    for _ in range(2):
        _poison()
        o = o0.clone()
        ops.colsum(x, o, workspace=torch.empty(ops.colsum_workspace(N), device="cuda"))
        torch.cuda.synchronize()
        outs.append(o)
    assert _same_bits(outs[0], outs[1])
    of = o0.clone()
    ops.colsum(x, of)
    ref = o0.double() + x.double().sum(0)
    assert _rel(outs[0] - o0, ref - o0.double()) <= 1e-4 and _rel(of - o0, ref - o0.double()) <= 1e-4


def _embed_case(rows, S, V, ids_kind, rating, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = lambda *s: torch.randn(*s, device="cuda", generator=g)
    pad = 1
    if ids_kind == "one_id":          # every row the same id, pad ids mixed in
        ids = torch.full((rows,), 7, device="cuda", dtype=torch.int32)
        ids[torch.rand(rows, device="cuda", generator=g) < 0.3] = pad
    elif ids_kind == "few_ids":
        ids = torch.randint(0, 5, (rows,), device="cuda", generator=g, dtype=torch.int32)
    else:
        ids = torch.randint(0, V, (rows,), device="cuda", generator=g, dtype=torch.int32)
        ids[rows // 3:rows // 2] = pad
    E, P = f(V, D) * 0.1, f(S + 2, D) * 0.1
    rd = f(rows // S) if rating else None
    remb = f(D) * 0.1 if rating else None
    gamma = torch.rand(D, device="cuda", generator=g) + 0.5
    z = E[ids.long()] + P[torch.arange(rows, device="cuda") % S + 2]
    if rating:
        z = z + rd.repeat_interleave(S)[:, None] * remb
    mean, rstd = z.mean(1), torch.rsqrt(z.var(1, unbiased=False) + 1e-5)
    dout = f(rows, D).to(torch.bfloat16)
    dout2 = f(rows, D).to(torch.bfloat16)
    return dict(dout=dout, dout2=dout2, ids=ids, E=E, P=P, rd=rd, remb=remb, gamma=gamma, mean=mean, rstd=rstd, pad=pad)


@pytest.mark.parametrize("rows,S,V,ids_kind,rating", [(18432, 128, 50265, "one_id", True), (13312, 104, 50265, "random", False),
                                                      (18432, 128, 50265, "random", True), (4096, 128, 3000, "few_ids", True)])
def test_ordered_embedding_backward_is_bitwise_reproducible(rows, S, V, ids_kind, rating):
    """Token-embedding scatter with heavy id duplication (all rows one id, pad ids mixed in), position and rating-embedding sums
    and dgamma / dbeta: the ordered call twice after poisoning bit for bit, the pad row exactly 0, and the atomic call within
    fp32 rounding."""
    from multimodalsum_b200 import ops
    c = _embed_case(rows, S, V, ids_kind, rating, rows + V)
    g = torch.Generator(device="cuda").manual_seed(5)
    dP0, dr0 = torch.randn(S + 2, D, device="cuda", generator=g), torch.randn(D, device="cuda", generator=g)
    dg0, db0 = torch.randn(D, device="cuda", generator=g), torch.randn(D, device="cuda", generator=g)
    step = torch.tensor([2], device="cuda", dtype=torch.int32)

    def run(ws):
        dE = torch.zeros(V, D, device="cuda")
        dP, dr, dg, db = dP0.clone(), dr0.clone(), dg0.clone(), db0.clone()
        dz = torch.empty(rows, D, device="cuda")
        ops.embed_ln_bwd(c["dout"], c["dout2"], c["ids"], c["E"], c["P"], c["rd"], c["remb"], c["gamma"], c["mean"], c["rstd"],
                         dE, dP, dr if rating else None, dg, db, dz, rows, S, c["pad"], 0.1, 3, 9, step_dev=step, workspace=ws)
        torch.cuda.synchronize()
        return dE, dP, dr, dg, db, dz

    outs = []
    for _ in range(2):
        _poison()
        outs.append(run(torch.empty(ops.embed_ln_bwd_workspace(rows, S, V), device="cuda")))
    fast = run(None)
    for a, b in zip(outs[0], outs[1]):
        assert _same_bits(a, b)
    dE, dP, dr, dg, db, dz = outs[0]
    assert torch.equal(dz, fast[5])
    assert (dE[c["pad"]] == 0).all() and _same_bits(dE[c["pad"]], torch.zeros(D, device="cuda"))
    used = torch.zeros(V, dtype=torch.bool, device="cuda")
    used[c["ids"].long()] = True
    used[c["pad"]] = False
    assert (dE[~used] == 0).all()
    # reference for dE: fp64 sum of the dz rows per id
    ref = torch.zeros(V, D, device="cuda", dtype=torch.float64)
    keep = c["ids"] != c["pad"]
    ref.index_add_(0, c["ids"][keep].long(), dz[keep].double())
    assert _rel(dE, ref) <= 1e-4 and _rel(fast[0], ref) <= 1e-4
    for i, base in ((1, dP0), (3, dg0), (4, db0)) + (((2, dr0),) if rating else ()):
        assert _rel(outs[0][i] - base, fast[i] - base) <= 1e-5, i


def test_table_bits_backward_is_bitwise_reproducible():
    """No ordered variant needed: one thread sums each dW element in a fixed order and adds it once."""
    from multimodalsum_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    B, F = 16, 47
    dX = torch.randn(B * F, 2 * D, device="cuda", generator=g).to(torch.bfloat16)
    bits = torch.randint(0, 2, (B, 7, 4), device="cuda", generator=g)
    W0 = torch.randn(D, 4, device="cuda", generator=g)
    outs = []
    for _ in range(2):
        _poison()
        W = W0.clone()
        ops.table_bits_bwd(dX, bits, W, B, F, 40, 7, 4)
        torch.cuda.synchronize()
        outs.append(W)
    assert _same_bits(outs[0], outs[1])
    ref = torch.einsum("brj,brc->cj", bits.double(), dX.view(B, F, 2 * D)[:, 40:47, D:].double())
    assert _rel(outs[0] - W0, ref) <= 1e-4


# ============================================================================================================== step level
def _batch_args(cfg, b):
    if cfg.dataset == "text":
        return (b.reviews, b.reviews_mask, b.reviews_rating), {}
    if cfg.dataset == "img":
        return (b.img, b.img_mask), dict(labels=b.labels)
    if cfg.dataset.startswith("table_"):
        return (b.field, b.field_value), dict(labels=b.labels)
    return (b.reviews, b.reviews_mask, b.reviews_rating, b.field, b.field_value, b.img, b.img_mask), \
        dict(max_review_len=getattr(b, "max_review_len", None))


def _make_model(cfg, sd=None):
    from multimodalsum_b200.modules import (AmazonTableEncoder, ImgSupervised, MultimodalSum, TableSupervised, TextSupervised,
                                            YelpTableEncoder)
    torch.manual_seed(0)
    if cfg.dataset == "text":
        model = TextSupervised(config=cfg, label_smoothing=None)
    elif cfg.dataset == "img":
        model = ImgSupervised(config=cfg, label_smoothing=0.1)
    elif cfg.dataset.startswith("table_"):
        model = TableSupervised(TableEncoder=YelpTableEncoder if cfg.table == "yelp" else AmazonTableEncoder, config=cfg,
                                label_smoothing=0.1)
    else:
        model = MultimodalSum(TableEncoder=YelpTableEncoder if cfg.dataset == "yelp" else AmazonTableEncoder, config=cfg,
                              label_smoothing=0.1)
    if sd is not None:
        model.load_state_dict(sd, strict=False)
    return model.cuda().train()


def _case(name):
    """(cfg, state_dict or None = torch.manual_seed(0) init, 3 batches on the device)."""
    from multimodalsum_b200.synth import ModelConfig, make_batch
    if name in ("yelp_b16", "amazon_b8"):
        amazon = name == "amazon_b8"
        cfg = ModelConfig(dataset="amazon" if amazon else "yelp", dropout=0.1)
        B = 8 if amazon else 16
        batches = [make_batch(cfg, B, seed=1234 + 17 * i, fixed_len=70 if amazon else 100,
                              n_valid_imgs=1 if amazon else 10).with_length_hint().to("cuda") for i in range(3)]
        return cfg, None, batches
    from golden_util import load_golden
    gold = load_golden(name)
    cfg = gold["cfg"]
    cfg.dropout = 0.1
    b = gold["batch"].to("cuda")
    return cfg, gold["sd"], [b, b, b]          # the weights and the dropout masks still change from step to step


def _run_steps(model, cfg, batches, graph=False, stock=False):
    """Three training steps from the model's current state: loss, gradient arena after each backward, parameters at the end."""
    from multimodalsum_b200.optim import get_optimizer
    eng = model._ensure_engine(torch.device("cuda"))
    eng.enable_graph(graph)
    if stock:
        opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=0.01)
    else:
        opt = get_optimizer(eng, 1e-3, ["bias", "LayerNorm.weight"], list(model.named_parameters()), None, max_grad_norm=1.0)
    losses, grads = [], []
    for b in batches:
        a, kw = _batch_args(cfg, b)
        loss = model(*a, **kw)[0]
        model.zero_grad(set_to_none=True)
        loss.backward()
        grads.append(eng.G32.clone())
        if stock:
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        losses.append(loss.detach().reshape(1).clone())
    torch.cuda.synchronize()
    return torch.cat(losses), grads, eng.W32.clone()


def _reset(model, w0, rng0):
    eng = model.engine
    eng.W32.copy_(w0)
    eng.mark_weights_dirty()
    eng.set_rng_state(rng0)
    model.zero_grad(set_to_none=True)
    torch.cuda.synchronize()


def _prepare(name):
    cfg, sd, batches = _case(name)
    model = _make_model(cfg, sd)
    eng = model._ensure_engine(torch.device("cuda"))
    return cfg, model, batches, eng.W32.clone(), eng.rng_state()


def _assert_same_run(r0, r1, what):
    (l0, g0, w0), (l1, g1, w1) = r0, r1
    assert _same_bits(l0, l1), (what, l0.tolist(), l1.tolist())
    for i, (a, b) in enumerate(zip(g0, g1)):
        assert _same_bits(a, b), (what, "gradients of step", i, (a != b).sum().item())
    assert _same_bits(w0, w1), (what, "parameters", (w0 != w1).sum().item())


def _hashes(run):
    losses, grads, w = run
    h = lambda t: hashlib.sha256(_bits(t).cpu().numpy().tobytes()).hexdigest()
    return dict(loss=h(losses), grads=[h(g) for g in grads], params=h(w))


def test_benchmark_step_is_bitwise_reproducible(det):
    """The benchmarked configuration (Yelp, 16 businesses, 12 + 12 layers, dropout 0.1) with FusedAdamW: three steps from the
    same state give the same loss, gradient arena and parameters bit for bit — twice with plain launches (allocator cache and
    on-chip memory poisoned in between), with graph replay, and in a second Python process."""
    cfg, model, batches, w0, rng0 = _prepare("yelp_b16")
    runs = []
    for graph in (False, False, True):
        _poison()
        _reset(model, w0, rng0)
        runs.append(_run_steps(model, cfg, batches, graph=graph))
    assert torch.isfinite(runs[0][0]).all() and runs[0][0][0] != runs[0][0][2]
    _assert_same_run(runs[0], runs[1], "plain twice")
    _assert_same_run(runs[0], runs[2], "plain vs graph replay")
    ent = next(iter(model.engine._graphs.values()))
    assert "fwd" in ent and "bwd" in ent                        # steps 2 and 3 were replays
    mine = _hashes(runs[0])
    del model, runs
    torch.cuda.empty_cache()
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "yelp_b16"], cwd=ROOT, env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=1800)
    assert p.returncode == 0, p.stderr[-4000:]
    other = json.loads(p.stdout.strip().splitlines()[-1])
    assert other == mine


@pytest.mark.parametrize("name,stock", [("amazon_b8", False), ("small_text", False), ("small_img", False),
                                        ("small_table_yelp", False), ("small_table_amazon", False), ("small_yelp_gates_open", True)])
def test_smaller_steps_are_bitwise_reproducible(det, name, stock):
    """Amazon shape, text-only, image stage, table stages; the last case with torch's AdamW + clip_grad_norm_ instead of
    FusedAdamW.  Plain launches twice (poisoned in between) and graph replay: bit for bit."""
    cfg, model, batches, w0, rng0 = _prepare(name)
    runs = []
    for graph in (False, False, True):
        _poison()
        _reset(model, w0, rng0)
        runs.append(_run_steps(model, cfg, batches, graph=graph, stock=stock))
    _assert_same_run(runs[0], runs[1], "plain twice")
    _assert_same_run(runs[0], runs[2], "plain vs graph replay")


def test_graph_replay_across_encoder_frames(det):
    """Batches whose longest review changes from step to step run on different encoder frames, each with its own recorded
    graphs, replayed in turn.  The ordered scratch is sized for every frame of the shape before the first graph is recorded (it
    never moves afterwards), and every replayed step equals the same step with plain launches bit for bit."""
    from multimodalsum_b200.synth import make_batch
    cfg, model, _, w0, rng0 = _prepare("small_yelp_gates_open")
    batches = [make_batch(cfg, 3, seed=90 + hi, n_reviews=4, max_imgs=3, len_range=(20, hi)).with_length_hint().to("cuda")
               for hi in (70, 100, 30)]
    order = [0, 1, 2, 0, 1, 2, 0, 2, 1]
    eng = model.engine

    def run(graph):
        _reset(model, w0, rng0)
        eng.enable_graph(graph)
        out, ptrs, frames = [], set(), set()
        for i in order:
            a, kw = _batch_args(cfg, batches[i])
            loss = model(*a, **kw)[0]
            model.zero_grad(set_to_none=True)
            loss.backward()
            torch.cuda.synchronize()
            out.append((loss.detach().clone(), eng.G32.clone()))
            ptrs.add((eng.det_ws.data_ptr(), eng.det_ws_side.data_ptr()))
            frames.add(eng.ws["S_enc"] if not graph else None)
        return out, ptrs, frames

    plain, _, frames = run(False)
    assert len(frames) == 3, frames
    graphed, ptrs, _ = run(True)
    assert len(ptrs) == 1
    assert len(eng._graphs) == 3 and all("bwd" in e for e in eng._graphs.values())
    for i, ((l0, g0), (l1, g1)) in enumerate(zip(plain, graphed)):
        assert _same_bits(l0, l1) and _same_bits(g0, g1), i


@pytest.mark.parametrize("name", ["small_yelp", "small_yelp_gates_open", "small_amazon", "small_text", "small_img",
                                  "small_table_yelp", "small_table_amazon", "full_yelp_b1_gates_open"])
def test_deterministic_step_matches_reference(name):
    """Parity of the ordered step with the reference goldens and the fp32 oracle, at the tolerances of test_step_gpu.py."""
    from golden_util import load_golden
    from oracle import mmsum_oracle as OR
    from test_step_gpu import _check, _run_cuda_step
    gold = load_golden(name)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    with deterministic(True):
        loss, grads, model = _run_cuda_step(gold)
        assert model.engine.det
    grads = {n: g.cpu() for n, g in grads.items()}
    del model
    torch.cuda.empty_cache()
    _, ograds, _ = OR.step_loss_and_grads(gold["sd"], gold["cfg"], gold["batch"], gold["label_smoothing"], dtype=torch.float32,
                                          device="cuda")
    _check(gold, loss, grads, {n: g.cpu() for n, g in ograds.items()})


# ============================================================================================================ switch plumbing
class _Recorder:
    """Stands in for the loaded library and records the name of every C-ABI call."""

    def __init__(self, real):
        self.real, self.calls = real, []

    def __getattr__(self, name):
        fn = getattr(self.real, name)

        def call(*a):
            self.calls.append(name)
            return fn(*a)
        return call


@contextlib.contextmanager
def _recording():
    from multimodalsum_b200 import _lib
    real = _lib.lib()
    rec = _Recorder(real)
    _lib._lib = rec
    try:
        yield rec
    finally:
        _lib._lib = real


def test_switch_toggles_between_steps():
    """off -> on -> off -> on between steps of one model: the ordered entry points run exactly in the steps taken with the switch
    on; the off steps call the library in the same sequence before and after an on step; and the graph keys keep the modes
    apart."""
    from multimodalsum_b200 import ops
    cfg, model, batches, w0, rng0 = _prepare("small_yelp_gates_open")
    b = batches[0]
    a, kw = _batch_args(cfg, b)

    def step(on):
        with deterministic(on), _recording() as rec:        # (the workspace-size query launches nothing and is left out)
            before = dict(ops.ORDERED_CALLS)
            loss = model(*a, **kw)[0]
            model.zero_grad(set_to_none=True)
            loss.backward()
            torch.cuda.synchronize()
        delta = {k: v - before.get(k, 0) for k, v in ops.ORDERED_CALLS.items() if v != before.get(k, 0)}
        return [c for c in rec.calls if c != "mmsum_gemm_ordered_workspace"], delta, model.engine.G32.clone()

    seqs = []
    for on in (False, True, False, True):
        _reset(model, w0, rng0)
        calls, delta, g = step(on)
        seqs.append((calls, delta, g))
        if on:
            assert set(delta) == {"gemm", "add_ln_bwd", "colsum", "embed_ln_bwd"}, delta
            assert delta["embed_ln_bwd"] == 2 and "mmsum_embed_ln_bwd" not in calls and "mmsum_add_ln_bwd" not in calls
            assert "mmsum_colsum" not in calls
        else:
            assert delta == {} and not any(c.endswith("_ordered") for c in calls)
    assert seqs[0][0] == seqs[2][0]                                   # the off step is unchanged by an on step before it
    assert seqs[1][0] == seqs[3][0] and _same_bits(seqs[1][2], seqs[3][2])
    # graph mode: a graph recorded in one mode is never replayed in the other
    eng = model.engine
    _reset(model, w0, rng0)
    eng.enable_graph(True)
    for on in (False, False, True, True, False, True):
        with deterministic(on):
            loss = model(*a, **kw)[0]
            model.zero_grad(set_to_none=True)
            loss.backward()
            torch.cuda.synchronize()
            assert eng.det == on
    keys = list(eng._graphs)
    assert sorted(k[-1] for k in keys) == [False, True]
    assert all("fwd" in eng._graphs[k] and "bwd" in eng._graphs[k] for k in keys)


def test_public_paths_run_under_the_switch(det):
    """Sub-module forwards, the inference surface and beam / sampled generate() run with the switch on (no torch op of the host
    glue raises), and give what they give with it off (their reductions are already in a fixed order)."""
    from golden_util import load_golden
    from multimodalsum_b200.modules import LabelSmoothingLoss, MultimodalSum, TextSupervised, YelpTableEncoder
    gold = load_golden("small_yelp_gates_open")
    cfg, sd = gold["cfg"], gold["sd"]
    model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg)
    model.load_state_dict(sd, strict=False)
    model = model.cuda().eval()
    b = gold["batch"].to("cuda")
    B, R, S = b.reviews.shape

    def surface():
        out = {}
        with torch.no_grad():
            out["enc"] = model.bart_model.model.encoder(input_ids=b.reviews.view(B * R, S), attention_mask=b.reviews_mask.view(B * R, S))[0]
            out["tab"] = model.table_encoder(b.field, b.field_value)[0]
            out["img"] = model.img_encoder(b.img)
            _, th, tm, tabh, tabm, ih, im = model.get_multimodal_outputs(b.reviews, b.reviews_mask, b.field, b.field_value, b.img,
                                                                         b.img_mask)
            rd = torch.zeros(B, 1, device="cuda")
            out["logits"] = model.bart_model(th[:, 1:], tm[:, 1:], tabh, tabm, ih, im, rating_diff=rd, labels=b.reviews[:, 0])[0]
            out["beam"] = model.bart_model.generate(th, tm, tabh, tabm, ih, im, rating_diff=rd, num_beams=4, max_length=24,
                                                    no_repeat_ngram_size=3, early_stopping=True)
            torch.manual_seed(3)
            out["sample"] = model.bart_model.generate(th, tm, tabh, tabm, ih, im, rating_diff=rd, do_sample=True, top_p=0.9,
                                                      num_return_sequences=2, max_length=24)
        pred = torch.randn(64, 777, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)).requires_grad_(True)
        loss = LabelSmoothingLoss(777, smoothing=0.1)(pred, torch.arange(64, device="cuda"))
        loss.backward()
        out["ls"], out["ls_grad"] = loss.detach(), pred.grad
        return out

    on = surface()
    with deterministic(False):
        off = surface()
    for k in on:
        assert on[k].shape == off[k].shape and torch.equal(on[k], off[k]), k
    tgold = load_golden("small_text")
    tm_ = TextSupervised(config=tgold["cfg"], label_smoothing=None)
    tm_.load_state_dict(tgold["sd"], strict=False)
    tm_ = tm_.cuda().eval()
    tb = tgold["batch"].to("cuda")
    B, R, S = tb.reviews.shape
    with torch.no_grad():
        th = tm_.bart_model.model.encoder(input_ids=tb.reviews.view(B * R, S), attention_mask=tb.reviews_mask.view(B * R, S))[0]
        th = th.reshape(B, R, S, -1)
        ids = tm_.bart_model.generate(th[:, 1:], tb.reviews_mask[:, 1:], rating_diff=torch.zeros(B, 1, device="cuda"), num_beams=2,
                                      max_length=16)
    assert ids.shape[0] == B


if __name__ == "__main__":
    # second-process half of test_benchmark_step_is_bitwise_reproducible: the same three steps, hashes of the results
    torch.use_deterministic_algorithms(True)
    cfg_, model_, batches_, _, _ = _prepare(sys.argv[1])
    print(json.dumps(_hashes(_run_steps(model_, cfg_, batches_))))
