"""The device sampler (csrc/sample_sm100.cu) and generate(do_sample=True) on the GPU, against generation.sample_scores (the
restatement of the vendored transformers 3.0.2 score processing, checked on the CPU in test_sampling_cpu.py).

All randomness comes from fixed seeds, so the statistical checks are deterministic; their bounds sit at about p = 1e-4 for a
fair sampler."""
import itertools
import math

import numpy as np
import pytest
import torch
from scipy import stats

from multimodalsum_b200 import generation as G
from multimodalsum_b200 import ops
from multimodalsum_b200.synth import ModelConfig, make_batch, make_state_dict

pytestmark = pytest.mark.gpu

V = 50265
EOS, PAD = 2, 1


def _buffers(rows, L=128, cur=20, seed=7, hist_range=(3, 40)):
    g = torch.Generator().manual_seed(seed)
    ids = torch.full((rows, L), PAD, dtype=torch.long)
    ids[:, 0] = EOS
    ids[:, 1:cur] = torch.randint(*hist_range, (rows, cur - 1), generator=g)
    return ids.cuda(), torch.tensor([cur], dtype=torch.long, device="cuda")


def _logits(rows, seed=0, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    z = torch.empty(rows, (V + 3) // 4 * 4)
    z[:, :V] = torch.randn(rows, V, generator=g) * scale
    return z.cuda()[:, :V]


def _sample(logits, ids, cur_t, seed, min_length=0, ngram=0, temperature=1.0, top_k=0, top_p=1.0, penalty=1.0, next32=None):
    rows = logits.shape[0]
    unf = torch.ones(rows, dtype=torch.uint8, device="cuda")
    sd = torch.tensor([seed], dtype=torch.long, device="cuda")
    ops.sample_token(logits, V, ids, cur_t, sd, min_length, ngram, EOS, PAD, temperature, top_k, top_p, penalty, unf, next32)
    return ids[:, int(cur_t.item())].clone(), unf


def test_kept_set_is_exact():
    """[256, 50265] tie-free logits with token histories: every drawn token lies in the restatement's kept set over the
    grid of the CPU test; with top_k = 1 or top_p = 0 the draw is the arg-max of the processed scores."""
    rows, cur = 256, 20
    logits = _logits(rows)
    ids0, cur_t = _buffers(rows, cur=cur)
    grid = list(itertools.product((0, 1, 50, V + 5), (1.0, 0.9, 0.3, 0.0), (0.7, 1.0, 1.5), (1.0, 1.3)))
    for i, (top_k, top_p, temperature, penalty) in enumerate(grid):
        min_length, ngram = (30, 3) if i % 2 else (0, 0)
        ids = ids0.clone()
        tok, _ = _sample(logits, ids, cur_t, 1000 + i, min_length, ngram, temperature, top_k, top_p, penalty)
        ref = G.sample_scores(logits, ids0, cur, min_length, ngram, temperature, top_k, top_p, penalty, EOS)
        kept = torch.isfinite(ref)
        what = (top_k, top_p, temperature, penalty, min_length, ngram)
        assert bool(kept.gather(1, tok[:, None]).all()), what
        if top_k == 1 or top_p == 0.0:
            assert torch.equal(tok, ref.argmax(-1)), what


def _chi2_case(row_logits, steps=64, rows=1024, **kw):
    """One row replicated over `rows` rows, `steps` launches with the step counter advanced -> counts [V] and the
    restatement's probabilities (float64)."""
    logits = row_logits.expand(rows, -1)
    buf = torch.empty(rows, (V + 3) // 4 * 4, device="cuda")
    buf[:, :V] = logits
    logits = buf[:, :V]
    ids, cur_t = _buffers(rows, L=steps + 2, cur=1)
    counts = torch.zeros(V, dtype=torch.long, device="cuda")
    for s in range(steps):
        tok, _ = _sample(logits, ids, cur_t, 12345, **kw)
        counts += torch.bincount(tok, minlength=V)
        cur_t += 1
    ref = G.sample_scores(row_logits[None], ids[:1], 1, 0, 0, kw.get("temperature", 1.0), kw.get("top_k", 0),
                          kw.get("top_p", 1.0), 1.0, EOS)[0]
    return counts.cpu(), torch.softmax(ref.double(), -1).cpu(), torch.isfinite(ref).cpu()


def _assert_chi2(counts, p, kept):
    n = int(counts.sum())
    assert int(counts[~kept].sum()) == 0
    exp = p * n
    big = exp >= 5
    obs = torch.cat([counts[big].double(), counts[~big].double().sum()[None]])
    e = torch.cat([exp[big], exp[~big].sum()[None]])
    keep = e > 0
    obs, e = obs[keep], e[keep]
    chi2 = float(((obs - e) ** 2 / e).sum())
    df = int(keep.sum()) - 1
    assert chi2 < stats.chi2.ppf(1 - 1e-4, df), (chi2, df)


@pytest.mark.parametrize("case", ["top_k50", "nucleus0.9", "t1.5_30live"])
def test_distribution_matches_restatement(case):
    g = torch.Generator().manual_seed(3)
    row = (torch.randn(V, generator=g) * 3).cuda()
    if case == "top_k50":
        kw = dict(top_k=50)
    elif case == "nucleus0.9":
        kw = dict(top_k=0, top_p=0.9)
    else:
        live = torch.randperm(V, generator=g)[:30].cuda()
        r = torch.full_like(row, float("-inf"))
        r[live] = row[live] / 3
        row, kw = r, dict(top_k=0, temperature=1.5)
    counts, p, kept = _chi2_case(row, **kw)
    _assert_chi2(counts, p, kept)


def test_counter_semantics():
    """A draw is a function of (seed, row, step): the same at 1, 7 and 256 rows; different rows of one step agree at the rate
    sum(p^2) of independent draws."""
    g = torch.Generator().manual_seed(4)
    row = (torch.randn(V, generator=g) * 3).cuda()
    def run(rows, steps):
        buf = torch.empty(rows, (V + 3) // 4 * 4, device="cuda")
        buf[:, :V] = row
        ids, cur_t = _buffers(rows, L=steps + 2, cur=1)
        out = []
        for _ in range(steps):
            out.append(_sample(buf[:, :V], ids, cur_t, 99, top_k=20)[0])
            cur_t += 1
        return torch.stack(out, 1)
    a256, a7, a1 = run(256, 64), run(7, 64), run(1, 64)
    assert torch.equal(a256[:7], a7) and torch.equal(a7[:1], a1)
    p = torch.softmax(G.sample_scores(row[None], torch.full((1, 1), EOS, device="cuda"), 1, 0, 0, 1.0, 20, 1.0, 1.0,
                                      EOS)[0].double(), -1)
    q = float((p * p).sum())
    pairs = (a256[0::2] == a256[1::2]).double()
    n = pairs.numel()
    rate = float(pairs.mean())
    assert abs(rate - q) < 3.9 * math.sqrt(q * (1 - q) / n), (rate, q)
    assert not torch.equal(a256[:, 0], a256[:, 1])                  # the step counter changes the draw


# ---- end to end ------------------------------------------------------------------------------------------------
def _setup(name):
    import json
    import os
    from golden_util import GOLDEN_DIR
    from multimodalsum_b200.generation import Generator
    from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    case = json.loads(str(z["case"]))
    cfg = ModelConfig(**case["cfg"])
    sd = make_state_dict(cfg, **case["sd"])
    bk = dict(case["batch"])
    batch = make_batch(cfg, bk.pop("B"), **bk).to("cuda")
    model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg)
    model.load_state_dict(sd, strict=False)
    model = model.cuda().eval()
    return Generator(model), model, cfg, batch, case["gen"], torch.from_numpy(z["tokens"])


def _greedy_no_beam(gen, st, cfg, N, max_length, min_length, ngram):
    """_generate_no_beam_search driven by last_logits, arg-max of the processed scores (what top_k = 1 samples)."""
    ids = torch.full((N, 1), cfg.eos_token_id, dtype=torch.long, device="cuda")
    unf = torch.ones(N, dtype=torch.bool, device="cuda")
    rd = torch.zeros(N, device="cuda")
    while ids.shape[1] < max_length:
        cur = ids.shape[1]
        scores = G.sample_scores(gen.last_logits(st, ids, rd), ids, cur, min_length, ngram, 1.0, 0, 1.0, 1.0, cfg.eos_token_id)
        tok = torch.where(unf, scores.argmax(-1), torch.full_like(unf, cfg.pad_token_id, dtype=torch.long))
        ids = torch.cat([ids, tok[:, None]], 1)
        unf &= tok != cfg.eos_token_id
        if not bool(unf.any()):
            break
    return ids


@pytest.mark.parametrize("use_cache", [True, False])
def test_top1_sampling_equals_greedy_no_beam_loop(use_cache):
    gen, model, cfg, b, gk, _ = _setup("gen_small_yelp_biased")
    args = (b.reviews, b.reviews_mask, b.field, b.field_value, b.img, b.img_mask)
    B = b.reviews.shape[0]
    kw = dict(max_length=gk["max_length"], min_length=4, no_repeat_ngram_size=gk["no_repeat_ngram_size"])
    st = gen.encode(*args, 1)
    ref = _greedy_no_beam(gen, st, cfg, B, **{k: kw[k] for k in ("max_length", "min_length")},
                          ngram=kw["no_repeat_ngram_size"])
    out = gen.generate(*args, num_beams=1, do_sample=True, top_k=1, use_cache=use_cache, **kw)
    assert torch.equal(out, ref), (out.tolist(), ref.tolist())
    out3 = gen.generate(*args, num_beams=1, do_sample=True, top_k=1, num_return_sequences=3, use_cache=use_cache, **kw)
    assert out3.shape[0] == 3 * B
    for i in range(3):
        assert torch.equal(out3[i::3], ref)


def test_sampling_is_reproducible_under_manual_seed():
    gen, model, cfg, b, gk, _ = _setup("gen_small_yelp_biased")
    args = (b.reviews, b.reviews_mask, b.field, b.field_value, b.img, b.img_mask)
    # this model's logits have wide margins (it is the tie-free beam case): a high temperature spreads the draws
    kw = dict(num_beams=1, do_sample=True, top_k=0, top_p=0.95, temperature=20.0, num_return_sequences=4, max_length=20)
    torch.manual_seed(11)
    a = gen.generate(*args, **kw)
    torch.manual_seed(11)
    b2 = gen.generate(*args, **kw)
    assert gen.last_used_graph
    assert torch.equal(a, b2)
    assert a.data_ptr() != b2.data_ptr()                          # results are copies, not views of the plan's buffers
    torch.manual_seed(12)
    c = gen.generate(*args, **kw)
    W = max(a.shape[1], c.shape[1])
    padw = lambda t: torch.nn.functional.pad(t, (0, W - t.shape[1]), value=cfg.pad_token_id)
    assert not torch.equal(padw(a), padw(c))


def test_beam_n_best_kernel_equals_tensor_path():
    B, k, Vb, L = 6, 4, 777, 16
    outs = []
    for use_kernel in (True, False):
        g = torch.Generator().manual_seed(8)
        bs = G.BeamSearch(B, Vb, "cuda", k, L, 0, 1.0, 3, True, 1, 0, 2)
        bs.use_kernel = use_kernel
        buf = torch.empty(B * k, (Vb + 3) // 4 * 4, device="cuda")
        while bs.cur_len < L:
            z = torch.randn(B * k, Vb, generator=g) * 2
            z[:, 2] += 1.0
            buf[:, :Vb] = z.cuda()
            bs.advance(buf[:, :Vb])
        assert bs.kernel_path == use_kernel
        outs.append(bs.finalize(3))
    assert torch.equal(outs[0], outs[1])


def test_beam_n_best_first_row_is_todays_output():
    gen, model, cfg, b, gk, ref = _setup("gen_small_yelp_biased")
    args = (b.reviews, b.reviews_mask, b.field, b.field_value, b.img, b.img_mask)
    for n in (2, 4):
        out = gen.generate(*args, num_return_sequences=n, **gk)
        assert out.shape[0] == n * ref.shape[0]
        assert torch.equal(out[::n, :ref.shape[1]].cpu(), ref)


def test_sampler_ignores_stale_state():
    rows = 64
    logits = _logits(rows, seed=5)
    ids0, cur_t = _buffers(rows, cur=12)
    res = []
    for poison in (False, True):
        ids = ids0.clone()
        nxt = torch.full((rows,), -7, dtype=torch.int32, device="cuda")
        if poison:
            ids[:, 12:] = -(1 << 40)
            nxt.view(torch.float32).fill_(float("nan"))
            ops.debug_poison()
        tok, unf = _sample(logits, ids, cur_t, 77, 15, 3, 1.3, 50, 0.8, 1.2, nxt)
        res.append((tok, unf, nxt.clone(), ids[:, :13].clone()))
    for a, b in zip(*res):
        assert torch.equal(a, b)


def test_config5_shape_sampling():
    """64 businesses x 4 samples, BART-large widths (2 + 2 layers), top_p 0.9, no_repeat_ngram_size 3, min_length 10: the
    output is well formed, and teacher-forced along each row's own prefix (last_logits) every sampled token lies in the
    restatement's kept set, up to tokens within 0.1 nats of the top-p boundary (bf16: the sampler saw the cached decoder's
    logits)."""
    from multimodalsum_b200.generation import Generator
    from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
    B, n = 64, 4
    cfg = ModelConfig(dataset="yelp", encoder_layers=2, decoder_layers=2, dropout=0.0)
    sd = make_state_dict(cfg, seed=41, gates_open=True, logits_bias_std=1.0)
    batch = make_batch(cfg, B, seed=42, n_reviews=8, seq_len=158, len_range=(100, 150)).to("cuda")
    model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg)
    model.load_state_dict(sd, strict=False)
    model = model.cuda().eval()
    gen = Generator(model)
    args = (batch.reviews, batch.reviews_mask, batch.field, batch.field_value, batch.img, batch.img_mask)
    torch.manual_seed(5)
    out = gen.generate(*args, num_beams=1, do_sample=True, top_p=0.9, num_return_sequences=n, no_repeat_ngram_size=3,
                       min_length=10, max_length=128)
    N, W = out.shape
    assert N == B * n and W <= 128 and (out[:, 0] == EOS).all()
    eos_at = [(r[1:] == EOS).nonzero() for r in out.cpu()]
    for r, e in zip(out.cpu(), eos_at):
        if len(e):
            f = int(e[0, 0]) + 1
            assert f >= 10 and (r[f + 1:] == PAD).all()
        grams = [tuple(r[i:i + 3].tolist()) for i in range(W - 2) if PAD not in r[i:i + 3].tolist()]
        assert len(grams) == len(set(grams))
    st = gen.encode(*args, n)
    rd = torch.zeros(N, device="cuda")
    unf = torch.ones(N, dtype=torch.bool, device="cuda")
    outside = 0
    for t in range(1, W):
        ids = out[:, :t].contiguous()
        logits = gen.last_logits(st, ids, rd)
        proc = G.sample_scores(logits, ids, t, 10, 3, 1.0, 50, 0.9, 1.0, EOS)
        tok = out[:, t]
        s_tok = G.sample_scores(logits, ids, t, 10, 3, 1.0, 0, 1.0, 1.0, EOS).gather(1, tok[:, None])[:, 0]
        assert bool(torch.isfinite(s_tok[unf]).all()), t                      # bans (min length, n-grams) are exact
        kept = torch.isfinite(proc).gather(1, tok[:, None])[:, 0]
        floor = torch.where(torch.isfinite(proc), proc, torch.full_like(proc, float("inf"))).min(-1).values
        bad = unf & ~kept & (s_tok < floor - 0.1)
        assert not bool(bad.any()), (t, bad.nonzero().flatten().tolist())
        outside += int((unf & ~kept).sum())
        unf &= tok != EOS
    assert outside <= 0.01 * N * W


def test_signed_zeros_tie_as_equal_scores():
    """-0.0 and +0.0 are one score (torch compares them equal): with the k-th value a zero, zeros of both signs survive
    top-k and are drawn."""
    rows = 1024
    row = torch.full((V,), float("-inf"))
    row[10:13] = 0.5
    row[100:110] = 0.0
    row[200:210] = -0.0
    buf = torch.empty(rows, (V + 3) // 4 * 4, device="cuda")
    buf[:, :V] = row.cuda()
    ids, cur_t = _buffers(rows, L=8, cur=1)
    tok, _ = _sample(buf[:, :V], ids, cur_t, 5, top_k=5)
    ref = G.sample_scores(row[None].cuda(), ids[:1], 1, 0, 0, 1.0, 5, 1.0, 1.0, EOS)[0]
    assert bool(torch.isfinite(ref)[200:210].all())
    assert bool(torch.isfinite(ref).gather(0, tok).all())
    assert bool(((tok >= 200) & (tok < 210)).any())


def test_out_of_range_step_writes_nothing():
    """A step counter outside 1 <= cur < L leaves the history, the decoder input and the unfinished flags untouched."""
    rows, L = 8, 16
    logits = _logits(rows, seed=2)
    for cur in (0, L, L + 40):
        ids, _ = _buffers(rows, L=L, cur=L)
        before = ids.clone()
        cur_t = torch.tensor([cur], dtype=torch.long, device="cuda")
        unf = torch.ones(rows, dtype=torch.uint8, device="cuda")
        nxt = torch.full((rows,), -7, dtype=torch.int32, device="cuda")
        ops.sample_token(logits, V, ids, cur_t, torch.tensor([1], dtype=torch.long, device="cuda"), 0, 3, EOS, PAD, 1.0, 50, 0.9,
                         1.0, unf, nxt)
        torch.cuda.synchronize()
        assert torch.equal(ids, before) and bool((unf == 1).all()) and bool((nxt == -7).all()), cur


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_sampler_runs_on_every_device():
    """The shared-memory opt-in is made per device: sampling on one device and then another works on both."""
    out = []
    for d in range(torch.cuda.device_count()):
        with torch.cuda.device(d):
            logits = _logits(4, seed=1).to(f"cuda:{d}")
            ids = torch.full((4, 8), PAD, dtype=torch.long, device=f"cuda:{d}")
            ids[:, 0] = EOS
            cur_t = torch.tensor([1], dtype=torch.long, device=f"cuda:{d}")
            unf = torch.ones(4, dtype=torch.uint8, device=f"cuda:{d}")
            ops.sample_token(logits, V, ids, cur_t, torch.tensor([3], dtype=torch.long, device=f"cuda:{d}"), 0, 0, EOS, PAD, 1.0,
                             50, 1.0, 1.0, unf)
            out.append(ids[:, 1].cpu())
    for o in out[1:]:
        assert torch.equal(o, out[0])                   # same seed, same rows, same step: same draws on every device
