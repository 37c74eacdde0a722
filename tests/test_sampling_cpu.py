"""Sampling in generate() without a GPU: the score processing restated in generation.sample_scores against a line-by-line
transcription of the vendored transformers 3.0.2 functions the reference's _generate_no_beam_search calls, the argument
resolution, the host-side checks of mmsum_sample_token, and the n-best output of BeamSearch.finalize."""
import ctypes as C
import itertools

import pytest
import torch
import torch.nn.functional as F

from multimodalsum_b200 import _lib
from multimodalsum_b200 import generation as G


# ---- transformers 3.0.2 generation_utils.py, transcribed (only the batch_size * num_beams = N convention kept) ----------
def hf_enforce_repetition_penalty_(lprobs, batch_size, num_beams, prev_output_tokens, repetition_penalty):
    for i in range(batch_size * num_beams):
        for previous_token in set(prev_output_tokens[i].tolist()):
            # if score < 0 then repetition penalty has to multiplied to reduce the previous token probability
            if lprobs[i, previous_token] < 0:
                lprobs[i, previous_token] *= repetition_penalty
            else:
                lprobs[i, previous_token] /= repetition_penalty


def hf_calc_banned_ngram_tokens(prev_input_ids, num_hypos, no_repeat_ngram_size, cur_len):
    if cur_len + 1 < no_repeat_ngram_size:
        return [[] for _ in range(num_hypos)]
    generated_ngrams = [{} for _ in range(num_hypos)]
    for idx in range(num_hypos):
        gen_tokens = prev_input_ids[idx].tolist()
        generated_ngram = generated_ngrams[idx]
        for ngram in zip(*[gen_tokens[i:] for i in range(no_repeat_ngram_size)]):
            prev_ngram_tuple = tuple(ngram[:-1])
            generated_ngram[prev_ngram_tuple] = generated_ngram.get(prev_ngram_tuple, []) + [ngram[-1]]

    def _get_generated_ngrams(hypo_idx):
        start_idx = cur_len + 1 - no_repeat_ngram_size
        ngram_idx = tuple(prev_input_ids[hypo_idx, start_idx:cur_len].tolist())
        return generated_ngrams[hypo_idx].get(ngram_idx, [])

    return [_get_generated_ngrams(hypo_idx) for hypo_idx in range(num_hypos)]


def hf_postprocess_next_token_scores(scores, input_ids, no_repeat_ngram_size, bad_words_ids, cur_len, min_length, max_length,
                                     eos_token_id, repetition_penalty, batch_size, num_beams):
    if repetition_penalty != 1.0:
        hf_enforce_repetition_penalty_(scores, batch_size, num_beams, input_ids, repetition_penalty)
    if eos_token_id is not None and cur_len < min_length:
        scores[:, eos_token_id] = -float("inf")
    if no_repeat_ngram_size > 0:
        num_batch_hypotheses = batch_size * num_beams
        banned_batch_tokens = hf_calc_banned_ngram_tokens(input_ids, num_batch_hypotheses, no_repeat_ngram_size, cur_len)
        for i, banned_tokens in enumerate(banned_batch_tokens):
            scores[i, banned_tokens] = -float("inf")
    return scores


def hf_top_k_top_p_filtering(logits, top_k=0, top_p=1.0, filter_value=-float("Inf"), min_tokens_to_keep=1):
    if top_k > 0:
        top_k = min(max(top_k, min_tokens_to_keep), logits.size(-1))
        indices_to_remove = logits < torch.topk(logits, top_k)[0][..., -1, None]
        logits[indices_to_remove] = filter_value
    if top_p < 1.0:
        sorted_logits, sorted_indices = torch.sort(logits, descending=True)
        cumulative_probs = torch.cumsum(F.softmax(sorted_logits, dim=-1), dim=-1)
        sorted_indices_to_remove = cumulative_probs > top_p
        if min_tokens_to_keep > 1:
            sorted_indices_to_remove[..., :min_tokens_to_keep] = 0
        sorted_indices_to_remove[..., 1:] = sorted_indices_to_remove[..., :-1].clone()
        sorted_indices_to_remove[..., 0] = 0
        indices_to_remove = sorted_indices_to_remove.scatter(1, sorted_indices, sorted_indices_to_remove)
        logits[indices_to_remove] = filter_value
    return logits


def hf_sample_step_scores(next_token_logits, input_ids, cur_len, min_length, no_repeat_ngram_size, temperature, top_k, top_p,
                          repetition_penalty, eos):
    """The do_sample branch of _generate_no_beam_search up to the softmax (no adjust_logits_during_generation there)."""
    scores = hf_postprocess_next_token_scores(next_token_logits.clone(), input_ids, no_repeat_ngram_size, None, cur_len,
                                              min_length, 128, eos, repetition_penalty, input_ids.shape[0], 1)
    if temperature != 1.0:
        scores = scores / temperature
    return hf_top_k_top_p_filtering(scores, top_k=top_k, top_p=top_p)


def _case(V=97, N=6, cur_len=9, seed=0):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(N, V, generator=g) * 3.0                      # both signs, continuous: tie-free
    ids = torch.randint(3, 9, (N, cur_len), generator=g)              # few distinct ids: repeats and n-gram hits
    ids[:, 0] = 2
    ids[0, :6] = torch.tensor([2, 5, 6, 5, 6, 5])                    # a row that certainly bans a 2-gram / 3-gram continuation
    return logits, ids


@pytest.mark.parametrize("penalty", [1.0, 1.3])
@pytest.mark.parametrize("temperature", [0.7, 1.0, 1.5])
def test_restatement_matches_transformers_transcription(penalty, temperature):
    V = 97
    logits, ids = _case(V)
    cur_len = ids.shape[1]
    for top_k, top_p, min_length, ngram in itertools.product((0, 1, 50, V + 5), (1.0, 0.9, 0.3, 0.0), (0, 20), (0, 2, 3)):
        ref = hf_sample_step_scores(logits, ids, cur_len, min_length, ngram, temperature, top_k, top_p, penalty, 2)
        got = G.sample_scores(logits, ids, cur_len, min_length, ngram, temperature, top_k, top_p, penalty, 2)
        what = (top_k, top_p, min_length, ngram)
        assert torch.equal(torch.isfinite(ref), torch.isfinite(got)), what
        assert torch.equal(torch.softmax(ref, -1), torch.softmax(got, -1)), what
        if top_k == 1 or top_p == 0.0:
            assert int(torch.isfinite(got).sum(-1).max()) == 1, what
    assert torch.isinf(G.sample_scores(logits, ids, cur_len, 20, 0, 1.0, 0, 1.0, 1.0, 2)[:, 2]).all()


def test_restatement_tie_rules():
    """Ties at the k-th value survive top-k; inside top-p, equal scores are ranked by token id."""
    s = torch.tensor([[1.0, 3.0, 2.0, 2.0, 0.0, 2.0]])
    ids = torch.full((1, 1), 2)
    got = G.sample_scores(s, ids, 1, 0, 0, 1.0, 2, 1.0, 1.0, 2)
    assert torch.isfinite(got[0]).tolist() == [False, True, True, True, False, True]
    flat = torch.zeros(1, 8)
    got = G.sample_scores(flat, ids, 1, 0, 0, 1.0, 0, 0.3, 1.0, 2)   # masses 1/8 each: 0, 1/8, 2/8 <= 0.3 -> ids 0, 1, 2 kept
    assert torch.isfinite(got[0]).tolist() == [True, True, True] + [False] * 5


def test_defaults_and_validation():
    r = G.resolve_generate_args
    beam = dict(num_beams=4, max_length=60, min_length=0, no_repeat_ngram_size=3, early_stopping=True)
    # the beam-search argument set is exactly what it was before sampling existed
    assert r(beam) == dict(beam, length_penalty=1.0, use_cache=True)
    assert r(dict(beam, do_sample=False, num_return_sequences=1, top_k=None, temperature=None)) == r(beam)
    a = r(dict(do_sample=True))
    assert (a["num_beams"], a["temperature"], a["top_k"], a["top_p"], a["repetition_penalty"], a["num_return_sequences"]) == \
        (1, 1.0, 50, 1.0, 1.0, 1)
    assert r(dict(beam, num_return_sequences=2))["num_return_sequences"] == 2
    for bad in (dict(do_sample=True, temperature=0.0), dict(do_sample=True, temperature=-1.0), dict(do_sample=True, top_k=-1),
                dict(do_sample=True, top_k=2.5), dict(do_sample=True, top_p=1.5), dict(do_sample=True, top_p=-0.1),
                dict(do_sample=True, repetition_penalty=0.9), dict(do_sample=True, num_return_sequences=0),
                dict(num_beams=1, num_return_sequences=2), dict(num_beams=4, num_return_sequences=5),
                dict(temperature=0.0)):
        with pytest.raises(ValueError):
            r(bad)
    for bad, word in ((dict(do_sample=True, num_beams=4), "beam sampling"), (dict(bad_words_ids=[[5]]), "bad_words_ids"),
                      (dict(do_sample=True, bad_words_ids=[[5]]), "bad_words_ids"),
                      (dict(num_beams=4, repetition_penalty=1.2), "repetition_penalty"),
                      (dict(num_beams=1, repetition_penalty=1.2), "repetition_penalty")):
        with pytest.raises(NotImplementedError, match=word):
            r(bad)


def test_sample_token_rejects_invalid_arguments_on_the_host():
    """Every bad argument of mmsum_sample_token comes back as -1 before any launch (one bad argument per call)."""
    L = _lib.lib()
    P = C.c_void_p(4096)
    ok = dict(logits=P, ld=C.c_int64(50268), rows=256, V=50265, ids=P, L=128, cur_dev=P, seed_dev=P, min_length=0, ngram=3,
              eos=2, pad=1, temperature=C.c_float(1.0), top_k=50, top_p=C.c_float(0.9), penalty=C.c_float(1.0), unfinished=P,
              next_tok32=P, stream=None)
    order = list(ok)
    bads = [dict(logits=None), dict(ids=None), dict(cur_dev=None), dict(seed_dev=None), dict(unfinished=None),
            dict(rows=0), dict(V=16), dict(V=60000, ld=C.c_int64(60000)), dict(L=1), dict(L=161),
            dict(ld=C.c_int64(50266)), dict(ld=C.c_int64(1000)), dict(logits=C.c_void_p(4100)),
            dict(ngram=-1), dict(ngram=9), dict(min_length=-1), dict(eos=50265), dict(pad=-1),
            dict(temperature=C.c_float(0.0)), dict(temperature=C.c_float(float("nan"))), dict(top_k=-1),
            dict(top_p=C.c_float(1.01)), dict(top_p=C.c_float(-0.5)), dict(penalty=C.c_float(0.5))]
    for bad in bads:
        args = dict(ok, **bad)
        assert L.mmsum_sample_token(*[args[k] for k in order]) == -1, bad


def _run_beams(B, k, V, L, seed, eos_bias=1.5):
    g = torch.Generator().manual_seed(seed)
    bs = G.BeamSearch(B, V, "cpu", k, L, 0, 1.0, 2, False, 1, 0, 2)
    while bs.cur_len < L:
        logits = torch.randn(B * k, V, generator=g) * 2
        logits[:, 2] += eos_bias                     # EOS likely enough that pools fill before the frame ends
        bs.advance(logits)
        if bool(bs.done.all()):
            break
    return bs


# (14, 3, 1.5): every width equal; (30, 2, 1.0): the n-best output is wider; (30, 1, 0.0): wider, and the n = 1 output had no
# closing EOS (all its hypotheses had one length)
@pytest.mark.parametrize("L,seed,eos_bias", [(14, 3, 1.5), (30, 2, 1.0), (30, 1, 0.0)])
@pytest.mark.parametrize("n", [2, 3, 4])
def test_beam_finalize_n_best(n, L, seed, eos_bias):
    B, k, V = 5, 4, 40
    one = _run_beams(B, k, V, L, seed, eos_bias).finalize()
    bs = _run_beams(B, k, V, L, seed, eos_bias)
    out = bs.finalize(n)
    assert out.shape[0] == B * n
    W = one.shape[1]
    assert torch.equal(out[::n, :W], one)
    # the padding rule of the reference's output: a hypothesis holds no EOS after the start token; when lengths differ, every
    # row shorter than the frame gets exactly one closing EOS at its own length, then pad
    any_eos = bool((out[:, 1:] == 2).any())
    for r in out:
        e = ((r[1:] == 2).nonzero().flatten() + 1).tolist()
        assert len(e) <= 1, r.tolist()
        if e:
            assert bool((r[e[0] + 1:] == 1).all()), r.tolist()
        else:
            assert out.shape[1] == L or not any_eos, r.tolist()
    # beyond the n = 1 width, row i*n continues with pad, or with its closing EOS when the n = 1 output had none
    for i in range(B):
        tail = out[i * n, W:]
        if tail.numel() == 0:
            continue
        if bool((one[i, 1:] == 2).any()):
            assert bool((tail == 1).all()), tail.tolist()
        else:
            assert int(tail[0]) == 2 and bool((tail[1:] == 1).all()), tail.tolist()
    sc = bs.out_scores.view(B, n)
    assert bool((sc[:, 1:] <= sc[:, :-1]).all())
    with pytest.raises(ValueError):
        _run_beams(B, k, V, L, seed, eos_bias).finalize(k + 1)


def test_cpu_sampling_loop_bookkeeping():
    """sample_search on the CPU tensor path: the start token, pad after a row's EOS, the width of the reference's output
    (the step in which the last row appended EOS), and no EOS before min_length."""
    B, n, V = 3, 2, 30
    g = torch.Generator().manual_seed(4)

    def logits_fn(ids):
        z = torch.randn(ids.shape[0], V, generator=g)
        z[:, 2] += 0.8 * ids.shape[1]                 # EOS more and more likely
        return z

    torch.manual_seed(0)
    out = G.sample_search(logits_fn, B, V, "cpu", num_return_sequences=n, max_length=40, min_length=4, no_repeat_ngram_size=2,
                          top_k=10, top_p=0.9, temperature=0.8, repetition_penalty=1.2)
    assert out.shape[0] == B * n and (out[:, 0] == 2).all()
    first = [(r[1:] == 2).nonzero()[0, 0].item() + 1 for r in out]
    assert min(first) >= 4 and max(first) == out.shape[1] - 1
    for r, f in zip(out, first):
        assert (r[f + 1:] == 1).all()
