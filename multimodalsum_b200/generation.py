"""Beam-search generation (BASELINE config 5, SURVEY §8 row a16) and sampling on the CUDA kernels of the training step.

Reference: BartForMultiEncConditionalGeneration.generate / _generate_beam_search / adjust_logits_during_generation
(src/transformer/modeling_multimodalsum.py:2295-3101), postprocess_next_token_scores / calc_banned_ngram_tokens /
BeamHypotheses (src/transformer/generation_utils.py:57-99, 848-868, 948-993), driven by src/test.py:152-158.

Design (B200-first, not the reference's):
  * the multimodal memory is encoded ONCE and its cross-attention K|V is projected ONCE per decoder layer and kept
    UN-EXPANDED per business — all beams of a business attend to the same memory (the reference expands every memory
    num_beams times and re-gathers the expanded K/V cache with index_select at every token, :2598-2627, :3004-3010);
  * decoding is incremental (`Generator.step_logits`): only the newest token of every hypothesis runs through the
    decoder, on decode-shaped attention kernels (csrc/decode_sm100.cu: one query row per hypothesis, K|V streamed once
    per business and head for all beams; self-attention caches that never move, addressed through a slot table that the
    beam re-ranking permutes), and the ~200 launches of a step are replayed from one CUDA graph.  `last_logits`
    recomputes the whole prefix in a 128-position causal frame with the training kernels and is kept as the cross-check
    of the cached path; both run the layer forwards of `layers.py`, on different attention and embedding kernels;
  * the beam bookkeeping is VECTORISED OVER BUSINESSES AND RUNS ON THE DEVICE (`BeamSearch`): n-gram blocking, the
    top-2k candidate merge, the per-business hypothesis pools and the early-stopping flags are tensor ops without a
    single `.item()` / `.tolist()` in the token loop (the reference loops over batch x beam in Python with host syncs
    every token, :2933-2983).  Termination is polled every few tokens through a pinned flag; steps taken after every
    business is done cannot change the result (finished businesses no longer admit hypotheses).
  * sampling (`do_sample=True`, _generate_no_beam_search of the vendored transformers 3.0.2 generation_utils.py) runs the
    same token loop with `SampleSearch` in place of `BeamSearch`: one kernel per token (csrc/sample_sm100.cu) processes the
    scores, draws from a counter-based Philox stream and does the loop bookkeeping; `sample_scores` is its restatement.
Review frames up to 208 tokens are supported (src/test.py uses 158 / 118).
"""
import torch

from . import inference as INF
from . import layers as L
from . import ops

NEG = float("-inf")


class BeamSearch:
    """State of one batched beam search: `B` businesses x `k` beams, hypotheses of a business adjacent.

    Semantics of _generate_beam_search (do_sample=False) + BeamHypotheses, restated on tensors:
      pool_score / pool_tok / pool_len [B, k]   finished hypotheses per business, score = sum_logprobs / len**length_penalty;
                                                a new one enters while the pool is not full or when it beats the pool's worst,
                                                which it then replaces
      done [B]                                  pool full and (early_stopping or the pool's worst >= best running score)
    """

    def __init__(self, B, V, dev, num_beams, max_length, min_length, length_penalty, no_repeat_ngram_size, early_stopping,
                 pad, bos, eos):
        k = num_beams
        self.B, self.k, self.V, self.dev = B, k, V, dev
        self.max_length, self.min_length = max_length, min_length
        self.length_penalty, self.ngram, self.early_stopping = length_penalty, no_repeat_ngram_size, early_stopping
        self.pad, self.bos, self.eos = pad, bos, eos
        N = B * k
        self.ids = torch.full((N, max_length), pad, dtype=torch.long, device=dev)
        self.ids[:, 0] = eos                                  # decoder_start_token_id = 2 (cfg/bart-large.json)
        self.cur_len = 1
        bs = torch.zeros(B, k, device=dev)
        bs[:, 1:] = -1e9                                      # only the first beam of a business is live at the start
        self.beam_scores = bs.view(-1).contiguous()
        self.done = torch.zeros(B, dtype=torch.bool, device=dev)
        self.pool_score = torch.full((B, k), NEG, device=dev)
        self.pool_tok = torch.full((B, k, max_length), pad, dtype=torch.long, device=dev)
        self.pool_len = torch.zeros(B, k, dtype=torch.long, device=dev)
        self.pool_n = torch.zeros(B, dtype=torch.long, device=dev)
        self.rows = torch.arange(B, device=dev)
        self.slot_ids = torch.arange(k, device=dev)
        self.row0 = (self.rows * k)[:, None]
        self.scores_ext = torch.empty(N, V + 1, device=dev)   # column V absorbs the "nothing banned" scatter writes
        lt = lambda v: torch.tensor([v], dtype=torch.long, device=dev)
        self.cur_t = lt(1)                                    # current length as a device scalar (see advance)
        self.bos_t, self.eos_t, self.pad_t, self.v_col = lt(bos), lt(eos), lt(pad), lt(V)
        self.neg_t = torch.full((1,), NEG, device=dev)
        n = no_repeat_ngram_size
        self.ng_ar = torch.arange(max(n - 1, 0), device=dev)
        self.win_ar = torch.arange(max(max_length - n + 1, 0), device=dev)
        self.own = self.row0 + self.slot_ids[None, :]
        self.beam_idx = torch.arange(N, device=dev)
        self.next_tok = torch.zeros(N, dtype=torch.long, device=dev)
        self.cand_val = self.cand_tok = None
        self.use_kernel = True                                # fused beam kernels on CUDA (tests switch them off)
        self.kernel_path = False                              # set when a step went through the kernels
        self.dec_ids32 = self.dec_hist = None                 # optional decoder hooks (see attach_decoder)

    def reset(self):
        """Back to the start state, in place (the buffers are baked into a recorded CUDA graph)."""
        self.ids.fill_(self.pad)
        self.ids[:, 0] = self.eos
        self.cur_len = 1
        self.cur_t.fill_(1)
        bs = self.beam_scores.view(self.B, self.k)
        bs.zero_()
        bs[:, 1:] = -1e9
        self.done.zero_()
        self.pool_score.fill_(NEG)
        self.pool_tok.fill_(self.pad)
        self.pool_len.zero_()
        self.pool_n.zero_()
        self.kernel_path = False

    def attach_decoder(self, ids32, hist):
        """The incremental decoder's next-token input [N] (int32) and self-attention slot table [N, 128] (int32): the beam
        update kernel writes / permutes them directly, so no separate re-ordering pass is needed."""
        self.dec_ids32, self.dec_hist = ids32, hist

    # -- hypothesis pool --------------------------------------------------------------------------------
    def _admit(self, active, score, tokens, length):
        """Offer one hypothesis per business (rows where `active`) to the pools."""
        k = self.k
        filled = self.slot_ids[None, :] < self.pool_n[:, None]
        worst, worst_slot = torch.where(filled, self.pool_score, torch.full_like(self.pool_score, float("inf"))).min(dim=1)
        full = self.pool_n >= k
        accept = active & (~full | (score > worst))
        slot = torch.where(full, worst_slot, self.pool_n.clamp(max=k - 1))
        r = self.rows
        self.pool_score[r, slot] = torch.where(accept, score, self.pool_score[r, slot])
        self.pool_tok[r, slot] = torch.where(accept[:, None], tokens, self.pool_tok[r, slot])
        length = length if torch.is_tensor(length) else torch.full((1,), length, dtype=torch.long, device=self.dev)
        self.pool_len[r, slot] = torch.where(accept, length.expand_as(accept), self.pool_len[r, slot])
        self.pool_n += (accept & ~full).long()

    def _pool_worst(self):
        filled = self.slot_ids[None, :] < self.pool_n[:, None]
        return torch.where(filled, self.pool_score, torch.full_like(self.pool_score, 1e9)).min(dim=1).values

    # -- one token --------------------------------------------------------------------------------------
    def advance(self, logits):
        """logits: fp32 [N, V] next-token logits of the current prefixes.  Returns beam_idx [N] (hypothesis i continues
        hypothesis beam_idx[i]) for the decoder's cache re-ordering.

        Every shape is static and every piece of per-step state (`cur_t`, `ids`, `beam_scores`, `done`, the pools,
        `beam_idx`, `next_tok`) is a fixed device buffer updated in place: the current length enters as the device scalar
        `cur_t`, never as a Python value, so the whole update can be recorded once in a CUDA graph (together with the decoder
        step) and replayed for every token."""
        B, k, V, L = self.B, self.k, self.V, self.max_length
        cur = self.cur_t                                                           # long [1]
        if self.use_kernel and logits.is_cuda and 2 * k in (2, 4, 8, 16) and L <= 160 and logits.stride(0) % 4 == 0:
            # fused per-row kernel (csrc/beam_sm100.cu): forced tokens, log-softmax, bans, + beam score, top-2k of the row;
            # the top-2k of a business is then merged from its k x 2k row candidates
            if self.cand_val is None:
                self.cand_val = torch.empty(B * k, 2 * k, device=self.dev)
                self.cand_tok = torch.empty(B * k, 2 * k, device=self.dev, dtype=torch.int32)
            ops.beam_topk(logits, V, self.beam_scores, self.ids, cur, self.min_length, self.ngram, self.bos, self.eos, 2 * k,
                          self.cand_val, self.cand_tok)
            # ... and the per-business bookkeeping (pools, next beams, history / slot-table permutation) in a second kernel
            ops.beam_update(self.cand_val, self.cand_tok, self.ids, self.beam_scores, self.done, self.pool_score, self.pool_tok,
                            self.pool_len, self.pool_n, cur, self.beam_idx, self.next_tok, self.dec_ids32, self.dec_hist, B, k,
                            self.eos, self.pad, self.early_stopping, self.length_penalty)
            self.kernel_path = True
            cur.add_(1)
            self.cur_len += 1
            return self.beam_idx
        # adjust_logits_during_generation (:3084-3089): only BOS may follow the start token, only EOS may close the frame
        forced_now = (cur == 1) | (cur == L - 1)
        forced_tok = torch.where(cur == 1, self.bos_t, self.eos_t).expand(logits.shape[0], 1)
        forced_logits = torch.full_like(logits, NEG).scatter_(1, forced_tok, logits.gather(1, forced_tok))
        logits = torch.where(forced_now, forced_logits, logits)
        scores = self.scores_ext
        torch.log_softmax(logits, dim=-1, out=scores[:, :V])
        # postprocess_next_token_scores (generation_utils.py:57-99)
        if self.min_length > 0:
            scores[:, self.eos] = torch.where(cur < self.min_length, self.neg_t, scores[:, self.eos])
        n = self.ngram
        if n > 0 and L >= n:
            # calc_banned_ngram_tokens (:848-868): a token is banned when it would complete an n-gram already in the prefix.
            # windows over the whole frame; window i is real when it ends inside the prefix (i <= cur - n)
            win = self.ids.unfold(1, n, 1)                                          # [N, L-n+1, n]
            sfx = self.ids.gather(1, (cur - n + 1 + self.ng_ar).clamp(min=0)[None, :].expand(self.ids.shape[0], -1))
            hit = (win[:, :, :n - 1] == sfx[:, None, :]).all(dim=-1) & (self.win_ar <= cur - n)[None, :]
            scores.scatter_(1, torch.where(hit, win[:, :, n - 1], self.v_col), NEG)
        cand = (scores[:, :V] + self.beam_scores[:, None]).view(B, k * V)
        cs, ci = torch.topk(cand, 2 * k, dim=1, largest=True, sorted=True)
        return self._update(cs, ci % V, self.row0 + ci // V)

    def _update(self, cs, tok, src):
        """cs / tok / src [B, 2k]: score, token and effective (global) beam index of the 2k best continuations per business."""
        k, cur = self.k, self.cur_t
        is_eos = tok == self.eos
        # finished candidates among the first k ranks enter the pool of their business (:2949-2957)
        live = ~self.done
        norm = cur.to(cs.dtype) ** self.length_penalty
        for r in range(k):
            self._admit(is_eos[:, r] & live, cs[:, r] / norm, self.ids[src[:, r]], cur)
        # the first k unfinished candidates, in rank order, are the next beams (:2958-2966)
        order = torch.argsort(is_eos.long(), dim=1, stable=True)[:, :k]
        nscore, ntok, nsrc = cs.gather(1, order), tok.gather(1, order), src.gather(1, order)
        # is_done (generation_utils.py:980-993), evaluated with the best candidate of this step
        if self.early_stopping:
            finished = self.pool_n >= k
        else:
            finished = (self.pool_n >= k) & (self._pool_worst() >= cs[:, 0] / norm)
        # businesses that were already done keep dummy beams (score 0, pad token); their rows are never read again
        nscore = torch.where(live[:, None], nscore, torch.zeros_like(nscore))
        ntok = torch.where(live[:, None], ntok, self.pad_t)
        nsrc = torch.where(live[:, None], nsrc, self.own)
        self.done.logical_or_(finished)
        self.beam_idx.copy_(nsrc.reshape(-1))
        self.next_tok.copy_(ntok.reshape(-1))
        self.beam_scores.copy_(nscore.reshape(-1))
        self.ids.copy_(self.ids[self.beam_idx])
        self.ids.scatter_(1, cur.expand(self.ids.shape[0], 1), self.next_tok[:, None])
        cur.add_(1)
        self.cur_len += 1
        return self.beam_idx

    def all_done(self):
        """Device bool: every business is done (the token loop's stop flag)."""
        return self.done.all()

    # -- result -----------------------------------------------------------------------------------------
    def finalize(self, num_return_sequences=1):
        """Unfinished businesses contribute their open beams (:3012-3026); the `num_return_sequences` best hypotheses per
        business in descending score order (rows i*n .. i*n+n-1 belong to business i), padded like the reference's output
        (:3036-3061).  Row i*n is the n = 1 result (ties go to the lower pool slot, as argmax)."""
        k, cur = self.k, self.cur_len
        live = ~self.done
        norm = float(cur) ** self.length_penalty
        for j in range(k):
            row = self.row0[:, 0] + j
            self._admit(live, self.beam_scores[row] / norm, self.ids[row], cur)
        filled = self.slot_ids[None, :] < self.pool_n[:, None]
        masked = torch.where(filled, self.pool_score, torch.full_like(self.pool_score, NEG))
        n = num_return_sequences
        if n == 1:
            best = masked.argmax(dim=1)
            tok = self.pool_tok[self.rows, best]
            lens = self.pool_len[self.rows, best]
        else:
            if n > k:
                raise ValueError("num_return_sequences (%d) must not exceed num_beams (%d)" % (n, k))
            order = torch.sort(masked, dim=1, descending=True, stable=True).indices[:, :n]
            best = order.reshape(-1)
            tok = self.pool_tok[self.rows[:, None], order].reshape(self.B * n, -1)
            lens = self.pool_len[self.rows[:, None], order].reshape(-1)
            self.out_scores = masked[self.rows.repeat_interleave(n), best]      # score of each returned row
        lo, hi = int(lens.min().item()), int(lens.max().item())
        if lo == hi:
            return tok[:, :hi].contiguous()
        width = min(hi + 1, self.max_length)
        pos = torch.arange(width, device=self.dev)[None, :]
        out = torch.where(pos < lens[:, None], tok[:, :width], torch.full_like(tok[:, :width], self.pad))
        return torch.where((pos == lens[:, None]) & (lens[:, None] < self.max_length), torch.full_like(out, self.eos), out)


def beam_search(logits_fn, B, V, dev, num_beams=4, max_length=20, min_length=0, length_penalty=1.0, no_repeat_ngram_size=3,
                early_stopping=True, pad=1, bos=0, eos=2, reorder_fn=None, poll_every=8, num_return_sequences=1):
    """_generate_beam_search (modeling_multimodalsum.py:2803-3067), do_sample=False.  `logits_fn(input_ids[N, cur_len])`
    returns the fp32 next-token logits [N, V] of the last position (N = B*num_beams, beams of a business adjacent);
    `reorder_fn(beam_idx)` re-orders an incremental decoder's caches (`_reorder_cache`, :3103-3115)."""
    bs = BeamSearch(B, V, dev, num_beams, max_length, min_length, length_penalty, no_repeat_ngram_size, early_stopping,
                    pad, bos, eos)
    cuda = torch.device(dev).type == "cuda"
    flag = torch.zeros(1, dtype=torch.bool, pin_memory=True) if cuda else None
    ev = None
    while bs.cur_len < max_length:
        beam_idx = bs.advance(logits_fn(bs.ids[:, :bs.cur_len]))
        if not cuda:
            if bool(bs.done.all()):
                break
        else:
            # poll the "every business done" flag without stalling the launch queue: the copy issued `poll_every` tokens
            # ago is read now
            if ev is not None and ev.query():
                if bool(flag[0]):
                    break
                ev = None
            if ev is None and bs.cur_len % poll_every == 0:
                flag.copy_(bs.done.all().reshape(1), non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
        if reorder_fn is not None and bs.cur_len < max_length:
            reorder_fn(beam_idx)
    return bs.finalize(num_return_sequences)


# ---------------------------------------------------------------------------------------------------- sampling
# Defaults of the reference's PretrainedConfig (vendored transformers 3.0.2 configuration_utils.py), which `generate` falls
# back to for every argument left at None.
SAMPLE_DEFAULTS = dict(do_sample=False, temperature=1.0, top_k=50, top_p=1.0, repetition_penalty=1.0, num_return_sequences=1)


def validate_generate_args(num_beams, do_sample, temperature, top_k, top_p, repetition_penalty, num_return_sequences,
                           bad_words_ids=None):
    """The argument checks of GenerationMixin.generate (generation_utils.py, its asserts) as ValueError, plus what this
    implementation does not cover as NotImplementedError.  Runs before any device work."""
    def is_int(v):
        return isinstance(v, int) and not isinstance(v, bool)
    if not is_int(num_beams) or num_beams < 1:
        raise ValueError("num_beams must be a positive integer, got %r" % (num_beams,))
    if not temperature > 0:
        raise ValueError("temperature must be > 0, got %r" % (temperature,))
    if not is_int(top_k) or top_k < 0:
        raise ValueError("top_k must be an integer >= 0, got %r" % (top_k,))
    if not 0 <= top_p <= 1:
        raise ValueError("top_p must be in [0, 1], got %r" % (top_p,))
    if not repetition_penalty >= 1.0:
        raise ValueError("repetition_penalty must be >= 1, got %r" % (repetition_penalty,))
    if not is_int(num_return_sequences) or num_return_sequences < 1:
        raise ValueError("num_return_sequences must be a positive integer, got %r" % (num_return_sequences,))
    if num_beams == 1 and not do_sample and num_return_sequences > 1:
        raise ValueError("greedy decoding (num_beams=1, do_sample=False) returns one sequence per input; "
                         "num_return_sequences=%d needs do_sample=True or num_beams >= %d" % (num_return_sequences,
                                                                                              num_return_sequences))
    if num_beams > 1 and num_return_sequences > num_beams:
        raise ValueError("num_return_sequences (%d) must not exceed num_beams (%d)" % (num_return_sequences, num_beams))
    if bad_words_ids is not None:
        raise NotImplementedError("bad_words_ids is not implemented")
    if do_sample and num_beams > 1:
        raise NotImplementedError("beam sampling (do_sample=True with num_beams > 1) is not implemented")
    if not do_sample and repetition_penalty != 1.0:
        raise NotImplementedError("repetition_penalty is implemented for do_sample=True only (greedy and beam search run "
                                  "the beam-search path)")


def resolve_generate_args(kw):
    """`generate(**kw)` keyword arguments -> the keyword arguments of Generator.generate_from_memory.  None means the
    default, as in the reference; everything is validated here, before any device work.  With do_sample=False and
    num_return_sequences=1 the result is exactly the beam-search argument set."""
    s = {k: (v if kw.get(k) is None else kw[k]) for k, v in SAMPLE_DEFAULTS.items()}
    args = dict(num_beams=kw.get("num_beams") or 1, max_length=kw.get("max_length") or 20, min_length=kw.get("min_length") or 0,
                length_penalty=1.0 if kw.get("length_penalty") is None else kw["length_penalty"],
                no_repeat_ngram_size=kw.get("no_repeat_ngram_size") or 0,
                early_stopping=bool(kw.get("early_stopping")), use_cache=kw.get("use_cache") is not False)
    validate_generate_args(args["num_beams"], bool(s["do_sample"]), s["temperature"], s["top_k"], s["top_p"],
                           s["repetition_penalty"], s["num_return_sequences"], kw.get("bad_words_ids"))
    if s["do_sample"]:
        args.update(do_sample=True, temperature=float(s["temperature"]), top_k=s["top_k"], top_p=float(s["top_p"]),
                    repetition_penalty=float(s["repetition_penalty"]), num_return_sequences=s["num_return_sequences"])
    elif s["num_return_sequences"] != 1:
        args.update(num_return_sequences=s["num_return_sequences"])
    return args


def sample_scores(logits, ids, cur_len, min_length, no_repeat_ngram_size, temperature, top_k, top_p, repetition_penalty,
                  eos):
    """The score processing of one sampling step, restated on tensors: logits fp32 [N, V] of the last position, ids [N, >=
    cur_len] the prefixes -> processed scores [N, V] with -inf for every token that cannot be drawn.  In the order of
    _generate_no_beam_search (generation_utils.py):
      1. postprocess_next_token_scores -> enforce_repetition_penalty_: each distinct id of the prefix (start token included)
         once, score / penalty if > 0 (>= 0 in the reference's `< 0 ? * : /`), * penalty if < 0;
      2. ... EOS score -inf while cur_len < min_length;
      3. ... calc_banned_ngram_tokens: a token that would complete an n-gram already in the prefix is -inf;
      4. NO adjust_logits_during_generation: the reference calls it on the beam path only (forced BOS / EOS do not apply);
      5. scores / temperature;
      6. top_k_top_p_filtering(min_tokens_to_keep=1): top-k keeps every token >= the k-th largest score (ties at the k-th
         value survive; k = min(top_k, V), 0 = off); top-p on what is left keeps a token iff the softmax mass ranked strictly
         before it is <= top_p (the crossing token and the top token are kept).  Equal scores are ranked by ascending
         token id: that tie rule is ours (torch.sort leaves the order of equal values unspecified).
    The draw is softmax over the result (7)."""
    scores = logits.float().clone()
    N, V = scores.shape
    prev = ids[:, :cur_len]
    if repetition_penalty != 1.0:
        seen = torch.zeros(N, V, dtype=torch.bool, device=scores.device).scatter_(1, prev, True)
        scores = torch.where(seen, torch.where(scores < 0, scores * repetition_penalty, scores / repetition_penalty), scores)
    if cur_len < min_length:
        scores[:, eos] = NEG
    n = no_repeat_ngram_size
    if n > 0 and cur_len + 1 >= n:
        for r in range(N):
            gen = prev[r].tolist()
            tail = tuple(gen[cur_len - n + 1:])
            banned = [gen[i + n - 1] for i in range(cur_len - n + 1) if tuple(gen[i:i + n - 1]) == tail]
            if banned:
                scores[r, banned] = NEG
    if temperature != 1.0:
        scores = scores / temperature
    if top_k > 0:
        kth = torch.topk(scores, min(top_k, V), dim=-1).values[:, -1:]
        scores = scores.masked_fill(scores < kth, NEG)
    if top_p < 1.0:
        sorted_s, sorted_i = torch.sort(scores, dim=-1, descending=True, stable=True)
        cum = torch.softmax(sorted_s, dim=-1).cumsum(dim=-1)
        remove = cum > top_p
        remove[:, 1:] = remove[:, :-1].clone()
        remove[:, 0] = False
        scores = scores.masked_fill(remove.scatter(1, sorted_i, remove), NEG)
    return scores


class SampleSearch:
    """State of one batched sampling loop (_generate_no_beam_search with do_sample=True): `B` businesses x `n` samples,
    rows i*n .. i*n+n-1 belong to business i and are never re-ranked (the decoder's slot table stays the identity).

      ids [N, max_length]   token histories (decoder start token = eos first), pad after a row's EOS by construction
      unfinished [N]        uint8, 0 once the row appended EOS
      seed [1]              int64 Philox key, drawn from torch's default generator of the device at every reset()

    Every piece of per-step state is a fixed device buffer updated in place and the length enters as the device scalar
    `cur_t`, so one step records into a CUDA graph.  On CUDA the step is csrc/sample_sm100.cu (no other path); on the CPU it
    is `sample_scores` + torch.multinomial, the tensor restatement the kernel is tested against."""

    def __init__(self, B, V, dev, num_return_sequences, max_length, min_length, no_repeat_ngram_size, temperature, top_k,
                 top_p, repetition_penalty, pad, eos):
        n = num_return_sequences
        self.B, self.n, self.V, self.dev = B, n, V, dev
        self.max_length, self.min_length, self.ngram = max_length, min_length, no_repeat_ngram_size
        self.temperature, self.top_k, self.top_p, self.penalty = temperature, top_k, top_p, repetition_penalty
        self.pad, self.eos = pad, eos
        N = B * n
        self.ids = torch.empty((N, max_length), dtype=torch.long, device=dev)
        self.unfinished = torch.empty(N, dtype=torch.uint8, device=dev)
        self.cur_t = torch.empty(1, dtype=torch.long, device=dev)
        self.seed = torch.zeros(1, dtype=torch.long, device=dev)
        self.kernel_path = torch.device(dev).type == "cuda"
        self.dec_ids32 = None
        self._gen = None
        self._clear()

    def _clear(self):
        self.ids.fill_(self.pad)
        self.ids[:, 0] = self.eos
        self.unfinished.fill_(1)
        self.cur_len = 1
        self.cur_t.fill_(1)

    def reset(self):
        """Back to the start state, in place, and this call's seed: one draw from torch's default generator of the device
        (no host sync), so torch.manual_seed makes a call reproducible and consecutive calls differ."""
        self._clear()
        self.seed.random_()
        if not self.kernel_path:
            self._gen = torch.Generator().manual_seed(int(self.seed.item()))

    def attach_decoder(self, ids32, hist):
        """The decoder's next-token input [N] (int32), written by the sampler.  The slot table needs no work: rows are never
        re-ranked and the decode self-attention writes hist[n][t] = n itself."""
        self.dec_ids32 = ids32

    def all_done(self):
        return self.unfinished.eq(0).all()

    def advance(self, logits):
        """logits: fp32 [N, V] next-token logits of the current prefixes; appends one token per row."""
        if self.kernel_path:
            ops.sample_token(logits, self.V, self.ids, self.cur_t, self.seed, self.min_length, self.ngram, self.eos, self.pad,
                             self.temperature, self.top_k, self.top_p, self.penalty, self.unfinished, self.dec_ids32)
        else:
            cur = self.cur_len
            scores = sample_scores(logits, self.ids, cur, self.min_length, self.ngram, self.temperature, self.top_k,
                                   self.top_p, self.penalty, self.eos)
            tok = torch.multinomial(torch.softmax(scores, dim=-1), 1, generator=self._gen).squeeze(1)
            tok = torch.where(self.unfinished.bool(), tok, torch.full_like(tok, self.pad))     # tokens_to_add
            self.ids[:, cur] = tok
            self.unfinished.mul_((tok != self.eos).to(torch.uint8))
            if self.dec_ids32 is not None:
                self.dec_ids32.copy_(tok)
        self.cur_t.add_(1)
        self.cur_len += 1

    def finalize(self):
        """The reference returns input_ids when the loop ends: at max_length, or right after the step in which the last row
        appended EOS.  Steps the token loop ran after that (it polls the stop flag with a lag) only appended pad."""
        ids = self.ids[:, :self.cur_len]
        if not (bool(self.unfinished.any()) or self.cur_len <= 1):
            first_eos = (ids[:, 1:] == self.eos).long().argmax(dim=1) + 1
            ids = ids[:, :int(first_eos.max()) + 1]
        return ids.clone()                    # never a view of the plan's buffer: the next call overwrites it


def sample_search(logits_fn, B, V, dev, num_return_sequences=1, max_length=20, min_length=0, no_repeat_ngram_size=0,
                  temperature=1.0, top_k=50, top_p=1.0, repetition_penalty=1.0, pad=1, eos=2, poll_every=8):
    """_generate_no_beam_search with do_sample=True.  `logits_fn(input_ids[N, cur_len])` returns the fp32 next-token logits
    [N, V] of the last position (N = B * num_return_sequences, the rows of a business adjacent)."""
    ss = SampleSearch(B, V, dev, num_return_sequences, max_length, min_length, no_repeat_ngram_size, temperature, top_k,
                      top_p, repetition_penalty, pad, eos)
    ss.reset()
    cuda = torch.device(dev).type == "cuda"
    flag = torch.zeros(1, dtype=torch.bool, pin_memory=True) if cuda else None
    ev = None
    while ss.cur_len < max_length:
        ss.advance(logits_fn(ss.ids[:, :ss.cur_len]))
        if not cuda:
            if bool(ss.all_done()):
                break
        else:
            if ev is not None and ev.query():
                if bool(flag[0]):
                    break
                ev = None
            if ev is None and ss.cur_len % poll_every == 0:
                flag.copy_(ss.all_done().reshape(1), non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
    return ss.finalize()


class DecodeState:
    """Per-call decoding state: the projected memory plus the incremental decoder's workspaces."""

    def __init__(self, mem, beams):
        self.mem, self.beams = mem, beams
        self.cws = None


class Generator:
    def __init__(self, model):
        self.model = model
        self.eng = None
        self._plans = {}

    def _engine(self, device):
        eng = self.model._ensure_engine(device)
        if eng is not self.eng:
            self._plans.clear()               # recorded graphs hold the previous engine's arena pointers
        self.eng = eng
        return self.eng

    # ------------------------------------------------------------------ memory
    @torch.no_grad()
    def encode(self, reviews, reviews_mask, field, field_value, img, img_mask, num_beams):
        """MultimodalSum.get_multimodal_outputs (src/multimodal_train.py:165-193) + the per-layer cross K|V projection."""
        return self.prepare(self.encode_memory(reviews, reviews_mask, field, field_value, img, img_mask), num_beams)

    @torch.no_grad()
    def encode_memory(self, reviews, reviews_mask, field, field_value, img, img_mask):
        """get_multimodal_outputs -> packed cross-attention memory (not yet projected to K|V)."""
        eng = self._engine(reviews.device)
        eng.refresh_bf16_weights()
        B, R, S = reviews.shape
        text = INF.encoder_forward(eng, reviews.reshape(B * R, S), reviews_mask.reshape(B * R, S)).reshape(B, R, S, -1)
        if eng.cfg.dataset == "text":
            mem = INF.build_memory(eng, [text], [reviews_mask])
        else:
            tab, tab_valid = INF.table_forward(eng, field, field_value)
            imgh = INF.image_forward(eng, img)
            imask = img_mask.reshape(B, -1, 1).expand(-1, -1, imgh.shape[2])
            mem = INF.build_memory(eng, [text, tab.unsqueeze(1), imgh], [reviews_mask, tab_valid.unsqueeze(1), imask])
        return mem

    @torch.no_grad()
    def prepare(self, mem, num_beams):
        eng = self._engine(mem.MEM.device)
        eng.refresh_bf16_weights()
        INF.project_memory(eng, mem)
        return DecodeState(mem, num_beams)

    # ------------------------------------------------------------------ one decode step, prefix recomputed
    @torch.no_grad()
    def last_logits(self, st, input_ids, rating_diff):
        """input_ids [N, cur_len] (N = B*beams, beams of a business adjacent) -> fp32 logits [N, V] of the last position."""
        x = INF.decoder_hidden(self.eng, st.mem, input_ids, rating_diff, per_biz=st.beams)
        return INF.lm_head(self.eng, x[:, input_ids.shape[1] - 1])      # strided [N, D] view: the GEMM reads it in place

    # ------------------------------------------------------------------ one cached decode step (all beams)
    def _decode_ws(self, st, N, dev):
        eng, cfg, mem = self.eng, self.eng.cfg, st.mem
        D, H, V, FF, L = cfg.d_model, cfg.heads, cfg.vocab_size, cfg.ffn_dim, cfg.decoder_layers
        S = INF.FRAME
        nm = len(mem.mods)
        bf = lambda *s: torch.empty(s, device=dev, dtype=torch.bfloat16)
        f32 = lambda *s: torch.empty(s, device=dev, dtype=torch.float32)
        w = dict(x=bf(N, D), x1=bf(N, D), x2=bf(N, D), nxt=bf(N, D), o=bf(N, D), qc=bf(N, D), a=bf(N, FF), f=bf(N, D),
                 qkv=bf(N, 3 * D), ctx=bf(N, D),
                 kvs=[torch.zeros(N, S, 2 * D, device=dev, dtype=torch.bfloat16) for _ in range(L)],   # self K|V caches: never move
                 hist=torch.zeros(N, S, device=dev, dtype=torch.int32),                                 # slot table (see decode_sm100.cu)
                 hist_alt=torch.zeros(N, S, device=dev, dtype=torch.int32),
                 A3=bf(nm, N, D), O3=bf(nm, N, D), U=bf(2, N, D), AB=bf(2, N, D), yc=bf(N, D),
                 mean=f32(N), rstd=f32(N), ids=torch.zeros(N, device=dev, dtype=torch.int32),
                 pos_dev=torch.zeros(1, device=dev, dtype=torch.int32), rd=torch.zeros(N, device=dev),
                 logits=f32(N, (V + 3) // 4 * 4)[:, :V],                                               # 16-byte row pitch for TMA
                 inv_n=mem.inv_n.repeat_interleave(st.beams, dim=0).contiguous(), pos=-1, graph=None,
                 side=torch.cuda.Stream(device=dev), ev_fork=torch.cuda.Event(), ev_join=torch.cuda.Event())
        return w

    def _decode_launches(self, st):
        """Every kernel of one decode step; all per-step state (token ids, position, slot table) is read from device memory."""
        eng, cfg, mem, w = self.eng, self.eng.cfg, st.mem, st.cws
        N = w["x"].shape[0]
        stats, scale = (w["mean"], w["rstd"]), cfg.head_dim ** -0.5
        x, nxt = w["x"], w["nxt"]
        ops.embed_ln_decode(w["ids"], *L.embed_params(eng, "decoder", w["rd"]), x, *stats, N, w["pos_dev"])
        cross = L.cross_attn_args(eng, w["qc"], mem.kv[0], w["A3"], None, mem.mods, mem.mem_valid, mem.ent_valid, w["inv_n"],
                                  N, st.beams)
        fork = (w["side"], w["ev_fork"], w["ev_join"])     # the two gate GEMMs are 16-CTA GEMMs: run them side by side
        for l in range(cfg.decoder_layers):
            lp = L.BM + "decoder.layers.%d." % l
            cross.KV = mem.kv[l].data_ptr()
            attend = lambda qkv, ctx, l=l: ops.attn_decode_self(qkv, w["kvs"][l], w["hist"], w["pos_dev"], ctx, cfg.heads, scale)
            L.self_block(eng, lp, x, w, attend, stats, L.NO_DROP)
            L.cross_block(eng, lp, w["x1"], w, lambda qc, A3: ops.attn_decode_cross(cross), stats, L.NO_DROP, mem.pres,
                          st.beams, fork)
            L.ffn_block(eng, lp, w["x2"], w, nxt, stats, L.NO_DROP)
            x, nxt = nxt, x
        ops.gemm(x, eng.w16(L.BM + "shared.weight"), w["logits"], bias=eng.w32_flb())

    @torch.no_grad()
    def step_logits(self, st, input_ids, rating_diff):
        """Incremental decoding (`_use_saved_state` / cached branch of `get_head_output`, modeling_multimodalsum.py:774-815,
        889-920): only the newest token of every hypothesis goes through the decoder.  input_ids [N, cur_len] -> fp32 logits
        [N, V] of the last position (a buffer that the next call overwrites).  Call `reorder_cache(st, beam_idx)` after every
        beam re-ranking (`_reorder_cache`, :3103-3115).

        Decode-shaped kernels (csrc/decode_sm100.cu): the self-attention K|V of earlier positions stay where they were written
        and are found through a slot table that `reorder_cache` permutes (128 KB instead of 12 layers of caches); the
        cross-attention reads the un-expanded per-business K|V once per business and head for all of its beams.  The ~200
        launches of a step take their per-step inputs (token ids, position, slot table) from device memory, so from the second
        token on the whole step is replayed from ONE CUDA graph (MMSUM_DECODE_GRAPH=0 launches it kernel by kernel)."""
        import os
        dev = input_ids.device
        N, cur = input_ids.shape
        if cur > INF.FRAME:
            raise ValueError("decoder frames up to 128 tokens")
        if st.beams > 8:
            raise ValueError("the decode attention kernel handles up to 8 beams per business")
        t = cur - 1
        if st.cws is None:
            st.cws = self._decode_ws(st, N, dev)
        w = st.cws
        if w.get("fused"):
            raise RuntimeError("this DecodeState is driven by the fused token loop; build a fresh one with encode()/prepare()")
        if t != w["pos"] + 1:
            raise ValueError("step_logits must be called with consecutive lengths (got position %d after %d)" % (t, w["pos"]))
        w["pos"] = t
        w["ids"].copy_(input_ids[:, t])
        w["rd"].copy_(rating_diff.reshape(-1))
        if w["graph"] is None:
            self._decode_launches(st)                 # first token: plain launches (also sets the one-time function attributes)
            w["graph"] = False
            if os.environ.get("MMSUM_DECODE_GRAPH", "1") != "0":
                try:
                    graph = torch.cuda.CUDAGraph()
                    torch.cuda.synchronize()
                    with torch.cuda.graph(graph):
                        self._decode_launches(st)     # re-records the same step; replays read the then-current device state
                    w["graph"] = graph
                except Exception as e:                # noqa: BLE001 — same kernels, launched one by one
                    import warnings
                    warnings.warn("CUDA-graph capture of the decode step failed (%s); launching kernel by kernel" % (e,))
                    w["graph"] = False
        elif w["graph"] is False:
            self._decode_launches(st)
        else:
            w["graph"].replay()
        w["pos_dev"].add_(1)
        return w["logits"]

    @torch.no_grad()
    def reorder_cache(self, st, beam_idx):
        """`_reorder_cache` (:3103-3115): hypothesis i continues hypothesis beam_idx[i].  Only the slot table moves: the
        self-attention caches stay in place and the cross-attention K|V are per business (beam_idx never crosses businesses)."""
        w = st.cws
        if w is None:
            return
        torch.index_select(w["hist"], 0, beam_idx, out=w["hist_alt"])
        w["hist"].copy_(w["hist_alt"])

    # ------------------------------------------------------------------ fused token loop (one CUDA graph per token)
    def _plan(self, mem, k, kw, sample=None):
        """Static buffers + the recorded token step for one (memory layout, search setting): the K|V projections of a
        new memory are written into the plan's buffers and the same CUDA graph is replayed — capture and instantiation
        (~0.15 s for ~220 nodes) are paid once per shape, not once per generate() call.  `k` rows per business: beams, or
        samples when `sample` holds the sampling parameters (a SampleSearch then replaces the BeamSearch)."""
        cfg = self.eng.cfg
        dev = mem.MEM.device
        if sample is None:
            key = (mem.B, k, tuple(mem.mods), mem.MEM.shape[0], mem.Et, mem.pres is None, kw["max_length"], kw["min_length"],
                   float(kw["length_penalty"]), kw["no_repeat_ngram_size"], bool(kw["early_stopping"]), str(dev))
        else:
            key = ("sample", mem.B, k, tuple(mem.mods), mem.MEM.shape[0], mem.Et, mem.pres is None, kw["max_length"],
                   kw["min_length"], kw["no_repeat_ngram_size"], sample["temperature"], sample["top_k"], sample["top_p"],
                   sample["repetition_penalty"], str(dev))
        plan = self._plans.get(key)
        if plan is not None:
            return plan
        D, L = cfg.d_model, cfg.decoder_layers
        smem = INF.Memory(MEM=mem.MEM[:0], B=mem.B, mods=list(mem.mods), mem_valid=torch.empty_like(mem.mem_valid),
                          ent_valid=torch.empty_like(mem.ent_valid), inv_n=torch.empty_like(mem.inv_n),
                          pres=None if mem.pres is None else torch.empty_like(mem.pres), Et=mem.Et,
                          kv=[torch.empty(mem.MEM.shape[0], 2 * D, device=dev, dtype=torch.bfloat16) for _ in range(L)])
        st = DecodeState(smem, k)
        N = mem.B * k
        st.cws = self._decode_ws(st, N, dev)
        st.cws["fused"] = True
        if sample is None:
            bs = BeamSearch(mem.B, cfg.vocab_size, dev, k, kw["max_length"], kw["min_length"], kw["length_penalty"],
                            kw["no_repeat_ngram_size"], kw["early_stopping"], cfg.pad_token_id, cfg.bos_token_id, cfg.eos_token_id)
        else:
            bs = SampleSearch(mem.B, cfg.vocab_size, dev, k, kw["max_length"], kw["min_length"], kw["no_repeat_ngram_size"],
                              sample["temperature"], sample["top_k"], sample["top_p"], sample["repetition_penalty"],
                              cfg.pad_token_id, cfg.eos_token_id)
        bs.attach_decoder(st.cws["ids"], st.cws["hist"])
        plan = dict(st=st, bs=bs, graph=None, captured=False)
        if len(self._plans) >= 4:                     # a handful of shapes at most; drop the oldest
            self._plans.pop(next(iter(self._plans)))
        self._plans[key] = plan
        return plan

    @torch.no_grad()
    def _fused_beam_search(self, mem, rd, poll_every=8, sample=None, num_return_sequences=1, **kw):
        """Decoder step + beam update + cache re-ranking of one token recorded ONCE and replayed: the host issues a single
        graph launch per token (the reference runs ~47 k eager ops and several host syncs per token, :2857-3010).  The very
        first token of a new shape runs kernel by kernel (one-time function attributes, allocator warm-up), the capture
        follows it; later calls with the same shape replay the graph from the first token on.  With `sample` (the sampling
        parameters) the same loop runs the sampler over num_beams = samples per business instead of the beam update."""
        import os
        eng = self.eng
        cfg = eng.cfg
        k = kw.pop("num_beams")
        plan = self._plan(mem, k, kw, sample)
        st, bs = plan["st"], plan["bs"]
        w, smem = st.cws, st.mem
        # ---- this call's memory: validity bookkeeping copied, K|V projected straight into the plan's buffers
        smem.mem_valid.copy_(mem.mem_valid); smem.ent_valid.copy_(mem.ent_valid); smem.inv_n.copy_(mem.inv_n)
        if smem.pres is not None:
            smem.pres.copy_(mem.pres)
        w["inv_n"].copy_(mem.inv_n.repeat_interleave(k, dim=0))
        for l in range(cfg.decoder_layers):
            if mem.kv:
                smem.kv[l].copy_(mem.kv[l])
            else:
                L.project_kv(eng, mem.MEM, l, smem.kv[l])
        # ---- reset the per-call state in place
        bs.reset()
        w["rd"].copy_(rd.reshape(-1))
        w["ids"].copy_(bs.ids[:, 0])
        w["pos_dev"].zero_()
        w["hist"].zero_()

        def token_step():
            self._decode_launches(st)
            beam_idx = bs.advance(w["logits"])
            if not bs.kernel_path:              # tensor-op beam update: re-rank the slot table / feed the tokens here
                torch.index_select(w["hist"], 0, beam_idx, out=w["hist_alt"])   # _reorder_cache: only the slot table moves
                w["hist"].copy_(w["hist_alt"])
                w["ids"].copy_(bs.next_tok)
            w["pos_dev"].add_(1)

        max_length = kw["max_length"]
        if max_length <= 1:
            return bs.finalize() if sample is not None else bs.finalize(num_return_sequences)
        if not plan["captured"]:
            plan["captured"] = True
            token_step()
            if bs.cur_len < max_length and os.environ.get("MMSUM_DECODE_GRAPH", "1") != "0":
                host_len = bs.cur_len
                try:
                    g = torch.cuda.CUDAGraph()
                    torch.cuda.synchronize()
                    with torch.cuda.graph(g):
                        token_step()
                    plan["graph"] = g
                except Exception as e:            # noqa: BLE001 — same kernels, launched one by one
                    import warnings
                    warnings.warn("CUDA-graph capture of the token step failed (%s); launching kernel by kernel" % (e,))
                bs.cur_len = host_len             # the capture ran the Python bookkeeping once without executing anything
        graph = plan["graph"]
        self.last_used_graph = graph is not None
        flag = torch.zeros(1, dtype=torch.bool, pin_memory=True)
        ev = None
        while bs.cur_len < max_length:
            if graph is not None:
                graph.replay()
                bs.cur_len += 1
            else:
                token_step()
            if ev is not None and ev.query():
                if bool(flag[0]):
                    break
                ev = None
            if ev is None and bs.cur_len % poll_every == 0:
                flag.copy_(bs.all_done().reshape(1), non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
        self.last_decode_steps = bs.cur_len - 1
        return bs.finalize() if sample is not None else bs.finalize(num_return_sequences)

    # ------------------------------------------------------------------ public entry points
    @torch.no_grad()
    def generate_from_memory(self, mem, rating_diff=None, num_beams=4, max_length=20, min_length=0, length_penalty=1.0,
                             no_repeat_ngram_size=3, early_stopping=True, use_cache=True, do_sample=False, temperature=1.0,
                             top_k=50, top_p=1.0, repetition_penalty=1.0, num_return_sequences=1):
        """`bart_model.generate(text_hiddens, ..., rating_diff=..., num_beams=...)` as src/test.py:156-158 calls it ->
        token ids [B * num_return_sequences, <= max_length], the rows of a business adjacent.  do_sample=True (num_beams
        must be 1): _generate_no_beam_search with num_return_sequences samples per business on the device sampler
        (`SampleSearch`); otherwise beam search, returning the num_return_sequences best hypotheses per business."""
        validate_generate_args(num_beams, do_sample, temperature, top_k, top_p, repetition_penalty, num_return_sequences)
        cfg = self.model.cfg
        B, dev = mem.B, mem.MEM.device
        rows = num_return_sequences if do_sample else num_beams
        rd = torch.zeros(B, device=dev) if rating_diff is None else rating_diff.reshape(B).float()
        rd = rd.repeat_interleave(rows).contiguous()
        if rows > 8:
            use_cache = False                     # the decode attention kernel holds up to 8 rows (beams, samples) per business
        sample = dict(temperature=float(temperature), top_k=int(top_k), top_p=float(top_p),
                      repetition_penalty=float(repetition_penalty)) if do_sample else None
        if use_cache:
            eng = self._engine(dev)
            eng.refresh_bf16_weights()
            return self._fused_beam_search(mem, rd, num_beams=rows, max_length=max_length, min_length=min_length,
                                           length_penalty=length_penalty, no_repeat_ngram_size=no_repeat_ngram_size,
                                           early_stopping=early_stopping, sample=sample,
                                           num_return_sequences=num_return_sequences)
        st = self.prepare(mem, rows)
        logits_fn, reorder_fn = (lambda ids: self.last_logits(st, ids, rd)), None
        if sample is not None:
            return sample_search(logits_fn, B, cfg.vocab_size, dev, num_return_sequences=rows, max_length=max_length,
                                 min_length=min_length, no_repeat_ngram_size=no_repeat_ngram_size, pad=cfg.pad_token_id,
                                 eos=cfg.eos_token_id, **sample)
        return beam_search(logits_fn, B, cfg.vocab_size, dev, num_beams=num_beams, max_length=max_length, min_length=min_length,
                           length_penalty=length_penalty, no_repeat_ngram_size=no_repeat_ngram_size, early_stopping=early_stopping,
                           pad=cfg.pad_token_id, bos=cfg.bos_token_id, eos=cfg.eos_token_id, reorder_fn=reorder_fn,
                           num_return_sequences=num_return_sequences)

    @torch.no_grad()
    def generate(self, reviews, reviews_mask, field, field_value, img, img_mask, rating_diff=None, **kw):
        """get_multimodal_outputs + generate in one call.  use_cache=True: incremental decoding with self-attention K|V
        caches (`step_logits`); False: recompute the whole prefix every step (`last_logits`)."""
        mem = self.encode_memory(reviews, reviews_mask, field, field_value, img, img_mask)
        return self.generate_from_memory(mem, rating_diff, **kw)
