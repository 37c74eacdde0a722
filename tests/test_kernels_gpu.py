"""Per-kernel parity tests (GPU): every C-ABI entry point against a plain torch fp32 restatement of the reference op
on the same seeded inputs.  Tolerances are bf16-storage tolerances, stated per test."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

D = 1024


def _dev():
    return torch.device("cuda")


def _ops():
    from multimodalsum_b200 import ops
    return ops


def _close(a, b, rtol, name=""):
    a, b = a.float(), b.float()
    err = (a - b).abs().max().item()
    scale = max(b.abs().max().item(), 1e-6)
    assert err <= rtol * scale, "%s: max err %.4g vs scale %.4g" % (name, err, scale)


# ------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K,a_t,b_t,f32,acc", [
    (128, 256, 64, 0, 0, 0, 0), (1000, 776, 520, 0, 0, 0, 0), (512, 1024, 1024, 0, 1, 0, 0),
    (1024, 1024, 4096, 1, 1, 1, 1), (1024, 2048, 1000, 1, 1, 1, 1), (384, 50264, 1024, 0, 0, 0, 0),
    (752, 1024, 2048, 0, 0, 0, 0), (640, 1024, 50265, 0, 1, 0, 0),
])
def test_gemm_variants(M, N, K, a_t, b_t, f32, acc):
    ops = _ops()
    torch.manual_seed(0)
    ldk = (K + 7) // 8 * 8
    A = torch.randn((K, M) if a_t else (M, ldk), device=_dev()).to(torch.bfloat16)
    B = torch.randn((K, N) if b_t else (N, ldk), device=_dev()).to(torch.bfloat16)
    if not a_t:
        A = A[:, :K]
    if not b_t:
        B = B[:, :K]
    out = torch.randn(M, N, device=_dev()) if acc else None
    base = out.clone() if acc else 0
    Dm = ops.gemm(A, B, out, a_t=bool(a_t), b_t=bool(b_t), out_dtype=torch.float32 if f32 else torch.bfloat16, accumulate=bool(acc))
    Af = A.float().t() if a_t else A.float()
    Bf = B.float().t() if b_t else B.float()
    _close(Dm, Af @ Bf.t() + base, 1.5e-2 if not f32 else 2e-3, "gemm")


@pytest.mark.parametrize("M,N,K,block_n", [(256, 1024, 4096, 128), (256, 3072, 1024, 128), (256, 1024, 1024, 0), (768, 1024, 1024, 0),
                                            (256, 50265, 1024, 0)])
def test_gemm_skinny_decode_shapes(M, N, K, block_n):
    """Decode-step GEMMs (256 hypotheses): 128-wide tiles over several N tiles, bias, strided fp32 output for the LM head."""
    ops = _ops()
    torch.manual_seed(4)
    A = torch.randn(M, K, device=_dev()).to(torch.bfloat16)
    B = (torch.randn(N, K, device=_dev()) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, device=_dev())
    if N == 50265:
        out = torch.empty(M, (N + 3) // 4 * 4, device=_dev())[:, :N]
        ops.gemm(A, B, out, bias=bias)
    else:
        out = ops.gemm(A, B, bias=bias, block_n=block_n)
    _close(out, A.float() @ B.float().t() + bias, 1e-2, "skinny gemm")


def test_gemm_epilogues_and_cat():
    ops = _ops()
    torch.manual_seed(1)
    M, N, K = 512, 1024, 1024
    A = torch.randn(M, K, device=_dev()).to(torch.bfloat16)
    B = (torch.randn(N, K, device=_dev()) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, device=_dev())
    aux = torch.empty(M, N, device=_dev(), dtype=torch.bfloat16)
    out = ops.gemm(A, B, bias=bias, act=ops.ACT_GELU, aux=aux, aux_mode=ops.AUX_STORE_PREACT)
    pre = A.float() @ B.float().t() + bias
    _close(aux, pre, 1e-2, "preact")
    _close(out, F.gelu(pre), 1e-2, "gelu")
    h = torch.randn(M, N, device=_dev()).to(torch.bfloat16)
    out = ops.gemm(A, B, act=ops.ACT_GELU, aux=h, aux_mode=ops.AUX_MUL_DACT)
    hf = h.float().requires_grad_(True)
    F.gelu(hf).sum().backward()
    _close(out, (A.float() @ B.float().t()) * hf.grad, 1e-2, "dgelu")
    # the pair the training step uses: the forward epilogue saves GELU'(pre-activation), backward multiplies by it
    dact = torch.empty(M, N, device=_dev(), dtype=torch.bfloat16)
    out = ops.gemm(A, B, bias=bias, act=ops.ACT_GELU, aux=dact, aux_mode=ops.AUX_STORE_DACT)
    pf = pre.clone().requires_grad_(True)
    F.gelu(pf).sum().backward()
    _close(out, F.gelu(pre), 1e-2, "gelu (derivative saved)")
    _close(dact, pf.grad, 1e-2, "saved gelu'")
    out = ops.gemm(A, B, aux=h, aux_mode=ops.AUX_MUL)
    _close(out, (A.float() @ B.float().t()) * h.float(), 1e-2, "multiply by aux")
    A2 = torch.randn(M, K, device=_dev()).to(torch.bfloat16)
    B2 = (torch.randn(N, 2 * K, device=_dev()) * 0.05).to(torch.bfloat16)
    out = ops.gemm_cat(A, A2, B2, bias=bias)
    _close(out, torch.cat([A, A2], 1).float() @ B2.float().t() + bias, 1e-2, "cat")


@pytest.mark.parametrize("a_t,b_t,f32,acc", [(0, 0, 0, 0), (0, 1, 0, 0), (1, 1, 1, 1), (1, 0, 0, 0), (0, 0, 1, 1)])
def test_gemm_cta_pair_shapes(a_t, b_t, f32, acc):
    """Problems large enough for the CTA-pair kernel (tcgen05.mma.cta_group::2, M = 256 per instruction, each CTA staging half
    of the B tile): an odd number of m-tiles (the last pair has an out-of-range second tile), ragged M / N / K edges, all four
    operand layouts, bf16 and fp32-accumulating (split-K) outputs."""
    ops = _ops()
    torch.manual_seed(2)
    M, N, K = 2400, 2040, 1000          # 19 x 8 tiles of 128 x 256: 80 pairs >= 74
    ldk = (K + 7) // 8 * 8
    A = torch.randn((K, M) if a_t else (M, ldk), device=_dev()).to(torch.bfloat16)
    B = torch.randn((K, N) if b_t else (N, ldk), device=_dev()).to(torch.bfloat16)
    if not a_t:
        A = A[:, :K]
    if not b_t:
        B = B[:, :K]
    out = torch.randn(M, N, device=_dev()) if acc else None
    base = out.clone() if acc else 0
    Dm = ops.gemm(A, B, out, a_t=bool(a_t), b_t=bool(b_t), out_dtype=torch.float32 if f32 else torch.bfloat16, accumulate=bool(acc))
    Af = A.float().t() if a_t else A.float()
    Bf = B.float().t() if b_t else B.float()
    _close(Dm, Af @ Bf.t() + base, 1.5e-2 if not f32 else 2e-3, "pair gemm")


def test_gemm_cta_pair_epilogues_and_cat():
    """Fused-activation epilogues and the K-concatenated A operand on the CTA-pair kernel (step-sized M)."""
    ops = _ops()
    torch.manual_seed(3)
    M, N, K = 4736, 1024, 512           # 37 x 4 tiles: 76 pairs
    A = torch.randn(M, K, device=_dev()).to(torch.bfloat16)
    B = (torch.randn(N, K, device=_dev()) * 0.05).to(torch.bfloat16)
    bias = torch.randn(N, device=_dev())
    aux = torch.empty(M, N, device=_dev(), dtype=torch.bfloat16)
    out = ops.gemm(A, B, bias=bias, act=ops.ACT_GELU, aux=aux, aux_mode=ops.AUX_STORE_PREACT)
    pre = A.float() @ B.float().t() + bias
    _close(aux, pre, 1e-2, "preact")
    _close(out, F.gelu(pre), 1e-2, "gelu")
    h = torch.randn(M, N, device=_dev()).to(torch.bfloat16)
    out = ops.gemm(A, B, act=ops.ACT_GELU, aux=h, aux_mode=ops.AUX_MUL_DACT)
    hf = h.float().requires_grad_(True)
    F.gelu(hf).sum().backward()
    _close(out, (A.float() @ B.float().t()) * hf.grad, 1e-2, "dgelu")
    Bt = (torch.randn(K, N, device=_dev()) * 0.05).to(torch.bfloat16)
    out = ops.gemm(A, Bt, b_t=True, act=ops.ACT_GELU, aux=h, aux_mode=ops.AUX_MUL_DACT)
    _close(out, (A.float() @ Bt.float()) * hf.grad, 1e-2, "dgelu, B MN-major")
    A2 = torch.randn(M, K, device=_dev()).to(torch.bfloat16)
    B2 = (torch.randn(N, 2 * K, device=_dev()) * 0.05).to(torch.bfloat16)
    out = ops.gemm_cat(A, A2, B2, bias=bias)
    _close(out, torch.cat([A, A2], 1).float() @ B2.float().t() + bias, 1e-2, "cat")


# ------------------------------------------------------------------ LayerNorm blocks
def test_add_ln_fwd_bwd():
    ops = _ops()
    torch.manual_seed(2)
    rows = 1000
    res = torch.randn(rows, D, device=_dev()).to(torch.bfloat16)
    y = torch.randn(rows, D, device=_dev()).to(torch.bfloat16)
    gamma = 1 + 0.1 * torch.randn(D, device=_dev())
    beta = 0.1 * torch.randn(D, device=_dev())
    out = torch.empty_like(res)
    mean = torch.empty(rows, device=_dev())
    rstd = torch.empty(rows, device=_dev())
    ops.add_ln_fwd(res, y, gamma, beta, out, mean, rstd, 0.0, 1, 1)
    rf, yf = res.float().requires_grad_(True), y.float().requires_grad_(True)
    gf, bf = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    ref = F.layer_norm(rf + yf, (D,), gf, bf, 1e-5)
    _close(out, ref, 1e-2, "ln fwd")
    d1 = torch.randn(rows, D, device=_dev()).to(torch.bfloat16)
    d2 = torch.randn(rows, D, device=_dev()).to(torch.bfloat16)
    ref.backward(d1.float() + d2.float())
    dres = torch.empty_like(res)
    dg = torch.zeros(D, device=_dev())
    db = torch.zeros(D, device=_dev())
    ops.add_ln_bwd(d1, d2, res, y, gamma, mean, rstd, dres, dres, dg, db, 0.0, 1, 1)
    _close(dres, rf.grad, 1e-2, "ln dres")
    _close(dg, gf.grad, 2e-3, "ln dgamma")
    _close(db, bf.grad, 2e-3, "ln dbeta")


def test_add_ln_dropout_mask_consistency():
    ops = _ops()
    torch.manual_seed(3)
    rows, p = 512, 0.1
    res = torch.zeros(rows, D, device=_dev(), dtype=torch.bfloat16)
    y = torch.ones(rows, D, device=_dev(), dtype=torch.bfloat16)
    gamma, beta = torch.ones(D, device=_dev()), torch.zeros(D, device=_dev())
    out = torch.empty_like(res)
    mean, rstd = torch.empty(rows, device=_dev()), torch.empty(rows, device=_dev())
    ops.add_ln_fwd(res, y, gamma, beta, out, mean, rstd, p, 7, 3)
    # z = mask/keep -> LN maps kept entries to a positive value, dropped to a negative one
    keep = (out.float() > 0)
    frac = keep.float().mean().item()
    assert abs(frac - (1 - p)) < 5e-3, frac
    # backward regenerates the same mask: dy is zero exactly where forward dropped
    d1 = torch.ones(rows, D, device=_dev(), dtype=torch.bfloat16) * torch.randn(rows, D, device=_dev()).to(torch.bfloat16)
    dres, dy = torch.empty_like(res), torch.empty_like(res)
    dg, db = torch.zeros(D, device=_dev()), torch.zeros(D, device=_dev())
    ops.add_ln_bwd(d1, None, res, y, gamma, mean, rstd, dres, dy, dg, db, p, 7, 3)
    assert torch.equal(dy.float() == 0, ~keep | (dres.float() == 0))
    # a different stream id gives a different mask
    out2 = torch.empty_like(res)
    ops.add_ln_fwd(res, y, gamma, beta, out2, mean, rstd, p, 7, 4)
    assert not torch.equal(out2 > 0, out > 0)


def test_embed_ln_fwd_bwd_exact_gather():
    ops = _ops()
    torch.manual_seed(4)
    V, S, nseq = 777, 128, 6
    rows = nseq * S
    E = torch.randn(V, D, device=_dev()) * 0.02
    E[1].zero_()
    P = torch.randn(S + 2, D, device=_dev()) * 0.02
    ids = torch.randint(0, V, (rows,), device=_dev(), dtype=torch.int32)
    ids[5::7] = 1
    rd = torch.randn(nseq, device=_dev())
    remb = torch.randn(D, device=_dev()) * 0.02
    gamma, beta = 1 + 0.1 * torch.randn(D, device=_dev()), 0.1 * torch.randn(D, device=_dev())
    out = torch.empty(rows, D, device=_dev(), dtype=torch.bfloat16)
    mean, rstd = torch.empty(rows, device=_dev()), torch.empty(rows, device=_dev())
    ops.embed_ln_fwd(ids, E, P, rd, remb, gamma, beta, out, mean, rstd, rows, S, 0.0, 1, 1)
    Ef, Pf, rf = E.clone().requires_grad_(True), P.clone().requires_grad_(True), remb.clone().requires_grad_(True)
    gf, bf = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    pos = torch.arange(S, device=_dev()).repeat(nseq) + 2
    z = F.embedding(ids.long(), Ef, padding_idx=1) + Pf[pos] + rd.repeat_interleave(S)[:, None] * rf
    # the gather itself is exact: the fp32 row sums give bit-identical LN statistics inputs
    assert torch.allclose(mean, z.mean(-1), atol=1e-6)
    ref = F.layer_norm(z, (D,), gf, bf, 1e-5)
    _close(out, ref, 1e-2, "embed fwd")
    d1 = torch.randn(rows, D, device=_dev()).to(torch.bfloat16)
    ref.backward(d1.float())
    dE, dP, dr = torch.zeros_like(E), torch.zeros_like(P), torch.zeros_like(remb)
    dg, db = torch.zeros(D, device=_dev()), torch.zeros(D, device=_dev())
    dz = torch.empty(rows, D, device=_dev())
    ops.embed_ln_bwd(d1, None, ids, E, P, rd, remb, gamma, mean, rstd, dE, dP, dr, dg, db, dz, rows, S, 1, 0.0, 1, 1)
    _close(dE, Ef.grad, 2e-3, "dE")
    assert dE[1].abs().max().item() == 0.0   # padding_idx row receives nothing from the gather path
    _close(dP, Pf.grad, 2e-3, "dP")
    _close(dr, rf.grad, 2e-3, "dremb")
    _close(dg, gf.grad, 2e-3, "dgamma")
    _close(db, bf.grad, 2e-3, "dbeta")


def test_colsum_and_cast():
    ops = _ops()
    torch.manual_seed(5)
    x = torch.randn(3000, 2048, device=_dev()).to(torch.bfloat16)
    out = torch.ones(1024, device=_dev())
    ops.colsum(x[:, 1024:], out)
    _close(out, x[:, 1024:].float().sum(0) + 1, 1e-4, "colsum")
    src = torch.randn(100003, device=_dev())
    dst = torch.empty(100003, device=_dev(), dtype=torch.bfloat16)
    ops.cast_bf16(src, dst)
    assert torch.equal(dst, src.to(torch.bfloat16))


# ------------------------------------------------------------------ cross entropy
@pytest.mark.parametrize("eps,V", [(0.1, 50265), (None, 50265), (0.1, 512), (None, 1000)])
def test_ce_fwd_bwd(eps, V):
    ops = _ops()
    torch.manual_seed(6)
    rows = 300
    ld = (V + 7) // 8 * 8
    logits = torch.zeros(rows, ld, device=_dev(), dtype=torch.bfloat16)
    logits[:, :V] = (torch.randn(rows, V, device=_dev()) * 2).to(torch.bfloat16)
    tgt = torch.randint(0, V, (rows,), device=_dev(), dtype=torch.int32)
    lf = logits[:, :V].float().requires_grad_(True)
    logp = torch.log_softmax(lf, -1)
    if eps is None:
        ref_rows = -logp.gather(1, tgt.long()[:, None])[:, 0]
    else:
        dist = torch.full_like(logp, eps / (V - 1))
        dist.scatter_(1, tgt.long()[:, None], 1 - eps)
        ref_rows = (-dist * logp).sum(-1)
    ref_rows.mean().backward()
    loss_rows = torch.empty(rows, device=_dev())
    loss = torch.empty(1, device=_dev())
    lse = torch.empty(rows, device=_dev())
    ops.ce_fwd_bwd(logits, V, tgt, eps, 0.0, None, loss_rows, loss, 1.0 / rows, False, lse_rows=lse)
    assert torch.allclose(loss_rows, ref_rows.detach(), rtol=2e-5, atol=2e-5)
    assert abs(loss.item() - ref_rows.mean().item()) < 1e-4
    assert torch.allclose(lse, torch.logsumexp(lf.detach(), -1), rtol=1e-5, atol=1e-5)
    gs = torch.full((1,), 2.0, device=_dev())
    saved = logits.clone()
    ops.ce_fwd_bwd(logits, V, tgt, eps, 1.0 / rows, gs, loss_rows, None, 0.0, True)        # statistics recomputed
    got = logits[:, :V].float()
    ref = 2.0 * lf.grad
    assert (got - ref).abs().max().item() <= 1e-2 * ref.abs().max().item()
    ops.ce_fwd_bwd(saved, V, tgt, eps, 1.0 / rows, gs, loss_rows, None, 0.0, True, lse_rows=lse)   # saved log-sum-exp
    assert torch.equal(saved[:, :V], logits[:, :V])


# ------------------------------------------------------------------ attention
def _ref_attention(q, k, v, valid, causal, scale):
    # q [N,H,S,hd] k,v [N,H,Sk,hd]; valid [N,Sk] bool
    w = (q @ k.transpose(-1, -2)) * scale
    if causal:
        S = q.shape[2]
        w = w + torch.triu(torch.full((S, S), float("-inf"), device=q.device), 1)
    w = w.masked_fill(~valid[:, None, None, :], float("-inf"))
    return torch.softmax(w, -1) @ v


@pytest.mark.parametrize("n_seq", [6, 72])   # 72 sequences: the kernels switch to one CTA per sequence with heads as items
@pytest.mark.parametrize("causal", [False, True])
def test_self_attention_fwd_bwd(causal, n_seq):
    ops = _ops()
    torch.manual_seed(7)
    N, H, S, hd = n_seq, 16, 128, 64
    T = N * S
    qkv = (torch.randn(T, 3 * D, device=_dev()) * 1.0).to(torch.bfloat16)
    lens = torch.randint(20, S + 1, (N,), device=_dev())
    valid = torch.arange(S, device=_dev())[None, :] < lens[:, None]
    kvalid = valid.reshape(-1).to(torch.uint8)
    ctx = torch.empty(T, D, device=_dev(), dtype=torch.bfloat16)
    lse = torch.empty(N, H, 1, S, device=_dev())
    kw = dict(Q=qkv, ldq=3 * D, q_col=0, KV=qkv, ldkv=3 * D, k_col=D, v_col=2 * D, O=ctx, ldo=D, LSE=lse, key_valid=kvalid,
              ent_valid=None, inv_n=None, n_qseq=N, H=H, R=1, causal=int(causal), E_total=1, scale=hd ** -0.5, mods=[(0, 0, 1, S, 0, 0)])
    ops.attn_fwd(ops.attn_args(**kw))
    x = qkv.float().view(N, S, 3, H, hd).requires_grad_(True)
    q, k, v = [x[:, :, i].transpose(1, 2) for i in range(3)]
    ref = _ref_attention(q, k, v, valid, causal, hd ** -0.5).transpose(1, 2).reshape(T, D)
    _close(ctx, ref, 1.5e-2, "attn fwd")
    dctx = torch.randn(T, D, device=_dev()).to(torch.bfloat16)
    ref.backward(dctx.float())
    dqkv = torch.zeros(T, 3 * D, device=_dev(), dtype=torch.bfloat16)
    delta = torch.empty(N, H, 1, S, device=_dev())
    kw.update(O=dctx, DELTA=delta, dQ=dqkv, lddq=3 * D, dq_col=0, dKV=dqkv, lddkv=3 * D, dk_col=D, dv_col=2 * D)
    ops.attn_bwd(ops.attn_args(**kw))
    gref = x.grad.reshape(T, 3 * D)
    for i, nm in enumerate(("dq", "dk", "dv")):
        _close(dqkv[:, i * D:(i + 1) * D], gref[:, i * D:(i + 1) * D], 2e-2, nm)


@pytest.mark.parametrize("n_seq,frame", [(6, 112), (72, 112), (72, 80), (5, 48)])
def test_self_attention_short_frames(n_seq, frame):
    """Encoder self-attention on frames of `frame` < 128 rows per sequence (q_rows in the ABI): the 128-row query tile of a
    sequence then overlaps the next sequence's rows, which must be neither written (forward, dQ) nor allowed to contribute
    (dK/dV).  Every buffer is pre-filled so that a stray write or a foreign contribution shows."""
    ops = _ops()
    torch.manual_seed(9)
    N, H, hd = n_seq, 16, 64
    T = N * frame
    qkv = torch.randn(T, 3 * D, device=_dev()).to(torch.bfloat16)
    lens = torch.randint(10, frame + 1, (N,), device=_dev())
    lens[0] = frame
    valid = torch.arange(frame, device=_dev())[None, :] < lens[:, None]
    kvalid = valid.reshape(-1).to(torch.uint8)
    ctx = torch.full((T + 128, D), 7.0, device=_dev(), dtype=torch.bfloat16)            # + guard rows behind the last frame
    lse = torch.full((N, H, 1, 128), float("nan"), device=_dev())
    kw = dict(Q=qkv, ldq=3 * D, q_col=0, KV=qkv, ldkv=3 * D, k_col=D, v_col=2 * D, O=ctx, ldo=D, LSE=lse, key_valid=kvalid,
              ent_valid=None, inv_n=None, n_qseq=N, H=H, R=1, causal=0, E_total=1, scale=hd ** -0.5, q_rows=frame,
              mods=[(0, 0, 1, frame, 0, 0)])
    ops.debug_poison()
    ops.attn_fwd(ops.attn_args(**kw))
    x = qkv.float().view(N, frame, 3, H, hd).requires_grad_(True)
    q, k, v = [x[:, :, i].transpose(1, 2) for i in range(3)]
    ref = _ref_attention(q, k, v, valid, False, hd ** -0.5).transpose(1, 2).reshape(T, D)
    _close(ctx[:T], ref, 1.5e-2, "short-frame attn fwd")
    assert (ctx[T:] == 7.0).all()                                                         # nothing written behind the last frame
    dctx = torch.randn(T, D, device=_dev()).to(torch.bfloat16)
    ref.backward(dctx.float())
    dqkv = torch.full((T + 128, 3 * D), 7.0, device=_dev(), dtype=torch.bfloat16)
    delta = torch.full((N, H, 1, 128), float("nan"), device=_dev())
    kw.update(O=dctx, DELTA=delta, dQ=dqkv, lddq=3 * D, dq_col=0, dKV=dqkv, lddkv=3 * D, dk_col=D, dv_col=2 * D)
    ops.debug_poison()
    ops.attn_bwd(ops.attn_args(**kw))
    gref = x.grad.reshape(T, 3 * D)
    for i, nm in enumerate(("dq", "dk", "dv")):
        _close(dqkv[:T, i * D:(i + 1) * D], gref[:, i * D:(i + 1) * D], 2e-2, "short-frame " + nm)
    assert (dqkv[T:] == 7.0).all()


@pytest.mark.parametrize("n_seq", [6, 72])
def test_attention_scores_growing_along_the_keys(n_seq):
    """The forward kernel reads every score chunk once and keeps a reference that is raised lazily (csrc/attention_sm100.cu,
    attn_fwd_tc3_kernel): keys whose scores grow by hundreds of nats from chunk to chunk force the raise-and-rescale path on most
    rows (and no raise on the rows whose scores shrink instead).  Output, log-sum-exp (through the backward pass) and
    gradients must still match the max-first softmax of the reference."""
    ops = _ops()
    torch.manual_seed(12)
    N, H, S, hd = n_seq, 16, 128, 64
    T = N * S
    qkv = torch.randn(T, 3 * D, device=_dev())
    ramp = torch.linspace(1.0, 40.0, S, device=_dev()).repeat(N)[:, None]          # key norm grows 40x along the sequence
    u = torch.randn(1, H, 1, hd, device=_dev()).expand(N, H, S, hd).transpose(1, 2).reshape(T, D)
    qkv[:, D:2 * D] = u * ramp                                                         # k_j = ramp_j * u: scores = ramp_j * (q . u)
    qkv = qkv.to(torch.bfloat16)
    lens = torch.randint(100, S + 1, (N,), device=_dev())
    valid = torch.arange(S, device=_dev())[None, :] < lens[:, None]
    kvalid = valid.reshape(-1).to(torch.uint8)
    ctx = torch.empty(T, D, device=_dev(), dtype=torch.bfloat16)
    lse = torch.empty(N, H, 1, S, device=_dev())
    kw = dict(Q=qkv, ldq=3 * D, q_col=0, KV=qkv, ldkv=3 * D, k_col=D, v_col=2 * D, O=ctx, ldo=D, LSE=lse, key_valid=kvalid,
              ent_valid=None, inv_n=None, n_qseq=N, H=H, R=1, causal=0, E_total=1, scale=hd ** -0.5, mods=[(0, 0, 1, S, 0, 0)])
    ops.attn_fwd(ops.attn_args(**kw))
    x = qkv.float().view(N, S, 3, H, hd).requires_grad_(True)
    q, k, v = [x[:, :, i].transpose(1, 2) for i in range(3)]
    w = (q @ k.transpose(-1, -2)) * hd ** -0.5
    assert (w.amax(-1) - w[..., :32].amax(-1)).max().item() > 100.0                    # the raise path is really exercised
    ref = _ref_attention(q, k, v, valid, False, hd ** -0.5).transpose(1, 2).reshape(T, D)
    assert torch.isfinite(ctx.float()).all()
    _close(ctx, ref, 1.5e-2, "attn fwd, growing scores")
    lse_ref = torch.logsumexp(w.masked_fill(~valid[:, None, None, :], float("-inf")), -1) * 1.4426950408889634   # log2 domain
    assert (lse[:, :, 0] - lse_ref).abs().max().item() <= 2e-2 + 1e-3 * lse_ref.abs().max().item()
    dctx = torch.randn(T, D, device=_dev()).to(torch.bfloat16)
    ref.backward(dctx.float())
    dqkv = torch.zeros(T, 3 * D, device=_dev(), dtype=torch.bfloat16)
    delta = torch.empty(N, H, 1, S, device=_dev())
    kw.update(O=dctx, DELTA=delta, dQ=dqkv, lddq=3 * D, dq_col=0, dKV=dqkv, lddkv=3 * D, dk_col=D, dv_col=2 * D)
    ops.attn_bwd(ops.attn_args(**kw))
    gref = x.grad.reshape(T, 3 * D)
    _close(dqkv[:, 2 * D:], gref[:, 2 * D:], 3e-2, "dv, growing scores")


def test_multi_entity_cross_attention_fwd_bwd():
    """Leave-one-out text entities + a partially masked table + images with null entities / a null-image business,
    against the restated reference semantics (per-entity softmax, masked mean, -2^16 fill)."""
    ops = _ops()
    from oracle import mmsum_oracle as OR
    torch.manual_seed(8)
    B, R, S, H, hd, F_, n_img, ik = 2, 3, 128, 16, 64, 47, 3, 196
    N, T = B * R, B * R * S
    Tm = T + B * F_ + B * n_img * ik
    Et = R + 1 + n_img
    dev = _dev()
    qc = torch.randn(T, D, device=dev).to(torch.bfloat16)
    kv = torch.randn(Tm, 2 * D, device=dev).to(torch.bfloat16)
    lens = torch.randint(30, S + 1, (B, R), device=dev)
    tvalid = torch.arange(S, device=dev)[None, None, :] < lens[:, :, None]           # [B,R,S]
    tabvalid = torch.rand(B, 1, F_, device=dev) > 0.3
    tabvalid[:, :, 0] = True
    imask = torch.tensor([[True, False, True], [False, False, False]], device=dev)   # business 1 has no image
    ivalid = imask[:, :, None].expand(B, n_img, ik)
    mem_valid = torch.cat([tvalid.reshape(-1), tabvalid.reshape(-1), ivalid.reshape(-1)]).to(torch.uint8)
    ent_valid = torch.cat([tvalid.any(-1), tabvalid.any(-1), imask], dim=1).to(torch.uint8).contiguous()  # [B, Et]
    inv_n = torch.zeros(N, 3, device=dev)
    for b in range(B):
        for i in range(R):
            nt = int(tvalid[b].any(-1).sum().item()) - 1
            inv_n[b * R + i, 0] = 1.0 / nt
            inv_n[b * R + i, 1] = 1.0
            ni = int(imask[b].sum().item())
            inv_n[b * R + i, 2] = 1.0 / ni if ni > 0 else 0.0
    A3 = torch.empty(3, T, D, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(N, H, Et, S, device=dev)
    mods = [(0, 0, R, S, 1, 0), (T, T * D, 1, F_, 0, R), (T + B * F_, 2 * T * D, n_img, ik, 0, R + 1)]
    kw = dict(Q=qc, ldq=D, q_col=0, KV=kv, ldkv=2 * D, k_col=0, v_col=D, O=A3, ldo=D, LSE=lse, key_valid=mem_valid,
              ent_valid=ent_valid, inv_n=inv_n, n_qseq=N, H=H, R=R, causal=0, E_total=Et, scale=hd ** -0.5, mods=mods)
    ops.attn_fwd(ops.attn_args(**kw))

    # reference: loop over targets exactly like src/multimodal_train.py:150-163 does
    qf = qc.float().requires_grad_(True)
    kvf = kv.float().requires_grad_(True)

    def ref_modality(q_rows, k, v, valid):
        # q_rows [B,S,D]; k,v [B,E,Sk,D]; valid [B,E,Sk]
        Bq, E, Sk = k.shape[0], k.shape[1], k.shape[2]
        q = q_rows.view(Bq, S, H, hd).transpose(1, 2) * hd ** -0.5
        kk = k.view(Bq, E, Sk, H, hd).permute(0, 1, 3, 2, 4)
        vv = v.view(Bq, E, Sk, H, hd).permute(0, 1, 3, 2, 4)
        wgt = q[:, None] @ kk.transpose(-1, -2)
        wgt = wgt.masked_fill(~valid[:, :, None, None, :], OR.NEG_CROSS)
        o = torch.softmax(wgt, -1) @ vv
        null = ~valid.any(-1)
        o = o.masked_fill(null[:, :, None, None, None], 0.0)
        n = (~null).sum(1).clamp(min=1).float()
        return (o.sum(1) / n[:, None, None, None]).transpose(1, 2).reshape(Bq, S, D)

    ktext, vtext = kvf[:T, :D].view(B, R, S, D), kvf[:T, D:].view(B, R, S, D)
    ktab, vtab = kvf[T:T + B * F_, :D].view(B, 1, F_, D), kvf[T:T + B * F_, D:].view(B, 1, F_, D)
    kimg, vimg = kvf[T + B * F_:, :D].view(B, n_img, ik, D), kvf[T + B * F_:, D:].view(B, n_img, ik, D)
    ref = torch.zeros(3, B, R, S, D, device=dev)
    outs = []
    for i in range(R):
        others = [j for j in range(R) if j != i]
        qi = qf.view(B, R, S, D)[:, i]
        outs.append(torch.stack([ref_modality(qi, ktext[:, others], vtext[:, others], tvalid[:, others]),
                                 ref_modality(qi, ktab, vtab, tabvalid),
                                 ref_modality(qi, kimg, vimg, ivalid)]))
    ref = torch.stack(outs, dim=2).reshape(3, T, D)   # [3, B, R, S, D]
    _close(A3, ref, 1.5e-2, "cross fwd")
    assert A3[2].view(B, R * S, D)[1].abs().max().item() == 0.0   # business without images -> exactly 0

    dA3 = torch.randn(3, T, D, device=dev).to(torch.bfloat16)
    ref.backward(dA3.float())
    dqc = torch.zeros(T, D, device=dev, dtype=torch.bfloat16)
    dkv = torch.full((Tm, 2 * D), 7.0, device=dev, dtype=torch.bfloat16)   # must be fully overwritten
    delta = torch.empty(N, H, Et, S, device=dev)
    kw.update(O=dA3, DELTA=delta, dQ=dqc, lddq=D, dq_col=0, dKV=dkv, lddkv=2 * D, dk_col=0, dv_col=D)
    ops.attn_bwd(ops.attn_args(**kw))
    _close(dqc, qf.grad, 2e-2, "cross dq")
    _close(dkv[:, :D], kvf.grad[:, :D], 2e-2, "cross dk")
    _close(dkv[:, D:], kvf.grad[:, D:], 2e-2, "cross dv")


def _stale_state_cross_case(seed):
    """Multi-entity cross-attention with null images inside packed dK/dV tiles, ragged reviews and a masked table."""
    torch.manual_seed(seed)
    B, R, S, H, hd, F_, n_img, ik = 3, 4, 128, 16, 64, 47, 3, 196
    N, T = B * R, B * R * S
    Tm = T + B * F_ + B * n_img * ik
    Et = R + 1 + n_img
    dev = _dev()
    qc = torch.randn(T, D, device=dev).to(torch.bfloat16)
    kv = torch.randn(Tm, 2 * D, device=dev).to(torch.bfloat16)
    lens = torch.randint(30, S + 1, (B, R), device=dev)
    tvalid = torch.arange(S, device=dev)[None, None, :] < lens[:, :, None]
    tabvalid = torch.rand(B, 1, F_, device=dev) > 0.3
    tabvalid[:, :, 0] = True
    imask = torch.tensor([[True, False, False], [False, False, False], [False, True, True]], device=dev)
    ivalid = imask[:, :, None].expand(B, n_img, ik)
    mem_valid = torch.cat([tvalid.reshape(-1), tabvalid.reshape(-1), ivalid.reshape(-1)]).to(torch.uint8)
    ent_valid = torch.cat([tvalid.any(-1), tabvalid.any(-1), imask], dim=1).to(torch.uint8).contiguous()
    inv_n = torch.zeros(N, 3, device=dev)
    ni = imask.sum(1).float()
    inv_n[:, 0] = 1.0 / (R - 1)
    inv_n[:, 1] = 1.0
    inv_n[:, 2] = torch.where(ni > 0, 1.0 / ni.clamp(min=1), torch.zeros_like(ni)).repeat_interleave(R)
    mods = [(0, 0, R, S, 1, 0), (T, T * D, 1, F_, 0, R), (T + B * F_, 2 * T * D, n_img, ik, 0, R + 1)]
    kw = dict(Q=qc, ldq=D, q_col=0, KV=kv, ldkv=2 * D, k_col=0, v_col=D, ldo=D, key_valid=mem_valid, ent_valid=ent_valid,
              inv_n=inv_n, n_qseq=N, H=H, R=R, causal=0, E_total=Et, scale=hd ** -0.5, mods=mods)
    dA3 = torch.randn(3, T, D, device=dev).to(torch.bfloat16)
    return kw, dA3, (N, H, Et, S, T, Tm)


def test_kernels_ignore_stale_onchip_state():
    """Masked score columns, pad keys and null entities are handled by SELECTING zeros, never by multiplying stale data by
    zero: with every SM's shared / tensor memory and every unwritten LSE / DELTA row filled with NaN patterns before each
    launch, forward and backward attention (deterministic kernels, no atomics) and a ragged GEMM must return exactly the
    bits of an unpoisoned run.  (Found in round 2: 0 * stale dP' columns beyond n16 in the dQ kernel, and 0 * DELTA of a
    null image inside a packed dK/dV tile, turned every gradient into NaN depending on which kernel ran before.)"""
    ops = _ops()
    kw, dA3, (N, H, Et, S, T, Tm) = _stale_state_cross_case(21)
    dev = _dev()

    def run(poisoned):
        fill = float("nan") if poisoned else 0.0
        A3 = torch.full((3, T, D), fill, device=dev, dtype=torch.bfloat16)
        lse = torch.full((N, H, Et, S), fill, device=dev)
        delta = torch.full((N, H, Et, S), fill, device=dev)
        dqc = torch.full((T, D), fill, device=dev, dtype=torch.bfloat16)
        dkv = torch.full((Tm, 2 * D), fill, device=dev, dtype=torch.bfloat16)
        if poisoned:
            ops.debug_poison()
        ops.attn_fwd(ops.attn_args(O=A3, LSE=lse, **kw))
        if poisoned:
            ops.debug_poison()
        ops.attn_bwd(ops.attn_args(O=dA3, LSE=lse, DELTA=delta, dQ=dqc, lddq=D, dq_col=0, dKV=dkv, lddkv=2 * D, dk_col=0,
                                   dv_col=D, **kw))
        torch.cuda.synchronize()
        return A3, dqc, dkv

    clean = run(False)
    for _ in range(2):
        dirty = run(True)
        for nm, a, b in zip(("out", "dq", "dkv"), clean, dirty):
            assert torch.isfinite(b.float()).all(), nm
            assert torch.equal(a, b), nm
    # causal self-attention with pad keys, entity mode (6 sequences) and head mode (72)
    for n_seq in (6, 72):
        torch.manual_seed(5)
        N, H, S, hd = n_seq, 16, 128, 64
        T = N * S
        qkv = torch.randn(T, 3 * D, device=_dev()).to(torch.bfloat16)
        lens = torch.randint(20, S + 1, (N,), device=_dev())
        kvalid = (torch.arange(S, device=_dev())[None, :] < lens[:, None]).reshape(-1).to(torch.uint8)
        dctx = torch.randn(T, D, device=_dev()).to(torch.bfloat16)
        res = []
        for poisoned in (False, True):
            fill = float("nan") if poisoned else 0.0
            ctx = torch.full((T, D), fill, device=_dev(), dtype=torch.bfloat16)
            lse = torch.full((N, H, 1, S), fill, device=_dev())
            delta = torch.full((N, H, 1, S), fill, device=_dev())
            dqkv = torch.full((T, 3 * D), fill, device=_dev(), dtype=torch.bfloat16)
            kw = dict(Q=qkv, ldq=3 * D, q_col=0, KV=qkv, ldkv=3 * D, k_col=D, v_col=2 * D, ldo=D, LSE=lse, key_valid=kvalid,
                      ent_valid=None, inv_n=None, n_qseq=N, H=H, R=1, causal=1, E_total=1, scale=hd ** -0.5, mods=[(0, 0, 1, S, 0, 0)])
            if poisoned:
                ops.debug_poison()
            ops.attn_fwd(ops.attn_args(O=ctx, **kw))
            if poisoned:
                ops.debug_poison()
            ops.attn_bwd(ops.attn_args(O=dctx, DELTA=delta, dQ=dqkv, lddq=3 * D, dq_col=0, dKV=dqkv, lddkv=3 * D, dk_col=D,
                                       dv_col=2 * D, **kw))
            torch.cuda.synchronize()
            res.append((ctx, dqkv))
        for nm, a, b in zip(("self out", "self dqkv"), res[0], res[1]):
            assert torch.isfinite(b.float()).all(), (nm, n_seq)
            assert torch.equal(a, b), (nm, n_seq)
    # ragged GEMM (TMA zero fill on M, N and K edges), bf16 and fp32-accumulating outputs
    torch.manual_seed(6)
    A = torch.randn(1000, 520, device=_dev()).to(torch.bfloat16)
    Bm = torch.randn(776, 520, device=_dev()).to(torch.bfloat16)
    ref = ops.gemm(A, Bm)
    ops.debug_poison()
    got = ops.gemm(A, Bm)
    assert torch.equal(ref, got)
    A = torch.randn(2400, 1000, device=_dev()).to(torch.bfloat16)      # CTA-pair kernel
    Bm = torch.randn(2040, 1000, device=_dev()).to(torch.bfloat16)
    ref = ops.gemm(A, Bm)
    ops.debug_poison()
    got = ops.gemm(A, Bm)
    assert torch.equal(ref, got)


# ------------------------------------------------------------------ decode-step attention
@pytest.mark.parametrize("beams,Sk_text", [(4, 158), (1, 128), (8, 208)])
def test_decode_cross_attention(beams, Sk_text):
    """One query row per hypothesis, the beams of a business share its un-expanded memory: text entities with ragged valid
    lengths, a partially masked table, images with null entities and a business without images."""
    ops = _ops()
    from oracle import mmsum_oracle as OR
    torch.manual_seed(11)
    B, R, H, hd, F_, n_img, ik = 3, 4, 16, 64, 47, 3, 196
    N = B * beams
    Tt = B * R * Sk_text
    Tm = Tt + B * F_ + B * n_img * ik
    Et = R + 1 + n_img
    dev = _dev()
    q = torch.randn(N, D, device=dev).to(torch.bfloat16)
    kv = torch.randn(Tm, 2 * D, device=dev).to(torch.bfloat16)
    lens = torch.randint(30, Sk_text + 1, (B, R), device=dev)
    tvalid = torch.arange(Sk_text, device=dev)[None, None, :] < lens[:, :, None]
    tvalid[0, 1] = False                                                             # a null review
    tabvalid = torch.rand(B, 1, F_, device=dev) > 0.3
    tabvalid[:, :, 0] = True
    imask = torch.tensor([[True, False, True], [False, False, False], [True, True, True]], device=dev)
    ivalid = imask[:, :, None].expand(B, n_img, ik)
    mem_valid = torch.cat([tvalid.reshape(-1), tabvalid.reshape(-1), ivalid.reshape(-1)]).to(torch.uint8)
    ent_valid = torch.cat([tvalid.any(-1), tabvalid.any(-1), imask], dim=1).to(torch.uint8).contiguous()
    cnt = torch.stack([tvalid.any(-1).sum(1), tabvalid.any(-1).sum(1), imask.sum(1)], dim=1).float()
    inv_n = torch.where(cnt > 0, 1.0 / cnt.clamp(min=1), torch.zeros_like(cnt)).repeat_interleave(beams, dim=0).contiguous()
    A3 = torch.full((3, N, D), 7.0, device=dev, dtype=torch.bfloat16)               # must be fully overwritten
    mods = [(0, 0, R, Sk_text, 0, 0), (Tt, N * D, 1, F_, 0, R), (Tt + B * F_, 2 * N * D, n_img, ik, 0, R + 1)]
    a = ops.attn_args(Q=q, ldq=D, q_col=0, KV=kv, ldkv=2 * D, k_col=0, v_col=D, O=A3, ldo=D, LSE=None, key_valid=mem_valid,
                      ent_valid=ent_valid, inv_n=inv_n, n_qseq=N, H=H, R=beams, causal=0, E_total=Et, scale=hd ** -0.5, mods=mods)
    ops.attn_decode_cross(a)
    kvf, qf = kv.float(), q.float().view(B, beams, H, hd).transpose(1, 2) * hd ** -0.5   # [B,H,beams,hd]

    def ref_modality(k, v, valid):
        E, Sk = k.shape[1], k.shape[2]
        kk = k.view(B, E, Sk, H, hd).permute(0, 1, 3, 2, 4)
        vv = v.view(B, E, Sk, H, hd).permute(0, 1, 3, 2, 4)
        wgt = (qf[:, None] @ kk.transpose(-1, -2)).masked_fill(~valid[:, :, None, None, :], OR.NEG_CROSS)
        o = (torch.softmax(wgt, -1) @ vv).masked_fill((~valid.any(-1))[:, :, None, None, None], 0.0)
        n = valid.any(-1).sum(1).clamp(min=1).float()
        return (o.sum(1) / n[:, None, None, None]).transpose(1, 2).reshape(N, D)

    ref = torch.stack([
        ref_modality(kvf[:Tt, :D].view(B, R, Sk_text, D), kvf[:Tt, D:].view(B, R, Sk_text, D), tvalid),
        ref_modality(kvf[Tt:Tt + B * F_, :D].view(B, 1, F_, D), kvf[Tt:Tt + B * F_, D:].view(B, 1, F_, D), tabvalid),
        ref_modality(kvf[Tt + B * F_:, :D].view(B, n_img, ik, D), kvf[Tt + B * F_:, D:].view(B, n_img, ik, D), ivalid)])
    _close(A3, ref, 1.5e-2, "decode cross")
    assert A3[2].view(B, beams, D)[1].abs().max().item() == 0.0                     # business without images -> exactly 0


def test_decode_self_attention_with_slot_table():
    """Token-by-token causal self-attention against caches that never move: after every step the hypotheses are re-ranked
    (children may share a parent) by permuting the slot table only."""
    ops = _ops()
    torch.manual_seed(12)
    N, H, hd, S = 12, 16, 64, 128
    dev = _dev()
    cache = torch.zeros(N, S, 2 * D, device=dev, dtype=torch.bfloat16)
    hist = torch.zeros(N, S, device=dev, dtype=torch.int32)
    pos = torch.zeros(1, device=dev, dtype=torch.int32)
    out = torch.empty(N, D, device=dev, dtype=torch.bfloat16)
    Kh = torch.zeros(N, S, D, device=dev)     # reference: per-hypothesis history, physically re-gathered as the reference does
    Vh = torch.zeros(N, S, D, device=dev)
    g = torch.Generator().manual_seed(3)
    for t in range(40):
        qkv = torch.randn(N, 3 * D, device=dev).to(torch.bfloat16)
        ops.attn_decode_self(qkv, cache, hist, pos, out, H, hd ** -0.5)
        Kh[:, t], Vh[:, t] = qkv[:, D:2 * D].float(), qkv[:, 2 * D:].float()
        qf = qkv[:, :D].float().view(N, H, 1, hd) * hd ** -0.5
        kk = Kh[:, :t + 1].view(N, t + 1, H, hd).transpose(1, 2)
        vv = Vh[:, :t + 1].view(N, t + 1, H, hd).transpose(1, 2)
        ref = (torch.softmax(qf @ kk.transpose(-1, -2), -1) @ vv).transpose(1, 2).reshape(N, D)
        _close(out, ref, 1.5e-2, "decode self t=%d" % t)
        src = ((torch.arange(N) // 4) * 4 + torch.randint(0, 4, (N,), generator=g)).to(dev)
        hist.copy_(hist.index_select(0, src))
        Kh, Vh = Kh[src], Vh[src]
        pos += 1


# ------------------------------------------------------------------ gates
def test_gate_fwd_bwd():
    ops = _ops()
    torch.manual_seed(9)
    nb, rpb = 3, 256
    rows = nb * rpb
    dev = _dev()
    o3 = torch.randn(3, rows, D, device=dev).to(torch.bfloat16)
    u = torch.randn(2, rows, D, device=dev).to(torch.bfloat16)
    pres = torch.tensor([[1, 1], [1, 0], [0, 1]], device=dev, dtype=torch.uint8)
    y = torch.empty(rows, D, device=dev, dtype=torch.bfloat16)
    ab = torch.empty(2, rows, D, device=dev, dtype=torch.bfloat16)
    ops.gate_fwd(o3, u, pres, y, ab, rows, rpb, D)
    of, uf = o3.float().requires_grad_(True), u.float().requires_grad_(True)
    pm = pres.float().repeat_interleave(rpb, 0)
    alpha = torch.relu(torch.tanh(uf[0])) * pm[:, :1]
    beta = torch.relu(torch.tanh(uf[1])) * pm[:, 1:]
    ref = of[0] + alpha * of[1] + beta * of[2]
    _close(y, ref, 1e-2, "gate y")
    dy = torch.randn(rows, D, device=dev).to(torch.bfloat16)
    ref.backward(dy.float())
    du = torch.empty_like(u)
    ops.gate_bwd_u(dy, o3, ab, du, rows, D)
    _close(du, uf.grad, 2e-2, "gate du")
    dca = torch.randn(rows, 2 * D, device=dev).to(torch.bfloat16)
    dcb = torch.randn(rows, 2 * D, device=dev).to(torch.bfloat16)
    do3 = torch.empty_like(o3)
    ops.gate_bwd_o(dy, ab, dca, dcb, do3, rows, D)
    exp = of.grad.clone()
    exp[0] += dca[:, :D].float() + dcb[:, :D].float()
    exp[1] += dca[:, D:].float()
    exp[2] += dcb[:, D:].float()
    _close(do3, exp, 2e-2, "gate dO3")


# ------------------------------------------------------------------ integer bookkeeping + table front end
# (ids, masks, validity: bit-exact; the bf16 sum-pooled table features: equal up to the summation order of the fp32 pool, i.e.
#  the rare element whose fp32 sum sits on a bf16 rounding boundary may differ by one ulp)
@pytest.mark.parametrize("dataset", ["yelp", "amazon"])
def test_prep_and_table_exact(dataset):
    ops = _ops()
    from multimodalsum_b200.synth import ModelConfig, make_batch, make_state_dict
    from oracle import mmsum_oracle as OR
    cfg = ModelConfig(encoder_layers=1, decoder_layers=1, ffn_dim=64, vocab_size=512, max_position_embeddings=128, dataset=dataset)
    sd = make_state_dict(cfg, seed=11)
    B, R, S = 3, 4, 128
    batch = make_batch(cfg, B, seed=12, n_reviews=R, max_imgs=2).to(_dev())
    dev = _dev()
    F_ = 47 if dataset == "yelp" else 133
    n_img, ik = batch.img.shape[1], 196
    E = sd["bart_model.model.shared.weight"].to(dev)
    t = "table_encoder."
    if dataset == "yelp":
        W0, W1 = sd[t + "rating_embedding.weight"].to(dev), sd[t + "hours_embedding.weight"].to(dev)
    else:
        W0, W1 = sd[t + "price_embedding.weight"].to(dev), sd[t + "rating_embedding.weight"].to(dev)
    X = torch.empty(B * F_, 2 * D, device=dev, dtype=torch.bfloat16)
    tv = torch.zeros(B, F_, device=dev, dtype=torch.uint8)
    ops.table_fwd(dataset, B, E, batch.field, batch.field_value, W0, W1, X, tv)
    # oracle front end: rebuild the [names | values] matrix the way the reference does
    p = {k: v.to(dev) for k, v in sd.items() if k.startswith("table_encoder.")}
    captured = {}
    orig = OR._lin

    def spy(x, pp, name, bias=True):
        if name.endswith("table_encoder.fc"):
            captured["x"] = x
        return orig(x, pp, name, bias)

    OR._lin = spy
    try:
        enc = OR.yelp_table_encoder if dataset == "yelp" else OR.amazon_table_encoder
        _, valid = enc(p, batch.field, batch.field_value)
    finally:
        OR._lin = orig
    assert torch.equal(tv.bool(), valid)
    ref = captured["x"].reshape(B * F_, 2 * D)
    refb = ref.to(torch.bfloat16)
    neq = X != refb
    assert neq.float().mean().item() <= 2e-3, neq.float().mean().item()                       # rounding-boundary ties only
    assert ((X.float() - refb.float()).abs() <= refb.float().abs() * 2.0 ** -7 + 1e-30).all()     # ... and at most one ulp apart

    T = B * R * S
    Tm = T + B * F_ + B * n_img * ik
    Et = R + 1 + n_img
    i32 = lambda n: torch.zeros(n, device=dev, dtype=torch.int32)
    u8 = lambda *s: torch.zeros(s, device=dev, dtype=torch.uint8)
    outs = dict(enc_ids=i32(T), dec_ids=i32(T), labels=i32(T), enc_valid=u8(T), dec_valid=u8(T), mem_valid=u8(Tm),
                ent_valid=u8(B, Et), pres=u8(B, 2), rating_diff=torch.zeros(B * R, device=dev), inv_n=torch.zeros(B * R, 3, device=dev))
    ops.prep_step(batch.reviews, batch.reviews_mask, batch.reviews_rating, tv, batch.img_mask.view(torch.uint8),
                  B=B, R=R, S=S, F=F_, n_img=n_img, img_keys=ik, n_mod=3, pad_id=1, bos_id=0, eos_id=2, **outs)
    for i in range(R):
        ref_ids = OR.shift_tokens_right(batch.reviews[:, i], 1, 0, 2)
        got = outs["dec_ids"].view(B, R, S)[:, i]
        assert torch.equal(got.long(), ref_ids)
        others = [j for j in range(R) if j != i]
        rd = batch.reviews_rating[:, i] - batch.reviews_rating[:, others].mean(1)
        assert torch.allclose(outs["rating_diff"].view(B, R)[:, i], rd, atol=1e-6)
    assert torch.equal(outs["enc_ids"].long(), batch.reviews.reshape(-1))
    assert torch.equal(outs["dec_valid"].bool(), outs["dec_ids"] != 1)
    assert torch.equal(outs["mem_valid"][:T].bool(), batch.reviews_mask.reshape(-1).bool())
    assert torch.equal(outs["mem_valid"][T:T + B * F_].bool(), valid.reshape(-1))
    assert torch.equal(outs["mem_valid"][T + B * F_:].view(B, n_img, ik)[:, :, 0].bool(), batch.img_mask)
    assert torch.equal(outs["pres"][:, 1].bool(), batch.img_mask.any(1))
    # trimmed encoder frame (S_enc): the encoder-side arrays hold the first S_enc tokens of every review, everything else is unchanged
    S_enc = min(S, (int(batch.reviews_mask.sum(-1).max().item()) + 15) // 16 * 16)
    o2 = dict(enc_ids=i32(T), dec_ids=i32(T), labels=i32(T), enc_valid=u8(T), dec_valid=u8(T), mem_valid=u8(Tm),
              ent_valid=u8(B, Et), pres=u8(B, 2), rating_diff=torch.zeros(B * R, device=dev), inv_n=torch.zeros(B * R, 3, device=dev))
    ops.prep_step(batch.reviews, batch.reviews_mask, batch.reviews_rating, tv, batch.img_mask.view(torch.uint8),
                  B=B, R=R, S=S, S_enc=S_enc, F=F_, n_img=n_img, img_keys=ik, n_mod=3, pad_id=1, bos_id=0, eos_id=2, **o2)
    Te = B * R * S_enc
    assert torch.equal(o2["enc_ids"][:Te].long(), batch.reviews[:, :, :S_enc].reshape(-1))
    assert torch.equal(o2["enc_valid"][:Te].bool(), batch.reviews_mask[:, :, :S_enc].reshape(-1).bool())
    assert torch.equal(o2["mem_valid"][:Te].bool(), batch.reviews_mask[:, :, :S_enc].reshape(-1).bool())
    assert torch.equal(o2["mem_valid"][Te:Te + B * F_].bool(), valid.reshape(-1))
    assert torch.equal(o2["mem_valid"][Te + B * F_:Te + B * F_ + B * n_img * ik], outs["mem_valid"][T + B * F_:])
    for k in ("dec_ids", "labels", "dec_valid", "ent_valid", "pres", "rating_diff", "inv_n"):
        assert torch.equal(o2[k], outs[k]), k
