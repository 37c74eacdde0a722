"""Thin torch-tensor -> C-ABI wrappers.  torch is used for device memory and streams only."""
import ctypes as C

import torch

from . import _lib
from ._lib import GemmArgs
from ._lib import check as _check_rc

LAUNCHES = 0      # kernels launched through the C-ABI since import (bench.py: gpu_launches)
# Optional instrumentation hook (bench.py roofline): callable(kind, work) -> context manager that brackets ONE C-ABI call with
# CUDA events on the launching stream.  kind / work: "gemm" FLOPs; "attn_fwd" / "attn_bwd" FLOPs; row kernels algorithmic bytes.
KERNEL_TIMER = None

ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2
AUX_NONE, AUX_STORE_PREACT, AUX_MUL_DACT, AUX_STORE_DACT, AUX_MUL = 0, 1, 2, 3, 4


def check(rc, what, n_kernels=1):
    global LAUNCHES
    _check_rc(rc, what)
    LAUNCHES += n_kernels


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _check2d(t, name, dtype=None):
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError("%s must be 2-D with unit inner stride, got %s / %s" % (name, tuple(t.shape), t.stride()))
    if dtype is not None and t.dtype != dtype:
        raise ValueError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor (no CPU fallback)" % name)


def gemm(A, B, out=None, *, a_t=False, b_t=False, out_dtype=torch.bfloat16, bias=None, act=ACT_NONE,
         aux=None, aux_mode=AUX_NONE, alpha=1.0, accumulate=False, splits=0, block_n=0, raster_m_fast=False):
    """out[M,N] (+)= epi(alpha * A·Bᵀ).

    A: [M,K] (a_t=False) or [K,M] (a_t=True, read MN-major, no copy); B: [N,K] or [K,N] (b_t=True).
    """
    _check2d(A, "A", torch.bfloat16)
    _check2d(B, "B", torch.bfloat16)
    if a_t:
        K, M = A.shape
    else:
        M, K = A.shape
    if b_t:
        Kb, N = B.shape
    else:
        N, Kb = B.shape
    if K != Kb:
        raise ValueError("contraction mismatch: %d vs %d" % (K, Kb))
    if out is None:
        out = torch.empty((M, N), device=A.device, dtype=out_dtype)
        if accumulate:
            out.zero_()
    _check2d(out, "out")
    if tuple(out.shape) != (M, N):
        raise ValueError("out shape %s != (%d,%d)" % (tuple(out.shape), M, N))
    if out.dtype not in (torch.bfloat16, torch.float32):
        raise ValueError("out must be bf16 or fp32")
    if bias is not None and (bias.dtype != torch.float32 or bias.numel() != N or not bias.is_contiguous()):
        raise ValueError("bias must be contiguous fp32 [N]")
    if aux_mode != AUX_NONE:
        _check2d(aux, "aux", torch.bfloat16)
    a = GemmArgs()
    a.A, a.B, a.D = A.data_ptr(), B.data_ptr(), out.data_ptr()
    a.lda, a.ldb, a.ldd = A.stride(0), B.stride(0), out.stride(0)
    a.M, a.N, a.K = M, N, K
    a.a_mn_major, a.b_mn_major = int(a_t), int(b_t)
    a.out_f32 = int(out.dtype == torch.float32)
    a.accumulate = int(accumulate)
    a.splits, a.block_n, a.raster_m_fast = splits, block_n, int(raster_m_fast)
    a.alpha = alpha
    a.bias = bias.data_ptr() if bias is not None else None
    a.act, a.aux_mode = act, aux_mode
    a.aux = aux.data_ptr() if aux is not None else None
    a.ld_aux = aux.stride(0) if aux is not None else 0
    if KERNEL_TIMER is not None:
        with KERNEL_TIMER("gemm", 2.0 * M * N * K):
            check(_lib.lib().mmsum_gemm_bf16(C.byref(a), _stream()), "mmsum_gemm_bf16")
    else:
        check(_lib.lib().mmsum_gemm_bf16(C.byref(a), _stream()), "mmsum_gemm_bf16")
    return out


def gemm_cat(A, A2, B, out=None, *, bias=None, out_dtype=torch.bfloat16):
    """out = [A | A2]·Bᵀ + bias with the concatenation along K done by the TMA producer (no cat buffer)."""
    _check2d(A, "A", torch.bfloat16)
    _check2d(A2, "A2", torch.bfloat16)
    _check2d(B, "B", torch.bfloat16)
    M, K1 = A.shape
    K = K1 + A2.shape[1]
    N = B.shape[0]
    if A2.shape[0] != M or B.shape[1] != K:
        raise ValueError("gemm_cat shape mismatch")
    if out is None:
        out = torch.empty((M, N), device=A.device, dtype=out_dtype)
    a = GemmArgs()
    a.A, a.B, a.D = A.data_ptr(), B.data_ptr(), out.data_ptr()
    a.lda, a.ldb, a.ldd = A.stride(0), B.stride(0), out.stride(0)
    a.M, a.N, a.K = M, N, K
    a.out_f32 = int(out.dtype == torch.float32)
    a.alpha = 1.0
    a.bias = bias.data_ptr() if bias is not None else None
    a.A2, a.lda2, a.k_split = A2.data_ptr(), A2.stride(0), K1
    if KERNEL_TIMER is not None:
        with KERNEL_TIMER("gemm", 2.0 * M * N * K):
            check(_lib.lib().mmsum_gemm_bf16(C.byref(a), _stream()), "mmsum_gemm_bf16(cat)")
    else:
        check(_lib.lib().mmsum_gemm_bf16(C.byref(a), _stream()), "mmsum_gemm_bf16(cat)")
    return out


def _timed(kind, work, fn):
    if KERNEL_TIMER is None:
        return fn()
    with KERNEL_TIMER(kind, work):
        return fn()


def cast_bf16(src, dst):
    check(_lib.lib().mmsum_cast_f32_bf16(_ptr(src), _ptr(dst), C.c_int64(src.numel()), _stream()), "mmsum_cast_f32_bf16")
    return dst


def embed_ln_fwd(ids, E, P, rating_diff, remb, gamma, beta, out, mean, rstd, rows, S, p_drop, seed, sid, step_dev=None):
    # algorithmic bytes: one fp32 table row read + one bf16 row written per token (positions / LN parameters stay in L2)
    _timed("embed_ln_fwd", rows * E.shape[1] * 6.0, lambda: _embed_ln_fwd(ids, E, P, rating_diff, remb, gamma, beta, out, mean, rstd, rows, S, p_drop, seed, sid, step_dev))


def _embed_ln_fwd(ids, E, P, rating_diff, remb, gamma, beta, out, mean, rstd, rows, S, p_drop, seed, sid, step_dev):
    check(_lib.lib().mmsum_embed_ln_fwd(_ptr(ids), _ptr(E), _ptr(P), _ptr(rating_diff), _ptr(remb), _ptr(gamma), _ptr(beta),
                                        _ptr(out), _ptr(mean), _ptr(rstd), rows, S, E.shape[1], C.c_float(p_drop),
                                        C.c_uint64(seed), C.c_uint32(sid), _ptr(step_dev), _stream()), "mmsum_embed_ln_fwd")


def embed_ln_bwd(dout, dout2, ids, E, P, rating_diff, remb, gamma, mean, rstd, dE, dP, dremb, dgamma, dbeta, dz, rows, S,
                 pad_id, p_drop, seed, sid, step_dev=None):
    check(_lib.lib().mmsum_embed_ln_bwd(_ptr(dout), _ptr(dout2), _ptr(ids), _ptr(E), _ptr(P), _ptr(rating_diff), _ptr(remb),
                                        _ptr(gamma), _ptr(mean), _ptr(rstd), _ptr(dE), _ptr(dP), _ptr(dremb), _ptr(dgamma),
                                        _ptr(dbeta), _ptr(dz), rows, S, E.shape[1], pad_id, C.c_float(p_drop),
                                        C.c_uint64(seed), C.c_uint32(sid), _ptr(step_dev), _stream()), "mmsum_embed_ln_bwd", 2)


def add_ln_fwd(res, y, gamma, beta, out, mean, rstd, p_drop, seed, sid, step_dev=None):
    rows, d = res.shape
    _timed("add_ln_fwd", 3.0 * rows * d * 2, lambda: _add_ln_fwd(res, y, gamma, beta, out, mean, rstd, p_drop, seed, sid, step_dev))


def _add_ln_fwd(res, y, gamma, beta, out, mean, rstd, p_drop, seed, sid, step_dev):
    rows, d = res.shape
    check(_lib.lib().mmsum_add_ln_fwd(_ptr(res), _ptr(y), _ptr(gamma), _ptr(beta), _ptr(out), _ptr(mean), _ptr(rstd), rows, d,
                                      C.c_float(p_drop), C.c_uint64(seed), C.c_uint32(sid), _ptr(step_dev), _stream()), "mmsum_add_ln_fwd")


def add_ln_bwd(d1, d2, res, y, gamma, mean, rstd, dres, dy, dgamma, dbeta, p_drop, seed, sid, step_dev=None):
    rows, d = res.shape
    n_mats = 3 + (1 if d2 is not None else 0) + 1 + (1 if dy.data_ptr() != dres.data_ptr() else 0)   # d1 (+d2), res, y in; dres (+dy) out
    _timed("add_ln_bwd", float(n_mats) * rows * d * 2, lambda: _add_ln_bwd(d1, d2, res, y, gamma, mean, rstd, dres, dy, dgamma, dbeta, p_drop, seed, sid, step_dev))


def _add_ln_bwd(d1, d2, res, y, gamma, mean, rstd, dres, dy, dgamma, dbeta, p_drop, seed, sid, step_dev):
    rows, d = res.shape
    check(_lib.lib().mmsum_add_ln_bwd(_ptr(d1), _ptr(d2), _ptr(res), _ptr(y), _ptr(gamma), _ptr(mean), _ptr(rstd), _ptr(dres),
                                      _ptr(dy), _ptr(dgamma), _ptr(dbeta), rows, d, C.c_float(p_drop), C.c_uint64(seed),
                                      C.c_uint32(sid), _ptr(step_dev), _stream()), "mmsum_add_ln_bwd")


def colsum(x, out):
    """out[n] += Σ_r x[r, n]  (x bf16 2-D, possibly a column-slice view)."""
    _check2d(x, "x", torch.bfloat16)
    _timed("colsum", 2.0 * x.shape[0] * x.shape[1], lambda: _colsum(x, out))


def _colsum(x, out):
    check(_lib.lib().mmsum_colsum(_ptr(x), C.c_int64(x.stride(0)), x.shape[0], x.shape[1], _ptr(out), _stream()), "mmsum_colsum")


def gate_fwd(o3, u, pres, y, ab, rows, rows_per_biz, d):
    _timed("gate", 8.0 * rows * d * 2, lambda: _gate_fwd(o3, u, pres, y, ab, rows, rows_per_biz, d))


def _gate_fwd(o3, u, pres, y, ab, rows, rows_per_biz, d):
    check(_lib.lib().mmsum_gate_fwd(_ptr(o3), _ptr(u), _ptr(pres), _ptr(y), _ptr(ab), rows, rows_per_biz, d, _stream()), "mmsum_gate_fwd")


def gate_bwd_u(dy, o3, ab, du, rows, d):
    _timed("gate", 8.0 * rows * d * 2, lambda: _gate_bwd_u(dy, o3, ab, du, rows, d))


def _gate_bwd_u(dy, o3, ab, du, rows, d):
    check(_lib.lib().mmsum_gate_bwd_u(_ptr(dy), _ptr(o3), _ptr(ab), _ptr(du), rows, d, _stream()), "mmsum_gate_bwd_u")


def gate_bwd_o(dy, ab, dca, dcb, do3, rows, d):
    _timed("gate", 10.0 * rows * d * 2, lambda: _gate_bwd_o(dy, ab, dca, dcb, do3, rows, d))


def _gate_bwd_o(dy, ab, dca, dcb, do3, rows, d):
    check(_lib.lib().mmsum_gate_bwd_o(_ptr(dy), _ptr(ab), _ptr(dca), _ptr(dcb), _ptr(do3), rows, d, _stream()), "mmsum_gate_bwd_o")


def ce_fwd_bwd(logits, V, target, eps, gscale, gscale_dev, loss_rows, loss_out, loss_scale, write_grad, lse_rows=None):
    """lse_rows (optional fp32 [rows]): written by the loss pass, read by the gradient pass (one read of the logits, not two)."""
    rows = logits.shape[0]
    _timed("ce_bwd" if write_grad else "ce_fwd", (2.0 if write_grad else 1.0) * rows * V * 2,
           lambda: _ce_fwd_bwd(logits, V, target, eps, gscale, gscale_dev, loss_rows, loss_out, loss_scale, write_grad, lse_rows))


def _ce_fwd_bwd(logits, V, target, eps, gscale, gscale_dev, loss_rows, loss_out, loss_scale, write_grad, lse_rows):
    rows = logits.shape[0]
    check(_lib.lib().mmsum_ce_fwd_bwd(_ptr(logits), C.c_int64(logits.stride(0)), rows, V, _ptr(target),
                                      C.c_float(-1.0 if eps is None else eps), C.c_float(gscale), _ptr(gscale_dev),
                                      _ptr(loss_rows), _ptr(loss_out), C.c_float(loss_scale), _ptr(lse_rows), int(write_grad), _stream()),
          "mmsum_ce_fwd_bwd", 2 if loss_out is not None else 1)


def attn_args(**kw):
    a = _lib.AttnArgs()
    mods = kw.pop("mods")
    for k, v in kw.items():
        if isinstance(v, torch.Tensor):
            v = v.data_ptr()
        setattr(a, k, v)
    a.n_mod = len(mods)
    for i, m in enumerate(mods):
        a.mods[i].kv_row_base, a.mods[i].o_off, a.mods[i].E, a.mods[i].Sk, a.mods[i].loo, a.mods[i].ent_base = m[:6]
        a.mods[i].ent_stride = m[6] if len(m) > 6 else 0
    return a


def attn_flops(a):
    """Algorithmic forward FLOPs of one attention call (SURVEY App. C): QK^T + PV over dense 128 x keys tiles of every
    (sequence, head, entity) pair that is attended (the leave-one-out entity excluded; causal / pad savings not credited)."""
    keys = 0
    for i in range(a.n_mod):
        m = a.mods[i]
        keys += (m.E - (1 if m.loo else 0)) * m.Sk
    return 4.0 * 128 * 64 * keys * a.n_qseq * a.H


def attn_fwd(a):
    kind = "attn_self_fwd" if a.n_mod == 1 and a.mods[0].E == 1 else "attn_cross_fwd"
    _timed(kind, attn_flops(a), lambda: check(_lib.lib().mmsum_attn_fwd(C.byref(a), _stream()), "mmsum_attn_fwd"))


def attn_bwd(a):
    # backward = 2.5 x forward algorithmic FLOPs (S, dP, dQ, dK, dV products; SURVEY App. H); two kernels (dQ, then dK/dV)
    kind = "attn_self_bwd" if a.n_mod == 1 and a.mods[0].E == 1 else "attn_cross_bwd"
    _timed(kind, 2.5 * attn_flops(a), lambda: check(_lib.lib().mmsum_attn_bwd(C.byref(a), _stream()), "mmsum_attn_bwd", 2))


def debug_poison():
    """Test aid: fill every SM's shared and tensor memory with NaN patterns (see include/mmsum_b200.h)."""
    check(_lib.lib().mmsum_debug_poison(_stream()), "mmsum_debug_poison")


def attn_decode_cross(a):
    """One query row per hypothesis against the un-expanded per-business memory (see include/mmsum_b200.h)."""
    check(_lib.lib().mmsum_attn_decode_cross(C.byref(a), _stream()), "mmsum_attn_decode_cross")


def attn_decode_self(qkv, cache, hist, pos_dev, out, H, scale):
    n = qkv.shape[0]
    check(_lib.lib().mmsum_attn_decode_self(_ptr(qkv), C.c_int64(qkv.stride(0)), _ptr(cache), _ptr(hist), _ptr(pos_dev), _ptr(out),
                                            C.c_int64(out.stride(0)), n, H, C.c_float(scale), _stream()), "mmsum_attn_decode_self")


def embed_ln_decode(ids, E, P, rating_diff, remb, gamma, beta, out, mean, rstd, rows, pos_dev):
    check(_lib.lib().mmsum_embed_ln_decode(_ptr(ids), _ptr(E), _ptr(P), _ptr(rating_diff), _ptr(remb), _ptr(gamma), _ptr(beta),
                                           _ptr(out), _ptr(mean), _ptr(rstd), rows, E.shape[1], _ptr(pos_dev), _stream()),
          "mmsum_embed_ln_decode")


def beam_topk(logits, V, beam_scores, ids, cur_dev, min_length, ngram, bos, eos, K, out_val, out_tok):
    """Per-row candidate selection of one beam-search token (see include/mmsum_b200.h)."""
    check(_lib.lib().mmsum_beam_topk(_ptr(logits), C.c_int64(logits.stride(0)), logits.shape[0], V, _ptr(beam_scores), _ptr(ids),
                                     ids.shape[1], _ptr(cur_dev), min_length, ngram, bos, eos, K, _ptr(out_val), _ptr(out_tok),
                                     _stream()), "mmsum_beam_topk")


def beam_update(cand_val, cand_tok, ids, beam_scores, done, pool_score, pool_tok, pool_len, pool_n, cur_dev, beam_idx, next_tok,
                next_tok32, hist, B, k, eos, pad, early_stopping, length_penalty):
    """Per-business beam update of one token (see include/mmsum_b200.h); every argument is device state updated in place."""
    check(_lib.lib().mmsum_beam_update(_ptr(cand_val), _ptr(cand_tok), _ptr(ids), _ptr(beam_scores), _ptr(done), _ptr(pool_score),
                                       _ptr(pool_tok), _ptr(pool_len), _ptr(pool_n), _ptr(cur_dev), _ptr(beam_idx), _ptr(next_tok),
                                       _ptr(next_tok32), _ptr(hist), B, k, cand_val.shape[1], ids.shape[1], eos, pad,
                                       int(bool(early_stopping)), C.c_float(length_penalty), _stream()), "mmsum_beam_update")


def prep_step(reviews, reviews_mask, rating, table_valid, img_mask, **kw):
    a = _lib.PrepArgs()
    for k, v in kw.items():
        setattr(a, k, v.data_ptr() if isinstance(v, torch.Tensor) else v)
    check(_lib.lib().mmsum_prep_step(_ptr(reviews), _ptr(reviews_mask), _ptr(rating), _ptr(table_valid), _ptr(img_mask),
                                     C.byref(a), _stream()), "mmsum_prep_step")


def table_fwd(dataset, B, E, field, values, W0, W1, X, valid):
    a = _lib.TableArgs()
    a.dataset, a.B = (0 if dataset == "yelp" else 1), B
    a.E, a.field = E.data_ptr(), field.data_ptr()
    for i, v in enumerate(values):
        setattr(a, "v%d" % i, v.data_ptr())
    a.W0, a.W1, a.X, a.valid = W0.data_ptr(), W1.data_ptr(), X.data_ptr(), valid.data_ptr()
    check(_lib.lib().mmsum_table_fwd(C.byref(a), _stream()), "mmsum_table_fwd")


def table_bits_bwd(dX, bits, dW, B, F, f0, nrows, nb):
    check(_lib.lib().mmsum_table_bits_bwd(_ptr(dX), _ptr(bits), _ptr(dW), B, F, f0, nrows, nb, _stream()), "mmsum_table_bits_bwd")
