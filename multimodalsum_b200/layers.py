"""Forward of the BART sub-layers on the kernels, written once for every caller: the training step
(engine.StepEngine.forward), the inference surface (inference.encoder_forward / decoder_hidden / table_forward) and the
cached decode step (generation.Generator._decode_launches).  Only training has a backward; it stays in engine.py.

Callers pass data, not modes:
  lp       parameter prefix of the layer ("bart_model.model.{encoder,decoder}.layers.<l>.")
  buf      the layer's activation buffers by name ("qkv", "ctx", "o", "x1", "qc", "A3", "O3", "U", "AB", "yc", "x2", "a", "f")
  attend   callable(q, out): the attention of the block over the q buffer
  stats    (mean, rstd) written by the block's add + LayerNorm
  drop     (p, seed, sid, step_dev) of the dropout in front of that LayerNorm; NO_DROP at inference
"""
import torch

from . import ops

BM = "bart_model.model."
NO_DROP = (0.0, 0, 0, None)


def table_dims(dataset):
    """Fields of the table memory: Yelp 47, Amazon 133 (src/table_encoder.py); 0 for a model without a table."""
    return {None: 0, "yelp": 47, "amazon": 133}[dataset]


def _add_ln(eng, name, res, y, out, stats, drop):
    ops.add_ln_fwd(res, y, eng.w32(name + ".weight"), eng.w32(name + ".bias"), out, *stats, *drop)


# ---------------------------------------------------------------------------------------------- front ends
def embed_params(eng, side, rating_diff):
    """(E, P, rating_diff, rating table, LN gamma, LN beta): the parameters of the "encoder" / "decoder" embedding kernels
    (ops.embed_ln_fwd, ops.embed_ln_decode); the rating embedding joins when rating_diff is given (decoder)."""
    pre = BM + side + "."
    remb = None if rating_diff is None else eng.w32(pre + "rating_embeddings")
    return (eng.w32(BM + "shared.weight"), eng.w32(pre + "embed_positions.weight"), rating_diff, remb,
            eng.w32(pre + "layernorm_embedding.weight"), eng.w32(pre + "layernorm_embedding.bias"))


def table_embed(eng, field, values, tabX, valid):
    """The table kernel: field / value codes -> tabX bf16 [B*F, 2D] and field validity u8 [B, F]."""
    t = "table_encoder."
    rating = eng.w32(t + "rating_embedding.weight")
    if eng.cfg.table == "yelp":
        W0, W1 = rating, eng.w32(t + "hours_embedding.weight")
    else:
        W0, W1 = eng.w32(t + "price_embedding.weight"), rating
    ops.table_fwd(eng.cfg.table, valid.shape[0], eng.w32(BM + "shared.weight"), field, values, W0, W1, tabX, valid)


def table_project(eng, tabX, tab_h, out):
    """fc + ReLU into tab_h, then the linear projection into the memory rows `out`."""
    t = "table_encoder."
    ops.gemm(tabX, eng.w16(t + "fc.weight"), tab_h, bias=eng.w32(t + "fc.bias"), act=ops.ACT_RELU)
    ops.gemm(tab_h, eng.w16(t + "linear.weight"), out)


def project_kv(eng, MEM, l, out):
    """Cross-attention K|V of the memory for decoder layer l: one GEMM (k_proj | v_proj are adjacent in the arena)."""
    c = BM + "decoder.layers.%d.encoder_attn." % l
    return ops.gemm(MEM, eng.w16(c + "k_proj.weight", c + "v_proj.weight"), out,
                    bias=eng.w32(c + "k_proj.bias", c + "v_proj.bias"))


# ---------------------------------------------------------------------------------------------- attention arguments
def self_attn_args(eng, qkv, out, lse, key_valid, n_qseq, causal, Sk, R=1, q_rows=0, ent_stride=0, **bwd):
    """Self-attention over a fused q|k|v buffer [rows, 3D]: n_qseq query sequences (R query tiles share a key frame of
    Sk keys, ent_stride rows apart; 0 = Sk), q_rows rows per sequence (0 = 128).  `bwd`: the backward's extra fields."""
    D = eng.cfg.d_model
    return ops.attn_args(Q=qkv, ldq=3 * D, q_col=0, KV=qkv, ldkv=3 * D, k_col=D, v_col=2 * D, O=out, ldo=D, LSE=lse,
                         key_valid=key_valid, ent_valid=None, inv_n=None, n_qseq=n_qseq, H=eng.cfg.heads, R=R,
                         causal=int(causal), E_total=1, scale=eng.cfg.head_dim ** -0.5, q_rows=q_rows,
                         mods=[(0, 0, 1, Sk, 0, 0, ent_stride)], **bwd)


def cross_attn_args(eng, qc, kv, out3, lse, mods, mem_valid, ent_valid, inv_n, n_qseq, R, loo=False, **bwd):
    """Cross-attention of qc [rows, D] over the K|V [Tm, 2D] of a memory given as (row_base, E, Sk) per modality, one
    output per modality in out3 [n_mod, rows, D].  loo: the first modality is left-one-out (training's text memory: target
    i does not see review i).  `bwd`: the backward's extra fields."""
    D = eng.cfg.d_model
    table, eb = [], 0
    for i, (base, E, Sk) in enumerate(mods):
        table.append((base, i * out3[0].numel(), E, Sk, int(loo and i == 0), eb, 0))
        eb += E
    return ops.attn_args(Q=qc, ldq=D, q_col=0, KV=kv, ldkv=2 * D, k_col=0, v_col=D, O=out3, ldo=D, LSE=lse,
                         key_valid=mem_valid, ent_valid=ent_valid, inv_n=inv_n, n_qseq=n_qseq, H=eng.cfg.heads, R=R,
                         causal=0, E_total=eb, scale=eng.cfg.head_dim ** -0.5, mods=table, **bwd)


# ---------------------------------------------------------------------------------------------- blocks
def self_block(eng, lp, x, buf, attend, stats, drop):
    """buf["x1"] = LN(x + drop(out_proj(attend(qkv(x)))))."""
    s = lp + "self_attn."
    ops.gemm(x, eng.w16(s + "q_proj.weight", s + "v_proj.weight"), buf["qkv"], bias=eng.w32(s + "q_proj.bias", s + "v_proj.bias"))
    attend(buf["qkv"], buf["ctx"])
    ops.gemm(buf["ctx"], eng.w16(s + "out_proj.weight"), buf["o"], bias=eng.w32(s + "out_proj.bias"))
    _add_ln(eng, lp + "self_attn_layer_norm", x, buf["o"], buf["x1"], stats, drop)


def _gate_proj(eng, c, O3, U, i):
    """U[i] = [O3[0] | O3[1 + i]]·Wᵀ + b: alpha (i = 0, text | table) or beta (i = 1, text | image)."""
    n = c + ("alpha_proj", "beta_proj")[i]
    ops.gemm_cat(O3[0], O3[1 + i], eng.w16(n + ".weight"), U[i], bias=eng.w32(n + ".bias"))


def cross_block(eng, lp, x1, buf, attend, stats, drop, pres, rows_per_biz, fork=None):
    """buf["x2"] = LN(x1 + drop(y)): y = out_proj of the attention over each memory modality, fused by the alpha / beta
    gates when there are three (SelfAttention.forward, multimodal branch :722-745).  fork: (side stream, fork event, join
    event) to run the two gate GEMMs side by side; None runs them one after the other on the current stream."""
    c = lp + "encoder_attn."
    ops.gemm(x1, eng.w16(c + "q_proj.weight"), buf["qc"], bias=eng.w32(c + "q_proj.bias"))
    A3, O3 = buf["A3"], buf["O3"]
    attend(buf["qc"], A3)
    nm, rows, D = A3.shape
    ops.gemm(A3.view(nm * rows, D), eng.w16(c + "out_proj.weight"), O3.view(nm * rows, D), bias=eng.w32(c + "out_proj.bias"))
    y = O3[0]
    if nm == 3:
        U = buf["U"]
        if fork is None:
            _gate_proj(eng, c, O3, U, 0)
            _gate_proj(eng, c, O3, U, 1)
        else:
            side, ev_fork, ev_join = fork
            main = torch.cuda.current_stream()
            ev_fork.record(main)
            side.wait_event(ev_fork)
            with torch.cuda.stream(side):
                _gate_proj(eng, c, O3, U, 1)
                ev_join.record(side)
            _gate_proj(eng, c, O3, U, 0)
            main.wait_event(ev_join)
        y = buf["yc"]
        ops.gate_fwd(O3, U, pres, y, buf["AB"], rows, rows_per_biz, D)
    _add_ln(eng, lp + "encoder_attn_layer_norm", x1, y, buf["x2"], stats, drop)


def ffn_block(eng, lp, xin, buf, out, stats, drop, dact=None):
    """out = LN(xin + drop(fc2(gelu(fc1(xin))))).  dact: where fc1 also stores GELU'(pre-activation) for the backward."""
    ops.gemm(xin, eng.w16(lp + "fc1.weight"), buf["a"], bias=eng.w32(lp + "fc1.bias"), act=ops.ACT_GELU, aux=dact,
             aux_mode=ops.AUX_NONE if dact is None else ops.AUX_STORE_DACT)
    ops.gemm(buf["a"], eng.w16(lp + "fc2.weight"), buf["f"], bias=eng.w32(lp + "fc2.bias"))
    _add_ln(eng, lp + "final_layer_norm", xin, buf["f"], out, stats, drop)
