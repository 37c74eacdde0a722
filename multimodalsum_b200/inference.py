"""Inference-side forwards of the reference's sub-modules on the step engine's kernels (no autograd graph).

These are the bodies behind the drop-in surface of SURVEY §8(b):
  encoder_forward          BartEncoder.forward                              modeling_multimodalsum.py:346-404
  table_forward            YelpTableEncoder / AmazonTableEncoder.forward    src/table_encoder.py:14-83, 95-167
  image_forward            Resnet.forward tail (flatten + linear)           src/img_encoder.py:39-40
  build_memory             what BartDecoder.forward does with its memory lists (mask inversion :572-575, null entities
                           :856-866, modality presence :732-736) — integer bookkeeping, torch on the device
  decoder_hidden, lm_head  BartDecoder.forward :530-660 + LM head :2281 over full 128-position frames
Training does NOT go through here: `MultimodalSum.forward` runs the fused step (engine.StepEngine); both run the layer
forwards of `layers.py`, on the same C-ABI kernels (bf16 activations, fp32 statistics).  Torch only allocates and does
the integer mask bookkeeping.  All functions expect CUDA tensors and raise otherwise (no CPU path).
"""
import math
from dataclasses import dataclass, field as dc_field

import torch

from . import layers as L
from . import ops

FRAME = 128          # query tile of the attention kernels
MAX_KEYS = 208       # keys per memory entity the attention kernels hold in tensor memory


def _bf(dev, *s):
    return torch.empty(s, device=dev, dtype=torch.bfloat16)


def _f32(dev, *s):
    return torch.empty(s, device=dev, dtype=torch.float32)


def _need_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: mmsum_b200 has no CPU path" % what)


# ---------------------------------------------------------------------------------------------- modality encoders
@torch.no_grad()
def table_forward(eng, field, field_value, out=None):
    """-> (emb bf16 [B, F, D], valid uint8 [B, F]).  `out`: optional [B*F, D] destination (a slice of a memory buffer)."""
    cfg = eng.cfg
    if cfg.table is None:
        raise RuntimeError("this model has no table encoder")
    _need_cuda(field, "field")
    dev = field.device
    D = cfg.d_model
    F = L.table_dims(cfg.table)
    vals = [v.to(torch.int64).contiguous() for v in field_value]
    B = vals[0].shape[0]
    tabX, valid, tab_h = _bf(dev, B * F, 2 * D), torch.zeros(B, F, device=dev, dtype=torch.uint8), _bf(dev, B * F, D)
    L.table_embed(eng, field.to(torch.int64).contiguous(), vals, tabX, valid)
    if out is None:
        out = _bf(dev, B * F, D)
    L.table_project(eng, tabX, tab_h, out)
    return out.view(B, F, D), valid


@torch.no_grad()
def image_forward(eng, feats, out=None):
    """Pooled ResNet-101 stage-3 features [B, n_img, keys, 1024] (fp32 or bf16) -> bf16 [B, n_img, keys, D]."""
    _need_cuda(feats, "img")
    dev = feats.device
    B, n_img, ik, C = feats.shape
    if C != 1024:
        raise ValueError("image features must have 1024 channels (ResNet-101 stage 3), got %d" % C)
    x = feats.reshape(B * n_img * ik, C)
    if x.dtype != torch.bfloat16:
        x = ops.cast_bf16(x.float().contiguous(), _bf(dev, B * n_img * ik, C))
    if out is None:
        out = _bf(dev, B * n_img * ik, eng.cfg.d_model)
    ops.gemm(x.contiguous(), eng.w16("img_encoder.linear.weight"), out)
    return out.view(B, n_img, ik, eng.cfg.d_model)


@torch.no_grad()
def encoder_forward(eng, input_ids, attention_mask=None):
    """BartEncoder.forward in eval mode.  input_ids [N, S] (S <= 208), attention_mask [N, S] 1 = token (None: ids != pad).
    Returns bf16 [N, S, D] (a view of the 128-row-tiled frame buffer)."""
    cfg = eng.cfg
    _need_cuda(input_ids, "input_ids")
    dev = input_ids.device
    D, H = cfg.d_model, cfg.heads
    N, S = input_ids.shape
    if S > MAX_KEYS:
        raise ValueError("encoder frames up to %d tokens are supported, got %d" % (MAX_KEYS, S))
    if attention_mask is None:
        attention_mask = input_ids.ne(cfg.pad_token_id)
    Sp = FRAME * math.ceil(S / FRAME)
    tiles = Sp // FRAME
    T = N * Sp
    ids = torch.full((N, Sp), cfg.pad_token_id, device=dev, dtype=torch.int32)
    ids[:, :S] = input_ids.to(torch.int32)
    valid = torch.zeros(N, Sp, device=dev, dtype=torch.uint8)
    valid[:, :S] = (attention_mask != 0).to(torch.uint8)
    kvalid = valid.reshape(-1)
    x, nxt = _bf(dev, T, D), _bf(dev, T, D)
    buf = dict(qkv=_bf(dev, T, 3 * D), ctx=_bf(dev, T, D), o=_bf(dev, T, D), x1=_bf(dev, T, D), a=_bf(dev, T, cfg.ffn_dim),
               f=_bf(dev, T, D))
    stats = (_f32(dev, T), _f32(dev, T))
    lse = _f32(dev, N * tiles, H, 1, FRAME)
    ops.embed_ln_fwd(ids.reshape(-1), *L.embed_params(eng, "encoder", None), x, *stats, T, Sp, *L.NO_DROP)
    # a frame of Sp rows = Sp/128 query tiles attending to one key entity of <= 208 rows
    attend = lambda qkv, ctx: ops.attn_fwd(L.self_attn_args(eng, qkv, ctx, lse, kvalid, N * tiles, False, min(Sp, MAX_KEYS),
                                                            R=tiles, ent_stride=Sp))
    for l in range(cfg.encoder_layers):
        lp = L.BM + "encoder.layers.%d." % l
        L.self_block(eng, lp, x, buf, attend, stats, L.NO_DROP)
        L.ffn_block(eng, lp, buf["x1"], buf, nxt, stats, L.NO_DROP)
        x, nxt = nxt, x
    return x.view(N, Sp, D)[:, :S]


# ---------------------------------------------------------------------------------------------- decoder memory
@dataclass
class Memory:
    """Cross-attention memory of B businesses, packed [text | table | image] along rows (bf16 [Tm, D]), plus the validity
    bookkeeping the attention / gate kernels read.  `kv[l]` = the K|V projection of layer l ([Tm, 2D]), made once and shared
    by every beam of a business (the reference expands and re-gathers it per hypothesis, :2598-2627, :3004-3010)."""
    MEM: torch.Tensor
    B: int
    mods: list                      # per modality (row_base, E, Sk) in MEM rows
    mem_valid: torch.Tensor         # u8 [Tm]
    ent_valid: torch.Tensor         # u8 [B, Et]
    inv_n: torch.Tensor             # f32 [B, n_mod]   1 / #valid entities (0 when none)
    pres: torch.Tensor              # u8 [B, 2] table / image present (None for a single-modality memory)
    Et: int
    kv: list = dc_field(default_factory=list)


def _ent_bookkeeping(valid_b_e_s):
    """valid [B, E, S] bool -> (entity validity u8 [B, E], 1/#valid f32 [B])."""
    ent = valid_b_e_s.any(dim=2)
    cnt = ent.sum(dim=1).float()
    inv = torch.where(cnt > 0, 1.0 / cnt.clamp(min=1), torch.zeros_like(cnt))
    return ent.to(torch.uint8), inv


@torch.no_grad()
def build_memory(eng, hiddens, masks):
    """hiddens: list of [B, E_m, S_m, D] tensors (1 entry: single-modality model; 3: text, table, image);
    masks: list of [B, E_m, S_m] (1/True = attend; None = all valid)."""
    cfg = eng.cfg
    if len(hiddens) not in (1, 3):
        raise ValueError("memory must hold 1 or 3 modalities")
    dev = hiddens[0].device
    _need_cuda(hiddens[0], "memory")
    D = cfg.d_model
    B = hiddens[0].shape[0]
    rows, mods, valids, ent_v, inv_n = [], [], [], [], []
    base = 0
    for h, m in zip(hiddens, masks):
        Bm, E, S, Dh = h.shape
        if Bm != B or Dh != D:
            raise ValueError("memory tensors must be [B, E, S, %d]" % D)
        if S > MAX_KEYS:
            raise ValueError("memory entities of up to %d keys are supported, got %d" % (MAX_KEYS, S))
        rows.append(h.reshape(B * E * S, D).to(torch.bfloat16))
        v = torch.ones(B, E, S, device=dev, dtype=torch.bool) if m is None else (m.reshape(B, E, S) != 0)
        valids.append(v.reshape(-1).to(torch.uint8))
        e, i = _ent_bookkeeping(v)
        ent_v.append(e)
        inv_n.append(i)
        mods.append((base, E, S))
        base += B * E * S
    MEM = torch.cat(rows, dim=0).contiguous()
    ent_valid = torch.cat(ent_v, dim=1).contiguous()
    pres = None
    if len(hiddens) == 3:
        # table present: entity 0 only (:732); image present: any entity (:735)
        pres = torch.stack([ent_v[1][:, 0], ent_v[2].max(dim=1).values], dim=1).contiguous()
    return Memory(MEM=MEM, B=B, mods=mods, mem_valid=torch.cat(valids).contiguous(), ent_valid=ent_valid,
                  inv_n=torch.stack(inv_n, dim=1).contiguous(), pres=pres, Et=ent_valid.shape[1])


@torch.no_grad()
def project_memory(eng, mem):
    """Cross-attention K|V of the whole memory, one GEMM per decoder layer."""
    if mem.kv:
        return mem
    for l in range(eng.cfg.decoder_layers):
        mem.kv.append(L.project_kv(eng, mem.MEM, l, _bf(mem.MEM.device, mem.MEM.shape[0], 2 * eng.cfg.d_model)))
    return mem


# ---------------------------------------------------------------------------------------------- decoder (full frames)
@torch.no_grad()
def decoder_hidden(eng, mem, dec_ids, rating_diff=None, per_biz=1, dec_valid=None):
    """BartDecoder.forward (eval) over 128-position causal frames.  dec_ids [N, T<=128] with N = mem.B * per_biz (the
    `per_biz` sequences of a business are adjacent and attend to the same memory); dec_valid [N, T] 1 = key position may
    be attended (None: all).  Returns bf16 [N, 128, D]; rows >= T are padding."""
    cfg = eng.cfg
    dev = dec_ids.device
    _need_cuda(dec_ids, "decoder_input_ids")
    D, H, FF = cfg.d_model, cfg.heads, cfg.ffn_dim
    N, cur = dec_ids.shape
    S = FRAME
    if cur > S:
        raise ValueError("decoder frames up to %d tokens" % S)
    if N != mem.B * per_biz:
        raise ValueError("decoder batch %d != businesses %d x %d" % (N, mem.B, per_biz))
    if per_biz > 32:
        raise ValueError("at most 32 sequences per business")
    project_memory(eng, mem)
    T = N * S
    nm = len(mem.mods)
    ids = torch.full((N, S), cfg.pad_token_id, device=dev, dtype=torch.int32)
    ids[:, :cur] = dec_ids.to(torch.int32)
    kvalid = None
    if dec_valid is not None:
        kv_ = torch.zeros(N, S, device=dev, dtype=torch.uint8)
        kv_[:, :cur] = (dec_valid != 0).to(torch.uint8)
        kvalid = kv_.reshape(-1)
    rd = torch.zeros(N, device=dev) if rating_diff is None else rating_diff.reshape(N).float().contiguous()
    x, nxt = _bf(dev, T, D), _bf(dev, T, D)
    buf = dict(qkv=_bf(dev, T, 3 * D), ctx=_bf(dev, T, D), o=_bf(dev, T, D), x1=_bf(dev, T, D), qc=_bf(dev, T, D),
               A3=_bf(dev, nm, T, D), O3=_bf(dev, nm, T, D), x2=_bf(dev, T, D), a=_bf(dev, T, FF), f=_bf(dev, T, D))
    if nm == 3:
        buf.update(U=_bf(dev, 2, T, D), AB=_bf(dev, 2, T, D), yc=_bf(dev, T, D))
    stats = (_f32(dev, T), _f32(dev, T))
    lse, lse_c = _f32(dev, N, H, 1, S), _f32(dev, N, H, mem.Et, S)
    inv_n = mem.inv_n.repeat_interleave(per_biz, dim=0).contiguous() if per_biz > 1 else mem.inv_n
    ops.embed_ln_fwd(ids.reshape(-1), *L.embed_params(eng, "decoder", rd), x, *stats, T, S, *L.NO_DROP)
    attend_self = lambda qkv, ctx: ops.attn_fwd(L.self_attn_args(eng, qkv, ctx, lse, kvalid, N, True, S))
    for l in range(cfg.decoder_layers):
        lp = L.BM + "decoder.layers.%d." % l
        attend_mem = lambda qc, A3: ops.attn_fwd(L.cross_attn_args(eng, qc, mem.kv[l], A3, lse_c, mem.mods, mem.mem_valid,
                                                                   mem.ent_valid, inv_n, N, per_biz))
        L.self_block(eng, lp, x, buf, attend_self, stats, L.NO_DROP)
        L.cross_block(eng, lp, buf["x1"], buf, attend_mem, stats, L.NO_DROP, mem.pres, per_biz * S)
        L.ffn_block(eng, lp, buf["x2"], buf, nxt, stats, L.NO_DROP)
        x, nxt = nxt, x
    return x.view(N, S, D)


@torch.no_grad()
def lm_head(eng, x_rows):
    """F.linear(x, shared.weight, final_logits_bias) (:2281): bf16 rows [M, D] (any row stride) -> fp32 logits [M, V]."""
    V = eng.cfg.vocab_size
    M = x_rows.shape[0]
    out = _f32(x_rows.device, M, (V + 3) // 4 * 4)[:, :V]      # 16-byte row pitch for the TMA store
    ops.gemm(x_rows, eng.w16("bart_model.model.shared.weight"), out, bias=eng.w32_flb())
    return out


def shift_tokens_right(labels, pad, bos, eos):
    """modeling_multimodalsum.py:225-246 on the device without the reference's host sync: the position of the last non-pad
    token becomes pad, shift right, start token = BOS unless the batch already starts with BOS (decided from labels[0, 0]
    for the whole batch, quirk Q3)."""
    idx_eos = labels.ne(pad).sum(dim=1, keepdim=True) - 1
    body = labels.scatter(1, idx_eos.clamp(min=0), pad)
    start = torch.where(labels[0, 0] == bos, torch.full_like(labels[0, 0], eos), torch.full_like(labels[0, 0], bos))
    return torch.cat([start.expand(labels.shape[0], 1), body[:, :-1]], dim=1)
