"""TEST INFRASTRUCTURE — CPU restatement (plain torch fp32/fp64, functional) of the reference algorithm for
the MultimodalSum training step.  It is the checker for the CUDA path; only tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / --impl reference legs may import it.  The product path never does.

Pinned against the reference itself: tests/golden/*.npz were produced by running the UNMODIFIED reference
(through oracle/ref_harness.py) on synthetic weights/inputs from multimodalsum_b200.synth;
tests/test_oracle_golden.py checks this file against those vectors, tests/test_oracle_vs_reference.py against the
live reference when a checkout of it is present (see oracle/ref_harness.py).  (The reference's own test-suite holds no
vectors for this path — SURVEY.md §4.)

All file:line citations are relative to the reference's src/.  Every function takes the flat reference state_dict
(`p`, keys of SURVEY App. B) so that no nn.Module of the reference is needed.  The algorithm is the AS-WRITTEN one:
9 sequential leave-one-out decoder passes, K/V re-projected in every pass, logits materialised.
"""
import math

import torch
import torch.nn.functional as F

NEG_CROSS = -2.0 ** 16  # finite mask value of the cross-attention (transformer/modeling_multimodalsum.py:844)


def _lin(x, p, name, bias=True):
    return F.linear(x, p[name + ".weight"], p[name + ".bias"] if bias else None)


def _ln(x, p, name):
    # LayerNorm factory, eps 1e-5 (transformer/modeling_multimodalsum.py:972-980)
    return F.layer_norm(x, (x.shape[-1],), p[name + ".weight"], p[name + ".bias"], 1e-5)


def _drop(x, pdrop, training):
    return F.dropout(x, p=pdrop, training=training) if pdrop > 0 else x


def _split_heads(x, H):
    # [B, T, D] -> [B, H, T, hd]   (SelfAttention._shape, modeling_multimodalsum.py:706-709)
    B, T, D = x.shape
    return x.view(B, T, H, D // H).transpose(1, 2)


def self_attention(x, p, pre, H, key_pad, causal):
    """Unimodal self-attention, modeling_multimodalsum.py:746-749 + get_head_output :783-853.
    x [B,T,D]; key_pad bool [B,T] True = pad (or None); additive causal triu(-inf) for the decoder."""
    B, T, D = x.shape
    hd = D // H
    q = _split_heads(_lin(x, p, pre + "q_proj") * hd ** -0.5, H)
    k = _split_heads(_lin(x, p, pre + "k_proj"), H)
    v = _split_heads(_lin(x, p, pre + "v_proj"), H)
    w = q @ k.transpose(-1, -2)  # [B,H,T,T]
    if causal:
        w = w + torch.triu(torch.full((T, T), float("-inf"), dtype=x.dtype, device=x.device), 1)
    if key_pad is not None:
        w = w.masked_fill(key_pad[:, None, None, :], float("-inf"))
    a = torch.softmax(w, dim=-1) @ v
    a = a.transpose(1, 2).reshape(B, T, D)
    return _lin(a, p, pre + "out_proj")  # aggregate_head_output :877-886


def cross_attention_modality(x, mem, mem_valid, p, pre, H):
    """One modality of the multi-entity cross-attention (get_head_output cross path :768-869 +
    aggregate_head_output :877-886).  x [B,T,D]; mem [B,E,S,D]; mem_valid bool [B,E,S] True = attend.
    Independent softmax per entity, pad keys filled with -2^16, mean over entities that have any valid key,
    all-null business -> 0, then the shared out_proj."""
    B, T, D = x.shape
    E, S = mem.shape[1], mem.shape[2]
    hd = D // H
    q = _split_heads(_lin(x, p, pre + "q_proj") * hd ** -0.5, H)             # [B,H,T,hd]
    k = _lin(mem, p, pre + "k_proj").view(B, E, S, H, hd).permute(0, 1, 3, 2, 4)  # [B,E,H,S,hd]
    v = _lin(mem, p, pre + "v_proj").view(B, E, S, H, hd).permute(0, 1, 3, 2, 4)
    w = q[:, None] @ k.transpose(-1, -2)                                      # [B,E,H,T,S]
    pad = ~mem_valid
    w = w.masked_fill(pad[:, :, None, None, :], NEG_CROSS)
    o = torch.softmax(w, dim=-1) @ v                                          # [B,E,H,T,hd]
    null_ent = pad.all(dim=-1)                                                # [B,E] (:856)
    o = o.masked_fill(null_ent[:, :, None, None, None], 0.0)
    n = (~null_ent).sum(dim=1).clamp(min=1).to(x.dtype)                       # (:859-865)
    a = o.sum(dim=1) / n[:, None, None, None]
    a = a.transpose(1, 2).reshape(B, T, D)
    return _lin(a, p, pre + "out_proj")


def multimodal_cross_attention(x, mems, valids, p, pre, H):
    """SelfAttention.forward multimodal branch, modeling_multimodalsum.py:722-745."""
    text = cross_attention_modality(x, mems[0], valids[0], p, pre, H)
    table = cross_attention_modality(x, mems[1], valids[1], p, pre, H)
    img = cross_attention_modality(x, mems[2], valids[2], p, pre, H)
    no_table = (~valids[1]).all(dim=2)[:, 0]          # entity 0 only (:732)
    no_img = (~valids[2]).all(dim=2).all(dim=1)       # (:735)
    alpha = torch.relu(torch.tanh(_lin(torch.cat([text, table], -1), p, pre + "alpha_proj")))
    beta = torch.relu(torch.tanh(_lin(torch.cat([text, img], -1), p, pre + "beta_proj")))
    alpha = alpha.masked_fill(no_table[:, None, None], 0.0)
    beta = beta.masked_fill(no_img[:, None, None], 0.0)
    return text + alpha * table + beta * img


def embed(ids, p, pre, rating_diff=None):
    """tokens + learned positions (offset 2) [+ rating_diff * rating_embeddings] -> layernorm_embedding
    (BartEncoder.forward :368-371, BartDecoder.forward :588-596, LearnedPositionalEmbedding :961-969)."""
    T = ids.shape[1]
    # nn.Embedding(padding_idx=1) (:1001): gather-path gradient to the pad row is dropped; positions are frame
    # positions + 2 and never hit the pad row.
    x = F.embedding(ids, p[pre + "embed_tokens.weight"], padding_idx=1) + \
        p[pre + "embed_positions.weight"][torch.arange(T, device=ids.device) + 2]
    if rating_diff is not None:
        x = x + (rating_diff * p[pre + "rating_embeddings"]).unsqueeze(1)
    return _ln(x, p, pre + "layernorm_embedding")


def encoder(p, cfg, ids, valid, training=False):
    """BartEncoder.forward :346-404 with EncoderLayer :276-309 (post-LN).  ids [N,S], valid [N,S] 1 = token."""
    pre = "bart_model.model.encoder."
    pd = cfg.dropout
    key_pad = valid.eq(0)
    x = _drop(embed(ids, p, pre), pd, training)
    for i in range(cfg.encoder_layers):
        lp = pre + "layers.%d." % i
        x = _ln(x + _drop(self_attention(x, p, lp + "self_attn.", cfg.heads, key_pad, False), pd, training), p, lp + "self_attn_layer_norm")
        h = _lin(F.gelu(_lin(x, p, lp + "fc1")), p, lp + "fc2")
        x = _ln(x + _drop(h, pd, training), p, lp + "final_layer_norm")
    return x


def shift_tokens_right(labels, pad, bos, eos):
    """modeling_multimodalsum.py:225-246: position of the last non-pad token (EOS) becomes pad, shift right,
    start with BOS (or EOS when the batch already starts with BOS — decided from labels[0,0] as the reference does)."""
    idx_eos = labels.ne(pad).sum(dim=1) - 1
    body = labels.clone()
    body[torch.arange(labels.shape[0], device=labels.device), idx_eos] = pad
    out = torch.empty_like(labels)
    out[:, 0] = bos if labels[0, 0].item() != bos else eos
    out[:, 1:] = body[:, :-1]
    return out


def decoder(p, cfg, dec_ids, mems, valids, rating_diff, training=False, use_pad_mask=True):
    """BartDecoder.forward :530-660 with DecoderLayer :432-494; mems/valids lists [text, table, img] or a single
    text memory (text-only model).  Returns hidden states [B,T,D]."""
    pre = "bart_model.model.decoder."
    pd = cfg.dropout
    pad_mask = dec_ids.eq(cfg.pad_token_id)
    key_pad = pad_mask if (use_pad_mask and bool(pad_mask.any())) else None   # make_padding_mask :249-254; generation passes no mask (:2253)
    x = _drop(embed(dec_ids, p, pre, rating_diff), pd, training)
    for i in range(cfg.decoder_layers):
        lp = pre + "layers.%d." % i
        x = _ln(x + _drop(self_attention(x, p, lp + "self_attn.", cfg.heads, key_pad, True), pd, training), p, lp + "self_attn_layer_norm")
        if isinstance(mems, (list, tuple)):
            c = multimodal_cross_attention(x, mems, valids, p, lp + "encoder_attn.", cfg.heads)
        else:
            c = cross_attention_modality(x, mems, valids, p, lp + "encoder_attn.", cfg.heads)
        x = _ln(x + _drop(c, pd, training), p, lp + "encoder_attn_layer_norm")
        h = _lin(F.gelu(_lin(x, p, lp + "fc1")), p, lp + "fc2")
        x = _ln(x + _drop(h, pd, training), p, lp + "final_layer_norm")
    return x


def lm_logits(x, p):
    """F.linear(x, shared.weight, final_logits_bias) — modeling_multimodalsum.py:2281."""
    return F.linear(x, p["bart_model.model.shared.weight"], p["bart_model.final_logits_bias"])


def label_smoothing_loss(logits, target, eps):
    """utils.py:32-38 (LabelSmoothingLoss); eps None -> nn.CrossEntropyLoss() (text_pretrain.py:97).  Pad positions
    are NOT ignored."""
    logp = torch.log_softmax(logits, dim=-1)
    if eps is None:
        return -logp.gather(1, target.unsqueeze(1)).mean()
    V = logits.shape[-1]
    dist = torch.full_like(logp, eps / (V - 1))
    dist.scatter_(1, target.unsqueeze(1), 1.0 - eps)
    return (-dist * logp).sum(dim=-1).mean()


def _masked_sum_embed(E, ids):
    return (E[ids] * ids.ne(1).unsqueeze(-1).to(E.dtype)).sum(dim=-2)


def yelp_table_encoder(p, field, field_value):
    """table_encoder.py:14-83 (YelpTableEncoder.forward).  Gathers run under no_grad on the shared embedding."""
    pre = "table_encoder."
    name, category, str_cat, str_bool, rating, hours = field_value
    with torch.no_grad():
        E = p[pre + "bart_embedding.weight"]
        field_name = _masked_sum_embed(E, field)                                  # [47,D]
        name_e = _masked_sum_embed(E, name).unsqueeze(1)                          # [B,1,D]
        cat_tok = _masked_sum_embed(E, category)                                  # [B,6,D]
        cat_valid = category.ne(1).any(dim=-1, keepdim=True).to(E.dtype)          # [B,6,1]
        cat_e = (cat_tok * cat_valid).sum(dim=1, keepdim=True) / (cat_valid.sum(dim=1, keepdim=True) + 1e-6)
        sc_e = _masked_sum_embed(E, str_cat)                                      # [B,5,D]
        sb_e = E[str_bool.squeeze(-1)] * str_bool.ne(1).to(E.dtype)               # [B,32,D]
    dt = p[pre + "fc.weight"].dtype
    rating_e = F.linear(rating.to(dt), p[pre + "rating_embedding.weight"]).unsqueeze(1)
    hours_e = F.linear(hours.to(dt), p[pre + "hours_embedding.weight"])
    B = name.shape[0]
    values = torch.cat([name_e, cat_e, sc_e, sb_e, rating_e, hours_e], dim=1)     # [B,47,D]
    x = torch.cat([field_name.unsqueeze(0).expand(B, -1, -1), values], dim=-1)
    x = F.linear(torch.relu(_lin(x, p, pre + "fc")), p[pre + "linear.weight"])
    ones = torch.ones(B, 1, dtype=torch.bool, device=name.device)
    valid = torch.cat([ones, category[:, :1, 0].ne(1), str_cat[:, :, 0].ne(1), str_bool[:, :, 0].ne(1), ones,
                       hours.sum(dim=-1) != 0], dim=1)                            # [B,47] (:75-82)
    return x, valid


def amazon_table_encoder(p, field, field_value):
    """table_encoder.py:95-167 (AmazonTableEncoder.forward)."""
    pre = "table_encoder."
    price, rating, brand, name, category, desc = field_value
    with torch.no_grad():
        E = p[pre + "bart_embedding.weight"]
        fn = E[field].squeeze(1)
        field_name = torch.cat([fn[:-1], fn[-1:].expand(128, -1)])                # [133,D]
        brand_e = _masked_sum_embed(E, brand).unsqueeze(1)
        name_e = _masked_sum_embed(E, name).unsqueeze(1)
        cat_tok = _masked_sum_embed(E, category)                                  # [B,3,8,D]
        v2 = category.ne(1).any(dim=-1)                                           # [B,3,8]
        v2f = v2.unsqueeze(-1).to(E.dtype)
        cat_mid = (cat_tok * v2f).sum(dim=2) / (v2f.sum(dim=2) + 1e-6)            # [B,3,D]
        v1f = v2.any(dim=-1).unsqueeze(-1).to(E.dtype)                            # [B,3,1]
        cat_e = (cat_mid * v1f).sum(dim=1, keepdim=True) / (v1f.sum(dim=1, keepdim=True) + 1e-6)
        desc_e = E[desc]
    dt = p[pre + "fc.weight"].dtype
    price_e = F.linear(price.to(dt), p[pre + "price_embedding.weight"]).unsqueeze(1)
    rating_e = F.linear(rating.to(dt), p[pre + "rating_embedding.weight"]).unsqueeze(1)
    B = price.shape[0]
    values = torch.cat([price_e, rating_e, brand_e, name_e, cat_e, desc_e], dim=1)
    x = torch.cat([field_name.unsqueeze(0).expand(B, -1, -1), values], dim=-1)
    x = F.linear(torch.relu(_lin(x, p, pre + "fc")), p[pre + "linear.weight"])
    ones = torch.ones(B, 1, dtype=torch.bool, device=price.device)
    valid = torch.cat([price.sum(dim=1, keepdim=True) != 0, ones, brand[:, :1].ne(1), name[:, :1].ne(1), ones,
                       desc.ne(1)], dim=1)
    return x, valid


def multimodal_memories(p, cfg, batch, training=False):
    """MultimodalSum.get_multimodal_outputs, multimodal_train.py:165-193 (pooled image features in)."""
    B, R, S = batch.reviews.shape
    text = encoder(p, cfg, batch.reviews.view(B * R, S), batch.reviews_mask.view(B * R, S), training).view(B, R, S, -1)
    text_valid = batch.reviews_mask.bool()
    if cfg.dataset == "text":
        return text, text_valid, None, None, None, None
    tenc = yelp_table_encoder if cfg.table == "yelp" else amazon_table_encoder
    table, table_valid = tenc(p, batch.field, batch.field_value)
    img = F.linear(batch.img.to(text.dtype), p["img_encoder.linear.weight"])      # img_encoder.py:39-40
    img_valid = batch.img_mask.unsqueeze(-1).expand(-1, -1, img.shape[2])
    return text, text_valid, table.unsqueeze(1), table_valid.unsqueeze(1), img, img_valid


def step_loss_passes(p, cfg, batch, label_smoothing=0.1, training=False, return_logits=False):
    """MultimodalSum.forward, multimodal_train.py:124-163 (and TextSupervised.forward, text_pretrain.py:71-113 for
    cfg.dataset == 'text'): generator over the R leave-one-out passes, yielding (loss_i, logits_i or None)."""
    text, text_valid, table, table_valid, img, img_valid = multimodal_memories(p, cfg, batch, training)
    B, R, S = batch.reviews.shape
    rating = batch.reviews_rating.to(text.dtype)
    for i in range(R):
        others = [j for j in range(R) if j != i]
        rating_diff = (rating[:, i] - rating[:, others].mean(dim=1)).unsqueeze(1)
        labels = batch.reviews[:, i, :]
        dec_ids = shift_tokens_right(labels, cfg.pad_token_id, cfg.bos_token_id, cfg.eos_token_id)
        if cfg.dataset == "text":
            mems, valids = text[:, others], text_valid[:, others]
        else:
            mems = [text[:, others], table, img]
            valids = [text_valid[:, others], table_valid, img_valid]
        x = decoder(p, cfg, dec_ids, mems, valids, rating_diff, training)
        logits = lm_logits(x, p)
        yield label_smoothing_loss(logits.view(-1, logits.shape[-1]), labels.reshape(-1), label_smoothing), \
            (logits if return_logits else None)


def step_loss(p, cfg, batch, label_smoothing=0.1, training=False, return_logits=False):
    """Mean of the R pass losses (multimodal_train.py:162)."""
    losses, all_logits = [], []
    for li, lg in step_loss_passes(p, cfg, batch, label_smoothing, training, return_logits):
        losses.append(li)
        all_logits.append(lg)
    loss = torch.stack(losses).mean()
    return (loss, all_logits) if return_logits else loss


def stage_step_loss(p, cfg, batch, label_smoothing=0.1, training=False):
    """ImgSupervised.forward (img_pretrain.py:91-141) / TableSupervised.forward (table_pretrain.py:90-129): the memory is
    the projected image features [B, max_imgs, 196, D] (mask repeated over the 196 keys) or the table encoder's output
    [B, 1, F, D]; rating_diff = 0; decoder inputs = shift_tokens_right(labels); one loss over all B*128 rows."""
    if cfg.image:
        mem = F.linear(batch.img.to(p["img_encoder.linear.weight"].dtype), p["img_encoder.linear.weight"])
        valid = batch.img_mask.unsqueeze(-1).expand(-1, -1, mem.shape[2])
    else:
        tenc = yelp_table_encoder if cfg.table == "yelp" else amazon_table_encoder
        mem, valid = tenc(p, batch.field, batch.field_value)
        mem, valid = mem.unsqueeze(1), valid.unsqueeze(1)
    labels = batch.labels
    rd = torch.zeros(labels.shape[0], 1, dtype=mem.dtype, device=mem.device)
    dec_ids = shift_tokens_right(labels, cfg.pad_token_id, cfg.bos_token_id, cfg.eos_token_id)
    x = decoder(p, cfg, dec_ids, mem, valid, rd, training)
    logits = lm_logits(x, p)
    return label_smoothing_loss(logits.view(-1, logits.shape[-1]), labels.reshape(-1), label_smoothing)


def step_loss_and_grads(sd, cfg, batch, label_smoothing=0.1, dtype=torch.float32, device="cpu", training=False, low_memory=False):
    """Forward + backward of the oracle; returns (loss, {name: grad}) keyed like the reference's named_parameters().
    `low_memory`: back-propagate each leave-one-out pass as soon as its loss exists (same sum of gradients, one pass of
    activations alive at a time) — for the full-size GPU comparisons at 16 businesses."""
    p = {}
    leaf = {}
    for k, v in sd.items():
        if any(k.endswith(a) for a in ("encoder.embed_tokens.weight", "decoder.embed_tokens.weight",
                                       "table_encoder.bart_embedding.weight")):
            continue
        t = v.to(device=device, dtype=dtype).clone()
        if not k.endswith("final_logits_bias"):
            t.requires_grad_(True)
            leaf[k] = t
        p[k] = t
    shared = p["bart_model.model.shared.weight"]
    p["bart_model.model.encoder.embed_tokens.weight"] = shared
    p["bart_model.model.decoder.embed_tokens.weight"] = shared
    if cfg.table is not None:
        p["table_encoder.bart_embedding.weight"] = shared
    b = batch.to(device)
    if low_memory and cfg.text_memory:
        R = b.reviews.shape[1]
        loss = torch.zeros((), dtype=dtype, device=device)
        for li, _ in step_loss_passes(p, cfg, b, label_smoothing, training):
            (li / R).backward(retain_graph=True)
            loss = loss + li.detach() / R
            del li
    else:
        loss = (step_loss if cfg.text_memory else stage_step_loss)(p, cfg, b, label_smoothing, training)
        loss.backward()
    grads = {k: t.grad for k, t in leaf.items() if t.grad is not None}
    return loss.detach(), grads, p


def generation_logits_fn(p, cfg, batch, num_beams):
    """Next-token logits for beam search as the reference computes them in `generate` (modeling_multimodalsum.py:2857-2866):
    memories from get_multimodal_outputs, rating_diff = 0 (src/test.py:155), every beam of a business attends to the same
    memory, no decoder padding mask.  The reference's incremental cache (:889-920) is a pure optimisation: the logits of the
    last position over the full prefix are identical, which is what this closure evaluates."""
    with torch.no_grad():
        text, text_valid, table, table_valid, img, img_valid = multimodal_memories(p, cfg, batch, training=False)
        rep = lambda t: t.repeat_interleave(num_beams, dim=0)
        mems = [rep(text), rep(table), rep(img)]
        valids = [rep(text_valid), rep(table_valid), rep(img_valid)]
        rd = torch.zeros(mems[0].shape[0], 1, dtype=text.dtype, device=text.device)

    def fn(input_ids):
        with torch.no_grad():
            x = decoder(p, cfg, input_ids, mems, valids, rd, training=False, use_pad_mask=False)
            return lm_logits(x[:, -1], p).float()
    return fn
