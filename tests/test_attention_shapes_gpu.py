"""Attention kernels at the shapes and dispatch modes the benchmarked workloads run, against one plain fp32 reference.

test_kernels_gpu.py checks the attention kernels on small, regular shapes.  The training step, the generation encoder and
beam-search decoding run them elsewhere: 9 reviews with leave-one-out, 10 images (20 entities, image keys tiled as one
packed range per business in dK/dV), Amazon's 133-key table (a 5-key second tile), 256-row encoder frames with 208 keys
per entity, head mode with all 16 heads per CTA, decode positions up to 127.  Every case of the training kernels states
which host dispatch paths it reaches (`attn_paths`, a restatement of the predicates in csrc/attention_sm100.cu), so that a later change of
shape cannot silently drop one.

Tolerances are the bf16-storage ones of test_kernels_gpu.py (forward 1.5e-2, backward 2e-2, relative to the max-abs of
the reference), applied separately to every modality output and every memory region (text / table / image rows of dK and
of dV), so that an error in a small block cannot hide under the scale of a large one.  What must be exact is checked
exactly: dK/dV rows of masked or null keys are 0, and sentinel-filled buffers keep the sentinel wherever the kernels must
not write (LSE / DELTA of entities that are not attended, rows behind the last frame)."""
import math
from types import SimpleNamespace

import pytest
import torch

pytestmark = pytest.mark.gpu

D, H, HD = 1024, 16, 64
SCALE = HD ** -0.5
LOG2E = 1.4426950408889634
GUARD = 128                      # sentinel rows behind every output buffer
FWD_TOL, BWD_TOL = 1.5e-2, 2e-2

# host-side constants of csrc/attention_sm100.cu / common.cuh
SQ, K_MAX_ENT, K_MAX_KEYS, N_SMS = 128, 24, 208, 148


@pytest.fixture(autouse=True)
def _fp32_reference_matmul():
    """The reference is fp32: TF32 products would put its own error (1e-3 relative) next to the kernels'."""
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _ops():
    from multimodalsum_b200 import ops
    return ops


def _dev():
    return torch.device("cuda")


# ------------------------------------------------------------------ which kernel paths a call takes
def _mod_packed(E, Sk, loo, stride):
    """mod_packed (csrc/attention_sm100.cu:842): the dK/dV kernel tiles the business' entities as one contiguous key range."""
    return E > 1 and not loo and stride in (0, Sk) and Sk >= SQ and Sk % SQ != 0


def attn_paths(mods, n_qseq, R, h=H):
    """The host dispatch of mmsum_attn_fwd / mmsum_attn_bwd for these arguments (mods: 7-tuples as in ops.attn_args)."""
    base, _o, E, Sk, loo, _eb, _st = mods[0]
    single = len(mods) == 1 and E == 1 and not loo
    head = single and h <= K_MAX_ENT and n_qseq >= 64                                      # :1261
    hpc = (h // 2 if h % 2 == 0 and n_qseq <= 2 * N_SMS else h) if head else 0             # :1262
    dq_head = single and Sk <= SQ and h <= K_MAX_ENT and n_qseq >= 64                       # :1301
    kv_heads = 4 if single and n_qseq // R >= 64 and h % 4 == 0 else 1                      # :1308
    packed = [_mod_packed(m[2], m[3], m[4], m[6]) for m in mods]
    return dict(fwd_hpc=hpc, dq_head=dq_head, dkv_heads_per_cta=kv_heads, packed=packed)


# ------------------------------------------------------------------ the reference
def _ent_rows(base, B, E, Sk, stride, dev):
    """KV row of key j of entity e of business b: [B, E, Sk]."""
    st = stride or Sk
    b = torch.arange(B, device=dev)[:, None, None]
    e = torch.arange(E, device=dev)[None, :, None]
    return base + (b * E + e) * st + torch.arange(Sk, device=dev)


def ref_attention(q, k, v, mods, key_valid, ent_valid, R, E_total, qs, causal=False, fill=None):
    """Multi-entity attention in fp32, restated from the references of test_multi_entity_cross_attention_fwd_bwd and
    test_decode_cross_attention.  q: [n_qseq * qs, D] (query sequence = business * R + target); k, v: [memory rows, D].
    Per modality, per entity: softmax over the entity's keys (masked keys filled with `fill`: -2^16 for cross-attention,
    -inf for self-attention), entity e skipped for target e under leave-one-out, entities without a valid key dropped, the
    mean over the remaining n entities taken as (1/n) sum, and 0 for a modality with none.
    Returns the per-modality outputs [n_qseq * qs, D], the log2-domain log-sum-exp [n_qseq, H, E_total, qs] (NaN where an
    entity is not attended) and the attended-entity mask [n_qseq, E_total]."""
    dev = q.device
    n_qseq = q.shape[0] // qs
    B = n_qseq // R
    fill = float("-inf") if fill is None else fill
    qh = q.view(B, R, qs, H, HD).permute(0, 1, 3, 2, 4) * SCALE                          # [B, R, H, qs, hd]
    lse = torch.full((B, R, H, E_total, qs), float("nan"), device=dev)
    inc_all = torch.zeros(B, R, E_total, dtype=torch.bool, device=dev)
    outs = []
    for base, _o, E, Sk, loo, eb, stride in mods:
        rows = _ent_rows(base, B, E, Sk, stride, dev)
        kk = k[rows].view(B, E, Sk, H, HD).permute(0, 1, 3, 2, 4)                          # [B, E, H, Sk, hd]
        vv = v[rows].view(B, E, Sk, H, HD).permute(0, 1, 3, 2, 4)
        valid = key_valid[rows] != 0
        if ent_valid is not None:
            valid = valid & (ent_valid[:, eb:eb + E, None] != 0)
        keep = valid[:, None, :, None, None, :]                                            # [B, 1, E, 1, 1, Sk]
        if causal:
            keep = keep & torch.ones(qs, Sk, dtype=torch.bool, device=dev).tril()
        w = qh[:, :, None] @ kk[:, None].transpose(-1, -2)                                 # [B, R, E, H, qs, Sk]
        o = torch.softmax(w.masked_fill(~keep, fill), -1) @ vv[:, None]
        inc = valid.any(-1)[:, None, :].expand(B, R, E).clone()
        if loo:
            inc &= ~torch.eye(R, E, dtype=torch.bool, device=dev)[None]
        o = o.masked_fill(~inc[:, :, :, None, None, None], 0.0)
        n = inc.sum(2).clamp(min=1).float()
        outs.append((o.sum(2) / n[:, :, None, None, None]).permute(0, 1, 3, 2, 4).reshape(n_qseq * qs, D))
        with torch.no_grad():
            l2 = torch.logsumexp(w.masked_fill(~keep, float("-inf")), -1) * LOG2E           # [B, R, E, H, qs]
            lse[:, :, :, eb:eb + E] = torch.where(inc[:, :, :, None, None], l2, float("nan")).transpose(2, 3)
        inc_all[:, :, eb:eb + E] = inc
    return outs, lse.view(n_qseq, H, E_total, qs), inc_all.view(n_qseq, E_total)


def entity_bookkeeping(mods, key_valid, B, R):
    """ent_valid [B, E_total] (an entity has a valid key) and inv_n [B * R, n_mod] (1 / #attended entities, 0 for none),
    the arrays the training step's prep kernel and the generation memory builder hand to the kernels."""
    ev, inv = [], []
    for base, _o, E, Sk, loo, _eb, stride in mods:
        ent = (key_valid[_ent_rows(base, B, E, Sk, stride, key_valid.device)] != 0).any(-1)      # [B, E]
        cnt = ent.sum(1, keepdim=True).float().expand(B, R)
        if loo:
            cnt = cnt - ent[:, :R].float()
        ev.append(ent)
        inv.append(torch.where(cnt > 0, 1.0 / cnt.clamp(min=1), torch.zeros_like(cnt)).reshape(-1))
    return torch.cat(ev, 1).to(torch.uint8).contiguous(), torch.stack(inv, 1).contiguous()


# ------------------------------------------------------------------ comparisons
def _close(name, got, ref, rtol):
    got, ref = got.float(), ref.float()
    assert torch.isfinite(got).all(), "%s: non-finite values" % name
    scale = max(ref.abs().max().item(), 1e-6)
    err = (got - ref).abs().max().item()
    assert err <= rtol * scale, "%s: max err %.4g vs scale %.4g (rtol %.3g)" % (name, err, scale, rtol)


def _regions(c):
    """(name, first row, end row) of every modality's block of memory rows."""
    B = c.n_qseq // c.R
    return [(nm, m[0], m[0] + B * m[2] * (m[6] or m[3])) for nm, m in zip(c.mod_names, c.mods)]


def _row_valid(c):
    """Per memory row: the key can be attended by some query (valid key of a non-null entity)."""
    B = c.n_qseq // c.R
    rv = torch.zeros(c.kv_rows, dtype=torch.bool, device=_dev())
    for base, _o, E, Sk, loo, eb, stride in c.mods:
        rows = _ent_rows(base, B, E, Sk, stride, rv.device)
        ok = c.key_valid[rows] != 0
        if c.ent_valid is not None:
            ok &= c.ent_valid[:, eb:eb + E, None] != 0
        rv[rows.reshape(-1)] = ok.reshape(-1)
    return rv


# ------------------------------------------------------------------ cases
def _case(Q, q_col, KV, k_col, v_col, fused, key_valid, mods, mod_names, n_qseq, R, q_rows=0, causal=False, fill=None,
          bookkeeping=True, dO=True):
    B = n_qseq // R
    qs = q_rows or SQ
    Tq = n_qseq * qs
    mods = [tuple(m[:1]) + (i * Tq * D,) + tuple(m[2:6]) + ((m[6] if len(m) > 6 else 0),) for i, m in enumerate(mods)]
    E_total = sum(m[2] for m in mods)
    ent_valid, inv_n = entity_bookkeeping(mods, key_valid, B, R) if bookkeeping else (None, None)
    c = SimpleNamespace(Q=Q, q_col=q_col, KV=KV, k_col=k_col, v_col=v_col, fused=fused, key_valid=key_valid, ent_valid=ent_valid,
                        inv_n=inv_n, mods=mods, mod_names=mod_names, n_qseq=n_qseq, R=R, E_total=E_total, q_rows=q_rows, qs=qs,
                        Tq=Tq, causal=causal, fill=fill)
    c.kv_rows = max(m[0] + B * m[2] * (m[6] or m[3]) for m in mods)
    c.paths = attn_paths(mods, n_qseq, R)
    if dO:
        c.dO = torch.randn(len(mods) * Tq, D, device=_dev()).to(torch.bfloat16)
    return c


def cross_case(seed, B, R, S_text, F, n_img, text_lens, tab_valid, img_mask, ik=196):
    """Decoder cross-attention of the training step: 128 decoder rows per (business, target review) against the memory
    [text B*R*S_text | table B*F | image B*n_img*ik] (engine._cross_attn_args)."""
    dev = _dev()
    torch.manual_seed(seed)
    N = B * R
    T = N * SQ
    Tt = B * R * S_text
    Tm = Tt + B * F + B * n_img * ik
    qc = torch.randn(T, D, device=dev).to(torch.bfloat16)
    kv = torch.randn(Tm, 2 * D, device=dev).to(torch.bfloat16)
    tvalid = torch.arange(S_text, device=dev)[None, None, :] < text_lens.to(dev)[:, :, None]
    ivalid = img_mask.to(dev)[:, :, None].expand(B, n_img, ik)
    key_valid = torch.cat([tvalid.reshape(-1), tab_valid.to(dev).reshape(-1), ivalid.reshape(-1)]).to(torch.uint8).contiguous()
    mods = [(0, 0, R, S_text, 1, 0), (Tt, 0, 1, F, 0, R), (Tt + B * F, 0, n_img, ik, 0, R + 1)]
    return _case(qc, 0, kv, 0, D, False, key_valid, mods, ("text", "table", "image"), N, R, fill=_neg_cross())


def self_case(seed, n_seq, causal, frame=SQ, lens_lo=20):
    """Encoder / decoder self-attention over frames of `frame` rows (q_rows = frame when < 128), pad keys at the tail."""
    dev = _dev()
    torch.manual_seed(seed)
    T = n_seq * frame
    qkv = torch.randn(T, 3 * D, device=dev).to(torch.bfloat16)
    lens = torch.randint(min(lens_lo, frame), frame + 1, (n_seq,), device=dev)
    lens[0] = frame
    key_valid = (torch.arange(frame, device=dev)[None, :] < lens[:, None]).reshape(-1).to(torch.uint8).contiguous()
    return _case(qkv, 0, qkv, D, 2 * D, True, key_valid, [(0, 0, 1, frame, 0, 0)], ("self",), n_seq, 1,
                 q_rows=0 if frame == SQ else frame, causal=causal, bookkeeping=False)


def encoder_case(seed, N, S):
    """The generation encoder's call (inference.encoder_forward): frames of Sp = 256 rows, R = 2 query tiles per sequence,
    one key entity of Sk = 208 rows at an entity stride of Sp.  Sequence 0 is S tokens long, the others are ragged."""
    dev = _dev()
    torch.manual_seed(seed)
    Sp = SQ * math.ceil(S / SQ)
    Sk = min(Sp, K_MAX_KEYS)
    qkv = torch.randn(N * Sp, 3 * D, device=dev).to(torch.bfloat16)
    lens = torch.randint(S // 2, S + 1, (N,), device=dev)
    lens[0] = S
    valid = torch.zeros(N, Sp, device=dev, dtype=torch.uint8)
    valid[:, :S] = (torch.arange(S, device=dev)[None, :] < lens[:, None]).to(torch.uint8)
    c = _case(qkv, 0, qkv, D, 2 * D, True, valid.reshape(-1).contiguous(), [(0, 0, 1, Sk, 0, 0, Sp)], ("self",), N * (Sp // SQ),
              Sp // SQ, bookkeeping=False, dO=False)
    c.lens = lens
    return c


def _neg_cross():
    from oracle import mmsum_oracle as OR
    return OR.NEG_CROSS


def yelp_case(seed=31):
    """Yelp training step: 9 reviews (one null review in the middle of business 0), trimmed encoder frame 112, a partially
    masked 47-key table, 10 images (20 entities) — business 0's images alternate valid / null inside the packed key range,
    business 1 has none."""
    B, R, S_text, F, n_img = 3, 9, 112, 47, 10
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(20, S_text + 1, (B, R), generator=g)
    lens[:, 0] = S_text
    lens[0, 4] = 0                                                    # a null review between valid ones
    tab = torch.rand(B, F, generator=g) > 0.3
    tab[:, 0] = True
    img = torch.ones(B, n_img, dtype=torch.bool)
    img[0] = torch.arange(n_img) % 2 == 0                             # valid / null alternating across the packed tiles
    img[1] = False                                                    # no images
    img[2, 7] = False
    return cross_case(seed, B, R, S_text, F, n_img, lens, tab, img)


def amazon_case(seed=32):
    """Amazon training step: 9 reviews on an 80-row frame, a 133-key table (second dK/dV tile of 5 keys) with a ragged mask
    and one business whose table is fully masked, one image per business (E = 1: not packed, tiles of 128 + 68 keys)."""
    B, R, S_text, F, n_img = 3, 9, 80, 133, 1
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(10, S_text + 1, (B, R), generator=g)
    lens[:, 1] = S_text
    tab = torch.rand(B, F, generator=g) > 0.4
    tab[0, 128:] = True                                               # keys of the 5-key tail tile attended ...
    tab[2, 130:] = False                                              # ... and partly masked
    tab[2, 128] = True
    tab[1] = False                                                    # a business without a table
    img = torch.tensor([[True], [True], [False]])
    return cross_case(seed, B, R, S_text, F, n_img, lens, tab, img)


def ceiling_case(seed=33, n_img=15):
    """8 reviews + table + n_img images: 24 entities (kMaxEnt) at n_img = 15."""
    B, R, S_text, F = 2, 8, 96, 47
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(20, S_text + 1, (B, R), generator=g)
    tab = torch.rand(B, F, generator=g) > 0.3
    tab[:, 0] = True
    img = torch.rand(B, n_img, generator=g) > 0.3
    img[0, 0] = img[1, n_img - 1] = True
    img[1, 5:9] = False
    return cross_case(seed, B, R, S_text, F, n_img, lens, tab, img)


# ------------------------------------------------------------------ running the kernels
def _args(c, O, LSE, **bwd):
    ops = _ops()
    return ops.attn_args(Q=c.Q, ldq=c.Q.stride(0), q_col=c.q_col, KV=c.KV, ldkv=c.KV.stride(0), k_col=c.k_col, v_col=c.v_col,
                         O=O, ldo=D, LSE=LSE, key_valid=c.key_valid, ent_valid=c.ent_valid, inv_n=c.inv_n, n_qseq=c.n_qseq, H=H,
                         R=c.R, causal=int(c.causal), E_total=c.E_total, scale=SCALE, q_rows=c.q_rows, mods=c.mods, **bwd)


def run_kernels(c, bwd=True, poisoned=False):
    """Forward (+ backward) into sentinel-filled buffers: 7.0 in the bf16 outputs, NaN in LSE / DELTA.  `poisoned`: NaN
    everywhere, and every SM's shared / tensor memory filled with NaN patterns before each launch."""
    ops = _ops()
    dev = _dev()
    s = float("nan") if poisoned else 7.0
    n_mod = len(c.mods)
    r = SimpleNamespace()
    r.O = torch.full((n_mod * c.Tq + GUARD, D), s, device=dev, dtype=torch.bfloat16)
    r.LSE = torch.full((c.n_qseq, H, c.E_total, SQ), float("nan"), device=dev)
    if poisoned:
        ops.debug_poison()
    ops.attn_fwd(_args(c, r.O, r.LSE))
    if bwd:
        r.DELTA = torch.full((c.n_qseq, H, c.E_total, SQ), float("nan"), device=dev)
        if c.fused:
            r.dQ = r.dKV = torch.full((c.Tq + GUARD, 3 * D), s, device=dev, dtype=torch.bfloat16)
            cols = dict(lddq=3 * D, dq_col=0, lddkv=3 * D, dk_col=D, dv_col=2 * D)
        else:
            r.dQ = torch.full((c.Tq + GUARD, D), s, device=dev, dtype=torch.bfloat16)
            r.dKV = torch.full((c.kv_rows + GUARD, 2 * D), s, device=dev, dtype=torch.bfloat16)
            cols = dict(lddq=D, dq_col=0, lddkv=2 * D, dk_col=0, dv_col=D)
        if poisoned:
            ops.debug_poison()
        ops.attn_bwd(_args(c, c.dO, r.LSE, DELTA=r.DELTA, dQ=r.dQ, dKV=r.dKV, **cols))
        r.dq = r.dQ[:c.Tq, :D]
        r.dk = r.dKV[:c.kv_rows, cols["dk_col"]:cols["dk_col"] + D]
        r.dv = r.dKV[:c.kv_rows, cols["dv_col"]:cols["dv_col"] + D]
    torch.cuda.synchronize()
    return r


def check_parity(c, name, bwd=True):
    """Kernel outputs against ref_attention, per modality and per memory region, plus the exact checks."""
    r = run_kernels(c, bwd)
    q = c.Q[:c.Tq, c.q_col:c.q_col + D].float().requires_grad_(bwd)
    k = c.KV[:c.kv_rows, c.k_col:c.k_col + D].float().requires_grad_(bwd)
    v = c.KV[:c.kv_rows, c.v_col:c.v_col + D].float().requires_grad_(bwd)
    outs, lse_ref, inc = ref_attention(q, k, v, c.mods, c.key_valid, c.ent_valid, c.R, c.E_total, c.qs, c.causal, c.fill)
    for m, nm in enumerate(c.mod_names):
        _close("%s fwd %s" % (name, nm), r.O[m * c.Tq:(m + 1) * c.Tq], outs[m], FWD_TOL)
    assert (r.O[len(c.mods) * c.Tq:] == 7.0).all(), "%s: output written behind the last frame" % name
    # log-sum-exp: written for every attended (sequence, head, entity), never for the others
    got = r.LSE[:, :, :, :c.qs].permute(0, 2, 1, 3)[inc]
    want = lse_ref.permute(0, 2, 1, 3)[inc]
    err = (got - want).abs().max().item()
    assert err <= 2e-3 + 1e-4 * want.abs().max().item(), "%s: LSE max err %.4g" % (name, err)
    assert r.LSE.permute(0, 2, 1, 3)[~inc].isnan().all(), "%s: LSE written for an entity that is not attended" % name
    if not bwd:
        return r
    torch.autograd.backward(outs, [c.dO[m * c.Tq:(m + 1) * c.Tq].float() for m in range(len(c.mods))])
    assert r.DELTA.permute(0, 2, 1, 3)[~inc].isnan().all(), "%s: DELTA written for an entity that is not attended" % name
    _close("%s dq" % name, r.dq, q.grad, BWD_TOL)
    for nm, a, b in _regions(c):
        _close("%s dk %s rows" % (name, nm), r.dk[a:b], k.grad[a:b], BWD_TOL)
        _close("%s dv %s rows" % (name, nm), r.dv[a:b], v.grad[a:b], BWD_TOL)
    dead = ~_row_valid(c)
    assert (r.dk[dead] == 0).all() and (r.dv[dead] == 0).all(), "%s: dK/dV of a masked or null key is not exactly 0" % name
    assert (r.dQ[c.Tq:] == 7.0).all(), "%s: dQ written behind the last frame" % name
    if not c.fused:
        assert (r.dKV[c.kv_rows:] == 7.0).all(), "%s: dK/dV written behind the memory" % name
    return r


def check_stale_state(c, name, bwd=True):
    """Bit-identical results with NaN-filled buffers after every SM's shared / tensor memory was filled with NaN patterns."""
    clean = run_kernels(c, bwd)
    for _ in range(2):
        dirty = run_kernels(c, bwd, poisoned=True)
        pairs = [("out", clean.O[:len(c.mods) * c.Tq], dirty.O[:len(c.mods) * c.Tq])]
        if bwd:
            pairs += [("dq", clean.dq, dirty.dq), ("dk", clean.dk, dirty.dk), ("dv", clean.dv, dirty.dv)]
        for nm, a, b in pairs:
            assert torch.isfinite(b.float()).all(), (name, nm)
            assert torch.equal(a, b), (name, nm)
        inc = ~clean.LSE.isnan()
        assert torch.equal(inc, ~dirty.LSE.isnan()) and torch.equal(clean.LSE[inc], dirty.LSE[inc]), (name, "LSE")


# ------------------------------------------------------------------ training-step cross-attention
def test_yelp_training_cross_attention():
    c = yelp_case()
    assert c.paths["packed"] == [False, False, True] and c.paths["fwd_hpc"] == 0 and not c.paths["dq_head"]
    assert c.E_total == 20
    check_parity(c, "yelp")


def test_amazon_training_cross_attention():
    c = amazon_case()
    assert c.paths["packed"] == [False, False, False] and c.paths["dkv_heads_per_cta"] == 1
    assert c.mods[1][3] == 133 and c.mods[2][2:4] == (1, 196)
    check_parity(c, "amazon")


def test_entity_ceiling():
    c = ceiling_case()
    assert c.E_total == K_MAX_ENT and c.paths["packed"] == [False, False, True]
    check_parity(c, "24 entities")
    over = ceiling_case(n_img=16)
    assert over.E_total == K_MAX_ENT + 1
    ops = _ops()
    from multimodalsum_b200._lib import MmsumError
    O = torch.full((3 * over.Tq, D), 7.0, device=_dev(), dtype=torch.bfloat16)
    LSE = torch.full((over.n_qseq, H, over.E_total, SQ), float("nan"), device=_dev())
    launches = ops.LAUNCHES
    with pytest.raises(MmsumError):
        ops.attn_fwd(_args(over, O, LSE))
    torch.cuda.synchronize()
    assert ops.LAUNCHES == launches and (O == 7.0).all() and LSE.isnan().all()


# ------------------------------------------------------------------ generation encoder
@pytest.mark.parametrize("N,hpc", [(5, 0), (40, H // 2), (160, H)])
@pytest.mark.parametrize("S", [150, 208])
def test_generation_encoder_frames(S, N, hpc):
    """Forward with exactly the arguments of inference.encoder_forward; every row of the 256-row frame (pad query rows
    included) against self-attention over the frame's valid keys.  S = 208 with an all-valid sequence: a 208-column score
    tile, whose TMEM columns overlap the previous head's O accumulator."""
    c = encoder_case(40 + N, N, S)
    assert c.mods[0][3:] == (K_MAX_KEYS, 0, 0, 256) and c.R == 2
    assert c.paths["fwd_hpc"] == hpc
    if S == K_MAX_KEYS:
        assert int(c.lens.max()) == K_MAX_KEYS        # n16 = 208 > the O accumulator's first column (192)
    check_parity(c, "encoder S=%d N=%d" % (S, N), bwd=False)


# ------------------------------------------------------------------ self-attention dispatch boundaries
@pytest.mark.parametrize("causal", [0, 1])
@pytest.mark.parametrize("n_seq", [63, 64, 296, 297])
def test_self_attention_dispatch_boundaries(n_seq, causal):
    c = self_case(50 + n_seq, n_seq, causal)
    p = c.paths
    assert p["fwd_hpc"] == (0 if n_seq < 64 else (H // 2 if n_seq <= 2 * N_SMS else H))
    assert p["dq_head"] == (n_seq >= 64) and p["dkv_heads_per_cta"] == (4 if n_seq >= 64 else 1)
    check_parity(c, "self n=%d causal=%d" % (n_seq, causal))


@pytest.mark.parametrize("frame", list(range(16, SQ + 1, 16)))
def test_self_attention_trimmed_frames_head_mode(frame):
    c = self_case(60 + frame, 64, False, frame=frame, lens_lo=frame // 2)
    assert c.paths["fwd_hpc"] == H // 2 and c.paths["dq_head"] and c.paths["dkv_heads_per_cta"] == 4
    check_parity(c, "self frame=%d" % frame)


# ------------------------------------------------------------------ decode-step attention
@pytest.mark.parametrize("Sk_text,F,n_img", [(158, 47, 10), (158, 133, 1), (208, 47, 10)])
def test_decode_cross_attention_production(Sk_text, F, n_img):
    """Beam-search cross-attention at the config-5 shape: 64 businesses x 4 beams, 8 reviews + table + images."""
    ops = _ops()
    dev = _dev()
    torch.manual_seed(70 + F)
    B, beams, R = 64, 4, 8
    N = B * beams
    Tt = B * R * Sk_text
    Tm = Tt + B * F + B * n_img * 196
    q = torch.randn(N, D, device=dev).to(torch.bfloat16)
    kv = torch.randn(Tm, 2 * D, device=dev).to(torch.bfloat16)
    lens = torch.randint(30, Sk_text + 1, (B, R), device=dev)
    lens[:, 0] = Sk_text
    lens[3, 2] = lens[9, 7] = 0                                         # null reviews
    tab = torch.rand(B, F, device=dev) > 0.3
    tab[:, 0] = True
    tab[5] = False                                                      # no table
    img = torch.rand(B, n_img, device=dev) > 0.3
    img[0] = torch.arange(n_img, device=dev) % 2 == 0
    img[1] = False                                                      # no images
    key_valid = torch.cat([(torch.arange(Sk_text, device=dev)[None, None] < lens[:, :, None]).reshape(-1), tab.reshape(-1),
                           img[:, :, None].expand(B, n_img, 196).reshape(-1)]).to(torch.uint8).contiguous()
    mods = [(0, 0, R, Sk_text, 0, 0, 0), (Tt, N * D, 1, F, 0, R, 0), (Tt + B * F, 2 * N * D, n_img, 196, 0, R + 1, 0)]
    assert sum(m[2] for m in mods) == R + 1 + n_img
    ent_valid, inv_n = entity_bookkeeping(mods, key_valid, B, beams)
    A3 = torch.full((3 * N + GUARD, D), 7.0, device=dev, dtype=torch.bfloat16)
    ops.attn_decode_cross(ops.attn_args(Q=q, ldq=D, q_col=0, KV=kv, ldkv=2 * D, k_col=0, v_col=D, O=A3, ldo=D, LSE=None,
                                        key_valid=key_valid, ent_valid=ent_valid, inv_n=inv_n, n_qseq=N, H=H, R=beams, causal=0,
                                        E_total=R + 1 + n_img, scale=SCALE, mods=mods))
    outs, _, _ = ref_attention(q.float(), kv[:, :D].float(), kv[:, D:].float(), mods, key_valid, ent_valid, beams,
                               R + 1 + n_img, 1, fill=_neg_cross())
    for m, nm in enumerate(("text", "table", "image")):
        _close("decode cross %s" % nm, A3[m * N:(m + 1) * N], outs[m], FWD_TOL)
    assert (A3[N:2 * N].view(B, beams, D)[5] == 0).all() and (A3[2 * N:3 * N].view(B, beams, D)[1] == 0).all()
    assert (A3[3 * N:] == 7.0).all()


def test_decode_self_attention_whole_cache():
    """Token-by-token causal self-attention over all 128 cache positions (every score slot of a lane, positions 0..127),
    the slot table permuted after every step as beam search re-ranks hypotheses."""
    ops = _ops()
    torch.manual_seed(80)
    N, S = 16, 128
    dev = _dev()
    cache = torch.zeros(N, S, 2 * D, device=dev, dtype=torch.bfloat16)
    hist = torch.zeros(N, S, device=dev, dtype=torch.int32)
    pos = torch.zeros(1, device=dev, dtype=torch.int32)
    out = torch.empty(N, D, device=dev, dtype=torch.bfloat16)
    Kh = torch.zeros(N, S, D, device=dev)
    Vh = torch.zeros(N, S, D, device=dev)
    g = torch.Generator().manual_seed(81)
    for t in range(S):
        qkv = torch.randn(N, 3 * D, device=dev).to(torch.bfloat16)
        ops.attn_decode_self(qkv, cache, hist, pos, out, H, SCALE)
        Kh[:, t], Vh[:, t] = qkv[:, D:2 * D].float(), qkv[:, 2 * D:].float()
        qf = qkv[:, :D].float().view(N, H, 1, HD) * SCALE
        kk = Kh[:, :t + 1].view(N, t + 1, H, HD).transpose(1, 2)
        vv = Vh[:, :t + 1].view(N, t + 1, H, HD).transpose(1, 2)
        ref = (torch.softmax(qf @ kk.transpose(-1, -2), -1) @ vv).transpose(1, 2).reshape(N, D)
        _close("decode self t=%d" % t, out, ref, FWD_TOL)
        src = ((torch.arange(N) // 4) * 4 + torch.randint(0, 4, (N,), generator=g)).to(dev)
        hist.copy_(hist.index_select(0, src))
        Kh, Vh = Kh[src], Vh[src]
        pos += 1


# ------------------------------------------------------------------ stale on-chip state on the new paths
def test_head_mode_208_keys_ignores_stale_onchip_state():
    c = encoder_case(90, 160, K_MAX_KEYS)
    assert c.paths["fwd_hpc"] == H
    check_stale_state(c, "encoder 208 keys, hpc = H", bwd=False)


def test_packed_images_backward_ignores_stale_onchip_state():
    c = yelp_case(91)
    assert c.paths["packed"][2]
    check_stale_state(c, "yelp packed images")


def test_amazon_table_backward_ignores_stale_onchip_state():
    c = amazon_case(92)
    check_stale_state(c, "amazon table")
