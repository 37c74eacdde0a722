"""requires_grad=False in the training step (DESIGN.md §4, "Frozen parameters"): the kernels' partial-output variants, and the
step with the freezing patterns users write against the all-trainable step on the same inputs and seed, under
torch.use_deterministic_algorithms(True) so that the gradients compare bit for bit."""
import types

import pytest
import torch

from test_deterministic_gpu import _batch_args, _case, _make_model, _rel, _same_bits, deterministic

pytestmark = pytest.mark.gpu

D = 1024
BM = "bart_model.model."
ENC, DEC, SHARED = BM + "encoder.", BM + "decoder.", BM + "shared.weight"


# ============================================================================================================ kernel level
def _ln_inputs(rows, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    bf = lambda *s: torch.randn(*s, device="cuda", generator=g).to(torch.bfloat16)   # noqa: E731
    res, y, d1, d2 = bf(rows, D), bf(rows, D), bf(rows, D), bf(rows, D)
    z = res.float() + y.float()
    mean, rstd = z.mean(1), torch.rsqrt(z.var(1, unbiased=False) + 1e-5)
    return res, y, d1, d2, torch.rand(D, device="cuda", generator=g) + 0.5, mean, rstd


@pytest.mark.parametrize("rows,p_drop,ordered", [(18432, 0.1, False), (18432, 0.1, True), (18432, 0.0, False), (752, 0.1, True)])
def test_add_ln_bwd_without_gamma_beta(rows, p_drop, ordered):
    """dgamma = dbeta = NULL: dres and dy bitwise those of the full call; one kernel."""
    from multimodalsum_b200 import ops
    res, y, d1, d2, gamma, mean, rstd = _ln_inputs(rows, rows + int(ordered))
    step = torch.tensor([3], device="cuda", dtype=torch.int32)
    ws = torch.empty(ops.ADD_LN_BWD_WORKSPACE, device="cuda") if ordered else None

    def run(grads):
        dres = torch.full_like(res, float("nan"))
        dy = dres if p_drop == 0 else torch.full_like(res, float("nan"))
        dg, db = (torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")) if grads else (None, None)
        n0 = ops.LAUNCHES
        ops.add_ln_bwd(d1, d2, res, y, gamma, mean, rstd, dres, dy, dg, db, p_drop, 7, 11, step_dev=step, workspace=ws)
        torch.cuda.synchronize()
        return dres, dy, ops.LAUNCHES - n0

    full, frozen = run(True), run(False)
    assert torch.equal(full[0], frozen[0]) and torch.equal(full[1], frozen[1]) and torch.isfinite(frozen[0]).all()
    assert frozen[2] == 1 and full[2] == (2 if ordered else 1)


def _embed_case(rows, S, V, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = lambda *s: torch.randn(*s, device="cuda", generator=g)    # noqa: E731
    ids = torch.randint(0, V, (rows,), device="cuda", generator=g, dtype=torch.int32)
    ids[rows // 3:rows // 2] = 1
    E, P, rd, remb = f(V, D) * 0.1, f(S + 2, D) * 0.1, f(rows // S), f(D) * 0.1
    gamma = torch.rand(D, device="cuda", generator=g) + 0.5
    z = E[ids.long()] + P[torch.arange(rows, device="cuda") % S + 2] + rd.repeat_interleave(S)[:, None] * remb
    mean, rstd = z.mean(1), torch.rsqrt(z.var(1, unbiased=False) + 1e-5)
    return dict(dout=f(rows, D).to(torch.bfloat16), dout2=f(rows, D).to(torch.bfloat16), ids=ids, E=E, P=P, rd=rd, remb=remb,
                gamma=gamma, mean=mean, rstd=rstd)


@pytest.mark.parametrize("ordered", [True, False])
@pytest.mark.parametrize("drop", [("dE",), ("dP",), ("dremb",), ("ln",), ("dE", "ln"), ("dP", "dremb"), ("dE", "dP", "dremb")])
def test_embed_ln_bwd_with_outputs_null(drop, ordered):
    """Each output (and combinations) NULL: the others bitwise those of the full call (atomic path: the single-writer outputs
    dP and dz; the ordered path: every output), the NULL ones untouched, and the kernels that only served them not launched."""
    from multimodalsum_b200 import ops
    rows, S, V = 18432, 128, 50265
    c = _embed_case(rows, S, V, 11)
    ws = torch.empty(ops.embed_ln_bwd_workspace(rows, S, V), device="cuda") if ordered else None
    step = torch.tensor([2], device="cuda", dtype=torch.int32)

    def run(skip):
        out = dict(dE=torch.zeros(V, D, device="cuda"), dP=torch.zeros(S + 2, D, device="cuda"), dremb=torch.zeros(D, device="cuda"),
                   dg=torch.zeros(D, device="cuda"), db=torch.zeros(D, device="cuda"))
        arg = {k: (None if k in skip or (k in ("dg", "db") and "ln" in skip) else v) for k, v in out.items()}
        dz = torch.empty(rows, D, device="cuda")
        n0 = ops.LAUNCHES
        ops.embed_ln_bwd(c["dout"], c["dout2"], c["ids"], c["E"], c["P"], c["rd"], c["remb"], c["gamma"], c["mean"], c["rstd"],
                         arg["dE"], arg["dP"], arg["dremb"], arg["dg"], arg["db"], dz, rows, S, 1, 0.1, 3, 9, step_dev=step,
                         workspace=ws)
        torch.cuda.synchronize()
        return out, dz, ops.LAUNCHES - n0

    full, dz_full, n_full = run(())
    part, dz_part, n_part = run(drop)
    assert torch.equal(dz_full, dz_part) and n_part <= n_full
    if ordered and "dE" in drop:
        assert n_full - n_part >= 3                                               # no id sort, tile or span scatter
    if "dP" in drop and "dremb" in drop:
        assert n_full - n_part >= 1                                               # no position / rating-embedding kernel
    for k in ("dE", "dP", "dremb", "dg", "db"):
        key = "ln" if k in ("dg", "db") else k
        if key in drop:
            assert (part[k] == 0).all(), k                                        # not written
        elif ordered or k == "dP":
            assert _same_bits(part[k], full[k]), k
        else:
            assert _rel(part[k], full[k]) <= 1e-5, k                              # fp32 atomics: order-dependent rounding


def _cross_case(seed):
    """A Yelp-shaped cross-attention: text (2 businesses x 3 reviews, leave-one-out), table (47 rows), image (2 x 196 keys)."""
    from multimodalsum_b200 import layers as L
    from multimodalsum_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    B, R, S, F, n_img, ik, H = 2, 3, 128, 47, 2, 196, 16
    Tt, Tm, T = B * R * S, B * R * S + B * F + B * n_img * ik, B * R * S
    bf = lambda *s: (torch.randn(*s, device="cuda", generator=g) * 0.5).to(torch.bfloat16)   # noqa: E731
    eng = types.SimpleNamespace(cfg=types.SimpleNamespace(d_model=D, heads=H, head_dim=64))
    qc, kv, O3, dA3 = bf(T, D), bf(Tm, 2 * D), torch.empty(3, T, D, device="cuda", dtype=torch.bfloat16), bf(3, T, D)
    lse = torch.empty(B * R, H, R + 1 + n_img, S, device="cuda")
    mem_valid = torch.ones(Tm, device="cuda", dtype=torch.uint8)
    ent_valid = torch.ones(B, R + 1 + n_img, device="cuda", dtype=torch.uint8)
    inv_n = torch.tensor([1.0 / (R - 1), 1.0, 0.5], device="cuda").repeat(B * R, 1).contiguous()
    mods = [(0, R, S), (Tt, 1, F), (Tt + B * F, n_img, ik)]
    args = lambda **bwd: L.cross_attn_args(eng, qc, kv, O3 if not bwd else dA3, lse, mods, mem_valid, ent_valid, inv_n, B * R, R,  # noqa: E731
                                           loo=True, **bwd)
    ops.attn_fwd(args())
    rows = dict(text=(0, Tt), table=(Tt, Tt + B * F), image=(Tt + B * F, Tm))
    return args, T, Tm, rows


@pytest.mark.parametrize("skip", [("text",), ("text", "table", "image"), ("table", "image")])
def test_attn_bwd_skips_dkv_of_flagged_modalities(skip):
    from multimodalsum_b200 import ops
    args, T, Tm, rows = _cross_case(5)
    delta = torch.empty(6, 16, 6, 128, device="cuda")

    def run(no_dkv):
        dq = torch.full((T, D), float("nan"), device="cuda", dtype=torch.bfloat16)
        dkv = torch.full((Tm, 2 * D), float("nan"), device="cuda", dtype=torch.bfloat16)
        n0 = ops.LAUNCHES
        ops.attn_bwd(args(DELTA=delta, dQ=dq, lddq=D, dq_col=0, dKV=dkv, lddkv=2 * D, dk_col=0, dv_col=D, no_dkv=no_dkv))
        torch.cuda.synchronize()
        return dq, dkv, ops.LAUNCHES - n0

    dq0, dkv0, n0 = run(None)
    dq1, dkv1, n1 = run([m in skip for m in ("text", "table", "image")])
    assert torch.isfinite(dq0).all() and torch.isfinite(dkv0).all()
    assert torch.equal(dq0, dq1)
    for m, (r0, r1) in rows.items():
        if m in skip:
            assert torch.isnan(dkv1[r0:r1].float()).all(), m                      # the sentinel is left in place
        else:
            assert torch.equal(dkv0[r0:r1], dkv1[r0:r1]), m
    assert n0 == 2 and n1 == (1 if len(skip) == 3 else 2)


# ============================================================================================================== step level
def _set_frozen(model, frozen):
    for n, p in model.named_parameters():
        p.requires_grad_(not frozen(n))


def _step(model, cfg, batch):
    from multimodalsum_b200 import ops
    a, kw = _batch_args(cfg, batch)
    n0 = ops.LAUNCHES
    loss = model(*a, **kw)[0]
    model.zero_grad(set_to_none=True)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach().clone(), ops.LAUNCHES - n0


def _compare_pattern(name, frozen, narrowed=(), must_drop=True):
    """One step all trainable, one with `frozen` applied, from the same weights, dropout seed and batch."""
    cfg, sd, batches = _case(name)
    model = _make_model(cfg, sd)
    eng = model._ensure_engine(torch.device("cuda"))
    w0, rng0 = eng.W32.clone(), eng.rng_state()
    with deterministic(True):
        loss_a, n_a = _step(model, cfg, batches[0])
        g_all = eng.G32.clone()
        eng.set_rng_state(rng0)
        _set_frozen(model, frozen)
        loss_f, n_f = _step(model, cfg, batches[0])
    assert _same_bits(eng.W32, w0)
    assert _same_bits(loss_a, loss_f)
    n_frozen = 0
    for n, p in eng.params.items():
        o, k = eng.offsets[n], p.numel()
        if frozen(n):
            n_frozen += 1
            assert p.grad is None, n
            assert (eng.G32[o:o + k] == 0).all() and not torch.signbit(eng.G32[o:o + k]).any(), n
        elif n in narrowed:
            assert _rel(eng.G32[o:o + k], g_all[o:o + k]) <= 1e-5, n
        else:
            assert p.grad is not None and p.grad.data_ptr() == eng.G32[o:].data_ptr(), n
            assert _same_bits(eng.G32[o:o + k], g_all[o:o + k]), (n, (eng.G32[o:o + k] != g_all[o:o + k]).sum().item())
    assert n_frozen > 0
    assert (n_f < n_a) if must_drop else (n_f <= n_a), (n_f, n_a)
    return model, eng


def _lower_half(name):
    cfg = _case(name)[0]
    low = tuple(DEC + "layers.%d." % l for l in range(cfg.decoder_layers // 2))
    return lambda n: not n.startswith(DEC + "layers.") or n.startswith(low)


PATTERNS = {
    "img_bart_frozen": ("small_img", lambda n: n.startswith("bart_model."), ()),
    "table_yelp_bart_frozen": ("small_table_yelp", lambda n: n.startswith("bart_model."), ()),
    "table_amazon_bart_frozen": ("small_table_amazon", lambda n: n.startswith("bart_model."), ()),
    "encoder_and_shared_frozen": ("small_yelp_gates_open", lambda n: n.startswith(ENC) or n == SHARED, ()),
    "lower_decoder_and_below_frozen": ("small_amazon", None, ()),
    "only_gates_trainable": ("small_yelp_gates_open", lambda n: "alpha_proj" not in n and "beta_proj" not in n, ()),
    "one_cross_k_proj_frozen": ("small_yelp_gates_open", lambda n: n.startswith(DEC + "layers.1.encoder_attn.k_proj."),
                                (DEC + "layers.1.encoder_attn.v_proj.weight", DEC + "layers.1.encoder_attn.v_proj.bias")),
    "one_layernorm_frozen": ("small_yelp", lambda n: n.startswith(DEC + "layers.0.final_layer_norm."), ()),
    "shared_frozen": ("small_yelp_gates_open", lambda n: n == SHARED, ()),
}


@pytest.mark.parametrize("pattern", list(PATTERNS))
def test_frozen_pattern_matches_the_all_trainable_step(pattern):
    """Trainable gradients bitwise equal (a narrowed fused group within fp32 reduction-order tolerance: its weight gradient is a
    narrower GEMM), frozen `.grad` None and frozen arena ranges exactly +0, fewer kernel launches (the narrowed group runs one
    GEMM either way, so there the count may stay)."""
    name, frozen, narrowed = PATTERNS[pattern]
    if frozen is None:
        frozen = _lower_half(name)
    _compare_pattern(name, frozen, narrowed, must_drop=pattern != "one_cross_k_proj_frozen")


def test_frozen_encoder_at_the_benchmark_shape():
    """Yelp, 16 businesses, BART-large 12 + 12 layers: encoder + shared frozen (the common fine-tuning set-up)."""
    _compare_pattern("yelp_b16", lambda n: n.startswith(ENC) or n == SHARED)


def test_image_stage_trajectory_with_bart_frozen():
    """Three steps of make_loops(stage='img')'s body (forward, zero_grad, backward, clip_grad_norm_ over what the stage clips,
    step) with a FusedAdamW over img_encoder built without max_grad_norm: BART frozen or not, the img_encoder weights are
    bitwise the same and BART does not move."""
    from multimodalsum_b200.optim import get_optimizer
    from multimodalsum_b200.train_utils import _stage_table
    cfg, sd, batches = _case("small_img")
    model = _make_model(cfg, sd)
    eng = model._ensure_engine(torch.device("cuda"))
    w0, rng0 = eng.W32.clone(), eng.rng_state()
    clip = _stage_table(type("A", (), {"dataset": "yelp"})(), None, "img")["clip"]
    img = "img_encoder.linear.weight"
    o, k = eng.offsets[img], eng.params[img].numel()
    finals = []
    with deterministic(True):
        for freeze in (False, True):
            eng.W32.copy_(w0)
            eng.mark_weights_dirty()
            eng.set_rng_state(rng0)
            _set_frozen(model, lambda n: freeze and n.startswith("bart_model."))
            opt = get_optimizer(eng, 1e-3, ["bias", "LayerNorm.weight"], list(model.img_encoder.named_parameters()))
            for b in batches:
                a, kw = _batch_args(cfg, b)
                loss = model(*a, **kw)[0]
                opt.zero_grad()
                loss.backward()
                torch.nn.utils.clip_grad_norm_(clip(model), 0.5)
                opt.step()
            torch.cuda.synchronize()
            finals.append(eng.W32.clone())
    assert _same_bits(finals[0][o:o + k], finals[1][o:o + k]) and not _same_bits(finals[0][o:o + k], w0[o:o + k])
    for f in finals:
        assert _same_bits(torch.cat([f[:o], f[o + k:]]), torch.cat([w0[:o], w0[o + k:]]))


def test_stock_adamw_leaves_a_frozen_encoder_unchanged():
    cfg, sd, batches = _case("small_yelp_gates_open")
    model = _make_model(cfg, sd)
    eng = model._ensure_engine(torch.device("cuda"))
    model.bart_model.model.encoder.requires_grad_(False)
    assert not model.bart_model.model.shared.weight.requires_grad            # frozen too, through embed_tokens
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=0.01)
    for b in batches[:2]:
        a, kw = _batch_args(cfg, b)
        loss = model(*a, **kw)[0]
        opt.zero_grad()
        loss.backward()
        opt.step()
    torch.cuda.synchronize()
    moved = 0
    for n, p in model.named_parameters():
        if n.startswith(ENC) or n == SHARED:
            assert p.grad is None and _same_bits(p.detach(), before[n]), n
        else:
            moved += not _same_bits(p.detach(), before[n])
    assert moved > 0 and eng.plan.mem["text"] is False


def test_graph_replay_with_the_trainable_set_toggled():
    """Steps alternating between two trainable sets replay recorded graphs (one per set) and equal plain launches bit for bit."""
    cfg, sd, batches = _case("small_yelp_gates_open")
    model = _make_model(cfg, sd)
    eng = model._ensure_engine(torch.device("cuda"))
    w0, rng0 = eng.W32.clone(), eng.rng_state()
    sets = [lambda n: False, lambda n: n.startswith(ENC) or n == SHARED]
    runs = []
    with deterministic(True):
        for graph in (False, True):
            eng.W32.copy_(w0)
            eng.mark_weights_dirty()
            eng.set_rng_state(rng0)
            eng.enable_graph(graph)
            out = []
            for i in range(6):
                _set_frozen(model, sets[i % 2])
                loss, _ = _step(model, cfg, batches[0])
                out.append((loss, eng.G32.clone(), [p.grad is None for p in eng.params.values()]))
            runs.append(out)
            if graph:
                assert len(eng._graphs) == 2 and all("bwd" in e for e in eng._graphs.values())
    eng.enable_graph(False)
    for (l0, g0, n0), (l1, g1, n1) in zip(*runs):
        assert _same_bits(l0, l1) and _same_bits(g0, g1) and n0 == n1


def test_no_trainable_parameter_gives_a_loss_without_grad():
    cfg, sd, batches = _case("small_yelp")
    model = _make_model(cfg, sd)
    model.requires_grad_(False)
    a, kw = _batch_args(cfg, batches[0])
    loss = model(*a, **kw)[0]
    assert not loss.requires_grad and torch.isfinite(loss)
    with pytest.raises(RuntimeError):
        loss.backward()
    model.requires_grad_(True)
    assert model(*a, **kw)[0].requires_grad
