"""Host side of requires_grad=False in the training step: the backward plan for the freezing patterns users write, the C-ABI's
rejection of malformed partial-output calls, the data-parallel exchange of trainable ranges only, and FusedAdamW's handling of
frozen parameters."""
import ctypes as C
import math
import os
import socket
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from multimodalsum_b200 import _lib
from multimodalsum_b200.engine import ALIGN, _arena_order, backward_plan
from multimodalsum_b200.synth import ModelConfig

BM = "bart_model.model."
ENC, DEC, SHARED = BM + "encoder.", BM + "decoder.", BM + "shared.weight"


def _cfg(dataset, **kw):
    return ModelConfig(dataset=dataset, encoder_layers=2, decoder_layers=4, ffn_dim=256, vocab_size=512, max_position_embeddings=128,
                       **kw)


def _plan(cfg, frozen):
    names = _arena_order(cfg)
    return names, backward_plan(cfg, names, [n for n in names if not frozen(n)])


def _full_labels(cfg):
    labels = {"head.in"}
    for l in range(cfg.decoder_layers):
        t = "dec.%d." % l
        labels |= {t + "ffn.dH", t + "ffn.in", t + "cross.dO3", t + "cross.dA3", t + "cross.in", t + "self.dctx", t + "self.in"}
        if cfg.multimodal:
            labels.add(t + "cross.dU")
    if cfg.text_memory:
        for l in range(cfg.encoder_layers):
            t = "enc.%d." % l
            labels |= {t + "ffn.dH", t + "ffn.in", t + "self.dctx", t + "self.in"}
    if cfg.table is not None:
        labels |= {"table.dtab_h", "table.dtabX"}
    return labels


@pytest.mark.parametrize("dataset", ["yelp", "amazon", "text", "img", "table_yelp", "table_amazon"])
def test_all_trainable_plan_is_the_full_backward(dataset):
    cfg = _cfg(dataset)
    names, p = _plan(cfg, lambda n: False)
    mods = tuple(m for m, on in (("text", cfg.text_memory), ("table", cfg.table is not None), ("image", cfg.image)) if on)
    assert p.run and p.dgrad == _full_labels(cfg)
    assert p.dkv == (mods,) * cfg.decoder_layers
    assert {m for m, on in p.mem.items() if on} == set(mods)
    assert all(p.dec_in) and (all(p.enc_in) if cfg.text_memory else p.enc_in == ())
    # every parameter the step reaches gets its gradient (the img / table stages never run the encoder)
    assert p.grads == {n for n in names if cfg.text_memory or not n.startswith(ENC)}


@pytest.mark.parametrize("dataset", ["img", "table_yelp", "table_amazon"])
def test_pretraining_stages_with_bart_frozen(dataset):
    cfg = _cfg(dataset)
    names, p = _plan(cfg, lambda n: n.startswith("bart_model."))
    head = {n for n in names if not n.startswith("bart_model.")}
    mod = "image" if dataset == "img" else "table"
    assert p.grads == head and p.mem == dict(text=False, table=mod == "table", image=mod == "image")
    assert p.dkv == ((mod,),) * cfg.decoder_layers              # the memory needs dK/dV of its rows at every layer
    assert p.enc_in == () and p.dec_in[0] is False and all(p.dec_in[1:])
    # layer 0: no chain below it, so neither the cross-attention's dQ side nor the self block
    assert "dec.0.cross.in" not in p.dgrad and "dec.0.self.dctx" not in p.dgrad and "dec.0.cross.dA3" in p.dgrad
    assert "dec.1.self.in" in p.dgrad and "head.in" in p.dgrad
    assert ("table.dtab_h" in p.dgrad and "table.dtabX" in p.dgrad) == (mod == "table")


def test_multimodal_with_the_encoder_and_shared_frozen():
    cfg = _cfg("yelp")
    names, p = _plan(cfg, lambda n: n.startswith(ENC) or n == SHARED)
    assert p.mem == dict(text=False, table=True, image=True)
    assert p.enc_in == () and not any(l.startswith("enc.") for l in p.dgrad)
    assert SHARED not in p.grads and p.run and "head.in" in p.dgrad
    assert p.dkv == (("text", "table", "image"),) * cfg.decoder_layers   # k / v projections are trainable: all rows
    assert all(p.dec_in)                                                  # positions / rating / LN embeddings are trainable


def test_lower_decoder_layers_and_everything_below_frozen():
    cfg = _cfg("yelp")
    low = tuple(DEC + "layers.%d." % l for l in (0, 1))
    names, p = _plan(cfg, lambda n: not n.startswith(DEC + "layers.") or n.startswith(low))
    assert p.dec_in == (False, False, False, True, True)
    assert p.dkv[:2] == ((), ()) and p.dkv[2:] == (("text", "table", "image"),) * 2
    assert not any(l.startswith(("dec.0.", "dec.1.")) for l in p.dgrad)
    assert "dec.2.self.dctx" in p.dgrad and "dec.2.self.in" not in p.dgrad and "dec.2.cross.in" in p.dgrad
    assert not any(p.mem.values()) and p.enc_in == ()


def test_only_the_gates_trainable():
    cfg = _cfg("yelp")
    names, p = _plan(cfg, lambda n: "alpha_proj" not in n and "beta_proj" not in n)
    assert p.grads == {n for n in names if "alpha_proj" in n or "beta_proj" in n}
    assert p.dkv == ((),) * cfg.decoder_layers                    # nothing trainable needs dK/dV: the dQ/DELTA pass only
    assert "dec.0.cross.dU" in p.dgrad and "dec.0.cross.dO3" not in p.dgrad and "dec.0.cross.dA3" not in p.dgrad
    assert "dec.1.cross.dA3" in p.dgrad and "dec.1.cross.in" in p.dgrad      # layer 0's gates need the chain through layer 1
    assert "dec.0.ffn.in" in p.dgrad and "dec.0.self.dctx" not in p.dgrad


def test_one_cross_k_proj_frozen_narrows_the_fused_group():
    cfg = _cfg("yelp")
    k = DEC + "layers.2.encoder_attn.k_proj."
    names, p = _plan(cfg, lambda n: n.startswith(k))
    full = _plan(cfg, lambda n: False)[1]
    assert p.dgrad == full.dgrad and p.dkv == full.dkv and p.mem == full.mem
    assert p.grads == full.grads - {k + "weight", k + "bias"}
    eng = types.SimpleNamespace(plan=p)
    from multimodalsum_b200.engine import StepEngine
    runs = StepEngine._fused_runs(eng, [k + "weight", DEC + "layers.2.encoder_attn.v_proj.weight"])
    assert runs == [[1, 2]]                                        # v only: the column slice dy[:, D:2D]
    s = DEC + "layers.2.self_attn."
    eng.plan = _plan(cfg, lambda n: n == s + "k_proj.weight")[1]
    assert StepEngine._fused_runs(eng, [s + "q_proj.weight", s + "k_proj.weight", s + "v_proj.weight"]) == [[0, 1], [2, 3]]
    eng.plan = full
    assert StepEngine._fused_runs(eng, [s + "q_proj.weight", s + "k_proj.weight", s + "v_proj.weight"]) == [[0, 3]]


def test_one_layernorm_frozen_and_shared_frozen():
    cfg = _cfg("amazon")
    ln = DEC + "layers.1.encoder_attn_layer_norm."
    names, p = _plan(cfg, lambda n: n.startswith(ln))
    full = _plan(cfg, lambda n: False)[1]
    assert p.grads == full.grads - {ln + "weight", ln + "bias"} and p.dgrad == full.dgrad and p.dkv == full.dkv
    names, p = _plan(cfg, lambda n: n == SHARED)
    # the text memory is still needed (the encoder is trainable), the embeddings run without their token-table output
    assert SHARED not in p.grads and p.mem["text"] and p.dgrad == full.dgrad and all(p.enc_in) and all(p.dec_in)


def test_encoder_backward_stops_at_the_lowest_trainable_layer():
    cfg = _cfg("text")
    names, p = _plan(cfg, lambda n: not n.startswith(ENC + "layers.1.fc"))
    assert p.enc_in == (False, False, True) and p.mem["text"]
    assert "enc.1.ffn.dH" in p.dgrad and "enc.1.ffn.in" not in p.dgrad and not any(l.startswith("enc.0.") for l in p.dgrad)
    names, p = _plan(cfg, lambda n: True)
    assert not p.run and p.grads == frozenset() and p.dgrad == frozenset()


# ------------------------------------------------------------------------------------------------------------ C-ABI
P = C.c_void_p(4096)
i32, i64, f32, u32, u64 = C.c_int32, C.c_int64, C.c_float, C.c_uint32, C.c_uint64


def test_partial_output_calls_reject_malformed_combinations_on_the_host():
    L = _lib.lib()
    ln = dict(d1=P, d2=None, res=P, y=P, gamma=P, mean=P, rstd=P, dres=P, dy=C.c_void_p(8192), dgamma=P, dbeta=P, rows=18432,
              d_model=1024, p_drop=f32(0.1), seed=u64(1), sid=u32(2), step_dev=None)
    for bad in (dict(dgamma=None), dict(dbeta=None)):                  # gamma / beta: both or neither
        args = dict(ln, **bad)
        assert L.mmsum_add_ln_bwd(*args.values(), None) == -1, bad
        assert L.mmsum_add_ln_bwd_ordered(*args.values(), P, i64(444 * 2048), None) == -1, bad
    rows, S, V = 18432, 128, 50265
    emb = dict(dout=P, dout2=None, ids=P, E=P, Pos=P, rd=P, remb=P, gamma=P, mean=P, rstd=P, dE=P, dP=P, dremb=P, dgamma=P,
               dbeta=P, dz=P, rows=rows, S=S, d_model=1024, pad=1, p_drop=f32(0.1), seed=u64(1), sid=u32(3), step_dev=None)
    ws = (V, P, i64(1 << 30), None)
    for bad in (dict(dgamma=None), dict(dbeta=None), dict(dgamma=None, dE=None, dP=None, dremb=None, dbeta=P),
                dict(remb=None, dremb=None)):
        args = dict(emb, **bad)
        assert L.mmsum_embed_ln_bwd(*args.values(), None) == -1, bad
        assert L.mmsum_embed_ln_bwd_ordered_subset(*args.values(), *ws) == -1, bad
    # nothing to compute: the ordered subset call is malformed; the plain call is a no-op (the host skips it anyway)
    none = dict(emb, dE=None, dP=None, dremb=None, dgamma=None, dbeta=None)
    assert L.mmsum_embed_ln_bwd_ordered_subset(*none.values(), *ws) == -1
    assert L.mmsum_embed_ln_bwd(*none.values(), None) == 0
    # the full ordered entry point still requires every output
    for bad in (dict(dE=None), dict(dP=None), dict(dremb=None), dict(dgamma=None, dbeta=None)):
        assert L.mmsum_embed_ln_bwd_ordered(*dict(emb, **bad).values(), *ws) == -1, bad


def test_attn_bwd_rejects_a_no_dkv_flag_other_than_0_or_1():
    L = _lib.lib()
    a = _lib.AttnArgs(Q=4096, KV=4096, O=4096, LSE=4096, DELTA=4096, dQ=4096, dKV=4096, ldq=1024, ldkv=2048, ldo=1024, lddq=1024,
                      lddkv=2048, v_col=1024, dv_col=1024, n_qseq=16, H=16, R=1, n_mod=1, E_total=1, scale=0.125)
    a.mods[0].E, a.mods[0].Sk = 1, 128
    for flag in (2, -1):
        a.mods[0].no_dkv = flag
        assert L.mmsum_attn_bwd(C.byref(a), None) == -1, flag


# ---------------------------------------------------------------------------------------------------- data parallel
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


HOLES = [(0, 3000), (3000, 5000), (9000, 12000), (20000, 40000), (60000, 65536)]   # trainable ranges (0,3000)+(3000,5000) merge


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from multimodalsum_b200.dp import GradAllReducer
    n = 1 << 16
    merged = [(0, 5000), (9000, 12000), (20000, 40000), (60000, 65536)]
    eng = types.SimpleNamespace(G32=torch.zeros(n), numel=n, device=torch.device("cpu"), grad_ready_hook=None,
                                grad_ranges=lambda: merged)
    red = GradAllReducer(eng, bucket_mb=0.0625)           # 16 Ki fp32 elements per bucket
    torch.manual_seed(100 + rank)
    local = torch.randn(n)
    mask = torch.zeros(n, dtype=torch.bool)
    for lo, hi in merged:
        mask[lo:hi] = True
    local[~mask] = 0.0                                    # frozen ranges are zero in the arena
    local[~mask & (torch.arange(n) % 2 == 0)] = float(rank + 1)   # a frozen range is never read: plant a per-rank value there
    cuts = [1000, 9000, 20000, 20001, 50000, n]
    lo = 0
    for hi in cuts:
        eng.G32[lo:hi] = local[lo:hi]
        eng.grad_ready_hook(hi)
        lo = hi
    torch.manual_seed(100)
    g0 = torch.randn(n)
    torch.manual_seed(101)
    g1 = torch.randn(n)
    ok = torch.allclose(eng.G32[mask], ((g0 + g1) / 2)[mask], atol=1e-6)
    ok = ok and bool((eng.G32[~mask] == local[~mask]).all())          # untouched
    # buckets as before ([0,20000) [20000,50000) [50000,n)); all-reduces only over their trainable parts: (0,5000) (9000,12000) |
    # (20000,40000) | (60000,65536)
    ok = ok and red.n_buckets == 3 and red.n_allreduce == 4 and red.lo == 0 and not red.works
    q.put((rank, bool(ok), red.n_allreduce))
    dist.destroy_process_group()


def test_grad_allreducer_exchanges_only_trainable_ranges_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
    assert all(ok for _, ok, _ in res), res


# -------------------------------------------------------------------------------------------------------- optimizer
def _fake_engine():
    shapes = {"a.weight": (8, 8), "a.bias": (8,), "b.weight": (100,), "c.weight": (4, 16)}
    params, offsets, off = {}, {}, 0
    for n, sh in shapes.items():
        params[n] = torch.nn.Parameter(torch.zeros(sh))
        offsets[n] = off
        off += (math.prod(sh) + ALIGN - 1) // ALIGN * ALIGN
    eng = types.SimpleNamespace(params=params, offsets=offsets, shapes=shapes, numel=off, device=torch.device("cpu"),
                                trainable=frozenset(shapes))
    return eng


def test_fused_adamw_skips_frozen_parameters():
    from multimodalsum_b200.optim import FusedAdamW
    eng = _fake_engine()
    p = eng.params
    eng.trainable = frozenset({"a.weight", "a.bias", "c.weight"})           # b.weight frozen before the optimizer is built
    opt = FusedAdamW(eng, [{"params": [p["a.weight"], p["b.weight"]], "weight_decay": 0.01},
                           {"params": [p["a.bias"]], "weight_decay": 0.0}])
    f = opt.flags.tolist()
    blk = lambda n: slice(eng.offsets[n] // ALIGN, (eng.offsets[n] + math.prod(eng.shapes[n]) + ALIGN - 1) // ALIGN)   # noqa: E731
    assert f[blk("a.weight")] == [3] and f[blk("a.bias")] == [1]
    assert f[blk("b.weight")] == [0, 0] and f[blk("c.weight")] == [0]      # frozen / in no group
    # the set may change freely before the first step
    eng.trainable = frozenset(eng.shapes)
    opt._sync_flags()
    assert opt.flags.tolist()[blk("b.weight")] == [3, 3]
    eng.trainable = frozenset({"a.weight", "a.bias", "c.weight"})
    opt._sync_flags()
    # after a step the state has no entry for the never-updated parameter (index 1 = b.weight), as torch's AdamW leaves it
    opt.step_count = 1
    sd = opt.state_dict()
    assert sorted(sd["state"]) == [0, 2] and sd["param_groups"][0]["params"] == [0, 1]
    # a parameter outside the groups may change; one of the groups may not
    eng.trainable = frozenset({"a.weight", "a.bias"})
    opt._sync_flags()
    eng.trainable = frozenset({"a.weight"})
    with pytest.raises(ValueError, match="a.bias"):
        opt.step(lr=1e-3)
    eng.trainable = frozenset(eng.shapes) - {"c.weight"}
    with pytest.raises(ValueError, match="b.weight"):
        opt.step(lr=1e-3)
