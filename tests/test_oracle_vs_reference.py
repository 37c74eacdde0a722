"""LIVE pin of the test infrastructure against the UNMODIFIED reference tree (skipped unless a checkout of it is present
at $MMSUM_REF, oracle/_ref or baseline/_ref; it is not part of this repository, and the committed goldens carry the
same pin everywhere else):
  * oracle/mmsum_oracle.py vs the reference's own forward + backward (multimodal, text-only, img / table stages);
  * the golden files can be regenerated bit-for-bit (one case re-run);
  * checkpoint + optimizer-state interchange: what multimodalsum_b200.train_utils.save_checkpoint writes loads into the
    reference model / the reference's AdamW (src/train_utils.py:79-97, src/test.py:205)."""
import os

import numpy as np
import pytest
import torch

from golden_util import GOLDEN_DIR, load_golden, load_optimizer_golden
from multimodalsum_b200.synth import ModelConfig, make_batch, make_state_dict
from oracle import mmsum_oracle as OR
from oracle import ref_harness as RH

pytestmark = pytest.mark.skipif(not RH.available(), reason="needs a checkout of the unmodified reference ($MMSUM_REF, oracle/_ref or baseline/_ref)")

SMALL = dict(encoder_layers=1, decoder_layers=2, ffn_dim=128, vocab_size=300, max_position_embeddings=128, dropout=0.0)


def _rel(a, b):
    return (a.double() - b.double()).norm().item() / max(b.double().norm().item(), 1e-30)


def _compare(gref, gor):
    assert set(gref) <= set(gor) | {n for n in gref if n.endswith("final_logits_bias")}
    for n, g in gref.items():
        if n.endswith("k_proj.bias"):
            continue       # identically zero in exact arithmetic (softmax shift invariance): rounding noise on both sides
        assert _rel(gor[n], g) <= 2e-4, (n, _rel(gor[n], g))


@pytest.mark.parametrize("dataset", ["yelp", "amazon"])
def test_oracle_step_matches_live_reference(dataset):
    cfg = ModelConfig(dataset=dataset, **SMALL)
    sd = make_state_dict(cfg, seed=13, gates_open=True)
    batch = make_batch(cfg, 2, seed=14, n_reviews=3, max_imgs=2)
    lref, gref, _ = RH.reference_step(cfg, sd, batch, dtype=torch.float32)
    lor, gor, _ = OR.step_loss_and_grads(sd, cfg, batch, 0.1, dtype=torch.float32)
    assert abs(lref.item() - lor.item()) <= 2e-6 * abs(lref.item())
    _compare(gref, gor)


def test_oracle_text_step_matches_live_reference():
    cfg = ModelConfig(dataset="text", **SMALL)
    sd = make_state_dict(cfg, seed=15)
    batch = make_batch(cfg, 2, seed=16, n_reviews=3)
    lref, gref, _ = RH.reference_text_step(cfg, sd, batch, dtype=torch.float32, label_smoothing=None)
    lor, gor, _ = OR.step_loss_and_grads(sd, cfg, batch, None, dtype=torch.float32)
    assert abs(lref.item() - lor.item()) <= 2e-6 * abs(lref.item())
    _compare(gref, gor)


@pytest.mark.parametrize("dataset", ["img", "table_yelp", "table_amazon"])
def test_oracle_stage_step_matches_live_reference(dataset):
    cfg = ModelConfig(dataset=dataset, **SMALL)
    sd = make_state_dict(cfg, seed=17)
    batch = make_batch(cfg, 3, seed=18, max_imgs=2)
    lref, gref, _ = RH.reference_stage_step(cfg, sd, batch, dtype=torch.float32)
    lor, gor, _ = OR.step_loss_and_grads(sd, cfg, batch, 0.1, dtype=torch.float32)
    assert abs(lref.item() - lor.item()) <= 2e-6 * abs(lref.item())
    _compare(gref, gor)


def test_committed_golden_is_reproducible_from_the_reference():
    gold = load_golden("small_yelp")
    loss, grads, _ = RH.reference_step(gold["cfg"], gold["sd"], gold["batch"], dtype=torch.float32)
    assert loss.item() == gold["loss"]
    for n in gold["names"]:
        assert abs(grads[n].double().norm().item() - gold["norms"][n]) <= 1e-12 + 1e-9 * gold["norms"][n], n


def test_checkpoint_and_optimizer_state_interchange_with_reference(tmp_path):
    """A CPU-resident engine (arenas only, no kernels) is enough to exercise the writers."""
    from multimodalsum_b200.engine import StepEngine
    from multimodalsum_b200.modules import MultimodalSum
    from multimodalsum_b200.optim import get_optimizer
    from multimodalsum_b200.train_utils import LinearWarmupSchedule, save_checkpoint
    cfg = ModelConfig(dataset="yelp", **SMALL)
    sd = make_state_dict(cfg, seed=19)
    model = MultimodalSum(config=cfg)
    model.load_state_dict(sd, strict=False)
    eng = StepEngine(cfg, "cpu")
    eng.bind(model.named_parameters())
    object.__setattr__(model, "engine", eng)
    no_decay = ["bias", "LayerNorm.weight"]
    opt = get_optimizer(eng, 1e-3, no_decay, model.named_parameters(), None, max_grad_norm=1.0)
    torch.manual_seed(0)
    opt.m.normal_()
    opt.v.uniform_()
    opt.step_count = 2
    sched = LinearWarmupSchedule(opt, 2, 8)
    for option in ("whole", "text", "img", "table"):
        save_checkpoint(model, opt, sched, 0, str(tmp_path / option), save_option=option)
    # (1) src/test.py:205 — the unmodified reference model loads the whole-model file strictly
    ref = RH.build_reference_model(cfg, torch.load(str(tmp_path / "whole" / "pytorch_model.bin")))
    for n, p in ref.named_parameters():
        assert torch.equal(p.detach(), sd[n]), n
    # (2) stage hand-off files (src/multimodal_train.py:116-122): text -> bart_model, table -> table_encoder, img -> img_encoder
    ref.bart_model.load_state_dict(torch.load(str(tmp_path / "text" / "pytorch_model.bin")))
    ref.table_encoder.load_state_dict(torch.load(str(tmp_path / "table" / "pytorch_model.bin")))
    assert set(torch.load(str(tmp_path / "img" / "pytorch_model.bin"))) == {"linear.weight"}
    # (3) training_state.bin: the reference's own AdamW (built by the reference's get_optimizer over the same generator) loads it
    import train_utils as TU
    ref_opt = TU.get_optimizer(1e-3, no_decay, ref.named_parameters(), None)
    state = torch.load(str(tmp_path / "whole" / "training_state.bin"))
    assert state["epoch"] == 0 and state["scheduler"]["last_epoch"] == 0
    ref_opt.load_state_dict(state["optimizer"])
    named = dict(ref.named_parameters())
    by_name = {n: p for n, p in model.named_parameters()}
    checked = 0
    for n, p in named.items():
        if any(nd in n for nd in no_decay):
            assert p not in ref_opt.state                 # quirk Q1 on both sides
            continue
        st = ref_opt.state[p]
        o, k = eng.offsets[n], p.numel()
        assert st["step"] == 2
        assert torch.equal(st["exp_avg"].reshape(-1), opt.m[o:o + k]) and torch.equal(st["exp_avg_sq"].reshape(-1), opt.v[o:o + k]), n
        checked += 1
    assert checked > 20 and by_name


def test_vendored_adamw_reproduces_optimizer_golden():
    gold = load_optimizer_golden()
    z = np.load(os.path.join(GOLDEN_DIR, "adamw_small.npz"), allow_pickle=False)
    assert len(z["lrs"]) == gold["case"]["steps"]
    import argparse
    c = gold["case"]
    model = RH.build_reference_model(gold["cfg"], gold["sd"], dtype=torch.float32)
    import train_utils as TU
    opt = TU.get_optimizer(c["lr"], c["no_decay"], model.named_parameters(), None)
    sched = TU.get_scheduler(argparse.Namespace(num_epochs=c["num_epochs"], warmup_ratio=c["warmup_ratio"]), c["t_epoch"], opt)
    named = dict(model.named_parameters())
    for _ in range(c["steps"]):
        for n, p in named.items():
            p.grad = gold["grads"][n].clone()
        torch.nn.utils.clip_grad_norm_(model.parameters(), c["max_grad_norm"])
        opt.step()
        sched.step()
    for n in gold["names"]:
        assert abs(named[n].detach().double().norm().item() - gold["norms"][n]) <= 1e-9 * gold["norms"][n] + 1e-12, n
