"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference on the synthetic
weights/inputs of multimodalsum_b200.synth.  Needs a checkout of the reference at $MMSUM_REF,
oracle/_ref or baseline/_ref (see oracle/ref_harness.py):

    python tests/golden/make_golden.py [small|full|all]

Each .npz holds: the case description (json), the reference's fp32 loss, the L2 norm of every parameter gradient
and the first 64 entries (stride 997) of every gradient.  Weights/inputs are NOT stored: they are rebuilt from the
seeds in the case description (torch CPU generators are deterministic for the pinned torch build).
"""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from multimodalsum_b200.synth import ModelConfig, make_batch, make_state_dict  # noqa: E402
from oracle import ref_harness as RH  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

SMALL = dict(encoder_layers=2, decoder_layers=2, ffn_dim=256, vocab_size=512, max_position_embeddings=128, dropout=0.0)
CASES = {
    # name: (cfg kwargs, state-dict kwargs, batch kwargs)
    "small_yelp": (dict(SMALL, dataset="yelp"), dict(seed=0), dict(B=2, seed=1, n_reviews=4, max_imgs=2)),
    "small_yelp_gates_open": (dict(SMALL, dataset="yelp"), dict(seed=0, gates_open=True), dict(B=3, seed=2, n_reviews=3, max_imgs=3)),
    "small_amazon": (dict(SMALL, dataset="amazon"), dict(seed=3), dict(B=2, seed=4, n_reviews=4)),
    "small_text": (dict(SMALL, dataset="text"), dict(seed=5), dict(B=2, seed=6, n_reviews=3)),
    "full_yelp_b1": (dict(dataset="yelp", dropout=0.0), dict(seed=0), dict(B=1, seed=1, n_reviews=9, n_valid_imgs=4)),
    "full_yelp_b1_gates_open": (dict(dataset="yelp", dropout=0.0), dict(seed=0, gates_open=True), dict(B=1, seed=7, n_reviews=9)),
    "full_text_b1": (dict(dataset="text", dropout=0.0), dict(seed=0), dict(B=1, seed=8, n_reviews=9)),
    # single-modality pretraining stages (src/img_pretrain.py, src/table_pretrain.py)
    "small_img": (dict(SMALL, dataset="img"), dict(seed=9), dict(B=3, seed=10, max_imgs=3)),
    "small_table_yelp": (dict(SMALL, dataset="table_yelp"), dict(seed=9), dict(B=3, seed=11)),
    "small_table_amazon": (dict(SMALL, dataset="table_amazon"), dict(seed=9), dict(B=3, seed=12)),
}


GEN_CFG = dict(encoder_layers=2, decoder_layers=2, ffn_dim=256, vocab_size=512, max_position_embeddings=256, dropout=0.0,
               dataset="yelp")
GEN_CASES = {
    # name: (cfg kwargs, state-dict kwargs, batch kwargs, generate kwargs) — BASELINE config 5 semantics at toy size
    "gen_small_yelp_s128": (GEN_CFG, dict(seed=21, gates_open=True), dict(B=3, seed=31, n_reviews=3, max_imgs=2, seq_len=128, len_range=(68, 118)),
                            dict(num_beams=4, max_length=24, length_penalty=1.0, no_repeat_ngram_size=3, early_stopping=True)),
    # tie-free variant: a wide random final_logits_bias (seed 77, std 2) separates the candidates by far more than bf16 noise,
    # so the CUDA path must reproduce the ids exactly
    "gen_small_yelp_biased": (GEN_CFG, dict(seed=21, gates_open=True, logits_bias_std=2.0), dict(B=3, seed=33, n_reviews=3, max_imgs=2, seq_len=150, len_range=(90, 140)),
                              dict(num_beams=4, max_length=24, length_penalty=1.0, no_repeat_ngram_size=3, early_stopping=True)),
    "gen_small_yelp_s150": (GEN_CFG, dict(seed=21, gates_open=True), dict(B=3, seed=32, n_reviews=3, max_imgs=2, seq_len=150, len_range=(90, 140)),
                            dict(num_beams=4, max_length=24, length_penalty=1.0, no_repeat_ngram_size=3, early_stopping=True)),
}


def make_generation_goldens():
    for name, (ck, sk, bk, gk) in GEN_CASES.items():
        t0 = time.time()
        cfg = ModelConfig(**ck)
        sd = make_state_dict(cfg, **sk)
        bk2 = dict(bk)
        batch = make_batch(cfg, bk2.pop("B"), **bk2)
        out = RH.reference_generate(cfg, sd, batch, **gk)
        np.savez_compressed(os.path.join(HERE, name + ".npz"),
                            case=json.dumps(dict(name=name, cfg=ck, sd=sk, batch=bk, gen=gk, torch=torch.__version__, ref_dtype="float32")),
                            tokens=out.numpy())
        print("%s: tokens %s, %.1fs" % (name, tuple(out.shape), time.time() - t0), flush=True)


def build_case(name):
    ck, sk, bk = CASES[name]
    cfg = ModelConfig(**ck)
    sd = make_state_dict(cfg, **sk)
    bk = dict(bk)
    batch = make_batch(cfg, bk.pop("B"), **bk)
    return cfg, sd, batch


def sample(g):
    return g.flatten()[::997][:64].double().numpy()


def main(which):
    for name in CASES:
        if which != "all" and not name.startswith(which):
            continue
        t0 = time.time()
        cfg, sd, batch = build_case(name)
        if cfg.dataset == "text":
            loss, grads, _ = RH.reference_text_step(cfg, sd, batch, dtype=torch.float32, label_smoothing=None)
        elif not cfg.text_memory:
            loss, grads, _ = RH.reference_stage_step(cfg, sd, batch, dtype=torch.float32, label_smoothing=0.1)
        else:
            loss, grads, _ = RH.reference_step(cfg, sd, batch, dtype=torch.float32, label_smoothing=0.1)
        out = {"case": json.dumps(dict(name=name, cfg=CASES[name][0], sd=CASES[name][1], batch=CASES[name][2],
                                       torch=torch.__version__, ref_dtype="float32")),
               "loss": np.float64(loss.item())}
        names = sorted(grads)
        out["names"] = np.array(names)
        out["norms"] = np.array([grads[n].double().norm().item() for n in names])
        out["samples"] = np.stack([np.pad(sample(grads[n]), (0, 64 - len(sample(grads[n])))) for n in names])
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print("%s: loss %.9f, %d grads, %.1fs" % (name, loss.item(), len(names), time.time() - t0), flush=True)


OPT_CASE = dict(cfg=dict(SMALL, dataset="yelp"), sd=dict(seed=0), grads=dict(seed=4, std=1e-3), lr=1e-3, steps=3,
                max_grad_norm=1.0, num_epochs=1, t_epoch=4, warmup_ratio=0.5, no_decay=["bias", "LayerNorm.weight"])


def make_optimizer_golden():
    """clip_grad_norm_ + AdamW + linear warm-up schedule exactly as src/multimodal_train.py:359-364 drives them:
    the reference's own get_optimizer / get_scheduler (src/train_utils.py:49-63, incl. the exhausted-generator quirk Q1),
    the vendored transformers-3.0.2 AdamW (src/transformer/optimization.py:168-267), torch's clip_grad_norm_."""
    import argparse
    from multimodalsum_b200.synth import make_grads
    c = OPT_CASE
    cfg = ModelConfig(**c["cfg"])
    sd = make_state_dict(cfg, **c["sd"])
    grads = make_grads(cfg, **c["grads"])
    model = RH.build_reference_model(cfg, sd, dtype=torch.float32)
    import train_utils as TU          # the reference's (RH put the checkout's src/ on sys.path)
    opt = TU.get_optimizer(c["lr"], c["no_decay"], model.named_parameters(), None)
    sched = TU.get_scheduler(argparse.Namespace(num_epochs=c["num_epochs"], warmup_ratio=c["warmup_ratio"]), c["t_epoch"], opt)
    named = dict(model.named_parameters())
    lrs, gnorms = [], []
    for _ in range(c["steps"]):
        opt.zero_grad()
        for n, p in named.items():
            p.grad = grads[n].clone()
        lrs.append(opt.param_groups[0]["lr"])
        gnorms.append(float(torch.nn.utils.clip_grad_norm_(model.parameters(), c["max_grad_norm"])))
        opt.step()
        sched.step()
    names = sorted(named)
    np.savez_compressed(os.path.join(HERE, "adamw_small.npz"),
                        case=json.dumps(dict(name="adamw_small", torch=torch.__version__, **c)),
                        names=np.array(names), lrs=np.array(lrs), gnorms=np.array(gnorms),
                        norms=np.array([named[n].detach().double().norm().item() for n in names]),
                        delta_norms=np.array([(named[n].detach().double() - sd[n].double()).norm().item() for n in names]),
                        samples=np.stack([np.pad(sample(named[n].detach()), (0, 64 - len(sample(named[n].detach())))) for n in names]),
                        sched_lrs=np.array([TU_lr for TU_lr in _sched_table(c)]))
    print("adamw_small: lrs %s, grad norms %s" % (lrs, gnorms), flush=True)


def _sched_table(c):
    """lr after k scheduler steps, k = 0..t_total+1, from the reference's get_scheduler on a dummy optimizer."""
    import argparse
    import train_utils as TU
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=c["lr"])
    sched = TU.get_scheduler(argparse.Namespace(num_epochs=c["num_epochs"], warmup_ratio=c["warmup_ratio"]), c["t_epoch"], opt)
    out = [opt.param_groups[0]["lr"]]
    for _ in range(c["t_epoch"] * c["num_epochs"] + 1):
        opt.step()
        sched.step()
        out.append(opt.param_groups[0]["lr"])
    return out


if __name__ == "__main__":
    which = sys.argv[1] if len(sys.argv) > 1 else "all"
    if which in ("all", "gen"):
        make_generation_goldens()
    if which in ("all", "opt"):
        make_optimizer_golden()
    if which not in ("gen", "opt"):
        main(which)
