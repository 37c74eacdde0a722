"""What freezing parameters (requires_grad=False) saves in the training step, BART-large 12 + 12 layers, 16 businesses, dropout 0.1,
plain launches, FusedAdamW with the fused clip, the two arms of each workload alternating in one process:

  * image stage (ImgSupervised, 10 images per business): all trainable vs BART frozen; the optimizer covers img_encoder in both
    arms, as the reference's does;
  * table stage (TableSupervised, Yelp): all trainable vs BART frozen; the optimizer covers the table encoder's own weights;
  * multimodal step (bench.py's Yelp workload, config 2): all trainable vs encoder + shared.weight frozen, one optimizer per arm
    over its trainable parameters.

ms/step from CUDA events around STEPS steps, REPS rounds per arm (median, min, max), and C-ABI kernel launches per step.  Also the
LayerNorm backward alone at the decoder shape (18432 rows, dropout 0.1) with and without the gamma / beta reduction, CUDA events
around 50 calls.  Prints the GPU name and power limit with the numbers."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from multimodalsum_b200 import ops
from multimodalsum_b200.modules import ImgSupervised, MultimodalSum, TableSupervised, YelpTableEncoder
from multimodalsum_b200.optim import get_optimizer
from multimodalsum_b200.synth import ModelConfig, make_batch

B, STEPS, REPS, WARM = 16, 5, 5, 2
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                     text=True).stdout.strip().splitlines()
print("gpu: %s" % (smi[0] if smi else torch.cuda.get_device_name()))
NO_DECAY = ["bias", "LayerNorm.weight"]


def workload(name):
    torch.manual_seed(0)
    if name == "img":
        cfg = ModelConfig(dataset="img", dropout=0.1)
        model = ImgSupervised(config=cfg).cuda().train()
        b = make_batch(cfg, B, seed=1234, n_valid_imgs=10).to("cuda")
        call = lambda: model(b.img, b.img_mask, labels=b.labels)[0]                            # noqa: E731
        head = lambda n: n.startswith("img_encoder.")                                          # noqa: E731
        frozen = lambda n: n.startswith("bart_model.")                                         # noqa: E731
    elif name == "table":
        cfg = ModelConfig(dataset="table_yelp", dropout=0.1)
        model = TableSupervised(TableEncoder=YelpTableEncoder, config=cfg).cuda().train()
        b = make_batch(cfg, B, seed=1234).to("cuda")
        call = lambda: model(b.field, b.field_value, labels=b.labels)[0]                       # noqa: E731
        head = lambda n: n.startswith("table_encoder.")                                        # noqa: E731
        frozen = lambda n: n.startswith("bart_model.")                                         # noqa: E731
    else:
        cfg = ModelConfig(dataset="yelp", dropout=0.1)
        model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg, label_smoothing=0.1).cuda().train()
        b = make_batch(cfg, B, seed=1234, fixed_len=100, n_valid_imgs=10).with_length_hint().to("cuda")
        call = lambda: model(b.reviews, b.reviews_mask, b.reviews_rating, b.field, b.field_value, b.img, b.img_mask,  # noqa: E731
                             max_review_len=b.max_review_len)[0]
        head = lambda n: True                                                                  # noqa: E731
        frozen = lambda n: n.startswith("bart_model.model.encoder.") or n == "bart_model.model.shared.weight"   # noqa: E731
    return model, call, head, frozen


def run(name):
    model, call, head, frozen = workload(name)
    eng = model._ensure_engine(torch.device("cuda"))
    named = list(model.named_parameters())
    arms = {}
    for arm, fr in (("all trainable", lambda n: False), ("frozen", frozen)):
        opt = get_optimizer(eng, 1e-5, NO_DECAY, [(n, p) for n, p in named if head(n) and not fr(n)], None, max_grad_norm=1.0)
        arms[arm] = (fr, opt)

    def step(arm):
        fr, opt = arms[arm]
        for n, p in named:
            p.requires_grad_(not fr(n))
        loss = call()
        opt.zero_grad()
        loss.backward()
        opt.step(lr=1e-5)

    for arm in arms:
        for _ in range(WARM):
            step(arm)
    torch.cuda.synchronize()
    times, launches = {a: [] for a in arms}, {}
    for _ in range(REPS):
        for arm in arms:
            step(arm)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            n0 = ops.LAUNCHES
            s.record()
            for _ in range(STEPS):
                step(arm)
            e.record()
            torch.cuda.synchronize()
            launches[arm] = (ops.LAUNCHES - n0) / STEPS
            times[arm].append(s.elapsed_time(e) / STEPS)
    med = {}
    for arm, t in times.items():
        ts = sorted(t)
        med[arm] = ts[len(ts) // 2]
        print("%-10s %-14s ms/step median %7.2f (min %7.2f, max %7.2f; %d rounds of %d steps)  launches/step %5.0f"
              % (name, arm, med[arm], ts[0], ts[-1], len(ts), STEPS, launches[arm]))
    print("%-10s frozen / all trainable: %.3f" % (name, med["frozen"] / med["all trainable"]))
    del model, arms
    torch.cuda.empty_cache()


for w in ("img", "table", "multimodal"):
    run(w)

# ---- LayerNorm backward alone at the decoder shape, with and without gamma / beta
rows, D = 16 * 9 * 128, 1024
g = torch.Generator(device="cuda").manual_seed(0)
bf = lambda *s: torch.randn(*s, device="cuda", generator=g).to(torch.bfloat16)      # noqa: E731
res, y, d1, d2 = bf(rows, D), bf(rows, D), bf(rows, D), bf(rows, D)
mean, rstd, gamma = torch.zeros(rows, device="cuda"), torch.ones(rows, device="cuda"), torch.ones(D, device="cuda")
dres, dy, dg, db = torch.empty_like(res), torch.empty_like(res), torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
res_us = {}
for _ in range(3):
    for arm, (a, b_) in (("with gamma/beta", (dg, db)), ("without", (None, None))):
        for i in range(60):
            if i == 10:
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
            ops.add_ln_bwd(d1, d2, res, y, gamma, mean, rstd, dres, dy, a, b_, 0.1, 3, 5)
        e.record()
        torch.cuda.synchronize()
        res_us.setdefault(arm, []).append(s.elapsed_time(e) / 50 * 1e3)
for arm, t in res_us.items():
    print("add_ln_bwd %d x 1024, dropout 0.1, %-16s %6.1f us/call (min of 3 rounds of 50)" % (rows, arm, min(t)))
