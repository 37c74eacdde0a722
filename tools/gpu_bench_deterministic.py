"""Cost of the bitwise-reproducible step: bench.py's workload (Yelp, 16 businesses, BART-large 12 + 12 layers, dropout 0.1,
FusedAdamW, plain launches) with torch.use_deterministic_algorithms off and on, the two arms alternating in one process.

  * ms/step of each arm: CUDA events around STEPS steps, REPS rounds per arm, arms interleaved;
  * per-kernel split of each arm through ops.KERNEL_TIMER (CUDA events around every C-ABI call, bias-gradient column sums moved
    onto the main stream so that their events time the kernels, as bench.py does), in separate instrumented steps;
  * the embedding backward alone (decoder shape: 18432 rows, V = 50265, rating embedding), atomic vs ordered, for token ids
    uniform over V (the synthetic batches above), Zipf-distributed (s = 1.1: natural-text frequencies, where common tokens
    form groups of hundreds to thousands of rows) and all one id: CUDA events around 20 calls each.
Prints the GPU name and power limit with the numbers."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from multimodalsum_b200 import ops
from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
from multimodalsum_b200.optim import get_optimizer
from multimodalsum_b200.synth import ModelConfig, make_batch

B, STEPS, REPS, WARM = 16, 10, 5, 3
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                     text=True).stdout.strip().splitlines()
print("gpu: %s" % (smi[0] if smi else torch.cuda.get_device_name()))

cfg = ModelConfig(dataset="yelp", dropout=0.1)
torch.manual_seed(0)
model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg, label_smoothing=0.1).cuda().train()
batch = make_batch(cfg, B, seed=1234, fixed_len=100, n_valid_imgs=10).with_length_hint().to("cuda")
opt = [None]


def step():
    loss = model(batch.reviews, batch.reviews_mask, batch.reviews_rating, batch.field, batch.field_value, batch.img,
                 batch.img_mask, max_review_len=batch.max_review_len)[0]
    model.zero_grad(set_to_none=True)
    loss.backward()
    if opt[0] is not None:
        opt[0].step(lr=1e-5)


step()
eng = model.engine
opt[0] = get_optimizer(eng, 1e-5, ["bias", "LayerNorm.weight"], list(model.named_parameters()), None, max_grad_norm=1.0)
ARMS = (("off", False), ("on", True))
for _, on in ARMS:
    torch.use_deterministic_algorithms(on)
    for _ in range(WARM):
        step()
torch.cuda.synchronize()

times = {name: [] for name, _ in ARMS}
for _ in range(REPS):
    for name, on in ARMS:
        torch.use_deterministic_algorithms(on)
        step()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s.record()
        for _ in range(STEPS):
            step()
        e.record()
        torch.cuda.synchronize()
        times[name].append(s.elapsed_time(e) / STEPS)
for name, t in times.items():
    ts = sorted(t)
    print("deterministic %-3s  ms/step median %.2f  (min %.2f, max %.2f; %d rounds of %d steps)" % (name, ts[len(ts) // 2], ts[0], ts[-1],
                                                                                                     len(ts), STEPS))
off, on = sorted(times["off"])[REPS // 2], sorted(times["on"])[REPS // 2]
print("overhead of the ordered reductions: %+.2f ms/step (%+.1f %%)" % (on - off, 100.0 * (on - off) / off))


class Timer:
    def __init__(self):
        self.events = []

    def __call__(self, kind, work):
        import contextlib

        @contextlib.contextmanager
        def cm():
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            yield
            e.record()
            self.events.append((kind, s, e))
        return cm()


split = {}
side, eng.side_stream = eng.side_stream, None
for name, on in ARMS:
    torch.use_deterministic_algorithms(on)
    step()
    t = Timer()
    ops.KERNEL_TIMER = t
    for _ in range(2):
        step()
    ops.KERNEL_TIMER = None
    torch.cuda.synchronize()
    agg = {}
    for kind, s, e in t.events:
        a = agg.setdefault(kind, [0, 0.0])
        a[0] += 1
        a[1] += s.elapsed_time(e) / 2
    split[name] = agg
eng.side_stream = side
torch.use_deterministic_algorithms(False)
kinds = sorted(set(split["off"]) | set(split["on"]), key=lambda k: -max(split["off"].get(k, [0, 0])[1], split["on"].get(k, [0, 0])[1]))
print("%-22s %18s %18s" % ("C-ABI call (timed)", "off: calls  ms", "on: calls  ms"))
for k in kinds:
    o, n = split["off"].get(k, [0, 0.0]), split["on"].get(k, [0, 0.0])
    print("%-22s %8d %9.3f %8d %9.3f" % (k, o[0] / 2, o[1], n[0] / 2, n[1]))
print("(per step; 'gemm_ordered' = split-K weight gradients with more than one split, partial store + ordered reduce; "
      "embed_ln_bwd is not timed on the atomic path)")


# ---- the embedding backward alone, by token-id distribution
rows, S, V, D = 16 * 9 * 128, 128, cfg.vocab_size, 1024
g = torch.Generator(device="cuda").manual_seed(0)
f = lambda *sh: torch.randn(*sh, device="cuda", generator=g)
E, P, remb, gamma = f(V, D) * 0.1, f(S + 2, D) * 0.1, f(D) * 0.1, torch.rand(D, device="cuda", generator=g) + 0.5
rd, mean, rstd = f(rows // S), torch.zeros(rows, device="cuda"), torch.ones(rows, device="cuda")
dout = f(rows, D).to(torch.bfloat16)
dE, dP, dr, dg, db, dz = (torch.zeros(V, D, device="cuda"), torch.zeros(S + 2, D, device="cuda"), torch.zeros(D, device="cuda"),
                          torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda"), torch.empty(rows, D, device="cuda"))
ws = torch.empty(ops.embed_ln_bwd_workspace(rows, S, V), device="cuda")
rank = torch.arange(1, V + 1, device="cuda", dtype=torch.float64)
zipf = torch.multinomial((rank ** -1.1).float(), rows, replacement=True, generator=g).to(torch.int32) + 2
dists = {"uniform": torch.randint(2, V, (rows,), device="cuda", generator=g, dtype=torch.int32), "zipf s=1.1": zipf.clamp(max=V - 1),
         "one id": torch.full((rows,), 7, device="cuda", dtype=torch.int32)}
for name, ids in dists.items():
    biggest = torch.bincount(ids.long()).max().item()
    res = []
    for w in (None, ws):
        for i in range(25):
            if i == 5:
                s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s_.record()
            ops.embed_ln_bwd(dout, None, ids, E, P, rd, remb, gamma, mean, rstd, dE, dP, dr, dg, db, dz, rows, S, 1, 0.1, 3, 9,
                             workspace=w)
        e_.record()
        torch.cuda.synchronize()
        res.append(s_.elapsed_time(e_) / 20 * 1e3)
    print("embed_ln_bwd %-11s (largest group %5d rows): atomic %7.1f us, ordered %7.1f us" % (name, biggest, res[0], res[1]))
