"""Sampling vs beam search at the BASELINE config-5 shape: 64 businesses, 8 reviews x 158 tokens + 47 table fields + 10 images,
BART-large (12 + 12 layers) random init, max_length 128 (EOS banned until then, so every call decodes 127 tokens).

  * ms per decoded token of generate(do_sample=True, top_p=0.9, num_return_sequences=4) (top_k 50, the default) against
    beam-4, alternating in one process, memory encoded once (generate_from_memory);
  * the stand-alone sampler kernel (mmsum_sample_token) on [256, 50265] fp32 logits: CUDA events around each of >= 100
    launches, L2 overwritten (a 256 MB write) before every launch.
Prints the GPU name and power limit with the numbers."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from multimodalsum_b200 import ops
from multimodalsum_b200.generation import Generator
from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
from multimodalsum_b200.synth import ModelConfig, make_batch

B, L, REPS = 64, 128, 3
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                     text=True).stdout.strip().splitlines()
print("gpu: %s" % (smi[0] if smi else torch.cuda.get_device_name()))

cfg = ModelConfig(dataset="yelp", dropout=0.0)
torch.manual_seed(0)
model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg).cuda().eval()
batch = make_batch(cfg, B, seed=5, n_reviews=8, seq_len=158, fixed_len=150, n_valid_imgs=10).to("cuda")
gen = Generator(model)
mem = gen.encode_memory(batch.reviews, batch.reviews_mask, batch.field, batch.field_value, batch.img, batch.img_mask)
arms = {
    "beam-4": dict(num_beams=4, max_length=L, min_length=L, no_repeat_ngram_size=3, early_stopping=True),
    "sample top_p=0.9 n=4": dict(num_beams=1, do_sample=True, top_p=0.9, num_return_sequences=4, max_length=L, min_length=L,
                                 no_repeat_ngram_size=3),
}


def run(kw):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    out = gen.generate_from_memory(mem, **kw)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / gen.last_decode_steps, tuple(out.shape)


for kw in arms.values():                     # plan, capture, warm-up
    run(kw)
res = {k: [] for k in arms}
for _ in range(REPS):
    for name, kw in arms.items():
        res[name].append(run(kw))
for name, r in res.items():
    print("%-22s ms/token %s  (output %s)" % (name, " ".join("%.3f" % t for t, _ in r), r[-1][1]))

# ---- the sampler kernel alone
V, rows = cfg.vocab_size, 256
logits = (torch.randn(rows, (V + 3) // 4 * 4, device="cuda") * 3)[:, :V]          # 16-byte row pitch
ids = torch.full((rows, L), 1, dtype=torch.long, device="cuda")
ids[:, 0] = 2
cur = torch.tensor([20], dtype=torch.long, device="cuda")
ids[:, 1:20] = torch.randint(3, 1000, (rows, 19), device="cuda")
seed = torch.tensor([1], dtype=torch.long, device="cuda")
unf = torch.ones(rows, dtype=torch.uint8, device="cuda")
flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
for label, kw in (("top_k=50 top_p=0.9", dict(top_k=50, top_p=0.9)), ("top_k=0 top_p=0.9", dict(top_k=0, top_p=0.9)),
                  ("top_k=50", dict(top_k=50, top_p=1.0))):
    times = []
    for i in range(110):
        flush.fill_(float(i))
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ops.sample_token(logits, V, ids, cur, seed, 0, 3, 2, 1, 1.0, kw["top_k"], kw["top_p"], 1.0, unf)
        e.record()
        torch.cuda.synchronize()
        if i >= 10:
            times.append(s.elapsed_time(e) * 1e3)
    times.sort()
    mb = rows * V * 4 / 1e6
    print("sample_token_kernel [%d, %d] %-20s median %.1f us (min %.1f, max %.1f) over %d launches, L2 overwritten before "
          "each; %.1f MB of logits -> %.0f GB/s" % (rows, V, label, times[len(times) // 2], times[0], times[-1], len(times), mb,
                                                     mb / 1e3 / (times[len(times) // 2] * 1e-6)))
