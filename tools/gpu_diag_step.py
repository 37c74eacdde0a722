"""Diagnostic: per-tensor gradient errors of the CUDA step vs the fp32 oracle on the GPU for one golden case."""
import sys
import torch
sys.path.insert(0, "."); sys.path.insert(0, "tests")
from golden_util import load_golden
from test_step_gpu import _run_cuda_step
from oracle import mmsum_oracle as OR
name = sys.argv[1] if len(sys.argv) > 1 else "small_yelp"
gold = load_golden(name)
torch.backends.cuda.matmul.allow_tf32 = False
lo, og, _ = OR.step_loss_and_grads(gold["sd"], gold["cfg"], gold["batch"], gold["label_smoothing"], dtype=torch.float32, device="cuda")
loss, grads, model = _run_cuda_step(gold)
print("loss cuda %.6f oracle %.6f golden %.6f" % (loss, lo.item(), gold["loss"]))
eng = model.engine
w = eng.ws
for k in ("loss_rows",):
    t = w[k]
    print(k, "nan:", torch.isnan(t).sum().item(), "of", t.numel())
def nanrep(tag, t):
    n = torch.isnan(t.float()).sum().item()
    if n: print("  NaN in", tag, n, "/", t.numel())
nanrep("MEM", w["MEM"]); nanrep("logits", w["logits"][:, :gold["cfg"].vocab_size]); nanrep("x_out", w["x_out"])
for l, a in enumerate(w["enc"]):
    for k, t in a.items():
        if isinstance(t, torch.Tensor): nanrep("enc%d.%s" % (l, k), t)
for l, a in enumerate(w["dec"]):
    for k, t in a.items():
        if isinstance(t, torch.Tensor): nanrep("dec%d.%s" % (l, k), t)
for k in ("delta", "dMEM16", "dA3", "dO3", "dqkv", "dkv", "dz32", "dH"):
    if k in w: nanrep("bwd." + k, w[k])
nbad = [n for n in gold["names"] if not torch.isfinite(grads[n]).all()]
print("non-finite grads:", len(nbad), "of", len(gold["names"]), nbad[:6])
if len(sys.argv) > 2:
    sys.exit(0)
rows = []
for n in gold["names"]:
    g, o = grads[n].double(), og[n].double().cuda()
    sc = max(o.norm().item(), 1e-30)
    rows.append(((g - o).norm().item() / sc, n, g.norm().item(), o.norm().item()))
rows.sort(reverse=True)
for r in rows[:40]:
    print("%.4f %s cuda=%.4g oracle=%.4g" % r)
