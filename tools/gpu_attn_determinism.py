"""Run-to-run determinism / stale-state check of the attention forward kernel.
(1) kernel level: the multi-entity cross-attention at small ragged shapes and the config-2 shape, the forward launched
    repeatedly with every SM's shared and tensor memory poisoned with NaN patterns in between; outputs must be finite and bitwise
    identical from launch to launch.
(2) step level: forward of the small graph-test configuration run twice on the same inputs; every workspace buffer is compared
    bitwise between the two runs (first difference = the non-deterministic kernel)."""
import ctypes as C
import sys

import torch

sys.path.insert(0, "."); sys.path.insert(0, "tests")
from multimodalsum_b200 import _lib, ops

D = 1024
dev = torch.device("cuda")
lib = _lib.lib()


def poison():
    rc = lib.mmsum_debug_poison(C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc


def cross_case(B, R, F_, n_img, ik, seed, nan_pad=False):
    torch.manual_seed(seed)
    S, H, hd = 128, 16, 64
    N, T = B * R, B * R * S
    Tm = T + B * F_ + B * n_img * ik
    Et = R + 1 + n_img
    qc = torch.randn(T, D, device=dev).to(torch.bfloat16)
    kv = torch.randn(Tm, 2 * D, device=dev).to(torch.bfloat16)
    lens = torch.randint(30, S + 1, (B, R), device=dev)
    tvalid = torch.arange(S, device=dev)[None, None, :] < lens[:, :, None]
    tabvalid = torch.rand(B, 1, F_, device=dev) > 0.3
    tabvalid[:, :, 0] = True
    imask = torch.rand(B, n_img, device=dev) > 0.3
    imask[0] = False
    ivalid = imask[:, :, None].expand(B, n_img, ik)
    mem_valid = torch.cat([tvalid.reshape(-1), tabvalid.reshape(-1), ivalid.reshape(-1)]).to(torch.uint8)
    ent_valid = torch.cat([tvalid.any(-1), tabvalid.any(-1), imask], dim=1).to(torch.uint8).contiguous()
    inv_n = torch.zeros(N, 3, device=dev)
    nt = (tvalid.any(-1).sum(1) - 1).clamp(min=1).float()
    ni = imask.sum(1).float()
    inv_n[:, 0] = (1.0 / nt).repeat_interleave(R)
    inv_n[:, 1] = 1.0
    inv_n[:, 2] = torch.where(ni > 0, 1.0 / ni.clamp(min=1), torch.zeros_like(ni)).repeat_interleave(R)
    A3 = torch.empty(3, T, D, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(N, H, Et, S, device=dev)
    mods = [(0, 0, R, S, 1, 0), (T, T * D, 1, F_, 0, R), (T + B * F_, 2 * T * D, n_img, ik, 0, R + 1)]
    kw = dict(Q=qc, ldq=D, q_col=0, KV=kv, ldkv=2 * D, k_col=0, v_col=D, O=A3, ldo=D, LSE=lse, key_valid=mem_valid,
              ent_valid=ent_valid, inv_n=inv_n, n_qseq=N, H=H, R=R, causal=0, E_total=Et, scale=hd ** -0.5, mods=mods)
    return kw, A3, lse, (qc, kv, mem_valid, ent_valid, inv_n)


def kernel_level():
    for shape in [(2, 5, 47, 2, 196, 1), (3, 4, 47, 3, 196, 2), (16, 9, 47, 10, 196, 3)]:
        kw, A3, lse, keep = cross_case(*shape)
        a = ops.attn_args(**kw)
        outs = []
        for it in range(6):
            A3.fill_(float("nan")); lse.fill_(float("nan"))
            if it % 2:
                poison()
            ops.attn_fwd(a)
            torch.cuda.synchronize()
            outs.append((A3.clone(), lse.clone()))
        fin = all(torch.isfinite(o.float()).all().item() for o, _ in outs)
        same = all(torch.equal(outs[0][0], o) and torch.equal(outs[0][1].nan_to_num(7.0, 7.0, 7.0), l.nan_to_num(7.0, 7.0, 7.0))
                   for o, l in outs)
        print("shape", shape, "finite", fin, "bitwise-reproducible", same, flush=True)


def step_level():
    from golden_util import load_golden
    from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
    from multimodalsum_b200.synth import make_batch
    gold = load_golden("small_yelp")
    cfg = gold["cfg"]
    cfg.dropout = 0.0
    torch.manual_seed(0)
    model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg, label_smoothing=0.1)
    model.load_state_dict(gold["sd"], strict=False)
    model = model.cuda().train()
    b = make_batch(cfg, 2, seed=50, n_reviews=4, max_imgs=2).to("cuda")

    def snap(w, pre=""):
        out = {}
        for k, t in w.items():
            if isinstance(t, torch.Tensor):
                out[pre + k] = t.clone()
            elif isinstance(t, list):
                for i, d in enumerate(t):
                    if isinstance(d, dict):
                        out.update(snap(d, "%s%s%d." % (pre, k, i)))
        return out

    runs = []
    for it in range(4):
        if it % 2:
            poison()
        loss = model(b.reviews, b.reviews_mask, b.reviews_rating, b.field, b.field_value, b.img, b.img_mask)[0]
        model.zero_grad(set_to_none=True)
        loss.backward()
        torch.cuda.synchronize()
        g = {"grad." + n: p.grad.detach().clone() for n, p in model.named_parameters()}
        s = snap(model.engine.ws)
        s.update(g)
        runs.append((loss.item(), s))
    print("losses", [r[0] for r in runs], flush=True)
    base = runs[0][1]
    for it in range(1, 4):
        diff = [k for k, t in base.items()
                if not torch.equal(t.view(torch.uint8) if t.dtype != torch.bool else t, runs[it][1][k].view(torch.uint8) if t.dtype != torch.bool else runs[it][1][k])]
        nf = [k for k, t in runs[it][1].items() if t.is_floating_point() and k.startswith("grad.") and not torch.isfinite(t).all()]
        print("  run", it, "buffers differing from run 0:", len(diff), diff[:30], "non-finite grads:", len(nf), flush=True)


def first_nonfinite(with_poison):
    """Wraps the op layer: after every backward op, checks its outputs; prints the first op that produces a non-finite value."""
    from golden_util import load_golden
    from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
    from multimodalsum_b200.synth import make_batch
    gold = load_golden("small_yelp")
    cfg = gold["cfg"]
    cfg.dropout = 0.0
    torch.manual_seed(0)
    model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg, label_smoothing=0.1)
    model.load_state_dict(gold["sd"], strict=False)
    model = model.cuda().train()
    b = make_batch(cfg, 2, seed=50, n_reviews=4, max_imgs=2).to("cuda")
    print("img_mask", b.img_mask.tolist(), "reviews_mask valid per review", b.reviews_mask.sum(-1).tolist(), flush=True)
    state = dict(on=False, n=0, found=False)
    stash = {}
    orig = {k: getattr(ops, k) for k in ("gemm", "attn_bwd", "add_ln_bwd", "gate_bwd_u", "gate_bwd_o", "attn_args", "colsum",
                                           "embed_ln_bwd", "cast_bf16", "ce_fwd_bwd")}

    def bad(t):
        return not torch.isfinite(t.float()).all().item()

    def report(kind, what):
        if not state["found"]:
            state["found"] = True
            print("   FIRST non-finite: op #%d %s -> %s" % (state["n"], kind, what), flush=True)

    def wrap(kind, outs):
        f = orig[kind]

        def g(*a, **kw):
            r = f(*a, **kw)
            if state["on"] and not state["found"]:
                state["n"] += 1
                if with_poison:
                    pass
                torch.cuda.synchronize()
                for idx in outs:
                    t = a[idx] if isinstance(idx, int) else kw.get(idx)
                    if isinstance(t, torch.Tensor) and bad(t):
                        ins = [i for i, x in enumerate(a) if isinstance(x, torch.Tensor) and i not in outs and bad(x)]
                        report(kind, "arg %s shape %s (non-finite inputs: %s) kw=%s" % (idx, tuple(t.shape), ins,
                                                                                       {k: v for k, v in kw.items() if not isinstance(v, torch.Tensor)}))
            return r
        return g

    def attn_args(**kw):
        a = orig["attn_args"](**kw)
        stash[id(a)] = kw
        return a

    def attn_bwd(a):
        if state["on"] and with_poison:
            poison()
        r = orig["attn_bwd"](a)
        if state["on"] and not state["found"]:
            state["n"] += 1
            torch.cuda.synchronize()
            kw = stash[id(a)]
            for k in ("dQ", "dKV", "DELTA"):
                t = kw[k]
                if k == "DELTA":
                    continue
                if bad(t):
                    ins = [kk for kk in ("Q", "KV", "O") if bad(kw[kk])]
                    lse = kw["LSE"]
                    report("attn_bwd", "%s shape %s n_mod=%d (non-finite inputs: %s; LSE nan %d +inf %d -inf %d)" %
                           (k, tuple(t.shape), len(kw["mods"]), ins, torch.isnan(lse).sum().item(), (lse == float("inf")).sum().item(),
                            (lse == float("-inf")).sum().item()))
                    if k == "dQ":
                        rows = (~torch.isfinite(t.float())).any(-1).nonzero().flatten()
                        print("      bad dQ rows:", rows[:20].tolist(), "of", t.shape[0], "cols", (~torch.isfinite(t.float())).any(0).nonzero().flatten()[:8].tolist())
                    else:
                        rows = (~torch.isfinite(t.float())).any(-1).nonzero().flatten()
                        print("      bad dKV rows:", rows[:40].tolist(), "n", rows.numel(), "of", t.shape[0], "cols", (~torch.isfinite(t.float())).any(0).nonzero().flatten()[:8].tolist())
        return r

    ops.gemm = wrap("gemm", [2])
    ops.add_ln_bwd = wrap("add_ln_bwd", [7, 8])
    ops.gate_bwd_u = wrap("gate_bwd_u", [3])
    ops.gate_bwd_o = wrap("gate_bwd_o", [4])
    ops.attn_args = attn_args
    ops.attn_bwd = attn_bwd
    try:
        for it in range(2):
            loss = model(b.reviews, b.reviews_mask, b.reviews_rating, b.field, b.field_value, b.img, b.img_mask)[0]
            model.zero_grad(set_to_none=True)
            state.update(on=True, n=0, found=False)
            loss.backward()
            torch.cuda.synchronize()
            state["on"] = False
            nf = [n for n, p in model.named_parameters() if not torch.isfinite(p.grad).all()]
            print("poison", with_poison, "run", it, "loss", loss.item(), "non-finite grads", len(nf), nf[:4], flush=True)
    finally:
        for k, f in orig.items():
            setattr(ops, k, f)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "nan":
        first_nonfinite(False)
        first_nonfinite(True)
        sys.exit(0)
    kernel_level()
    step_level()
