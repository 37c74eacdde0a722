#!/usr/bin/env python
"""bench.py — headline benchmark: MultimodalSum data-parallel training step, businesses/s (BASELINE.json).

  python bench.py [--gpus N] [--steps K] [--warmup W]            this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference [--steps K] [--warmup W]      the reference's CPU implementation of the same step on the
                                                                 host cores (the unmodified reference tree when it is present,
                                                                 else the oracle port), same metric / config
  python bench.py --workload amazon                              BASELINE configs[3] shape (133 table rows, 1 image, 70 tokens)
  python bench.py --workload generate                            BASELINE configs[4]: beam-4 generation, 64 businesses
  python bench.py --dump-outputs DIR                             also write what the last timed step computed to DIR/*.npy

Default workload = BASELINE.json configs[1]: one step = forward + backward (+ bucketed gradient all-reduce when N > 1)
+ fused clip/AdamW of `MultimodalSum.forward` over 16 synthetic Yelp-shaped businesses per GPU (9 reviews x 128-token frame
with 100 valid tokens, 47 table fields, 10 images x 196 pooled ResNet features, BART-large, bf16 compute, dropout 0.1).
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how each field is obtained.
"""
import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TFLOP_PER_BUSINESS = {"yelp": 4.187, "amazon": 3.640}   # algorithmic fwd+bwd FLOPs per business, SURVEY.md §8(d) / App. C
METRIC = "train businesses/sec (BART-large, Yelp shape)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=["yelp", "amazon", "generate"],
                    help="yelp = BASELINE configs[1-2] (headline, default); amazon = configs[3] shape; generate = configs[4]")
    ap.add_argument("--dataset", default=None, choices=["yelp", "amazon"], help="alias of --workload (round-1 flag)")
    ap.add_argument("--businesses", type=int, default=None, help="businesses per GPU (train: 16, generate: 64)")
    ap.add_argument("--max-length", type=int, default=128, help="generate: decoder frame (src/test.py --max_length)")
    ap.add_argument("--graph", action="store_true", help="train workloads: replay forward / backward from recorded CUDA graphs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the Amazon / generation workloads appended to the default run")
    ap.add_argument("--cpu-seconds", type=float, default=240.0, help="time budget of the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy: training workloads "
                         "loss, grads and params (fixed per-tensor samples, see sampled_parameters); generate generated_ids")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs records the CUDA path (--impl b200)")
    a.workload = a.workload or a.dataset or "yelp"
    if a.businesses is None:
        a.businesses = 64 if a.workload == "generate" else 16
    return a


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"], source="measured")
    except Exception:
        return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


def load_traffic():
    """DRAM bytes per launch from the committed ncu capture (profiles/r02_traffic.json, written by tools/ncu_traffic.py)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm / cpu baseline
def cpu_reference_steps(steps, warmup, budget_s, dataset="yelp"):
    """Time the reference's CPU implementation of the step (MultimodalSum.forward + backward as written: 9-pass loop, fp32,
    dropout 0.1, no optimizer — BASELINE.md §3) on the host cores.  One step = ONE business.  Runs the UNMODIFIED reference
    through oracle/ref_harness.py when its tree is present (kind 'reference'), else the oracle port (kind 'port')."""
    import torch
    from multimodalsum_b200.synth import ModelConfig, make_batch, make_state_dict
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = ModelConfig(dataset=dataset, dropout=0.1)
    sd = make_state_dict(cfg, seed=0, perturb=False)
    amazon = dataset == "amazon"
    batch = make_batch(cfg, 1, seed=1, fixed_len=70 if amazon else 100, n_valid_imgs=1 if amazon else 10)
    kind, run = "port", None
    from oracle import ref_harness as RH
    if RH.available():
        try:
            model = RH.build_reference_model(cfg, sd, dtype=torch.float32, label_smoothing=0.1, dropout=0.1)

            def run():
                loss = model(batch.reviews, batch.reviews_mask, batch.reviews_rating, batch.field, batch.field_value, batch.img, batch.img_mask)[0]
                model.zero_grad()
                loss.backward()
            kind = "reference"
        except Exception as e:                                  # noqa: BLE001 — fall back to the port, say why
            sys.stderr.write("reference tree at %s unusable (%s); timing the oracle port\n" % (RH.REF_ROOT, e))
            run = None
    if run is None:
        from oracle import mmsum_oracle as OR

        def run():
            OR.step_loss_and_grads(sd, cfg, batch, 0.1, dtype=torch.float32, device="cpu", training=True)
    times = []
    t_start = time.time()
    n_done = 0
    dt = 0.0
    for i in range(warmup + steps):
        t0 = time.time()
        run()
        dt = time.time() - t0
        if i >= warmup:
            times.append(dt)
        n_done += 1
        elapsed = time.time() - t_start
        if i < warmup and elapsed + dt * (warmup - i - 1 + steps) > budget_s:
            warmup = i + 1                      # cut warm-up short to keep the run within the budget
        if times and elapsed + dt > budget_s:
            break
    if not times:
        times = [dt]
    med = statistics.median(times)
    shape = "9x128-token reviews, 133 table rows, 1x196 image keys" if amazon else "9x128-token reviews, 47 table fields, 10x196 image keys"
    return dict(value=1.0 / med, ms_per_step=1000.0 * med, steps=len(times), warmup=min(warmup, n_done - len(times)), cores=cores, kind=kind,
                sample="1 business per step (B=1, full %s shape: %s), %s fwd+bwd, fp32, dropout 0.1, %d warm-up + %d timed step(s), median"
                       % (dataset, shape, "unmodified reference" if kind == "reference" else "oracle port", min(warmup, n_done - len(times)), len(times)))


def train_config(args, world, cpu=None):
    amazon = args.workload == "amazon"
    cfg = {"workload": ("BASELINE configs[3] shape: Amazon-shape multimodal_train step" if amazon else
                        "BASELINE configs[1]: Yelp-shape multimodal_train step") + ", BART-large random init",
           "businesses_per_gpu": args.businesses, "reviews": 9, "frame": 128, "valid_tokens": 70 if amazon else 100,
           "encoder_frame": "encoder rows trimmed to ceil16(longest review) = %d per review (pad rows are masked and carry zero gradient: results unchanged)" % (80 if amazon else 112),
           "table_fields": 133 if amazon else 47, "images": "1x196" if amazon else "10x196", "dropout": 0.1, "label_smoothing": 0.1}
    return cfg


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "generate":
        print(json.dumps({"impl": "reference", "unavailable": "the reference arm times the training step (BASELINE metric); "
                          "the reference's CPU generate at 64 businesses x beam 4 does not fit a bounded run (BASELINE.md §2: 2.1 s/step for 8 hypotheses)"}), flush=True)
        return
    r = cpu_reference_steps(args.steps, args.warmup, args.cpu_seconds, args.workload)
    cfg = train_config(args, 1)
    cfg.update({"parallelism": "cpu x%d threads" % r["cores"],
                "sample": "1 business per timed step (the reference's per-business cost is independent of the batch)",
                "step": "fwd + bwd of the reference step on the host cores (the b200 arm additionally runs the fused clip/AdamW)"})
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "businesses/s", "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": r["value"], "unit": "businesses/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "businesses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ helpers of the GPU arms
def _dist_env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local_rank


def _build_record():
    """Which library ran: the record build() wrote next to libmmsum_b200.so and whether it matches the sources of this tree."""
    from multimodalsum_b200 import _lib
    b = _lib.build_info()
    return {"library": os.path.relpath(b["path"], ROOT), "nvcc": b.get("nvcc"), "arch": b.get("arch"),
            "source_digest": (b.get("source_digest") or "")[:16], "matches_sources": b["matches_sources"]}


DUMP_PER_TENSOR = 4096          # entries kept per parameter tensor: 566 BART-large tensors -> < 10 MB per array
DUMP_LIMIT_BYTES = 64 << 20
# The training step is not bitwise reproducible: the embedding / LayerNorm / column-sum gradient kernels
# (multimodalsum_b200/csrc/rowwise.cu) accumulate with float atomicAdd, so the summation order varies between runs and the
# difference carries through AdamW into later steps.  Two runs of the same build (default workload, --steps 10 --warmup 3,
# one B200 at its 1000 W power limit) differed by 1.4e-2 in the relative L2 norm of grads.npy, 3e-7 in params.npy and 2e-6
# in loss.npy.  params.npy and loss.npy are therefore the sharp comparisons between two builds; grads.npy only shows
# differences well above that 1e-2 spread.


def sampled_parameters(model):
    """{"grads": ..., "params": ...}: for every parameter in `model.named_parameters()` order, its gradient and its (updated)
    value at the same fixed entries — all of them for tensors of at most DUMP_PER_TENSOR entries, else DUMP_PER_TENSOR sorted
    distinct flat indices drawn from a generator seeded with crc32(name), so a tensor's sample depends on its name and size
    only — concatenated into one float32 array each."""
    import zlib

    import numpy as np
    import torch
    grads, params = [], []
    for name, p in model.named_parameters():
        g, w = p.grad.detach().reshape(-1), p.detach().reshape(-1)
        if w.numel() > DUMP_PER_TENSOR:
            idx = np.sort(np.random.default_rng(zlib.crc32(name.encode())).choice(w.numel(), DUMP_PER_TENSOR, replace=False))
            idx = torch.from_numpy(idx).to(w.device)
            g, w = g[idx], w[idx]
        grads.append(g.float().cpu())
        params.append(w.float().cpu())
    return {"grads": torch.cat(grads).numpy(), "params": torch.cat(params).numpy()}


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy in float32 / float64 (at most DUMP_LIMIT_BYTES in all)."""
    import numpy as np
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError("outputs to dump take %d bytes, more than %d" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


class KernelTimer:
    """ops.KERNEL_TIMER hook: brackets every C-ABI call of the instrumented steps with CUDA events on the launching stream."""

    def __init__(self, torch):
        self.torch = torch
        self.events = []

    @contextlib.contextmanager
    def __call__(self, kind, work):
        s, e = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        s.record()
        yield
        e.record()
        self.events.append((kind, work, s, e))

    def summary(self):
        agg = {}
        for kind, work, s, e in self.events:
            a = agg.setdefault(kind, [0, 0.0, 0.0])
            a[0] += 1
            a[1] += work
            a[2] += s.elapsed_time(e)
        return agg


TENSOR_KINDS = ("gemm", "attn_cross_fwd", "attn_cross_bwd", "attn_self_fwd", "attn_self_bwd")
KERNEL_OF = {"gemm": "gemm_tcgen05_kernel", "attn_cross_fwd": "attn_fwd_tc3_kernel (multi-entity cross-attention)",
             "attn_cross_bwd": "attn_bwd_dq_tc_kernel + attn_bwd_dkv_tc_kernel (cross)", "attn_self_fwd": "attn_fwd_tc3_kernel (self)",
             "attn_self_bwd": "attn_bwd_dq_tc_kernel + attn_bwd_dkv_tc_kernel (self)", "add_ln_fwd": "add_ln_fwd_kernel",
             "add_ln_bwd": "add_ln_bwd_kernel", "embed_ln_fwd": "embed_ln_fwd_kernel", "ce_fwd": "ce_fwd_bwd_kernel (loss pass)",
             "ce_bwd": "ce_fwd_bwd_kernel (gradient pass)", "colsum": "colsum_kernel", "gate": "gate_fwd/bwd kernels"}


def roofline_kernels(agg, n_steps, peaks, step_ms, traffic):
    out = {}
    for kind, (n, work, ms) in sorted(agg.items()):
        if ms <= 0:
            continue
        tensor = kind in TENSOR_KINDS
        achieved = work / (ms / 1e3) / (1e12 if tensor else 1e9)
        peak = peaks["tf_sustained"] if tensor else peaks["hbm_gbs"]
        ent = {"kernel": KERNEL_OF.get(kind, kind), "bound": "tensor" if tensor else "hbm", "launches_per_step": n / n_steps,
               "avg_us": 1e3 * ms / n, "achieved": achieved, "peak": peak, "unit": "TFLOP/s" if tensor else "GB/s",
               "frac": achieved / peak, "share_of_step": ms / n_steps / step_ms}
        if kind in traffic:
            ent["traffic"] = traffic[kind]
        out[kind] = ent
    return out


# ------------------------------------------------------------------------------------------------ training workloads
def run_train(args):
    import torch
    import torch.distributed as dist
    from multimodalsum_b200 import ops
    from multimodalsum_b200.dp import GradAllReducer
    from multimodalsum_b200.modules import AmazonTableEncoder, MultimodalSum, YelpTableEncoder
    from multimodalsum_b200.optim import get_optimizer
    from multimodalsum_b200.synth import ModelConfig, make_batch

    world, rank, local_rank = _dist_env()
    dev = torch.device("cuda", local_rank)
    B = args.businesses
    amazon = args.workload == "amazon"
    cfg = ModelConfig(dataset=args.workload, dropout=0.1)
    torch.manual_seed(0)                                   # identical random-init bart-large weights on every rank
    model = MultimodalSum(TableEncoder=AmazonTableEncoder if amazon else YelpTableEncoder, config=cfg, label_smoothing=0.1).to(dev).train()
    # distinct synthetic shards per rank (businesses are independent units: weak scaling, no data-path collective)
    n_host_batches = 2
    host = [make_batch(cfg, B, seed=1234 + rank * 17 + i, fixed_len=70 if amazon else 100, n_valid_imgs=1 if amazon else 10).with_length_hint().pin()
            for i in range(n_host_batches)]
    resident = host[0].to(dev)

    opt = [None]

    def step(batch):
        # src/multimodal_train.py:357-364: forward, zero_grad, backward (+ bucketed all-reduce), clip, AdamW, schedule
        loss = model(batch.reviews, batch.reviews_mask, batch.reviews_rating, batch.field, batch.field_value, batch.img, batch.img_mask,
                     max_review_len=batch.max_review_len)[0]       # the collate-time length hint (host metadata, no device read-back)
        model.zero_grad(set_to_none=True)
        loss.backward()
        if opt[0] is not None:
            opt[0].step(lr=1e-5)
        return loss

    if args.graph and world == 1:
        model.enable_cuda_graph()
    step(resident)                                          # builds the engine, arenas and workspaces
    eng = model.engine
    reducer = GradAllReducer(eng) if world > 1 else None    # noqa: F841 (hooks the engine)
    # all parameters in a group (a list, not the reference's exhausted generator: every tensor is updated here)
    opt[0] = get_optimizer(eng, 1e-5, ["bias", "LayerNorm.weight"], list(model.named_parameters()), None, max_grad_norm=1.0)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()
        return ms

    # ---------------- device-resident timing (value): nothing but the step inside the timed region
    W = max(args.warmup, 3)
    for _ in range(W):
        step(resident)
    barrier()
    launches0 = ops.LAUNCHES
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start.record()
    for _ in range(args.steps):
        loss = step(resident)
    t_end.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = ops.LAUNCHES - launches0
    ms = max_over_ranks(t_start.elapsed_time(t_end))
    ms_per_step = ms / args.steps
    value = B * world / (ms_per_step / 1000.0)
    if args.dump_outputs and rank == 0:
        # what the caller holds after the last timed step: its loss, every .grad and the parameters AdamW updated
        dump_outputs(args.dump_outputs, dict(loss=loss.detach().double().reshape(1).cpu().numpy(), **sampled_parameters(model)))

    # ---------------- instrumented steps (outside `value`): every C-ABI call bracketed with CUDA events
    n_inst = 2
    timer = KernelTimer(torch)
    barrier()
    ops.KERNEL_TIMER = timer
    side, eng.side_stream = eng.side_stream, None      # bias-gradient column sums inline, so that their events time the kernel
    for _ in range(n_inst):
        step(resident)
    eng.side_stream = side
    ops.KERNEL_TIMER = None
    barrier()
    agg = timer.summary()

    # ---------------- end-to-end timing through the public API with HOST (pinned) inputs
    # The timed region is one "epoch" of the reference's train() (src/multimodal_train.py:344-379) over K host batches, written as
    # the reference writes it: construct the dataset's prefetcher on the loader, `next()`, and loop until it returns None.  The
    # prefetcher is this repo's public input pipeline (multimodalsum_b200/prefetch.py: resident staging slots filled on a copy
    # stream, so there is no device allocation churn inside the loop — with freshly allocated tensors + record_stream, the caching
    # allocator's occasional cudaMalloc showed up as 5-10 % dips of this number in one run out of three).  All K host -> device
    # copies (batch 0's included: the prefetcher is constructed after the start event) and the loss read-backs are inside.
    from multimodalsum_b200.prefetch import amazon_data_prefetcher, yelp_data_prefetcher
    Prefetcher = amazon_data_prefetcher if amazon else yelp_data_prefetcher
    field = resident.field                                  # src/multimodal_train.py:469-470: `field` is moved to the GPU once

    def loader(n):
        for i in range(n):
            h = host[i % n_host_batches]
            yield (h.reviews, h.reviews_mask, h.reviews_rating, *h.field_value, h.img, h.img_mask)

    def epoch(n, on_loss):
        prefetcher = Prefetcher(loader(n), device=dev)
        reviews, reviews_mask, reviews_rating, field_value, img, img_mask = prefetcher.next()
        while reviews is not None:
            loss = model(reviews, reviews_mask, reviews_rating, field, field_value, img, img_mask)[0]   # length hint rides on reviews_mask
            model.zero_grad(set_to_none=True)
            loss.backward()
            opt[0].step(lr=1e-5)
            on_loss(loss)
            reviews, reviews_mask, reviews_rating, field_value, img, img_mask = prefetcher.next()
        return prefetcher

    epoch(max(3, args.warmup), lambda loss: loss.item())
    barrier()
    loss_host = torch.empty(1, pin_memory=True)
    e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_start.record()
    pf = epoch(args.steps, lambda loss: loss_host.copy_(loss.detach().reshape(1), non_blocking=True))   # device -> host read of the result
    e_end.record()
    barrier()
    assert pf.n_served == args.steps
    h2d_bytes = pf.h2d_bytes // args.steps                  # counted from the tensors the prefetcher copied
    e2e_ms = max_over_ranks(e_start.elapsed_time(e_end))
    e2e_value = B * world / (e2e_ms / args.steps / 1000.0)
    final_loss = float(loss_host.item())

    if rank != 0:
        return None
    peaks = load_peaks()
    traffic = load_traffic()
    tfb = TFLOP_PER_BUSINESS[args.workload]
    rk = roofline_kernels(agg, n_inst, peaks, ms_per_step, traffic)
    gemm = rk.get("gemm", {})
    cfg_line = train_config(args, world)
    cfg_line.update({"step": "fwd + bwd%s + fused clip/AdamW" % (" + bucketed NCCL grad all-reduce overlapped with backward" if world > 1 else ""),
                     "parallelism": "dp%d" % world,
                     "cuda_graph": bool(args.graph and world == 1),
                     "l2_policy": "per-step working set (>25 GB activations + 2.8 GB weights) exceeds the 126 MB L2",
                     "final_loss": final_loss})
    tensor_ms = sum(agg[k][2] for k in TENSOR_KINDS if k in agg) / n_inst
    tensor_flops = sum(agg[k][1] for k in TENSOR_KINDS if k in agg) / n_inst
    line = {
        "metric": METRIC, "value": value, "unit": "businesses/s", "n_gpus": world, "steps": args.steps, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": cfg_line, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "businesses/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches,
        "tc_fraction_step": {"algorithmic_tflop_per_business": tfb,
                             "achieved_tflops_per_gpu": value / world * tfb,
                             "frac_of_sustained_peak": value / world * tfb / peaks["tf_sustained"],
                             "tensor_kernels": {"tflops": tensor_flops / (tensor_ms / 1e3) / 1e12 if tensor_ms > 0 else None,
                                                "frac_of_sustained_peak": tensor_flops / (tensor_ms / 1e3) / 1e12 / peaks["tf_sustained"] if tensor_ms > 0 else None,
                                                "share_of_step": tensor_ms / ms_per_step}},
        "roofline": {"kernel": "gemm_tcgen05_kernel (all %d GEMM launches of a step, timed in %d instrumented steps after the timed region)"
                               % (int(gemm.get("launches_per_step", 0)), n_inst),
                     "bound": "tensor", "achieved": gemm.get("achieved"), "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                     "frac": gemm.get("frac"),
                     # ncu dram__bytes_read.sum + dram__bytes_write.sum per launch (committed capture, profiles/r02_traffic.json)
                     "traffic": (traffic.get("gemm") or {}).get("dram_bytes_per_launch"), "traffic_detail": traffic.get("gemm"),
                     "peak_source": peaks["source"] + " (sustained bf16)", "gemm_share_of_step": gemm.get("share_of_step")},
        "roofline_kernels": rk,
        "build": _build_record(),
    }
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_steps(3, 1, 60.0, args.workload)
        line["cpu_baseline"] = {"value": r["value"], "unit": "businesses/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
    return line


# ------------------------------------------------------------------------------------------------ generation workload (config 5)
def run_generate(args):
    """BASELINE configs[4]: src/test.py-style beam-4 generation, 64 businesses per GPU, 8 reviews in 158-token frames + 47
    table fields + 10 x 196 image keys, max_length 128, no_repeat_ngram_size 3, early_stopping.  One step = one complete
    `generate` call (memory encoding, per-layer cross K|V projection, beam search).  Replicas only for N > 1 (no collective)."""
    import torch
    import torch.distributed as dist
    from multimodalsum_b200 import ops
    from multimodalsum_b200.generation import Generator
    from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
    from multimodalsum_b200.synth import ModelConfig, make_batch

    world, rank, local_rank = _dist_env()
    dev = torch.device("cuda", local_rank)
    B, beams, max_length = args.businesses, 4, args.max_length
    cfg = ModelConfig(dataset="yelp", dropout=0.0)
    torch.manual_seed(0)
    model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg).to(dev).eval()
    host = make_batch(cfg, B, seed=5 + rank, n_reviews=8, seq_len=158, fixed_len=150, n_valid_imgs=10).pin()
    resident = host.to(dev)
    gen = Generator(model)
    kw = dict(num_beams=beams, max_length=max_length, length_penalty=1.0, no_repeat_ngram_size=3, early_stopping=True)

    def run(b):
        return gen.generate(b.reviews, b.reviews_mask, b.field, b.field_value, b.img, b.img_mask, **kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()
        return ms

    W = max(args.warmup, 3)
    for _ in range(W):
        out = run(resident)
    barrier()
    launches0 = ops.LAUNCHES
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    s.record()
    for _ in range(args.steps):
        out = run(resident)
    e.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = ops.LAUNCHES - launches0
    ms_per_step = max_over_ranks(s.elapsed_time(e)) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"generated_ids": out.cpu().numpy().astype("float64")})
    tokens = max_length - 1                       # decode steps of a full frame (random-init weights never finish early)
    value = B * world * tokens / (ms_per_step / 1e3)
    # memory encoding alone (encoder + table + image heads + 12 cross K|V projections)
    s.record()
    for _ in range(3):
        st = gen.encode(resident.reviews, resident.reviews_mask, resident.field, resident.field_value, resident.img, resident.img_mask, beams)
    e.record()
    torch.cuda.synchronize()
    enc_ms = s.elapsed_time(e) / 3
    # decode-step-only timing: the incremental decoder alone, 16 consecutive positions
    st = gen.encode(resident.reviews, resident.reviews_mask, resident.field, resident.field_value, resident.img, resident.img_mask, beams)
    N = B * beams
    rd = torch.zeros(N, device=dev)
    ids = torch.randint(3, cfg.vocab_size, (N, 40), device=dev)
    perm = torch.arange(N, device=dev)
    for cur in range(1, 9):
        gen.step_logits(st, ids[:, :cur], rd); gen.reorder_cache(st, perm)
    torch.cuda.synchronize()
    s.record()
    for cur in range(9, 25):
        gen.step_logits(st, ids[:, :cur], rd); gen.reorder_cache(st, perm)
    e.record()
    torch.cuda.synchronize()
    dec_ms = s.elapsed_time(e) / 16
    # end to end: pinned host inputs -> device, generate, ids -> host
    out_host = torch.empty(B, max_length, dtype=torch.long).pin_memory()
    barrier()
    s.record()
    for _ in range(args.steps):
        b = host.to(dev, non_blocking=True)
        o = run(b)
        out_host[:, :o.shape[1]].copy_(o, non_blocking=True)
    e.record()
    barrier()
    e2e_ms = max_over_ranks(s.elapsed_time(e)) / args.steps
    if rank != 0:
        return None
    peaks = load_peaks()
    mem = st.mem
    D = cfg.d_model
    kv_bytes = mem.MEM.shape[0] * 2 * D * 2 * cfg.decoder_layers                 # every cross K|V row read once per step
    dec_w = sum(p.numel() for n, p in model.named_parameters() if ".decoder.layers." in n) * 2 + cfg.vocab_size * D * 2
    self_bytes = N * 24 * 2 * D * 2 * cfg.decoder_layers * 2                      # ~24 cached positions read + re-ordered
    step_bytes = kv_bytes + dec_w + self_bytes
    line = {
        "metric": "beam-4 generation, business x tokens / sec (src/test.py path, BASELINE configs[4])", "value": value,
        "unit": "business*tokens/s", "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "BASELINE configs[4]: beam-4 generation, %d businesses/GPU, 8 reviews x 158-token frames + 47 table fields + "
                               "10x196 image keys, max_length %d, no_repeat_ngram_size 3, early_stopping; BART-large random init; one step = "
                               "one generate() call (encode + cross K|V projection + %d decode steps)" % (B, max_length, tokens),
                   "businesses_per_gpu": B, "beams": beams, "parallelism": "replicas x%d" % world,
                   "l2_policy": "cross-attention K|V (%.1f GB) streamed every decode step exceeds the 126 MB L2" % (kv_bytes / 1e9),
                   "output_shape": list(out.shape)},
        "clocks": clocks,
        "e2e": {"value": B * world * tokens / (e2e_ms / 1e3), "unit": "business*tokens/s", "h2d_bytes_per_step": host.nbytes(),
                "d2h_bytes_per_step": int(out.numel() * 8), "ms_per_step": e2e_ms},
        "gpu_launches": launches,
        "roofline": {"kernel": "incremental decode step (all kernels of one token: 12 decoder layers + LM head)", "bound": "hbm",
                     "achieved": step_bytes / (dec_ms / 1e3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": step_bytes / (dec_ms / 1e3) / 1e9 / peaks["hbm_gbs"], "traffic": None,
                     "peak_source": peaks["source"], "decode_step_ms": dec_ms, "encode_ms": enc_ms,
                     "token_ms_incl_beam_update": (ms_per_step - enc_ms) / tokens,
                     "algorithmic_bytes_per_step": {"cross_kv": kv_bytes, "decoder_weights_and_lm_head": dec_w, "self_kv_cache": self_bytes}},
    }
    return line


def _free_gpu():
    import gc
    import torch
    gc.collect()
    torch.cuda.empty_cache()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import copy
    import torch
    import torch.distributed as dist
    world, rank, local_rank = _dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", init_method="env://", device_id=torch.device("cuda", local_rank))
    line = run_generate(args) if args.workload == "generate" else run_train(args)
    if args.workload == "yelp" and not args.no_secondary:
        # the other BASELINE configs, measured in the same run so that the driver's default invocation records them:
        # configs[3] (Amazon shape, every N) and configs[4] (beam-4 generation; replicas only, so N = 1)
        sec = {}
        _free_gpu()
        a2 = copy.copy(args)
        a2.workload, a2.businesses, a2.steps, a2.no_cpu_baseline = "amazon", 16, min(args.steps, 5), True
        a2.dump_outputs = None
        r = run_train(a2)
        if r is not None:
            sec["amazon_configs3"] = {k: r[k] for k in ("value", "unit", "ms_per_step", "n_gpus", "steps", "e2e", "config", "clocks", "tc_fraction_step")}
            sec["amazon_configs3"]["roofline_frac_gemm"] = r["roofline"]["frac"]
        if world == 1:
            _free_gpu()
            a3 = copy.copy(args)
            a3.workload, a3.businesses, a3.steps, a3.dump_outputs = "generate", 64, min(args.steps, 3), None
            r = run_generate(a3)
            if r is not None:
                sec["generate_configs4"] = {k: r[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "e2e", "config", "clocks", "roofline")}
        if line is not None:
            line["secondary"] = sec
    if line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
