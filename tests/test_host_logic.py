"""CPU-side checks: C-ABI library loads and exports every symbol the header declares; arena layout, module
state_dict keys and synthetic generators are consistent with the reference's parameter inventory (SURVEY App. B)."""
import os
import re

import pytest
import torch

from multimodalsum_b200 import _lib
from multimodalsum_b200.engine import ALIGN, StepEngine, _arena_order
from multimodalsum_b200.synth import ModelConfig, make_batch, make_state_dict, param_shapes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = dict(encoder_layers=2, decoder_layers=2, ffn_dim=256, vocab_size=512, max_position_embeddings=128)


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "mmsum_b200.h")).read()
    declared = sorted(set(re.findall(r"\bint\s+(mmsum_\w+)\s*\(", header)))
    assert declared, "no declarations found"
    lib = _lib.lib()           # raises if the .so is missing: there is no fallback
    for name in declared:
        assert hasattr(lib, name), "libmmsum_b200.so does not export %s" % name
    assert sorted(_lib.EXPORTS) == declared


def test_ops_refuse_cpu_tensors():
    from multimodalsum_b200 import ops
    a = torch.zeros(128, 64, dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        ops.gemm(a, a)


@pytest.mark.parametrize("dataset", ["yelp", "amazon", "text"])
def test_arena_order_covers_reference_parameters(dataset):
    cfg = ModelConfig(dataset=dataset, **SMALL)
    names = _arena_order(cfg)
    assert len(names) == len(set(names))
    shapes = param_shapes(cfg)
    aliases = ("encoder.embed_tokens.weight", "decoder.embed_tokens.weight", "table_encoder.bart_embedding.weight")
    expected = {n for n in shapes if not n.endswith(aliases) and not n.endswith("final_logits_bias")}
    assert set(names) == expected
    # fused groups must be adjacent in the arena (one GEMM serves q|k|v and k|v)
    idx = {n: i for i, n in enumerate(names)}
    for n in names:
        if n.endswith("self_attn.q_proj.weight"):
            b = n[:-len("q_proj.weight")]
            assert idx[b + "k_proj.weight"] == idx[n] + 1 and idx[b + "v_proj.weight"] == idx[n] + 2
            assert idx[b + "k_proj.bias"] == idx[b + "q_proj.bias"] + 1 and idx[b + "v_proj.bias"] == idx[b + "q_proj.bias"] + 2
        if n.endswith("encoder_attn.k_proj.weight"):
            b = n[:-len("k_proj.weight")]
            assert idx[b + "v_proj.weight"] == idx[n] + 1 and idx[b + "v_proj.bias"] == idx[b + "k_proj.bias"] + 1
    # shared embedding is last: its gradient is final only after the encoder's gather backward
    assert names[-1] == "bart_model.model.shared.weight"


@pytest.mark.parametrize("dataset", ["yelp", "amazon", "text"])
def test_module_state_dict_matches_reference_keys(dataset):
    from multimodalsum_b200.modules import AmazonTableEncoder, MultimodalSum, TextSupervised, YelpTableEncoder
    cfg = ModelConfig(dataset=dataset, **SMALL)
    if dataset == "text":
        m = TextSupervised(config=cfg)
    else:
        m = MultimodalSum(TableEncoder=YelpTableEncoder if dataset == "yelp" else AmazonTableEncoder, config=cfg)
    sd = m.state_dict()
    shapes = param_shapes(cfg)
    assert set(sd.keys()) == set(shapes.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(shapes[k]), k
    # aliasing contract: shared == encoder.embed_tokens == decoder.embed_tokens == table_encoder.bart_embedding
    shared = m.bart_model.model.shared.weight
    assert m.bart_model.model.encoder.embed_tokens.weight is shared
    assert m.bart_model.model.decoder.embed_tokens.weight is shared
    if dataset != "text":
        assert m.table_encoder.bart_embedding.weight is shared
    # loads the synthetic reference-keyed state_dict without missing / unexpected keys
    missing, unexpected = m.load_state_dict(make_state_dict(cfg, seed=0), strict=False)
    assert not missing and not unexpected
    # parameter names seen by the engine == arena order set
    assert {n for n, _ in m.named_parameters()} == set(_arena_order(cfg))
    # reference init recipe (:188-199): pad row of the shared embedding is zero
    m2 = MultimodalSum(config=ModelConfig(dataset="yelp", **SMALL)) if dataset == "yelp" else None
    if m2 is not None:
        assert m2.bart_model.model.shared.weight[1].abs().sum().item() == 0.0


def test_no_cpu_fallback():
    from multimodalsum_b200.modules import MultimodalSum
    cfg = ModelConfig(dataset="yelp", **SMALL)
    m = MultimodalSum(config=cfg)
    b = make_batch(cfg, 1, seed=0, n_reviews=3, max_imgs=1)
    with pytest.raises(RuntimeError):
        m(b.reviews, b.reviews_mask, b.reviews_rating, b.field, b.field_value, b.img, b.img_mask)


def test_synthetic_batch_shapes_and_invariants():
    cfg = ModelConfig(dataset="yelp")
    b = make_batch(cfg, 2, seed=3)
    assert b.reviews.shape == (2, 9, 128) and b.img.shape == (2, 10, 196, 1024) and b.field.shape == (47, 6)
    lens = b.reviews_mask.sum(-1)
    assert lens.min() >= 60 and lens.max() <= 100
    idx = (lens - 1).unsqueeze(-1)
    assert (b.reviews.gather(-1, idx) == 2).all()            # EOS closes every review
    assert (b.reviews[:, :, 0] != 0).all()                   # never BOS at position 0 (SURVEY §8d)
    assert ((b.reviews == 1) == (b.reviews_mask == 0)).all()
    b2 = make_batch(ModelConfig(dataset="amazon"), 2, seed=3)
    assert b2.img.shape == (2, 1, 196, 1024) and b2.field.shape == (6, 1) and b2.field_value[4].shape == (2, 3, 8, 12)


def test_encoder_frame_views_and_length_cache():
    """Host logic of the trimmed encoder frames (engine._encoder_frame / _alloc / _frame_view), on CPU tensors: the frame is
    the next multiple of 16 above the longest review (hint, read-back, cache keyed on the tensor's identity and version), the
    workspace is allocated once for full frames and a step works on views of the same storage, and the encoder-sized scratch
    pool hands out row-cut views of the shared buffers."""
    import torch
    from multimodalsum_b200.engine import StepEngine
    from multimodalsum_b200.synth import ModelConfig, make_batch
    cfg = ModelConfig(dataset="yelp", encoder_layers=1, decoder_layers=2, ffn_dim=64, vocab_size=512, max_position_embeddings=128)
    eng = StepEngine(cfg, device="cpu")
    b = make_batch(cfg, 2, seed=3, n_reviews=3, max_imgs=2, len_range=(20, 70))
    longest = int(b.reviews_mask.sum(-1).max())
    frame = (longest + 15) // 16 * 16
    assert eng._encoder_frame(b, 128) == frame                       # read back from the mask
    assert eng._len_cache[0]() is b.reviews_mask and eng._len_cache[2] == longest
    b.reviews_mask[0, 0, 100] = 1                                    # in-place change bumps the version: the cache must miss
    assert eng._encoder_frame(b, 128) == 112
    b.reviews_mask[0, 0, 100] = 0
    other = b.reviews_mask.clone()                                   # a different tensor object never hits the cache
    b2 = make_batch(cfg, 2, seed=3, n_reviews=3, max_imgs=2, len_range=(20, 70))
    b2.reviews_mask = other
    assert eng._encoder_frame(b2, 128) == frame
    assert b.with_length_hint().max_review_len == longest
    b.max_review_len = 17
    assert eng._encoder_frame(b, 128) == 32                          # the hint wins (a wrong one fails loudly on the device)
    b.max_review_len = 1
    assert eng._encoder_frame(b, 128) == 16
    eng.trim_frames = False
    assert eng._encoder_frame(b, 128) == 128
    eng.trim_frames = True

    B, R, S, F, n_img, ik = 2, 3, 128, 47, 2, 196
    w = eng._alloc(B, R, S, F, n_img, ik, 80)
    full = eng.ws_full
    assert (w["S_enc"], w["Te"], w["Tt"]) == (80, B * R * 80, B * R * 80)
    assert w["Tm"] == B * R * 80 + B * F + B * n_img * ik and w["T"] == B * R * S
    assert w["MEM"].shape[0] == w["Tm"] and w["MEM"].data_ptr() == full["MEM"].data_ptr()
    assert w["enc"][0]["qkv"].shape == (w["Te"], 3 * cfg.d_model) and w["enc"][0]["qkv"].data_ptr() == full["enc"][0]["qkv"].data_ptr()
    assert w["enc"][0]["lse"] is full["enc"][0]["lse"]
    assert w["dec"][0]["kv"].shape[0] == w["Tm"] and w["dec"][0]["x"] is full["dec"][0]["x"]
    assert w["dkv_all"].shape == (w["Tm"], cfg.decoder_layers * 2 * cfg.d_model)
    assert eng._alloc(B, R, S, F, n_img, ik, 80) is w                # cached view, nothing reallocated
    assert eng._alloc(B, R, S, F, n_img, ik, 128) is full
    assert eng._alloc(B, R, S, F, n_img, ik, 96)["MEM"].data_ptr() == full["MEM"].data_ptr()
    pool = w["pool_e"]
    x = pool.get()
    y = pool.get()
    assert x.shape == (w["Te"], cfg.d_model) and x.data_ptr() != y.data_ptr()
    n_free = len(full["pool"].free)
    pool.put(x, y)
    assert len(full["pool"].free) == n_free + 2 and all(t.shape[0] == B * R * S for t in full["pool"].free)


def test_bench_reference_arm_prints_the_contract_line(monkeypatch, capsys):
    """`bench.py --impl reference` (the driver's reference arm): ONE JSON line with the b200 arm's metric / unit / workload, the
    extra keys of the tier contract (impl, cpu_baseline, e2e with zero copy bytes); under torchrun only rank 0 works (the other
    ranks exit 0 without output).  The timing loop itself (a 40-second full-size CPU step) is stubbed here."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2"], env=env,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""
    sys.path.insert(0, root)
    import bench
    seen = {}

    def fake_steps(steps, warmup, budget_s, dataset="yelp"):
        seen.update(steps=steps, warmup=warmup, budget_s=budget_s, dataset=dataset)
        return dict(value=0.25, ms_per_step=4000.0, steps=steps, warmup=warmup, cores=8, kind="reference", sample="1 business per step (stub)")

    monkeypatch.setattr(bench, "cpu_reference_steps", fake_steps)
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--gpus", "4", "--steps", "2", "--warmup", "1"])
    bench.main()
    lines = [l for l in capsys.readouterr().out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert seen == dict(steps=2, warmup=1, budget_s=240.0, dataset="yelp")
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "businesses/s" and d["n_gpus"] == 4
    assert d["higher_is_better"] is True and d["value"] == 0.25 and d["steps"] == 2 and d["warmup"] == 1 and d["scaling"] == "weak"
    assert d["cpu_baseline"] == {"value": 0.25, "unit": "businesses/s", "cores": 8, "kind": "reference", "sample": "1 business per step (stub)"}
    assert d["e2e"] == {"value": 0.25, "unit": "businesses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    # same workload description as the b200 arm (the driver compares the two lines' configs)
    args = bench.parse()
    assert d["config"]["workload"] == bench.train_config(args, 1)["workload"] and d["config"]["workload"].startswith("BASELINE configs[1]")


def test_bench_dump_outputs_samples_and_writes_float_arrays(monkeypatch, tmp_path):
    """--dump-outputs: the same entries of every gradient / parameter on every run, written as float32 / float64 .npy files
    within the size limit; --steps below 1 and a dump of the CPU reference arm are refused."""
    import sys

    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit):
            bench.parse()

    def model():
        torch.manual_seed(3)
        m = torch.nn.Sequential(torch.nn.Linear(100, 80), torch.nn.LayerNorm(80))
        for p in m.parameters():
            p.grad = torch.randn_like(p)
        return m

    a, b = bench.sampled_parameters(model()), bench.sampled_parameters(model())
    n = bench.DUMP_PER_TENSOR + 80 + 80 + 80          # the 8000-entry weight is sampled, the small tensors are kept whole
    assert set(a) == {"grads", "params"} and a["grads"].shape == a["params"].shape == (n,)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    m = model()
    w = m[0].weight.detach().reshape(-1).numpy()
    assert np.isin(a["params"][:bench.DUMP_PER_TENSOR], w).all() and np.array_equal(a["params"][-80:], m[1].bias.detach().numpy())
    bench.dump_outputs(str(tmp_path / "out"), dict(a, loss=np.array([1.5]), ids=np.arange(6).reshape(2, 3)))
    got = {f: np.load(tmp_path / "out" / f) for f in sorted(os.listdir(tmp_path / "out"))}
    assert sorted(got) == ["grads.npy", "ids.npy", "loss.npy", "params.npy"]
    assert got["loss.npy"].dtype == np.float64 and got["ids.npy"].dtype == np.float32 and got["ids.npy"].tolist() == [[0, 1, 2], [3, 4, 5]]
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, np.float32)})


def test_library_is_tied_to_the_sources_it_was_built_from(monkeypatch):
    """build() leaves a record (source digest, nvcc, flags) next to the library; loading a library whose record does not match
    csrc/ + include/ raises instead of running stale kernels (file mtimes do not survive the snapshot to the GPU box)."""
    from multimodalsum_b200 import build as B
    info = _lib.build_info()
    if B.read_build_info() is None:
        pytest.skip("library shipped without a build record")
    assert info["matches_sources"] is True and info["source_digest"] == B.source_digest()
    assert "arch=compute_100a,code=sm_100a" in info["flags"] and "-lineinfo" in info["flags"] and info["arch"] == "sm_100a"
    assert B.build(force=False) == B.LIB                          # current: nothing is recompiled
    monkeypatch.setattr(B, "source_digest", lambda: "0" * 64)     # as if a .cu file had been edited after the build
    assert B.is_current() is False
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(_lib.MmsumError, match="built from different sources"):
        _lib.lib()
    monkeypatch.setenv("MMSUM_ALLOW_STALE_LIB", "1")              # explicit override (A/B tooling)
    assert _lib.lib() is not None


def test_engine_rng_state_round_trip_cpu():
    """Dropout stream state (seed, step counter) is checkpointable: set before or after the arenas are bound, the device-side step
    counter follows; the default seed follows torch.manual_seed and differs per data-parallel rank."""
    from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
    cfg = ModelConfig(dataset="yelp", encoder_layers=1, decoder_layers=1, ffn_dim=64, vocab_size=300, max_position_embeddings=128)
    torch.manual_seed(11)
    a = StepEngine(cfg, device="cpu")
    torch.manual_seed(12)
    b = StepEngine(cfg, device="cpu")
    assert a.seed != b.seed and a.rng_state() == {"seed": a.seed, "step_count": 0}
    os.environ["RANK"] = "3"
    try:
        torch.manual_seed(11)
        assert StepEngine(cfg, device="cpu").seed != a.seed          # same torch seed, another rank: other masks
    finally:
        del os.environ["RANK"]
    a.set_rng_state({"seed": 2 ** 63 + 5, "step_count": 7})           # before bind(): the counter is created from it
    model = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg)
    a.bind(model.named_parameters())
    assert a.rng_state() == {"seed": 2 ** 63 + 5, "step_count": 7} and int(a.step_dev.item()) == 7
    a.set_rng_state({"seed": 9, "step_count": 21})                    # after bind(): the device counter is rewritten
    assert int(a.step_dev.item()) == 21 and a.seed == 9 and a._graphs == {}


def test_c_abi_rejects_invalid_arguments_on_the_host():
    """Error behaviour of the boundary (include/mmsum_b200.h): invalid arguments are detected on the host BEFORE any launch and come
    back as a negative status (-1 invalid argument, -2 driver / tensor-map failure) — no exception, no crash, no device needed;
    the Python side turns any non-zero status into MmsumError."""
    import ctypes as C
    L = _lib.lib()
    i64, i32 = C.c_int64, C.c_int32
    assert L.mmsum_gemm_bf16(None, None) == -1
    assert L.mmsum_gemm_bf16(C.byref(_lib.GemmArgs()), None) == -1                              # null operands
    ok = dict(A=4096, B=4096, D=4096, lda=64, ldb=64, ldd=64, M=128, N=128, K=64)
    for bad in (dict(M=0), dict(K=-3), dict(accumulate=1), dict(aux_mode=1), dict(block_n=96), dict(splits=2),
                dict(out_f32=1, act=1), dict(A=4097)):                                         # misaligned pointer: TMA needs 16 B
        assert L.mmsum_gemm_bf16(C.byref(_lib.GemmArgs(**dict(ok, **bad))), None) < 0, bad
    for fn in (L.mmsum_attn_fwd, L.mmsum_attn_bwd, L.mmsum_attn_decode_cross):
        assert fn(None, None) == -1 and fn(C.byref(_lib.AttnArgs()), None) == -1
    a = _lib.AttnArgs(Q=4096, KV=4096, O=4096, LSE=4096, ldq=1024, ldkv=1024, ldo=1024, n_qseq=1, H=16, R=1, n_mod=5)
    assert L.mmsum_attn_fwd(C.byref(a), None) == -1                                             # at most 3 memory modalities
    assert L.mmsum_table_fwd(None, None) == -1 and L.mmsum_table_fwd(C.byref(_lib.TableArgs(dataset=7, B=1)), None) == -1
    assert L.mmsum_cast_f32_bf16(None, None, i64(16), None) == -1
    assert L.mmsum_cast_f32_bf16(C.c_void_p(4096), C.c_void_p(4096), i64(-1), None) == -1
    assert L.mmsum_colsum(None, i64(8), i32(4), i32(8), None, None) == -1
    assert L.mmsum_grad_sumsq(None, i64(4), None, i32(4), None, None) == -1
    with pytest.raises(_lib.MmsumError, match="rc=-1"):
        _lib.check(-1, "mmsum_gemm_bf16")
    _lib.check(0, "mmsum_gemm_bf16")


def test_bench_roofline_arithmetic():
    """bench.roofline_kernels: achieved = algorithmic work / summed event time; tensor kernels against the sustained bf16 peak in
    TFLOP/s, the others against the HBM peak in GB/s; shares are of the step time; ncu DRAM traffic attached where captured."""
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    peaks = dict(hbm_gbs=6500.0, tf_burst=1600.0, tf_sustained=1400.0, source="measured")
    agg = {"gemm": [984, 2 * 58.0e12, 2 * 46.0], "add_ln_fwd": [120, 120 * 113.2e6, 120 * 0.0283], "idle": [1, 0.0, 0.0]}
    rk = bench.roofline_kernels(agg, 2, peaks, 93.5, {"gemm": {"dram_bytes": 1.0}})
    assert set(rk) == {"gemm", "add_ln_fwd"}                                   # kinds without time are dropped
    g, l = rk["gemm"], rk["add_ln_fwd"]
    assert g["bound"] == "tensor" and g["unit"] == "TFLOP/s" and g["peak"] == 1400.0 and g["launches_per_step"] == 492
    assert g["achieved"] == pytest.approx(58.0e12 / 46.0e-3 / 1e12) and g["frac"] == pytest.approx(g["achieved"] / 1400.0)
    assert g["share_of_step"] == pytest.approx(46.0 / 93.5) and g["traffic"] == {"dram_bytes": 1.0} and g["kernel"] == "gemm_tcgen05_kernel"
    assert l["bound"] == "hbm" and l["unit"] == "GB/s" and l["peak"] == 6500.0 and l["avg_us"] == pytest.approx(28.3)
    assert l["achieved"] == pytest.approx(113.2e6 / 28.3e-6 / 1e9) and "traffic" not in l
    p = bench.load_peaks()
    assert p["tf_sustained"] <= p["tf_burst"] and p["hbm_gbs"] > 1000 and p["source"] in ("measured", "fallback")
