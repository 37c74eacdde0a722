"""Train-step glue around the fused step (SURVEY §8 row a17): `train_model` (src/train_utils.py:65-97), `set_environments`
(:12-31), and the epoch bodies `train` / `validate` (src/multimodal_train.py:346-408) built by `make_loops`.  The orchestration is
checked on CPU with stub loops; the epoch bodies run on the GPU against a hand-written loop over the same batches."""
import types

import pytest
import torch

from multimodalsum_b200 import train_utils as TU
from multimodalsum_b200.synth import ModelConfig, make_batch, make_state_dict

SMALL = dict(encoder_layers=1, decoder_layers=1, ffn_dim=128, vocab_size=300, max_position_embeddings=128, dropout=0.0)


class _Sampler:
    def __init__(self):
        self.epochs = []

    def set_epoch(self, e):
        self.epochs.append(e)


class _Dataset:
    def __init__(self):
        self.reshuffles = 0

    def set_epoch(self):
        self.reshuffles += 1


class _Stateful:
    def __init__(self, tag):
        self.tag, self.n = tag, 0

    def state_dict(self):
        return {"tag": self.tag, "n": self.n}


@pytest.mark.parametrize("early_stopping", [False, True])
def test_train_model_orchestration(tmp_path, early_stopping):
    """Epoch order, sampler / dataset epoch bookkeeping, and which epochs write checkpoints (every epoch, or only a new best
    validation loss under --early_stopping) — src/train_utils.py:65-97."""
    args = types.SimpleNamespace(num_epochs=4, distributed=True, local_rank=0, early_stopping=early_stopping, ckpt=str(tmp_path / "ckpt"))
    model = torch.nn.Linear(2, 2)
    sampler, loader = _Sampler(), types.SimpleNamespace(dataset=_Dataset())
    opt, sch = _Stateful("opt"), _Stateful("sch")
    val_losses = [3.0, 2.0, 2.5, 2.0]
    calls, saved = [], []

    def train(start_time, train_dataloader, m, optimizer, scheduler, e, t_epoch):
        assert train_dataloader is loader and m is model and optimizer is opt and scheduler is sch and t_epoch == 7
        calls.append(("train", e))
        opt.n += 1
        with torch.no_grad():
            model.weight.fill_(float(e))

    def validate(val_dataloader, m, e):
        calls.append(("validate", e))
        return val_losses[e]

    real_save = TU.save_checkpoint

    def spy(*a, **k):
        saved.append(a[3])
        return real_save(*a, **k)

    TU.save_checkpoint, keep = spy, TU.save_checkpoint
    try:
        out = TU.train_model(args, model, sampler, loader, "val", train, validate, opt, sch, 7, "whole", log=lambda *_: None)
    finally:
        TU.save_checkpoint = keep
    assert out == val_losses
    assert calls == [(k, e) for e in range(4) for k in ("train", "validate")]
    assert sampler.epochs == [0, 1, 2, 3] and loader.dataset.reshuffles == 3        # `if e != 0: dataset.set_epoch()`
    assert saved == ([0, 1, 3] if early_stopping else [0, 1, 2, 3])                 # `val_loss <= min(val_loss_list)` (ties save)
    sd = torch.load(tmp_path / "ckpt" / "pytorch_model.bin")
    st = torch.load(tmp_path / "ckpt" / "training_state.bin")
    assert bool((sd["weight"] == 3.0).all()) and st["epoch"] == 3 and st["optimizer"] == {"tag": "opt", "n": 4}
    # other ranks never write
    args2 = types.SimpleNamespace(num_epochs=1, distributed=False, local_rank=1, early_stopping=False, ckpt=str(tmp_path / "rank1"))
    TU.train_model(args2, model, None, loader, "val", train, validate, opt, sch, 7, log=lambda *_: None)
    assert not (tmp_path / "rank1").exists()


def test_set_environments_single_process(tmp_path, monkeypatch):
    for k in ("WORLD_SIZE", "LOCAL_RANK", "RANK"):
        monkeypatch.delenv(k, raising=False)
    args = types.SimpleNamespace(local_rank=0, ckpt=str(tmp_path / "run"), dataset="yelp", batch_size=4)
    out = TU.set_environments(args)
    assert out is args and args.distributed is False and args.world_size == 1 and args.gpu == 0
    saved = torch.load(tmp_path / "run" / "training_args.bin")
    assert saved["dataset"] == "yelp" and saved["batch_size"] == 4                 # vars(args), src/train_utils.py:16
    monkeypatch.setenv("WORLD_SIZE", "1")
    assert TU.set_environments(types.SimpleNamespace(local_rank=0, ckpt=str(tmp_path / "run"))).distributed is False


def test_average_meter():
    m = TU.AverageMeter()
    m.update(2.0, 4)
    m.update(5.0, 2)
    assert m.val == 5.0 and m.count == 6 and m.sum == 18.0 and m.avg == 3.0


def test_checkpoint_resume_round_trip(tmp_path):
    """save_checkpoint -> load_checkpoint: weights, optimizer moments and the schedule position come back; the next epoch index is
    returned; files with foreign keys are refused."""
    from multimodalsum_b200.optim import LinearWarmupSchedule

    def make():
        torch.manual_seed(0)
        m = torch.nn.Sequential(torch.nn.Linear(4, 4), torch.nn.Linear(4, 2))
        o = torch.optim.AdamW(m.parameters(), lr=1e-2)
        return m, o, LinearWarmupSchedule(o, 2, 10)

    m, o, sch = make()
    for _ in range(3):
        o.zero_grad()
        m(torch.ones(1, 4)).sum().backward()
        o.step()
        sch.step()
    TU.save_checkpoint(m, o, sch, 1, str(tmp_path / "c"))
    m2, o2, s2 = make()
    assert TU.load_checkpoint(m2, o2, s2, str(tmp_path / "c")) == 2
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    assert s2.last_epoch == 3 and o2.param_groups[0]["lr"] == o.param_groups[0]["lr"]
    k = next(iter(o.state))
    k2 = next(iter(o2.state))
    assert torch.equal(o.state[k]["exp_avg"], o2.state[k2]["exp_avg"]) and o2.state[k2]["step"] == o.state[k]["step"]
    for mm, oo, ss in ((m, o, sch), (m2, o2, s2)):                  # both continue identically
        oo.zero_grad()
        mm(torch.ones(1, 4)).sum().backward()
        oo.step()
        ss.step()
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    sd = torch.load(tmp_path / "c" / "pytorch_model.bin")
    sd["bogus.weight"] = torch.zeros(1)
    torch.save(sd, tmp_path / "c" / "pytorch_model.bin")
    with pytest.raises(KeyError, match="unexpected keys"):
        TU.load_checkpoint(m2, o2, s2, str(tmp_path / "c"))


def test_checkpoint_files_match_the_reference_inventory(tmp_path):
    """save_checkpoint writes what the reference's model, its stage sub-modules and its AdamW load (src/test.py:205,
    src/multimodal_train.py:116-122, src/train_utils.py:79-97), checked against what the unmodified reference recorded in
    tests/golden/adamw_small.npz: the names of its parameters, and which of them its own get_optimizer + AdamW updated
    (quirk Q1: the no-decay group is empty, so those parameters carry no optimizer state).  A CPU-resident engine (arenas
    only, no kernels) is enough to exercise the writers."""
    from golden_util import load_optimizer_golden
    from multimodalsum_b200.engine import StepEngine
    from multimodalsum_b200.modules import MultimodalSum
    gold = load_optimizer_golden()
    cfg, sd, names, c = gold["cfg"], gold["sd"], gold["names"], gold["case"]
    model = MultimodalSum(config=cfg)
    model.load_state_dict(sd, strict=False)
    eng = StepEngine(cfg, "cpu")
    eng.bind(model.named_parameters())
    object.__setattr__(model, "engine", eng)
    opt = TU.get_optimizer(eng, c["lr"], c["no_decay"], model.named_parameters(), None, max_grad_norm=c["max_grad_norm"])
    torch.manual_seed(0)
    opt.m.normal_()
    opt.v.uniform_()
    opt.step_count = 2
    sched = TU.LinearWarmupSchedule(opt, 2, 8)
    for option in ("whole", "text", "img", "table"):
        TU.save_checkpoint(model, opt, sched, 0, str(tmp_path / option), save_option=option)

    def load(option, f="pytorch_model.bin"):
        return torch.load(str(tmp_path / option / f))

    # whole model: the reference's parameters, plus the entries of its state_dict that are not parameters of their own
    # (the final_logits_bias buffer, and the token embedding that BART and the table encoder share under three more names)
    shared = "bart_model.model.shared.weight"
    aliases = {"bart_model.model.encoder.embed_tokens.weight", "bart_model.model.decoder.embed_tokens.weight",
               "table_encoder.bart_embedding.weight"}
    whole = load("whole")
    assert set(whole) == set(names) | aliases | {"bart_model.final_logits_bias"}
    for n, t in whole.items():
        assert t.shape == sd[n].shape and torch.equal(t, sd[n]), n      # sd: the weights the reference loaded for the golden
    assert all(torch.equal(whole[n], whole[shared]) for n in aliases)
    # stage hand-offs: text -> bart_model, table -> table_encoder, img -> img_encoder
    for option, prefix in (("text", "bart_model."), ("table", "table_encoder."), ("img", "img_encoder.")):
        assert set(load(option)) == {n[len(prefix):] for n in whole if n.startswith(prefix)}, option
    assert set(load("img")) == {"linear.weight"}
    # training_state.bin: transformers-AdamW layout, state exactly for the parameters the reference's AdamW updated
    state = load("whole", "training_state.bin")
    assert state["epoch"] == 0 and state["scheduler"]["last_epoch"] == 0
    updated = {n for n in names if gold["delta_norms"][n] > 0}
    assert 0 < len(updated) < len(names)
    groups = state["optimizer"]["param_groups"]
    assert [g["weight_decay"] for g in groups] == [0.01, 0.0] and all(g["correct_bias"] for g in groups)
    assert groups[0]["params"] == list(range(len(updated))) and groups[1]["params"] == []
    order = [n for n, _ in model.named_parameters() if not any(nd in n for nd in c["no_decay"])]
    assert set(order) == updated
    st = state["optimizer"]["state"]
    assert sorted(st) == groups[0]["params"]
    for i, n in enumerate(order):
        o, k = eng.offsets[n], sd[n].numel()
        assert st[i]["step"] == 2 and st[i]["exp_avg"].shape == st[i]["exp_avg_sq"].shape == sd[n].shape, n
        assert torch.equal(st[i]["exp_avg"].reshape(-1), opt.m[o:o + k]) and torch.equal(st[i]["exp_avg_sq"].reshape(-1), opt.v[o:o + k]), n


class _StubModel(torch.nn.Module):
    """Stands in for the four stage modules on the CPU: records how it was called, returns a loss that depends on one tensor of
    the batch and on its parameters (so backward / clip / step do something)."""

    def __init__(self, pick):
        super().__init__()
        self.img_encoder = torch.nn.Linear(1, 1, bias=False)
        self.table_encoder = torch.nn.Module()
        self.table_encoder.fc = torch.nn.Linear(1, 1, bias=False)
        self.table_encoder.bart_embedding = torch.nn.Linear(1, 1, bias=False)
        self.other = torch.nn.Parameter(torch.ones(1))
        with torch.no_grad():
            for p in self.parameters():
                p.fill_(1.0)
        self.pick, self.calls = pick, []

    def forward(self, *a, **k):
        self.calls.append((self.training, torch.is_grad_enabled(), len(a), sorted(k)))
        x = self.pick(a, k).float().mean()
        w = self.img_encoder.weight.sum() + self.table_encoder.fc.weight.sum() + self.table_encoder.bart_embedding.weight.sum() + self.other.sum()
        return (x * w * 100.0,)


@pytest.mark.parametrize("stage", ["multimodal", "text", "img", "table"])
def test_stage_loops_call_the_model_as_the_reference_scripts_do(stage):
    """make_loops(stage=...) on CPU tensors (device='cpu' prefetchers, stub model): the positional / keyword layout of each
    script's model call, clip_grad_norm_ restricted to the trained head in the img / table stages, size-weighted validation."""
    cfg = ModelConfig(dataset="yelp", **SMALL)
    bs = [make_batch(cfg, n, seed=s, n_reviews=2, max_imgs=2) for s, n in ((1, 2), (2, 2), (3, 1))]
    g = torch.Generator().manual_seed(0)
    labels = [torch.randint(3, 50, (b.reviews.shape[0], 16), generator=g) for b in bs]
    field = bs[0].field
    if stage == "multimodal":
        loader = [_tuple(b) for b in bs]
        pick, want_call = (lambda a, k: a[5]), (7, [])                                     # img
        expect = [b.img.float().mean().item() for b in bs]
    elif stage == "text":
        loader = [(b.reviews, b.reviews_mask, b.reviews_rating) for b in bs]
        pick, want_call = (lambda a, k: a[2]), (3, [])                                     # reviews_rating
        expect = [b.reviews_rating.mean().item() for b in bs]
    elif stage == "img":
        loader = [(b.img[:, 0], b.img_mask, l) for b, l in zip(bs, labels)]
        pick, want_call = (lambda a, k: k["labels"]), (2, ["labels"])
        expect = [l.float().mean().item() for l in labels]
    else:
        loader = [(*b.field_value, l) for b, l in zip(bs, labels)]
        pick, want_call = (lambda a, k: k["labels"] + 0 * a[0].sum() + 0 * a[1][5].sum()), (2, ["labels"])   # (field, field_value, labels=)
        expect = [l.float().mean().item() for l in labels]
    args = types.SimpleNamespace(dataset="yelp", max_grad_norm=1, log_interval=1, distributed=False, world_size=1, local_rank=0)
    model = _StubModel(pick)
    opt = torch.optim.SGD(model.parameters(), lr=0.0)                                       # lr 0: the loss stays a function of the batch only
    sch = torch.optim.lr_scheduler.LambdaLR(opt, lambda step: 1.0)
    logs = []
    train, validate = TU.make_loops(args, field, log=logs.append, stage=stage, device="cpu")
    assert train(0.0, loader, model, opt, sch, 0, 3) == 3
    assert [c[2:] for c in model.calls] == [want_call] * 3 and all(c[0] and c[1] for c in model.calls)
    got = [float(l.rsplit(" ", 1)[1]) for l in logs]
    assert got == pytest.approx([x * 4 * 100.0 for x in expect], rel=1e-5)
    # gradient clipping: the whole model in the multimodal / text stages, only the trained head in the pretraining stages
    gn = {n: p.grad.abs().item() for n, p in [("img", model.img_encoder.weight), ("fc", model.table_encoder.fc.weight),
                                                ("bart", model.table_encoder.bart_embedding.weight), ("other", model.other)]}
    raw = abs(expect[-1]) * 100.0
    if stage in ("multimodal", "text"):
        assert all(v == pytest.approx(0.5, rel=1e-4) for v in gn.values())                 # 4 equal gradients clipped to total norm 1
    elif stage == "img":
        assert gn["img"] == pytest.approx(1.0, rel=1e-4) and gn["fc"] == pytest.approx(raw, rel=1e-4) and gn["other"] == pytest.approx(raw, rel=1e-4)
    else:
        assert gn["fc"] == pytest.approx(1.0, rel=1e-4) and gn["bart"] == pytest.approx(raw, rel=1e-4) and gn["img"] == pytest.approx(raw, rel=1e-4)
    model.calls.clear()
    avg = validate(loader, model, 0)
    assert all((not c[0]) and (not c[1]) for c in model.calls) and len(model.calls) == 3   # eval mode, under no_grad
    sizes = [2, 2, 1]
    assert avg == pytest.approx(sum(x * 400.0 * n for x, n in zip(expect, sizes)) / 5, rel=1e-5)
    with pytest.raises(ValueError):
        TU.make_loops(args, field, stage="bogus")


def test_generation_loop_of_test_py_on_stubs():
    """make_test_loop: the body of src/test.py:137-165 — one get_multimodal_outputs + generate per batch with the reference's
    arguments, summaries of all businesses in loader order, decoded when a tokenizer is given."""
    cfg = ModelConfig(dataset="yelp", **SMALL)
    bs = [make_batch(cfg, n, seed=s, n_reviews=2, max_imgs=2) for s, n in ((1, 2), (2, 1))]
    seen = []

    class _Bart:
        def generate(self, th, tm, tbh, tbm, ih, im, **kw):
            seen.append((tuple(th.shape), kw["rating_diff"].shape, {k: v for k, v in kw.items() if k != "rating_diff"}, torch.is_grad_enabled()))
            return torch.arange(th.size(0) * 3).reshape(th.size(0), 3) + 10 * len(seen)

    class _Model(torch.nn.Module):
        bart_model = _Bart()

        def get_multimodal_outputs(self, reviews, reviews_mask, field, field_value, img, img_mask):
            assert field.shape == (47, 6) and len(field_value) == 6 and not self.training
            B = reviews.size(0)
            return (reviews.size(1), torch.zeros(B, 2, 128, 4), reviews_mask, torch.zeros(B, 1, 47, 4), torch.ones(B, 1, 47),
                    torch.zeros(B, 2, 196, 4), torch.ones(B, 2, 196))

    args = types.SimpleNamespace(dataset="yelp", num_beams=4, length_penalty=1.0, max_length=128)
    logs = []
    test = TU.make_test_loop(args, bs[0].field, log=logs.append, device="cpu")
    out = test([_tuple(b) for b in bs], _Model(), None)
    assert [o.tolist() for o in out] == [[10, 11, 12], [13, 14, 15], [20, 21, 22]] and logs == ["1 / 2", "2 / 2"]
    want_kw = dict(num_beams=4, length_penalty=1.0, max_length=128, no_repeat_ngram_size=3, early_stopping=True)
    assert seen == [((2, 2, 128, 4), torch.Size([2, 1]), want_kw, False), ((1, 2, 128, 4), torch.Size([1, 1]), want_kw, False)]
    tok = types.SimpleNamespace(decode=lambda g, skip_special_tokens, clean_up_tokenization_spaces: " ".join(str(int(x)) for x in g))
    assert test([_tuple(bs[1])], _Model(), tok) == ["30 31 32"]


# ------------------------------------------------------------------------------------------------ GPU
def _tuple(b):
    return (b.reviews, b.reviews_mask, b.reviews_rating, *b.field_value, b.img, b.img_mask)


@pytest.mark.gpu
def test_epoch_bodies_match_a_hand_written_loop_gpu(tmp_path):
    """`train` / `validate` from make_loops (the reference's signatures) over a list loader with a short last validation batch:
    the training losses and weight updates agree with the same statements written out by hand on resident batches, the
    validation average is weighted by batch size (`losses.update(loss, reviews.size(0))`), and `train_model` leaves loadable files."""
    from multimodalsum_b200.modules import MultimodalSum, YelpTableEncoder
    from multimodalsum_b200.optim import get_optimizer, get_scheduler
    cfg = ModelConfig(dataset="yelp", **SMALL)
    sd = make_state_dict(cfg, seed=0, gates_open=True)
    train_b = [make_batch(cfg, 2, seed=20 + i, n_reviews=3, max_imgs=2) for i in range(3)]
    val_b = [make_batch(cfg, n, seed=40 + i, n_reviews=3, max_imgs=2) for i, n in enumerate([2, 1])]
    field = train_b[0].field.cuda()
    args = types.SimpleNamespace(dataset="yelp", max_grad_norm=1, log_interval=2, distributed=False, world_size=1, local_rank=0,
                                 num_epochs=1, warmup_ratio=0.0, early_stopping=False, ckpt=str(tmp_path / "ckpt"))

    def fresh():
        m = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg, label_smoothing=0.1)
        m.load_state_dict(sd, strict=False)
        m = m.cuda()
        eng = m._ensure_engine(torch.device("cuda"))
        opt = get_optimizer(eng, 1e-3, ["bias", "layer_norm.weight"], list(m.named_parameters()), None, max_grad_norm=1.0)
        return m, opt, get_scheduler(args, len(train_b), opt)

    # by hand: src/multimodal_train.py:357-364 on resident batches
    m1, opt1, sch1 = fresh()
    m1.train()
    want = []
    for b in train_b:
        d = b.to("cuda")
        loss = m1(d.reviews, d.reviews_mask, d.reviews_rating, field, d.field_value, d.img, d.img_mask)[0]
        opt1.zero_grad()
        loss.backward()
        opt1.step()
        sch1.step()
        want.append(loss.item())
    m1.eval()
    vl = []
    with torch.no_grad():
        for b in val_b:
            d = b.to("cuda")
            vl.append(m1(d.reviews, d.reviews_mask, d.reviews_rating, field, d.field_value, d.img, d.img_mask)[0].item())
    want_val = (vl[0] * 2 + vl[1] * 1) / 3

    m2, opt2, sch2 = fresh()
    logs = []
    train, validate = TU.make_loops(args, field, log=logs.append)
    out = TU.train_model(args, m2, None, [_tuple(b) for b in train_b], [_tuple(b) for b in val_b], train, validate, opt2, sch2,
                         len(train_b), "whole", log=logs.append)
    got = [float(l.rsplit(" ", 1)[1]) for l in logs if "batch id" in l]
    # log_interval 2: batches 1 and 3.  The first loss is bit-equal (same kernels, same inputs); after optimizer steps the two runs
    # agree to the run-to-run rounding of the fp32 reduction order in the weight gradients (split-K / atomics; measured 4e-7)
    assert len(got) == 2 and got[0] == pytest.approx(want[0], rel=1e-6) and got[1] == pytest.approx(want[2], rel=1e-4)
    assert out == [pytest.approx(want_val, rel=1e-4)] and any("epoch valid loss" in l for l in logs)
    d1 = torch.cat([(p.detach().float().cpu() - sd[n].float()).reshape(-1) for n, p in m1.named_parameters() if n in sd])
    d2 = torch.cat([(p.detach().float().cpu() - sd[n].float()).reshape(-1) for n, p in m2.named_parameters() if n in sd])
    assert d1.norm() > 0 and torch.nn.functional.cosine_similarity(d1, d2, dim=0).item() > 0.9    # the same three updates
    assert opt2.step_count == 3 and sch2.last_epoch == 3
    re = MultimodalSum(TableEncoder=YelpTableEncoder, config=cfg, label_smoothing=0.1)
    missing = re.load_state_dict(torch.load(tmp_path / "ckpt" / "pytorch_model.bin"), strict=False)
    assert not missing.unexpected_keys
    assert torch.load(tmp_path / "ckpt" / "training_state.bin")["epoch"] == 0


def test_train_synthetic_script_keeps_the_reference_flags():
    """tools/train_synthetic.py (main() of src/multimodal_train.py on the drop-in): the reference's flags and defaults (:411-439)."""
    import importlib.util
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "train_synthetic.py")
    spec = importlib.util.spec_from_file_location("train_synthetic", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    a = mod.parse([])
    assert (a.dataset, a.batch_size, a.num_epochs, a.warmup_ratio, a.max_grad_norm, a.learning_rate, a.label_smoothing,
            a.early_stopping, a.workers, a.local_rank) == ("yelp", 1, 5, 0.05, 1, 1e-5, 0.1, False, 4, 0)
    b = mod.parse(["--dataset", "amazon", "--early_stopping", "true", "--batch_size", "16"])
    assert b.dataset == "amazon" and b.early_stopping is True and b.batch_size == 16
    with pytest.raises(SystemExit):
        mod.parse(["--early_stopping", "maybe"])
