"""TEST INFRASTRUCTURE — runs the UNMODIFIED reference (nc-ai/MultimodalSum) from a checkout of it.

The checkout is not part of this repository.  It is found at $MMSUM_REF, else at oracle/_ref or baseline/_ref inside the
repository (both git-ignored).  Used by tests/golden/make_golden.py to produce the committed golden vectors, by
tests/test_oracle_vs_reference.py to pin oracle/mmsum_oracle.py, and by bench.py's CPU reference arm when present.
Nothing on the product path, in the `-m gpu` tests or smoke() imports this file.

Recipe (SURVEY.md §8c / App. G): put <checkout>/src on sys.path, stub the two imports that no longer exist
(`apex.parallel.DistributedDataParallel`, `transformers.AdamW`), build `MultimodalSum` without its network-bound
constructor, and call the reference's own `MultimodalSum.forward` (src/multimodal_train.py:124-163).  Only the image
branch of `get_multimodal_outputs` (:188-192, which hard-codes a ResNet over [*,3,224,224]) is restated so pooled
features [B, max_imgs, 196, 1024] can be fed to `img_encoder.linear` (src/img_encoder.py:39-40).
"""
import argparse
import os
import sys
import types

import torch
import torch.nn as nn

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def find_reference():
    """The first reference checkout among $MMSUM_REF, oracle/_ref and baseline/_ref, or None."""
    for cand in (os.environ.get("MMSUM_REF"), os.path.join(_REPO, "oracle", "_ref"), os.path.join(_REPO, "baseline", "_ref")):
        if cand and os.path.isdir(os.path.join(cand, "src", "transformer")):
            return cand
    return None


REF_ROOT = find_reference()


def available():
    return REF_ROOT is not None


_mods = {}


def _import_reference():
    if _mods:
        return _mods
    if not available():
        raise RuntimeError("no reference checkout at $MMSUM_REF, oracle/_ref or baseline/_ref")
    sys.dont_write_bytecode = True
    src = os.path.join(REF_ROOT, "src")
    if src not in sys.path:
        sys.path.insert(0, src)
    # stubs for imports that do not exist in this image (not edits to the reference)
    if "apex" not in sys.modules:
        apex = types.ModuleType("apex")
        apex_parallel = types.ModuleType("apex.parallel")
        apex_parallel.DistributedDataParallel = torch.nn.parallel.DistributedDataParallel
        apex.parallel = apex_parallel
        sys.modules["apex"] = apex
        sys.modules["apex.parallel"] = apex_parallel
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import transformer  # vendored HF 3.0.2
        import transformers
        if not hasattr(transformers, "AdamW"):
            from transformer.optimization import AdamW as _RefAdamW  # vendored copy of transformers 3.0.2 AdamW
            transformers.AdamW = _RefAdamW
        import multimodal_train as MT
        import table_encoder as TE
        import utils as U
        from transformer.modeling_multimodalsum import BartForMultiEncConditionalGeneration, BartForEncConditionalGeneration
        from transformer.configuration_bart import BartConfig
    _mods.update(dict(MT=MT, TE=TE, U=U, BartConfig=BartConfig, transformer=transformer,
                      MultiEnc=BartForMultiEncConditionalGeneration, Enc=BartForEncConditionalGeneration))
    return _mods


class _FeatProj(nn.Module):
    """Stand-in for src/img_encoder.py Resnet with the trunk removed: only `.linear` (1024 -> d_model, no bias)."""

    def __init__(self, d_model):
        super().__init__()
        self.linear = nn.Linear(1024, d_model, bias=False)

    def forward(self, feats):
        return self.linear(feats)


def _get_multimodal_outputs(self, reviews, reviews_mask, field, field_value, img, img_mask):
    # restatement of src/multimodal_train.py:165-193 with pooled features instead of raw pixels
    bsz, n_reviews, seq_len = reviews.size()
    text_hiddens = self.bart_model.model.encoder(input_ids=reviews.view(bsz * n_reviews, seq_len),
                                                 attention_mask=reviews_mask.view(bsz * n_reviews, seq_len))[0]
    text_hiddens = text_hiddens.view(bsz, n_reviews, seq_len, -1)
    table_hiddens, table_mask = self.table_encoder(field, field_value)
    img_hiddens = self.img_encoder(img)
    img_attention_mask = img_mask.unsqueeze(-1).repeat(1, 1, img_hiddens.size(2))
    return (n_reviews, text_hiddens, reviews_mask, table_hiddens.unsqueeze(1), table_mask.unsqueeze(1),
            img_hiddens, img_attention_mask)


def build_reference_model(cfg, state_dict, dtype=torch.float32, label_smoothing=0.1, dropout=0.0):
    """cfg: multimodalsum_b200.synth.ModelConfig; returns the reference MultimodalSum with `state_dict` loaded."""
    m = _import_reference()
    MT = m["MT"]
    MT.args = argparse.Namespace(label_smoothing=label_smoothing)
    bcfg = m["BartConfig"].from_json_file(os.path.join(REF_ROOT, "cfg", "bart-large.json"))
    for k, v in cfg.to_reference_dict().items():
        setattr(bcfg, k, v)
    bcfg.dropout = dropout
    model = MT.MultimodalSum.__new__(MT.MultimodalSum)
    nn.Module.__init__(model)
    model.bart_model = m["MultiEnc"](bcfg)
    TableEnc = m["TE"].YelpTableEncoder if cfg.table == "yelp" else m["TE"].AmazonTableEncoder
    model.table_encoder = TableEnc(model.bart_model.model.shared)
    model.img_encoder = _FeatProj(cfg.d_model)
    model.get_multimodal_outputs = types.MethodType(_get_multimodal_outputs, model)
    missing, unexpected = model.load_state_dict(state_dict, strict=False)
    assert not unexpected, unexpected
    assert not missing, missing
    model = model.to(dtype)
    model.train()
    return model


def reference_step(cfg, state_dict, batch, dtype=torch.float64, label_smoothing=0.1):
    """Run the reference's forward + backward; returns (loss, {name: grad})."""
    model = build_reference_model(cfg, state_dict, dtype=dtype, label_smoothing=label_smoothing)
    img = batch.img.to(dtype)
    loss = model(batch.reviews, batch.reviews_mask, batch.reviews_rating.to(dtype), batch.field, batch.field_value,
                 img, batch.img_mask)[0]
    model.zero_grad()
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return loss.detach(), grads, model


def reference_text_step(cfg, state_dict, batch, dtype=torch.float32, label_smoothing=None):
    """BASELINE config 1: the reference's text-only step — text_pretrain.TextSupervised.forward
    (src/text_pretrain.py:71-113) around BartForEncConditionalGeneration, plain CrossEntropyLoss by default."""
    m = _import_reference()
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import text_pretrain as TP
    TP.args = argparse.Namespace(label_smoothing=label_smoothing)
    if label_smoothing is not None:
        TP.LabelSmoothingLoss = m["U"].LabelSmoothingLoss  # quirk Q6: text_pretrain.py never imports it
    bcfg = m["BartConfig"].from_json_file(os.path.join(REF_ROOT, "cfg", "bart-large.json"))
    for k, v in cfg.to_reference_dict().items():
        setattr(bcfg, k, v)
    bcfg.dropout = 0.0
    model = TP.TextSupervised.__new__(TP.TextSupervised)
    nn.Module.__init__(model)
    model.bart_model = m["Enc"](bcfg)
    missing, unexpected = model.load_state_dict(state_dict, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    model = model.to(dtype).train()
    loss = model(batch.reviews, batch.reviews_mask, batch.reviews_rating.to(dtype))[0]
    model.zero_grad()
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return loss.detach(), grads, model


class _FeatBox:
    """Lets the UNMODIFIED ImgSupervised.forward (src/img_pretrain.py:108-113) run on pooled features: it only calls
    `.size()` and `.reshape([-1, 3, 224, 224])` on its image input before handing it to `img_encoder`."""

    def __init__(self, feats):
        self.feats = feats

    def size(self):
        return self.feats.size()

    def reshape(self, shape):
        return self.feats


def reference_stage_step(cfg, state_dict, batch, dtype=torch.float32, label_smoothing=0.1):
    """The reference's single-modality pretraining steps, unmodified: img_pretrain.ImgSupervised.forward
    (src/img_pretrain.py:91-141) / table_pretrain.TableSupervised.forward (src/table_pretrain.py:90-129)."""
    m = _import_reference()
    import warnings
    bcfg = m["BartConfig"].from_json_file(os.path.join(REF_ROOT, "cfg", "bart-large.json"))
    for k, v in cfg.to_reference_dict().items():
        setattr(bcfg, k, v)
    bcfg.dropout = 0.0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if cfg.image:
            import img_pretrain as SP
            model = SP.ImgSupervised.__new__(SP.ImgSupervised)
            nn.Module.__init__(model)
            model.bart_model = m["Enc"](bcfg)
            model.img_encoder = _FeatProj(cfg.d_model)
        else:
            import table_pretrain as SP
            model = SP.TableSupervised.__new__(SP.TableSupervised)
            nn.Module.__init__(model)
            model.bart_model = m["Enc"](bcfg)
            TableEnc = m["TE"].YelpTableEncoder if cfg.table == "yelp" else m["TE"].AmazonTableEncoder
            model.table_encoder = TableEnc(model.bart_model.model.shared)
    SP.args = argparse.Namespace(label_smoothing=label_smoothing)
    missing, unexpected = model.load_state_dict(state_dict, strict=False)
    assert not unexpected and not missing, (missing, unexpected)
    model = model.to(dtype).train()
    if cfg.image:
        loss = model(_FeatBox(batch.img.to(dtype)), batch.img_mask, labels=batch.labels)[0]
    else:
        loss = model(batch.field, batch.field_value, labels=batch.labels)[0]
    model.zero_grad()
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return loss.detach(), grads, model


def reference_generate(cfg, state_dict, batch, num_beams=4, max_length=20, length_penalty=1.0, no_repeat_ngram_size=3,
                       early_stopping=True, dtype=torch.float32):
    """BASELINE config 5: the reference's own generation path, as src/test.py:152-158 drives it —
    get_multimodal_outputs (no_grad), rating_diff = 0, bart_model.generate(beam search)."""
    model = build_reference_model(cfg, state_dict, dtype=dtype)
    model.eval()
    with torch.no_grad():
        _, th, tm, tabh, tabm, ih, im = model.get_multimodal_outputs(batch.reviews, batch.reviews_mask, batch.field, batch.field_value,
                                                                       batch.img.to(dtype), batch.img_mask)
        rating_diff = torch.zeros([th.size(0), 1], dtype=dtype)
        out = model.bart_model.generate(th, tm, tabh, tabm, ih, im, rating_diff=rating_diff, num_beams=num_beams,
                                        length_penalty=length_penalty, max_length=max_length,
                                        no_repeat_ngram_size=no_repeat_ngram_size, early_stopping=early_stopping)
    return out
