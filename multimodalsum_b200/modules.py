"""Drop-in `nn.Module` surface of the reference for the training-step path (SURVEY §8b).

Same class names, constructor meaning, forward signatures, return tuples and `state_dict` keys/shapes as
  MultimodalSum                         src/multimodal_train.py:111-193   (.forward, .get_multimodal_outputs)
  TextSupervised                        src/text_pretrain.py:66-113
  ImgSupervised / TableSupervised       src/img_pretrain.py:85-141, src/table_pretrain.py:84-129
  BartForMultiEncConditionalGeneration  src/transformer/modeling_multimodalsum.py:2181-2292 (.forward), :2295 (.generate)
  BartForEncConditionalGeneration       :1290-1396
  BartEncoder                           :321-404
  YelpTableEncoder / AmazonTableEncoder src/table_encoder.py:14-83, 95-167
  Resnet (projection head only)         src/img_encoder.py:26,39-40  (pooled stage-3 features in, trunk out of scope)
  LabelSmoothingLoss                    src/utils.py:22-38

The modules HOLD the parameters (fp32 masters, re-pointed into the engine's flat arena on first use); all compute runs
in the CUDA kernels behind the C-ABI.  Two kinds of forward:
  * the TRAINING step — `MultimodalSum / TextSupervised / ImgSupervised / TableSupervised.forward` — is one fused
    forward+backward engine (`engine.StepEngine`) behind a single autograd node;
  * the sub-module forwards (`BartEncoder`, table / image encoders, `BartFor*ConditionalGeneration.forward/.generate`,
    `get_multimodal_outputs`) are the INFERENCE paths src/test.py drives: same kernels, no autograd graph
    (activations come back as bf16 tensors, logits as fp32).
There is no eager/CPU fallback: without a CUDA device and the built library every forward raises.
"""
import os
import weakref

import torch
import torch.nn as nn

from . import inference as INF
from . import ops
from .engine import StepEngine
from .synth import Batch, ModelConfig


def _init_linear(m, std):
    m.weight.data.normal_(mean=0.0, std=std)
    if m.bias is not None:
        m.bias.data.zero_()


# ---------------------------------------------------------------------------------------------- engine ownership
class _EngineRoot:
    """Mixin of the modules that can own a StepEngine (the flat parameter arenas + kernels).  Sub-modules reach the engine
    of the root that adopted them; a stand-alone BartFor*ConditionalGeneration is its own root."""

    _param_prefix = ""          # prefix that maps this module's parameter names onto the reference MultimodalSum keys

    def _adopt_children(self):
        ref = weakref.ref(self)
        for m in self.modules():
            if m is not self:
                object.__setattr__(m, "_root_ref", ref)

    def enable_cuda_graph(self, on=True):
        """Replay the training step from recorded CUDA graphs (engine.StepEngine.enable_graph); call after `.cuda()`."""
        dev = next(self.parameters()).device
        self._ensure_engine(dev).enable_graph(on)
        return self

    def _ensure_engine(self, device):
        device = torch.device(device)
        if getattr(self, "engine", None) is None:
            if device.type != "cuda":
                raise RuntimeError("mmsum_b200 has no CPU path: move the module and its inputs to a CUDA device")
            eng = StepEngine(self.cfg, device)
            eng.bind((self._param_prefix + n, p) for n, p in self.named_parameters())
            flb = self.bart_model.final_logits_bias if hasattr(self, "bart_model") else self.final_logits_bias
            eng.final_logits_bias = flb
            object.__setattr__(self, "engine", eng)
        return self.engine


def _engine_of(module, device):
    ref = getattr(module, "_root_ref", None)
    root = ref() if ref is not None else None
    if root is None:
        if isinstance(module, _EngineRoot):
            root = module
        else:
            raise RuntimeError("%s must be part of a MultimodalSum / TextSupervised / BartFor*ConditionalGeneration model to run: "
                               "its kernels read the model's parameter arena" % type(module).__name__)
    while getattr(root, "_root_ref", None) is not None and root._root_ref() is not None:
        root = root._root_ref()
    eng = root._ensure_engine(device)
    eng.refresh_bf16_weights()
    return eng


# ---------------------------------------------------------------------------------------------- BART containers
class _Attention(nn.Module):
    def __init__(self, d, cross=False, multimodal=False):
        super().__init__()
        # registration order k, v, q, out as in the reference (modeling_multimodalsum.py:695-698)
        self.k_proj = nn.Linear(d, d)
        self.v_proj = nn.Linear(d, d)
        self.q_proj = nn.Linear(d, d)
        self.out_proj = nn.Linear(d, d)
        if cross and multimodal:
            self.alpha_proj = nn.Linear(2 * d, d)
            self.beta_proj = nn.Linear(2 * d, d)


class _EncoderLayer(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        d = cfg.d_model
        self.self_attn = _Attention(d)
        self.self_attn_layer_norm = nn.LayerNorm(d)
        self.fc1 = nn.Linear(d, cfg.ffn_dim)
        self.fc2 = nn.Linear(cfg.ffn_dim, d)
        self.final_layer_norm = nn.LayerNorm(d)


class _DecoderLayer(nn.Module):
    def __init__(self, cfg, multimodal):
        super().__init__()
        d = cfg.d_model
        self.self_attn = _Attention(d)
        self.self_attn_layer_norm = nn.LayerNorm(d)
        self.encoder_attn = _Attention(d, cross=True, multimodal=multimodal)
        self.encoder_attn_layer_norm = nn.LayerNorm(d)
        self.fc1 = nn.Linear(d, cfg.ffn_dim)
        self.fc2 = nn.Linear(cfg.ffn_dim, d)
        self.final_layer_norm = nn.LayerNorm(d)


class BartEncoder(nn.Module):
    def __init__(self, cfg, embed_tokens):
        super().__init__()
        self.embed_tokens = embed_tokens
        self.embed_positions = nn.Embedding(cfg.max_position_embeddings + 2, cfg.d_model, padding_idx=cfg.pad_token_id)
        self.layers = nn.ModuleList([_EncoderLayer(cfg) for _ in range(cfg.encoder_layers)])
        self.layernorm_embedding = nn.LayerNorm(cfg.d_model)

    def forward(self, input_ids, attention_mask=None, **unused):
        """modeling_multimodalsum.py:346-404 (eval): input_ids [N, S], attention_mask [N, S] 1 = token -> (x [N, S, D],)."""
        eng = _engine_of(self, input_ids.device)
        return (INF.encoder_forward(eng, input_ids, attention_mask),)


class BartDecoder(nn.Module):
    def __init__(self, cfg, embed_tokens, multimodal):
        super().__init__()
        self.embed_tokens = embed_tokens
        self.rating_embeddings = nn.Parameter(torch.empty(cfg.d_model).normal_(mean=0.0, std=cfg.init_std))
        self.embed_positions = nn.Embedding(cfg.max_position_embeddings + 2, cfg.d_model, padding_idx=cfg.pad_token_id)
        self.layers = nn.ModuleList([_DecoderLayer(cfg, multimodal) for _ in range(cfg.decoder_layers)])
        self.layernorm_embedding = nn.LayerNorm(cfg.d_model)


class BartModel(nn.Module):
    def __init__(self, cfg, multimodal):
        super().__init__()
        self.shared = nn.Embedding(cfg.vocab_size, cfg.d_model, padding_idx=cfg.pad_token_id)
        self.encoder = BartEncoder(cfg, self.shared)
        self.decoder = BartDecoder(cfg, self.shared, multimodal)


def _as_engine_cfg(config, multimodal):
    """A stand-alone BART container runs on an engine without table / image encoders: 'yelp' keeps the gated three-modality
    decoder layout, 'text' the single-memory one."""
    want = ("yelp", "amazon") if multimodal else ("text", "img", "table_yelp", "table_amazon")
    if config.dataset in want:
        return config
    import dataclasses
    return dataclasses.replace(config, dataset=want[0])


class _BartLMBase(nn.Module, _EngineRoot):
    _param_prefix = "bart_model."

    def __init__(self, config: ModelConfig, multimodal):
        super().__init__()
        self.config = config
        self.cfg = _as_engine_cfg(config, multimodal)
        self.model = BartModel(config, multimodal)
        self.register_buffer("final_logits_bias", torch.zeros((1, config.vocab_size)))
        self.apply(self._init_weights)
        self.engine = None
        self._adopt_children()

    def _init_weights(self, m):
        # PretrainedBartModel._init_weights, modeling_multimodalsum.py:188-199
        std = self.config.init_std
        if isinstance(m, nn.Linear):
            _init_linear(m, std)
        elif isinstance(m, nn.Embedding):
            m.weight.data.normal_(mean=0.0, std=std)
            if m.padding_idx is not None:
                m.weight.data[m.padding_idx].zero_()

    # -- shared bodies ------------------------------------------------------------------------------------
    @torch.no_grad()
    def _lm_forward(self, hiddens, masks, rating_diff, decoder_input_ids, decoder_attention_mask, decoder_past_key_values, labels):
        eng = _engine_of(self, hiddens[0].device)
        cfg = eng.cfg
        if decoder_past_key_values is not None:
            raise NotImplementedError("the incremental-cache calling convention is internal to .generate(); call generate() or "
                                      "pass the full decoder_input_ids")
        if labels is not None:
            # _prepare_bart_decoder_inputs (:160-181): decoder inputs = shift_tokens_right(labels) unless given, pad mask from them
            if decoder_input_ids is None:
                decoder_input_ids = INF.shift_tokens_right(labels, cfg.pad_token_id, cfg.bos_token_id, cfg.eos_token_id)
            if decoder_attention_mask is None:
                decoder_attention_mask = decoder_input_ids.ne(cfg.pad_token_id)
        elif decoder_input_ids is None:
            raise ValueError("labels or decoder_input_ids required")
        mem = INF.build_memory(eng, hiddens, masks)
        N, T = decoder_input_ids.shape
        x = INF.decoder_hidden(eng, mem, decoder_input_ids, rating_diff, per_biz=N // mem.B, dec_valid=decoder_attention_mask)
        logits = INF.lm_head(eng, x[:, :T].reshape(N * T, cfg.d_model))
        return (logits.reshape(N, T, cfg.vocab_size),)

    @torch.no_grad()
    def _lm_generate(self, hiddens, masks, rating_diff, kw):
        from .generation import Generator, resolve_generate_args
        args = resolve_generate_args(kw)     # defaults and validation (beam sampling, bad_words_ids: NotImplementedError)
        eng = _engine_of(self, hiddens[0].device)
        root = self._root_ref() if getattr(self, "_root_ref", None) is not None else self
        mem = INF.build_memory(eng, hiddens, masks)
        gen = getattr(root, "_generator", None)
        if gen is None:                       # one Generator per model: it caches the recorded token-step graphs per shape
            gen = Generator(root)
            object.__setattr__(root, "_generator", gen)
        return gen.generate_from_memory(mem, rating_diff, **args)


class BartForMultiEncConditionalGeneration(_BartLMBase):
    """Three-memory decoder with gated fusion (`multimodal=True`) — modeling_multimodalsum.py:2181-2292."""

    def __init__(self, config: ModelConfig, multimodal=True):
        super().__init__(config, multimodal)

    def forward(self, text_hiddens, text_attention_mask, table_hiddens, table_attention_mask, img_hiddens, img_attention_mask,
                rating_diff=None, decoder_input_ids=None, decoder_attention_mask=None, decoder_past_key_values=None, labels=None,
                use_cache=None, output_attentions=False, output_hidden_states=False, return_dict=False, **unused):
        """-> (lm_logits [B, T, V] fp32,).  Memories [B, E, S, D] with masks [B, E, S] (1 = attend), as the reference."""
        return self._lm_forward([text_hiddens, table_hiddens, img_hiddens],
                                [text_attention_mask, table_attention_mask, img_attention_mask],
                                rating_diff, decoder_input_ids, decoder_attention_mask, decoder_past_key_values, labels)

    def generate(self, text_hiddens, text_attention_mask, table_hiddens, table_attention_mask, img_hiddens, img_attention_mask,
                 input_ids=None, rating_diff=None, **kw):
        """Beam search, greedy decoding or sampling (do_sample=True, temperature, top_k, top_p, repetition_penalty) over the
        given memories (:2295-2693) -> token ids [B * num_return_sequences, <= max_length]."""
        return self._lm_generate([text_hiddens, table_hiddens, img_hiddens],
                                 [text_attention_mask, table_attention_mask, img_attention_mask], rating_diff, kw)


class BartForEncConditionalGeneration(_BartLMBase):
    """Single-memory decoder (text-only / img / table stages) — modeling_multimodalsum.py:1290-1396."""

    def __init__(self, config: ModelConfig):
        super().__init__(config, multimodal=False)

    def forward(self, encoder_hiddens, rating_diff=None, encoder_attention_mask=None, decoder_input_ids=None,
                decoder_attention_mask=None, decoder_past_key_values=None, labels=None, use_cache=None, output_attentions=False,
                output_hidden_states=False, return_dict=False, **unused):
        return self._lm_forward([encoder_hiddens], [encoder_attention_mask], rating_diff, decoder_input_ids,
                                decoder_attention_mask, decoder_past_key_values, labels)

    def generate(self, encoder_hiddens, encoder_attention_mask=None, input_ids=None, rating_diff=None, **kw):
        return self._lm_generate([encoder_hiddens], [encoder_attention_mask], rating_diff, kw)


# ---------------------------------------------------------------------------------------------- modality encoders
class _TableEncoderBase(nn.Module):
    def forward(self, field, field_value):
        """src/table_encoder.py:14-83 / 95-167 -> (emb [B, F, D], mask bool [B, F])."""
        eng = _engine_of(self, field.device)
        emb, valid = INF.table_forward(eng, field, list(field_value))
        return emb, valid.bool()


class YelpTableEncoder(_TableEncoderBase):
    def __init__(self, bart_embedding):
        super().__init__()
        self.bart_embedding = bart_embedding
        self.rating_embedding = nn.Linear(4, 1024, bias=False)
        self.hours_embedding = nn.Linear(4, 1024, bias=False)
        self.fc = nn.Linear(2048, 1024)
        self.linear = nn.Linear(1024, 1024, bias=False)


class AmazonTableEncoder(_TableEncoderBase):
    def __init__(self, bart_embedding):
        super().__init__()
        self.bart_embedding = bart_embedding
        self.price_embedding = nn.Linear(11, 1024, bias=False)
        self.rating_embedding = nn.Linear(4, 1024, bias=False)
        self.fc = nn.Linear(2048, 1024)
        self.linear = nn.Linear(1024, 1024, bias=False)


class Resnet(nn.Module):
    """Projection head of src/img_encoder.py (`linear`, 1024 -> d_model, no bias).  The ResNet-101 trunk is outside the
    hot path (north star): `img` inputs are its pooled stage-3 features [B, max_imgs, 196, 1024]."""

    def __init__(self, embedding_dim):
        super().__init__()
        self.linear = nn.Linear(1024, embedding_dim, bias=False)

    def forward(self, x):
        """Pooled features [..., 196, 1024] -> [..., 196, d_model] (src/img_encoder.py:39-40)."""
        eng = _engine_of(self, x.device)
        lead = x.shape[:-2]
        y = INF.image_forward(eng, x.reshape(1, -1, x.shape[-2], x.shape[-1]))
        return y.reshape(*lead, x.shape[-2], -1)


class _LSLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, eps):
        rows, V = pred.shape
        ld = (V + 7) // 8 * 8
        z = torch.empty(rows, ld, device=pred.device, dtype=torch.bfloat16)
        z[:, :V] = pred.detach()
        loss_rows = torch.empty(rows, device=pred.device)
        loss = torch.empty(1, device=pred.device)
        tgt = target.to(torch.int32).contiguous()
        ops.ce_fwd_bwd(z, V, tgt, eps, 0.0, None, loss_rows, loss, 1.0 / rows, False)
        ctx.save_for_backward(z, tgt)
        ctx.eps, ctx.V, ctx.dtype = eps, V, pred.dtype
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        z, tgt = ctx.saved_tensors
        rows = z.shape[0]
        scratch = torch.empty(rows, device=z.device)
        g = z.clone()
        ops.ce_fwd_bwd(g, ctx.V, tgt, ctx.eps, 1.0 / rows, grad_out.reshape(1).float().contiguous(), scratch, None, 0.0, True)
        return g[:, :ctx.V].to(ctx.dtype), None, None


class LabelSmoothingLoss(nn.Module):
    """src/utils.py:22-38 on the fused soft-max cross-entropy kernel: `LabelSmoothingLoss(classes, smoothing)(pred, target)`
    with pred [rows, classes] logits -> mean over rows of sum_v -dist_v log_softmax(pred)_v (pad rows are NOT ignored).
    The kernel reads bf16 logits; the gradient w.r.t. `pred` is available through autograd."""

    def __init__(self, classes, smoothing=0.0, dim=-1):
        super().__init__()
        self.confidence = 1.0 - smoothing
        self.smoothing = smoothing
        self.cls = classes
        self.dim = dim

    def forward(self, pred, target):
        if not pred.is_cuda:
            raise RuntimeError("mmsum_b200 has no CPU path: LabelSmoothingLoss needs CUDA tensors")
        if pred.dim() != 2 or pred.shape[1] != self.cls or self.dim not in (-1, 1):
            raise ValueError("pred must be [rows, classes] with the class axis last")
        return _LSLossFn.apply(pred, target, float(self.smoothing))


# ---------------------------------------------------------------------------------------------- training steps
class _StepFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, module, batch, label_smoothing):
        eng = module.engine
        loss = eng.forward_step(batch, label_smoothing, module.training)
        ctx.engine = eng
        ctx.generation = eng.fwd_generation
        return loss.reshape(()).clone()

    @staticmethod
    def backward(ctx, grad_out):
        eng = ctx.engine
        if ctx.generation != eng.fwd_generation:
            raise RuntimeError("backward() of a stale step: another forward ran on this model since this loss was computed "
                               "(the engine keeps the activations of ONE step); call backward before the next forward")
        eng.backward_step(grad_out.contiguous().float())
        return None, None, None, None


def _ids(t):
    return t.to(torch.int64).contiguous()


def _check_device(dev, *tensors):
    for t in tensors:
        if t is not None and t.device != dev:
            raise RuntimeError("all step inputs must live on %s (got a tensor on %s)" % (dev, t.device))


def _load(path):
    return torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu")


class MultimodalSum(nn.Module, _EngineRoot):
    """`MultimodalSum(bart_pretrained, table_pretrained, img_pretrained, TableEncoder)` as in src/multimodal_train.py:111-122.

    `*_pretrained` are local checkpoint directories holding `pytorch_model.bin` (no hub download in this build; `None`
    = random init by the reference's recipe).  `config` selects the model dims (default: cfg/bart-large.json values).
    `label_smoothing` replaces the reference's module-global `args.label_smoothing` (default 0.1, :433)."""

    def __init__(self, bart_pretrained=None, table_pretrained=None, img_pretrained=None, TableEncoder=YelpTableEncoder,
                 config: ModelConfig = None, label_smoothing=0.1):
        super().__init__()
        ds = "yelp" if TableEncoder is YelpTableEncoder else "amazon"
        cfg = config if config is not None else ModelConfig(dataset=ds)
        if cfg.dataset != ds:
            raise ValueError("config.dataset %r does not match the TableEncoder (%s)" % (cfg.dataset, ds))
        self.cfg = cfg
        self.label_smoothing = label_smoothing
        self.bart_model = BartForMultiEncConditionalGeneration(cfg)
        if bart_pretrained is not None:
            self.bart_model.load_state_dict(_load(bart_pretrained), strict=False)  # alpha/beta_proj are authorized missing keys (:2183)
        self.table_encoder = TableEncoder(self.bart_model.model.shared)
        if table_pretrained is not None:
            self.table_encoder.load_state_dict(_load(table_pretrained))
        self.img_encoder = Resnet(cfg.d_model)
        if img_pretrained is not None:
            self.img_encoder.load_state_dict(_load(img_pretrained), strict=False)
        self.engine = None
        self._adopt_children()

    def forward(self, reviews, reviews_mask, reviews_rating, field, field_value, img, img_mask, max_review_len=None, **unused):
        """-> (loss,)  — same arguments as the reference (src/multimodal_train.py:124-139); `img` holds pooled
        ResNet-101 stage-3 features [B, max_imgs, 196, 1024] (fp32 or bf16).  `max_review_len` (optional, not in the reference):
        what the collate function knows — no review has a valid token at or beyond that position; the encoder then runs on
        frames trimmed to it without the engine reading the mask back from the device."""
        eng = self._ensure_engine(reviews.device)
        _check_device(reviews.device, reviews_mask, reviews_rating, field, img, img_mask, *field_value)
        if max_review_len is None:
            max_review_len = getattr(reviews_mask, "max_review_len", None)      # attached by prefetch.*_data_prefetcher
        batch = Batch(_ids(reviews), _ids(reviews_mask), reviews_rating.float().contiguous(), _ids(field),
                      [_ids(v) for v in field_value], img if img.dtype == torch.bfloat16 else img.float(),
                      img_mask.to(torch.bool).contiguous(), max_review_len=max_review_len)
        loss = _StepFn.apply(eng.step_anchor(), self, batch, self.label_smoothing)
        return (loss,)

    @torch.no_grad()
    def get_multimodal_outputs(self, reviews, reviews_mask, field, field_value, img, img_mask):
        """src/multimodal_train.py:165-193 -> (n_reviews, text_hiddens [B,R,S,D], text_attention_mask [B,R,S],
        table_hiddens [B,1,F,D], table_attention_mask [B,1,F], img_hiddens [B,n,196,D], img_attention_mask [B,n,196])."""
        bsz, n_reviews, seq_len = reviews.size()
        text_hiddens = self.bart_model.model.encoder(input_ids=reviews.reshape(bsz * n_reviews, seq_len),
                                                     attention_mask=reviews_mask.reshape(bsz * n_reviews, seq_len))[0]
        text_hiddens = text_hiddens.reshape(bsz, n_reviews, seq_len, -1)
        table_hiddens, table_attention_mask = self.table_encoder(field, field_value)
        img_hiddens = self.img_encoder(img)
        img_attention_mask = None
        if img_mask is not None:
            img_attention_mask = img_mask.unsqueeze(-1).repeat([1, 1, img_hiddens.size(2)])
        return (n_reviews, text_hiddens, reviews_mask, table_hiddens.unsqueeze(1), table_attention_mask.unsqueeze(1),
                img_hiddens, img_attention_mask)


class TextSupervised(nn.Module, _EngineRoot):
    """Text-only step of src/text_pretrain.py:66-113 (BASELINE config 1): same engine, one text memory,
    plain cross-entropy unless `label_smoothing` is given."""

    def __init__(self, bart_pretrained=None, config: ModelConfig = None, label_smoothing=None):
        super().__init__()
        cfg = config if config is not None else ModelConfig(dataset="text")
        if cfg.dataset != "text":
            raise ValueError("TextSupervised needs config.dataset == 'text'")
        self.cfg = cfg
        self.label_smoothing = label_smoothing
        self.bart_model = BartForEncConditionalGeneration(cfg)
        if bart_pretrained is not None:
            self.bart_model.load_state_dict(_load(bart_pretrained), strict=False)
        self.engine = None
        self._adopt_children()

    def forward(self, reviews, reviews_mask, reviews_rating, max_review_len=None, **unused):
        eng = self._ensure_engine(reviews.device)
        _check_device(reviews.device, reviews_mask, reviews_rating)
        if max_review_len is None:
            max_review_len = getattr(reviews_mask, "max_review_len", None)      # attached by prefetch.text_data_prefetcher
        batch = Batch(_ids(reviews), _ids(reviews_mask), reviews_rating.float().contiguous(), max_review_len=max_review_len)
        loss = _StepFn.apply(eng.step_anchor(), self, batch, self.label_smoothing)
        return (loss,)


class ImgSupervised(nn.Module, _EngineRoot):
    """Image pretraining stage, src/img_pretrain.py:85-141: the single-memory decoder attends to the projected image
    features of a business and is trained to emit one of its reviews (`labels`); rating_diff = 0.  The reference trains
    only `img_encoder` in this stage (`get_optimizer(..., model.img_encoder.named_parameters(), ...)`, BART frozen)."""

    def __init__(self, bart_pretrained=None, config: ModelConfig = None, label_smoothing=0.1):
        super().__init__()
        cfg = config if config is not None else ModelConfig(dataset="img")
        if cfg.dataset != "img":
            raise ValueError("ImgSupervised needs config.dataset == 'img'")
        self.cfg = cfg
        self.label_smoothing = label_smoothing
        self.bart_model = BartForEncConditionalGeneration(cfg)
        if bart_pretrained is not None:
            self.bart_model.load_state_dict(_load(bart_pretrained), strict=False)
        self.img_encoder = Resnet(cfg.d_model)
        self.engine = None
        self._adopt_children()

    def forward(self, input_imgs, input_imgs_mask=None, decoder_input_ids=None, decoder_attention_mask=None,
                decoder_past_key_values=None, labels=None, **unused):
        """input_imgs: pooled features [B, max_imgs, 196, 1024]; input_imgs_mask [B, max_imgs]; labels [B, 128] -> (loss,)."""
        if labels is None:
            raise ValueError("ImgSupervised.forward is the training step: labels are required")
        eng = self._ensure_engine(input_imgs.device)
        B, n = input_imgs.shape[:2]
        mask = torch.ones(B, n, dtype=torch.bool, device=input_imgs.device) if input_imgs_mask is None else input_imgs_mask
        _check_device(input_imgs.device, mask, labels)
        batch = Batch(None, None, None, img=input_imgs if input_imgs.dtype == torch.bfloat16 else input_imgs.float(),
                      img_mask=mask.to(torch.bool).contiguous(), labels=_ids(labels))
        return (_StepFn.apply(eng.step_anchor(), self, batch, self.label_smoothing),)


class TableSupervised(nn.Module, _EngineRoot):
    """Table pretraining stage, src/table_pretrain.py:84-129: memory = the table encoder's output (one entity of 47 / 133
    field rows), target = one review of the business, rating_diff = 0."""

    def __init__(self, bart_pretrained=None, TableEncoder=YelpTableEncoder, config: ModelConfig = None, label_smoothing=0.1):
        super().__init__()
        ds = "table_yelp" if TableEncoder is YelpTableEncoder else "table_amazon"
        cfg = config if config is not None else ModelConfig(dataset=ds)
        if cfg.dataset != ds:
            raise ValueError("config.dataset %r does not match the TableEncoder (%s)" % (cfg.dataset, ds))
        self.cfg = cfg
        self.label_smoothing = label_smoothing
        self.bart_model = BartForEncConditionalGeneration(cfg)
        if bart_pretrained is not None:
            self.bart_model.load_state_dict(_load(bart_pretrained), strict=False)
        self.table_encoder = TableEncoder(self.bart_model.model.shared)
        self.engine = None
        self._adopt_children()

    def forward(self, field, field_value, decoder_input_ids=None, decoder_attention_mask=None, decoder_past_key_values=None,
                labels=None, **unused):
        if labels is None:
            raise ValueError("TableSupervised.forward is the training step: labels are required")
        eng = self._ensure_engine(field.device)
        _check_device(field.device, labels, *field_value)
        batch = Batch(None, None, None, field=_ids(field), field_value=[_ids(v) for v in field_value], labels=_ids(labels))
        return (_StepFn.apply(eng.step_anchor(), self, batch, self.label_smoothing),)
