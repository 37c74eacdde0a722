"""Step engine: orchestrates the hand-written CUDA kernels (through the C-ABI) into the forward and backward of
MultimodalSum.forward (reference: src/multimodal_train.py:124-163).

B200-first design decisions (see DESIGN.md):
  * batched leave-one-out: the reference's 9 sequential decoder passes are ONE decoder pass over 9·B sequences in
    which target i simply does not see review i (SURVEY App. F) — decoder GEMMs get M = 9·B·128 rows and the
    cross-attention K/V of every memory token is projected once per layer instead of 9 times;
  * one K|V GEMM per layer over the concatenated text+table+image memory (k/v projections are shared by the modalities);
  * parameters live in three flat arenas (fp32 master, bf16 compute copy, fp32 gradient) ordered by the time their
    gradients become final in backward, so data-parallel buckets are contiguous slices that can be all-reduced while
    backward is still running; fused weights (q|k|v, k|v) are adjacent in the arena so one GEMM serves them;
  * activations are token-major [rows, 1024] bf16, saved per layer (≈1.2 GB / decoder layer at 16 businesses) — no
    recomputation; all workspaces are allocated once per shape.
torch is used for memory (arenas, workspaces), streams and torch.distributed only.
"""
import math
import os
import types
import weakref

import torch

from . import layers as L
from . import ops
from .synth import ModelConfig

ALIGN = 64


def _arena_order(cfg: ModelConfig):
    """Parameter names (reference state_dict keys, SURVEY App. B) in backward-completion order."""
    names = []
    bm = "bart_model.model."

    def self_attn(lp):
        a = lp + "self_attn."
        return [a + "out_proj.weight", a + "out_proj.bias",
                a + "q_proj.weight", a + "k_proj.weight", a + "v_proj.weight",
                a + "q_proj.bias", a + "k_proj.bias", a + "v_proj.bias",
                lp + "self_attn_layer_norm.weight", lp + "self_attn_layer_norm.bias"]

    def ffn(lp):
        return [lp + "fc2.weight", lp + "fc2.bias", lp + "fc1.weight", lp + "fc1.bias",
                lp + "final_layer_norm.weight", lp + "final_layer_norm.bias"]

    for i in reversed(range(cfg.decoder_layers)):
        lp = bm + "decoder.layers.%d." % i
        names += ffn(lp)
        c = lp + "encoder_attn."
        if cfg.multimodal:
            names += [c + "alpha_proj.weight", c + "alpha_proj.bias", c + "beta_proj.weight", c + "beta_proj.bias"]
        names += [c + "out_proj.weight", c + "out_proj.bias", c + "q_proj.weight", c + "q_proj.bias",
                  c + "k_proj.weight", c + "v_proj.weight", c + "k_proj.bias", c + "v_proj.bias",
                  lp + "encoder_attn_layer_norm.weight", lp + "encoder_attn_layer_norm.bias"]
        names += self_attn(lp)
    names += [bm + "decoder.layernorm_embedding.weight", bm + "decoder.layernorm_embedding.bias",
              bm + "decoder.rating_embeddings", bm + "decoder.embed_positions.weight"]
    if cfg.table is not None:
        t = "table_encoder."
        names += [t + "linear.weight", t + "fc.weight", t + "fc.bias"]
        names += [t + "rating_embedding.weight", t + ("hours_embedding.weight" if cfg.table == "yelp" else "price_embedding.weight")]
    if cfg.image:
        names += ["img_encoder.linear.weight"]
    for i in reversed(range(cfg.encoder_layers)):
        lp = bm + "encoder.layers.%d." % i
        names += ffn(lp)
        names += self_attn(lp)
    names += [bm + "encoder.layernorm_embedding.weight", bm + "encoder.layernorm_embedding.bias",
              bm + "encoder.embed_positions.weight", bm + "shared.weight"]
    return names


def backward_plan(cfg: ModelConfig, names, trainable):
    """Which parts of the backward run when only the parameters in `trainable` want a gradient: autograd's rule, a gradient is
    computed iff it reaches a trainable parameter.  A pure function of the configuration, the arena's parameter names and the
    trainable set.
      grads    parameters whose gradient the backward writes (the trainable ones the step reaches)
      dgrad    activation gradients of the dgrad chain that are computed, by label: "dec.<l>.ffn.dH" (fc2 dgrad), "dec.<l>.ffn.in"
               (d of the block input), "dec.<l>.cross.dU" / ".dO3" / ".dA3" / ".in", "dec.<l>.self.dctx" / ".in", the same for
               "enc.<l>.", "head.in" (LM-head dgrad), "table.dtab_h", "table.dtabX"
      mem      per memory modality: whether its rows of the memory gradient are needed (its producer has a trainable parameter)
      dkv      per decoder layer: the modalities whose cross-attention dK/dV runs
      dec_in / enc_in   whether the gradient into layer l's input is needed (index n_layers = the stack's output)"""
    bm = "bart_model.model."
    enc, dec, shared = bm + "encoder.", bm + "decoder.", bm + "shared.weight"
    names = list(names)
    tset = frozenset(trainable) & frozenset(names)
    tr = lambda n: n in tset                                           # noqa: E731
    anyp = lambda *pre: any(n.startswith(pre) for n in tset)            # noqa: E731
    text, table, image = cfg.text_memory, cfg.table is not None, cfg.image
    mods = [m for m, on in (("text", text), ("table", table), ("image", image)) if on]
    mem = {"text": text and (anyp(enc) or tr(shared)), "table": table and anyp("table_encoder."),
           "image": image and tr("img_encoder.linear.weight")}
    mem_any = any(mem.values())
    dgrad = set()

    def ffn(tag, lp, need_in):
        if tr(lp + "fc1.weight") or tr(lp + "fc1.bias") or need_in:
            dgrad.add(tag + "ffn.dH")
        if need_in:
            dgrad.add(tag + "ffn.in")

    def self_attn(tag, lp, need_in):
        s = lp + "self_attn."
        if anyp(s + "q_proj.", s + "k_proj.", s + "v_proj.") or need_in:
            dgrad.add(tag + "self.dctx")
        if need_in:
            dgrad.add(tag + "self.in")

    # decoder: layer l's input gradient is needed when anything trainable lies below it (memory producers included: the
    # cross-attention dK/dV of the layers below needs the chain)
    L_d = cfg.decoder_layers
    dec_in = [tr(shared) or anyp(dec + "embed_positions.", dec + "rating_embeddings", dec + "layernorm_embedding.")]
    for l in range(L_d):
        dec_in.append(dec_in[l] or anyp(dec + "layers.%d." % l) or mem_any)
    dkv = []
    for l in range(L_d):
        lp, tag = dec + "layers.%d." % l, "dec.%d." % l
        c = lp + "encoder_attn."
        if not dec_in[l + 1]:
            dkv.append(())
            continue
        self_out = dec_in[l] or anyp(lp + "self_attn.", lp + "self_attn_layer_norm.")
        cross_out = self_out or anyp(c, lp + "encoder_attn_layer_norm.") or mem_any
        ffn(tag, lp, cross_out)
        if cross_out:
            kv = anyp(c + "k_proj.", c + "v_proj.")
            want = tuple(m for m in mods if kv or mem[m])
            dA3 = tr(c + "q_proj.weight") or tr(c + "q_proj.bias") or self_out or bool(want)
            dO3 = tr(c + "out_proj.weight") or tr(c + "out_proj.bias") or dA3
            if cfg.multimodal and (anyp(c + "alpha_proj.", c + "beta_proj.") or dO3):
                dgrad.add(tag + "cross.dU")
            dgrad.update(t for t, on in ((tag + "cross.dO3", dO3), (tag + "cross.dA3", dA3), (tag + "cross.in", self_out)) if on)
            dkv.append(want if dA3 else ())
        else:
            dkv.append(())
        if self_out:
            self_attn(tag, lp, dec_in[l])
    if dec_in[L_d]:
        dgrad.add("head.in")
    if mem["table"]:
        t = "table_encoder."
        emb = tr(t + "rating_embedding.weight") or tr(t + "hours_embedding.weight") or tr(t + "price_embedding.weight")
        if anyp(t + "fc.") or emb:
            dgrad.add("table.dtab_h")
        if emb:
            dgrad.add("table.dtabX")
    # encoder: runs down to the lowest layer with something trainable at or below it (the embeddings count as below layer 0)
    enc_in = []
    if mem["text"]:
        enc_in = [tr(shared) or anyp(enc + "embed_positions.", enc + "layernorm_embedding.")]
        for l in range(cfg.encoder_layers):
            enc_in.append(enc_in[l] or anyp(enc + "layers.%d." % l))
        for l in range(cfg.encoder_layers):
            lp, tag = enc + "layers.%d." % l, "enc.%d." % l
            if enc_in[l + 1]:
                self_out = enc_in[l] or anyp(lp + "self_attn.", lp + "self_attn_layer_norm.")
                ffn(tag, lp, self_out)
                if self_out:
                    self_attn(tag, lp, enc_in[l])
    grads = frozenset(n for n in tset if text or not n.startswith(enc))
    return types.SimpleNamespace(trainable=tset, grads=grads, dgrad=frozenset(dgrad), mem=mem, dkv=tuple(dkv),
                                 dec_in=tuple(dec_in), enc_in=tuple(enc_in), run=dec_in[L_d] or tr(shared))


class _Pool:
    """Free-list of equally shaped scratch tensors.  The step runs on one stream (plus the bias-gradient side stream,
    which `before_put` joins), so a buffer may be handed out again as soon as its last consumer has been enqueued."""

    def __init__(self, n, shape, device):
        self.free = [torch.empty(shape, device=device, dtype=torch.bfloat16) for _ in range(n)]
        self.before_put = None

    def get(self):
        if not self.free:
            raise RuntimeError("scratch pool exhausted (a buffer was not returned with put())")
        return self.free.pop()

    def put(self, *ts):
        if self.before_put is not None:
            self.before_put()
        for t in ts:
            if t is not None and all(t is not f for f in self.free):
                self.free.append(t)


class _PoolRows:
    """The same free-list handing out the first `rows` rows of its buffers (encoder-sized operands: a GEMM's M is the row count
    of its tensors)."""

    def __init__(self, base, rows):
        self.base, self.rows = base, rows
        self.out = {}

    def get(self):
        b = self.base.get()
        v = b[:self.rows]
        self.out[v.data_ptr()] = b
        return v

    def put(self, *ts):
        self.base.put(*[self.out.pop(t.data_ptr(), t) for t in ts if t is not None])


class StepEngine:
    def __init__(self, cfg: ModelConfig, device="cuda"):
        if cfg.d_model != 1024 or cfg.head_dim != 64:
            raise ValueError("kernels are specialised to d_model 1024 / head_dim 64 (bart-large)")
        self.cfg = cfg
        self.device = torch.device(device)
        self.names = _arena_order(cfg)
        self.shapes = {}
        self.offsets = {}
        self.numel = 0
        self.bound = False
        self.ws = None
        self.ws_full = None
        # A/B switch (default = the faster variant, DESIGN.md section 2)
        self.trim_frames = os.environ.get("MMSUM_TRIM_FRAMES", "1") != "0"
        self._len_cache = None
        self.ws_key = None
        # dropout stream = f(seed, step_count, layer, element): the seed follows torch.manual_seed / torch.initial_seed and
        # differs per data-parallel rank; `seed` and `step_count` are plain attributes so a resume can restore them
        self.seed = self._default_seed()
        self.step_count = 0
        self.fwd_generation = 0          # bumped by every forward; backward refuses to run on a stale workspace
        self.dropout = cfg.dropout
        self.grad_ready_hook = None      # callable(lo, hi): gradient arena range [lo, hi) is final (data-parallel buckets)
        self.graph_mode = False          # replay forward / backward from recorded CUDA graphs (see forward_step)
        # torch.are_deterministic_algorithms_enabled() as read by the last forward: its backward then runs the ordered
        # (bitwise-reproducible) reductions, with their fp32 scratch (main stream / bias-gradient stream) sized per step shape
        self.det = False
        self.det_ws = None
        self.det_ws_side = None
        self._det_sized = set()
        # the parameters that require grad, as read by the last forward, and the backward plan of that set (backward_plan)
        self.trainable = frozenset()
        self.plan = None
        self._plans = {}
        self._graphs = {}
        self._graph_entry = None
        self._w16_fresh = False          # True only right after a fused optimizer wrote W16 itself
        self._w16_versions = -1
        self.anchor = None
        # bias-gradient side stream (see _bias_grad); MMSUM_BIAS_SIDE_STREAM=0 keeps everything on one stream
        self.side_stream = None
        self._side_pending = False
        if self.device.type == "cuda" and os.environ.get("MMSUM_BIAS_SIDE_STREAM", "1") != "0":
            prio = int(os.environ.get("MMSUM_SIDE_PRIORITY", "-1"))   # high priority: its short kernels slot in at once
            self.side_stream = torch.cuda.Stream(device=self.device, priority=prio)
            self._ev_main = torch.cuda.Event()
            self._ev_side = torch.cuda.Event()

    # ------------------------------------------------------------------ parameters
    def bind(self, named_params):
        """Move the parameters into the flat arenas and re-point `.data` at the arena views."""
        named = dict(named_params)
        off = 0
        # a stand-alone BartFor*ConditionalGeneration owns no table / image encoder: those arena entries are dropped
        self.names = [n for n in self.names if n in named or not n.startswith(("table_encoder.", "img_encoder."))]
        for n in self.names:
            if n not in named:
                raise KeyError("parameter %s missing" % n)
            self.shapes[n] = tuple(named[n].shape)
            self.offsets[n] = off
            off += (named[n].numel() + ALIGN - 1) // ALIGN * ALIGN
        extra = set(named) - set(self.names)
        if extra:
            raise KeyError("unexpected parameters: %s" % sorted(extra)[:4])
        self.numel = off
        dev = self.device
        self.W32 = torch.zeros(off, device=dev, dtype=torch.float32)
        self.W16 = torch.empty(off, device=dev, dtype=torch.bfloat16)
        self.G32 = torch.zeros(off, device=dev, dtype=torch.float32)
        self.params = {}
        with torch.no_grad():
            for n in self.names:
                p = named[n]
                v = self.w32(n)
                v.copy_(p.data.to(device=dev, dtype=torch.float32))
                p.data = v
                self.params[n] = p
        self.anchor = torch.zeros(1, device=dev, requires_grad=True)
        self.trainable = frozenset(n for n, p in self.params.items() if p.requires_grad)
        self._plans = {}
        self._ln_sink = torch.empty(2, self.cfg.d_model, device=dev, dtype=torch.float32)  # gamma / beta of a half-frozen LayerNorm
        self.step_dev = torch.full((1,), self.step_count, device=dev, dtype=torch.int32)   # dropout step counter, incremented by every forward
        self.bound = True
        self._w16_fresh = False

    def _view(self, arena, n, n2=None):
        o = self.offsets[n]
        if n2 is None:
            return arena[o:o + math.prod(self.shapes[n])].view(self.shapes[n])
        # fused view over adjacent tensors n..n2 (same trailing dims, no padding in between)
        o2 = self.offsets[n2] + math.prod(self.shapes[n2])
        tail = self.shapes[n][1:]
        return arena[o:o2].view((-1,) + tail)

    def w32(self, n, n2=None):
        return self._view(self.W32, n, n2)

    def w16(self, n, n2=None):
        return self._view(self.W16, n, n2)

    def g32(self, n, n2=None):
        return self._view(self.G32, n, n2)

    @staticmethod
    def _default_seed():
        rank = 0
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                rank = dist.get_rank()
            else:
                rank = int(os.environ.get("RANK", "0"))
        except Exception:
            rank = 0
        return (torch.initial_seed() ^ (0x5EED + rank * 0x9E3779B97F4A7C15)) & 0xFFFFFFFFFFFFFFFF

    def rng_state(self):
        """What the dropout masks of the next step depend on besides the layer / element index: saved by
        train_utils.save_checkpoint, so a resumed run draws the masks the uninterrupted run would have drawn."""
        return {"seed": int(self.seed), "step_count": int(self.step_count)}

    def set_rng_state(self, state):
        self.seed = int(state["seed"]) & 0xFFFFFFFFFFFFFFFF
        self.step_count = int(state["step_count"])
        if getattr(self, "step_dev", None) is not None:
            self.step_dev.fill_(self.step_count)
        self._graphs.clear()                      # recorded graphs baked the old seed into their kernel arguments
        self._graph_entry = None

    def _param_versions(self):
        return sum(p._version for p in self.params.values())

    def refresh_bf16_weights(self, force=False):
        """Re-cast the fp32 masters into the bf16 compute copy.  The masters are updated through the Parameters
        (`p.data.addcdiv_` in transformers' AdamW, torch.optim, load_state_dict, ...), which the arena's own version counter
        never sees, so the cast runs on EVERY call (2.8 GB of traffic, < 0.5 ms) unless a fused optimizer that writes W16
        itself has just declared it fresh (`mark_w16_fresh`) and no Parameter has been written in place since."""
        vs = self._param_versions()
        if force or not self._w16_fresh or vs != self._w16_versions:
            ops.cast_bf16(self.W32, self.W16)
        self._w16_fresh = False
        self._w16_versions = vs

    def mark_w16_fresh(self):
        self._w16_fresh = True
        self._w16_versions = self._param_versions()

    def mark_weights_dirty(self):
        self._w16_fresh = False

    # ------------------------------------------------------------------ trainable set (requires_grad)
    def _read_trainable(self):
        """Read which parameters require grad (at every forward, like the deterministic switch) and select the backward plan of
        that set.  A parameter that has just been frozen gets its arena range zeroed: nothing writes it afterwards, so the fused
        clip and the data-parallel buckets see zeros there."""
        t = frozenset(n for n, p in self.params.items() if p.requires_grad)
        if t != self.trainable:
            with torch.no_grad():
                for n in self.trainable - t:
                    self.g32(n).zero_()
            self.trainable = t
        plan = self._plans.get(t)
        if plan is None:
            plan = self._plans[t] = backward_plan(self.cfg, self.names, t)
            plan.grad_ranges = self._merged_ranges(n for n in self.names if n in t)
        self.plan = plan
        return plan

    def _merged_ranges(self, names):
        out = []
        for n in names:
            lo = self.offsets[n]
            hi = lo + (math.prod(self.shapes[n]) + ALIGN - 1) // ALIGN * ALIGN
            if out and out[-1][1] == lo:
                out[-1][1] = hi
            else:
                out.append([lo, hi])
        return [tuple(r) for r in out]

    def grad_ranges(self):
        """Arena ranges [lo, hi) of the trainable parameters, adjacent ones merged, in arena order (data-parallel buckets)."""
        return (self.plan or self._read_trainable()).grad_ranges

    def step_anchor(self):
        """The autograd input of a training step: detached when no parameter requires grad, so the loss does not either (as in
        torch: its backward() then raises)."""
        return self.anchor if any(p.requires_grad for p in self.params.values()) else self.anchor.detach()

    def _point_grads(self):
        """`.grad` of a trainable parameter is its arena view; a frozen parameter's is None."""
        tset = self.plan.trainable
        for n, p in self.params.items():
            if n in tset:
                if p.grad is None:
                    p.grad = self.g32(n)
            elif p.grad is not None:
                p.grad = None

    # ------------------------------------------------------------------ workspaces
    def _frame_view(self, full, S_enc):
        """Views of the full-size workspace for a step whose encoder runs on S_enc-row frames (see _alloc): every encoder
        buffer, the memory and its per-layer K|V / gradient buffers cut to the rows this step uses.  The storage never moves,
        so recorded CUDA graphs of different frames stay valid side by side; the views are built once per frame."""
        if S_enc == full["S"] or full["Tt"] == 0:
            return full
        views = full.setdefault("_views", {})
        if S_enc in views:
            return views[S_enc]
        B, R, F, n_img, ik = full["B"], full["R"], full["F"], full["n_img"], full["img_keys"]
        Te = B * R * S_enc
        Tm = Te + B * F + B * n_img * ik
        w = dict(full)
        w.update(S_enc=S_enc, Te=Te, Tt=Te, Tm=Tm)
        cut = lambda t, n: t[:n] if isinstance(t, torch.Tensor) else t
        w["enc"] = [{k: (v if k == "lse" else cut(v, Te)) for k, v in a.items()} for a in full["enc"]]
        for k in ("enc_x0", "enc_m0", "enc_r0"):
            w[k] = full[k][:Te]
        w["dec"] = [dict(a, kv=a["kv"][:Tm]) for a in full["dec"]]
        for k in ("MEM", "dkv_all", "dMEM16", "mem_valid"):
            if k in full:
                w[k] = full[k][:Tm]
        w["pool_e"] = _PoolRows(full["pool"], Te)
        views[S_enc] = w
        return w

    def _alloc(self, B, R, S, F, n_img, img_keys, S_enc=None):
        """Workspaces of one step shape.  B businesses, R decoder sequences per business (the leave-one-out targets; 1 in
        the img / table stages), S = 128; memory rows = [text B*R*S_enc (when the model has a text memory) | table B*F | image].
        S_enc <= S is the ENCODER frame: when no review of the batch is longer than S_enc tokens, the encoder (and the text
        rows of the memory) run on B*R*S_enc rows — rows beyond a review's last token are pad in every review, are masked as
        keys everywhere and receive exactly zero gradient, so dropping them changes no result (the decoder keeps its 128-row
        frames: its pad rows count in the loss, quirk Q2)."""
        S_enc = S if S_enc is None else S_enc
        key = (B, R, S, F, n_img, img_keys)
        if self.ws_key == key:
            return self._frame_view(self.ws_full, S_enc)
        self.ws_full = None
        S_enc_req, S_enc = S_enc, S              # storage for full frames; the step works on views cut to its frame
        self.ws, self.ws_key = None, None       # drop the old workspace before allocating the new one
        cfg, dev = self.cfg, self.device
        D, FF, H = cfg.d_model, cfg.ffn_dim, cfg.heads
        T = B * R * S
        has_text = cfg.text_memory
        Te = B * R * S_enc                        # encoder rows
        Tt = Te if has_text else 0
        Tm = Tt + B * F + B * n_img * img_keys
        N = B * R
        Et = (R if has_text else 0) + (1 if F > 0 else 0) + n_img
        nm = int(has_text) + int(F > 0) + int(n_img > 0)
        bf = lambda *s: torch.empty(s, device=dev, dtype=torch.bfloat16)
        f32 = lambda *s: torch.empty(s, device=dev, dtype=torch.float32)
        u8 = lambda *s: torch.zeros(s, device=dev, dtype=torch.uint8)
        i32 = lambda *s: torch.zeros(s, device=dev, dtype=torch.int32)
        w = dict(B=B, R=R, S=S, F=F, n_img=n_img, img_keys=img_keys, T=T, Tt=Tt, Tm=Tm, N=N, Et=Et, nm=nm, S_enc=S_enc, Te=Te)
        w.update(enc_ids=i32(T), dec_ids=i32(T), labels=i32(T), enc_valid=u8(T), dec_valid=u8(T), mem_valid=u8(Tm),
                 ent_valid=u8(B, Et), pres=u8(B, 2), rating_diff=f32(N), inv_n=f32(N, nm))
        w["MEM"] = bf(Tm, D)
        if F > 0:
            w.update(tabX=bf(B * F, 2 * D), tab_valid=u8(B, F), tab_h=bf(B * F, D))
        if n_img > 0:
            w.update(img16=bf(B * n_img * img_keys, 1024))
        L_e, L_d = (cfg.encoder_layers if has_text else 0), cfg.decoder_layers
        enc = []
        for l in range(L_e):
            enc.append(dict(x=bf(Te, D) if l > 0 else None, qkv=bf(Te, 3 * D), ctx=bf(Te, D), o=bf(Te, D), x1=bf(Te, D), h=bf(Te, FF),
                            a=bf(Te, FF), f=bf(Te, D), lse=f32(N, H, 1, S), m1=f32(Te), r1=f32(Te), m2=f32(Te), r2=f32(Te)))
        w["enc"] = enc
        if has_text:
            w["enc_x0"] = bf(Te, D)
            w["enc_m0"], w["enc_r0"] = f32(Te), f32(Te)
        dec = []
        U = bf(2, T, D) if cfg.multimodal else None      # gate pre-activations: forward scratch shared by the layers
        for l in range(L_d):
            d = dict(x=bf(T, D), qkv=bf(T, 3 * D), ctx=bf(T, D), o=bf(T, D), x1=bf(T, D), qc=bf(T, D), kv=bf(Tm, 2 * D),
                     A3=bf(nm, T, D), O3=bf(nm, T, D), x2=bf(T, D), h=bf(T, FF), a=bf(T, FF), f=bf(T, D),
                     lse=f32(N, H, 1, S), lse_c=f32(N, H, Et, S),
                     m1=f32(T), r1=f32(T), m2=f32(T), r2=f32(T), m3=f32(T), r3=f32(T))
            if cfg.multimodal:
                d.update(U=U, AB=bf(2, T, D), yc=bf(T, D))
            dec.append(d)
        w["dec"] = dec
        w["dec_m0"], w["dec_r0"] = f32(T), f32(T)
        w["x_out"] = bf(T, D)
        self.ldv = (cfg.vocab_size + 7) // 8 * 8
        w["logits"] = bf(T, self.ldv)
        w["loss_rows"] = f32(T)
        w["lse_rows"] = f32(T)
        w["loss"] = f32(1)
        # backward scratch
        w["pool"] = _Pool(5, (T, D), dev)
        w["pool"].before_put = self._side_join
        w["pool_e"] = w["pool"]                    # (a frame view hands out row-cut views of the same buffers)
        w["dH"] = bf(T, FF)
        w["dqkv"] = bf(T, 3 * D)
        # cross-attention K|V gradients of ALL decoder layers side by side: the memory gradient is then ONE GEMM over the
        # concatenated K (sum_l dkv_l W_l = [dkv_0 | dkv_1 | ...] [W_0; W_1; ...]) instead of L fp32 read-modify-write passes
        # over a [Tm, D] accumulator (TMA reduce-add: 2.5 ms per step at config 2, against 1.75 ms for the single product)
        w["dkv_all"] = bf(Tm, L_d * 2 * D)
        w["Wkv_cat"] = bf(L_d * 2 * D, D)
        w["delta"] = f32(N, H, Et, S)
        w["dMEM16"] = bf(Tm, D)
        w["dz32"] = f32(T, D)
        w["dA3"] = bf(nm, T, D)
        w["dO3"] = bf(nm, T, D)
        if cfg.multimodal:
            w.update(dU=bf(2, T, D), dca=bf(T, 2 * D), dcb=bf(T, 2 * D))
        if F > 0:
            w.update(dtab_h=bf(B * F, D), dtabX=bf(B * F, 2 * D))
        self.ws_full, self.ws_key = w, key
        return self._frame_view(w, S_enc_req)

    # ------------------------------------------------------------------ helpers
    def _sid(self, kind, layer):
        # the step number is added inside the kernels from the device-resident counter `step_dev` (graph-replayable)
        return kind * 64 + layer

    def _self_attn_args(self, w, qkv, out, lse, key_valid, causal, dqkv=None, frame=None):
        """frame: rows per sequence (the encoder's trimmed frame; None = 128).  dqkv: the backward's gradient buffer."""
        D, S = self.cfg.d_model, w["S"]
        fr = S if frame is None else frame
        bwd = {} if dqkv is None else dict(DELTA=w["delta"], dQ=dqkv, lddq=3 * D, dq_col=0, dKV=dqkv, lddkv=3 * D, dk_col=D,
                                           dv_col=2 * D)
        return L.self_attn_args(self, qkv, out, lse, key_valid, w["N"], causal, fr, q_rows=(0 if fr == S else fr), **bwd)

    def _cross_attn_args(self, w, qc, kv, out3, lse, dqc=None, dkv=None, no_dkv=None):
        """Memory rows = [text B*R*S_enc (leave-one-out over the R reviews of a business) | table B*F | image].  no_dkv (backward):
        per modality, whether its dK/dV is skipped."""
        D, B, R, F, n_img, Tt = self.cfg.d_model, w["B"], w["R"], w["F"], w["n_img"], w["Tt"]
        mods = ([(0, R, w["S_enc"])] if Tt > 0 else []) + ([(Tt, 1, F)] if F > 0 else []) + \
               ([(Tt + B * F, n_img, w["img_keys"])] if n_img > 0 else [])
        bwd = {} if dqc is None else dict(DELTA=w["delta"], dQ=dqc, lddq=D, dq_col=0, dKV=dkv, lddkv=dkv.stride(0), dk_col=0,
                                          dv_col=D, no_dkv=no_dkv)
        return L.cross_attn_args(self, qc, kv, out3, lse, mods, w["mem_valid"], w["ent_valid"], w["inv_n"], w["N"], R,
                                 loo=Tt > 0, **bwd)

    # ------------------------------------------------------------------ forward
    def _stage_bookkeeping(self, w, batch, img_mask_u8):
        """Integer bookkeeping of the img / table pretraining stages (src/img_pretrain.py:85-141, src/table_pretrain.py:84-129):
        one target per business given as `labels`, rating_diff = 0, one memory modality.  Small tensors; torch on the device."""
        from .inference import shift_tokens_right
        cfg = self.cfg
        B, F, n_img, ik = w["B"], w["F"], w["n_img"], w["img_keys"]
        lab = batch.labels.to(torch.int64)
        dec = shift_tokens_right(lab, cfg.pad_token_id, cfg.bos_token_id, cfg.eos_token_id)
        w["labels"].copy_(lab.reshape(-1))
        w["dec_ids"].copy_(dec.reshape(-1))
        w["dec_valid"].copy_(dec.ne(cfg.pad_token_id).reshape(-1))
        w["rating_diff"].zero_()
        if F > 0:
            w["mem_valid"].copy_(w["tab_valid"].reshape(-1))
            ent = w["tab_valid"].max(dim=1, keepdim=True).values
        else:
            w["mem_valid"].copy_(img_mask_u8.ne(0).to(torch.uint8)[:, :, None].expand(B, n_img, ik).reshape(-1))
            ent = img_mask_u8.ne(0).to(torch.uint8)
        w["ent_valid"].copy_(ent)
        cnt = ent.sum(dim=1).float()
        w["inv_n"].copy_(torch.where(cnt > 0, 1.0 / cnt.clamp(min=1), torch.zeros_like(cnt))[:, None])

    # ------------------------------------------------------------------ CUDA-graph replay of the step
    def enable_graph(self, on=True):
        """Record forward and backward of a step shape once and replay them (SURVEY §8f-2).  The step takes everything that
        changes between steps from device memory — inputs are copied into static buffers, the dropout step counter lives on the
        device, the upstream gradient is a device scalar — so a replay is two graph launches instead of ~940 kernel launches.
        It pays where the step is launch-bound (the reference's default of ONE business per GPU); at 16 businesses the step is
        GPU-bound either way.  Semantics in graph mode: gradients are zeroed at the start of every backward (= the
        `optimizer.zero_grad()` of src/multimodal_train.py:359), and a data-parallel reducer (NCCL inside the backward) keeps the
        step on plain launches."""
        self.graph_mode = bool(on)
        self._graphs = {}
        self._graph_entry = None

    @staticmethod
    def _batch_key(batch):
        return tuple((tuple(t.shape), str(t.dtype)) for t in batch.tensors())

    def forward_step(self, batch, label_smoothing, training):
        """`forward` behind the autograd node: plain launches, or warm-up -> capture -> replay in graph mode."""
        self._graph_entry = None
        if not self.graph_mode or self.grad_ready_hook is not None or self.device.type != "cuda":
            return self.forward(batch, label_smoothing, training)
        # the encoder frame is part of the recorded shapes (taken from the batch's length hint, else read back from the mask:
        # one small host sync per step, which costs a graph-launch latency, not the launch-bound step the graphs remove)
        S_in = batch.reviews.shape[-1] if batch.reviews is not None else 0
        frame = self._encoder_frame(batch, S_in) if self.cfg.text_memory else None
        self.det = torch.are_deterministic_algorithms_enabled()       # (a replay runs no forward(): the mode is read here too)
        plan = self._read_trainable()
        key = (self._batch_key(batch), bool(training), label_smoothing, frame, plan.trainable, self.det)
        ent = self._graphs.get(key)
        if ent is None:
            if len(self._graphs) >= 4:
                self._graphs.pop(next(iter(self._graphs)))
            from .synth import Batch
            cl = lambda t: None if t is None else t.clone()
            ent = dict(static=Batch(cl(batch.reviews), cl(batch.reviews_mask), cl(batch.reviews_rating), cl(batch.field),
                                    [cl(t) for t in batch.field_value], cl(batch.img), cl(batch.img_mask), cl(batch.labels)),
                       warm=False, gout=torch.ones(1, device=self.device))
            self._graphs[key] = ent
        for dst, src in zip(ent["static"].tensors(), batch.tensors()):
            dst.copy_(src)
        ent["static"].max_review_len = frame
        self.refresh_bf16_weights()                       # host-side decision: stays outside the recorded graph
        self._graph_entry = ent
        if not ent["warm"]:                               # first step of a shape: plain launches (one-time attributes, workspaces)
            ent["warm"] = True
            ent["eager"] = True
            return self.forward(ent["static"], label_smoothing, training, refresh=False)
        ent["eager"] = False
        if "fwd" not in ent:
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                self.forward(ent["static"], label_smoothing, training, refresh=False)
            ent["fwd"] = g
        else:
            self.fwd_generation += 1
            self.step_count += 1
        ent["fwd"].replay()
        return self.ws["loss"]

    def backward_step(self, grad_out):
        ent = self._graph_entry
        if ent is None or ent.get("eager", True):
            return self.backward(grad_out)
        ent["gout"].copy_(grad_out.reshape(1))
        if "bwd" not in ent:
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                self.backward(ent["gout"], force_zero=True)
            ent["bwd"] = g
        ent["bwd"].replay()
        self._point_grads()

    def forward(self, batch, label_smoothing=0.1, training=True, refresh=True):
        """batch: synth.Batch on the device.  Returns the scalar loss tensor (fp32, device)."""
        if not self.bound:
            raise RuntimeError("engine.bind(named_parameters) first")
        cfg = self.cfg
        V = cfg.vocab_size
        has_text, gates = cfg.text_memory, cfg.multimodal
        if has_text:
            B, R, S = batch.reviews.shape
        else:
            (B, S), R = batch.labels.shape, 1
        F = L.table_dims(cfg.table)
        n_img, img_keys = (batch.img.shape[1], batch.img.shape[2]) if cfg.image else (0, 0)
        if S != 128:
            raise ValueError("the attention kernels are specialised to 128-token frames")
        S_enc = self._encoder_frame(batch, S) if has_text else S
        w = self._alloc(B, R, S, F, n_img, img_keys, S_enc)
        self.ws = w
        self.det = torch.are_deterministic_algorithms_enabled()
        self._read_trainable()
        if self.det and training:
            self._size_ordered_workspaces()       # before any recorded graph of this shape can need it (backward re-checks)
        T, Tt, Te = w["T"], w["Tt"], w["Te"]
        w["batch"] = batch                 # backward re-reads the bit-code table fields
        self.step_count += 1
        self.step_dev.add_(1)
        self.fwd_generation += 1
        self.training = training
        pd = self.dropout if training else 0.0
        self.pd = pd
        self.label_smoothing = label_smoothing
        seed = self.seed
        if refresh:
            self.refresh_bf16_weights()
        bm = "bart_model.model."
        drop = lambda kind, l: (pd, seed, self._sid(kind, l), self.step_dev)

        # ---- table front end + step bookkeeping (integer work, bit-exact)
        img_mask_u8 = None
        if F > 0:
            L.table_embed(self, batch.field, batch.field_value, w["tabX"], w["tab_valid"])
        if n_img > 0:
            img_mask_u8 = batch.img_mask.view(torch.uint8) if batch.img_mask.dtype == torch.bool else batch.img_mask
        if has_text:
            ops.prep_step(batch.reviews, batch.reviews_mask, batch.reviews_rating,
                          w["tab_valid"] if gates else None, img_mask_u8 if gates else None,
                          B=B, R=R, S=S, S_enc=S_enc, F=F, n_img=n_img, img_keys=img_keys, n_mod=3 if gates else 1,
                          pad_id=cfg.pad_token_id, bos_id=cfg.bos_token_id, eos_id=cfg.eos_token_id,
                          enc_ids=w["enc_ids"], dec_ids=w["dec_ids"], labels=w["labels"], enc_valid=w["enc_valid"],
                          dec_valid=w["dec_valid"], mem_valid=w["mem_valid"], ent_valid=w["ent_valid"],
                          pres=w["pres"] if gates else None, rating_diff=w["rating_diff"], inv_n=w["inv_n"])
        else:
            self._stage_bookkeeping(w, batch, img_mask_u8)
        MEM = w["MEM"]
        if F > 0:
            L.table_project(self, w["tabX"], w["tab_h"], MEM[Tt:Tt + B * F])
        if n_img > 0:
            img = batch.img.reshape(B * n_img * img_keys, 1024)
            if img.dtype == torch.float32:
                ops.cast_bf16(img.contiguous(), w["img16"])
                img = w["img16"]
            w["img_in"] = img
            ops.gemm(img, self.w16("img_encoder.linear.weight"), MEM[Tt + B * F:])

        # ---- encoder (BartEncoder.forward :346-404)
        if has_text:
            x = w["enc_x0"]
            ops.embed_ln_fwd(w["enc_ids"], *L.embed_params(self, "encoder", None), x, w["enc_m0"], w["enc_r0"], Te, S_enc, *drop(0, 0))
            L_e = cfg.encoder_layers
            for l in range(L_e):
                a = w["enc"][l]
                a["x"] = x
                lp = bm + "encoder.layers.%d." % l
                out = MEM[:Te] if l == L_e - 1 else w["enc"][l + 1]["x"]
                attend = lambda qkv, ctx, a=a: ops.attn_fwd(self._self_attn_args(w, qkv, ctx, a["lse"], w["enc_valid"], False,
                                                                                 frame=S_enc))
                L.self_block(self, lp, x, a, attend, (a["m1"], a["r1"]), drop(1, l))
                L.ffn_block(self, lp, a["x1"], a, out, (a["m2"], a["r2"]), drop(2, l), dact=a["h"])   # a["h"]: GELU'
                x = out

        # ---- decoder, batched leave-one-out (BartDecoder.forward :530-660 over 9·B sequences)
        L_d = cfg.decoder_layers
        x = w["dec"][0]["x"]
        ops.embed_ln_fwd(w["dec_ids"], *L.embed_params(self, "decoder", w["rating_diff"]), x, w["dec_m0"], w["dec_r0"], T, S,
                         *drop(3, 0))
        for l in range(L_d):
            a = w["dec"][l]
            lp = bm + "decoder.layers.%d." % l
            out = w["x_out"] if l == L_d - 1 else w["dec"][l + 1]["x"]
            attend = lambda qkv, ctx, a=a: ops.attn_fwd(self._self_attn_args(w, qkv, ctx, a["lse"], w["dec_valid"], True))

            def attend_mem(qc, A3, a=a, l=l):
                L.project_kv(self, MEM, l, a["kv"])     # this layer's K|V of the memory, kept for the backward
                ops.attn_fwd(self._cross_attn_args(w, qc, a["kv"], A3, a["lse_c"]))

            L.self_block(self, lp, a["x"], a, attend, (a["m1"], a["r1"]), drop(4, l))
            L.cross_block(self, lp, a["x1"], a, attend_mem, (a["m2"], a["r2"]), drop(5, l), w["pres"], R * S)
            L.ffn_block(self, lp, a["x2"], a, out, (a["m3"], a["r3"]), drop(6, l), dact=a["h"])
            x = out

        # ---- LM head + loss (:2281, src/utils.py:32-38); mean over all 9·B·128 rows == mean of the 9 pass means
        logits = w["logits"]
        ops.gemm(x, self.w16(bm + "shared.weight"), logits[:, :V], bias=self.w32_flb(), raster_m_fast=True)
        ops.ce_fwd_bwd(logits, V, w["labels"], label_smoothing, 0.0, None, w["loss_rows"], w["loss"], 1.0 / T, False,
                       lse_rows=w["lse_rows"])
        return w["loss"]

    def _encoder_frame(self, batch, S):
        """Smallest multiple of 16 that holds every review's last valid token (the encoder frame, see _alloc).  Taken from the
        batch's host-side hint when there is one; otherwise read back from the mask once per mask tensor (a host sync)."""
        if not self.trim_frames:
            return S
        n = getattr(batch, "max_review_len", None)
        if n is None:
            m = batch.reviews_mask
            # cached only for the SAME tensor object at the same version (an address can be recycled by a new batch)
            c = self._len_cache
            if c is not None and c[0]() is m and c[1] == m._version:
                n = c[2]
            elif m.is_cuda and torch.cuda.is_current_stream_capturing():
                return S
            else:
                pos = torch.arange(1, S + 1, device=m.device, dtype=torch.int32)
                n = int((m.ne(0).to(torch.int32) * pos).max().item())
                self._len_cache = (weakref.ref(m), m._version, n)
        return min(S, max(16, (int(n) + 15) // 16 * 16))

    def _size_ordered_workspaces(self):
        """Scratch of the ordered backward, sized once per step shape (like the other workspaces) for every encoder frame the
        shape can run: the largest split-K partial set of the step's weight-gradient GEMMs, the LayerNorm and embedding partials
        (main stream), and the bias-gradient partials (side stream).  The split choice is not monotone in the frame, so all
        frames are visited.  A graph recorded in this mode holds the old scratch's address: when the scratch has to grow, those
        graphs are dropped.  The library rejects a call whose scratch is too small."""
        if self.ws_key in self._det_sized:
            return
        cfg, w = self.cfg, self.ws_full
        D, FF, V = cfg.d_model, cfg.ffn_dim, cfg.vocab_size
        B, R, S, F, T = w["B"], w["R"], w["S"], w["F"], w["T"]
        side = B * F + B * w["n_img"] * w["img_keys"]
        frames = range(16, S + 1, 16) if w["Tt"] > 0 and self.trim_frames else [S]
        shapes = {(V, D, T), (D, FF, T), (FF, D, T), (D, D, T), (3 * D, D, T), (D, D, w["nm"] * T)}
        need = max(ops.ADD_LN_BWD_WORKSPACE, ops.embed_ln_bwd_workspace(T, S, V))
        for f in frames:
            Te = B * R * f
            shapes.add((2 * D, D, (Te if w["Tt"] > 0 else 0) + side))
            if w["Tt"] > 0:
                shapes.update({(D, FF, Te), (FF, D, Te), (D, D, Te), (3 * D, D, Te)})
                need = max(need, ops.embed_ln_bwd_workspace(Te, f, V))
        if F > 0:
            shapes.update({(D, D, B * F), (D, 2 * D, B * F)})
        if w["n_img"] > 0:
            shapes.add((D, 1024, B * w["n_img"] * w["img_keys"]))
        need = max([need] + [ops.gemm_workspace_elems(*sh) for sh in shapes])
        need_side = ops.colsum_workspace(max(FF, 3 * D))
        grown = False
        if self.det_ws is None or self.det_ws.numel() < need:
            self.det_ws, grown = torch.empty(need, device=self.device, dtype=torch.float32), True
        if self.det_ws_side is None or self.det_ws_side.numel() < need_side:
            self.det_ws_side, grown = torch.empty(need_side, device=self.device, dtype=torch.float32), True
        if grown:
            self._graphs = {k: e for k, e in self._graphs.items() if not (k[-1] and "bwd" in e)}
        self._det_sized.add(self.ws_key)

    def _ows(self):
        """The main-stream scratch of the ordered reductions when this step runs them, else None (the atomic fast path)."""
        return self.det_ws if self.det else None

    def w32_flb(self):
        return self.final_logits_bias.view(-1) if getattr(self, "final_logits_bias", None) is not None else None

    # ------------------------------------------------------------------ backward
    def _wgrad(self, dy, x, gname, gname2=None, col_slice=None):
        """G[name] += dyᵀ·x   (dy [T, N_out], x [T, K_in]) — MN-major operands, split-K, TMA reduce-add."""
        out = self.g32(gname, gname2)
        if col_slice is not None:
            out = out[:, col_slice[0]:col_slice[1]]
        ops.gemm(dy, x, out, a_t=True, b_t=True, accumulate=True, workspace=self._ows())

    # Bias gradients (column sums of an upstream-gradient matrix) are short, launch-latency-dominated kernels that sit
    # off the critical dgrad chain: they run on a side stream and overlap the GEMMs that consume the same matrix.  The main
    # stream joins the side stream before any scratch buffer is recycled, before a gradient range is declared final and
    # at the end of backward.
    def _bias_grad(self, x, out):
        ws = self.det_ws_side if self.det else None
        if self.side_stream is None:
            ops.colsum(x, out, workspace=ws)
            return
        main = torch.cuda.current_stream()
        self._ev_main.record(main)
        self.side_stream.wait_event(self._ev_main)
        with torch.cuda.stream(self.side_stream):
            ops.colsum(x, out, workspace=ws)
            self._ev_side.record(self.side_stream)
        self._side_pending = True

    def _side_join(self):
        if self._side_pending:
            torch.cuda.current_stream().wait_event(self._ev_side)
            self._side_pending = False

    def _ready(self, name_last):
        self._side_join()
        if self.grad_ready_hook is not None:
            hi = self.offsets[name_last] + (math.prod(self.shapes[name_last]) + ALIGN - 1) // ALIGN * ALIGN
            self.grad_ready_hook(hi)

    def _ln_grads(self, ln):
        """(dgamma, dbeta) outputs of LayerNorm `ln`: (None, None) when both are frozen (the kernel variant without the reduction);
        a frozen half of a trainable pair writes into a sink instead of its arena range."""
        gw, gb = ln + ".weight" in self.plan.grads, ln + ".bias" in self.plan.grads
        if not gw and not gb:
            return None, None
        return (self.g32(ln + ".weight") if gw else self._ln_sink[0]), (self.g32(ln + ".bias") if gb else self._ln_sink[1])

    def _fused_runs(self, names):
        """Maximal runs [i0, i1) of adjacent members of a fused group (q|k|v, k|v: consecutive in the arena and in the columns of
        their upstream gradient) whose gradient is computed: one GEMM / column sum per run, nothing written into a frozen member."""
        runs = []
        for i, n in enumerate(names):
            if n in self.plan.grads:
                if runs and runs[-1][1] == i:
                    runs[-1][1] = i + 1
                else:
                    runs.append([i, i + 1])
        return runs

    def _fused_grads(self, dy, x, wnames, bnames):
        """Bias column sums and weight gradients of a fused group over the column slices of dy that belong to trainable members."""
        D = self.cfg.d_model
        for i0, i1 in self._fused_runs(bnames):
            self._bias_grad(dy[:, i0 * D:i1 * D], self.g32(bnames[i0], bnames[i1 - 1]))
        for i0, i1 in self._fused_runs(wnames):
            self._wgrad(dy[:, i0 * D:i1 * D], x, wnames[i0], wnames[i1 - 1])

    def _ffn_block_bwd(self, w, a, lp, d1, d2, xin, mk, rk, l, kind, tag, enc=False):
        """Backward of x_out = LN(xin + drop(fc2(gelu(fc1(xin))))).  Returns the two addends of d xin (None, None when the plan
        does not need it)."""
        pool, pd, P = (w["pool_e"] if enc else w["pool"]), self.pd, self.plan
        need_in = tag + "ffn.in" in P.dgrad
        dres = pool.get()
        df = pool.get() if pd > 0 else dres
        gam, bet = self._ln_grads(lp + "final_layer_norm")
        ops.add_ln_bwd(d1, d2, xin, a["f"], self.w32(lp + "final_layer_norm.weight"), a[mk], a[rk], dres, df, gam, bet, pd, self.seed,
                       self._sid(kind, l), step_dev=self.step_dev, workspace=self._ows())
        pool.put(d1, d2)
        if lp + "fc2.bias" in P.grads:
            self._bias_grad(df, self.g32(lp + "fc2.bias"))
        if lp + "fc2.weight" in P.grads:
            self._wgrad(df, a["a"], lp + "fc2.weight")
        dH = w["dH"][:xin.shape[0]]
        if tag + "ffn.dH" in P.dgrad:
            ops.gemm(df, self.w16(lp + "fc2.weight"), dH, b_t=True, act=ops.ACT_GELU, aux=a["h"], aux_mode=ops.AUX_MUL)
        if df is not dres:
            pool.put(df)
        if lp + "fc1.bias" in P.grads:
            self._bias_grad(dH, self.g32(lp + "fc1.bias"))
        if lp + "fc1.weight" in P.grads:
            self._wgrad(dH, xin, lp + "fc1.weight")
        if not need_in:
            pool.put(dres)
            return None, None
        dx = pool.get()
        ops.gemm(dH, self.w16(lp + "fc1.weight"), dx, b_t=True)
        return dres, dx

    def _self_block_bwd(self, w, a, lp, d1, d2, key_valid, causal, l, kind, tag, enc=False):
        """Backward of x1 = LN(x + drop(out_proj(attn(qkv(x))))).  Returns the two addends of d x (None, None when the plan does
        not need it)."""
        pool, pd, P = (w["pool_e"] if enc else w["pool"]), self.pd, self.plan
        s = lp + "self_attn."
        need_in = tag + "self.in" in P.dgrad
        dres = pool.get()
        do = pool.get() if pd > 0 else dres
        gam, bet = self._ln_grads(lp + "self_attn_layer_norm")
        ops.add_ln_bwd(d1, d2, a["x"], a["o"], self.w32(lp + "self_attn_layer_norm.weight"), a["m1"], a["r1"], dres, do, gam, bet, pd,
                       self.seed, self._sid(kind, l), step_dev=self.step_dev, workspace=self._ows())
        pool.put(d1, d2)
        if s + "out_proj.bias" in P.grads:
            self._bias_grad(do, self.g32(s + "out_proj.bias"))
        if s + "out_proj.weight" in P.grads:
            self._wgrad(do, a["ctx"], s + "out_proj.weight")
        if tag + "self.dctx" not in P.dgrad:
            pool.put(do, dres)
            return None, None
        dctx = pool.get()
        ops.gemm(do, self.w16(s + "out_proj.weight"), dctx, b_t=True)
        if do is not dres:
            pool.put(do)
        dqkv = w["dqkv"][:a["qkv"].shape[0]]
        ops.attn_bwd(self._self_attn_args(w, a["qkv"], dctx, a["lse"], key_valid, causal, dqkv=dqkv, frame=w["S_enc"] if enc else None))
        pool.put(dctx)
        self._fused_grads(dqkv, a["x"], [s + "q_proj.weight", s + "k_proj.weight", s + "v_proj.weight"],
                          [s + "q_proj.bias", s + "k_proj.bias", s + "v_proj.bias"])
        if not need_in:
            pool.put(dres)
            return None, None
        dx = pool.get()
        ops.gemm(dqkv, self.w16(s + "q_proj.weight", s + "v_proj.weight"), dx, b_t=True)
        return dres, dx

    def _mem_rows(self, w, m):
        Tt, BF = w["Tt"], w["B"] * w["F"]
        return {"text": (0, Tt), "table": (Tt, Tt + BF), "image": (Tt + BF, w["Tm"])}[m]

    def backward(self, grad_out=None, force_zero=False):
        """Writes the gradient of every trainable parameter into the fp32 gradient arena (+=) and points its `.grad` at it.  Runs
        the backward plan (backward_plan) of the trainable set the forward read: a frozen parameter's range is never written and
        its `.grad` is None; what only frozen parameters need is not computed."""
        cfg, w = self.cfg, self.ws
        if w is None:
            raise RuntimeError("backward() without a forward()")
        D, V = cfg.d_model, cfg.vocab_size
        T, Tt, Tm, B, R, S, F = w["T"], w["Tt"], w["Tm"], w["B"], w["R"], w["S"], w["F"]
        n_img, img_keys = w["n_img"], w["img_keys"]
        gates = cfg.multimodal
        pool, pd, seed = w["pool"], self.pd, self.seed
        bm = "bart_model.model."
        g = ops.gemm
        P = self.plan
        grads, dgrad = P.grads, P.dgrad
        if self.det:
            self._size_ordered_workspaces()
        first = next((p for n, p in self.params.items() if n in P.trainable), None)
        if force_zero or (first is not None and first.grad is None):
            self.G32.zero_()
        # ---- loss + LM head
        logits = w["logits"]
        if P.run:
            ops.ce_fwd_bwd(logits, V, w["labels"], self.label_smoothing, 1.0 / T, grad_out, w["loss_rows"], None, 0.0, True,
                           lse_rows=w["lse_rows"])
        dl = logits[:, :V]
        d1 = d2 = None
        if "head.in" in dgrad:
            d1 = pool.get()
            g(dl, self.w16(bm + "shared.weight"), d1, b_t=True)
        xfin = w["x_out"]
        if bm + "shared.weight" in grads:
            ops.gemm(dl, xfin, self.g32(bm + "shared.weight"), a_t=True, b_t=True, accumulate=True, workspace=self._ows())

        # ---- decoder layers, last to first
        pre = bm + "decoder."
        mem_any = any(P.mem.values())
        for l in reversed(range(cfg.decoder_layers)):
            a = w["dec"][l]
            lp = pre + "layers.%d." % l
            c = lp + "encoder_attn."
            tag = "dec.%d." % l
            if not P.dec_in[l + 1]:
                self._ready(lp + "self_attn_layer_norm.bias")
                continue
            d1, d2 = self._ffn_block_bwd(w, a, lp, d1, d2, a["x2"], "m3", "r3", l, 6, tag)
            if tag + "ffn.in" in dgrad:
                # cross block
                dres = pool.get()
                yc = a["yc"] if gates else a["O3"][0]
                dyc = pool.get() if pd > 0 else dres
                gam, bet = self._ln_grads(lp + "encoder_attn_layer_norm")
                ops.add_ln_bwd(d1, d2, a["x1"], yc, self.w32(lp + "encoder_attn_layer_norm.weight"), a["m2"], a["r2"], dres, dyc,
                               gam, bet, pd, seed, self._sid(5, l), step_dev=self.step_dev, workspace=self._ows())
                pool.put(d1, d2)
                nm = a["A3"].shape[0]
                dO3_on, dA3_on = tag + "cross.dO3" in dgrad, tag + "cross.dA3" in dgrad
                if gates:
                    dU, dO3 = w["dU"], w["dO3"]
                    if tag + "cross.dU" in dgrad:
                        ops.gate_bwd_u(dyc, a["O3"], a["AB"], dU, T, D)
                    if c + "alpha_proj.bias" in grads:
                        self._bias_grad(dU[0], self.g32(c + "alpha_proj.bias"))
                    if c + "beta_proj.bias" in grads:
                        self._bias_grad(dU[1], self.g32(c + "beta_proj.bias"))
                    if c + "alpha_proj.weight" in grads:
                        self._wgrad(dU[0], a["O3"][0], c + "alpha_proj.weight", col_slice=(0, D))
                        self._wgrad(dU[0], a["O3"][1], c + "alpha_proj.weight", col_slice=(D, 2 * D))
                    if c + "beta_proj.weight" in grads:
                        self._wgrad(dU[1], a["O3"][0], c + "beta_proj.weight", col_slice=(0, D))
                        self._wgrad(dU[1], a["O3"][2], c + "beta_proj.weight", col_slice=(D, 2 * D))
                    if dO3_on:
                        g(dU[0], self.w16(c + "alpha_proj.weight"), w["dca"], b_t=True)
                        g(dU[1], self.w16(c + "beta_proj.weight"), w["dcb"], b_t=True)
                        ops.gate_bwd_o(dyc, a["AB"], w["dca"], w["dcb"], dO3, T, D)
                    dO3f = dO3.view(nm * T, D)
                else:
                    dO3f = dyc
                if c + "out_proj.bias" in grads:
                    self._bias_grad(dO3f, self.g32(c + "out_proj.bias"))
                if c + "out_proj.weight" in grads:
                    self._wgrad(dO3f, a["A3"].view(nm * T, D), c + "out_proj.weight")
                dA3 = w["dA3"]
                if dA3_on:
                    g(dO3f, self.w16(c + "out_proj.weight"), dA3.view(nm * T, D), b_t=True)
                if dyc is not dres:
                    pool.put(dyc)
                need_x1 = tag + "cross.in" in dgrad
                dx1 = None
                if dA3_on:
                    dqc = pool.get()
                    dkv = w["dkv_all"][:, l * 2 * D:(l + 1) * 2 * D]
                    mods = [m for m, on in (("text", Tt > 0), ("table", F > 0), ("image", n_img > 0)) if on]
                    ops.attn_bwd(self._cross_attn_args(w, a["qc"], a["kv"], dA3, a["lse_c"], dqc, dkv,
                                                       no_dkv=[m not in P.dkv[l] for m in mods]))
                    if c + "q_proj.bias" in grads:
                        self._bias_grad(dqc, self.g32(c + "q_proj.bias"))
                    if c + "q_proj.weight" in grads:
                        self._wgrad(dqc, a["x1"], c + "q_proj.weight")
                    if need_x1:
                        dx1 = pool.get()
                        g(dqc, self.w16(c + "q_proj.weight"), dx1, b_t=True)
                    pool.put(dqc)
                    self._fused_grads(dkv, w["MEM"], [c + "k_proj.weight", c + "v_proj.weight"], [c + "k_proj.bias", c + "v_proj.bias"])
                if mem_any:
                    w["Wkv_cat"][l * 2 * D:(l + 1) * 2 * D].copy_(self.w16(c + "k_proj.weight", c + "v_proj.weight"))
                if need_x1:
                    # self block
                    d1, d2 = self._self_block_bwd(w, a, lp, dres, dx1, w["dec_valid"], True, l, 4, tag)
                else:
                    pool.put(dres)
                    d1, d2 = None, None
            self._ready(lp + "self_attn_layer_norm.bias")
        # decoder embedding
        if P.dec_in[0]:
            opt = lambda n: self.g32(n) if n in grads else None        # noqa: E731
            gam, bet = self._ln_grads(pre + "layernorm_embedding")
            ops.embed_ln_bwd(d1, d2, w["dec_ids"], self.w32(bm + "shared.weight"), self.w32(pre + "embed_positions.weight"),
                             w["rating_diff"], self.w32(pre + "rating_embeddings"), self.w32(pre + "layernorm_embedding.weight"),
                             w["dec_m0"], w["dec_r0"], opt(bm + "shared.weight"), opt(pre + "embed_positions.weight"),
                             opt(pre + "rating_embeddings"), gam, bet, w["dz32"], T, S, cfg.pad_token_id, pd, seed, self._sid(3, 0),
                             step_dev=self.step_dev, workspace=self._ows())
            pool.put(d1, d2)
        self._ready(pre + "embed_positions.weight")

        # ---- memory gradients: table, image, text (only the rows of modalities whose producer has a trainable parameter)
        dMEM = w["dMEM16"]
        runs = []
        for m in ("text", "table", "image"):
            if P.mem[m]:
                r0, r1 = self._mem_rows(w, m)
                if runs and runs[-1][1] == r0:
                    runs[-1][1] = r1
                else:
                    runs.append([r0, r1])
        for r0, r1 in runs:
            g(w["dkv_all"][r0:r1], w["Wkv_cat"], dMEM[r0:r1], b_t=True)
        if F > 0:
            t = "table_encoder."
            if P.mem["table"]:
                dtab = dMEM[Tt:Tt + B * F]
                if t + "linear.weight" in grads:
                    self._wgrad(dtab, w["tab_h"], t + "linear.weight")
                if "table.dtab_h" in dgrad:
                    g(dtab, self.w16(t + "linear.weight"), w["dtab_h"], b_t=True, act=ops.ACT_RELU, aux=w["tab_h"],
                      aux_mode=ops.AUX_MUL_DACT)
                if t + "fc.bias" in grads:
                    self._bias_grad(w["dtab_h"], self.g32(t + "fc.bias"))
                if t + "fc.weight" in grads:
                    self._wgrad(w["dtab_h"], w["tabX"], t + "fc.weight")
                if "table.dtabX" in dgrad:
                    g(w["dtab_h"], self.w16(t + "fc.weight"), w["dtabX"], b_t=True)
                batch = w["batch"]
                if cfg.table == "yelp":
                    bits = ((batch.field_value[4], t + "rating_embedding.weight", 39, 1, 4),
                            (batch.field_value[5], t + "hours_embedding.weight", 40, 7, 4))
                else:
                    bits = ((batch.field_value[0], t + "price_embedding.weight", 0, 1, 11),
                            (batch.field_value[1], t + "rating_embedding.weight", 1, 1, 4))
                for v, n, f0, nrows, nb in bits:
                    if n in grads:
                        ops.table_bits_bwd(w["dtabX"], v, self.g32(n), B, F, f0, nrows, nb)
            if n_img == 0:
                self._ready(t + ("hours_embedding.weight" if cfg.table == "yelp" else "price_embedding.weight"))
        if n_img > 0:
            if "img_encoder.linear.weight" in grads:
                self._wgrad(dMEM[Tt + B * F:], w["img_in"], "img_encoder.linear.weight")
            self._ready("img_encoder.linear.weight")

        # ---- encoder layers, last to first, down to the lowest one the plan needs (the img / table stages have no text memory)
        if Tt > 0 and P.mem["text"]:
            pre = bm + "encoder."
            Te, S_enc, pool = w["Te"], w["S_enc"], w["pool_e"]
            d1 = pool.get()
            d1.copy_(dMEM[:Te])
            d2 = None
            for l in reversed(range(cfg.encoder_layers)):
                a = w["enc"][l]
                lp = pre + "layers.%d." % l
                if P.enc_in[l + 1]:
                    tag = "enc.%d." % l
                    d1, d2 = self._ffn_block_bwd(w, a, lp, d1, d2, a["x1"], "m2", "r2", l, 2, tag, enc=True)
                    if tag + "ffn.in" in dgrad:
                        d1, d2 = self._self_block_bwd(w, a, lp, d1, d2, w["enc_valid"], False, l, 1, tag, enc=True)
                self._ready(lp + "self_attn_layer_norm.bias")
            if P.enc_in[0]:
                opt = lambda n: self.g32(n) if n in grads else None    # noqa: E731
                gam, bet = self._ln_grads(pre + "layernorm_embedding")
                ops.embed_ln_bwd(d1, d2, w["enc_ids"], self.w32(bm + "shared.weight"), self.w32(pre + "embed_positions.weight"), None,
                                 None, self.w32(pre + "layernorm_embedding.weight"), w["enc_m0"], w["enc_r0"],
                                 opt(bm + "shared.weight"), opt(pre + "embed_positions.weight"), None, gam, bet, w["dz32"], Te, S_enc,
                                 cfg.pad_token_id, pd, seed, self._sid(0, 0), step_dev=self.step_dev, workspace=self._ows())
                pool.put(d1, d2)
        self._ready(bm + "shared.weight")
        self._point_grads()
