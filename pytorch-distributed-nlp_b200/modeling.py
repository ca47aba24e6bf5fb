"""Drop-in ``BertForSequenceClassification`` whose forward/backward run on the sm_100a kernels of libb2ddpbert.so.

Mirrors the surface `multi-gpu-distributed-cls.py` uses (reference lines in brackets):
  * ``BertConfig(..., num_labels=6)`` / ``BertForSequenceClassification.from_pretrained(path, config=config)`` [:336-338]
  * ``model.cuda()`` [:340], ``model.train()/eval()`` [:166,:200]
  * ``model(input_ids=, token_type_ids=, attention_mask=, labels=)`` -> output with ``[0]`` = loss, ``[1]`` = logits
    [:132-136] and ``.logits`` (`predict.py:133`)
  * ``named_parameters()`` yielding the 201 HF parameter names (the no-decay filter at [:101-107] matches on them)
  * ``state_dict()/load_state_dict()`` in HF naming, fp32 (`test.py:96-101`, [:192,:362])
The arithmetic follows HF ``BertForSequenceClassification`` (SP/transformers/models/bert/modeling_bert.py:53-468,
1077-1154, eager attention) in bf16 with fp32 accumulation/statistics; fp32 master weights stay the parameters
the user sees.  There is no PyTorch fallback: without the CUDA library every call raises.
"""
import contextlib
import os
from collections import OrderedDict

import torch
import torch.nn as nn

from . import _lib as L


class BertConfig:
    """The subset of ``transformers.BertConfig`` the path reads; any object with these attributes works."""

    def __init__(self, vocab_size=21128, hidden_size=768, num_hidden_layers=12, num_attention_heads=12,
                 intermediate_size=3072, hidden_act="gelu", hidden_dropout_prob=0.1,
                 attention_probs_dropout_prob=0.1, max_position_embeddings=512, type_vocab_size=2,
                 initializer_range=0.02, layer_norm_eps=1e-12, pad_token_id=0, num_labels=2,
                 classifier_dropout=None, **kwargs):
        self.vocab_size = vocab_size
        self.hidden_size = hidden_size
        self.num_hidden_layers = num_hidden_layers
        self.num_attention_heads = num_attention_heads
        self.intermediate_size = intermediate_size
        self.hidden_act = hidden_act
        self.hidden_dropout_prob = hidden_dropout_prob
        self.attention_probs_dropout_prob = attention_probs_dropout_prob
        self.max_position_embeddings = max_position_embeddings
        self.type_vocab_size = type_vocab_size
        self.initializer_range = initializer_range
        self.layer_norm_eps = layer_norm_eps
        self.pad_token_id = pad_token_id
        self.num_labels = num_labels
        self.classifier_dropout = classifier_dropout
        for k, v in kwargs.items():
            setattr(self, k, v)

    @classmethod
    def from_pretrained(cls, path, **kwargs):
        import json
        cfg = {}
        f = os.path.join(path, "config.json")
        if os.path.exists(f):
            with open(f) as fp:
                cfg = json.load(fp)
        cfg.update(kwargs)
        return cls(**cfg)


# presets named in BASELINE.json
def chinese_bert_wwm_ext_config(num_labels=6, **kw):
    return BertConfig(vocab_size=21128, num_labels=num_labels, **kw)


def bert_base_config(num_labels=6, **kw):
    return BertConfig(vocab_size=30522, num_labels=num_labels, **kw)


def bert_large_config(num_labels=6, **kw):
    return BertConfig(vocab_size=30522, hidden_size=1024, num_hidden_layers=24, num_attention_heads=16,
                      intermediate_size=4096, num_labels=num_labels, **kw)


class SequenceClassifierOutput:
    """Tuple-like output: with labels ``(loss, logits)``, without ``(logits,)`` — as HF's ModelOutput indexes."""

    def __init__(self, loss=None, logits=None):
        self.loss = loss
        self.logits = logits

    def to_tuple(self):
        return tuple(v for v in (self.loss, self.logits) if v is not None)

    def __getitem__(self, i):
        if isinstance(i, str):
            return getattr(self, i)
        return self.to_tuple()[i]

    def __iter__(self):
        return iter(self.to_tuple())

    def __len__(self):
        return len(self.to_tuple())


def _round8(n):
    return (n + 7) // 8 * 8


class _Holder(nn.Module):
    """Name-only container so that ``named_parameters()`` reproduces the HF module paths."""


class _Layout:
    """Flat parameter space: HF tensors in forward order, each padded to 8 elements, Q/K/V stacked contiguously.
    Buckets (DDP exchange / AdamW launch units) = embeddings | encoder layer 0..L-2 | last layer + head.  The head
    (pooler + classifier, 0.6 M parameters) rides with the last encoder layer -- they are adjacent in the flat space and
    final within microseconds of each other at the start of backward -- instead of paying a barrier, an exchange and
    a kernel launch of its own."""

    def __init__(self, cfg):
        H, I, L_ = cfg.hidden_size, cfg.intermediate_size, cfg.num_hidden_layers
        self.entries = OrderedDict()  # hf name -> (offset, shape)
        self.buckets = []             # (begin, end, label)
        off = 0

        def add(name, shape):
            nonlocal off
            n = 1
            for s in shape:
                n *= s
            self.entries[name] = (off, tuple(shape))
            off += _round8(n)

        b0 = off
        add("bert.embeddings.word_embeddings.weight", (cfg.vocab_size, H))
        add("bert.embeddings.position_embeddings.weight", (cfg.max_position_embeddings, H))
        add("bert.embeddings.token_type_embeddings.weight", (cfg.type_vocab_size, H))
        add("bert.embeddings.LayerNorm.weight", (H,))
        add("bert.embeddings.LayerNorm.bias", (H,))
        self.buckets.append((b0, off, "embeddings"))
        for l in range(L_):
            p = "bert.encoder.layer.%d." % l
            b0 = off
            # stacked [3H, H] weight and [3H] bias: one GEMM for Q, K, V
            add(p + "attention.self.query.weight", (H, H))
            add(p + "attention.self.key.weight", (H, H))
            add(p + "attention.self.value.weight", (H, H))
            add(p + "attention.self.query.bias", (H,))
            add(p + "attention.self.key.bias", (H,))
            add(p + "attention.self.value.bias", (H,))
            add(p + "attention.output.dense.weight", (H, H))
            add(p + "attention.output.dense.bias", (H,))
            add(p + "attention.output.LayerNorm.weight", (H,))
            add(p + "attention.output.LayerNorm.bias", (H,))
            add(p + "intermediate.dense.weight", (I, H))
            add(p + "intermediate.dense.bias", (I,))
            add(p + "output.dense.weight", (H, I))
            add(p + "output.dense.bias", (H,))
            add(p + "output.LayerNorm.weight", (H,))
            add(p + "output.LayerNorm.bias", (H,))
            self.buckets.append((b0, off, "layer%d" % l))
        b0 = off
        add("bert.pooler.dense.weight", (H, H))
        add("bert.pooler.dense.bias", (H,))
        add("classifier.weight", (cfg.num_labels, H))
        add("classifier.bias", (cfg.num_labels,))
        if L_ > 0:
            lb, _le, lbl = self.buckets[-1]
            self.buckets[-1] = (lb, off, lbl + "+head")
        else:
            self.buckets.append((b0, off, "head"))
        self.head_in_last_layer = L_ > 0
        self.total = off

    def off(self, name):
        return self.entries[name][0]


# HF named_parameters() order (201 tensors for 12 layers); differs from the flat order only inside attention.self
def _hf_order(cfg):
    names = ["bert.embeddings.word_embeddings.weight", "bert.embeddings.position_embeddings.weight",
             "bert.embeddings.token_type_embeddings.weight", "bert.embeddings.LayerNorm.weight",
             "bert.embeddings.LayerNorm.bias"]
    for l in range(cfg.num_hidden_layers):
        p = "bert.encoder.layer.%d." % l
        for m in ("attention.self.query", "attention.self.key", "attention.self.value", "attention.output.dense",
                  "attention.output.LayerNorm", "intermediate.dense", "output.dense", "output.LayerNorm"):
            names += [p + m + ".weight", p + m + ".bias"]
    names += ["bert.pooler.dense.weight", "bert.pooler.dense.bias", "classifier.weight", "classifier.bias"]
    return names


class _StepFn(torch.autograd.Function):
    """logits (and HF's in-model loss) with a backward that runs the CUDA backward pass."""

    @staticmethod
    def forward(ctx, anchor, model, input_ids, token_type_ids, attention_mask, labels, packed=None):
        eng = model._engine
        logits, loss = eng.forward(input_ids, token_type_ids, attention_mask, labels, training=model.training,
                                   need_backward=True, packed=packed)
        ctx.model = model
        ctx.no_sync = model._no_sync     # as in torch DDP, whether this micro-batch accumulates is fixed at forward time
        ctx.has_loss = loss is not None
        ctx.set_materialize_grads(False)
        if loss is None:
            return logits.clone(), torch.zeros((), device=logits.device)
        return logits.clone(), loss.clone()

    @staticmethod
    def backward(ctx, d_logits, d_loss):
        model = ctx.model
        eng = model._engine
        if d_logits is None and (d_loss is None or not ctx.has_loss):
            raise RuntimeError("backward reached the model without any gradient")
        if model._optimizer is not None:
            # gradients are OVERWRITTEN by every backward outside no_sync() (bf16 bucket space): a second one before
            # optimizer.step() would silently drop the first one's gradients where torch would accumulate
            if model._grads_live:
                raise RuntimeError("backward() called twice without optimizer.step() in between: gradient "
                                   "accumulation is not supported on this path outside no_sync() (gradients are "
                                   "overwritten, not summed)")
            if not ctx.no_sync:
                model._grads_live = True
        # no_sync(): this micro-batch is added to the fp32 accumulator.  The first backward outside it folds the
        # accumulated sum back into the bf16 gradient space, where the exchange and the optimizer read it.
        if ctx.no_sync:
            eng.ensure_accum()
            fold = (L.ACCUM_ADD, 1.0)
        else:
            fold = (L.ACCUM_FINISH, 1.0) if eng.accum_pending else None
        eng.fold = fold
        try:
            eng.backward(d_logits, d_loss if ctx.has_loss else None)
        finally:
            eng.fold = None
        eng.accum_pending = eng.accum_pending + 1 if ctx.no_sync else 0
        model._notify_backward_done()
        # Gradients live in the engine's bf16 bucket space, not in `.grad`.  The anchor (classifier.bias) gets its
        # true gradient as a 6-float fp32 probe: it is the column sum of d_logits, so an inf/nan anywhere upstream
        # of the model shows up in it -- which is what torch.cuda.amp.GradScaler's inf check needs to see.
        off, shape = ctx.model._layout.entries["classifier.bias"]
        n = 1
        for d in shape:
            n *= d
        probe = eng.grads[off:off + n].float().view(shape)
        window = probe
        if fold is not None and fold[0] == L.ACCUM_FINISH:
            # the gradient space now holds the window's sum; autograd adds the probe to the .grad the earlier
            # micro-batches left, so return the difference: .grad ends as the window's sum, as torch's would
            prev = model._params_by_name["classifier.bias"].grad
            if prev is not None:
                probe = window - prev
        if model._ddp is not None and not ctx.no_sync:
            probe = model._ddp.consensus_probe(probe, window)   # covers every micro-batch of the window
        return probe, None, None, None, None, None, None


class BertForSequenceClassification(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        cfg = config
        assert cfg.hidden_size % cfg.num_attention_heads == 0
        if cfg.hidden_size // cfg.num_attention_heads != 64:
            raise ValueError("only head_dim 64 is on the path (BERT-base / BERT-large)")
        if getattr(cfg, "hidden_act", "gelu") != "gelu":
            raise ValueError("only the erf GELU of the reference config is on the path")
        self.num_labels = cfg.num_labels
        self._layout = _Layout(cfg)
        lay = self._layout
        # fp32 master weights: ONE flat tensor, every nn.Parameter is a view into it
        self._flat = torch.zeros(lay.total, dtype=torch.float32)
        self._build_skeleton()
        self._init_weights()
        self._engine = None
        self._optimizer = None
        self._ddp = None
        self._grads_live = False     # an eager backward has produced gradients no optimizer.step() has consumed yet
        self._no_sync = False        # inside no_sync(): training forwards accumulate their gradients

    # ---- module skeleton reproducing HF parameter paths -------------------------------------------------------
    def _build_skeleton(self):
        cfg = self.config
        self._params_by_name = OrderedDict()
        root = self

        def holder(parent, path):
            cur = parent
            for part in path:
                if part.isdigit():
                    cur = cur[int(part)]
                    continue
                if not hasattr(cur, part):
                    setattr(cur, part, nn.ModuleList() if part == "layer" else _Holder())
                cur = getattr(cur, part)
            return cur

        # registration order fixes named_parameters() order: embeddings, encoder, pooler, classifier (as HF)
        holder(root, ["bert", "embeddings"])
        enc = holder(root, ["bert", "encoder"])
        enc.layer = nn.ModuleList([_Holder() for _ in range(cfg.num_hidden_layers)])
        for name in _hf_order(cfg):
            off, shape = self._layout.entries[name]
            n = 1
            for s in shape:
                n *= s
            parts = name.split(".")
            mod = holder(root, parts[:-1])
            p = nn.Parameter(self._flat[off:off + n].view(shape))
            p._b2_owner = self
            p._b2_name = name
            mod.register_parameter(parts[-1], p)
            self._params_by_name[name] = p
        # transformers 4.28.1 (the reference's pin) keeps position_ids as a persistent buffer in checkpoints
        emb = holder(root, ["bert", "embeddings"])
        emb.register_buffer("position_ids", torch.arange(cfg.max_position_embeddings).unsqueeze(0), persistent=True)

    def _init_weights(self):
        """HF ``_init_weights``: N(0, initializer_range) for Linear/Embedding weights, zero pad row / biases,
        LayerNorm (1, 0)  (SP/transformers/models/bert/modeling_bert.py `_init_weights`)."""
        cfg = self.config
        with torch.no_grad():
            for name, p in self._params_by_name.items():
                if "LayerNorm.weight" in name:
                    p.fill_(1.0)
                elif name.endswith(".bias") or "LayerNorm.bias" in name:
                    p.zero_()
                else:
                    p.normal_(mean=0.0, std=cfg.initializer_range)
            pad = getattr(cfg, "pad_token_id", None)
            if pad is not None:
                self._params_by_name["bert.embeddings.word_embeddings.weight"][pad].zero_()

    # ---- construction helpers ----------------------------------------------------------------------------------
    @classmethod
    def from_config(cls, config, seed=None):
        if seed is not None:
            torch.manual_seed(seed)
        return cls(config)

    @classmethod
    def from_pretrained(cls, model_path, config=None, **kwargs):
        """Loads HF-format weights (``pytorch_model.bin`` / ``model.safetensors``) when present; like HF, tensors
        absent from the checkpoint (the fresh classifier) keep their random init."""
        if config is None:
            config = BertConfig.from_pretrained(model_path, **kwargs)
        model = cls(config)
        sd = None
        binf = os.path.join(model_path, "pytorch_model.bin")
        sft = os.path.join(model_path, "model.safetensors")
        if os.path.exists(binf):
            sd = torch.load(binf, map_location="cpu")
        elif os.path.exists(sft):
            from safetensors.torch import load_file
            sd = load_file(sft)
        if sd is None:
            raise FileNotFoundError("no pytorch_model.bin / model.safetensors under %s" % model_path)
        model.load_state_dict(sd, strict=False)
        return model

    # ---- device movement keeps the flat storage ---------------------------------------------------------------
    def _apply(self, fn, recurse=True):
        new_flat = fn(self._flat)
        if new_flat.dtype != torch.float32:
            raise TypeError("master weights stay fp32 (the kernels compute in bf16 from a shadow copy)")
        self._flat = new_flat.contiguous()
        for name, p in self._params_by_name.items():
            off, shape = self._layout.entries[name]
            n = p.numel()
            p.data = self._flat[off:off + n].view(shape)
        for mod in self.modules():
            for key, buf in list(mod._buffers.items()):
                if buf is not None:
                    mod._buffers[key] = fn(buf)
        if self._flat.is_cuda:
            self._engine = _Engine(self)
        else:
            self._engine = None
        return self

    def _rebind_flat(self, new_flat):
        """moves the fp32 masters into `new_flat` (same size; e.g. the DDP wrapper's peer-visible buffer) and re-points
        every nn.Parameter view at it"""
        if new_flat.dtype != torch.float32 or new_flat.numel() != self._flat.numel():
            raise ValueError("_rebind_flat: need an fp32 buffer of %d elements" % self._flat.numel())
        new_flat.copy_(self._flat)
        self._flat = new_flat
        for name, p in self._params_by_name.items():
            off, shape = self._layout.entries[name]
            p.data = self._flat[off:off + p.numel()].view(shape)

    # ---- state dict -----------------------------------------------------------------------------------------------
    def load_state_dict(self, state_dict, strict=True, assign=False):
        own = self._params_by_name
        missing = [k for k in own if k not in state_dict]
        unexpected = [k for k in state_dict if k not in own and not k.endswith("position_ids")
                      and not k.endswith("embeddings.token_type_ids")]
        if strict and (missing or unexpected):
            raise RuntimeError("Error(s) in loading state_dict: missing %s unexpected %s" % (missing, unexpected))
        with torch.no_grad():
            for k, p in own.items():
                if k in state_dict:
                    src = state_dict[k]
                    if tuple(src.shape) != tuple(p.shape):
                        raise RuntimeError("size mismatch for %s: %s vs %s" % (k, tuple(src.shape), tuple(p.shape)))
                    p.copy_(src.to(dtype=torch.float32))
        if self._engine is not None:
            self._engine.refresh_shadow()
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    def state_dict(self, *args, **kwargs):
        if self._optimizer is not None:
            self._optimizer.flush_pending()      # a pipelined train step may still owe its update
        if self._ddp is not None:
            self._ddp._gather_master()
        return super().state_dict(*args, **kwargs)

    # ---- forward ------------------------------------------------------------------------------------------------------
    def forward(self, input_ids=None, token_type_ids=None, attention_mask=None, labels=None, position_ids=None,
                segments=None, cls_index=None, **unused):
        """`position_ids` / `segments` / `cls_index` (all three or none): the batch is PACKED -- the rows of
        `input_ids` are the 128-token bins of `packing.pack_batch`, logits come back one row per original sequence."""
        if self._engine is None:
            raise RuntimeError("BertForSequenceClassification (b200) only runs on CUDA: call model.cuda() first; "
                               "there is no CPU path.")
        if input_ids is None:
            raise ValueError("input_ids is required")
        if self._optimizer is not None:
            self._optimizer.flush_pending()      # a pipelined train step may still owe its update
        packed = None
        if segments is not None or cls_index is not None:
            if position_ids is None or segments is None or cls_index is None:
                raise ValueError("a packed batch needs position_ids, segments and cls_index together")
            packed = (position_ids, segments, cls_index)
        elif position_ids is not None:
            raise ValueError("position_ids are only supported for packed batches (with segments and cls_index)")
        if torch.is_grad_enabled() and self.training:
            anchor = self._params_by_name["classifier.bias"]
            logits, loss = _StepFn.apply(anchor, self, input_ids, token_type_ids, attention_mask, labels, packed)
            return SequenceClassifierOutput(loss=loss if labels is not None else None, logits=logits)
        logits, loss = self._engine.forward(input_ids, token_type_ids, attention_mask, labels,
                                            training=self.training, need_backward=False, packed=packed)
        return SequenceClassifierOutput(loss=None if loss is None else loss.clone(), logits=logits.clone())

    @contextlib.contextmanager
    def no_sync(self):
        """Gradient accumulation, as torch DDP's ``no_sync()``: the backward of a training forward run inside the
        context ADDS its gradient to the model's fp32 accumulator (no exchange, no update).  The first backward outside
        it is the window's last micro-batch: the gradient space then holds the sum, and ``optimizer.step()`` applies it.
        Loss scaling stays with the caller (``criterion(...) / k``).  Needed on one GPU, where there is no wrapper."""
        prev = self._no_sync
        self._no_sync = True
        try:
            yield
        finally:
            self._no_sync = prev

    def _notify_backward_done(self):
        if self._ddp is not None:
            self._ddp._on_backward_done()

    # ---- test / tooling helpers -----------------------------------------------------------------------------------------
    def grad_dict(self):
        """fp32 copies of the (bf16) gradients of the last backward, keyed by HF parameter name."""
        if self._engine is None:
            raise RuntimeError("no engine (model not on CUDA)")
        out = OrderedDict()
        g = self._engine.grads
        for name, p in self._params_by_name.items():
            off, shape = self._layout.entries[name]
            out[name] = g[off:off + p.numel()].view(shape).float()
        return out


class _Engine:
    """Owns the device-side state of one model replica and drives the kernels (forward, backward)."""

    def __init__(self, model):
        L.load()
        self.model = model
        self.cfg = cfg = model.config
        self.lay = model._layout
        self.dev = model._flat.device
        self.H, self.I = cfg.hidden_size, cfg.intermediate_size
        self.heads, self.nl, self.C = cfg.num_attention_heads, cfg.num_hidden_layers, cfg.num_labels
        self.p_hidden = float(cfg.hidden_dropout_prob)
        self.p_attn = float(cfg.attention_probs_dropout_prob)
        cd = getattr(cfg, "classifier_dropout", None)
        self.p_cls = float(cd if cd is not None else cfg.hidden_dropout_prob)
        n = self.lay.total
        self.shadow = torch.empty(n, dtype=torch.bfloat16, device=self.dev)   # bf16 copy the GEMMs read
        self.grads = torch.zeros(n, dtype=torch.bfloat16, device=self.dev)    # bf16 gradient bucket space
        self.rng = torch.zeros(2, dtype=torch.int64, device=self.dev)         # {seed, step} for the dropout streams
        self.owner = torch.empty(cfg.vocab_size, dtype=torch.int32, device=self.dev)
        self.split_ws = torch.empty(64 << 20, dtype=torch.uint8, device=self.dev)
        self.partials = torch.empty(32 << 20, dtype=torch.uint8, device=self.dev)   # column-sum partials; the embedding
        # backward's fp32 owner-row accumulators ([tokens + seq*types][H] fp32 = 13.4 MB at config A)
        self._ws = {}
        self._saved = None
        # gradient accumulation (no_sync): fp32 sum over the pending micro-batches of a window, allocated by the first
        # accumulating backward; `fold` = (b2_grad_accumulate mode, scale) for the backward about to run, or None
        self.accum = None
        self.accum_pending = 0
        self.fold = None
        self.wgrad_stream = torch.cuda.Stream(device=self.dev)
        self.opt_stream = torch.cuda.Stream(device=self.dev)
        self.accum_dgrad = os.environ.get("B2_ACCUM_DGRAD", "1") != "0"
        self.grouped_wgrad = os.environ.get("B2_GROUPED_WGRAD", "1") != "0"
        # experimental, off: measured 4.17 ms/step vs 3.94 with the separate per-bucket AdamW launches -- the epilogue's
        # optimizer-state round trips (one 4 KB staging tile per warp) keep too few bytes in flight; see DESIGN.md 4.3
        self.fused_adamw = os.environ.get("B2_FUSED_ADAMW", "0") == "1"
        self.fused_adamw_active = False
        # cache of the forward's attention-dropout decisions for the backward (1 bit per (b, h, q, k), bit-exact against
        # the Philox replica): neutral in round 1 (3.96 vs 3.95 ms/step), +1.4 % now that the step body runs on a
        # high-priority stream (8 232 vs 8 117 samples/s, two A/B pairs in one run) -> on by default, B2_ATTN_KEEP_BITS=0
        # regenerates the masks in the backward instead
        self.attn_keep_bits = os.environ.get("B2_ATTN_KEEP_BITS", "1") != "0"
        self.use_wgrad_stream = os.environ.get("B2_WGRAD_STREAM", "1") != "0"
        # dense + bias + dropout + residual + LayerNorm as ONE cluster kernel (b2_gemm_ln_fwd) for the two N = hidden
        # GEMMs of a layer, when the hidden size has a row-cluster tiling (768, 1024) and the device can co-schedule
        # the 8-CTA clusters; otherwise (and with B2_FUSED_LN=0) the GEMM epilogue + separate LayerNorm launch
        self.fused_ln = (os.environ.get("B2_FUSED_LN", "1") != "0" and self.H in (768, 1024) and
                         int(L.load().b2_gemm_ln_max_clusters(self.H)) > 0)
        # fp32 accumulators for the bias gradients that kernels produce as a side effect of their epilogues (QKV bias
        # from attention backward, intermediate bias from the GELU' dgrad): per layer [3H | I]; one finishing launch
        # per step turns them into bf16 gradients and re-zeroes them
        # ... and for the LayerNorm-backward column sums (d_gamma, d_beta, dense-bias gradient of the branch): per
        # layer [3H qkv | I intermediate | 3H output-LN sets | 3H attention-output-LN sets]
        H_, I_ = self.H, self.I
        per = self.acc_per_layer = 9 * H_ + I_
        self.bias_acc = torch.zeros(max(1, self.nl * per), dtype=torch.float32, device=self.dev)
        segs = []
        for l in range(self.nl):
            pre = "bert.encoder.layer.%d." % l
            o = self.lay.off
            segs.append([l * per, o(pre + "attention.self.query.bias"), 3 * H_])
            segs.append([l * per + 3 * H_, o(pre + "intermediate.dense.bias"), I_])
            b2_ = l * per + 3 * H_ + I_
            segs.append([b2_, o(pre + "output.LayerNorm.weight"), H_])
            segs.append([b2_ + H_, o(pre + "output.LayerNorm.bias"), H_])
            segs.append([b2_ + 2 * H_, o(pre + "output.dense.bias"), H_])
            b1_ = b2_ + 3 * H_
            segs.append([b1_, o(pre + "attention.output.LayerNorm.weight"), H_])
            segs.append([b1_ + H_, o(pre + "attention.output.LayerNorm.bias"), H_])
            segs.append([b1_ + 2 * H_, o(pre + "attention.output.dense.bias"), H_])
        self.segs_per_layer = 8
        self.bias_segs = torch.tensor(segs if segs else [[0, 0, 0]], dtype=torch.int64, device=self.dev)
        s = self.stream()
        L.call("b2_embed_owner_init", L.ptr(self.owner), cfg.vocab_size, s)
        L.call("b2_rng_seed", L.ptr(self.rng), int(torch.initial_seed()) & ((1 << 63) - 1), 0, s)
        self.refresh_shadow()

    # ---- plumbing ----
    def stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def rebind(self, shadow, grads):
        """DDP moves the exchanged buffers into IPC-shared allocations."""
        shadow.copy_(self.shadow)
        grads.zero_()
        self.shadow, self.grads = shadow, grads

    def refresh_shadow(self):
        L.call("b2_cast_f32_to_bf16", L.ptr(self.model._flat), L.ptr(self.shadow), self.lay.total, self.stream())

    def ensure_accum(self):
        """the fp32 accumulator (zeroed; a local buffer, never shared with peers)"""
        if self.accum is None:
            self.accum = torch.zeros(self.lay.total, dtype=torch.float32, device=self.dev)
        return self.accum

    def fold_range(self, begin, end, mode, scale, stream):
        L.call("b2_grad_accumulate", self.ensure_accum().data_ptr(), self.grads.data_ptr(), begin, end, float(scale),
               mode, stream)

    def discard_accum(self):
        """drops the micro-batches not applied yet (optimizer.zero_grad)"""
        if self.accum_pending:
            L.call("b2_zero", self.accum.data_ptr(), 4 * self.accum.numel(), self.stream())
            self.accum_pending = 0

    def seed_dropout(self, seed, step=0):
        L.call("b2_rng_seed", L.ptr(self.rng), int(seed), int(step), self.stream())

    def w(self, name):
        return self.shadow.data_ptr() + 2 * self.lay.off(name)

    def g(self, name):
        return self.grads.data_ptr() + 2 * self.lay.off(name)

    def workspace(self, B, S, Bo=None):
        """B x S token rows; Bo = number of sequences the head sees (packed bins: B bins carry Bo >= B sequences)"""
        Bo = B if Bo is None else Bo
        key = (B, S, Bo)
        ws = self._ws.get(key)
        if ws is not None:
            return ws
        H, I, M, nl = self.H, self.I, B * S, self.nl
        bf, f32, dev = torch.bfloat16, torch.float32, self.dev

        def e(*shape, dtype=bf):
            return torch.empty(*shape, dtype=dtype, device=dev)

        ws = {
            "emb_out": e(M, H), "emb_pre": e(M, H), "emb_mean": e(M, dtype=f32), "emb_rstd": e(M, dtype=f32),
            # fp32 residual stream of the forward (fused dense + LayerNorm path): the LayerNorm outputs are kept
            # unrounded for the NEXT block's residual add; the bf16 copies above / below feed the GEMMs
            "emb_out_f": e(M, H, dtype=f32) if self.fused_ln else None,
            "ids32": e(M, dtype=torch.int32), "tt32": e(M, dtype=torch.int32), "pos32": e(M, dtype=torch.int32),
            "layers": [
                {"qkv": e(M, 3 * H), "ctx": e(M, H), "lse": e(B * self.heads * S, dtype=f32),
                 # attention-dropout decisions of the forward, 1 bit per (b, h, q, k): read back by the backward
                 "keep": (e(B * self.heads * S * (S // 64), dtype=torch.int64)
                          if (S == 128 and self.attn_keep_bits) else None),
                 "z1": e(M, H),
                 "x1": e(M, H), "mean1": e(M, dtype=f32), "rstd1": e(M, dtype=f32), "u": e(M, I), "h": e(M, I),
                 "z2": e(M, H), "x2": e(M, H), "mean2": e(M, dtype=f32), "rstd2": e(M, dtype=f32),
                 "x1f": e(M, H, dtype=f32) if self.fused_ln else None,
                 "x2f": e(M, H, dtype=f32) if (self.fused_ln and li < nl - 1) else None}
                for li in range(nl)],
            "pooled": e(Bo, H), "logits": e(Bo, self.C, dtype=f32), "loss": e((), dtype=f32),
            "dlogits": e(Bo, self.C, dtype=f32), "dloss_logits": e(Bo, self.C, dtype=f32),
            # gradient of the residual stream: fp32 (12 layers of residual adds would otherwise each round it to bf16);
            # dzd / dz1d are the bf16 (dropout-masked) copies the tensor cores consume
            "dxA": e(M, H, dtype=f32), "dxB": e(M, H, dtype=f32), "dz": e(M, H, dtype=f32),
            "dz1": e(M, H, dtype=f32), "emb_dx": e(M, H), "dctx": e(M, H), "head_scratch": e(2 * Bo, H, dtype=f32),
            # operands of the weight-gradient GEMMs, double-buffered by layer parity (see _backward_from_dlogits)
            "dzd": [e(M, H), e(M, H)], "dz1d": [e(M, H), e(M, H)], "dU": [e(M, I), e(M, I)],
            "dqkv": [e(M, 3 * H), e(M, 3 * H)],
            "dq_accum": e(M, H, dtype=f32) if S > 128 else None,
            "zeros_tt": torch.zeros(B, S, dtype=torch.int64, device=dev),
        }
        self._ws[key] = ws
        return ws

    def gemm_grouped(self, problems, stream):
        """independent GEMMs behind one launch where the library can group them (the layer's weight gradients)"""
        arr = (L.GemmArgs * len(problems))(*problems)
        L.call("b2_gemm_bf16_grouped", arr, len(problems), stream)

    def gemm(self, M, N, K, A, lda, a_major, Bm, ldb, b_major, D, ldd, epi=L.EPI_NONE, bias=None, aux_in=None,
             ld_aux_in=0, aux_out=None, ld_aux_out=0, p=0.0, site=0, split=False, stream=None, colsum=None,
             defer=None):
        """defer: a list -> the problem is appended to it instead of being launched (see gemm_grouped)"""
        a = L.GemmArgs()
        a.M, a.N, a.K = M, N, K
        a.A, a.lda, a.a_major = A, lda, a_major
        a.B, a.ldb, a.b_major = Bm, ldb, b_major
        a.D, a.ldd, a.epilogue = D, ldd, epi
        a.bias, a.aux_in, a.ld_aux_in, a.aux_out, a.ld_aux_out = bias, aux_in, ld_aux_in, aux_out, ld_aux_out
        a.dropout_p, a.rng_state, a.rng_site = p, self.rng.data_ptr(), site
        if split:
            a.workspace, a.workspace_bytes = self.split_ws.data_ptr(), self.split_ws.numel()
        else:
            a.workspace, a.workspace_bytes = None, 0
        a.force_bn = int(os.environ.get("B2_FORCE_BN", "0"))
        a.force_splits = 0
        a.force_kernel = int(os.environ.get("B2_FORCE_KERNEL", "0"))
        a.debug_timing = None
        a.colsum_out = colsum
        if defer is not None:
            defer.append(a)
            return
        L.call("b2_gemm_bf16", a, stream if stream is not None else self.stream())

    def dense_dropout_residual_layernorm(self, M, K, A, W, bias, resid, resid_f, p, site, gamma, beta, z, y, y_f, mean,
                                         rstd):
        """y = LayerNorm(dropout(A W^T + bias) + resid) with z = the pre-LN sum kept for the backward
        (BertSelfOutput / BertOutput, modeling_bert.py:294-298, :352-356).  Fused path: ONE cluster kernel, the
        residual comes in as fp32 (resid_f), the output leaves as bf16 (y) and fp32 (y_f, may be None)."""
        H = self.H
        s = self.stream()
        eps = float(self.cfg.layer_norm_eps)
        if self.fused_ln:
            a = L.GemmArgs()
            a.M, a.N, a.K = M, H, K
            a.A, a.lda, a.a_major = A, K, L.MAJOR_K
            a.B, a.ldb, a.b_major = W, K, L.MAJOR_K
            a.D, a.ldd, a.epilogue = z, H, L.EPI_BIAS_DROPOUT_RESIDUAL
            a.bias, a.aux_in, a.ld_aux_in, a.aux_out, a.ld_aux_out = bias, resid_f, H, None, 0
            a.dropout_p, a.rng_state, a.rng_site = p, self.rng.data_ptr(), site
            a.workspace, a.workspace_bytes = None, 0
            a.force_bn = a.force_splits = a.force_kernel = 0
            a.debug_timing, a.colsum_out = None, None
            L.call("b2_gemm_ln_fwd", a, gamma, beta, eps, y, H, y_f, H if y_f else 0, mean, rstd, s)
            return
        self.gemm(M, H, K, A, K, L.MAJOR_K, W, K, L.MAJOR_K, z, H, L.EPI_BIAS_DROPOUT_RESIDUAL, bias=bias,
                  aux_in=resid, ld_aux_in=H, p=p, site=site)
        L.call("b2_layernorm_fwd", z, gamma, beta, M, H, eps, y, mean, rstd, s)

    # ---- forward --------------------------------------------------------------------------------------------------------
    def forward(self, input_ids, token_type_ids, attention_mask, labels, training, need_backward, packed=None,
                weight_events=None):
        """packed: None, or (position_ids int64 [bins, 128], segments int32 [bins, 128], cls_index int64 [batch]) --
        the rows of `input_ids` are then 128-token bins produced by packing.pack_batch, not sequences.
        weight_events: None, or one event per bucket (forward order) after which that bucket's bf16 weights are
        current (pipelined optimizer, optim.AdamW.apply_pending): each is awaited right before its first use."""
        cfg, H, I = self.cfg, self.H, self.I
        if input_ids.dim() != 2:
            raise ValueError("input_ids must be [batch, seq]")
        B, S = input_ids.shape
        Bo = B
        if packed is not None:
            pos_ids, segs, cls_rows = packed
            if S != 128:
                raise ValueError("packed bins are 128 tokens long (got %d)" % S)
            if attention_mask is not None:
                raise ValueError("packed bins carry their own (block-diagonal) mask: pass attention_mask=None")
            for t, nm, dt, shape in ((pos_ids, "position_ids", torch.int64, (B, S)), (segs, "segments", torch.int32, (B, S)),
                                     (cls_rows, "cls_index", torch.int64, None)):
                if t.device != self.dev or t.dtype != dt or (shape is not None and tuple(t.shape) != shape):
                    raise TypeError("%s must be a %s tensor%s on %s" % (nm, dt, "" if shape is None else " of shape %s"
                                                                        % (shape,), self.dev))
            pos_ids, segs, cls_rows = pos_ids.contiguous(), segs.contiguous(), cls_rows.contiguous().view(-1)
            Bo = cls_rows.numel()
        if B == 0 or S == 0:
            raise ValueError("empty batch")
        if S % 128 != 0 or S > 512 or S > cfg.max_position_embeddings:
            raise ValueError("seq_len=%d: the attention kernel covers multiples of 128 up to 512 "
                             "(the reference pads every batch to max_seq_len=128)" % S)
        for t, nm in ((input_ids, "input_ids"), (token_type_ids, "token_type_ids"),
                      (attention_mask, "attention_mask"), (labels, "labels")):
            if t is not None:
                if t.device != self.dev:
                    raise RuntimeError("%s is on %s, model on %s" % (nm, t.device, self.dev))
                if t.dtype != torch.int64:
                    raise TypeError("%s must be int64 (as the reference Collate produces)" % nm)
        ws = self.workspace(B, S, Bo)
        M = B * S
        s = self.stream()
        ids = input_ids.contiguous()
        tt = (token_type_ids if token_type_ids is not None else ws["zeros_tt"]).contiguous()
        mask = attention_mask.contiguous() if attention_mask is not None else None
        p_h = self.p_hidden if training else 0.0
        p_a = self.p_attn if training else 0.0
        p_c = self.p_cls if training else 0.0
        rng = self.rng.data_ptr()
        w = self.w
        KM, MN = L.MAJOR_K, L.MAJOR_MN

        cur = torch.cuda.current_stream(self.dev)
        if weight_events is not None:
            cur.wait_event(weight_events[0])
        emb_w = (w("bert.embeddings.word_embeddings.weight"), w("bert.embeddings.position_embeddings.weight"),
                 w("bert.embeddings.token_type_embeddings.weight"), w("bert.embeddings.LayerNorm.weight"),
                 w("bert.embeddings.LayerNorm.bias"))
        emb_out = (L.ptr(ws["emb_out"]), L.ptr(ws["emb_out_f"]), L.ptr(ws["emb_pre"]), L.ptr(ws["emb_mean"]),
                   L.ptr(ws["emb_rstd"]), L.ptr(ws["ids32"]), L.ptr(ws["tt32"]))
        if packed is None:
            L.call("b2_embed_fwd", ids.data_ptr(), tt.data_ptr(), B, S, *emb_w, H, cfg.vocab_size, cfg.type_vocab_size,
                   float(cfg.layer_norm_eps), p_h, rng, 0, *emb_out, s)
        else:
            L.call("b2_embed_fwd_packed", ids.data_ptr(), tt.data_ptr(), pos_ids.data_ptr(),
                   cfg.max_position_embeddings, B, S, *emb_w, H, cfg.vocab_size, cfg.type_vocab_size,
                   float(cfg.layer_norm_eps), p_h, rng, 0, *emb_out, L.ptr(ws["pos32"]), s)
        x, xf = ws["emb_out"], ws["emb_out_f"]
        for l in range(self.nl):
            a = ws["layers"][l]
            pre = "bert.encoder.layer.%d." % l
            if weight_events is not None:
                cur.wait_event(weight_events[1 + l])
            self.gemm(M, 3 * H, H, x.data_ptr(), H, KM, w(pre + "attention.self.query.weight"), H, KM,
                      a["qkv"].data_ptr(), 3 * H, L.EPI_BIAS, bias=w(pre + "attention.self.query.bias"))
            if packed is None:
                L.call("b2_attention_fwd", a["qkv"].data_ptr(), L.ptr(mask), B, S, self.heads, 64, p_a, rng, 1 + 3 * l,
                       a["ctx"].data_ptr(), a["lse"].data_ptr(), L.ptr(a["keep"]) if need_backward else None, s)
            else:
                L.call("b2_attention_fwd_packed", a["qkv"].data_ptr(), segs.data_ptr(), B, self.heads, 64, p_a, rng,
                       1 + 3 * l, a["ctx"].data_ptr(), a["lse"].data_ptr(),
                       L.ptr(a["keep"]) if need_backward else None, s)
            self.dense_dropout_residual_layernorm(
                M, H, a["ctx"].data_ptr(), w(pre + "attention.output.dense.weight"),
                w(pre + "attention.output.dense.bias"), x.data_ptr(), L.ptr(xf), p_h, 2 + 3 * l,
                w(pre + "attention.output.LayerNorm.weight"), w(pre + "attention.output.LayerNorm.bias"),
                a["z1"].data_ptr(), a["x1"].data_ptr(), L.ptr(a["x1f"]), a["mean1"].data_ptr(), a["rstd1"].data_ptr())
            self.gemm(M, I, H, a["x1"].data_ptr(), H, KM, w(pre + "intermediate.dense.weight"), H, KM,
                      a["h"].data_ptr(), I, L.EPI_BIAS_GELU, bias=w(pre + "intermediate.dense.bias"),
                      aux_out=a["u"].data_ptr(), ld_aux_out=I)
            self.dense_dropout_residual_layernorm(
                M, I, a["h"].data_ptr(), w(pre + "output.dense.weight"), w(pre + "output.dense.bias"),
                a["x1"].data_ptr(), L.ptr(a["x1f"]), p_h, 3 + 3 * l, w(pre + "output.LayerNorm.weight"),
                w(pre + "output.LayerNorm.bias"), a["z2"].data_ptr(), a["x2"].data_ptr(), L.ptr(a["x2f"]),
                a["mean2"].data_ptr(), a["rstd2"].data_ptr())
            x, xf = a["x2"], a["x2f"]
        if weight_events is not None:
            cur.wait_event(weight_events[-1])         # the head's bucket (the last layer's, or its own)
        head_w = (w("bert.pooler.dense.weight"), w("bert.pooler.dense.bias"), w("classifier.weight"),
                  w("classifier.bias"))
        if packed is None:
            L.call("b2_head_fwd", x.data_ptr(), B, S, H, *head_w, self.C, p_c, rng, 1 + 3 * self.nl,
                   ws["pooled"].data_ptr(), ws["logits"].data_ptr(), s)
        else:
            L.call("b2_head_fwd_packed", x.data_ptr(), cls_rows.data_ptr(), Bo, H, *head_w, self.C, p_c, rng,
                   1 + 3 * self.nl, ws["pooled"].data_ptr(), ws["logits"].data_ptr(), s)
        loss = None
        if labels is not None:
            lab = labels.contiguous().view(-1)
            if lab.numel() != Bo:
                raise ValueError("labels must be [batch]")
            L.call("b2_ce_fwd_bwd", ws["logits"].data_ptr(), lab.data_ptr(), Bo, self.C, ws["loss"].data_ptr(),
                   ws["dloss_logits"].data_ptr() if need_backward else None, s)
            loss = ws["loss"]
        if need_backward:
            self._saved = (B, S, mask, p_h, p_a, p_c, None if packed is None else (segs, cls_rows))
        return ws["logits"], loss

    # ---- backward ---------------------------------------------------------------------------------------------------------
    def backward(self, d_logits, d_loss=None, stream=None):
        """d_logits: fp32 [B, C] gradient wrt the returned logits; d_loss: optional scalar gradient wrt HF's loss."""
        if self._saved is None:
            raise RuntimeError("backward called without a training forward")
        B, S, mask, p_h, p_a, p_c, packed = self._saved
        self._saved = None
        Bo = B if packed is None else packed[1].numel()
        ws = self.workspace(B, S, Bo)
        dl = ws["dlogits"]
        if d_logits is not None:
            dl.copy_(d_logits.to(torch.float32).reshape(Bo, self.C))
        else:
            dl.zero_()
        if d_loss is not None:
            dl.add_(ws["dloss_logits"] * d_loss.to(torch.float32))
        return self._backward_from_dlogits(dl, B, S, mask, p_h, p_a, p_c, packed)

    def _backward_from_dlogits(self, dl, B, S, mask, p_h, p_a, p_c, packed=None):
        cfg, H, I, M = self.cfg, self.H, self.I, B * S
        Bo = B if packed is None else packed[1].numel()
        ws = self.workspace(B, S, Bo)
        s = self.stream()
        rng = self.rng.data_ptr()
        w, g = self.w, self.g
        KM, MN = L.MAJOR_K, L.MAJOR_MN
        scratch, scratch_bytes = self.partials.data_ptr(), self.partials.numel()
        hooks = self.model._ddp

        # embedding-table gradients are scatter targets: clear the whole bucket (word rows not in the batch, unused
        # position rows and padding must read as zero for the dense DDP/AdamW pass, like the reference's dense grads)
        eb, ee, _ = self.lay.buckets[0]
        L.call("b2_zero", self.grads.data_ptr() + 2 * eb, 2 * (ee - eb), s)

        x_last = ws["layers"][-1]["x2"] if self.nl > 0 else ws["emb_out"]
        head_g = (g("bert.pooler.dense.weight"), g("bert.pooler.dense.bias"), g("classifier.weight"),
                  g("classifier.bias"))
        # data gradient (d_hidden) on the main stream; the four head parameter gradients on the weight-gradient stream
        # (they belong to the last layer's bucket, whose readiness waits for that stream's marker of the layer anyway).
        # A model without encoder layers announces its head bucket right away: keep everything on one stream there.
        main0 = torch.cuda.current_stream(self.dev)
        head_side = self.wgrad_stream if (self.use_wgrad_stream and self.nl > 0) else main0
        if head_side is not main0:
            # the side stream may still be busy with the previous step's tail; it must also not overtake this step
            head_side.wait_stream(main0)
        L.call("b2_head_bwd_split", dl.data_ptr(), x_last.data_ptr(), ws["pooled"].data_ptr(),
               None if packed is None else packed[1].data_ptr(), M, Bo, S, H, w("bert.pooler.dense.weight"),
               w("classifier.weight"), self.C, p_c, rng, 1 + 3 * self.nl, *head_g, ws["dxA"].data_ptr(), 1,
               ws["head_scratch"].data_ptr(), s, None if head_side is main0 else head_side.cuda_stream)
        dx, dx_other = ws["dxA"], ws["dxB"]
        # Weight gradients are off the critical path (only the optimizer consumes them): they run on a second stream,
        # overlapping the dgrad / LayerNorm / attention chain of the main stream.  Their A operands (dzd, dU, dz1d,
        # dqkv) are double-buffered by layer parity; the main stream may reuse a buffer set only after the weight
        # gradients of the layer two steps earlier have drained (done[l + 2]).
        main = torch.cuda.current_stream(self.dev)
        side = self.wgrad_stream if self.use_wgrad_stream else main
        ss = side.cuda_stream
        done = {}

        def fork():
            if side is not main:
                ev = torch.cuda.Event()
                ev.record(main)
                side.wait_event(ev)

        # (head bucket is announced right after these helpers are defined)
        opt = self.model._optimizer
        fold = self.fold
        accumulating = fold is not None and fold[0] == L.ACCUM_ADD
        overlap_opt = hooks is None and opt is not None and getattr(opt, "_armed", False)
        # single GPU, optimizer armed by the fused step, no GradScaler: the encoder weight matrices are updated in the
        # epilogue of the grouped weight-gradient GEMM itself (no gradient round trip, no separate HBM-bound pass over
        # 85 % of the parameters); the per-bucket AdamW launches then skip those vectors.  Not while accumulating: that
        # update would read this micro-batch's gradient instead of the window's sum.
        self.fused_adamw_active = bool(overlap_opt and self.grouped_wgrad and self.fused_adamw and fold is None and
                                       getattr(opt, "grad_scale", None) is None and
                                       not getattr(opt, "_amp_seen", False))
        # a world > 1 wrapper folds each bucket on its side stream, ahead of the bucket's barrier (ddp._bucket_ready)
        ddp_hooks = hooks is not None and hooks.world > 1
        fold_stream = hooks._side if ddp_hooks else self.opt_stream

        def bucket_ready(idx, wg_event=None):
            """bucket `idx` holds its final gradients once the main stream reaches this point (and `wg_event`,
            the weight-gradient stream's marker for the layer, has fired)"""
            if hooks is not None and (ddp_hooks or fold is None):
                hooks._bucket_ready(idx, wg_event, fold)
            elif overlap_opt or fold is not None:
                # single GPU: the fold and the HBM-bound AdamW of this bucket run on their own stream under the rest
                # of backward; a non-final micro-batch is only folded
                ev = torch.cuda.Event()
                ev.record(main)
                self.opt_stream.wait_event(ev)
                if wg_event is not None:
                    self.opt_stream.wait_event(wg_event)
                b0, e0, _lbl = self.lay.buckets[idx]
                if fold is not None:
                    self.fold_range(b0, e0, fold[0], fold[1], self.opt_stream.cuda_stream)
                if overlap_opt and not accumulating:
                    opt.update_range(b0, e0, 1, 0, [self.grads.data_ptr()], [self.shadow.data_ptr()],
                                     self.opt_stream.cuda_stream, background=(idx != 0))
                    opt._pending.add(idx)

        if not self.lay.head_in_last_layer:
            bucket_ready(len(self.lay.buckets) - 1)     # (a model without encoder layers: the head is its own bucket)
        for l in reversed(range(self.nl)):
            a = ws["layers"][l]
            x_in = ws["layers"][l - 1]["x2"] if l > 0 else ws["emb_out"]
            pre = "bert.encoder.layer.%d." % l
            st = l & 1
            dzd, dU, dz1d, dqkv = ws["dzd"][st], ws["dU"][st], ws["dz1d"][st], ws["dqkv"][st]
            if side is not main and (l + 2) in done:
                main.wait_event(done[l + 2])
            # --- BertOutput: LN2 backward (+ dropout mask, bias grad), FFN2 wgrad/dgrad(+GELU')
            acc_l = self.bias_acc.data_ptr() + 4 * l * self.acc_per_layer
            # column sums (d_gamma, d_beta, d_bias) are added into this layer's fp32 accumulators by the kernel itself
            L.call("b2_layernorm_bwd_accum", dx.data_ptr(), a["z2"].data_ptr(), a["mean2"].data_ptr(),
                   a["rstd2"].data_ptr(), w(pre + "output.LayerNorm.weight"), M, H, p_h, rng, 3 + 3 * l,
                   (dx_other if self.accum_dgrad else ws["dz"]).data_ptr(), dzd.data_ptr(),
                   acc_l + 4 * (3 * H + I), s)
            # the layer's four weight gradients: launched one by one on the side stream, or (grouped_wgrad) collected
            # and issued as ONE persistent launch once the last operand (dqkv) exists
            wgrads = [] if self.grouped_wgrad else None
            if wgrads is None:
                fork()
            self.gemm(H, I, M, dzd.data_ptr(), H, MN, a["h"].data_ptr(), I, MN, g(pre + "output.dense.weight"), I,
                      split=True, stream=ss, defer=wgrads)
            # dU = (dY2 W2) * gelu'(u); its column sums (= intermediate bias gradient) accumulate in the same epilogue
            self.gemm(M, I, H, dzd.data_ptr(), H, KM, w(pre + "output.dense.weight"), I, MN, dU.data_ptr(), I,
                      L.EPI_GELU_BWD, aux_in=a["u"].data_ptr(), ld_aux_in=I, colsum=acc_l + 4 * 3 * H)
            # --- BertIntermediate
            if wgrads is None:
                fork()
            self.gemm(I, H, M, dU.data_ptr(), I, MN, a["x1"].data_ptr(), H, MN,
                      g(pre + "intermediate.dense.weight"), H, split=True, stream=ss, defer=wgrads)
            # dX1 = dZ2 + dU W1.  accum_dgrad: LayerNorm backward left dZ2 (fp32) in dx_other and the GEMM adds into
            # it (split-K slices reduce in place at L2), else the epilogue reads dZ2 as an auxiliary tile
            if self.accum_dgrad:
                self.gemm(M, H, I, dU.data_ptr(), I, KM, w(pre + "intermediate.dense.weight"), H, MN,
                          dx_other.data_ptr(), H, L.EPI_ACCUM_F32)
            else:
                self.gemm(M, H, I, dU.data_ptr(), I, KM, w(pre + "intermediate.dense.weight"), H, MN,
                          dx_other.data_ptr(), H, L.EPI_RESIDUAL_F32, aux_in=ws["dz"].data_ptr(), ld_aux_in=H)
            # --- BertSelfOutput
            L.call("b2_layernorm_bwd_accum", dx_other.data_ptr(), a["z1"].data_ptr(), a["mean1"].data_ptr(),
                   a["rstd1"].data_ptr(), w(pre + "attention.output.LayerNorm.weight"), M, H, p_h, rng, 2 + 3 * l,
                   (dx if self.accum_dgrad else ws["dz1"]).data_ptr(), dz1d.data_ptr(),
                   acc_l + 4 * (6 * H + I), s)
            if wgrads is None:
                fork()
            self.gemm(H, H, M, dz1d.data_ptr(), H, MN, a["ctx"].data_ptr(), H, MN,
                      g(pre + "attention.output.dense.weight"), H, split=True, stream=ss, defer=wgrads)
            self.gemm(M, H, H, dz1d.data_ptr(), H, KM, w(pre + "attention.output.dense.weight"), H, MN,
                      ws["dctx"].data_ptr(), H)
            # --- BertSelfAttention
            if packed is None:
                L.call("b2_attention_bwd", a["qkv"].data_ptr(), L.ptr(mask), a["ctx"].data_ptr(),
                       ws["dctx"].data_ptr(), a["lse"].data_ptr(), B, S, self.heads, 64, p_a, rng, 1 + 3 * l,
                       dqkv.data_ptr(), L.ptr(ws["dq_accum"]), acc_l if S == 128 else None, L.ptr(a["keep"]), s)
            else:
                L.call("b2_attention_bwd_packed", a["qkv"].data_ptr(), packed[0].data_ptr(), a["ctx"].data_ptr(),
                       ws["dctx"].data_ptr(), a["lse"].data_ptr(), B, self.heads, 64, p_a, rng, 1 + 3 * l,
                       dqkv.data_ptr(), acc_l, L.ptr(a["keep"]), s)
            if S != 128:   # long-sequence parity configs: separate column-sum pass into the same accumulator slot
                L.call("b2_colsum", dqkv.data_ptr(), M, 3 * H, 3 * H, g(pre + "attention.self.query.bias"),
                       scratch, scratch_bytes, s)
            fork()
            self.gemm(3 * H, H, M, dqkv.data_ptr(), 3 * H, MN, x_in.data_ptr(), H, MN,
                      g(pre + "attention.self.query.weight"), H, split=True, stream=ss, defer=wgrads)
            if wgrads is not None:
                # 108 full-K 256x256 tiles (BERT-base) in two waves of one kernel instead of four small split-K GEMMs
                # and their reduce kernels; largest problems first
                wgrads.sort(key=lambda t: -(t.M * t.N))
                if self.fused_adamw_active:
                    hp = opt.hparams()
                    hp.skip_flags = None
                    arr = (L.GemmArgs * len(wgrads))(*wgrads)
                    L.call("b2_gemm_bf16_grouped_adamw", arr, opt.fused_targets(wgrads), len(wgrads), hp,
                           L.ptr(opt._state()["step"]), ss)
                else:
                    self.gemm_grouped(wgrads, ss)
            # fp32 accumulators -> bf16 bias gradients of this layer (and re-arm them); for S != 128 the QKV segment's
            # accumulator is unused (zero) and must not overwrite the colsum result: finish only the intermediate one.
            # Every kernel that adds into this layer's accumulators is behind the fork() above, and only the optimizer /
            # exchange reads the result: the launch rides the weight-gradient stream, off the critical path.
            spl = self.segs_per_layer
            seg0 = spl * l if S == 128 else spl * l + 1
            L.call("b2_accum_finish", self.bias_acc.data_ptr(), self.grads.data_ptr(),
                   self.bias_segs.data_ptr() + 24 * seg0, spl * (l + 1) - seg0, max(3 * H, I), ss)
            if side is not main:
                done[l] = torch.cuda.Event()
                done[l].record(side)
            if self.accum_dgrad:
                self.gemm(M, H, 3 * H, dqkv.data_ptr(), 3 * H, KM, w(pre + "attention.self.query.weight"), H, MN,
                          dx.data_ptr(), H, L.EPI_ACCUM_F32)
            else:
                self.gemm(M, H, 3 * H, dqkv.data_ptr(), 3 * H, KM, w(pre + "attention.self.query.weight"), H, MN,
                          dx.data_ptr(), H, L.EPI_RESIDUAL_F32, aux_in=ws["dz1"].data_ptr(), ld_aux_in=H)
            bucket_ready(1 + l, done.get(l))   # complete only with this layer's weight gradients
        emb_in = (dx.data_ptr(), 1, ws["emb_pre"].data_ptr(), ws["emb_mean"].data_ptr(), ws["emb_rstd"].data_ptr(),
                  w("bert.embeddings.LayerNorm.weight"), ws["ids32"].data_ptr(), ws["tt32"].data_ptr())
        emb_tail = (B, S, H, cfg.vocab_size, cfg.type_vocab_size,
                    -1 if getattr(cfg, "pad_token_id", None) is None else int(cfg.pad_token_id), p_h, rng, 0,
                    g("bert.embeddings.word_embeddings.weight"), g("bert.embeddings.position_embeddings.weight"),
                    g("bert.embeddings.token_type_embeddings.weight"), g("bert.embeddings.LayerNorm.weight"),
                    g("bert.embeddings.LayerNorm.bias"), ws["emb_dx"].data_ptr(), scratch, scratch_bytes,
                    self.owner.data_ptr(), s)
        if packed is None:
            L.call("b2_embed_bwd", *emb_in, *emb_tail)
        else:
            L.call("b2_embed_bwd_packed", *emb_in, ws["pos32"].data_ptr(), *emb_tail)
        # Whoever consumes the gradients next on the main stream (optimizer.step, grad_dict) must see the weight-gradient
        # stream's work.  Under an armed DDP exchange the side stream has taken those dependencies bucket by bucket
        # (ddp._bucket_ready) and optimizer.step() joins the side stream; in every other case join here.
        ddp_overlap = (hooks is not None and hooks.world > 1 and hooks.overlap and opt is not None and
                       getattr(opt, "_armed", False) and not accumulating)
        if side is not main and not ddp_overlap:
            for l in sorted(done)[:2]:       # the last two layers processed (0 and 1) may still be in flight
                main.wait_event(done[l])
        bucket_ready(0)
        if fold is not None:
            # ordering rule of accumulation: the next backward writes gradients (the embedding bucket's clear, the head
            # gradients) at its very start, so nothing may run on the main stream before every fold has read them
            main.wait_stream(fold_stream)
            if accumulating:
                # one dropout RNG step per micro-batch: micro-batch j of a window draws the masks of step r0 + j
                L.call("b2_step_advance", None, rng, None, s)
