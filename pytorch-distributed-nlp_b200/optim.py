"""HF-semantics ``AdamW`` + the reference's ``build_optimizer`` on top of the fused CUDA update.

Reference surface: ``build_optimizer(model, args)`` (multi-gpu-distributed-cls.py:100-111) returning an object with
``zero_grad()`` [:172] and ``step()`` [:174].  The arithmetic is transformers 4.28.1 ``optimization.py::AdamW.step``
(eps added to sqrt(v) before the bias correction, weight decay applied after the Adam update with the updated
weight, ``correct_bias=True``) — NOT ``torch.optim.AdamW``.  One kernel updates the whole flat parameter space
(or, under DDP, this rank's slice of every bucket, fused with the gradient mean over peers).
"""
import os

import torch

from . import _lib as L


class AdamW(torch.optim.Optimizer):
    # torch.cuda.amp.GradScaler contract for optimizers that unscale themselves (torch/amp/grad_scaler.py `step`):
    # the scaler sets `self.grad_scale` (device fp32 scalar) / `self.found_inf` around step() instead of walking
    # `.grad` tensors -- which do not exist here (gradients live in the bf16 bucket space).  This is what lets the
    # reference's -amp loop (multi-gpu-distributed-mp-amp-cls.py:166-171: autocast, scaler.scale(loss).backward(),
    # scaler.step(optimizer), scaler.update()) run unchanged.  bf16 has fp32's exponent range, so no overflow check
    # is needed: found_inf stays 0 and the scale only has to be divided out (exactly: it is a power of two).
    _step_supports_amp_scaling = True

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0, correct_bias=True,
                 no_deprecation_warning=True):
        if lr < 0.0:
            raise ValueError(f"Invalid learning rate: {lr} - should be >= 0.0")
        if not 0.0 <= betas[0] < 1.0:
            raise ValueError(f"Invalid beta parameter: {betas[0]} - should be in [0.0, 1.0)")
        if not 0.0 <= betas[1] < 1.0:
            raise ValueError(f"Invalid beta parameter: {betas[1]} - should be in [0.0, 1.0)")
        if not 0.0 <= eps:
            raise ValueError(f"Invalid epsilon value: {eps} - should be >= 0.0")
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, correct_bias=correct_bias)
        super().__init__(params, defaults)
        owners = {id(getattr(p, "_b2_owner", None)) for g in self.param_groups for p in g["params"]}
        first = self.param_groups[0]["params"][0]
        self._model = getattr(first, "_b2_owner", None)
        if self._model is None or len(owners) != 1:
            raise TypeError("this AdamW drives the fused CUDA update of ONE b200 BertForSequenceClassification; "
                            "got parameters that do not belong to such a model")
        g0 = self.param_groups[0]
        for g in self.param_groups[1:]:
            if (g["lr"], tuple(g["betas"]), g["eps"], g["correct_bias"]) != \
                    (g0["lr"], tuple(g0["betas"]), g0["eps"], g0["correct_bias"]):
                raise ValueError("param groups may differ only in weight_decay (as the reference's two groups do)")
        wds = sorted({float(g["weight_decay"]) for g in self.param_groups if g["weight_decay"] > 0})
        if len(wds) > 1:
            raise ValueError("at most one non-zero weight_decay value is supported")
        self._wd = wds[0] if wds else 0.0
        lay = self._model._layout
        covered = set()
        flags = torch.zeros(lay.total // 8, dtype=torch.uint8)
        for g in self.param_groups:
            for p in g["params"]:
                off, _shape = lay.entries[p._b2_name]
                covered.add(p._b2_name)
                if g["weight_decay"] > 0:
                    flags[off // 8:(off + (p.numel() + 7) // 8 * 8) // 8] = 1
        if covered != set(lay.entries):
            raise ValueError("the fused update steps every parameter of the model; %d of %d were passed"
                             % (len(covered), len(lay.entries)))
        self._decay_flags_cpu = flags
        self._dev_state = None
        self._armed = False      # set by FusedTrainStep: per-bucket updates may start during backward
        self._pending = set()    # buckets already updated (on the engine's optimizer stream) in this step
        self._background = os.environ.get("B2_ADAMW_BACKGROUND", "1") != "0"   # one-GPU update shaped to co-reside
        # pipelined form (one GPU, captured steps only; see apply_pending): the update of step i runs at the START of
        # step i + 1, bucket by bucket in forward order on the low-priority optimizer stream, while the forward pass
        # works its way up the layers
        self._pipelined = False
        self._deferred_pending = False
        self._amp_seen = False   # a GradScaler drives this optimizer: the scale is only known inside step(), so
                                 # per-bucket updates must not start during backward
        self._model._optimizer = self

    # -- device state (fp32 moments, step counter) ------------------------------------------------------------------
    def _state(self):
        eng = self._model._engine
        if eng is None:
            raise RuntimeError("optimizer.step(): the model is not on CUDA")
        if self._dev_state is None or self._dev_state["dev"] != eng.dev:
            n = self._model._layout.total
            self._dev_state = {
                "dev": eng.dev,
                "exp_avg": torch.zeros(n, dtype=torch.float32, device=eng.dev),
                "exp_avg_sq": torch.zeros(n, dtype=torch.float32, device=eng.dev),
                "step": torch.zeros(1, dtype=torch.int64, device=eng.dev),
                "step_size": torch.zeros(1, dtype=torch.float32, device=eng.dev),   # see b2_adamw_prepare
                # pipelined form: 1.0 = the gradient space holds nothing that is not applied yet (the update kernels
                # treat it like GradScaler's found_inf: non-zero -> skip), 0.0 = gradients of the last backward pending
                "no_grads": torch.ones(1, dtype=torch.float32, device=eng.dev),
                "decay": self._decay_flags_cpu.to(eng.dev),
                "skip": self._fused_skip_flags().to(eng.dev),
            }
            self._prepare(eng.stream())
        return self._dev_state

    # ---- pipelined update (FusedTrainStep / PackedTrainStep on one GPU) ------------------------------------------------
    def enable_pipelining(self):
        """Called by the captured train steps.  Measured (B2_DEBUG_SKIP_ADAMW): launched under the backward pass, the
        0.49 ms of optimizer kernels are exposed almost in full -- the backward keeps every SM busy with GEMM CTAs that
        own the whole register file.  The forward pass does not: its two dense + LayerNorm launches per layer occupy 96
        of the 148 SMs.  So the update of step i is applied at the beginning of step i + 1: bucket by bucket in FORWARD
        order on the optimizer stream (lowest priority), layer l of the forward waiting only for bucket l's event.
        Nothing is skipped: every captured step applies one full update (the previous step's), `state_dict()`, an eager
        forward, an evaluation step and `optimizer.step()` first flush what is pending, and the arithmetic (operands,
        order, step count) is exactly that of the unpipelined step."""
        model = self._model
        # Measured (config A, one B200): 8 013 samples/s pipelined vs 8 123 unpipelined -- under the forward the update
        # time-slices with the GEMM CTAs just as it does under the backward, and a layer that has to wait for its
        # bucket's event stalls the critical path.  Correct (tests/test_model.py::test_pipelined_adamw_is_the_same_
        # training run) but slower: opt-in only (B2_PIPELINED_ADAMW=1).
        if (os.environ.get("B2_PIPELINED_ADAMW", "0") != "1" or model._ddp is not None or self._amp_seen or
                getattr(model._engine, "fused_adamw", False)):
            return False
        self._pipelined = True
        self._armed = False          # no per-bucket launches under the backward
        return True

    def apply_pending(self, in_step):
        """Applies the gradients of the last backward if they have not been applied yet (device flag, so the same
        captured nodes serve the first replay, where nothing is pending).  in_step: launched from a train step body
        on the optimizer stream, returns one event per bucket (forward order); else: on the current stream."""
        st = self._state()
        model = self._model
        eng = model._engine
        main = torch.cuda.current_stream(eng.dev)
        stream = eng.opt_stream if in_step else main
        if in_step:
            ev0 = torch.cuda.Event()
            ev0.record(main)
            stream.wait_event(ev0)
        hp = self.hparams()
        hp.grad_scale, hp.skip_flags = None, None
        hp.found_inf = st["no_grads"].data_ptr()
        gptr, sptr = L.ptr_array([eng.grads.data_ptr()]), L.ptr_array([eng.shadow.data_ptr()])
        events = []
        for (b0, e0, _lbl) in model._layout.buckets:
            L.call("b2_bucket_reduce_adamw", gptr, sptr, 1, 0, L.ptr(model._flat), L.ptr(st["exp_avg"]),
                   L.ptr(st["exp_avg_sq"]), L.ptr(st["decay"]), b0, e0, hp, L.ptr(st["step"]), stream.cuda_stream)
            if in_step:
                ev = torch.cuda.Event()
                ev.record(stream)
                events.append(ev)
        L.call("b2_step_advance", L.ptr(st["step"]), None, st["no_grads"].data_ptr(), stream.cuda_stream)
        self._prepare(stream.cuda_stream)
        return events

    def mark_grads_pending(self):
        """end of a pipelined step body: the gradient space now holds an unapplied backward; bump the dropout stream"""
        st = self._state()
        eng = self._model._engine
        s = eng.stream()
        L.call("b2_zero", st["no_grads"].data_ptr(), 4, s)
        L.call("b2_step_advance", None, L.ptr(eng.rng), None, s)
        self._deferred_pending = True

    def flush_pending(self):
        """applies a pending pipelined update now (on the current stream): called before anything reads the weights or
        overwrites the gradients outside a pipelined step body"""
        if not self._deferred_pending:
            return
        self._deferred_pending = False
        self.apply_pending(in_step=False)
        self._dev_state["no_grads"].fill_(1.0)

    def _prepare(self, stream):
        """bias-corrected step size of the NEXT update -> device float (read by the background kernel)"""
        st = self._dev_state
        L.call("b2_adamw_prepare", self.hparams(), L.ptr(st["step"]), L.ptr(st["step_size"]), stream)

    def _fused_skip_flags(self):
        """uint8 per 8-element vector: 1 for the encoder weight matrices, which the single-GPU fused step updates in the
        epilogue of the grouped weight-gradient GEMM (b2_gemm_bf16_grouped_adamw); the per-bucket update skips them."""
        lay = self._model._layout
        flags = torch.zeros(lay.total // 8, dtype=torch.uint8)
        for l in range(self._model.config.num_hidden_layers):
            pre = "bert.encoder.layer.%d." % l
            for nm in ("attention.self.query.weight", "attention.self.key.weight", "attention.self.value.weight",
                       "attention.output.dense.weight", "intermediate.dense.weight", "output.dense.weight"):
                off, shape = lay.entries[pre + nm]
                flags[off // 8:(off + shape[0] * shape[1]) // 8] = 1
        return flags

    def fused_targets(self, problems):
        """b2_fused_adamw_target_t array for weight-gradient problems whose D pointers lie in the engine's bf16 gradient
        space: the optimizer state of the same elements."""
        st = self._state()
        model = self._model
        eng = model._engine
        gbase = eng.grads.data_ptr()
        arr = (L.FusedAdamWTarget * len(problems))()
        decay = self._decay_flags_cpu
        for i, pr in enumerate(problems):
            off = (pr.D - gbase) // 2
            arr[i].master = model._flat.data_ptr() + 4 * off
            arr[i].exp_avg = st["exp_avg"].data_ptr() + 4 * off
            arr[i].exp_avg_sq = st["exp_avg_sq"].data_ptr() + 4 * off
            arr[i].shadow = eng.shadow.data_ptr() + 2 * off
            arr[i].decay = int(decay[off // 8])
        return arr

    def hparams(self):
        g = self.param_groups[0]
        hp = L.AdamWHParams()
        hp.lr, hp.beta1, hp.beta2, hp.eps = float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"])
        hp.weight_decay = float(self._wd)
        hp.correct_bias = 1 if g["correct_bias"] else 0
        gs = getattr(self, "grad_scale", None)        # set by GradScaler.step() for the duration of step()
        hp.grad_scale = gs.data_ptr() if gs is not None else None
        if gs is not None and (gs.dtype != torch.float32 or not gs.is_cuda):
            raise TypeError("grad_scale must be a CUDA fp32 scalar (torch.cuda.amp.GradScaler's)")
        hp.found_inf = self._found_inf_ptr()
        eng = self._model._engine
        st = self._dev_state
        hp.skip_flags = (st["skip"].data_ptr() if (st is not None and getattr(eng, "fused_adamw_active", False))
                         else None)
        return hp

    def _found_inf_ptr(self):
        fi = getattr(self, "found_inf", None)         # GradScaler: 0-dim fp32 tensor (or int 0 when nothing was checked)
        if isinstance(fi, torch.Tensor):
            if fi.dtype != torch.float32 or not fi.is_cuda:
                raise TypeError("found_inf must be a CUDA fp32 scalar (torch.cuda.amp.GradScaler's)")
            self._found_inf_keep = fi                 # keep the tensor alive until the kernels that read it have run
            return fi.data_ptr()
        return None

    def zero_grad(self, set_to_none=True):
        """Gradients live in the bf16 bucket space and are overwritten by every backward: nothing to clear
        (the reference's zero_grad [:172] exists only because torch accumulates into .grad).  The one real `.grad`
        is the small fp32 probe the eager backward leaves on classifier.bias for GradScaler's inf check.  Micro-batches
        accumulated under no_sync() and not applied yet are discarded, as torch discards their .grad."""
        self._model._params_by_name["classifier.bias"].grad = None
        if self._model._engine is not None:
            self._model._engine.discard_accum()
        return None

    def update_range(self, begin, end, world, rank, peer_grads, peer_shadow, stream, background=False):
        """Fused (mean over peers +) HF-AdamW on flat elements [begin, end).  background=True (one GPU, the update of
        a bucket launched while the backward pass is still running): the form shaped to run beside the GEMM CTAs;
        with nothing left to hide behind (the last bucket, or a plain optimizer.step()) the 256-thread kernel is the
        faster one (5.2 vs 3.6 TB/s alone)."""
        if os.environ.get("B2_DEBUG_SKIP_ADAMW") == "1":
            return      # MEASUREMENT ONLY (how much of the optimizer is exposed in the step): weights are not updated
        st = self._state()
        hp = self.hparams()
        model = self._model
        if (background and world == 1 and self._background and hp.grad_scale is None and hp.found_inf is None and
                hp.skip_flags is None):
            # one GPU: the form that fits beside the GEMM CTAs (csrc/optim.cu, adamw_slim_kernel)
            L.call("b2_adamw_background", peer_grads[0], peer_shadow[0], L.ptr(model._flat), L.ptr(st["exp_avg"]),
                   L.ptr(st["exp_avg_sq"]), L.ptr(st["decay"]), begin, end, hp, L.ptr(st["step_size"]), stream)
            return
        L.call("b2_bucket_reduce_adamw", L.ptr_array(peer_grads), L.ptr_array(peer_shadow), world, rank,
               L.ptr(model._flat), L.ptr(st["exp_avg"]), L.ptr(st["exp_avg_sq"]), L.ptr(st["decay"]), begin, end,
               hp, L.ptr(st["step"]), stream)

    def advance(self, stream):
        st = self._state()
        L.call("b2_step_advance", L.ptr(st["step"]), L.ptr(self._model._engine.rng), self._found_inf_ptr(), stream)
        self._prepare(stream)

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        self.flush_pending()
        if getattr(self, "grad_scale", None) is not None:
            self._amp_seen = True
        model = self._model
        eng = model._engine
        if eng is None:
            raise RuntimeError("optimizer.step(): the model is not on CUDA")
        if model._ddp is not None and model._ddp.world > 1:
            if eng.accum_pending:
                raise RuntimeError("optimizer.step() after only no_sync() backwards: the last micro-batch of a window "
                                   "must run outside no_sync(), or the ranks would step on gradients never exchanged")
            model._ddp._optimizer_step(self)
        else:
            main = torch.cuda.current_stream(eng.dev)
            s = main.cuda_stream
            if eng.accum_pending:
                # only no_sync() backwards since the last step: apply their sum (the gradient space holds the last
                # micro-batch, already added, hence scale 0)
                main.wait_stream(eng.opt_stream)
                eng.fold_range(0, model._layout.total, L.ACCUM_FINISH, 0.0, s)
                eng.accum_pending = 0
            if self._pending:
                ev = torch.cuda.Event()
                ev.record(eng.opt_stream)
                main.wait_event(ev)
            if len(self._pending) == 0:
                self.update_range(0, model._layout.total, 1, 0, [eng.grads.data_ptr()], [eng.shadow.data_ptr()], s)
            else:
                for idx, (b0, e0, _lbl) in enumerate(model._layout.buckets):
                    if idx not in self._pending:
                        self.update_range(b0, e0, 1, 0, [eng.grads.data_ptr()], [eng.shadow.data_ptr()], s)
            self._pending = set()
            self.advance(s)
        model._grads_live = False
        # the inf-check probe has served its purpose (GradScaler reads it before calling step); the -amp scripts never
        # call zero_grad, so drop it here or it would accumulate
        model._params_by_name["classifier.bias"].grad = None
        return loss

    def moments(self):
        """(exp_avg, exp_avg_sq) fp32 by HF parameter name — for tests/checkpoint tooling."""
        st = self._state()
        out = {}
        for name, p in self._model._params_by_name.items():
            off, shape = self._model._layout.entries[name]
            out[name] = (st["exp_avg"][off:off + p.numel()].view(shape), st["exp_avg_sq"][off:off + p.numel()].view(shape))
        return out


def build_optimizer(model, args):
    """Same grouping rule as the reference (multi-gpu-distributed-cls.py:100-111): no weight decay for names
    containing 'bias' or 'LayerNorm.weight'; lr = args.learning_rate; HF AdamW defaults otherwise."""
    no_decay = ['bias', 'LayerNorm.weight']
    optimizer_grouped_parameters = [
        {'params': [p for n, p in model.named_parameters() if not any(nd in n for nd in no_decay)],
         'weight_decay': args.weight_decay},
        {'params': [p for n, p in model.named_parameters() if any(nd in n for nd in no_decay)],
         'weight_decay': 0.0}
    ]
    optimizer = AdamW(optimizer_grouped_parameters, lr=args.learning_rate)
    return optimizer
