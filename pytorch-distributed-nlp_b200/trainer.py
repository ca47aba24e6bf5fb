"""The reference's ``Trainer`` / ``Args`` surface (multi-gpu-distributed-cls.py:113-257) on the B200 step.

Same methods, same argument meaning: ``on_step`` [:126-137], ``loss_reduce`` [:139-143], ``output_reduce`` [:145-155],
``train`` [:157-197], ``dev`` [:199-220], ``test`` [:222-239].  Differences, all on the hot path's periphery:
  * host batches are staged through pinned memory and copied asynchronously (the reference does four pageable,
    synchronous ``.cuda()`` copies per step, :128-131);
  * the per-step ``torch.distributed.barrier()`` [:171] is dropped: ranks are ordered by the device-side flag barriers
    inside the gradient exchange, and a host-blocking barrier only serialises forward/backward across ranks;
  * ``loss_reduce`` / ``output_reduce`` go through the peer-memory kernels when the model is the b200 DDP wrapper;
  * ``train`` uses :class:`FusedTrainStep` (the whole step captured in one CUDA graph) when ``args.fused`` is set.
"""
import contextlib
import os
import time

import numpy as np
import torch

from . import _lib as L
from .ddp import DistributedDataParallel


class Args:
    model_path = "model_hub/chinese-bert-wwm-ext"
    ckpt_path = "output/multi-gpu-distributed-cls.pt"
    max_seq_len = 128
    ratio = 0.92
    train_batch_size = 32
    dev_batch_size = 32
    weight_decay = 0.01
    epochs = 1
    learning_rate = 3e-5
    eval_step = 50
    local_rank = None
    local_world_size = None
    device_ids = None
    rank = None
    dev = False
    use_amp = False       # the -amp scripts' flag (multi-gpu-distributed-mp-amp-cls.py:160): GradScaler loop on the eager path
    fused = True          # capture fwd + bwd + exchange + AdamW in one CUDA graph
    pack = False          # pack the valid prefixes of the padded [B, 128] batches into 128-token bins (packing.py): the
                          # reference pads every row to max_seq_len although real rows average 18 tokens [:76]
    log_every = 1         # the reference prints every step (forces a D2H sync per step)
    total_step = 0
    use_grad_accumulation = False   # fabric/fabric-cls.py's accumulation: the loss is divided by grad_accumulation and
    grad_accumulation = 4           # the optimizer steps when (step + 1) % grad_accumulation == 0 (per-epoch index)


def _unwrap(model):
    return model.module if isinstance(model, DistributedDataParallel) else model


def _arm_pipelining(optimizer, grad_accumulation):
    """the pipelined update (optim.AdamW.enable_pipelining) runs on step-local gradients: not while accumulating"""
    if grad_accumulation == 1:
        optimizer.enable_pipelining()     # one GPU: the update moves under the NEXT step's forward (optim.py)
    elif optimizer._pipelined:
        raise ValueError("gradient accumulation needs the unpipelined update (B2_PIPELINED_ADAMW=0)")


class _StagedGraphStep:
    """Shared plumbing of the graph-captured steps: one pinned staging buffer for the four host tensors of a batch, one
    async H2D copy, two eager warm-up passes (first launches set kernel attributes), then capture + replay."""

    def __init__(self, model, batch_size, seq_len, use_graph=True):
        self.wrapper = model if isinstance(model, DistributedDataParallel) else None
        self.model = _unwrap(model)
        self.eng = self.model._engine
        if self.eng is None:
            raise RuntimeError("%s: model must be on CUDA" % type(self).__name__)
        dev = self.eng.dev
        self.B, self.S = batch_size, seq_len
        z = lambda *s: torch.zeros(*s, dtype=torch.int64, device=dev)
        self.d_ids, self.d_tt, self.d_mask, self.d_lab = z(batch_size, seq_len), z(batch_size, seq_len), \
            z(batch_size, seq_len), z(batch_size)
        self.h_stage = torch.empty(3 * batch_size * seq_len + batch_size, dtype=torch.int64).pin_memory()
        self.d_stage = torch.empty_like(self.h_stage, device=dev)
        self.loss_out = torch.zeros((), dtype=torch.float32, device=dev)
        self.h_loss = torch.zeros((), dtype=torch.float32).pin_memory()
        self.use_graph = use_graph
        self.graph = None
        self._warm = 0
        # gradient accumulation (train steps built with grad_accumulation > 1): a second graph for the non-final
        # micro-batches of a window; `_final` selects which one the next run_device() replays
        self.grad_accumulation = 1
        self._final = True
        self._graph_accum = None
        self._warm_accum = 0
        self._h2d_done = None
        # The step body -- the critical chain of forward / dgrad kernels -- is issued (and captured) on a HIGH-priority
        # stream, so that when an SM frees up the block scheduler hands it to the critical path before the
        # weight-gradient / optimizer streams (default, i.e. lowest, priority): measured 7 990 -> 8 093 samples/s on
        # config A.  B2_STEP_PRIORITY=0 restores the plain current stream (A/B switch).
        self._prio_stream = None
        if os.environ.get("B2_STEP_PRIORITY", "1") != "0":
            self._prio_stream = torch.cuda.Stream(device=dev, priority=-1)

    def _unstage(self):
        n = self.B * self.S
        st = self.d_stage
        self.d_ids.copy_(st[0:n].view(self.B, self.S))
        self.d_tt.copy_(st[n:2 * n].view(self.B, self.S))
        self.d_mask.copy_(st[2 * n:3 * n].view(self.B, self.S))
        self.d_lab.copy_(st[3 * n:3 * n + self.B])

    def _body(self):
        raise NotImplementedError

    def stage(self, batch_data):
        """Host batch (the dict the reference Collate yields, int64 tensors) -> pinned staging -> async H2D."""
        n = self.B * self.S
        ids, tt, mask, lab = batch_data["input_ids"], batch_data["token_type_ids"], batch_data["attention_mask"], \
            batch_data["label"]
        if tuple(ids.shape) != (self.B, self.S):
            raise ValueError("%s was built for batch %dx%d, got %s"
                             % (type(self).__name__, self.B, self.S, tuple(ids.shape)))
        hs = self.h_stage
        if self._h2d_done is not None:
            self._h2d_done.synchronize()  # previous step's copy out of the pinned staging buffer has drained
        hs[0:n].copy_(ids.reshape(-1))
        hs[n:2 * n].copy_(tt.reshape(-1))
        hs[2 * n:3 * n].copy_(mask.reshape(-1))
        hs[3 * n:3 * n + self.B].copy_(lab.reshape(-1))
        self.d_stage.copy_(hs, non_blocking=True)
        self._h2d_done = torch.cuda.Event()
        self._h2d_done.record(torch.cuda.current_stream(self.eng.dev))

    def _run_body(self):
        if self._prio_stream is None:
            self._body()
            return
        cur = torch.cuda.current_stream(self.eng.dev)
        self._prio_stream.wait_stream(cur)
        with torch.cuda.stream(self._prio_stream):
            self._body()
        cur.wait_stream(self._prio_stream)

    def run_device(self, final=True):
        """The step with inputs already staged on the device (bench `value` path).  final=False (train steps built
        with grad_accumulation > 1): a non-final micro-batch, only added to the accumulator."""
        k = self.grad_accumulation
        if not final and k == 1:
            raise ValueError("a non-final micro-batch needs a train step built with grad_accumulation > 1")
        self._final = final
        if k > 1:
            self.eng.ensure_accum()          # allocated (and zeroed) outside any capture
        self._run_device()
        opt = getattr(self, "opt", None)
        if opt is not None and opt._pipelined:
            opt._deferred_pending = True      # (a graph replay runs no Python: keep the host-side flag current)
        if k > 1:
            self.eng.accum_pending = 0 if final else self.eng.accum_pending + 1

    def _run_device(self):
        if not self.use_graph:
            self._run_body()
            return
        if not self._final:
            self._graph_accum, self._warm_accum = self._replay(self._graph_accum, self._warm_accum)
            return
        self.graph, self._warm = self._replay(self.graph, self._warm)

    def _replay(self, graph, warm):
        """one run of the body through `graph`, capturing it after two eager warm-up runs; returns (graph, warm)"""
        if graph is None:
            if warm < 2:
                # eager warm-up: first launches set kernel attributes, DDP arms its overlap path
                self._run_body()
                return None, warm + 1
            torch.cuda.synchronize(self.eng.dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                self._run_body()
        graph.replay()
        return graph, warm

    def _train_body(self, forward):
        """forward(weight_events) -> (logits, loss): the common part of the captured train steps"""
        eng, opt = self.eng, self.opt
        events = opt.apply_pending(in_step=True) if opt._pipelined else None     # step i-1's update, see optim.py
        logits, loss = forward(events)
        B, S, mask, p_h, p_a, p_c, packed = eng._saved
        eng._saved = None
        Bo = B if packed is None else packed[1].numel()
        ws = eng.workspace(B, S, Bo)
        k = self.grad_accumulation
        if k > 1:
            # the reference's loss / k, applied by the fold: ADD for a non-final micro-batch (no update, no exchange),
            # FINISH ahead of each bucket's update or exchange for the last one
            eng.fold = (L.ACCUM_FINISH if self._final else L.ACCUM_ADD, 1.0 / k)
        try:
            # d(loss)/d(logits) was produced by the CE kernel: the reference's criterion(logits, label) [:169]
            eng._backward_from_dlogits(ws["dloss_logits"], B, S, mask, p_h, p_a, p_c, packed)
        finally:
            eng.fold = None
        if not self._final:
            self.loss_out.copy_(loss)
            return
        eng.accum_pending = 0
        if opt._pipelined:
            opt.mark_grads_pending()
            torch.cuda.current_stream(eng.dev).wait_stream(eng.opt_stream)   # (step counter bump of the applied update)
        else:
            opt.step()
        self.loss_out.copy_(loss)

    def loss_to_host(self):
        self.h_loss.copy_(self.loss_out, non_blocking=True)
        torch.cuda.current_stream(self.eng.dev).synchronize()
        return float(self.h_loss)


class FusedTrainStep(_StagedGraphStep):
    """One training step == one CUDA-graph replay: H2D of the batch, embeddings -> 12 layers -> head -> CE, the full
    backward, the peer-HBM gradient exchange fused with AdamW, and the device-side step/RNG bump.  Semantically the body
    of the reference loop [:166-176] without the host round trips."""

    def __init__(self, model, optimizer, batch_size, seq_len, use_graph=True, grad_accumulation=1):
        """grad_accumulation = k > 1: micro-batches of a window scaled by 1 / k (the reference's loss / k), the
        update applied by the call with final=True"""
        super().__init__(model, batch_size, seq_len, use_graph)
        self.opt = optimizer
        self.grad_accumulation = int(grad_accumulation)
        # the fused step owns backward + optimizer: per-bucket AdamW (and, under DDP, the peer exchange) may start
        # while backward is still running
        optimizer._armed = True
        _arm_pipelining(optimizer, self.grad_accumulation)
        self.kernel_launches = None

    # the step body, expressed only with stream-ordered work (capturable)
    def _body(self):
        self._unstage()
        self._train_body(lambda ev: self.eng.forward(self.d_ids, self.d_tt, self.d_mask, self.d_lab, training=True,
                                                     need_backward=True, weight_events=ev))

    def __call__(self, batch_data, final=True):
        """batch_data: the dict the reference Collate yields (host int64 tensors).  Returns the device loss scalar
        (local rank's mean CE, like `loss` at [:169]).  final=False: a non-final micro-batch (see grad_accumulation)."""
        self.stage(batch_data)
        self.run_device(final)
        return self.loss_out


class PackedTrainStep(_StagedGraphStep):
    """FusedTrainStep for PACKED batches (packing.pack_batch): `bins` 128-token bins carrying `batch` sequences.  One
    instance (staging buffers + CUDA graph) per bin count; the Trainer keeps a small cache of them, since the number of
    bins a batch packs into varies with its lengths."""

    def __init__(self, model, optimizer, bins, batch, use_graph=True, grad_accumulation=1):
        super().__init__(model, bins, 128, use_graph)
        dev = self.eng.dev
        self.bins, self.batch = bins, batch
        self.grad_accumulation = int(grad_accumulation)
        n = bins * 128
        # pinned staging: ids | token types | positions | segments (as int64) | cls rows | labels
        self.h_stage = torch.empty(4 * n + 2 * batch, dtype=torch.int64).pin_memory()
        self.d_stage = torch.empty_like(self.h_stage, device=dev)
        z = lambda *sh: torch.zeros(*sh, dtype=torch.int64, device=dev)
        self.d_pos, self.d_cls, self.d_lab = z(bins, 128), z(batch), z(batch)
        self.d_seg = torch.zeros(bins, 128, dtype=torch.int32, device=dev)
        self.opt = optimizer
        optimizer._armed = True
        _arm_pipelining(optimizer, self.grad_accumulation)

    def _unstage(self):
        n, st = self.bins * 128, self.d_stage
        self.d_ids.copy_(st[0:n].view(self.bins, 128))
        self.d_tt.copy_(st[n:2 * n].view(self.bins, 128))
        self.d_pos.copy_(st[2 * n:3 * n].view(self.bins, 128))
        self.d_seg.copy_(st[3 * n:4 * n].view(self.bins, 128))          # int64 -> int32
        self.d_cls.copy_(st[4 * n:4 * n + self.batch])
        self.d_lab.copy_(st[4 * n + self.batch:4 * n + 2 * self.batch])

    def stage(self, packed, label):
        n, hs = self.bins * 128, self.h_stage
        if packed["bins"] != self.bins or label.numel() != self.batch:
            raise ValueError("PackedTrainStep was built for %d bins / %d sequences" % (self.bins, self.batch))
        if self._h2d_done is not None:
            self._h2d_done.synchronize()
        hs[0:n].copy_(packed["input_ids"].reshape(-1))
        hs[n:2 * n].copy_(packed["token_type_ids"].reshape(-1))
        hs[2 * n:3 * n].copy_(packed["position_ids"].reshape(-1))
        hs[3 * n:4 * n].copy_(packed["segments"].reshape(-1))
        hs[4 * n:4 * n + self.batch].copy_(packed["cls_index"])
        hs[4 * n + self.batch:4 * n + 2 * self.batch].copy_(label.reshape(-1))
        self.d_stage.copy_(hs, non_blocking=True)
        self._h2d_done = torch.cuda.Event()
        self._h2d_done.record(torch.cuda.current_stream(self.eng.dev))

    def _body(self):
        self._unstage()
        packed = (self.d_pos, self.d_seg, self.d_cls)
        self._train_body(lambda ev: self.eng.forward(self.d_ids, self.d_tt, None, self.d_lab, training=True,
                                                     need_backward=True, packed=packed, weight_events=ev))

    def __call__(self, packed, label, final=True):
        self.stage(packed, label)
        self.run_device(final)
        return self.loss_out


class FusedEvalStep(_StagedGraphStep):
    """The reference's eval body (`on_step` + `criterion` under `no_grad`, [:204-208] / [:228-229]) as one CUDA-graph
    replay: H2D of the batch, the dropout-free forward, mean CE.  Returns device tensors that are overwritten by the
    next call (the callers below consume them before staging the next batch)."""

    def __init__(self, model, batch_size, seq_len, use_graph=True):
        super().__init__(model, batch_size, seq_len, use_graph)
        self.logits_out = torch.zeros(batch_size, self.model.num_labels, dtype=torch.float32, device=self.eng.dev)

    def _body(self):
        self._unstage()
        logits, loss = self.eng.forward(self.d_ids, self.d_tt, self.d_mask, self.d_lab, training=False,
                                        need_backward=False)
        self.logits_out.copy_(logits)
        self.loss_out.copy_(loss)

    def __call__(self, batch_data):
        if self.model._optimizer is not None:
            self.model._optimizer.flush_pending()     # a pipelined train step may still owe its update
        self.stage(batch_data)
        self.run_device()
        return self.logits_out, self.d_lab, self.loss_out


class Trainer:
    def __init__(self, args, config, model, criterion, optimizer):
        self.args = args
        self.config = config          # (the reference's `self.config = config,` stores a 1-tuple by accident, :121)
        self.model = model
        self.criterion = criterion
        self.optimizer = optimizer
        self._fused = None
        self._packed = {}     # bins -> PackedTrainStep
        self._scaler = None
        self._fused_eval = {}
        self._pin = {}

    def _to_device(self, batch_data):
        dev = _unwrap(self.model)._engine.dev
        out = {}
        for k in ("label", "input_ids", "token_type_ids", "attention_mask"):
            t = batch_data[k]
            if t.is_cuda:
                out[k] = t
                continue
            key = (k, tuple(t.shape))
            if key not in self._pin:
                self._pin[key] = [torch.empty(t.shape, dtype=t.dtype).pin_memory(), None]
            buf, ev = self._pin[key]
            if ev is not None:
                ev.synchronize()          # the previous async copy out of this staging buffer has drained
            buf.copy_(t)
            out[k] = buf.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            self._pin[key][1] = ev
        return out

    def on_step(self, batch_data):
        d = self._to_device(batch_data)
        label = d["label"]
        output = self.model(input_ids=d["input_ids"], token_type_ids=d["token_type_ids"],
                            attention_mask=d["attention_mask"], labels=label)
        logits = output[1]
        return logits, label

    def eval_step(self, batch_data):
        """`on_step` for the no-grad loops: the graph-captured forward when ``args.fused`` (one replay per batch instead
        of ~100 eager launches), else the eager call.  Returns (logits, label) like `on_step`."""
        if not getattr(self.args, "fused", True) or batch_data["input_ids"].is_cuda:
            return self.on_step(batch_data)
        B, S = batch_data["input_ids"].shape
        key = (id(_unwrap(self.model)), B, S)     # `test` may swap the model [:222-224]
        if key not in self._fused_eval:
            self._fused_eval[key] = FusedEvalStep(self.model, B, S)
        logits, label, _loss = self._fused_eval[key](batch_data)
        return logits, label

    def loss_reduce(self, loss):
        if isinstance(self.model, DistributedDataParallel):
            return self.model.loss_reduce(loss)
        return loss.clone()

    def output_reduce(self, outputs, targets):
        if isinstance(self.model, DistributedDataParallel):
            return self.model.all_gather_rows(outputs), self.model.all_gather_rows(targets)
        return outputs.clone(), targets.clone()

    def grad_accumulation(self):
        """micro-batches per optimizer step: args.grad_accumulation under args.use_grad_accumulation, else 1"""
        if not getattr(self.args, "use_grad_accumulation", False):
            return 1
        k = int(getattr(self.args, "grad_accumulation", 1))
        if k < 1:
            raise ValueError("grad_accumulation must be >= 1 (got %d)" % k)
        return k

    def train_step(self, batch_data, step_optimizer=True):
        """One step of the reference loop body [:166-176]; returns the rank-averaged loss (device scalar).
        step_optimizer=False: a non-final micro-batch of an accumulation window (fabric/fabric-cls.py:150-161): its
        loss / k gradient is added to the model's accumulator, with no exchange and no update.  The returned loss is
        the micro-batch's own, not divided by k."""
        k = self.grad_accumulation()
        final = bool(step_optimizer)
        if getattr(self.args, "fused", True) and getattr(self.args, "pack", False) and \
                batch_data["input_ids"].shape[1] == 128 and not batch_data["input_ids"].is_cuda:
            from .packing import pack_batch
            packed = pack_batch(batch_data["input_ids"], batch_data["token_type_ids"], batch_data["attention_mask"])
            key = (packed["bins"], batch_data["input_ids"].shape[0])
            if key in self._packed and self._packed[key].grad_accumulation != k:
                del self._packed[key]
            if key not in self._packed:
                if len(self._packed) >= 16:           # bound the graph cache: drop the oldest entry
                    self._packed.pop(next(iter(self._packed)))
                self._packed[key] = PackedTrainStep(self.model, self.optimizer, key[0], key[1], grad_accumulation=k)
            self.model.train()
            loss = self._packed[key](packed, batch_data["label"], final)
        elif getattr(self.args, "fused", True):
            B, S = batch_data["input_ids"].shape
            if self._fused is None or (self._fused.B, self._fused.S, self._fused.grad_accumulation) != (B, S, k):
                self._fused = FusedTrainStep(self.model, self.optimizer, B, S, grad_accumulation=k)
            self.model.train()
            loss = self._fused(batch_data, final)
        elif getattr(self.args, "use_amp", False):
            # the -amp scripts' loop body (multi-gpu-distributed-mp-amp-cls.py:166-171), scaler created once
            if self._scaler is None:
                self._scaler = torch.amp.GradScaler("cuda")
            self.model.train()
            with torch.autocast("cuda"), self._window(final):
                logits, label = self.on_step(batch_data)
                loss = self.criterion(logits, label)
            self._scaler.scale(loss / k if k > 1 else loss).backward()
            if final:
                self._scaler.step(self.optimizer)
                self._scaler.update()
        elif k > 1 or not final:
            # fabric-cls.py:150-161: loss / k, step and zero_grad once per window
            self.model.train()
            with self._window(final):
                logits, label = self.on_step(batch_data)
                loss = self.criterion(logits, label)
            (loss / k).backward()
            if final:
                self.optimizer.step()
                self.optimizer.zero_grad()
        else:
            self.model.train()
            logits, label = self.on_step(batch_data)
            loss = self.criterion(logits, label)
            self.optimizer.zero_grad()
            loss.backward()
            self.optimizer.step()
        return self.loss_reduce(loss.detach())

    def _window(self, final):
        """the forward of a non-final micro-batch runs under no_sync()"""
        return contextlib.nullcontext() if final else self.model.no_sync()

    def train(self, train_loader, dev_loader=None, train_sampler=None):
        gloabl_step = 1
        best_acc = 0.
        if self.args.local_rank == 0:
            start = time.time()
        for epoch in range(1, self.args.epochs + 1):
            if train_sampler is not None:
                train_sampler.set_epoch(epoch)
            for step, batch_data in enumerate(train_loader):
                if getattr(self.args, "use_grad_accumulation", False):
                    # per-epoch index, as fabric-cls.py:157: a window left open at the end of an epoch is completed
                    # by the first micro-batches of the next one
                    loss = self.train_step(batch_data, step_optimizer=(step + 1) % self.grad_accumulation() == 0)
                else:
                    loss = self.train_step(batch_data)
                if self.args.local_rank == 0 and gloabl_step % max(1, getattr(self.args, "log_every", 1)) == 0:
                    print("【train】 epoch：{}/{} step：{}/{} loss：{:.6f}".format(
                        epoch, self.args.epochs, gloabl_step, self.args.total_step, float(loss)
                    ))
                gloabl_step += 1
                if self.args.dev:
                    if gloabl_step % self.args.eval_step == 0:
                        loss, accuracy = self.dev(dev_loader)
                        improved = accuracy > best_acc   # identical on every rank (gathered outputs)
                        if self.args.local_rank == 0:
                            print("【dev】 loss：{:.6f} accuracy：{:.4f}".format(float(loss), accuracy))
                        if improved:
                            best_acc = accuracy
                            if self.args.local_rank == 0:
                                print("【best accuracy】 {:.4f}".format(best_acc))
                                # rank 0 alone, as in the reference [:190-192]: under DDP state_dict() pulls the fp32
                                # slices other ranks own out of their HBM one-sidedly (ddp.py::_gather_master)
                                torch.save(self.model.state_dict(), self.args.ckpt_path)
        if self.args.local_rank == 0:
            end = time.time()
            print("耗时：{}分钟".format((end - start) / 60))
        if not self.args.dev:
            if self.args.local_rank == 0:
                torch.save(self.model.state_dict(), self.args.ckpt_path)

    def dev(self, dev_loader):
        self.model.eval()
        correct_total = 0
        num_total = 0
        loss_total = 0.
        with torch.no_grad():
            for step, batch_data in enumerate(dev_loader):
                logits, label = self.eval_step(batch_data)
                loss = self.criterion(logits, label)
                loss = self.loss_reduce(loss)
                loss_total += loss
                logits, label = self.output_reduce(logits, label)
                logits = logits.detach().cpu().numpy()
                label = label.view(-1).detach().cpu().numpy()
                num_total += len(label)
                preds = np.argmax(logits, axis=1).flatten()
                correct_num = (preds == label).sum()
                correct_total += correct_num
        return loss_total, correct_total / num_total

    def test(self, model, test_loader, labels):
        self.model = model
        self.model.eval()
        preds = []
        trues = []
        with torch.no_grad():
            for step, batch_data in enumerate(test_loader):
                logits, label = self.eval_step(batch_data)
                logits, label = self.output_reduce(logits, label)
                label = label.view(-1).detach().cpu().numpy().tolist()
                logits = logits.detach().cpu().numpy()
                pred = np.argmax(logits, axis=1).flatten().tolist()
                trues.extend(label)
                preds.extend(pred)
        from sklearn.metrics import classification_report
        report = classification_report(trues, preds, target_names=labels)
        return report
