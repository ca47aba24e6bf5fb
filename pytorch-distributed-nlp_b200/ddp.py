"""``DistributedDataParallel``-compatible wrapper whose gradient exchange is a peer-HBM kernel, not NCCL.

Reference surface: ``torch.nn.parallel.DistributedDataParallel(model, device_ids=[rank])``
(multi-gpu-distributed-cls.py:341): module pass-through, ``module.``-prefixed ``state_dict`` keys
(:192, :362, test.py:96-101), rank-0 parameter broadcast at wrap time (SP/torch/nn/parallel/distributed.py:879-889),
gradient mean over ranks during ``loss.backward()`` (Reducer, distributed.py:1255-1280).

Design (SURVEY.md §8e): every rank owns a contiguous 1/world slice of every bucket (embeddings | layer i | head).
Gradients (bf16), shadow weights (bf16) and the fp32 master weights live in cudaMalloc'ed buffers that every peer maps
through CUDA IPC; the exchange is ``b2_bucket_reduce_adamw``: read my slice from all peers over NVSwitch, mean in fp32,
HF-AdamW on my fp32 master slice, store the new bf16 weights into every peer.  torch.distributed is used only for the
one-time handle exchange and the initial broadcast.  ``state_dict()`` is ONE-SIDED: the calling rank pulls the fp32
slices it does not own out of their owners' HBM with copy-engine peer copies, so the reference's
``if local_rank == 0: torch.save(model.state_dict())`` (:190-197) works without the other ranks taking part.
"""
import os

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib as L


class _DevBuf:
    """cudaMalloc'ed, IPC-exportable buffer exposed to torch through __cuda_array_interface__ (zero copy)."""

    def __init__(self, nbytes):
        import ctypes
        p = ctypes.c_void_p()
        L.call("b2_comm_alloc", nbytes, ctypes.byref(p))
        self.ptr, self.nbytes = p.value, nbytes

    def handle(self):
        import ctypes
        buf = ctypes.create_string_buffer(L.IPC_HANDLE_BYTES)
        L.call("b2_comm_export", self.ptr, buf)
        return bytes(buf.raw)

    def tensor(self, dtype, device):
        class _Iface:
            pass
        o = _Iface()
        o.__cuda_array_interface__ = {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False),
                                      "version": 2, "strides": None}
        t = torch.as_tensor(o, device=device)
        t._b2_keepalive = self
        return t.view(dtype)

    def free(self):
        if self.ptr:
            L.call("b2_comm_free", self.ptr)
            self.ptr = 0


def _import_handle(handle_bytes):
    import ctypes
    p = ctypes.c_void_p()
    L.call("b2_comm_import", handle_bytes, ctypes.byref(p))
    return p.value


# Local IPC buffers of wrappers that were dropped without close(): a peer may still be reading them (rank 0 pulling
# master slices for a checkpoint while this rank already moved on), so they are only freed at the next collective
# point every rank is known to have reached -- the barrier at the end of the next wrapper's constructor, or close().
_graveyard = []


def _drain_graveyard():
    while _graveyard:
        _graveyard.pop().free()


class PeerComm:
    """Symmetric buffers of one process group: one entry per name, local pointer + every peer's mapped pointer."""

    def __init__(self, device, group=None):
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.device = device
        self.local = {}
        self.peers = {}
        self.epochs = torch.zeros(L.FLAG_SLOTS, dtype=torch.int32, device=device)
        self.alloc("flags", L.FLAG_SLOTS * self.world * 4)
        self.alloc("scalar", 2 * self.world * 4)
        self.alloc("scalar_inf", 2 * self.world * 4)

    def alloc(self, name, nbytes):
        """Collective: every rank allocates `nbytes` under `name` and maps every peer's copy."""
        if name in self.local:
            self.release(name)
        buf = _DevBuf(nbytes)
        handles = [None] * self.world
        dist.all_gather_object(handles, buf.handle(), group=self.group)
        ptrs = []
        for r, h in enumerate(handles):
            ptrs.append(buf.ptr if r == self.rank else _import_handle(h))
        self.local[name] = buf
        self.peers[name] = ptrs
        return buf

    def release(self, name):
        """Unmaps the peers' copies of `name` (always safe: the mapping is mine) and parks the local buffer."""
        for r, p in enumerate(self.peers.pop(name, [])):
            if r != self.rank and p:
                L.call("b2_comm_unimport", p)
        buf = self.local.pop(name, None)
        if buf is not None:
            _graveyard.append(buf)

    def release_all(self):
        torch.cuda.synchronize(self.device)      # no kernel / copy of mine may still touch a mapping I am closing
        for name in list(self.local):
            self.release(name)

    def epoch_ptr(self, slot):
        return self.epochs.data_ptr() + 4 * slot

    def barrier(self, slot, stream):
        L.call("b2_peer_barrier", L.ptr_array(self.peers["flags"]), self.world, self.rank, slot,
               self.epoch_ptr(slot), stream)


# flag slots
_SLOT_GRADS_READY, _SLOT_UPDATE_DONE, _SLOT_LOSS, _SLOT_GATHER, _SLOT_INF, _SLOT_BUCKET0 = 0, 1, 2, 3, 4, 8
_GATHER_SLOT_BYTES = 64 << 10     # per-rank capacity of the two eval-gather buffers (grown on demand)


class DistributedDataParallel(nn.Module):
    def __init__(self, module, device_ids=None, output_device=None, process_group=None, overlap=True, **unused):
        super().__init__()
        if not hasattr(module, "_engine"):
            raise TypeError("this DistributedDataParallel wraps the b200 BertForSequenceClassification")
        if module._engine is None:
            raise RuntimeError("call model.cuda() before wrapping (as the reference does, :340-341)")
        self.module = module
        self.group = process_group
        if dist.is_available() and dist.is_initialized():
            self.world, self.rank = dist.get_world_size(process_group), dist.get_rank(process_group)
        else:
            self.world, self.rank = 1, 0
        self.overlap = overlap
        self.dma = False
        self.comm = None
        self._master_stale = False
        self._side = None
        self._pending = None
        self._closed = False
        self._gather_calls = 0
        self._gather_cap = 0
        # plain attribute, NOT a registered submodule (model -> wrapper -> model would be a module cycle)
        object.__setattr__(module, "_ddp", self)
        eng = module._engine
        if self.world > 1:
            import gc
            gc.collect()     # a dropped previous wrapper (module <-> wrapper cycle) parks its buffers now, see __del__
            if self.world > 8:
                raise ValueError("peer-HBM exchange covers one NVSwitch domain (world <= 8)")
            # DDP init sync: parameters of rank 0 win
            dist.broadcast(module._flat, src=0, group=process_group)
            self.comm = PeerComm(eng.dev, process_group)
            n = module._layout.total
            shadow = self.comm.alloc("shadow", 2 * n).tensor(torch.bfloat16, eng.dev)
            grads = self.comm.alloc("grads", 2 * n).tensor(torch.bfloat16, eng.dev)
            eng.rebind(shadow, grads)
            # fp32 masters move into a peer-visible buffer too: state_dict() pulls foreign slices one-sidedly
            module._rebind_flat(self.comm.alloc("master", 4 * n).tensor(torch.float32, eng.dev))
            eng.refresh_shadow()
            self._slices = self._make_slices()
            # staging for the DMA form of the exchange: my slice of every bucket as held by each peer
            # transport form of the exchange: the fused peer-HBM kernel (default) or copy-engine DMA + local reduce.
            # Round 1 measured the DMA form ahead (60.0 k vs 58.7 k samples/s on 8 B200); with the step body on a
            # high-priority stream the exchange kernels no longer hold SMs the GEMM chain is waiting for, and the
            # kernel form wins clearly: 66.0 k vs 54.6 k samples/s on 8 B200 (config A), 14.4 k vs 11.9 k (config C)
            self.dma = os.environ.get("B2_DDP_DMA", "0") == "1"
            self._stage_off, off = [], 0
            for (sb, se) in self._slices:
                row = {}
                for r in range(self.world):
                    if r != self.rank:
                        row[r] = off
                        off += (2 * (se - sb) + 255) // 256 * 256
                self._stage_off.append(row)
            self._stage = torch.empty(max(off, 256), dtype=torch.uint8, device=eng.dev)
            self._side = torch.cuda.Stream(device=eng.dev)
            self._grow_gather(_GATHER_SLOT_BYTES)
            torch.cuda.synchronize(eng.dev)
            dist.barrier(group=process_group)
            # every rank is past its previous wrapper (if any): buffers parked by dropped wrappers can go
            _drain_graveyard()

    @staticmethod
    def _bucket_slice(b, e, r, world):
        """rank r's 8-aligned 1/world slice of the bucket [b, e)"""
        per = ((e - b) // 8 + world - 1) // world * 8
        sb = min(e, b + r * per)
        return sb, min(e, sb + per)

    def _make_slices(self):
        return [DistributedDataParallel._bucket_slice(b, e, self.rank, self.world)
                for (b, e, _label) in self.module._layout.buckets]

    def forward(self, *args, **kwargs):
        return self.module(*args, **kwargs)

    def no_sync(self):
        """torch DDP's ``no_sync()``: backwards of forwards run inside the context add to the local fp32 accumulator,
        with no exchange; the first backward outside it exchanges the window's sum.  ``optimizer.step()`` after only
        no_sync() backwards raises (the ranks' gradients were never exchanged)."""
        return self.module.no_sync()

    # ---- checkpoint surface ---------------------------------------------------------------------------------------------
    def load_state_dict(self, state_dict, strict=True, assign=False):
        """`model.load_state_dict(torch.load(ckpt))` on the WRAPPED model (multi-gpu-distributed-cls.py:357-363): keys
        carry the `module.` prefix.  Delegates to the model's own loader so the bf16 shadow weights the kernels read are
        refreshed (nn.Module's per-leaf loader would update only the fp32 masters)."""
        sd = {}
        for k, v in state_dict.items():
            if strict and not k.startswith("module."):
                raise RuntimeError("Error(s) in loading state_dict for DistributedDataParallel: unexpected key %r "
                                   "(keys of a wrapped model start with 'module.')" % k)
            sd[k[len("module."):] if k.startswith("module.") else k] = v
        res = self.module.load_state_dict(sd, strict=strict)
        self._master_stale = False      # every rank loaded the full tensors: all slices are current everywhere
        return torch.nn.modules.module._IncompatibleKeys(["module." + k for k in res.missing_keys],
                                                         ["module." + k for k in res.unexpected_keys])

    # ---- teardown -------------------------------------------------------------------------------------------------------
    def close(self):
        """Collective teardown: unmaps the peers' buffers and frees the local ones after a barrier.  A wrapper that is
        simply dropped (the reference re-wraps for its test phase, :357-360) unmaps the peers and parks its buffers
        until the next wrap's barrier instead."""
        if self._closed:
            return
        self._closed = True
        if self.comm is not None:
            eng = self.module._engine
            torch.cuda.synchronize(eng.dev)
            dist.barrier(group=self.group)
            self._detach_module()            # pulls foreign master slices out of the peers' buffers ...
            torch.cuda.synchronize(eng.dev)
            dist.barrier(group=self.group)   # ... so nobody frees before everybody has pulled
            self.comm.release_all()
            _drain_graveyard()
            self.comm = None

    def _detach_module(self):
        """give the model private (non-IPC) copies of its buffers so it stays usable after the wrapper is gone"""
        module = self.module
        eng = module._engine
        if eng is not None and self.comm is not None and "shadow" in self.comm.local:
            self._gather_master()
            module._rebind_flat(torch.empty_like(module._flat))
            eng.rebind(torch.empty_like(eng.shadow), torch.empty_like(eng.grads))
            torch.cuda.synchronize(eng.dev)
        if getattr(module, "_ddp", None) is self:
            object.__setattr__(module, "_ddp", None)

    def __del__(self):
        try:
            if not self._closed and self.comm is not None:
                self._closed = True
                self.comm.release_all()      # peers unmapped now, local buffers parked until the next collective point
        except Exception:
            pass

    # ---- hooks called by the engine during backward (autograd thread) -----------------------------------------------
    def _bucket_ready(self, idx, wg_event=None, fold=None):
        """Bucket `idx` holds this rank's final local gradients once the main stream reaches this point and `wg_event`
        (the weight-gradient stream's marker for the layer) has fired.  With an optimizer attached and overlap on,
        start its exchange + update on the side stream right away so it hides behind the rest of backward.  Only the
        SIDE stream waits for the weight gradients: the main stream's dgrad chain never parks behind them.
        fold: gradient accumulation (engine.fold).  A no_sync() micro-batch is only added to the local accumulator: no
        barrier, no exchange.  The last one folds the window's sum into the bf16 gradients BEFORE the bucket's barrier,
        after which the peers read my slice."""
        opt = self.module._optimizer
        armed = self.world > 1 and self.overlap and opt is not None and getattr(opt, "_armed", False)
        if fold is None and not armed:
            return
        eng = self.module._engine
        main = torch.cuda.current_stream(eng.dev)
        ev = torch.cuda.Event()
        ev.record(main)
        self._side.wait_event(ev)
        if wg_event is not None:
            self._side.wait_event(wg_event)
        s = self._side.cuda_stream
        if fold is not None:
            b0, e0, _lbl = self.module._layout.buckets[idx]
            eng.fold_range(b0, e0, fold[0], fold[1], s)
            if fold[0] == L.ACCUM_ADD or not armed:
                return
        self.comm.barrier(_SLOT_BUCKET0 + idx, s)
        self._exchange_update(opt, idx, s)
        if self._pending is None:
            self._pending = set()
        self._pending.add(idx)

    def _exchange_update(self, opt, idx, s):
        """Mean over ranks + HF-AdamW on my slice of bucket `idx` + delivery of the new bf16 weights to every rank.
        Kernel form (default): the reduce kernel loads the peers' slices / stores the peers' shadows itself through the
        mapped pointers -- one launch per bucket does the one-shot peer-HBM reduction, the fp32 cast, the partitioned
        AdamW and the delivery of the new weights.  DMA form (B2_DDP_DMA=1, every bucket but the last one produced):
        the transfers are copy-engine copies over NVLink and the reduce kernel works on local memory only."""
        sb, se = self._slices[idx]
        if se <= sb:
            return
        peers_g, peers_s = self.comm.peers["grads"], self.comm.peers["shadow"]
        if not self.dma or idx == 0:
            opt.update_range(sb, se, self.world, self.rank, peers_g, peers_s, s)
            return
        nbytes = 2 * (se - sb)
        g_ptrs, s_ptrs = [], []
        for r in range(self.world):
            if r == self.rank:
                g_ptrs.append(peers_g[r])
                s_ptrs.append(peers_s[r])
                continue
            st = self._stage.data_ptr() + self._stage_off[idx][r]
            L.call("b2_copy_async", st, peers_g[r] + 2 * sb, nbytes, s)
            g_ptrs.append(st - 2 * sb)        # the kernel indexes base + absolute element index
            s_ptrs.append(None)
        opt.update_range(sb, se, self.world, self.rank, g_ptrs, s_ptrs, s)
        mine = peers_s[self.rank] + 2 * sb
        for r in range(self.world):
            if r != self.rank:
                L.call("b2_copy_async", peers_s[r] + 2 * sb, mine, nbytes, s)

    def _on_backward_done(self):
        pass

    def consensus_probe(self, probe, window=None):
        """GradScaler inf check under DDP (multi-gpu-distributed-mp-amp-cls.py:166-171): stock DDP all-reduces the
        gradients before the scaler looks at them, so a non-finite value on ONE rank makes EVERY rank skip the step and
        back off its scale.  Here the scaler only sees the 6-float probe on classifier.bias: poison it on every rank
        when any rank's probe is non-finite (one scalar exchange through peer memory, no host sync).  window: the
        probe's value summed over the accumulation window (no_sync), checked as well."""
        if self.world == 1:
            return probe
        eng = self.module._engine
        bad = (~torch.isfinite(probe)).any()
        if window is not None:
            bad = bad | (~torch.isfinite(window)).any()
        bad = bad.to(torch.float32).reshape(1)
        dst = torch.empty(1, dtype=torch.float32, device=eng.dev)
        L.call("b2_scalar_allreduce_mean", bad.data_ptr(), dst.data_ptr(), L.ptr_array(self.comm.peers["scalar_inf"]),
               L.ptr_array(self.comm.peers["flags"]), self.world, self.rank, _SLOT_INF,
               self.comm.epoch_ptr(_SLOT_INF), eng.stream())
        return torch.where(dst > 0, torch.full_like(probe, float("inf")), probe)

    def _optimizer_step(self, opt):
        """world > 1 body of ``optimizer.step()``."""
        eng = self.module._engine
        main = torch.cuda.current_stream(eng.dev)
        nb = len(self.module._layout.buckets)
        done = self._pending or set()
        if len(done) == nb:
            # everything was launched from the backward hooks: just join
            s = self._side.cuda_stream
            self.comm.barrier(_SLOT_UPDATE_DONE, s)
            opt.advance(s)
            ev = torch.cuda.Event()
            ev.record(self._side)
            main.wait_event(ev)
        else:
            if done:
                ev = torch.cuda.Event()
                ev.record(self._side)
                main.wait_event(ev)
            s = main.cuda_stream
            self.comm.barrier(_SLOT_GRADS_READY, s)
            for idx in range(nb):
                if idx in done:
                    continue
                self._exchange_update(opt, idx, s)
            self.comm.barrier(_SLOT_UPDATE_DONE, s)
            opt.advance(s)
        self._pending = None
        self._master_stale = True

    def _gather_master(self):
        """fp32 masters are updated slice-wise by their owner ranks.  Re-assemble them on THIS rank by pulling every
        foreign slice out of its owner's (IPC-mapped) master buffer -- one-sided, stream-ordered copy-engine copies.
        Safe without the owners' cooperation: every step ends with a device barrier after all updates
        (_SLOT_UPDATE_DONE), and an owner cannot start the NEXT update before this rank joins that step's bucket
        barriers -- so between steps the peers' masters are quiescent."""
        if self.world == 1 or not self._master_stale or self.comm is None:
            return
        eng = self.module._engine
        s = eng.stream()
        flat = self.module._flat
        peers_m = self.comm.peers["master"]
        for (b, e, _label) in self.module._layout.buckets:
            for r in range(self.world):
                if r == self.rank:
                    continue
                sb, se = self._bucket_slice(b, e, r, self.world)
                if se > sb:
                    L.call("b2_copy_async", flat.data_ptr() + 4 * sb, peers_m[r] + 4 * sb, 4 * (se - sb), s)
        self._master_stale = False

    # ---- the two small collectives of the reference Trainer -------------------------------------------------------------
    def loss_reduce(self, loss):
        """mean over ranks of a scalar loss (Trainer.loss_reduce, :139-143)."""
        if self.world == 1:
            return loss.clone()
        eng = self.module._engine
        src = loss.detach().to(torch.float32).reshape(1).contiguous()
        dst = torch.empty(1, dtype=torch.float32, device=eng.dev)
        L.call("b2_scalar_allreduce_mean", src.data_ptr(), dst.data_ptr(), L.ptr_array(self.comm.peers["scalar"]),
               L.ptr_array(self.comm.peers["flags"]), self.world, self.rank, _SLOT_LOSS,
               self.comm.epoch_ptr(_SLOT_LOSS), eng.stream())
        return dst.reshape(())

    def _grow_gather(self, per_rank_bytes):
        """(re)allocates the two eval-gather buffers -- collective, like the call that needs them"""
        cap = _GATHER_SLOT_BYTES
        while cap < per_rank_bytes:
            cap *= 2
        self.comm.alloc("gather0", cap * self.world)
        self.comm.alloc("gather1", cap * self.world)
        self._gather_cap = cap

    def all_gather_rows(self, t):
        """rank-ordered concatenation along dim 0 (Trainer.output_reduce, :145-155)."""
        if self.world == 1:
            return t.clone()
        eng = self.module._engine
        t = t.contiguous()
        nbytes = t.numel() * t.element_size()
        if nbytes % 4 != 0:
            raise ValueError("all_gather_rows: payload must be a multiple of 4 bytes")
        if nbytes > self._gather_cap:
            torch.cuda.synchronize(eng.dev)
            self._grow_gather(nbytes)
        # two buffers alternated per call (whatever the payload): a fast rank's next store can never land in a buffer
        # a slow rank is still reading (to reach call n+2 it must pass barrier n+1, which the slow rank only joins
        # after its read of call n was enqueued ahead of it on the same stream)
        self._gather_calls += 1
        key = "gather%d" % (self._gather_calls & 1)
        L.call("b2_allgather_rows", t.data_ptr(), nbytes, L.ptr_array(self.comm.peers[key]),
               L.ptr_array(self.comm.peers["flags"]), self.world, self.rank, _SLOT_GATHER,
               self.comm.epoch_ptr(_SLOT_GATHER), eng.stream())
        full = self.comm.local[key].tensor(torch.uint8, eng.dev)[:nbytes * self.world].view(t.dtype)
        return full.view((self.world * t.shape[0],) + tuple(t.shape[1:])).clone()
