"""Gradient accumulation: ``no_sync()`` micro-batches summed in fp32, one exchange and one update per window.

CPU: the accumulation oracle (tests/grad_accum_ref.py) against real torch, the Trainer's window logic, the export.
GPU: the b2_grad_accumulate kernel, gradient parity of accumulated windows, trajectories through the eager loop and the
captured Trainer steps, the surface rules (zero_grad, step, errors, GradScaler), and the world-2 DDP path."""
import contextlib
import os
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from grad_accum_ref import train_accum, window_grads
from parity import (TOL_GRAD_REL, TOL_LOSS, TOL_TRAJ, b2, bert_ref, full_config, grad_report, make_model,
                    oracle_masks, state_from_hf_init, tiny_config, to_dev)
from oracle import cpu_step, ddp_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _split(batch, k):
    n = batch["input_ids"].shape[0] // k
    return [{key: v[j * n:(j + 1) * n] for key, v in batch.items()} for j in range(k)]


class _Args:
    weight_decay, learning_rate = 0.01, 3e-5


# ---- CPU: the oracle against real torch ---------------------------------------------------------------------------------
def test_window_grads_equal_hf_accumulated_grad():
    """k calls of (loss / k).backward() on HF BertForSequenceClassification leave the oracle's sum in .grad"""
    cfg = tiny_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, num_hidden_layers=1)
    hf = cpu_step.build_hf_model(cfg, seed=123)
    state = {k: v.detach().clone() for k, v in hf.named_parameters()}
    micro = [bert_ref.synthetic_batch(cfg, 2, 128, 300 + j, padded=(j % 2 == 1)) for j in range(3)]
    for b in micro:
        out = hf(input_ids=b["input_ids"], token_type_ids=b["token_type_ids"], attention_mask=b["attention_mask"])
        (F.cross_entropy(out.logits, b["label"]) / len(micro)).backward()
    _, acc = window_grads(state, cfg, micro)
    for k, p in hf.named_parameters():
        assert float((acc[k] - p.grad).abs().max()) < 2e-6 + 1e-5 * float(p.grad.abs().max()), k


def _gloo_no_sync_worker(rank, world, port, out_path):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    cfg = tiny_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, num_hidden_layers=1)
    hf = cpu_step.build_hf_model(cfg, seed=123 + rank)
    ddp = torch.nn.parallel.DistributedDataParallel(hf)
    k = 3
    for j in range(k):
        b = bert_ref.synthetic_batch(cfg, 2, 128, 60 + 10 * rank + j)
        ctx = ddp.no_sync() if j < k - 1 else contextlib.nullcontext()
        with ctx:
            out = ddp(input_ids=b["input_ids"], token_type_ids=b["token_type_ids"],
                      attention_mask=b["attention_mask"])
            (F.cross_entropy(out.logits, b["label"]) / k).backward()
    if rank == 0:
        torch.save({n: v.grad.clone() for n, v in hf.named_parameters()}, out_path)
    dist.barrier()
    dist.destroy_process_group()


def test_window_mean_matches_torch_ddp_no_sync_on_gloo_world2(tmp_path):
    """rank mean of the per-rank window sums == what torch DDP with no_sync() leaves in .grad (gloo, world 2)"""
    ctx = mp.get_context("spawn")
    out_path = str(tmp_path / "ddp_no_sync_grads.pt")
    procs = [ctx.Process(target=_gloo_no_sync_worker, args=(r, 2, 29637, out_path)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=240)
        assert p.exitcode == 0
    got = torch.load(out_path)
    cfg = tiny_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0, num_hidden_layers=1)
    hf = cpu_step.build_hf_model(cfg, seed=123)
    state = {k: v.detach().clone() for k, v in hf.named_parameters()}
    sums = [window_grads(state, cfg, [bert_ref.synthetic_batch(cfg, 2, 128, 60 + 10 * r + j) for j in range(3)])[1]
            for r in range(2)]
    avg = ddp_ref.mean_grads(sums)
    for k in avg:
        assert float((avg[k] - got[k]).abs().max()) < 2e-6 + 1e-5 * float(got[k].abs().max()), k


# ---- CPU: Trainer window logic ------------------------------------------------------------------------------------------
class _StubTrainer(b2.Trainer):
    def __init__(self, args):
        super().__init__(args, None, None, None, None)
        self.calls = []

    def train_step(self, batch_data, *args, **kwargs):
        self.calls.append((batch_data, args, kwargs))
        return torch.zeros(())


def _stub_args(**kw):
    class A(b2.Args):
        epochs, dev, local_rank = 2, False, None
    for k, v in kw.items():
        setattr(A, k, v)
    return A


def test_trainer_steps_every_k_batches_with_carry_over():
    t = _StubTrainer(_stub_args(use_grad_accumulation=True, grad_accumulation=3))
    t.train(list(range(7)))
    got = [(b, kw["step_optimizer"]) for b, _a, kw in t.calls]
    # per-epoch index as fabric-cls.py:157: batch 6 of epoch 1 is carried into epoch 2's first window
    want = [(i, i in (2, 5)) for i in range(7)] * 2
    assert got == want


def test_trainer_without_the_flag_calls_train_step_as_before():
    t = _StubTrainer(_stub_args())
    assert b2.Args.use_grad_accumulation is False and b2.Args.grad_accumulation == 4
    t.train(list(range(7)))
    assert t.calls == [(i, (), {}) for i in range(7)] * 2


def test_grad_accumulate_is_exported_and_registered():
    from pytorch_distributed_nlp_b200 import _lib as L
    assert L._SIGNATURES["b2_grad_accumulate"] == [L.vp, L.vp, L.i64, L.i64, L.f32, L.i32, L.vp]
    assert "b2_grad_accumulate" in L.EXPORTED_SYMBOLS
    with open(os.path.join(ROOT, "include", "b2_ddp_bert.h")) as f:
        assert "int32_t b2_grad_accumulate(" in f.read()
    assert hasattr(L.load(), "b2_grad_accumulate")


# ---- GPU: kernel ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 0.3])
def test_grad_accumulate_kernel_against_torch(cuda_dev, scale):
    from pytorch_distributed_nlp_b200 import _lib as L
    gen = torch.Generator(device=cuda_dev).manual_seed(7)
    n, begin, end = 3 * 4096 + 200, 136, 3 * 4096 + 104          # several blocks, a ragged last one
    g1 = torch.randn(n, device=cuda_dev, generator=gen).to(torch.bfloat16)
    g2 = torch.randn(n, device=cuda_dev, generator=gen).to(torch.bfloat16)
    acc = torch.randn(n, device=cuda_dev, generator=gen)
    acc0, g2_0 = acc.clone(), g2.clone()
    s = torch.cuda.current_stream().cuda_stream
    L.call("b2_grad_accumulate", acc.data_ptr(), g1.data_ptr(), begin, end, scale, L.ACCUM_ADD, s)
    want_acc = acc0.clone()
    want_acc[begin:end] += scale * g1[begin:end].float()
    # FMA contraction: one rounding instead of two, so the result may differ by one ulp of the operands
    ulp = (acc0.abs() + scale * g1.float().abs()) * 2.0 ** -23
    if scale == 1.0:
        assert torch.equal(acc, want_acc)
    else:
        assert bool(((acc - want_acc).abs() <= ulp).all())
    assert torch.equal(acc[:begin], acc0[:begin]) and torch.equal(acc[end:], acc0[end:])
    mid = acc.clone()
    L.call("b2_grad_accumulate", acc.data_ptr(), g2.data_ptr(), begin, end, scale, L.ACCUM_FINISH, s)
    torch.cuda.synchronize()
    want_f = mid[begin:end] + scale * g2_0[begin:end].float()
    got = g2[begin:end]
    if scale == 1.0:
        assert torch.equal(got, want_f.to(torch.bfloat16))
    else:
        # one fp32 ulp before the bf16 rounding: the result is one of the two neighbouring bf16 values
        tol = (mid[begin:end].abs() + scale * g2_0[begin:end].float().abs()) * 2.0 ** -23
        lo = (want_f - tol).to(torch.bfloat16)
        hi = (want_f + tol).to(torch.bfloat16)
        assert bool(((got.float() >= lo.float()) & (got.float() <= hi.float())).all())
    assert float(acc[begin:end].abs().max()) == 0.0
    assert torch.equal(acc[:begin], acc0[:begin]) and torch.equal(acc[end:], acc0[end:])
    assert torch.equal(g2[:begin], g2_0[:begin]) and torch.equal(g2[end:], g2_0[end:])


# ---- GPU: gradient parity of one window -----------------------------------------------------------------------------------
def _window_backward(model, micro, dev, k=None):
    """micro-batches under model.no_sync(), the last one outside; each loss divided by k"""
    k = k or len(micro)
    losses = []
    for j, b in enumerate(micro):
        d = to_dev(b, dev)
        ctx = model.no_sync() if j < len(micro) - 1 else contextlib.nullcontext()
        with ctx:
            out = model(input_ids=d["input_ids"], token_type_ids=d["token_type_ids"],
                        attention_mask=d["attention_mask"], labels=d["label"])
        loss = F.cross_entropy(out[1], d["label"])
        (loss / k).backward()
        losses.append(float(loss))
    torch.cuda.synchronize()
    return losses


@pytest.mark.gpu
@pytest.mark.parametrize("padded", [False, True])
def test_tiny_window_grads_match_oracle_batch(cuda_dev, padded):
    """4 micro-batches of 4 rows == the gradient of the 16-row batch (mean CE over equal micro-batches)"""
    cfg = tiny_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    state = state_from_hf_init(cfg)
    model = make_model(cfg, state, cuda_dev).train()
    b2.build_optimizer(model, _Args)
    batch = bert_ref.synthetic_batch(cfg, 16, 128, 1500, padded=padded)
    _window_backward(model, _split(batch, 4), cuda_dev)
    assert model._engine.accum_pending == 0 and float(model._engine.accum.abs().max()) == 0.0
    _rl, _rz, rg = bert_ref.loss_and_grads(state, cfg, batch)
    worst, rows = grad_report(model.grad_dict(), rg)
    assert worst <= TOL_GRAD_REL, sorted(rows, key=lambda r: -r[1])[:5]


@pytest.mark.gpu
def test_full_config_window_matches_golden(cuda_dev):
    """config A, the batch of test_full_config_step_matches_golden (seed 1000, B = 32) as 4 x 8 rows with loss / 4"""
    gold = torch.load(os.path.join(GOLD, "config_a_step0.pt"))
    cfg = full_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    state = state_from_hf_init(cfg)
    model = make_model(cfg, state, cuda_dev).train()
    b2.build_optimizer(model, _Args)
    batch = bert_ref.synthetic_batch(cfg, 32, 128, 1000, padded=True)
    assert torch.equal(batch["input_ids"], gold["input_ids"])
    losses = _window_backward(model, _split(batch, 4), cuda_dev)
    assert abs(sum(losses) / 4 - gold["loss"]) <= TOL_LOSS
    g = model.grad_dict()
    scale = max(gold["grad_norms"].values())
    for k, n in gold["grad_norms"].items():
        got = float(g[k].double().norm())
        assert abs(got - n) <= TOL_GRAD_REL * max(n, 1e-3 * scale), (k, got, n)
    for k, ref in gold["grad_samples"].items():
        got = g[k].flatten()[: ref.numel()].cpu()
        assert float((got - ref).norm()) <= 3 * TOL_GRAD_REL * max(float(ref.norm()), 1e-3 * scale), k


@pytest.mark.gpu
def test_dropout_window_replays_one_rng_step_per_micro_batch(cuda_dev):
    cfg = tiny_config()
    state = state_from_hf_init(cfg)
    model = make_model(cfg, state, cuda_dev).train()
    b2.build_optimizer(model, _Args)
    seed, r0, k = 99, 7, 3
    model._engine.seed_dropout(seed, r0)
    micro = [bert_ref.synthetic_batch(cfg, 4, 128, 1700 + j, padded=(j == 1)) for j in range(k)]
    losses = _window_backward(model, micro, cuda_dev)
    masks = [oracle_masks(cfg, 4, 128, seed, r0 + j) for j in range(k)]
    rl, rg = window_grads(state, cfg, micro, masks=masks)
    for j in range(k):
        assert abs(losses[j] - float(rl[j])) <= TOL_LOSS, (j, losses[j], float(rl[j]))
    worst, rows = grad_report(model.grad_dict(), rg)
    assert worst <= TOL_GRAD_REL, sorted(rows, key=lambda r: -r[1])[:5]


# ---- GPU: trajectories ------------------------------------------------------------------------------------------------------
def _trajectory_setup(k, steps, seed0):
    cfg = tiny_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    state = state_from_hf_init(cfg)
    windows = [[bert_ref.synthetic_batch(cfg, 4, 128, seed0 + 10 * s + j, padded=((s + j) % 2 == 1))
                for j in range(k)] for s in range(steps)]
    ref = {n: v.clone() for n, v in state.items()}
    hist = train_accum(ref, cfg, [[w] for w in windows])
    return cfg, state, windows, ref, hist


def _check_trajectory(losses, hist, model, ref, what):
    for s, h in enumerate(hist):
        for j, lv in enumerate(losses[s]):
            want = float(h["loss_per_rank"][0][j])
            assert abs(lv - want) <= TOL_TRAJ, (what, s, j, lv, want)
    sd = model.state_dict()
    for n, v in ref.items():
        assert float((sd[n].cpu() - v).abs().max()) <= 2e-4, (what, n)


@pytest.mark.gpu
def test_trajectory_eager_and_captured_trainer_match_oracle(cuda_dev):
    """4 optimizer steps of k = 3 micro-batches through the eager no_sync() loop and Trainer(fused=True); k = 2 through
    Trainer(pack=True)"""
    k, steps = 3, 4
    cfg, state, windows, ref, hist = _trajectory_setup(k, steps, 3100)
    model = make_model(cfg, state, cuda_dev).train()
    opt = b2.build_optimizer(model, _Args)
    losses = []
    for w in windows:
        losses.append(_window_backward(model, w, cuda_dev))
        opt.step()
        opt.zero_grad()
    _check_trajectory(losses, hist, model, ref, "eager")

    def trainer_run(k, windows, **kw):
        class A(b2.Args):
            fused, use_grad_accumulation, grad_accumulation, pack = True, True, k, False
            weight_decay, learning_rate = 0.01, 3e-5
        for n, v in kw.items():
            setattr(A, n, v)
        m = make_model(cfg, state, cuda_dev).train()
        o = b2.build_optimizer(m, A)
        tr = b2.Trainer(A, cfg, m, torch.nn.CrossEntropyLoss(), o)
        out = []
        for w in windows:
            out.append([float(tr.train_step(b, step_optimizer=(j == k - 1))) for j, b in enumerate(w)])
        return m, tr, out

    m, tr, l2 = trainer_run(k, windows)
    assert tr._fused.graph is not None and tr._fused._graph_accum is not None
    _check_trajectory(l2, hist, m, ref, "fused")

    cfg2, state2, windows2, ref2, hist2 = _trajectory_setup(2, steps, 3500)
    assert cfg2.hidden_size == cfg.hidden_size
    m, tr, l3 = trainer_run(2, windows2, pack=True)
    assert tr._packed
    _check_trajectory(l3, hist2, m, ref2, "packed")


# ---- GPU: surface rules ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_zero_grad_step_and_error_rules(cuda_dev):
    cfg = tiny_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    state = state_from_hf_init(cfg)
    a, b = (bert_ref.synthetic_batch(cfg, 4, 128, 1900 + i, padded=True) for i in range(2))

    # zero_grad() discards the pending micro-batch: the final backward then leaves b's gradient alone
    m1 = make_model(cfg, state, cuda_dev).train()
    o1 = b2.build_optimizer(m1, _Args)
    o1.zero_grad()                                        # nothing pending: a no-op
    with m1.no_sync():
        d = to_dev(a, cuda_dev)
        out = m1(input_ids=d["input_ids"], attention_mask=d["attention_mask"], labels=d["label"])
    F.cross_entropy(out[1], d["label"]).backward()
    assert m1._engine.accum_pending == 1
    o1.zero_grad()
    assert m1._engine.accum_pending == 0 and float(m1._engine.accum.abs().max()) == 0.0
    _window_backward(m1, [b], cuda_dev)
    m2 = make_model(cfg, state, cuda_dev).train()
    b2.build_optimizer(m2, _Args)
    _window_backward(m2, [b], cuda_dev)
    g1, g2 = m1.grad_dict(), m2.grad_dict()
    assert all(torch.equal(g1[n], g2[n]) for n in g1)
    o1.step()

    # step() after only no_sync() backwards (one GPU) applies the sum: same weights as a window closed by a final one
    def run(close_outside):
        m = make_model(cfg, state, cuda_dev).train()
        o = b2.build_optimizer(m, _Args)
        for j, bb in enumerate((a, b)):
            d = to_dev(bb, cuda_dev)
            ctx = contextlib.nullcontext() if (close_outside and j == 1) else m.no_sync()
            with ctx:
                out = m(input_ids=d["input_ids"], attention_mask=d["attention_mask"], labels=d["label"])
            (F.cross_entropy(out[1], d["label"]) / 2).backward()
        o.step()
        return m.state_dict(), int(o._state()["step"])
    w_closed, t_closed = run(True)
    w_open, t_open = run(False)
    assert t_closed == t_open == 1
    assert all(torch.equal(w_closed[n], w_open[n]) for n in w_closed)

    # a second final backward without a step raises, and so does a no_sync() backward after an unstepped final one
    m3 = make_model(cfg, state, cuda_dev).train()
    o3 = b2.build_optimizer(m3, _Args)
    _window_backward(m3, [a], cuda_dev)
    with pytest.raises(RuntimeError, match="accumulation"):
        _window_backward(m3, [a], cuda_dev)
    with pytest.raises(RuntimeError, match="accumulation"):
        _window_backward(m3, [a, b], cuda_dev)
    o3.step()
    _window_backward(m3, [a, b], cuda_dev)                # fine again after the step
    o3.step()


@pytest.mark.gpu
def test_gradscaler_with_accumulation(cuda_dev):
    """scaler.scale(loss / k).backward() k times, then scaler.step / update: lands where the unscaled accumulation lands;
    an inf in a NON-final micro-batch skips the whole window's step and backs the scale off"""
    cfg = tiny_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    state = state_from_hf_init(cfg)
    k = 2
    windows = [[bert_ref.synthetic_batch(cfg, 4, 128, 2300 + 10 * s + j, padded=(j == 1)) for j in range(k)]
               for s in range(3)]

    def fwd(model, bb, no_sync, amp):
        d = to_dev(bb, cuda_dev)
        ctx = model.no_sync() if no_sync else contextlib.nullcontext()
        with ctx, (torch.autocast("cuda") if amp else contextlib.nullcontext()):
            out = model(input_ids=d["input_ids"], attention_mask=d["attention_mask"], labels=d["label"])
            return F.cross_entropy(out[1], d["label"])

    plain = make_model(cfg, state, cuda_dev).train()
    opt = b2.build_optimizer(plain, _Args)
    for w in windows:
        for j, bb in enumerate(w):
            (fwd(plain, bb, j < k - 1, False) / k).backward()
        opt.step()
    amp = make_model(cfg, state, cuda_dev).train()
    opt2 = b2.build_optimizer(amp, _Args)
    scaler = torch.amp.GradScaler("cuda")
    for w in windows:
        for j, bb in enumerate(w):
            scaler.scale(fwd(amp, bb, j < k - 1, True) / k).backward()
        scaler.step(opt2)
        scaler.update()
    assert float(scaler.get_scale()) == 65536.0
    sd, sd2 = plain.state_dict(), amp.state_dict()
    for n in sd:
        assert float((sd[n].double() - sd2[n].double()).abs().max()) <= 2e-5, n

    before = {n: v.clone() for n, v in amp.state_dict().items()}
    t_before = int(opt2._state()["step"])
    scaler.scale(fwd(amp, windows[0][0], True, True) * float("inf") / k).backward()
    scaler.scale(fwd(amp, windows[0][1], False, True) / k).backward()
    scaler.step(opt2)
    scaler.update()
    assert float(scaler.get_scale()) == 32768.0
    assert int(opt2._state()["step"]) == t_before
    after = amp.state_dict()
    for n in before:
        assert torch.equal(before[n], after[n]), n
    assert float(amp._engine.accum.abs().max()) == 0.0          # the poisoned window left nothing behind


# ---- GPU, two B200s: the DDP path ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_ddp_no_sync_world2_matches_oracle():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29591", os.path.join(ROOT, "tests", "grad_accum_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    for mode in ("eager", "amp", "fused"):
        assert "mode %s OK" % mode in r.stdout, r.stdout[-3000:]
