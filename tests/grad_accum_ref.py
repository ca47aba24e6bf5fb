"""Test oracle for gradient accumulation: torch DDP ``no_sync()`` semantics, restated on top of oracle/.

Every rank sums ``grad(loss_j / k)`` over the k micro-batches of a window in fp32 (what ``(loss / k).backward()`` k
times leaves in ``.grad``, fabric/fabric-cls.py:150-161), the DDP mean over ranks is taken once per window (the last
backward, outside ``no_sync()``), then HF AdamW steps.  tests/test_grad_accum.py pins this against real torch: HF
``BertForSequenceClassification`` on CPU, and torch DDP on gloo at world 2.
"""
import torch

from oracle import adamw_ref, bert_ref, ddp_ref


def window_grads(params, cfg, micro_batches, masks=None):
    """sum over micro-batches of grad(loss_j / k), fp32.  masks: None or one dropout mask dict per micro-batch."""
    k = len(micro_batches)
    acc, losses = None, []
    for j, b in enumerate(micro_batches):
        loss, _logits, g = bert_ref.loss_and_grads(params, cfg, b, masks=None if masks is None else masks[j])
        losses.append(loss)
        if acc is None:
            acc = {n: torch.zeros_like(v) for n, v in g.items()}
        for n, v in g.items():
            acc[n] += v / k
    return torch.stack(losses), acc


def train_accum(params, cfg, windows, lr=3e-5, weight_decay=0.01):
    """windows: list over steps of list over ranks of lists of micro-batch dicts.  Dropout off.  Updates `params` in
    place.  Returns per step: dict(loss_per_rank [world, k], grads (rank mean of the window sums))."""
    opt = adamw_ref.HFAdamW(params, lr=lr, weight_decay=weight_decay)
    history = []
    for rank_windows in windows:
        losses, sums = [], []
        for micro in rank_windows:
            l, g = window_grads(params, cfg, micro)
            losses.append(l)
            sums.append(g)
        avg = ddp_ref.mean_grads(sums)
        history.append({"loss_per_rank": torch.stack(losses), "grads": avg})
        opt.step(avg)
    return history
