"""One rank per GPU: gradient accumulation through the peer-HBM DDP wrapper vs tests/grad_accum_ref.train_accum.
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29591 \
        tests/grad_accum_worker.py
Three loops, k = 2 micro-batches per window: "eager" (ddp.no_sync() + (loss / k).backward(), step and zero_grad once per
window), "amp" (the same through GradScaler) and "fused" (Trainer with use_grad_accumulation: the two captured graphs).
Exits non-zero on any mismatch."""
import contextlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch
import torch.distributed as dist
import torch.nn.functional as F

from grad_accum_ref import train_accum
from parity import TOL_TRAJ, b2, bert_ref, state_from_hf_init, tiny_config
from pytorch_distributed_nlp_b200 import ddp as ddp_mod


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    cfg = tiny_config(hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    state = state_from_hf_init(cfg, seed=123)
    k, steps = 2, 4
    windows = [[[bert_ref.synthetic_batch(cfg, 4, 128, 8000 + 100 * s + 10 * r + j, padded=((s + j) % 2 == 1))
                 for j in range(k)] for r in range(world)] for s in range(steps)]
    ref = {n: v.clone() for n, v in state.items()}
    hist = train_accum(ref, cfg, windows)

    class A(b2.Args):
        weight_decay, learning_rate = 0.01, 3e-5
        fused, use_grad_accumulation, grad_accumulation, pack = True, True, k, False

    def forward(ddp, b, no_sync, amp):
        d = {n: v.to(dev) for n, v in b.items()}
        with (ddp.no_sync() if no_sync else contextlib.nullcontext()), \
                (torch.autocast("cuda") if amp else contextlib.nullcontext()):
            out = ddp(input_ids=d["input_ids"], token_type_ids=d["token_type_ids"],
                      attention_mask=d["attention_mask"], labels=d["label"])
            return F.cross_entropy(out[1], d["label"])

    nb = len(b2.BertForSequenceClassification(cfg)._layout.buckets)
    for mode in ("eager", "amp", "fused"):
        model = b2.BertForSequenceClassification(cfg)
        model.load_state_dict(state if rank == 0 else state_from_hf_init(cfg, seed=999))
        model.cuda()
        ddp = b2.DistributedDataParallel(model, device_ids=[local])
        opt = b2.build_optimizer(ddp, A)
        scaler = torch.amp.GradScaler("cuda") if mode == "amp" else None
        trainer = b2.Trainer(A, cfg, ddp, torch.nn.CrossEntropyLoss(), opt) if mode == "fused" else None
        torch.cuda.synchronize()
        ep0 = ddp.comm.epochs[ddp_mod._SLOT_BUCKET0:ddp_mod._SLOT_BUCKET0 + nb].clone()
        for s in range(steps):
            for j, b in enumerate(windows[s][rank]):
                final = j == k - 1
                if trainer is not None:
                    red = trainer.train_step(b, step_optimizer=final)
                    loss = None
                else:
                    loss = forward(ddp, b, not final, scaler is not None)
                    if scaler is not None:
                        scaler.scale(loss / k).backward()
                        if final:
                            scaler.step(opt)
                            scaler.update()
                    else:
                        (loss / k).backward()
                        if final:
                            opt.step()
                            opt.zero_grad()
                    red = ddp.loss_reduce(loss.detach())
                want = hist[s]["loss_per_rank"][:, j]
                if loss is not None:
                    assert abs(float(loss) - float(want[rank])) <= TOL_TRAJ, (mode, s, j, rank, float(loss))
                assert abs(float(red) - float(want.mean())) <= TOL_TRAJ, (mode, s, j, rank, float(red))
        torch.cuda.synchronize()
        # one barrier per bucket and window on the captured path (none per non-final micro-batch); the eager loops
        # exchange inside optimizer.step() behind one grads-ready barrier and use no bucket barrier at all
        adv = (ddp.comm.epochs[ddp_mod._SLOT_BUCKET0:ddp_mod._SLOT_BUCKET0 + nb] - ep0).tolist()
        assert adv == [steps if mode == "fused" else 0] * nb, (mode, adv)
        if scaler is not None:
            assert float(scaler.get_scale()) == 65536.0
        # every rank holds bit-identical bf16 weights
        sh = model._engine.shadow.clone()
        allsh = [torch.empty_like(sh) for _ in range(world)]
        dist.all_gather(allsh, sh)
        assert all(torch.equal(x, allsh[0]) for x in allsh), mode
        sd = ddp.state_dict()
        for n, v in ref.items():
            err = float((sd["module." + n].cpu() - v).abs().max())
            assert err <= 2e-4, (mode, n, err)
        if mode == "eager":
            # step() after only no_sync() backwards: the ranks never exchanged, stepping would let them diverge
            loss = forward(ddp, windows[0][rank][0], True, False)
            loss.backward()
            try:
                opt.step()
                raise AssertionError("step() after only no_sync() backwards did not raise")
            except RuntimeError as e:
                assert "no_sync" in str(e), e
            opt.zero_grad()
        if mode == "amp":
            # an inf on ONE rank in the first (non-final) micro-batch: every rank skips the window's step
            before = model._flat.clone()
            t_before = int(opt._state()["step"])
            loss = forward(ddp, windows[0][rank][0], True, True)
            scaler.scale(loss * (float("inf") if rank == world - 1 else 1.0) / k).backward()
            scaler.scale(forward(ddp, windows[0][rank][1], False, True) / k).backward()
            scaler.step(opt)
            scaler.update()
            torch.cuda.synchronize()
            assert float(scaler.get_scale()) == 32768.0, (rank, float(scaler.get_scale()))
            assert int(opt._state()["step"]) == t_before, rank
            assert torch.equal(model._flat, before), (rank, "a skipped window changed the weights")
        torch.cuda.synchronize()
        dist.barrier()
        if rank == 0:
            print("grad_accum_worker: mode %s OK (world %d)" % (mode, world), flush=True)
        ddp.close()
        del trainer, opt, ddp, model
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
