"""Gradient accumulation on the B200: the fold kernel alone, and training throughput at k = 1, 2, 4 micro-batches per
optimizer step.  One JSON line per measurement (to stdout and, with --out, appended to a file); every line records
the card and its power limit.

    python tools/grad_accum_bench.py --out /tmp/grad_accum_1gpu.jsonl
    python -m torch.distributed.run --nproc-per-node 2 tools/grad_accum_bench.py --out ...   (DDP lines)

Fold kernel: b2_grad_accumulate over the whole config-A flat space (409 MB of fp32 accumulator + 205 MB of bf16
gradients, larger than the 126 MB L2), ADD (10 B per parameter) and FINISH (12 B), CUDA events over 50 launches each.
Throughput: config A (B = 32, S = 128), the device-resident captured replays of Trainer.train_step's FusedTrainStep,
as bench.py's `value`; k = 1 is today's step.  The k = 1 / k = 4 pair is repeated to show the run's spread.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch
import torch.distributed as dist


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                            "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in q.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(), "unknown"
    return {"gpu": name, "power_limit": power}


def fold_kernel(model, reps=50):
    from pytorch_distributed_nlp_b200 import _lib as L
    eng = model._engine
    n = model._layout.total
    acc = eng.ensure_accum()
    eng.grads.copy_(torch.randn(n, device=eng.dev).to(torch.bfloat16))
    s = torch.cuda.current_stream().cuda_stream
    out = []
    for mode, name, per_param in ((L.ACCUM_ADD, "ADD", 10), (L.ACCUM_FINISH, "FINISH", 12)):
        for _ in range(3):
            L.call("b2_grad_accumulate", acc.data_ptr(), eng.grads.data_ptr(), 0, n, 0.25, mode, s)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            L.call("b2_grad_accumulate", acc.data_ptr(), eng.grads.data_ptr(), 0, n, 0.25, mode, s)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / reps
        out.append({"what": "fold_kernel", "mode": name, "params": n, "bytes": per_param * n, "us": round(us, 1),
                    "GB_s": round(per_param * n / us / 1e3, 1)})
    acc.zero_()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60, help="micro-batches per timed run (a multiple of every k)")
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--ks", default="1,2,4,1,4,1,4")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import pytorch_distributed_nlp_b200 as b2

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("grad_accum_bench needs a GPU")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    info = dict(card(), world=world, config="A", batch=32, seq=128)
    lines = []

    def emit(obj):
        obj = dict(info, **obj)
        lines.append(obj)
        if rank == 0:
            print(json.dumps(obj), flush=True)
            if args.out:
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, "a") as f:
                    f.write(json.dumps(obj) + "\n")

    cfg = b2.chinese_bert_wwm_ext_config(num_labels=6)
    b2.set_seed(123)
    model = b2.BertForSequenceClassification(cfg)
    model.cuda()
    if rank == 0 and world == 1:
        for o in fold_kernel(model):
            emit(o)
    net = b2.DistributedDataParallel(model, device_ids=[local]) if world > 1 else model
    B, S = 32, 128
    ring = [b2.synthetic_batch(cfg, B, S, 1000 + rank + 64 * i) for i in range(16)]
    dev_ring = [torch.cat([b["input_ids"].reshape(-1), b["token_type_ids"].reshape(-1),
                           b["attention_mask"].reshape(-1), b["label"].reshape(-1)]).to(dev) for b in ring]
    base = b2.Args()
    base.local_rank, base.local_world_size, base.rank = local, world, rank
    optimizer = b2.build_optimizer(net, base)
    trainers = {}

    def trainer_for(k):
        if k not in trainers:
            class A(b2.Args):
                use_grad_accumulation, grad_accumulation = k > 1, k
                local_rank, local_world_size, rank = local, world, rank
            tr = b2.Trainer(A, cfg, net, torch.nn.CrossEntropyLoss(), optimizer)
            for i in range(args.warmup):          # through the public call: warm-up runs, then both graphs captured
                tr.train_step(ring[i % len(ring)], step_optimizer=(i + 1) % k == 0)
            trainers[k] = tr
        return trainers[k]

    def sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for k in [int(x) for x in args.ks.split(",")]:
        assert args.steps % k == 0
        step = trainer_for(k)._fused
        assert step.grad_accumulation == k and step.graph is not None
        for i in range(2 * k):
            step.d_stage.copy_(dev_ring[i % len(dev_ring)])
            step.run_device(final=(i + 1) % k == 0)
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            step.d_stage.copy_(dev_ring[i % len(dev_ring)])
            step.run_device(final=(i + 1) % k == 0)
        e1.record()
        sync()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms)
        loss = step.loss_to_host()
        emit({"what": "throughput", "k": k, "micro_batches": args.steps, "optimizer_steps": args.steps // k,
              "ms_per_micro_batch": round(ms / args.steps, 4),
              "samples_per_s": round(world * B * args.steps / (ms / 1e3), 1), "last_loss": round(loss, 5)})
    if world > 1:
        net.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
