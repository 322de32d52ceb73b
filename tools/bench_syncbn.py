"""What nn.SyncBatchNorm costs the batch-sharded trainer.

    python tools/bench_syncbn.py [--out-dir DIR] [--steps K]     (on B200s; writes DIR/r06_bench_syncbn.json)

* AttentionUNet(1, 2, bilinear, 64), BatchShardedTrainer with FusedAdamW and its CUDA-graph replayed step, one
  process per GPU over NCCL, at 2 and 8 GPUs x (batch 4 at 512^2, batch 1 at 512^2, batch 1 at 1024^2) per GPU:
  ms per step (the slowest rank, over K steps after 6 warm-up steps, graph capture included in those) for the
  unconverted model and for the model after ``nn.SyncBatchNorm.convert_sync_batchnorm``, the latter with the
  gradient buckets all-reduced as they fill (the trainer's default) and after backward (UB2_ALLREDUCE_AT_END=1).
  A world size larger than the number of visible GPUs is reported as not measured.
* The bytes one rank exchanges per step for the BatchNorm statistics, computed from the shapes of the fp64 tables
  one converted training step hands to unet.syncbn.exchange (30 forward, 26 backward exchanges for this model),
  and how many exchanges that is.
* Card name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "unet-segment-pytorch_b200"))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402
import torch.nn as nn  # noqa: E402

WORLDS = (2, 8)
SHAPES = ((4, 512), (1, 512), (1, 1024))          # (images per GPU, image side)
SETTINGS = (("unconverted", False, "0"), ("syncbn_buckets_as_filled", True, "0"),
            ("syncbn_buckets_after_backward", True, "1"))


def _card():
    info = {"device": torch.cuda.get_device_name(), "gpus_visible": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        power, clock = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
        info.update(power_limit=power, sm_clock_max=clock)
    except Exception as e:  # a query failure leaves the numbers unlabelled; say so
        info.update(power_limit=None, sm_clock_max=None, query_error=str(e))
    return info


def _model(convert):
    from unet.models import AttentionUNet
    torch.manual_seed(0)
    model = AttentionUNet(1, 2, True, 64)
    return nn.SyncBatchNorm.convert_sync_batchnorm(model) if convert else model


def _batch(n, size, seed):
    from oracle import unet_oracle as O
    x, t = O.synthetic_batch(n, size, size, seed=seed, fg_fraction=0.01)
    return x.cuda(), t.cuda()


def _worker(rank, world, root, n, size, convert, at_end, steps):
    os.environ["UB2_ALLREDUCE_AT_END"] = at_end
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"file://{root}/init", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        from unet.optim import FusedAdamW
        from unet.parallel import BatchShardedTrainer
        from unet.utils.loss import DiceBCELoss
        model = _model(convert).cuda()
        tr = BatchShardedTrainer(model, DiceBCELoss(), FusedAdamW(model.parameters(), lr=1e-4), grad_clip=1.0,
                                 cuda_graph=True, graph_warmup=2)
        x, t = _batch(n, size, 1 + rank)
        for _ in range(6):
            tr.step(x, t)
        torch.cuda.synchronize()
        dist.barrier(device_ids=[rank])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            tr.step(x, t)
        e1.record()
        torch.cuda.synchronize()
        with open(f"{root}/ms.{rank}", "w") as f:
            f.write(str(e0.elapsed_time(e1) / steps))
        tr.release_graphs()
    finally:
        dist.destroy_process_group()


def step_ms(world, n, size, convert, at_end, steps):
    with tempfile.TemporaryDirectory() as root:
        mp.spawn(_worker, args=(world, root, n, size, convert, at_end, steps), nprocs=world, join=True)
        return max(float(open(f"{root}/ms.{r}").read()) for r in range(world))


def exchanged_bytes(n, size):
    """Bytes and count of the statistics tables one converted training step exchanges, from their shapes: one
    eager step with unet.syncbn's exchange replaced by a recorder (no process group needed)."""
    from unet import syncbn
    from unet.utils.loss import DiceBCELoss
    seen = []

    def record(partials, count, group):
        seen.append(partials.numel() * partials.element_size())
        return partials, count

    orig = syncbn.group_of, syncbn.exchange
    syncbn.group_of = lambda bn: "recorder" if isinstance(bn, nn.SyncBatchNorm) and bn.training else getattr(
        bn, "sync_group", None)
    syncbn.exchange = record
    try:
        model = _model(True).cuda().train()
        x, t = _batch(n, size, 1)
        out = model(x)
        forward = len(seen)
        DiceBCELoss()(out, t).backward()
        torch.cuda.synchronize()
    finally:
        syncbn.group_of, syncbn.exchange = orig
    return {"forward_exchanges": forward, "backward_exchanges": len(seen) - forward,
            "bytes_per_step": sum(seen), "bytes_forward": sum(seen[:forward])}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out-dir", default="bench_outputs")
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_syncbn.py measures on CUDA devices; none is visible")
    res = {"metric": "AttentionUNet(1,2,True,64) graph-replayed BatchShardedTrainer step, ms (slowest rank), "
                     "with and without nn.SyncBatchNorm", **_card(), "runs": []}
    for n, size in SHAPES:
        row = {"images_per_gpu": n, "size": size, **exchanged_bytes(n, size)}
        for world in WORLDS:
            for name, convert, at_end in SETTINGS:
                key = f"{world}gpu_{name}_ms"
                if world > torch.cuda.device_count():
                    row[key] = f"not measured: {torch.cuda.device_count()} GPU(s) visible"
                    continue
                row[key] = round(step_ms(world, n, size, convert, at_end, args.steps), 3)
        res["runs"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "r06_bench_syncbn.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
