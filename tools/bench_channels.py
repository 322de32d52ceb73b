"""Channel counts that are not multiples of 16: what the padded per-tap tensor-core path costs.

    python tools/bench_channels.py [--out-dir DIR]      (on a B200; writes DIR/bench_channels.json)

* training: AttentionUNet(1, 2, bilinear, bf) for bf in 24 / 32 / 40 / 48 and AttentionUNet(n, 2, bilinear, 64) for
  n in 1 / 5 / 16, BatchShardedTrainer with its CUDA-graph replayed step, batch 4 at 512^2: ms per step over 20 steps
  after 6 (graph warm-up and capture included in those);
* inference: InferenceEngine (graph replayed) on the same models, batch 8 at 512^2: ms per call over 20 calls;
* the convolutions that take the padded path (a source or the output channel count not a multiple of 16): one eager
  bf16 train step of each model with every conv_fwd / conv_wgrad launch bracketed by CUDA events, reported per
  launch shape as time and TFLOP/s of the unpadded algorithmic FLOPs (2 * pixels * Cout * taps * Cin).  The event
  pairs cost a little launch overhead; kernel times of 10 us and more are what these numbers are good for.
bf = 32 and n = 1 have no padded layer and are the comparison points.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "unet-segment-pytorch_b200"))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SIZE = 512
MODELS = [(1, bf) for bf in (24, 32, 40, 48)] + [(n, 64) for n in (1, 5, 16)]


def _card():
    info = {"device": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        power, clock = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
        info.update(power_limit=power, sm_clock_max=clock)
    except Exception as e:  # a query failure leaves the numbers unlabelled; say so
        info.update(power_limit=None, sm_clock_max=None, query_error=str(e))
    return info


def _ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _batch(n, nc, seed):
    from oracle import unet_oracle as O
    x, t = O.synthetic_batch(n, SIZE, SIZE, seed=seed, n_channels=nc, fg_fraction=0.01)
    return x.cuda(), t.cuda()


def train_step_ms(nc, bf):
    from unet.models import AttentionUNet
    from unet.optim import FusedAdamW
    from unet.parallel import BatchShardedTrainer
    from unet.utils.loss import DiceBCELoss
    torch.manual_seed(0)
    model = AttentionUNet(nc, 2, True, bf).cuda()
    tr = BatchShardedTrainer(model, DiceBCELoss(), FusedAdamW(model.parameters(), lr=1e-4), grad_clip=1.0,
                             cuda_graph=True, graph_warmup=2)
    x, t = _batch(4, nc, 1)
    return _ms(lambda: tr.step(x, t), iters=20, warmup=6)


def inference_ms(nc, bf):
    from unet.inference import InferenceEngine
    from unet.models import AttentionUNet
    torch.manual_seed(0)
    engine = InferenceEngine(AttentionUNet(nc, 2, True, bf).cuda())
    x, _ = _batch(8, nc, 2)
    return _ms(lambda: engine(x), iters=20, warmup=4)


def padded_launches(nc, bf):
    """Every padded conv_fwd / conv_wgrad launch of one eager bf16 train step, timed with CUDA events."""
    from unet import kernels as K
    from unet.models import AttentionUNet
    from unet.utils.loss import DiceBCELoss
    torch.manual_seed(0)
    model = AttentionUNet(nc, 2, True, bf).cuda().train()
    x, t = _batch(4, nc, 3)
    loss_fn = DiceBCELoss()
    loss_fn(model(x), t).backward()        # warm-up: module loads, workspaces
    torch.cuda.synchronize()
    rows = []
    orig_fwd, orig_wg = K.conv_fwd, K.conv_wgrad

    def timed(kind, n, h, w, cin, cout, taps, run):
        if cin[0] % 16 == 0 and cin[1] % 16 == 0 and cout % 16 == 0:
            return run()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = run()
        e1.record()
        rows.append((kind, f"{n}x{h}x{w} C {cin[0]}+{cin[1]} -> {cout} taps {taps}",
                     2.0 * n * h * w * cout * taps * (cin[0] + cin[1]), e0, e1))
        return out

    def conv_fwd(x0, wgt, taps, x1=None, **kw):
        n, h, w, c0 = x0.shape
        return timed("fwd" if kw.get("out1") is None and kw.get("split", 0) == 0 else "dgrad", n, h, w,
                     (c0, x1.shape[3] if x1 is not None else 0), wgt.shape[0], taps,
                     lambda: orig_fwd(x0, wgt, taps, x1=x1, **kw))

    def conv_wgrad(x0, dy, taps, x1=None, **kw):
        n, h, w, c0 = x0.shape
        return timed("wgrad", n, h, w, (c0, x1.shape[3] if x1 is not None else 0), dy.shape[3], taps,
                     lambda: orig_wg(x0, dy, taps, x1=x1, **kw))

    K.conv_fwd, K.conv_wgrad = conv_fwd, conv_wgrad
    try:
        model.zero_grad(set_to_none=True)
        loss_fn(model(x), t).backward()
    finally:
        K.conv_fwd, K.conv_wgrad = orig_fwd, orig_wg
    torch.cuda.synchronize()
    out = []
    for kind, shape, flops, e0, e1 in rows:
        us = e0.elapsed_time(e1) * 1e3
        out.append({"kind": kind, "shape": shape, "us": round(us, 2), "unpadded_tflops": round(flops / us / 1e6, 1)})
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out-dir", default="bench_outputs")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_channels.py measures on a CUDA device; none is visible")
    res = {"metric": "padded channel counts: train step (graph, batch 4) and inference (graph, batch 8) at 512^2",
           **_card(), "models": []}
    for nc, bf in MODELS:
        row = {"model": f"AttentionUNet({nc}, 2, True, {bf})", "n_channels": nc, "base_features": bf,
               "train_step_ms_b4": round(train_step_ms(nc, bf), 3), "inference_ms_b8": round(inference_ms(nc, bf), 3),
               "padded_conv_launches": padded_launches(nc, bf)}
        res["models"].append(row)
        print(json.dumps({k: v for k, v in row.items() if k != "padded_conv_launches"}), flush=True)
        torch.cuda.empty_cache()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "bench_channels.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
