"""Device-time breakdown of one eager training step by C-ABI entry point (CUDA events around
every call; a leading device-side sleep lets the host run ahead so that no launch gap is timed).

Usage: python tools/step_profile.py [batch] [--unet] [--detail] [--out FILE.md]
"""
import argparse
import collections
import ctypes
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "unet-segment-pytorch_b200"))
sys.path.insert(0, ROOT)
from bench import synthetic_batch  # noqa: E402  (the bench's own generator; oracle/ is for tests only)
from unet import _C  # noqa: E402
from unet.models import AttentionUNet, UNet  # noqa: E402
from unet.parallel import BatchShardedTrainer  # noqa: E402
from unet.utils.loss import DiceBCELoss  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("batch", nargs="?", type=int, default=4)
    ap.add_argument("--unet", action="store_true")
    ap.add_argument("--detail", action="store_true")
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda")
    torch.manual_seed(42)
    model = (UNet if args.unet else AttentionUNet)(1, 2, True, 64).to(dev)
    from unet.optim import FusedAdamW
    opt = FusedAdamW(model.parameters(), lr=5e-5, weight_decay=1e-4)
    tr = BatchShardedTrainer(model, DiceBCELoss(), opt, grad_clip=1.0)
    x, t = synthetic_batch(args.batch, 512, 512, seed=1234)
    x, t = x.to(dev), t.to(dev)
    for _ in range(3):
        tr.step(x, t)
    torch.cuda.synchronize()

    records = []
    orig_call = _C.call

    def timed_call(name, *a, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_call(name, *a, **kw)
        e1.record()
        dims = tuple(v for (_, t), v in zip(_C.SIGNATURES[name], a) if t is not ctypes.c_void_p)   # sizes, not pointers
        records.append((name, dims, e0, e1))

    _C.call = timed_call
    from unet import kernels as K
    K._C.call = timed_call
    totals = []
    for _ in range(args.steps):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(int(60e6))     # ~30 ms: the host gets ahead of the device
        s0.record()
        tr.step(x, t)
        s1.record()
        totals.append((s0, s1))
    torch.cuda.synchronize()
    _C.call = orig_call
    K._C.call = orig_call

    step_ms = sum(a.elapsed_time(b) for a, b in totals) / args.steps
    agg = collections.OrderedDict()
    for name, dims, e0, e1 in records:
        key = (name, dims) if args.detail else name
        ms = e0.elapsed_time(e1)
        c = agg.setdefault(key, [0, 0.0])
        c[0] += 1
        c[1] += ms
    ours = sum(v[1] for v in agg.values()) / args.steps
    lines = [f"# eager train step, {'UNet' if args.unet else 'AttentionUNet'} batch {args.batch} x 1x512x512, "
             f"CUDA events per C-ABI call, mean of {args.steps} steps",
             f"step {step_ms:.3f} ms; C-ABI kernels {ours:.3f} ms; torch-side (optimizer, clip, autograd adds, fills) "
             f"{step_ms - ours:.3f} ms", "",
             "| entry point | calls/step | ms/step | share |", "|---|---|---|---|"]
    for key, (n, ms) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        nm = key if isinstance(key, str) else f"{key[0]} {key[1]}"
        lines.append(f"| {nm} | {n / args.steps:.1f} | {ms / args.steps:.3f} | {100 * ms / args.steps / step_ms:.1f}% |")
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
