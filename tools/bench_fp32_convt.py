"""fp32 / TF32 mode with bilinear=False: the ConvTranspose2d up-sampling kernels, the layer, and the whole network.

    python tools/bench_fp32_convt.py [--out profiles/r04_bench_fp32_convt.json]     (on a B200)

* kernel times of ub2_f32_shuffle2x2_fwd / _bwd (the latter with its bias gradient) at the four decoder levels of
  AttentionUNet(1, 2, bilinear=False, 64) at 4 x 1 x 512^2: CUDA events over 200 back-to-back launches after
  warm-up.  Bytes from shapes: t (N,h,w,4C) read + out (N,2h,2w,C) written, and the reverse; the bound is those
  bytes at 6.55 TB/s (the copy bandwidth this project measured on a B200).  A level whose operands (in + out) fit
  the 126 MB L2 is marked L2-resident: back-to-back launches then read it from L2, not HBM;
* the fp32-mode layer forward + backward (fp32.conv_transpose2x2 in training) against F.conv_transpose2d + F.pad
  through cuDNN on the same fp32 operands, with TF32 off and on;
* the whole fp32-mode AttentionUNet(1, 2, bilinear, 64): eval forward at batch 1 and a training step (forward,
  DiceBCE, backward) at batch 4, 512^2, for bilinear=False next to bilinear=True.
The card's name, power limit and maximum SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "unet-segment-pytorch_b200"))

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from bench_input_grad import HBM_TBPS, _card, _time_us  # noqa: E402

L2_BYTES = 126e6
N, HW, BASE = 4, 512, 64
# (name, Cin, h): up1..up4 of AttentionUNet(1, 2, False, 64) at 512^2 — ConvTranspose2d(Cin, Cin/2) from h x h
LEVELS = [("up1", 16 * BASE, HW // 16), ("up2", 8 * BASE, HW // 8), ("up3", 4 * BASE, HW // 4), ("up4", 2 * BASE, HW // 2)]


def shuffle_kernels():
    from unet import _C
    from unet import kernels as K
    from unet._C import ptr, stream
    out = []
    g = torch.Generator(device="cuda").manual_seed(0)
    for name, cin, h in LEVELS:
        c = cin // 2
        t = torch.randn((N, h, h, 4 * c), device="cuda", generator=g)
        o = torch.empty((N, 2 * h, 2 * h, c), device="cuda")
        dt = torch.empty_like(t)
        rows = K._rows("ub2_f32_shuffle2x2_rows", N, h, h, c, 2 * h, 2 * h)
        part = torch.empty((rows, c), device="cuda", dtype=torch.float64)
        db = torch.zeros((c,), device="cuda")

        def fwd():
            _C.call("ub2_f32_shuffle2x2_fwd", ptr(t), 4 * c, ptr(o), c, N, h, h, c, 2 * h, 2 * h, stream())

        def bwd():
            _C.call("ub2_f32_shuffle2x2_bwd", ptr(o), c, ptr(dt), 4 * c, ptr(part), rows, ptr(db), N, h, h, c, 2 * h, 2 * h,
                    stream())

        nbytes = (t.numel() + o.numel()) * 4
        bound_us = nbytes / (HBM_TBPS * 1e12) * 1e6
        for direction, fn in (("fwd", fwd), ("bwd", bwd)):
            us = _time_us(fn, iters=200, warmup=20)
            out.append({"level": name, "direction": direction, "shape_in": list(t.shape if direction == "fwd" else o.shape),
                        "us": us, "bytes": nbytes, "GBps": nbytes / us / 1e3, "hbm_bound_us": bound_us,
                        "frac_of_hbm_bound": bound_us / us, "l2_resident": nbytes <= L2_BYTES})
        assert torch.equal(dt, t), "shuffle backward did not invert the forward"
        del t, o, dt, part
        torch.cuda.empty_cache()
    return out


def layer():
    from unet import fp32
    out = []
    g = torch.Generator(device="cuda").manual_seed(1)
    for name, cin, h in LEVELS:
        mod = nn.ConvTranspose2d(cin, cin // 2, kernel_size=2, stride=2).cuda().train()
        x = torch.randn((N, cin, h, h), device="cuda", generator=g).contiguous(memory_format=torch.channels_last)
        gout = torch.randn((N, cin // 2, 2 * h, 2 * h), device="cuda", generator=g).contiguous(memory_format=torch.channels_last)
        xr = x.detach().requires_grad_(True)

        def ours():
            mod.zero_grad(set_to_none=True)
            xr.grad = None
            fp32.conv_transpose2x2(mod, xr, 2 * h, 2 * h).backward(gout)

        def cudnn():
            mod.zero_grad(set_to_none=True)
            xr.grad = None
            F.pad(F.conv_transpose2d(xr, mod.weight, mod.bias, stride=2), [0, 0, 0, 0]).backward(gout)

        row = {"level": name, "x": list(x.shape), "ours_fwd_bwd_us": _time_us(ours, iters=50, warmup=5)}
        prev = torch.backends.cudnn.allow_tf32
        for tf32 in (False, True):
            torch.backends.cudnn.allow_tf32 = tf32
            row[f"cudnn_fp32_tf32_{'on' if tf32 else 'off'}_us"] = _time_us(cudnn, iters=50, warmup=5)
        torch.backends.cudnn.allow_tf32 = prev
        out.append(row)
        del x, gout, xr, mod
        torch.cuda.empty_cache()
    return out


def network():
    import unet
    from unet.models import AttentionUNet
    from unet.utils.loss import DiceBCELoss
    out = []
    unet.set_precision("tf32")
    try:
        for bilinear in (False, True):
            torch.manual_seed(0)
            model = AttentionUNet(1, 2, bilinear, BASE).cuda()
            x1 = torch.randn((1, 1, HW, HW), device="cuda")
            model.eval()

            def eval_fwd():
                with torch.no_grad():
                    model(x1)

            eval_ms = _time_us(eval_fwd, iters=20, warmup=3) / 1e3
            model.train()
            x4 = torch.randn((N, 1, HW, HW), device="cuda")
            t4 = (torch.rand((N, HW, HW), device="cuda") < 0.05).long()
            loss_fn = DiceBCELoss()

            def step():
                model.zero_grad(set_to_none=True)
                loss_fn(model(x4), t4).backward()

            step_ms = _time_us(step, iters=10, warmup=3) / 1e3
            out.append({"model": f"AttentionUNet(1, 2, {bilinear}, {BASE})", "bilinear": bilinear,
                        "eval_fwd_batch1_ms": eval_ms, "train_step_batch4_ms": step_ms})
            del model
            torch.cuda.empty_cache()
    finally:
        unet.set_precision("bf16")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_bench_fp32_convt.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp32_convt.py measures on a CUDA device; none is visible")
    res = {"metric": "fp32 / TF32 mode ConvTranspose2d up-sampling (bilinear=False)", **_card(),
           "hbm_bandwidth_assumed_TBps": HBM_TBPS, "l2_bytes": L2_BYTES, "shuffle": shuffle_kernels(), "layer": layer(),
           "network": network()}
    line = json.dumps(res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
