"""Gradients with respect to the network input: the stem data-gradient kernels and saliency-map throughput.

    python tools/bench_input_grad.py            (on a B200; prints one JSON line)

* kernel times of ub2_conv_in_dgrad (bf16 dy) and ub2_f32_conv_in_dgrad (fp32 dy) at N x 1 x 512^2, Cout 64,
  N = 4 and 32: CUDA events over 200 back-to-back launches after warm-up.  dy is 134 MB (bf16) / 268 MB (fp32)
  at N = 4, already larger than the 126 MB L2, so every launch streams dy from HBM.  Bounds from shapes: dy read
  + dx write at 6.55 TB/s (the copy bandwidth this project measured on a B200), and the FMA count at
  148 SMs x 128 FMA / clock at the SM clock the card reports as its maximum.  The same-box bar is
  torch.nn.grad.conv2d_input through cuDNN on the same operands (fp32 with TF32 off, and bf16 where cuDNN takes it);
* saliency throughput: AttentionUNet(1, 2, bilinear, 64) in eval with frozen parameters at 512^2, batch 1 / 4 / 16,
  forward + backward to the input, eager and CUDA-graph replayed, images/s, in both precisions.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "unet-segment-pytorch_b200"))

import torch  # noqa: E402

HBM_TBPS = 6.55


def _card():
    info = {"device": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        dev = torch.cuda.current_device()
        power, clock = [s.strip() for s in q[dev].split(",")]
        info.update(power_limit=power, sm_clock_max=clock)
    except Exception as e:  # a query failure leaves the numbers unlabelled; say so
        info.update(power_limit=None, sm_clock_max=None, query_error=str(e))
    return info


def _time_us(fn, iters=200, warmup=20):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def kernels(sm_mhz):
    from unet import kernels as K
    out = []
    g = torch.Generator(device="cuda").manual_seed(0)
    w = torch.randn((64, 1, 3, 3), device="cuda", generator=g) / 3
    for n in (4, 32):
        for dtype in (torch.bfloat16, torch.float32):
            dy = torch.randn((n, 512, 512, 64), device="cuda", generator=g).to(dtype)
            us = _time_us(lambda: K.conv_in_dgrad(dy, w, 1))
            nbytes = dy.numel() * dy.element_size() + n * 512 * 512 * 4
            fma = n * 512 * 512 * 64 * 9
            hbm_us = nbytes / (HBM_TBPS * 1e12) * 1e6
            fma_us = fma / (148 * 128 * sm_mhz * 1e6) * 1e6 if sm_mhz else None
            row = {"entry": "ub2_conv_in_dgrad" if dtype == torch.bfloat16 else "ub2_f32_conv_in_dgrad",
                   "shape": f"{n}x1x512x512 Cout 64", "us": us, "bytes": nbytes, "GBps": nbytes / us / 1e3,
                   "hbm_bound_us": hbm_us, "frac_of_hbm_bound": hbm_us / us, "fma": fma, "fma_bound_us": fma_us,
                   "frac_of_fma_bound": (fma_us / us) if fma_us else None}
            # cuDNN on the same operands (NHWC dy viewed as channels_last NCHW)
            dyc = dy.permute(0, 3, 1, 2)
            wc = w.to(dtype)
            prev = torch.backends.cudnn.allow_tf32
            torch.backends.cudnn.allow_tf32 = False
            try:
                row["cudnn_us"] = _time_us(lambda: torch.nn.grad.conv2d_input((n, 1, 512, 512), wc, dyc, padding=1),
                                           iters=50, warmup=5)
            except Exception as e:
                row["cudnn_us"], row["cudnn_error"] = None, str(e)[:200]
            finally:
                torch.backends.cudnn.allow_tf32 = prev
            out.append(row)
            del dy, dyc
            torch.cuda.empty_cache()
    return out


def saliency():
    import unet
    from unet.models import AttentionUNet
    out = []
    torch.manual_seed(0)
    model = AttentionUNet(1, 2, True, 64).cuda().eval()
    for p in model.parameters():
        p.requires_grad_(False)
    for precision in ("bf16", "tf32"):
        unet.set_precision(precision)
        for n in (1, 4, 16):
            xs = torch.randn((n, 1, 512, 512), device="cuda").requires_grad_(True)

            def step():
                (gx,) = torch.autograd.grad(model(xs).sum(), xs)
                return gx

            iters = max(5, 40 // n)
            eager_us = _time_us(step, iters=iters, warmup=3)
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    step()
            torch.cuda.current_stream().wait_stream(s)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step()
            graph_us = _time_us(graph.replay, iters=iters, warmup=3)
            out.append({"precision": precision, "batch": n, "eager_img_s": n / eager_us * 1e6,
                        "graph_img_s": n / graph_us * 1e6, "eager_ms": eager_us / 1e3, "graph_ms": graph_us / 1e3})
            del graph, xs
            torch.cuda.empty_cache()
    unet.set_precision("bf16")
    return out


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_input_grad.py measures on a CUDA device; none is visible")
    card = _card()
    try:
        sm_mhz = float(card["sm_clock_max"].split()[0])
    except Exception:
        sm_mhz = None
    res = {"metric": "stem data gradient (input gradient) kernels and saliency throughput", **card,
           "hbm_bandwidth_assumed_TBps": HBM_TBPS, "kernels": kernels(sm_mhz), "saliency": saliency()}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
