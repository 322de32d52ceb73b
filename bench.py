#!/usr/bin/env python
"""Benchmark of the B200 Attention U-Net hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference|reference-gpu]
                  [--dump-outputs DIR]

A "step" is one training step (forward, DiceBCELoss, backward, gradient all-reduce for N > 1,
clip 1.0, AdamW) of AttentionUNet(1, 2, bilinear, 64) on a synthetic batch of B 1x512x512
CT-shaped images per GPU — BASELINE.json configs[1] (B = 4).  One process per GPU; for N > 1
launch under torchrun.  Rank 0 prints ONE JSON line.

  value       whole-job images/s with the batch already resident in HBM (CUDA-event timed, max over ranks)
  e2e         the same through the public API (`BatchShardedTrainer.step`) with pinned HOST buffers: H2D of
              the batch and a D2H read of the loss inside the timed region
  roofline    tensor-pipe fraction of the dominant kernels (every 3x3 / 1x1 forward and data-gradient
              implicit GEMM): CUDA events around each launch in an eager pass of the same step, algorithmic
              FLOPs = 2*pixels*Cout*taps*Cin per launch; peak = the BURST bf16 figure of MEASURED_PEAKS.json
              when the SM clock sat at its maximum while the kernels were timed, else the sustained one
  roofline_wgrad / roofline_convs   the same for the weight-gradient GEMMs / all three passes together
  kernels     per C-ABI entry point: launches, time, achieved TFLOP/s or GB/s and the fraction of its roof
  sustained   the same step replayed for >= 3 s (what a training run sees: power-capped clocks)
  configs     BASELINE configs[2] (UNet, batch 32), configs[3]'s per-GPU shape (AttentionUNet, batch 32) and
              configs[4] (inference sweep 1..256 with the confusion-matrix update in the loop), N = 1 only
  dp_check    N > 1: the replicas hold bit-identical parameters after the timed steps
  cpu_baseline  `--impl reference` (below) run as a child process on a bounded sample (3 steps)
  gpu_library_baseline  `--impl reference-gpu` as a child process: the UNMODIFIED reference on the same
              B200 through PyTorch/cuDNN (fp32, TF32, bf16 autocast + channels_last) — the same-box bar

  --impl reference      the reference's own CPU path on all host cores: the unmodified `unet` package from
              baseline/_ref (installed by baseline/install_reference.py; kind "reference"), its model, loss
              and the loop of scripts/train.py:132-143, same workload (batch 4 per step, never shrunk).
              Without baseline/_ref the oracle port runs instead (kind "port").

  --dump-outputs DIR    --impl ours only: after the K timed steps, write what the last of them handed its
              caller as float32 DIR/<name>.npy (32 MB in all; see dump_outputs).  The inputs and the initial
              weights are seeded, so two builds run with the same arguments can be compared output for output.
              bench_outputs/ is git-ignored for such dumps.

The benchmark writes nothing into the tree it runs from (which may be read-only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # no __pycache__ in the tree (children run this file and set it too)

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "unet-segment-pytorch_b200")
REF = os.path.join(ROOT, "baseline", "_ref")

METRIC = "AttentionUNet 512^2 train images/sec (whole job; per GPU = value / n_gpus)"
H = W = 512
WORKLOAD = ("AttentionUNet(1,2,bilinear,64) train step: fwd + DiceBCELoss + bwd + clip 1.0 + AdamW, "
            "1x512x512 inputs (BASELINE configs[1])")
FLOPS_TRAIN = {"attention": 983_373_447_168, "plain": 957_509_271_552}   # per 512^2 image, SURVEY §8d
FLOPS_FWD = {"attention": 327_891_812_352, "plain": 319_270_420_480}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during a timed region."""

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.reasons, self._halt = gpu_index, [], set(), threading.Event()
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu)], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def synthetic_batch(n, h, w, seed):
    """CT-shaped synthetic inputs (SURVEY.md 8d): images ~ clamp(randn, -1, 1) (the reference feeds
    (px/255 - 0.5)/0.5, unet/data/dataset.py:146); int64 masks with 1-3 filled ellipses covering
    ~0.36 % of the pixels (README.md:135), ~10 % of the images left empty."""
    import math

    import torch

    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 1, h, w, generator=g).clamp_(-1, 1)
    t = torch.zeros(n, h, w, dtype=torch.long)
    yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
    for i in range(n):
        if torch.rand((), generator=g).item() < 0.1:
            continue
        k = int(torch.randint(1, 4, (), generator=g).item())
        area = 0.0036 * h * w / k
        for _ in range(k):
            cy, cx = torch.rand((), generator=g).item() * h, torch.rand((), generator=g).item() * w
            ratio = 0.5 + torch.rand((), generator=g).item()
            ry, rx = max(1.0, math.sqrt(area / math.pi * ratio)), max(1.0, math.sqrt(area / math.pi / ratio))
            t[i][((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0] = 1
    return x, t


def base_config(batch, world):
    return {"workload": WORKLOAD, "batch_per_gpu": batch, "global_batch": batch * world, "parallelism": f"dp{world}"}


def child_json(extra_args, timeout):
    """Run another arm of this script as a child process; its last stdout line is its JSON."""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")}
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__)] + extra_args, capture_output=True, text=True,
                           timeout=timeout, env=env, cwd=ROOT)
        lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
        if r.returncode == 0 and lines:
            return json.loads(lines[-1])
        return {"unavailable": f"child exited {r.returncode}: {(r.stderr or r.stdout)[-300:]}"}
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}


# ----------------------------------------------------------------------------- reference arms
def _reference_objects():
    """(AttentionUNet, DiceBCELoss, kind): the unmodified reference from baseline/_ref, else None."""
    if not os.path.isfile(os.path.join(REF, "unet", "models", "unet.py")):
        return None
    sys.path.insert(0, REF)
    from unet.models import AttentionUNet   # the reference's own package: nothing of this repo on the path
    from unet.utils.loss import DiceBCELoss
    import unet
    assert os.path.realpath(unet.__file__).startswith(os.path.realpath(REF)), unet.__file__
    return AttentionUNet, DiceBCELoss


def run_reference_arm(args):
    """The reference's own CPU implementation of the step, all host threads, the arm's own workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    batch = args.batch
    x, t = synthetic_batch(batch, H, W, seed=1234)
    ref = _reference_objects()
    if ref is not None:
        kind = "reference"
        AttentionUNet, DiceBCELoss = ref
        torch.manual_seed(42)   # configs/lung_tumor.yaml:69
        model = AttentionUNet(n_channels=1, n_classes=2, bilinear=True, base_features=64)
        criterion = DiceBCELoss()
        opt = torch.optim.AdamW(model.parameters(), lr=5e-5, weight_decay=1e-4)   # train.py:346-350
        model.train()

        def step():   # scripts/train.py:132-143 with accumulation_steps = 1
            opt.zero_grad()
            loss = criterion(model(x), t)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            opt.step()
            return loss.item()
    else:
        kind = "port"
        sys.path.insert(0, ROOT)
        from oracle import unet_oracle as O
        cfg = dict(n_channels=1, n_classes=2, bilinear=True, base_features=64, attention=True)
        sd = O.synthetic_state_dict(42, **cfg)
        keys = [k for k, v in sd.items() if v.is_floating_point() and not k.endswith(("running_mean", "running_var"))]
        params = [sd[k].requires_grad_(True) for k in keys]
        opt = torch.optim.AdamW(params, lr=5e-5, weight_decay=1e-4)

        def step():
            opt.zero_grad()
            loss = O.dice_bce_loss(O.unet_forward(x, sd, attention=True, training=True), t)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
            return loss.item()

    warm = max(0, min(args.warmup, 1))
    for _ in range(warm):
        step()
    times = []
    for _ in range(args.steps):   # the workload is never shrunk, and exactly --steps steps are timed
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    per = sum(times) / len(times)
    ips = batch / per
    sample = (f"{'unmodified reference (baseline/_ref)' if kind == 'reference' else 'oracle port'}: fp32 CPU train step "
              f"(fwd + DiceBCELoss + bwd + clip 1.0 + AdamW), batch {batch}x1x512x512, {len(times)} timed steps "
              f"(+{warm} warm-up), {cores} threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "steps_timed": len(times), "warmup": args.warmup, "ms_per_step": per * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the arm's config is the GPU arm's for this N (what the driver pairs it with); the CPU process itself always
        # runs one batch_per_gpu-sized step at a time: `sample`
        "config": base_config(batch, max(1, args.gpus)),
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_reference_gpu(args):
    """The unmodified reference on the B200 through PyTorch's own kernels (cuDNN): the same-box bar."""
    import torch

    ref = _reference_objects()
    if ref is None or not torch.cuda.is_available():
        print(json.dumps({"impl": "reference-gpu", "unavailable": "baseline/_ref or CUDA missing"}))
        return
    AttentionUNet, DiceBCELoss = ref
    dev = torch.device("cuda", 0)
    torch.backends.cudnn.benchmark = True   # unet/utils/general.py:35
    out = {"impl": "reference-gpu", "unit": "images/s",
           "what": "unmodified reference (baseline/_ref) AttentionUNet(1,2,True,64) + DiceBCELoss + clip + AdamW on "
                   "this B200 via PyTorch/cuDNN, CUDA-event timed, inputs resident", "train": {}, "eval": {}}

    def timed(fn, iters, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    def build(channels_last):
        torch.manual_seed(42)
        m = AttentionUNet(1, 2, True, 64).to(dev)
        if channels_last:
            m = m.to(memory_format=torch.channels_last)
        return m

    modes = [("fp32", False, None, False), ("tf32", True, None, False), ("bf16_autocast_channels_last", True, torch.bfloat16, True)]
    for batch in (4, 32):
        x, t = synthetic_batch(batch, H, W, seed=1234)
        x, t = x.to(dev), t.to(dev)
        for name, tf32, amp, cl in modes:
            if batch == 32 and name == "fp32":
                continue
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            try:
                model = build(cl).train()
                crit = DiceBCELoss()
                opt = torch.optim.AdamW(model.parameters(), lr=5e-5, weight_decay=1e-4)
                xin = x.contiguous(memory_format=torch.channels_last) if cl else x

                def step():
                    opt.zero_grad()
                    with torch.autocast("cuda", dtype=amp, enabled=amp is not None):
                        logits = model(xin)
                    loss = crit(logits.float(), t)
                    loss.backward()
                    torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
                    opt.step()

                ms = timed(step, 10 if batch == 4 else 4, 4 if batch == 4 else 2)
                out["train"][f"batch{batch}_{name}"] = {"images_per_s": batch / ms * 1e3, "ms_per_step": ms}
                del model, opt
            except Exception as e:  # noqa: BLE001
                out["train"][f"batch{batch}_{name}"] = {"error": f"{type(e).__name__}: {str(e)[:120]}"}
            torch.cuda.empty_cache()
    # inference (configs[4]): eval forward + argmax metrics are host-side in the reference; forward only here
    for batch in (1, 16):
        x, _ = synthetic_batch(batch, H, W, seed=2)
        x = x.to(dev)
        for name, tf32, amp, cl in modes[1:]:
            torch.backends.cudnn.allow_tf32 = tf32
            model = build(cl).eval()
            xin = x.contiguous(memory_format=torch.channels_last) if cl else x

            def fwd():
                with torch.no_grad(), torch.autocast("cuda", dtype=amp, enabled=amp is not None):
                    model(xin)

            ms = timed(fwd, 10, 4)
            out["eval"][f"batch{batch}_{name}"] = {"images_per_s": batch / ms * 1e3, "ms": ms}
            del model
            torch.cuda.empty_cache()
    print(json.dumps(out))


# ----------------------------------------------------------------------------- GPU arm
def _shutdown(trainer, world):
    """Leave a multi-rank run: drop the captured graphs (they pin the NCCL communicator), meet
    the other ranks, tear the process group down — and never hang on the way out."""
    sys.stdout.flush()
    if world == 1:
        return
    import torch
    import torch.distributed as dist

    guard = threading.Timer(20.0, lambda: os._exit(0))
    guard.daemon = True
    guard.start()
    try:
        trainer.release_graphs()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
    except Exception:  # noqa: BLE001  the measurement is already printed
        pass
    sys.stdout.flush()
    os._exit(0)


def kernel_table(prof, steps, peaks, tensor_peak):
    """Per C-ABI entry point: launches / step, time / step, achieved rate and fraction of its roof."""
    hbm = float(peaks.get("hbm_gbs", 6550.0))
    agg = {}
    for name, e0, e1, work in prof:
        a = agg.setdefault(name, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0, "claimed": 0})
        a["launches"] += 1
        a["ms"] += e0.elapsed_time(e1)
        if work is not None:
            a["flops"] += work[0]
            a["bytes"] += work[1]
            a["claimed"] += 1
    table = {}
    for name, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        row = {"launches_per_step": a["launches"] / steps, "us_per_step": a["ms"] * 1e3 / steps}
        if a["claimed"] == a["launches"] and a["ms"] > 0:
            tf = a["flops"] / (a["ms"] * 1e-3) / 1e12
            gb = a["bytes"] / (a["ms"] * 1e-3) / 1e9
            # which roof: arithmetic intensity against the ridge of the measured peaks
            if a["flops"] > 0 and a["flops"] / max(a["bytes"], 1.0) > tensor_peak * 1e12 / (hbm * 1e9):
                row.update(bound="tensor", achieved=tf, unit="TFLOP/s", frac=tf / tensor_peak)
            else:
                row.update(bound="hbm", achieved=gb, unit="GB/s", frac=gb / hbm)
        table[name.replace("ub2_", "")] = row
    return table


def replica_check(model, trainer, dev, world):
    """Every rank's parameters against rank 0's (broadcast), per parameter: replicas must be bit-identical."""
    import torch
    import torch.distributed as dist

    names, worst = [], 0.0
    for name, p in model.named_parameters():
        ref = p.detach().clone()
        dist.broadcast(ref, src=0)
        d = (p.detach() - ref).abs().max().reshape(1)
        dist.all_reduce(d, op=dist.ReduceOp.MAX)
        if d.item() != 0.0:
            names.append((name, d.item()))
            worst = max(worst, d.item())
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    sums = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
    dist.all_gather(sums, flat.double().sum().reshape(1))
    return {"max_abs_param_diff_vs_rank0": worst, "param_checksums_equal": len({s.item() for s in sums}) == 1,
            "params_that_differ": len(names), "first_differing": names[:6], "param_checksum": sums[0].item(),
            "optimizer_steps": trainer._steps,
            "what": "after the timed steps every rank's parameters are compared with rank 0's (broadcast) and the "
                    "per-rank fp64 checksums gathered: replicas must be bit-identical"}


DUMP_SAMPLE = 1 << 22   # elements of the sampled arrays: 16 MiB each in float32


def dump_outputs(out_dir, model, loss):
    """What one training step hands its caller, as float32 .npy files under out_dir:
      loss           the loss the step returned (0-dim)
      bn_running     every BatchNorm running_mean / running_var the step updated, concatenated in model order
      params_sample  the updated parameters, all of them flattened in model.parameters() order, at DUMP_SAMPLE
                     positions drawn once from a generator seeded with 0 (in ascending order)
      grads_sample   the gradients of the step at the same positions
    AttentionUNet(1,2,True,64) has 17.6 M parameters (70 MB per full array), hence the fixed sample."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    params = list(model.parameters())
    flat_p = torch.cat([p.detach().reshape(-1) for p in params])
    flat_g = torch.cat([p.grad.detach().reshape(-1) for p in params])   # views into the trainer's buckets
    idx = torch.randperm(flat_p.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE]
    idx = idx.sort().values.to(flat_p.device)
    running = [b.detach().reshape(-1) for n, b in model.named_buffers() if n.endswith(("running_mean", "running_var"))]
    arrays = {"loss": loss.detach().reshape(()), "bn_running": torch.cat(running),
              "params_sample": flat_p[idx], "grads_sample": flat_g[idx]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.float().cpu().numpy())


def run_ours(args):
    for p in (PKG, ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: anything libraries print there (NCCL's version banner)
    # goes to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from unet import _C   # the GPU arm never touches oracle/
    from unet.inference import InferenceEngine
    from unet.models import AttentionUNet, UNet
    from unet.optim import FusedAdamW
    from unet.parallel import BatchShardedTrainer
    from unet.utils.loss import DiceBCELoss
    from unet.utils.metrics import SegmentationMetrics

    peaks, peak_src = load_peaks()
    B = args.batch

    def make_trainer(attention=True, graph=True):
        torch.manual_seed(42)  # configs/lung_tumor.yaml:69
        model = (AttentionUNet if attention else UNet)(n_channels=1, n_classes=2, bilinear=True, base_features=64).to(dev)
        opt = FusedAdamW(model.parameters(), lr=5e-5, weight_decay=1e-4)   # train.py:346-350, fused with the clip
        return BatchShardedTrainer(model, DiceBCELoss(), opt, grad_clip=1.0, cuda_graph=graph)

    trainer = make_trainer(True, not args.no_graph)
    model = trainer.model

    x_host, t_host = synthetic_batch(B, H, W, seed=1234 + rank)
    x_host, t_host = x_host.pin_memory(), t_host.pin_memory()
    x_dev, t_dev = x_host.to(dev), t_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    warm = max(3, args.warmup)
    for _ in range(warm + (4 if not args.no_graph else 0)):
        trainer.step(x_dev, t_dev)   # includes the eager warm-up steps and the graph capture

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    last_loss = [None]

    def timed_step():
        last_loss[0] = trainer.step(x_dev, t_dev)

    ms = timed(timed_step, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, last_loss[0])   # before any later step changes the model
    dp_check_after_graph = replica_check(model, trainer, dev, world) if world > 1 else None

    def profile_eager(tr, x, t, steps):
        """Per-launch CUDA events (and the launch count) in an eager pass of the very same step — a
        replayed CUDA graph has no per-launch host hooks."""
        eager = BatchShardedTrainer.__new__(BatchShardedTrainer)
        eager.__dict__.update(tr.__dict__)
        eager.cuda_graph = False
        eager._side_enabled = False   # one stream: a launch's two events then bracket that kernel alone
        eager.step(x, t)
        torch.cuda.synchronize()
        s = ClockSampler(local) if rank == 0 else None
        if s:
            s.start()
        _C.PROFILE = []
        _C.LAUNCHES = 0
        ms_eager = timed(lambda: eager.step(x, t), steps)
        prof, _C.PROFILE = _C.PROFILE, None
        return prof, _C.LAUNCHES // steps, ms_eager / steps, (s.stop() if s else None)

    prof_steps = 3
    prof, launches_per_step, ms_eager, prof_clocks = profile_eager(trainer, x_dev, t_dev, prof_steps)

    # end to end through the public API: host buffers in, loss value out, every step
    def e2e_step():
        return trainer.step(x_host, t_host).item()

    for _ in range(5):
        e2e_step()                   # host-buffer inputs share the captured graph (same shapes)
    ms_e2e = timed(e2e_step, args.steps)

    # what a training run sees: the same replayed step for >= 3 s (clocks settle under the power cap)
    sustained = None
    if not args.no_extras:
        n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / (ms / args.steps)) + 1)
        s2 = ClockSampler(local) if rank == 0 else None
        if s2:
            s2.start()
        ms_sus = timed(lambda: trainer.step(x_dev, t_dev), n_sus)
        c2 = s2.stop() if s2 else None
        sustained = {"value": B * world * n_sus / (ms_sus * 1e-3), "unit": "images/s", "steps": n_sus,
                     "seconds": ms_sus * 1e-3, "ms_per_step": ms_sus / n_sus, "clocks": c2}

    # what the collective costs: the same replayed step with the all-reduce left out (measurement knob of the trainer)
    collective = None
    if world > 1 and not args.no_extras:
        os.environ["UB2_SKIP_ALLREDUCE"] = "1"
        try:
            t2 = make_trainer(True, not args.no_graph)
            for _ in range(warm + (4 if not args.no_graph else 0)):
                t2.step(x_dev, t_dev)
            ms_nc = timed(lambda: t2.step(x_dev, t_dev), args.steps)
            collective = {"ms_per_step_without_allreduce": ms_nc / args.steps, "exposed_ms_per_step": (ms - ms_nc) / args.steps,
                          "bytes_per_step": sum(b.flat.numel() * 4 for b in trainer.buckets), "buckets": len(trainer.buckets),
                          "what": "same step, same graph capture, gradient all-reduce skipped (replicas diverge: timing only)"}
            t2.release_graphs()
            del t2
        finally:
            os.environ.pop("UB2_SKIP_ALLREDUCE", None)
        torch.cuda.empty_cache()

    dp_check = None
    if world > 1:
        dp_check = replica_check(model, trainer, dev, world)

    if rank != 0:
        _shutdown(trainer, world)
        return

    def roofline_of(entries, name, burst):
        rows = [(e0.elapsed_time(e1), w[0]) for n, e0, e1, w in prof if n in entries and w is not None]
        t_ms = sum(r[0] for r in rows)
        fl = sum(r[1] for r in rows)
        achieved = fl / (t_ms * 1e-3) / 1e12 if t_ms > 0 else 0.0
        peak = float(peaks.get("bf16_tflops" if burst else "bf16_tflops_sustained", 1400.0))
        return {"bound": "tensor", "kernel": name, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "traffic": None,
                "peak_source": f"{peak_src} {'bf16_tflops (burst)' if burst else 'bf16_tflops_sustained'}: SM clock while "
                               f"the kernels were timed = {prof_clocks.get('sm_mhz') if prof_clocks else None} MHz of "
                               f"{prof_clocks.get('sm_max_mhz') if prof_clocks else None}",
                "launches_per_step": len(rows) // prof_steps, "kernel_ms_per_step": t_ms / prof_steps,
                "algorithmic_flops_per_step": fl / prof_steps,
                "share_of_step": (t_ms / prof_steps) / (ms / args.steps),
                "how": "CUDA events around every launch in an eager ONE-STREAM pass of the same step "
                       f"({ms_eager:.2f} ms/step eager) right after the timed region; the replayed step runs the "
                       "weight-gradient kernels on a side stream next to the BatchNorm-backward passes, so the "
                       "per-kernel times add up to more than ms_per_step"}

    burst = bool(prof_clocks and prof_clocks.get("sm_mhz") and prof_clocks.get("sm_max_mhz")
                 and prof_clocks["sm_mhz"] >= 0.985 * prof_clocks["sm_max_mhz"])
    roofline = roofline_of({"ub2_conv_fwd"}, "conv_halo2_kernel / conv_fwd2_kernel / conv_fwd_kernel (3x3 and 1x1 "
                           "forward + data-gradient implicit GEMM, tcgen05, one- and two-CTA)", burst)
    try:   # DRAM bytes per launch of the same kernels from the committed ncu --set full capture
        with open(os.path.join(ROOT, "profiles", "conv_traffic.json")) as f:
            tj = json.load(f)
        roofline["traffic"] = tj["traffic_bytes_per_launch"]
        roofline["traffic_note"] = (f"mean dram__bytes_read+write per launch, {tj['source']}; algorithmic operand "
                                    f"bytes of the same launches: {tj['algorithmic_bytes_per_launch']:.3e}")
    except Exception:
        pass
    roofline_wgrad = roofline_of({"ub2_conv_wgrad"}, "conv_wgrad_halo2_kernel / conv_wgrad2_kernel / conv_wgrad_kernel "
                                 "(weight-gradient implicit GEMM, split-K)", burst)
    roofline_convs = roofline_of({"ub2_conv_fwd", "ub2_conv_wgrad"}, "all tcgen05 convolution launches (fwd + dgrad + wgrad)", burst)
    tensor_peak = roofline["peak"]
    kernels = kernel_table(prof, prof_steps, peaks, tensor_peak)

    total_imgs = B * world * args.steps
    value = total_imgs / (ms * 1e-3)
    step_tflops = FLOPS_TRAIN["attention"] * B / (ms / args.steps * 1e-3) / 1e12
    cfg = base_config(B, world)
    cfg.update({"collective": "NCCL all-reduce of flat gradient buckets overlapped with backward" if world > 1 else "none",
                "cuda_graph": not args.no_graph,
                "l2_policy": "activations per step (>1 GB) exceed the 126 MB L2; no flush needed"})
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": cfg,
        "e2e": {"value": total_imgs / (ms_e2e * 1e-3), "unit": "images/s",
                "h2d_bytes_per_step": (x_host.numel() * 4 + t_host.numel() * 8) * world,
                "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches_per_step * args.steps, "clocks": clocks, "roofline": roofline,
        "roofline_wgrad": roofline_wgrad, "roofline_convs": roofline_convs,
        "step_tensor_frac": {"achieved_tflops": step_tflops, "frac_of_burst": step_tflops / float(peaks.get("bf16_tflops", 1640.0)),
                             "what": "training FLOPs of the whole step (SURVEY §8d) / step time: end-to-end tensor-pipe fraction"},
        "kernels": kernels, "sustained": sustained, "dp_check": dp_check, "dp_check_after_graph_steps": dp_check_after_graph,
        "collective": collective,
    }

    # ---------------------------------------------------------------- the other BASELINE configs (N = 1)
    if world == 1 and not args.no_extras:
        trainer.release_graphs()
        del trainer, model
        torch.cuda.empty_cache()
        line["configs"] = other_configs(dev, timed, profile_eager, make_trainer, roofline_peak=tensor_peak,
                                        InferenceEngine=InferenceEngine, AttentionUNet=AttentionUNet,
                                        SegmentationMetrics=SegmentationMetrics)
        trainer = None
    if world == 1 and not args.no_cpu_baseline:
        torch.cuda.empty_cache()
        if not args.no_extras:
            line["gpu_library_baseline"] = child_json(["--impl", "reference-gpu"], 400)
        cb = child_json(["--impl", "reference", "--steps", "3", "--warmup", "1", "--batch", str(min(B, 4))], 400)
        line["cpu_baseline"] = cb.get("cpu_baseline", cb)
    else:
        line["cpu_baseline"] = None
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if trainer is not None:
        _shutdown(trainer, world)


def other_configs(dev, timed, profile_eager, make_trainer, roofline_peak, InferenceEngine, AttentionUNet, SegmentationMetrics):
    """BASELINE configs[2], configs[3]'s per-GPU shape and configs[4], each with its own numbers."""
    import torch

    out = {}
    for key, attention, what in (("cfg3_unet_train_batch32", False, "plain UNet(1,2,True,64) train step, batch 32 (BASELINE configs[2])"),
                                 ("cfg4_shape_attention_train_batch32", True,
                                  "AttentionUNet train step at configs[3]'s per-GPU batch 32, one GPU")):
        try:
            tr = make_trainer(attention, True)
            x, t = synthetic_batch(32, H, W, seed=1)
            x, t = x.to(dev), t.to(dev)
            for _ in range(7):
                tr.step(x, t)
            steps = 8
            ms = timed(lambda: tr.step(x, t), steps) / steps
            prof, launches, ms_eager, _ = profile_eager(tr, x, t, 1)
            conv = [(e0.elapsed_time(e1), w[0]) for n, e0, e1, w in prof if n in ("ub2_conv_fwd", "ub2_conv_wgrad") and w]
            conv_ms, conv_fl = sum(c[0] for c in conv), sum(c[1] for c in conv)
            fl = FLOPS_TRAIN["attention" if attention else "plain"] * 32
            out[key] = {"workload": what, "value": 32 / ms * 1e3, "unit": "images/s", "ms_per_step": ms, "steps": steps,
                        "step_tflops": fl / ms / 1e9, "gpu_launches_per_step": launches,
                        "roofline": {"bound": "tensor", "kernel": "all tcgen05 convolution launches", "unit": "TFLOP/s",
                                     "achieved": conv_fl / conv_ms / 1e9, "peak": roofline_peak,
                                     "frac": conv_fl / conv_ms / 1e9 / roofline_peak, "kernel_ms_per_step": conv_ms,
                                     "share_of_step": conv_ms / ms},
                        "peak_mem_gib": torch.cuda.max_memory_allocated() / 2 ** 30}
            tr.release_graphs()
            del tr, x, t
        except Exception as e:  # noqa: BLE001
            out[key] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
    # configs[0] and the fp32 accuracy mode: fp32 activations; inference = single-pass TF32 with BN folded, training =
    # 3xTF32 forward / data gradient + bf16x3 weight gradient (unet/fp32.py)
    try:
        import unet
        unet.set_precision("tf32")
        torch.manual_seed(42)
        model = AttentionUNet(1, 2, True, 64).to(dev).eval()
        x1, _ = synthetic_batch(1, H, W, seed=1234)
        x1 = x1.to(dev)

        def fwd():
            with torch.no_grad():
                model(x1)

        for _ in range(3):
            fwd()
        ms = timed(fwd, 20) / 20
        out["cfg1_attention_fp32_forward_batch1"] = {
            "workload": "AttentionUNet(1,2) eval forward, 1x1x512x512, fp32 activations / TF32 tensor-core convolutions "
                        "(BASELINE configs[0]); logits within 1e-3 of the fp32 reference (tests/test_fp32_mode_gpu.py)",
            "value": 1e3 / ms, "unit": "images/s", "ms": ms, "tflops": FLOPS_FWD["attention"] / ms / 1e9}
        tr = make_trainer(True, False)
        x, t = synthetic_batch(4, H, W, seed=1234)
        x, t = x.to(dev), t.to(dev)
        for _ in range(2):
            tr.step(x, t)
        ms = timed(lambda: tr.step(x, t), 3) / 3
        out["fp32_mode_train_batch4"] = {
            "workload": "AttentionUNet train step, batch 4, fp32 accuracy mode (3xTF32 forward / data gradient, bf16x3 weight "
                        "gradient, fp32 everything else; gradients within 1e-3 per module: tests/test_fp32_train_gpu.py), eager",
            "value": 4e3 / ms, "unit": "images/s", "ms_per_step": ms}
        del tr, model, x, t
    except Exception as e:  # noqa: BLE001
        out["fp32_mode"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    finally:
        import unet
        unet.set_precision("bf16")
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    # configs[4]: inference, BN folded, fused threshold + confusion counts, batch sweep
    try:
        torch.manual_seed(42)
        model = AttentionUNet(1, 2, True, 64).to(dev).eval()
        sweep = {}
        for b in (1, 2, 4, 8, 16, 32, 64, 128, 256):
            x, t = synthetic_batch(min(b, 16), H, W, seed=2)
            reps = (b + x.shape[0] - 1) // x.shape[0]
            x = x.repeat(reps, 1, 1, 1)[:b].to(dev)
            t = t.repeat(reps, 1, 1)[:b].to(dev)
            engine = InferenceEngine(model)
            metrics = SegmentationMetrics(2)

            def step():
                metrics.update(engine(x), t, threshold=0.5)   # softmax[:,1] > 0.5 (predict.py:155-159) + counts

            for _ in range(4):
                step()
            iters = 20 if b <= 16 else (8 if b <= 64 else 4)
            ms = timed(step, iters) / iters
            res = metrics.compute()
            sweep[str(b)] = {"images_per_s": b / ms * 1e3, "ms": ms, "tflops": b * FLOPS_FWD["attention"] / ms / 1e9,
                             "mean_dice": res.get("mean_dice"), "pixels_counted": int(metrics.confusion_matrix.sum()),
                             "peak_mem_gib": torch.cuda.max_memory_allocated() / 2 ** 30}
            del engine, x, t
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
        out["cfg5_attention_inference_sweep"] = {
            "workload": "AttentionUNet eval forward (BN folded, ReLU fused) + sigmoid-threshold + confusion counts per batch, "
                        "InferenceEngine graph replay (BASELINE configs[4])", "unit": "images/s", "batches": sweep}
    except Exception as e:  # noqa: BLE001
        out["cfg5_attention_inference_sweep"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps (--impl reference-gpu times its own fixed counts per precision mode)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=4, help="images per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU and cuDNN child processes")
    ap.add_argument("--no-extras", action="store_true", help="skip sustained / other configs / library baseline")
    ap.add_argument("--sustain-seconds", type=float, default=3.0)
    ap.add_argument("--no-graph", action="store_true", help="issue every kernel eagerly (no CUDA-graph replay)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl ours only: write the loss, BatchNorm statistics and a fixed sample of the parameters "
                         "and gradients after the last timed step as float32 DIR/<name>.npy (bench_outputs/ is "
                         "git-ignored)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours only")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.impl == "reference-gpu":
        run_reference_gpu(args)
        return
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
