"""ORACLE — TEST INFRASTRUCTURE ONLY.  Never imported by the product path.

A CPU (plain fp32 torch / numpy) restatement of the reference's algorithm for the
Attention U-Net hot path, written functionally over a ``state_dict`` so that it
also pins the reference's parameter naming.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s cpu-baseline / ``--impl reference``
leg may import it, and only as the checker or the timed CPU baseline.

Parity status: **pinned** — the reference itself ships no tests or golden vectors
(SURVEY.md §4), so the oracle is pinned against outputs of the unmodified
reference run in the build container (``oracle/gen_golden.py`` →
``tests/golden/*.pt``) and, whenever ``$UNET_REFERENCE`` names a checkout, directly
against the imported reference (``tests/test_oracle_vs_reference.py``).

Every function cites the reference lines it restates (paths relative to the
reference repository root).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor
BN_EPS = 1e-5       # nn.BatchNorm2d default, unet/models/layers.py:33
BN_MOMENTUM = 0.1   # nn.BatchNorm2d default


# ------------------------------------------------------------------------------- storage model
# The product stores activations (raw conv outputs and post-ReLU tensors) in bf16.  The
# default oracle is pure fp32.  `bf16_storage()` makes the oracle round the same tensors to
# bf16 (straight-through gradient), so ReLU / max-pool decisions are taken on identical values
# and per-module input-gradient comparisons are not dominated by sign flips of near-zero
# pre-activations (a flip fraction f costs sqrt(f) relative L2, ~6 % for f = 0.3 %).
import contextlib

_STORAGE_BF16 = False


@contextlib.contextmanager
def bf16_storage(enabled: bool = True):
    global _STORAGE_BF16
    old, _STORAGE_BF16 = _STORAGE_BF16, enabled
    try:
        yield
    finally:
        _STORAGE_BF16 = old


def _st(t: Tensor) -> Tensor:
    if not _STORAGE_BF16:
        return t
    return t + (t.to(torch.bfloat16).to(t.dtype) - t).detach()


def _wq(w: Tensor) -> Tensor:
    """Tensor-core operand: the product feeds bf16-rounded conv weights to the MMA."""
    return _st(w)


# ------------------------------------------------------------------------------- blocks
def batch_norm(x: Tensor, sd: Dict[str, Tensor], p: str, training: bool) -> Tensor:
    """nn.BatchNorm2d (layers.py:33,36,153,159,165).  Train: biased batch variance to
    normalise, unbiased variance into running_var, momentum 0.1; updates ``sd`` in place."""
    w, b = sd[p + ".weight"], sd[p + ".bias"]
    if training:
        m = x.numel() // x.shape[1]
        mean = x.mean(dim=(0, 2, 3))
        var = x.var(dim=(0, 2, 3), unbiased=False)
        with torch.no_grad():
            sd[p + ".running_mean"].mul_(1 - BN_MOMENTUM).add_(BN_MOMENTUM * mean.detach())
            sd[p + ".running_var"].mul_(1 - BN_MOMENTUM).add_(
                BN_MOMENTUM * var.detach() * (m / max(m - 1, 1)))
            sd[p + ".num_batches_tracked"] += 1
    else:
        mean, var = sd[p + ".running_mean"], sd[p + ".running_var"]
    inv = torch.rsqrt(var + BN_EPS)
    return (x - mean[None, :, None, None]) * (inv * w)[None, :, None, None] + b[None, :, None, None]


def double_conv(x: Tensor, sd, p: str, training: bool) -> Tensor:
    """DoubleConv: (conv3x3 no-bias -> BN -> ReLU) x 2 (layers.py:31-38)."""
    for conv, bn in (("0", "1"), ("3", "4")):
        first_stem = conv == "0" and x.shape[1] % 16 != 0   # the stem conv runs in fp32 on CUDA cores
        w = sd[f"{p}.double_conv.{conv}.weight"]
        x = _st(F.conv2d(x, w if first_stem else _wq(w), None, 1, 1))
        x = _st(torch.relu(batch_norm(x, sd, f"{p}.double_conv.{bn}", training)))
    return x


def down(x: Tensor, sd, p: str, training: bool) -> Tensor:
    """Down: MaxPool2d(2) then DoubleConv (layers.py:55-58)."""
    return double_conv(F.max_pool2d(x, 2), sd, p + ".maxpool_conv.1", training)


def bilinear_to(x: Tensor, size) -> Tensor:
    """Bilinear resampling with align_corners=True (layers.py:78,183,212; unet.py:206-208)."""
    return F.interpolate(x, size=tuple(size), mode="bilinear", align_corners=True)


def attention_gate(g: Tensor, x: Tensor, sd, p: str, training: bool) -> Tensor:
    """AttentionGate.forward (layers.py:171-192): x * sigmoid(BN(psi(relu(BN(W_g up(g)) + BN(W_x x)))))."""
    if _STORAGE_BF16:
        # the product projects at low resolution (1x1 conv and bilinear resampling commute) and
        # stores that projection in bf16
        g1_raw = bilinear_to(_st(F.conv2d(g, _wq(sd[p + ".W_g.0.weight"]))), x.shape[2:])
    else:
        g1_raw = F.conv2d(bilinear_to(g, x.shape[2:]), sd[p + ".W_g.0.weight"])
    g1 = batch_norm(g1_raw, sd, p + ".W_g.1", training)
    x1 = batch_norm(_st(F.conv2d(x, _wq(sd[p + ".W_x.0.weight"]))), sd, p + ".W_x.1", training)
    s = torch.relu(g1 + x1)
    a = torch.sigmoid(batch_norm(F.conv2d(s, sd[p + ".psi.0.weight"]), sd, p + ".psi.1", training))
    return _st(x * a)


def up_block(x1: Tensor, x2: Tensor, sd, p: str, attention: bool, bilinear: bool, training: bool) -> Tensor:
    """Up.forward (layers.py:84-106) / AttentionUp.forward (layers.py:229-255).
    The gate sees the *un-upsampled* decoder tensor; concat order is [skip, upsampled]."""
    skip = attention_gate(x1, x2, sd, p + ".attention", training) if attention else x2
    if bilinear:
        up = _st(bilinear_to(x1, (2 * x1.shape[2], 2 * x1.shape[3])))
    else:
        up = _st(F.conv_transpose2d(x1, _wq(sd[p + ".up.weight"]), sd[p + ".up.bias"], stride=2))
    dy, dx = skip.shape[2] - up.shape[2], skip.shape[3] - up.shape[3]
    up = F.pad(up, [dx // 2, dx - dx // 2, dy // 2, dy - dy // 2])
    return double_conv(torch.cat([skip, up], dim=1), sd, p + ".conv", training)


def unet_forward(x: Tensor, sd, *, attention: bool, bilinear: bool = True, deep_supervision: bool = False,
                 training: bool = False):
    """UNet.forward (unet.py:67-92) / AttentionUNet.forward (unet.py:175-211)."""
    size = x.shape[2:]
    x1 = double_conv(x, sd, "inc", training)
    x2 = down(x1, sd, "down1", training)
    x3 = down(x2, sd, "down2", training)
    x4 = down(x3, sd, "down3", training)
    x5 = down(x4, sd, "down4", training)
    d4 = up_block(x5, x4, sd, "up1", attention, bilinear, training)
    d3 = up_block(d4, x3, sd, "up2", attention, bilinear, training)
    d2 = up_block(d3, x2, sd, "up3", attention, bilinear, training)
    d1 = up_block(d2, x1, sd, "up4", attention, bilinear, training)
    logits = F.conv2d(d1, sd["outc.conv.weight"], sd["outc.conv.bias"])
    if attention and deep_supervision and training:
        heads = []
        for name, d in (("ds_out1", d2), ("ds_out2", d3), ("ds_out3", d4)):
            heads.append(bilinear_to(F.conv2d(d, sd[name + ".conv.weight"], sd[name + ".conv.bias"]), size))
        return [logits] + heads
    return logits


# ------------------------------------------------------------------------------- parameters
def _double_conv_shapes(p, cin, cout, mid=None):
    mid = mid or cout
    out = {f"{p}.double_conv.0.weight": (mid, cin, 3, 3)}
    out.update(_bn_shapes(f"{p}.double_conv.1", mid))
    out[f"{p}.double_conv.3.weight"] = (cout, mid, 3, 3)
    out.update(_bn_shapes(f"{p}.double_conv.4", cout))
    return out


def _bn_shapes(p, c):
    return {f"{p}.weight": (c,), f"{p}.bias": (c,), f"{p}.running_mean": (c,), f"{p}.running_var": (c,),
            f"{p}.num_batches_tracked": ()}


def state_dict_shapes(n_channels=1, n_classes=2, bilinear=True, base_features=64, attention=True,
                      deep_supervision=False) -> Dict[str, tuple]:
    """Key -> shape table in the reference's registration order (unet.py:152-173, layers.py)."""
    bf = base_features
    factor = 2 if bilinear else 1
    shapes: Dict[str, tuple] = {}
    shapes.update(_double_conv_shapes("inc", n_channels, bf))
    for i, (ci, co) in enumerate([(bf, bf * 2), (bf * 2, bf * 4), (bf * 4, bf * 8), (bf * 8, bf * 16 // factor)], 1):
        shapes.update(_double_conv_shapes(f"down{i}.maxpool_conv.1", ci, co))
    ups = [(bf * 16, bf * 8 // factor), (bf * 8, bf * 4 // factor), (bf * 4, bf * 2 // factor), (bf * 2, bf)]
    for i, (ci, co) in enumerate(ups, 1):
        p = f"up{i}"
        if not bilinear:
            shapes[p + ".up.weight"] = (ci, ci // 2, 2, 2)
            shapes[p + ".up.bias"] = (ci // 2,)
        shapes.update(_double_conv_shapes(p + ".conv", ci, co, ci // 2 if bilinear else None))
        if attention:
            cg = ci // 2 if bilinear else ci
            cx = ci // 2
            inter = cx // 2
            shapes[p + ".attention.W_g.0.weight"] = (inter, cg, 1, 1)
            shapes.update(_bn_shapes(p + ".attention.W_g.1", inter))
            shapes[p + ".attention.W_x.0.weight"] = (inter, cx, 1, 1)
            shapes.update(_bn_shapes(p + ".attention.W_x.1", inter))
            shapes[p + ".attention.psi.0.weight"] = (1, inter, 1, 1)
            shapes.update(_bn_shapes(p + ".attention.psi.1", 1))
    shapes["outc.conv.weight"] = (n_classes, bf, 1, 1)
    shapes["outc.conv.bias"] = (n_classes,)
    if attention and deep_supervision:
        for name, c in (("ds_out3", bf * 8 // factor), ("ds_out2", bf * 4 // factor), ("ds_out1", bf * 2 // factor)):
            shapes[name + ".conv.weight"] = (n_classes, c, 1, 1)
            shapes[name + ".conv.bias"] = (n_classes,)
    return shapes


def synthetic_state_dict(seed: int = 0, **cfg) -> Dict[str, Tensor]:
    """Deterministic, init-order-independent synthetic parameters (one generator per key):
    conv weights U(+-1/sqrt(fan_in)) like the reference's default Kaiming(a=sqrt(5)) init,
    and *non-trivial* BN affine / running statistics so eval-mode parity exercises them."""
    sd: Dict[str, Tensor] = {}
    for i, (k, shape) in enumerate(state_dict_shapes(**cfg).items()):
        g = torch.Generator().manual_seed(seed * 100003 + i)
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.tensor(0, dtype=torch.long)
        elif k.endswith("running_mean"):
            sd[k] = 0.1 * torch.randn(shape, generator=g)
        elif k.endswith("running_var"):
            sd[k] = 0.5 + torch.rand(shape, generator=g)
        elif len(shape) == 4:
            fan_in = shape[1] * shape[2] * shape[3]
            sd[k] = (torch.rand(shape, generator=g) * 2 - 1) / math.sqrt(fan_in)
        elif ".conv.bias" in k or ".up.bias" in k:
            sd[k] = 0.1 * torch.randn(shape, generator=g)
        elif k.endswith(".weight"):  # BN gamma
            sd[k] = 0.75 + 0.5 * torch.rand(shape, generator=g)
        else:  # BN beta
            sd[k] = 0.1 * torch.randn(shape, generator=g)
    return sd


def synthetic_batch(n: int, h: int, w: int, seed: int = 1234, n_channels: int = 1, fg_fraction: float = 0.0036):
    """CT-shaped synthetic inputs (SURVEY.md §8d): images ~ clamp(randn, -1, 1) as the
    reference normalises to [-1, 1] (unet/data/dataset.py:146); masks are 1-3 filled
    ellipses covering ~0.36 % of the pixels (README.md:135), ~10 % of images left empty."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, n_channels, h, w, generator=g).clamp_(-1, 1)
    t = torch.zeros(n, h, w, dtype=torch.long)
    yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
    for i in range(n):
        if torch.rand((), generator=g).item() < 0.1:
            continue
        k = int(torch.randint(1, 4, (), generator=g).item())
        area = fg_fraction * h * w / k
        for _ in range(k):
            cy = torch.rand((), generator=g).item() * h
            cx = torch.rand((), generator=g).item() * w
            ratio = 0.5 + torch.rand((), generator=g).item()
            ry = max(1.0, math.sqrt(area / math.pi * ratio))
            rx = max(1.0, math.sqrt(area / math.pi / ratio))
            t[i][((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0] = 1
    return x, t


# ------------------------------------------------------------------------------- loss
def balanced_ce(logits: Tensor, targets: Tensor, class_weight: float = 0.5, smooth: float = 1e-6) -> Tensor:
    """BalancedCELoss.forward (unet/utils/loss.py:110-150): per image, class-1 pixels share
    weight cw, class-0 pixels share 1-cw, other labels get 0; sum over all pixels / N."""
    n = logits.shape[0]
    ce = F.cross_entropy(logits, targets, reduction="none")
    is1 = (targets == 1)
    is0 = (targets == 0)
    n1 = is1.flatten(1).sum(1).float() + smooth
    n0 = is0.flatten(1).sum(1).float() + smooth
    w = is1.float() * (class_weight / n1)[:, None, None] + is0.float() * ((1 - class_weight) / n0)[:, None, None]
    return (ce * w).sum() / n


def dice_loss(logits: Tensor, targets: Tensor, smooth: float = 1.0, ignore_background: bool = True) -> Tensor:
    """DiceLoss.forward, reduction='mean' (unet/utils/loss.py:45-85)."""
    c = logits.shape[1]
    p = torch.softmax(logits, dim=1)
    y = F.one_hot(targets, c).permute(0, 3, 1, 2).to(p.dtype)
    inter = (p * y).sum(dim=(2, 3))
    union = p.sum(dim=(2, 3)) + y.sum(dim=(2, 3))
    d = (2 * inter + smooth) / (union + smooth)
    if ignore_background and c > 1:
        d = d[:, 1:]
    return 1 - d.mean()


def dice_bce_loss(logits: Tensor, targets: Tensor, ce_weight=1.0, dice_weight=1.0, class_weight=0.5) -> Tensor:
    """DiceBCELoss.forward (unet/utils/loss.py:184-191)."""
    return ce_weight * balanced_ce(logits, targets, class_weight) + dice_weight * dice_loss(logits, targets)


def deep_supervision_loss(preds, targets: Tensor, weights=(1.0, 0.4, 0.2, 0.1), **kw) -> Tensor:
    """DeepSupervisionLoss.forward (unet/utils/loss.py:216-229)."""
    if isinstance(preds, (list, tuple)):
        return sum(w * dice_bce_loss(p, targets, **kw) for p, w in zip(preds, weights))
    return dice_bce_loss(preds, targets, **kw)


# ------------------------------------------------------------------------------- metrics
def confusion_matrix(pred, target, num_classes: int, ignore_index: Optional[int] = None) -> np.ndarray:
    """SegmentationMetrics.update (unet/utils/metrics.py:55-84), vectorised: argmax over
    dim 1 for logits (first maximum wins), count (t, p) pairs with both in [0, C)."""
    if isinstance(pred, Tensor) and pred.dim() == 4:
        pred = pred.argmax(dim=1)
    p = np.asarray(pred.cpu() if isinstance(pred, Tensor) else pred).reshape(-1).astype(np.int64)
    t = np.asarray(target.cpu() if isinstance(target, Tensor) else target).reshape(-1).astype(np.int64)
    keep = np.ones_like(t, dtype=bool)
    if ignore_index is not None:
        keep &= t != ignore_index
    keep &= (t >= 0) & (t < num_classes) & (p >= 0) & (p < num_classes)
    idx = t[keep] * num_classes + p[keep]
    return np.bincount(idx, minlength=num_classes * num_classes).reshape(num_classes, num_classes).astype(np.int64)


def metrics_from_confusion(cm: np.ndarray, class_names: Optional[List[str]] = None) -> dict:
    """SegmentationMetrics.compute (unet/utils/metrics.py:86-143)."""
    c = cm.shape[0]
    names = class_names or [f"class_{i}" for i in range(c)]
    total = cm.sum()
    if total == 0:
        return {"pixel_accuracy": 0.0, "mean_iou": 0.0, "mean_dice": 0.0,
                "class_iou": {n: 0.0 for n in names}, "class_dice": {n: 0.0 for n in names}}
    iou, dice = {}, {}
    for i in range(c):
        tp = cm[i, i]
        fp = cm[:, i].sum() - tp
        fn = cm[i, :].sum() - tp
        iou[names[i]] = tp / (tp + fp + fn) if (tp + fp + fn) > 0 else 0.0
        dice[names[i]] = 2 * tp / (2 * tp + fp + fn) if (2 * tp + fp + fn) > 0 else 0.0
    vi = [v for v in iou.values() if v > 0]
    vd = [v for v in dice.values() if v > 0]
    return {"pixel_accuracy": float(np.diag(cm).sum() / total),
            "mean_iou": float(np.mean(vi)) if vi else 0.0,
            "mean_dice": float(np.mean(vd)) if vd else 0.0,
            "class_iou": iou, "class_dice": dice}


def iou_per_class(pred: Tensor, target: Tensor, num_classes: int = 2, smooth: float = 1e-6) -> Tensor:
    """compute_iou (unet/utils/metrics.py:160-192)."""
    if pred.dim() == 4:
        pred = pred.argmax(dim=1)
    out = []
    for c in range(num_classes):
        a, b = pred == c, target == c
        out.append(((a & b).float().sum() + smooth) / ((a | b).float().sum() + smooth))
    return torch.stack(out)


def dice_per_class(pred: Tensor, target: Tensor, num_classes: int = 2, smooth: float = 1e-6) -> Tensor:
    """compute_dice (unet/utils/metrics.py:195-227)."""
    if pred.dim() == 4:
        pred = pred.argmax(dim=1)
    out = []
    for c in range(num_classes):
        a, b = (pred == c).float(), (target == c).float()
        out.append((2 * (a * b).sum() + smooth) / (a.sum() + b.sum() + smooth))
    return torch.stack(out)


# ------------------------------------------------------------------------------- either side of the model
def prepare_slices(images: np.ndarray, labels: Optional[np.ndarray] = None, flags: Optional[np.ndarray] = None,
                   mean: float = 0.5, std: float = 0.5, requantize: bool = True):
    """uint8 slices (N,H,W) -> (x fp32 (N,1,H,W), targets int64 (N,H,W) or None).

    LungTumorDataset.__getitem__ (unet/data/dataset.py:146-151): image = float32(px) / 255.0,
    mask = (label > 127) as int64; apply_basic_transforms (unet/data/augmentations.py:148-170):
    the image goes through uint8 once more, ``(image * 255).astype(np.uint8)`` then / 255.0 again
    (requantize), np.fliplr on both (flags bit 0; bit 1 = np.flipud, the albumentations pipeline's
    VerticalFlip, augmentations.py:78), ``(image - mean) / std`` in float32.  requantize=False is
    preprocess_image of scripts/predict.py:122-130 (one division, no flip)."""
    images = np.asarray(images, dtype=np.uint8)
    x = images.astype(np.float32) / 255.0
    if requantize:
        x = (x * 255).astype(np.uint8).astype(np.float32) / 255.0
    t = None if labels is None else (np.asarray(labels, dtype=np.uint8) > 127).astype(np.int64)
    if flags is not None:
        x, t = x.copy(), (None if t is None else t.copy())
        for n, f in enumerate(np.asarray(flags).reshape(-1)):
            if f & 1:
                x[n] = np.fliplr(x[n])
                if t is not None:
                    t[n] = np.fliplr(t[n])
            if f & 2:
                x[n] = np.flipud(x[n])
                if t is not None:
                    t[n] = np.flipud(t[n])
    x = (x - np.float32(mean)) / np.float32(std)
    return torch.from_numpy(np.ascontiguousarray(x)).unsqueeze(1).float(), (None if t is None else torch.from_numpy(t).long())


def predict_mask(logits: Tensor, threshold: float = 0.5):
    """postprocess_mask + tumor_ratio (scripts/predict.py:155-159, :238) per image: mask uint8 =
    255 * (softmax(logits, 1)[:, 1] > threshold), positives = number of set pixels."""
    prob = torch.softmax(logits.float(), dim=1)[:, 1].cpu().numpy()
    mask = (prob > threshold).astype(np.uint8) * 255
    return mask, (mask > 127).reshape(mask.shape[0], -1).sum(axis=1).astype(np.int64)


# ------------------------------------------------------------------------------- train step
def clone_state(sd):
    return {k: v.clone() for k, v in sd.items()}


def train_grads(x: Tensor, targets: Tensor, sd, *, attention: bool, loss_scale: float = 1.0, **cfg):
    """One micro-batch of train_one_epoch (scripts/train.py:128-136): forward in train mode,
    DiceBCE / accumulation_steps, backward.  Returns (loss, logits, grads by key); ``sd``'s BN
    buffers are updated in place exactly as the modules would."""
    params = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point()
              and not k.endswith(("running_mean", "running_var"))}
    work = dict(sd)
    work.update(params)
    logits = unet_forward(x, work, attention=attention, training=True, **cfg)
    loss = deep_supervision_loss(logits, targets) * loss_scale
    loss.backward()
    main = logits[0] if isinstance(logits, list) else logits
    return loss.detach(), main.detach(), {k: p.grad for k, p in params.items()}
