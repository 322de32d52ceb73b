"""Generate tests/golden/*.pt from the UNMODIFIED reference, a checkout of which $UNET_REFERENCE names.

    UNET_REFERENCE=<checkout> python oracle/gen_golden.py
    python oracle/gen_golden.py --oracle-only     # tests/golden/random_cases.pt from the oracle alone

Each fixture holds the seeds / configuration that regenerate the inputs (synthetic weights and
batches come from oracle.unet_oracle's deterministic generators) and the reference's outputs:
eval logits, train-mode logits, loss, per-parameter gradient norms + leading values, updated
BatchNorm buffers, DiceBCE values / gradients on random logits and confusion matrices.  The
script also asserts, on the spot, that the oracle reproduces every one of them.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("UNET_REFERENCE", "")
sys.path.insert(0, ROOT)
from oracle import unet_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def import_reference():
    """Import the reference's modules from files (its package is also called `unet`)."""
    import importlib.util

    if not (REF and os.path.isdir(os.path.join(REF, "unet"))):
        raise RuntimeError("set UNET_REFERENCE to a checkout of the unmodified reference")

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    import types
    pkg = types.ModuleType("refunet"); pkg.__path__ = [os.path.join(REF, "unet")]
    sys.modules["refunet"] = pkg
    mpkg = types.ModuleType("refunet.models"); mpkg.__path__ = [os.path.join(REF, "unet", "models")]
    sys.modules["refunet.models"] = mpkg
    layers = load("refunet.models.layers", "unet/models/layers.py")
    net = load("refunet.models.unet", "unet/models/unet.py")
    loss = load("refunet.loss", "unet/utils/loss.py")
    metrics = load("refunet.metrics", "unet/utils/metrics.py")
    return layers, net, loss, metrics


def grad_summary(named_grads):
    return {k: {"norm": g.norm().item(), "head": g.flatten()[:8].clone()} for k, g in named_grads.items()}


def model_case(net, loss_mod, attention, bf, seed, n, hw, **kw):
    cfg = dict(n_channels=1, n_classes=2, bilinear=kw.get("bilinear", True), base_features=bf, attention=attention,
               deep_supervision=kw.get("deep_supervision", False))
    sd = O.synthetic_state_dict(seed, **cfg)
    mk = dict(n_channels=1, n_classes=2, bilinear=cfg["bilinear"], base_features=bf)
    if attention:
        mk["deep_supervision"] = cfg["deep_supervision"]
    model = (net.AttentionUNet if attention else net.UNet)(**mk)
    assert list(model.state_dict().keys()) == list(sd.keys()), "state_dict key order"
    model.load_state_dict(sd, strict=True)
    x, t = O.synthetic_batch(n, hw, hw, seed=seed + 100, fg_fraction=0.05)

    model.eval()
    with torch.no_grad():
        eval_logits = model(x)
    model.train()
    out = model(x)
    crit = loss_mod.DiceBCELoss()
    if isinstance(out, list):
        crit = loss_mod.DeepSupervisionLoss(crit)
    loss = crit(out, t) / 8  # accumulation_steps = 8 (configs/lung_tumor.yaml:27)
    loss.backward()
    main = out[0] if isinstance(out, list) else out
    grads = {k: p.grad for k, p in model.named_parameters()}
    buffers = {k: v.clone() for k, v in model.state_dict().items()
               if k.endswith(("running_mean", "running_var", "num_batches_tracked")) and ("inc." in k or "up4" in k)}

    # the oracle must agree with the reference (fp32 both; tolerance = summation-order noise)
    ocfg = {k: cfg[k] for k in ("bilinear", "deep_supervision")}
    o_eval = O.unet_forward(x, sd, attention=attention, training=False, **ocfg)
    assert torch.allclose(o_eval, eval_logits, rtol=1e-4, atol=1e-5), (o_eval - eval_logits).abs().max()
    o_sd = O.clone_state(sd)
    o_loss, o_main, o_grads = O.train_grads(x, t, o_sd, attention=attention, loss_scale=1 / 8, **ocfg)
    assert torch.allclose(o_main, main.detach(), rtol=1e-3, atol=1e-4)
    assert abs(o_loss.item() - loss.item()) < 1e-5
    for k, g in grads.items():
        cos = torch.dot(o_grads[k].flatten(), g.flatten()) / (o_grads[k].norm() * g.norm() + 1e-30)
        assert cos > 0.9999, (k, cos)
    for k, v in buffers.items():
        assert torch.allclose(o_sd[k].float(), v.float(), rtol=1e-4, atol=1e-6), k
    return {"cfg": cfg, "seed": seed, "n": n, "hw": hw, "fg_fraction": 0.05, "loss_scale": 1 / 8,
            "eval_logits": eval_logits, "train_logits": main.detach(), "loss": loss.item(),
            "grads": grad_summary(grads), "buffers": buffers}


def loss_case(loss_mod):
    g = torch.Generator().manual_seed(11)
    z = 2 * torch.randn(3, 2, 40, 36, generator=g)
    t = (torch.rand(3, 40, 36, generator=g) < 0.1).long()
    t[0] = 0
    out = {"z": z, "t": t}
    for name, mod, fn in (("dice_bce", loss_mod.DiceBCELoss(), O.dice_bce_loss),
                          ("dice", loss_mod.DiceLoss(), O.dice_loss),
                          ("balanced_ce", loss_mod.BalancedCELoss(0.3), lambda a, b: O.balanced_ce(a, b, 0.3))):
        zr = z.clone().requires_grad_(True)
        v = mod(zr, t)
        v.backward()
        zo = z.clone().requires_grad_(True)
        vo = fn(zo, t)
        vo.backward()
        assert abs(v.item() - vo.item()) < 1e-6 and torch.allclose(zr.grad, zo.grad, rtol=1e-4, atol=1e-9), name
        out[name] = {"value": v.item(), "grad": zr.grad.clone()}
    return out


def metrics_case(metrics_mod):
    g = torch.Generator().manual_seed(12)
    out = []
    for c, ignore in ((2, None), (3, 2), (4, 255)):
        z = torch.randn(2, c, 24, 20, generator=g)
        z[:, :, :2] = 0.5
        t = torch.randint(0, c, (2, 24, 20), generator=g)
        if ignore is not None:
            t[torch.rand(2, 24, 20, generator=g) < 0.1] = ignore
        m = metrics_mod.SegmentationMetrics(num_classes=c, ignore_index=ignore)
        m.update(z, t)                       # the reference's per-pixel Python loop
        cm = m.get_confusion_matrix()
        res = m.compute()
        assert np.array_equal(cm, O.confusion_matrix(z, t, c, ignore))
        mine = O.metrics_from_confusion(cm)
        assert all(abs(mine[k] - res[k]) < 1e-12 for k in ("pixel_accuracy", "mean_iou", "mean_dice"))
        iou = metrics_mod.compute_iou(z, t, c)
        dice = metrics_mod.compute_dice(z, t, c)
        assert torch.allclose(iou, O.iou_per_class(z, t, c)) and torch.allclose(dice, O.dice_per_class(z, t, c))
        out.append({"c": c, "ignore": ignore, "z": z, "t": t, "cm": torch.from_numpy(cm),
                    "result": {k: res[k] for k in ("pixel_accuracy", "mean_iou", "mean_dice")},
                    "iou": iou, "dice": dice})
    return out


def io_case():
    """The per-slice host work either side of the model, through the reference's own functions:
    apply_basic_transforms (unet/data/augmentations.py:117-170) on top of the two lines of
    LungTumorDataset.__getitem__ that precede it (dataset.py:146-151), and preprocess_image /
    postprocess_mask of scripts/predict.py (which reads a PNG: one is written to a temp dir)."""
    import importlib.util
    import tempfile
    from pathlib import Path
    from PIL import Image

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    aug = load("ref_augmentations", "unet/data/augmentations.py")
    rng = np.random.default_rng(21)
    n, h, w = 3, 48, 48
    images = rng.integers(0, 256, (n, h, w), dtype=np.uint8)
    images[0, 0, :256 % w] = 0
    images[0].reshape(-1)[:256] = np.arange(256, dtype=np.uint8)      # every grey level once
    labels = (rng.random((n, h, w)) < 0.2).astype(np.uint8) * 255
    labels[1].reshape(-1)[:4] = (127, 128, 1, 254)                      # the > 127 boundary
    xs, ts, flags = [], [], []
    for i in range(n):
        image = np.array(Image.fromarray(images[i]).convert("L"), dtype=np.float32) / 255.0   # dataset.py:146
        mask = (np.array(Image.fromarray(labels[i]).convert("L"), dtype=np.uint8) > 127).astype(np.int64)  # :147-151
        # find a numpy seed whose first draw takes the branch wanted for this slice (flip for odd i)
        want = i % 2 == 1
        seed = next(s for s in range(100) if (np.random.RandomState(s).rand() > 0.5) == want)
        np.random.seed(seed)
        x, t = aug.apply_basic_transforms(image, mask, img_size=h, is_train=True)
        xs.append(x); ts.append(t); flags.append(1 if want else 0)
    x_ref, t_ref = torch.stack(xs), torch.stack(ts)
    flags = np.array(flags, dtype=np.uint8)
    ox, ot = O.prepare_slices(images, labels, flags)
    assert torch.equal(ox, x_ref) and torch.equal(ot, t_ref), "oracle vs apply_basic_transforms"

    sys.argv = ["predict.py"]
    saved = {k: sys.modules.get(k) for k in list(sys.modules) if k == "unet" or k.startswith("unet.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, REF)
    try:
        pred = load("ref_predict", "scripts/predict.py")
    finally:
        sys.path.remove(REF)
        for k in [k for k in sys.modules if k == "unet" or k.startswith("unet.")]:
            del sys.modules[k]
        sys.modules.update({k: v for k, v in saved.items() if v is not None})
    with tempfile.TemporaryDirectory() as d:
        path = Path(d) / "slice.png"
        Image.fromarray(images[0]).save(path)
        tensor, _, size = pred.preprocess_image(path, img_size=h)
    px, _ = O.prepare_slices(images[:1], requantize=False)
    assert size == (w, h) and torch.equal(px, tensor), "oracle vs preprocess_image"

    g = torch.Generator().manual_seed(22)
    z = 3 * torch.randn(2, 2, h, w, generator=g)
    masks, counts = [], []
    for i in range(2):
        m = pred.postprocess_mask(z[i:i + 1], (w, h), threshold=0.6)
        masks.append(m); counts.append(int((m > 127).sum()))
    om, oc = O.predict_mask(z, 0.6)
    assert np.array_equal(om, np.stack(masks)) and list(oc) == counts, "oracle vs postprocess_mask"
    return {"images": torch.from_numpy(images), "labels": torch.from_numpy(labels), "flags": torch.from_numpy(flags),
            "x": x_ref, "t": t_ref, "x_predict": tensor, "z": z, "threshold": 0.6,
            "mask": torch.from_numpy(np.stack(masks)), "positives": torch.tensor(counts)}


# Seeded cases of tests/test_oracle_vs_reference.py that the model cases above do not cover: 3 input
# channels and 3 classes (DiceBCE over more than one foreground class), odd non-square sizes under bilinear
# up-sampling (the F.pad path), and a confusion matrix with an out-of-range label and no ignore_index.
RANDOM_CASES = [(True, True, (33, 47)), (False, True, (40, 24)), (True, False, (32, 32))]


def random_case_inputs(attention, bilinear, hw):
    cfg = dict(n_channels=3, n_classes=3, bilinear=bilinear, base_features=8, attention=attention)
    sd = O.synthetic_state_dict(9, **cfg)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 3, *hw, generator=g)
    t = torch.randint(0, 3, (2, *hw), generator=g)
    return cfg, sd, x, t


def metrics_loop_inputs():
    g = torch.Generator().manual_seed(2)
    z = torch.randn(1, 4, 16, 16, generator=g)
    t = torch.randint(0, 5, (1, 16, 16), generator=g)  # label 4 is out of range -> skipped
    return z, t


def reference_train_step(net, loss_mod, attention, bilinear, hw):
    """(loss, train-mode logits, gradients by key) of the reference's modules on one random case."""
    cfg, sd, x, t = random_case_inputs(attention, bilinear, hw)
    mk = {k: cfg[k] for k in ("n_channels", "n_classes", "bilinear", "base_features")}
    model = (net.AttentionUNet if attention else net.UNet)(**mk)
    model.load_state_dict(sd, strict=True)
    model.train()
    out = model(x)
    loss = loss_mod.DiceBCELoss()(out, t)
    loss.backward()
    return loss, out.detach(), {k: p.grad for k, p in model.named_parameters()}


def random_cases(ref=None):
    """Outputs on RANDOM_CASES -> tests/golden/random_cases.pt: train-mode logits, loss, per-parameter gradient
    norm / largest magnitude / first 8 values, and the confusion matrix of metrics_loop_inputs().  With
    ref = import_reference() they are the reference's and the oracle must reproduce them on the spot (the
    tolerances of tests/test_oracle_vs_reference.py); without, they are the oracle's.  "source" says which."""
    out = {"source": "oracle" if ref is None else "reference", "models": []}
    for attention, bilinear, hw in RANDOM_CASES:
        cfg, sd, x, t = random_case_inputs(attention, bilinear, hw)
        o_loss, o_logits, o_grads = O.train_grads(x, t, O.clone_state(sd), attention=attention, bilinear=bilinear)
        loss, logits, grads = o_loss, o_logits, o_grads
        if ref is not None:
            loss, logits, grads = reference_train_step(ref[1], ref[2], attention, bilinear, hw)
            assert torch.allclose(o_logits, logits, rtol=1e-3, atol=1e-4)
            assert abs(o_loss.item() - loss.item()) < 1e-5
            for k, g in grads.items():
                assert torch.allclose(o_grads[k], g, rtol=5e-3, atol=1e-5 * g.abs().max().item() + 1e-9), k
        out["models"].append({"attention": attention, "bilinear": bilinear, "hw": hw, "logits": logits.detach().clone(),
                              "loss": loss.item(),
                              "grads": {k: {"norm": g.norm().item(), "absmax": g.abs().max().item(),
                                            "head": g.flatten()[:8].clone()} for k, g in grads.items()}})
    z, t = metrics_loop_inputs()
    cm = O.confusion_matrix(z, t, 4)
    if ref is not None:
        m = ref[3].SegmentationMetrics(4)
        m.update(z, t)
        assert np.array_equal(m.get_confusion_matrix(), cm)
        cm = m.get_confusion_matrix()
    out["confusion"] = torch.from_numpy(np.asarray(cm))
    return out


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    os.makedirs(OUT, exist_ok=True)
    if "--oracle-only" in sys.argv:
        torch.save(random_cases(), os.path.join(OUT, "random_cases.pt"))
        print("random_cases.pt", os.path.getsize(os.path.join(OUT, "random_cases.pt")), "bytes")
        return
    layers, net, loss_mod, metrics_mod = import_reference()
    torch.save(random_cases((layers, net, loss_mod, metrics_mod)), os.path.join(OUT, "random_cases.pt"))
    cases = {
        "attn_bf32": model_case(net, loss_mod, True, 32, 1, 2, 32),
        "unet_bf16": model_case(net, loss_mod, False, 16, 2, 2, 48),
        "attn_bf16_ds": model_case(net, loss_mod, True, 16, 3, 2, 32, deep_supervision=True),
        "attn_bf16_convT": model_case(net, loss_mod, True, 16, 4, 1, 40, bilinear=False),
    }
    torch.save(cases, os.path.join(OUT, "models.pt"))
    torch.save(loss_case(loss_mod), os.path.join(OUT, "loss.pt"))
    torch.save(metrics_case(metrics_mod), os.path.join(OUT, "metrics.pt"))
    torch.save(io_case(), os.path.join(OUT, "io.pt"))
    # default-initialisation fingerprint: same seed -> same parameters as the reference constructor
    torch.manual_seed(42)
    ref = net.AttentionUNet(1, 2, True, 16)
    fp = {k: (v.double().sum().item(), v.flatten()[:4].clone()) for k, v in ref.state_dict().items()}
    torch.save(fp, os.path.join(OUT, "init_fingerprint.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)), "bytes")


if __name__ == "__main__":
    main()
