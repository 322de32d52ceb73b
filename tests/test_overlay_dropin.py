"""The drop-in boundary against the reference's own scripts (SURVEY.md §8b).

The reference's scripts import, next to the hot-path modules this package rebuilds, orchestration
modules it does not (scripts/train.py:28-35, scripts/predict.py:29-30).  With a reference checkout
attached (``unet.overlay``) those imports must resolve — hot path here, the rest in the reference's
own files — and the objects must work together the way train.py uses them.  Runs wherever a
checkout is available and skips elsewhere: $UNET_REFERENCE (the variable build() and the oracle tests
read too), else the copy build() stages under baseline/_ref.  $UNET_REFERENCE_ROOT is what the package
itself attaches at run time; the cases set or clear it themselves.
Each case runs in a fresh interpreter (import state is the thing under test).
"""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "unet-segment-pytorch_b200")


def _checkout():
    for c in (os.environ.get("UNET_REFERENCE", ""), os.path.join(ROOT, "baseline", "_ref")):
        if c and os.path.isfile(os.path.join(c, "unet", "__init__.py")) and os.path.isfile(os.path.join(c, "scripts", "train.py")):
            return c
    return None


CHECKOUT = _checkout()
needs_checkout = pytest.mark.skipif(CHECKOUT is None, reason="no reference checkout (with scripts/) available")


def _run(*code, **env):
    e = dict(os.environ, PYTHONPATH=PKG)
    e.pop("UNET_REFERENCE_ROOT", None)
    e.update(env)
    src = "\n".join(textwrap.dedent(c) for c in code)
    r = subprocess.run([sys.executable, "-c", src], capture_output=True, text=True, env=e, cwd="/tmp")
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


IMPORT_BLOCKS = '''
import re, sys
def import_block(path):
    """the top-level `from unet... import ...` lines of a reference script"""
    return "\\n".join(l for l in open(path).read().splitlines() if re.match(r"from unet[. ]", l))
'''


@needs_checkout
def test_train_and_predict_import_blocks_resolve_and_compose(tmp_path):
    out = _run(IMPORT_BLOCKS, f'''
        import os, torch
        import unet                                   # this package first (what `python -m unet.dropin` does)
        sys.path.insert(0, {CHECKOUT!r})              # scripts/train.py:25-26 then puts its checkout in front
        exec(import_block(os.path.join({CHECKOUT!r}, "scripts", "train.py")))
        exec(import_block(os.path.join({CHECKOUT!r}, "scripts", "predict.py")))
        here = {PKG!r}
        for obj in (UNet, AttentionUNet, create_loss_function, DeepSupervisionLoss, SegmentationMetrics, ModelEMA):
            assert sys.modules[obj.__module__].__file__.startswith(here), obj       # hot path: this package
        for obj in (LungTumorDataset, get_train_transforms, set_seed, get_device, load_config, increment_path,
                    EarlyStopping, ModelCheckpoint, ReduceLROnPlateau, plot_training_curves):
            assert sys.modules[obj.__module__].__file__.startswith({CHECKOUT!r}), obj  # the rest: reference files
        # the objects of train.py:306-420, built the way it builds them (CPU construction, train.py:306)
        set_seed(42)
        cfg = load_config(os.path.join({CHECKOUT!r}, "configs", "lung_tumor.yaml"))
        m = cfg["model"]
        model = AttentionUNet(n_channels=m["n_channels"], n_classes=m["n_classes"], bilinear=m.get("bilinear", True),
                              base_features=16, deep_supervision=True)
        ema = ModelEMA(model, decay=0.99)
        crit = DeepSupervisionLoss(create_loss_function(loss_type="dice_bce"))
        opt = torch.optim.AdamW(model.parameters(), lr=5e-5, weight_decay=1e-4)
        ckpt = ModelCheckpoint({str(tmp_path)!r}, monitor="mean_dice", mode="max", verbose=False)
        ckpt.save(model, opt, 0, {{"mean_dice": 0.5}})
        saved = sorted(os.listdir({str(tmp_path)!r}))
        assert "best.pt" in saved and "last.pt" in saved, saved
        sd = torch.load(os.path.join({str(tmp_path)!r}, "best.pt"), weights_only=False)
        model.load_state_dict(sd["model_state_dict"], strict=True)
        ema.ema_model.load_state_dict(model.state_dict())                      # train.py:465
        assert isinstance(get_device("cpu"), torch.device)
        print("composed", len(sd["model_state_dict"]))
    ''')
    assert "composed 188" in out     # AttentionUNet + deep supervision: 188 state_dict entries (SURVEY App. A)


@needs_checkout
def test_package_level_reexports_follow_the_reference():
    _run(f'''
        import unet
        from unet import overlay
        overlay.attach({CHECKOUT!r})
        from unet.utils import DiceLoss, DiceBCELoss, create_loss_function, SegmentationMetrics      # ours
        from unet.utils import set_seed, get_device, load_config, EarlyStopping, ModelCheckpoint     # reference's
        from unet.data import LungTumorDataset, get_train_transforms, get_val_transforms, DeviceBatchPipeline
        import unet.utils.general as G
        assert G.ModelEMA.__module__ == "unet.utils.general" and G.set_seed.__module__ == "unet.utils._reference_general"
    ''')


@needs_checkout
def test_environment_variable_attaches():
    _run('''
        from unet.utils.general import increment_path, ModelEMA
        from unet.utils.callbacks import EarlyStopping
    ''', UNET_REFERENCE_ROOT=CHECKOUT)


def test_without_a_checkout_the_error_says_what_to_do():
    out = _run('''
        import unet
        try:
            from unet.utils.general import set_seed
        except ImportError as e:
            print("IMPORTERROR", e)
        try:
            import unet.utils.callbacks
        except ModuleNotFoundError as e:
            print("MODULENOTFOUND", e)
        import unet.utils.general as G
        try:
            G.get_device
        except AttributeError as e:
            print("ATTR", e)
    ''')
    assert "IMPORTERROR" in out and "MODULENOTFOUND" in out and "UNET_REFERENCE_ROOT" in out


@needs_checkout
def test_dropin_launcher_runs_the_reference_scripts():
    for script in ("train.py", "predict.py"):
        r = subprocess.run([sys.executable, "-m", "unet.dropin", os.path.join(CHECKOUT, "scripts", script), "--help"],
                           capture_output=True, text=True, env=dict(os.environ, PYTHONPATH=PKG), cwd="/tmp")
        assert r.returncode == 0 and "usage:" in r.stdout, r.stdout + r.stderr


# --------------------------------------------------------------------------- the scripts themselves, on the GPU
def _tiny_dataset(root, volumes=5, slices=4, size=64):
    """PNG slices in the layout LungTumorDataset expects (unet/data/dataset.py:24-34): images/ and labels/,
    <volume>_slice_<k>.png, 8-bit grey, label 255 inside a disc."""
    import numpy as np
    from PIL import Image
    rng = np.random.default_rng(0)
    for sub in ("images", "labels"):
        os.makedirs(os.path.join(root, sub), exist_ok=True)
    yy, xx = np.mgrid[:size, :size]
    for v in range(volumes):
        for k in range(slices):
            img = (rng.normal(110, 40, (size, size))).clip(0, 255).astype(np.uint8)
            cy, cx, r = rng.integers(16, size - 16, 2).tolist() + [int(rng.integers(4, 9))]
            lab = (((yy - cy) ** 2 + (xx - cx) ** 2) <= r * r).astype(np.uint8) * 255
            img[lab > 0] = np.minimum(255, img[lab > 0].astype(int) + 60).astype(np.uint8)
            name = f"{v}_slice_{k:04d}.png"
            Image.fromarray(img).save(os.path.join(root, "images", name))
            Image.fromarray(lab).save(os.path.join(root, "labels", name))


@pytest.mark.gpu
@needs_checkout
def test_reference_train_and_predict_scripts_run_on_the_b200_package(tmp_path):
    """The reference's own scripts/train.py and scripts/predict.py, unmodified, through ``python -m unet.dropin``:
    one epoch on a tiny PNG dataset (dataset, transforms, config, callbacks, checkpoint I/O from the reference's
    files; model, loss, metrics, EMA from this package, on CUDA), then prediction from the checkpoint it wrote."""
    import torch
    import yaml
    data = tmp_path / "dataset"
    _tiny_dataset(str(data))
    with open(os.path.join(CHECKOUT, "configs", "lung_tumor.yaml")) as f:
        cfg = yaml.safe_load(f)
    cfg["model"].update(base_features=32)
    cfg["data"].update(root=str(data), img_size=64, batch_size=2, num_workers=0)
    cfg["train"].update(epochs=2, accumulation_steps=2)
    cfg["scheduler"].update(warmup_epochs=1)
    cfg["ema"] = {"enabled": True, "decay": 0.9}
    cfg["augmentation"]["enabled"] = False
    cfg["output"].update(save_dir=str(tmp_path / "runs"), experiment_name="dropin")
    cfg["device"] = "cuda"
    cfg_path = tmp_path / "cfg.yaml"
    cfg_path.write_text(yaml.safe_dump(cfg))
    env = dict(os.environ, PYTHONPATH=PKG)
    r = subprocess.run([sys.executable, "-m", "unet.dropin", os.path.join(CHECKOUT, "scripts", "train.py"), "--config", str(cfg_path)],
                       capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:] + "\n" + r.stderr[-3000:])
    weights = [os.path.join(dp, f) for dp, _, fs in os.walk(tmp_path / "runs") for f in fs if f.endswith(".pt")]
    assert any(w.endswith("last.pt") for w in weights), weights
    ckpt = torch.load([w for w in weights if w.endswith("last.pt")][0], map_location="cpu", weights_only=False)
    sys.path.insert(0, PKG)
    from unet.models import AttentionUNet
    model = AttentionUNet(1, 2, True, 32)
    model.load_state_dict(ckpt["model_state_dict"], strict=True)
    assert all(torch.isfinite(v).all() for v in ckpt["model_state_dict"].values() if v.is_floating_point())
    out = tmp_path / "pred"
    img = sorted(os.listdir(data / "images"))[0]
    r = subprocess.run([sys.executable, "-m", "unet.dropin", os.path.join(CHECKOUT, "scripts", "predict.py"), "--weights",
                        [w for w in weights if w.endswith("last.pt")][0], "--source", str(data / "images" / img), "--output",
                        str(out), "--img-size", "64", "--device", "cuda"],
                       capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=300)
    assert r.returncode == 0, (r.stdout[-3000:] + "\n" + r.stderr[-3000:])
    assert any(f.endswith(".png") for _, _, fs in os.walk(out) for f in fs)
