"""CPU: the oracle against the golden vectors of oracle/gen_golden.py.  fp32 on both sides: tolerances are
summation-order noise.  models / loss / metrics / io / init_fingerprint hold outputs of the UNMODIFIED
reference.  random_cases.pt names its origin in "source": the committed copy is the output of the oracle as
it stood when it last matched the reference on these seeded cases (tests/test_oracle_vs_reference.py), so a
later change of the oracle on those paths is caught without a reference checkout; with one,
`UNET_REFERENCE=<checkout> python oracle/gen_golden.py` rewrites it from the reference."""
import os

import numpy as np
import pytest
import torch

from oracle import unet_oracle as O
from oracle.gen_golden import RANDOM_CASES, metrics_loop_inputs, random_case_inputs

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    return torch.load(os.path.join(GOLD, name), weights_only=False)


@pytest.mark.parametrize("case", ["attn_bf32", "unet_bf16", "attn_bf16_ds", "attn_bf16_convT"])
def test_model_cases(case):
    g = _load("models.pt")[case]
    cfg = g["cfg"]
    sd = O.synthetic_state_dict(g["seed"], **cfg)
    x, t = O.synthetic_batch(g["n"], g["hw"], g["hw"], seed=g["seed"] + 100, fg_fraction=g["fg_fraction"])
    ocfg = {k: cfg[k] for k in ("bilinear", "deep_supervision")}
    ev = O.unet_forward(x, sd, attention=cfg["attention"], training=False, **ocfg)
    assert torch.allclose(ev, g["eval_logits"], rtol=1e-4, atol=1e-5)
    loss, logits, grads = O.train_grads(x, t, sd, attention=cfg["attention"], loss_scale=g["loss_scale"], **ocfg)
    assert torch.allclose(logits, g["train_logits"], rtol=1e-3, atol=1e-4)
    assert abs(loss.item() - g["loss"]) < 1e-5
    for k, ref in g["grads"].items():
        assert abs(grads[k].norm().item() - ref["norm"]) <= 2e-3 * ref["norm"] + 1e-7, k
        assert torch.allclose(grads[k].flatten()[:8], ref["head"], rtol=2e-2, atol=1e-3 * ref["norm"] + 1e-8), k
    for k, v in g["buffers"].items():
        assert torch.allclose(sd[k].float(), v.float(), rtol=1e-4, atol=1e-6), k


def test_loss_cases():
    g = _load("loss.pt")
    z, t = g["z"], g["t"]
    for name, fn in (("dice_bce", O.dice_bce_loss), ("dice", O.dice_loss),
                     ("balanced_ce", lambda a, b: O.balanced_ce(a, b, 0.3))):
        zr = z.clone().requires_grad_(True)
        v = fn(zr, t)
        v.backward()
        assert abs(v.item() - g[name]["value"]) < 1e-6, name
        assert torch.allclose(zr.grad, g[name]["grad"], rtol=1e-4, atol=1e-9), name


def test_metrics_cases():
    for g in _load("metrics.pt"):
        cm = O.confusion_matrix(g["z"], g["t"], g["c"], g["ignore"])
        assert np.array_equal(cm, g["cm"].numpy())
        res = O.metrics_from_confusion(cm)
        for k, v in g["result"].items():
            assert abs(res[k] - v) < 1e-12
        assert torch.allclose(O.iou_per_class(g["z"], g["t"], g["c"]), g["iou"])
        assert torch.allclose(O.dice_per_class(g["z"], g["t"], g["c"]), g["dice"])


@pytest.mark.parametrize("i", range(len(RANDOM_CASES)), ids=[f"{a}-{b}-{h[0]}x{h[1]}" for a, b, h in RANDOM_CASES])
def test_random_cases(i):
    """3 channels / 3 classes, odd sizes through the F.pad path (oracle/gen_golden.py:random_cases); the
    tolerances of tests/test_oracle_vs_reference.py."""
    g = _load("random_cases.pt")["models"][i]
    assert (g["attention"], g["bilinear"], tuple(g["hw"])) == RANDOM_CASES[i]
    _, sd, x, t = random_case_inputs(*RANDOM_CASES[i])
    loss, logits, grads = O.train_grads(x, t, sd, attention=g["attention"], bilinear=g["bilinear"])
    assert torch.allclose(logits, g["logits"], rtol=1e-3, atol=1e-4)
    assert abs(loss.item() - g["loss"]) < 1e-5
    assert grads.keys() == g["grads"].keys()
    for k, ref in g["grads"].items():
        assert abs(grads[k].norm().item() - ref["norm"]) <= 5e-3 * ref["norm"] + 1e-9, k
        assert torch.allclose(grads[k].flatten()[:8], ref["head"], rtol=5e-3, atol=1e-5 * ref["absmax"] + 1e-9), k


def test_confusion_out_of_range_label():
    """A label >= num_classes without ignore_index is skipped, as the reference's loop does."""
    z, t = metrics_loop_inputs()
    assert (t == 4).any()
    assert np.array_equal(O.confusion_matrix(z, t, 4), _load("random_cases.pt")["confusion"].numpy())


def test_state_dict_shapes_match_appendix_a():
    shapes = O.state_dict_shapes()
    assert len(shapes) == 182                                   # SURVEY.md App. A
    n_params = sum(int(np.prod(s)) for k, s in shapes.items()
                   if not k.endswith(("running_mean", "running_var", "num_batches_tracked")))
    assert n_params == 17_612_458
    assert len(O.state_dict_shapes(attention=False)) == 110
    assert len(O.state_dict_shapes(deep_supervision=True)) == 188
    assert len(O.state_dict_shapes(bilinear=False)) == 190


def test_io_cases():
    """prepare_slices / predict_mask against apply_basic_transforms, preprocess_image and
    postprocess_mask of the reference (fixture written by oracle/gen_golden.py:io_case)."""
    g = _load("io.pt")
    x, t = O.prepare_slices(g["images"].numpy(), g["labels"].numpy(), g["flags"].numpy())
    assert torch.equal(x, g["x"]) and torch.equal(t, g["t"])
    xp, none = O.prepare_slices(g["images"][:1].numpy(), requantize=False)
    assert none is None and torch.equal(xp, g["x_predict"])
    # the transform's second uint8 round trip changes no grey level
    lv = np.arange(256, dtype=np.uint8).reshape(1, 16, 16)
    assert torch.equal(O.prepare_slices(lv, requantize=True)[0], O.prepare_slices(lv, requantize=False)[0])
    m, c = O.predict_mask(g["z"], g["threshold"])
    assert np.array_equal(m, g["mask"].numpy()) and np.array_equal(c, g["positives"].numpy())
