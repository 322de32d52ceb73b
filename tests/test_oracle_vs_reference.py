"""CPU: the oracle against the imported, unmodified reference on seeded random cases.  Runs where
$UNET_REFERENCE names a checkout of the reference (it is not part of this repository) and skips
elsewhere.  The same cases are checked on every machine against tests/golden/random_cases.pt
(tests/test_oracle_golden.py: test_random_cases, test_confusion_out_of_range_label)."""
import os

import pytest
import torch

from oracle import unet_oracle as O
from oracle.gen_golden import RANDOM_CASES, metrics_loop_inputs, random_case_inputs, reference_train_step

REF = os.environ.get("UNET_REFERENCE", "")
pytestmark = pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "unet"))),
                                reason="no reference checkout ($UNET_REFERENCE)")


@pytest.fixture(scope="module")
def ref():
    from oracle.gen_golden import import_reference
    return import_reference()


@pytest.mark.parametrize("attention,bilinear,hw", RANDOM_CASES)
def test_forward_backward_random(ref, attention, bilinear, hw):
    _, net, loss_mod, _ = ref
    loss, out, grads = reference_train_step(net, loss_mod, attention, bilinear, hw)
    _, sd, x, t = random_case_inputs(attention, bilinear, hw)
    o_loss, o_logits, o_grads = O.train_grads(x, t, O.clone_state(sd), attention=attention, bilinear=bilinear)
    assert torch.allclose(o_logits, out, rtol=1e-3, atol=1e-4)
    assert abs(o_loss.item() - loss.item()) < 1e-5
    for k, g in grads.items():
        assert torch.allclose(o_grads[k], g, rtol=5e-3, atol=1e-5 * g.abs().max().item() + 1e-9), k


def test_metrics_python_loop(ref):
    _, _, _, metrics_mod = ref
    z, t = metrics_loop_inputs()
    m = metrics_mod.SegmentationMetrics(4)
    m.update(z, t)
    assert (m.get_confusion_matrix() == O.confusion_matrix(z, t, 4)).all()
