"""The reference's OWN training loop, unmodified, running on the drop-in (VERDICT r1 "missing" #2).

baseline/stage_ref.py stages utils/utils_fit.py byte for byte from the reference; `load_with_shims` executes that file with
`nets.unet_training` and `utils.utils_metrics` in sys.modules pointing at this package's drop-in modules -- exactly the import
swap INTEGRATION.md describes -- and `fit_one_epoch_no_val` (utils/utils_fit.py:175-280) then drives the CUDA engine through
`model_train(imgs)`, `CE_Loss`, `Dice_loss`, `f_score`, `loss.backward()`, `optimizer.step()`.  The same loop with nothing
swapped (reference model, reference losses, CPU fp32) is the yardstick."""
import contextlib
import os
import sys
import tempfile

import numpy as np
import pytest
import torch

from oracle import unet_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _History:
    def __init__(self):
        self.losses = []

    def append_loss(self, epoch, loss, *rest):
        self.losses.append(float(loss))


def _staged():
    from baseline import stage_ref
    return stage_ref if (stage_ref.stage() is not None and stage_ref.available()) else None


def _batches(C, n, hw, count):
    out = []
    for i in range(count):
        imgs, pngs = O.make_inputs(n, C, hw, hw, seed=40 + i)
        out.append((imgs, pngs, O.one_hot(pngs, C)))
    return out


def _run_loop(fit, model, cuda, C, batches, epochs, dice=True, focal=False, lr=1e-4):
    hist = _History()
    opt = torch.optim.Adam(model.parameters(), lr, betas=(0.9, 0.999), weight_decay=0.0)       # train.py:402-403
    cls_weights = np.ones([C], np.float32)                                                       # train.py:241
    with tempfile.TemporaryDirectory() as tmp:
        for ep in range(epochs):
            fit(model, model, hist, opt, ep, len(batches), iter(batches), epochs, cuda, dice, focal, cls_weights, C, False, None,
                5, tmp, 0)
        saved = sorted(os.listdir(tmp))
    return hist.losses, saved


def test_shimmed_loop_binds_the_dropin(b2u):
    """CPU: the unmodified utils_fit.py, loaded with the import swap, calls this package's losses and metric."""
    S = _staged()
    if S is None:
        pytest.skip("baseline/_ref is not staged")
    import unet_pytorch_b200.nets.unet_training as ours_t
    import unet_pytorch_b200.utils.utils_metrics as ours_m
    fit = S.load_with_shims("utils/utils_fit.py", {"nets.unet_training": ours_t, "utils.utils_metrics": ours_m})
    assert fit.CE_Loss is ours_t.CE_Loss and fit.Dice_loss is ours_t.Dice_loss and fit.Focal_Loss is ours_t.Focal_Loss
    assert fit.f_score is ours_m.f_score
    ref = S.import_reference("utils.utils_fit")
    assert ref.CE_Loss is not ours_t.CE_Loss
    src = open(os.path.join(S.REF_DST, "utils", "utils_fit.py"), "rb").read()
    if os.path.isdir(S.REF_SRC):      # byte-identical to the reference checkout (build container only)
        assert src == open(os.path.join(S.REF_SRC, "utils", "utils_fit.py"), "rb").read()
    # the host helpers the training scripts import from nets.unet_training are the reference's own functions
    assert ours_t.get_lr_scheduler("cos", 1e-4, 1e-6, 100)(0) == S.import_reference("nets.unet_training").get_lr_scheduler("cos", 1e-4, 1e-6, 100)(0)


@pytest.mark.gpu
@pytest.mark.parametrize("backbone,C", [("vgg", 21), ("vgg", 2)])
def test_reference_fit_one_epoch_runs_on_the_dropin(b2u, cuda_device, backbone, C):
    S = _staged()
    if S is None:
        pytest.skip("baseline/_ref is not staged")
    import unet_pytorch_b200.nets.unet_training as ours_t
    import unet_pytorch_b200.utils.utils_metrics as ours_m
    fit_ours = S.load_with_shims("utils/utils_fit.py", {"nets.unet_training": ours_t, "utils.utils_metrics": ours_m}).fit_one_epoch_no_val
    fit_ref = S.import_reference("utils.utils_fit").fit_one_epoch_no_val
    RefUnet = S.import_reference("nets.unet").Unet

    params = O.make_params(C, seed=11)
    batches = _batches(C, 2, 64, 2)
    ref_model = RefUnet(num_classes=C, pretrained=False, backbone=backbone)
    ref_model.load_state_dict(params)
    ref_losses, ref_saved = _run_loop(fit_ref, ref_model.train(), False, C, batches, epochs=2)

    model = b2u.Unet(num_classes=C, pretrained=False, backbone=backbone)
    model.load_state_dict(params)
    model = model.train().to(cuda_device)
    lib = b2u._lib.lib()
    lib.b2u_reset_launch_count()
    losses, saved = _run_loop(fit_ours, model, True, C, batches, epochs=2)
    assert lib.b2u_launch_count() > 4 * 100          # four iterations of the CUDA engine, not a fallback
    assert saved == ref_saved                          # the loop's own checkpoint files (state_dict round trip)
    print(f"\n[fit_one_epoch_no_val {backbone} nc={C}] drop-in epoch losses {losses} | unmodified reference on CPU {ref_losses}")
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 1e-2 * abs(b)
    # the parameters after four Adam steps (lr 1e-4): every tensor moved like the reference's
    after = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    ref_after = ref_model.state_dict()
    num = sum(((after[k] - params[k]) - (ref_after[k] - params[k])).double().pow(2).sum().item() for k in params)
    den = sum((ref_after[k] - params[k]).double().pow(2).sum().item() for k in params)
    assert (num / den) ** 0.5 <= 0.15                  # Adam's sign-like first steps amplify bf16 gradient noise on tiny entries
    assert max((after[k] - ref_after[k]).abs().max().item() for k in params) <= 8.1e-4     # <= 2 x 4 steps x lr (opposite signs on a ~0 gradient)


@contextlib.contextmanager
def _build(b2u, name):
    """'bf16' = the product library; 'fp32' = the fp32 validation build of the same ABI and host engines (logic check)."""
    if name == "fp32":
        b2u.ops.set_validation_fp32(True)
    try:
        yield
    finally:
        if name == "fp32":
            b2u.ops.set_validation_fp32(False)


@pytest.mark.gpu
@pytest.mark.parametrize("build", ["bf16", "fp32"])
@pytest.mark.parametrize("cin", [1, 4])
def test_lightweight_unet_non_rgb_inputs(b2u, cuda_device, cin, build):
    """LightweightUnet(num_classes, in_channels=...) (nets/LightWeightUnet.py:133): the reference accepts any channel count; the
    graph engine zero-pads the image to one 64-channel block (two-term bf16 split while 2C <= 64).  Tiny random-init fixture in
    training mode (BatchNorm over 2 x 4 x 4 samples at the bridge): the fp32 validation build pins the engine's logic to the
    reference (1e-4), the product bf16 path is held to the noise level such fixtures show for every BatchNorm family
    (tests/test_model_gpu.py, `_direct`).  The reference is the oracle's restatement of LightweightUnet.forward (pinned to the
    reference's own outputs by tests/test_oracle.py) in training mode without Dropout, on the weights the module's
    constructor draws (the drop-in keeps the reference's module tree and init)."""
    zb, gb = (1e-1, 1.0) if build == "bf16" else (1e-4, 2e-2)      # measured: 4.0-5.4e-2 / 6.0-6.2e-1 (bf16), 1.3e-5 / 9.3e-3 (fp32)
    torch.manual_seed(3)
    sd = b2u.LightweightUnet(num_classes=3, in_channels=cin).state_dict()
    ref = {k: (v.to(cuda_device).requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.to(cuda_device))
           for k, v in sd.items()}
    with _build(b2u, build):
        ours = b2u.LightweightUnet(num_classes=3, in_channels=cin)
        ours.load_state_dict(sd)
        ours = ours.to(cuda_device).train()
        for ins in ours._engine_for(cuda_device).program:
            if ins["op"] == "drop":
                ins["p"] = 0.0
        x = torch.rand(2, cin, 64, 64, device=cuda_device)
        zr, _ = O.lw_forward(ref, x, training=True)
        zo = ours(x)
        assert zo.shape == zr.shape
        zerr = ((zo - zr).norm() / zr.norm()).item()
        zr.square().mean().backward()
        zo.square().mean().backward()
        w = "backbone.stage1.0.conv.0.weight"
        gr = ref[w].grad
        go = dict(ours.named_parameters())[w].grad
        gerr = ((go - gr).norm() / gr.norm()).item()
        print(f"\n[LightweightUnet in_channels={cin} {build}] logits {zerr:.2e} first-conv gradient {gerr:.2e}")
        assert go.shape == gr.shape and zerr <= zb and gerr <= gb


@pytest.mark.gpu
@pytest.mark.parametrize("build", ["bf16", "fp32"])
def test_repvgg_improved_segnet_train_and_deploy(b2u, cuda_device, build):
    """nets/RepVGG_Unet.py::ImprovedSegNet (SURVEY 8(f) rank 4): the training form (two conv + BatchNorm branches per RepVGGBlock)
    against the reference in fp32 on the GPU -- logits, loss gradients, BatchNorm running statistics -- and the deploy form
    after `switch_to_deploy()` (one re-parameterised conv3x3 + bias + ReLU per block, eval mode) against the reference's
    deployed model.  The reference is the oracle's restatement (oracle.isn_forward / isn_deploy_params: the topology, SE
    blocks, BatchNorm and pooling of ulu_forward, which tests/test_oracle.py pins to the reference's own outputs, with the
    RepVGG block in place of the depthwise one).  The training form sums two BatchNorm branches per block over as few as
    4 x 4 x 4 samples on this tiny random-init fixture, which amplifies bf16 rounding far beyond the other families: the fp32
    validation build pins the program's logic (logits 2e-5, gradients 1.4e-3 measured), the product path is a regression guard
    there and is held to 5e-2 in the deploy form, where no batch statistics are involved."""
    with _build(b2u, build):
        _repvgg_case(b2u, cuda_device, build)


def _repvgg_case(b2u, cuda_device, build):
    zb, gb, sb, db_, ab = (5e-1, 1.0, 1e-1, 5e-2, 0.95) if build == "bf16" else (1e-4, 5e-3, 1e-4, 1e-4, 0.999)
    dev = cuda_device
    C = 4
    torch.manual_seed(5)
    sd = b2u.ImprovedSegNet(num_classes=C).state_dict()          # the module's own init (the reference's module tree)
    ref = {k: (v.to(dev).requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.to(dev))
           for k, v in sd.items()}
    ours = b2u.ImprovedSegNet(num_classes=C)
    ours.load_state_dict(sd)
    ours = ours.to(dev).train()
    for ins in ours._engine_for(dev).program:
        if ins["op"] == "drop":
            ins["p"] = 0.0
    imgs, pngs = O.make_inputs(4, C, 64, 64, seed=17)
    imgs, pngs = imgs.to(dev), pngs.to(dev)
    w = torch.ones(C, device=dev)
    labels = O.one_hot(pngs.cpu(), C).to(dev)
    zr, stats = O.isn_forward(ref, imgs, training=True)
    live_names = [k for k, v in ref.items() if v.requires_grad]
    gr = dict(zip(live_names, torch.autograd.grad(O.ce_loss(zr, pngs, w, C) + O.dice_loss(zr, labels), [ref[k] for k in live_names])))
    zo = ours(imgs)
    (b2u.CE_Loss(zo, pngs, w, num_classes=C) + b2u.Dice_loss(zo, labels)).backward()
    zerr = ((zo - zr).norm() / zr.norm()).item()
    go = {k: p.grad for k, p in ours.named_parameters()}
    live = [k for k in gr if gr[k].norm().item() > 1e-9]
    num = sum((go[k] - gr[k]).double().pow(2).sum().item() for k in live)
    den = sum(gr[k].double().pow(2).sum().item() for k in live)
    gerr = (num / den) ** 0.5
    print(f"\n[ImprovedSegNet train {build}] logits {zerr:.2e} grads {gerr:.2e}")
    assert zerr <= zb and gerr <= gb
    for k, a in ours.named_buffers():
        if k.endswith("running_mean") or k.endswith("running_var"):
            b = stats[k]
            assert ((a - b).norm() / (b.norm() + 1e-12)).item() <= sb, k
    # deploy: fold every RepVGGBlock, eval mode
    # (the deploy form is built from identical states: the training step above left bf16-level differences in the running statistics)
    ref_sd = {k: v.detach() for k, v in ref.items()}
    ref_sd.update(stats)
    ours.load_state_dict(ref_sd)
    ours.eval(); ours.switch_to_deploy()
    deployed = O.isn_deploy_params(ref_sd)
    assert sorted(ours.state_dict()) == sorted(deployed)
    for k in deployed:
        assert torch.allclose(ours.state_dict()[k], deployed[k], rtol=1e-5, atol=1e-6), k
    with torch.no_grad():
        dr, _ = O.isn_forward(deployed, imgs, training=False, deploy=True)
        do = ours(imgs)
    derr = ((do - dr).norm() / dr.norm()).item()
    print(f"[ImprovedSegNet deploy {build}] logits {derr:.2e}")
    assert derr <= db_
    assert (do.argmax(1) == dr.argmax(1)).float().mean().item() >= ab
