"""GPU: the whole hot path (drop-in Unet + losses + backward, the fused trainer step) against the CPU oracle and
against golden vectors produced by the reference itself.

Tolerances (BASELINE.json north_star): bf16 logits and gradients rel-L2 <= 1e-2 against the fp32 reference, arg-max
masks >= 99.9 % identical, fast_hist / mIoU exact.  The golden fixtures use weights at the scale of torch's default
Conv2d init (gain 0.5 x He), where bf16 storage noise of the *gradient* is 3e-3..8e-3.  With full-He weights
(gain 1.0) the same network amplifies bf16 rounding of weights/activations into a 3e-2 gradient difference no matter
who computes it (oracle.train_step_bf16_storage, an fp32 CPU run that only rounds where bf16 tensors are stored,
shows 2.8e-2; torch's own bf16 autocast 1.7e-2, SURVEY.md Appendix B), so that fixture is judged against the bf16
storage model (<= 1e-2) and must not exceed 1.5x the model's own distance from fp32."""
import os
import re
import socket

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _global_rel(grads, ref):
    num = sum((grads[k].float().cpu() - ref[k]).double().pow(2).sum().item() for k in ref)
    den = sum(ref[k].double().pow(2).sum().item() for k in ref)
    return (num / den) ** 0.5


def _argmax_agreement(logits, ref):
    a, b = logits.cpu().argmax(1), ref.argmax(1)
    top2 = ref.topk(2, dim=1).values
    margin = top2[:, 0] - top2[:, 1]
    confident = margin > 0.02 * ref.abs().max()
    return (a == b).float().mean().item(), (a == b)[confident].float().mean().item()


def _direct(tag, outputs, z32, grads, g32, zbound, gbound):
    """Direct, absolute comparison with the fp32 oracle on the small random-init fixtures (32-64 px, where ResNet's layer4
    sees 8 samples per channel): fixed bounds taken from the measured values, no bf16-model yardstick.  The precision
    claim at BASELINE size (512x512, warm weights, float64 reference, torch autocast as peer) is tests/test_parity_512_gpu.py."""
    zr, gr = rel(outputs, z32), _global_rel(grads, g32)
    print(f"\n[direct {tag}] logits {zr:.3e} (bound {zbound:.1e})  grads {gr:.3e} (bound {gbound:.1e})")
    assert zr <= zbound, (tag, zr)
    assert gr <= gbound, (tag, gr)


CASES = [
    # tag, C, n, h, w, seed, medical, cls_w, dice, focal
    ("nc2_medical", 2, 2, 64, 64, 0, True, [1, 1], False, False),
    ("nc21_cedice", 21, 2, 64, 96, 1, False, [1] * 21, True, False),
    ("nc4_focaldice", 4, 1, 32, 32, 2, False, [1, 15, 1.5, 2], True, True),
]


@pytest.mark.parametrize("tag,C,n,h,w,seed,medical,cw,dice,focal", CASES)
def test_dropin_module_matches_oracle_and_reference_golden(b2u, cuda_device, golden_dir, tag, C, n, h, w, seed, medical, cw, dice, focal):
    dev = cuda_device
    params = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=seed, medical=medical)
    weights = torch.tensor(cw, dtype=torch.float32)
    loss_ref, logits_ref, grads_ref = O.train_step(params, imgs, pngs, weights, C, dice=dice, focal=focal)

    model = b2u.Unet(num_classes=C, pretrained=False, backbone="vgg")
    model.load_state_dict(params)
    model = model.train().to(dev)
    # exactly the calls of utils_fit.py:70-92
    outputs = model(imgs.to(dev))
    labels = O.one_hot(pngs, C).to(dev)
    if focal:
        loss = b2u.Focal_Loss(outputs, pngs.to(dev), weights.to(dev), num_classes=C)
    else:
        loss = b2u.CE_Loss(outputs, pngs.to(dev), weights.to(dev), num_classes=C)
    if dice:
        loss = loss + b2u.Dice_loss(outputs, labels)
    with torch.no_grad():
        fs = b2u.f_score(outputs, labels)
    loss.backward()

    assert outputs.shape == logits_ref.shape and outputs.dtype == torch.float32
    assert rel(outputs, logits_ref) <= 1e-2
    assert abs(loss.item() - loss_ref.item()) <= 1e-2 * abs(loss_ref.item())
    # default-init-scale logits are nearly tied (std ~0.05): the 99.9 % bar is checked on pixels whose fp32 top-2 margin
    # clears the bf16 noise floor; the full-He fixture below checks it on all pixels
    allpix, confident = _argmax_agreement(outputs.detach(), logits_ref)
    assert confident >= 0.999 and allpix >= 0.99
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert _global_rel(grads, grads_ref) <= 1e-2
    worst = max(rel(grads[k], grads_ref[k]) for k in grads_ref if k.endswith("weight"))
    assert worst <= 1.5e-1                                 # single deep-encoder tensors: bf16 noise (SURVEY.md Appendix B: up to 1.3e-1)

    # the same quantities as recorded from the UNMODIFIED reference
    g = np.load(os.path.join(golden_dir, f"unet_vgg_{tag}.npz"))
    assert rel(outputs, torch.from_numpy(g["logits"])) <= 1e-2
    assert abs(loss.item() - float(g["loss"])) <= 1e-2 * abs(float(g["loss"]))
    assert abs(fs.item() - float(g["f_score"])) <= 1e-2
    num = den = 0.0
    for k, p in model.named_parameters():
        flat = p.grad.reshape(-1).cpu()
        s = flat if flat.numel() <= 4096 else flat[torch.linspace(0, flat.numel() - 1, 4096).long()]
        r = torch.from_numpy(g["g:" + k])
        num += (s - r).double().pow(2).sum().item(); den += r.double().pow(2).sum().item()
    assert (num / den) ** 0.5 <= 1.5e-2


def test_harsh_fixture_against_bf16_storage_model(b2u, cuda_device):
    """Full-He weights (gain 1.0): compare with the oracle's bf16-storage model (same rounding points, fp32 math)."""
    dev = cuda_device
    C, n, h, w = 21, 2, 64, 64
    params = O.make_params(C, seed=11, gain=1.0)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=0)
    l32, z32, g32 = O.train_step(params, imgs, pngs, torch.ones(C), C, dice=True)
    lbf, zbf, gbf = O.train_step_bf16_storage(params, imgs, pngs, torch.ones(C), C, dice=True)
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=params, lr=0.0)
    out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    logits = tr.engine.forward(imgs.to(dev), tr.params, save=False)
    assert rel(logits, zbf) <= 8e-3 and rel(logits, z32) <= 1e-2
    assert abs(out[0].item() - lbf.item()) <= 2e-3 * abs(lbf.item())
    # in this regime the network amplifies 1-ulp differences (accumulation order) chaotically: two bf16 computations
    # differ from each other by about as much as each differs from fp32 (2.8e-2 here); scripts/gpu_model_check.py
    # shows 4e-4 .. 7e-4 against the same model on the default-init-scale fixtures
    model_noise = _global_rel(gbf, g32)
    assert _global_rel(tr.grads, gbf) <= model_noise
    assert _global_rel(tr.grads, g32) <= 1.5 * model_noise
    assert (logits.cpu().argmax(1) == z32.argmax(1)).float().mean().item() >= 0.999


def test_trainer_matches_bf16_storage_model_tightly(b2u, cuda_device):
    """On the default-init-scale fixture the CUDA path must agree with the oracle's bf16-storage model (fp32 math,
    rounding only where bf16 tensors are stored) far inside the bf16-vs-fp32 distance: this is the bug detector."""
    dev = cuda_device
    C, n, h, w = 21, 2, 64, 64
    params = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=5)
    lbf, zbf, gbf = O.train_step_bf16_storage(params, imgs, pngs, torch.ones(C), C, dice=True)
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=params, lr=0.0)
    out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert abs(out[0].item() - lbf.item()) <= 1e-4 * abs(lbf.item())
    assert _global_rel(tr.grads, gbf) <= 3e-3
    g1 = {k: v.clone() for k, v in tr.grads.items()}
    tr.train_step(imgs.to(dev), pngs.to(dev))
    assert all(torch.equal(g1[k], tr.grads[k]) for k in g1)          # bitwise reproducible


def test_trainer_step_matches_oracle_adam(b2u, cuda_device):
    """UnetTrainer.train_step == forward + CE + Dice + backward + Adam of the reference loop (train.py:403)."""
    dev = cuda_device
    C, n, h, w = 21, 2, 64, 64
    params = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=5)
    loss_ref, _, grads_ref = O.train_step(params, imgs, pngs, torch.ones(C), C, dice=True)
    ref_p = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    opt = torch.optim.Adam(list(ref_p.values()), lr=1e-4, betas=(0.9, 0.999))
    for k in ref_p:
        ref_p[k].grad = grads_ref[k].clone()
    opt.step()
    tr = b2u.UnetTrainer(num_classes=C, device=dev, lr=1e-4, state_dict=params, dice_loss=True)
    out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert abs(out[0].item() - loss_ref.item()) <= 1e-2 * abs(loss_ref.item())
    assert _global_rel(tr.grads, grads_ref) <= 1e-2
    sd = tr.state_dict()
    # Adam's first step moves every weight by ~lr * sign(g): compare the update direction where |g| is not tiny
    agree = tot = 0
    for k in ref_p:
        d_ref = (ref_p[k].detach() - params[k]).reshape(-1)
        d_got = (sd[k].cpu() - params[k]).reshape(-1)
        big = grads_ref[k].reshape(-1).abs() > 1e-3 * grads_ref[k].abs().max()
        agree += (torch.sign(d_ref[big]) == torch.sign(d_got[big])).sum().item(); tot += int(big.sum())
    assert agree / tot >= 0.97
    # second step runs with re-packed weights and changes the loss
    out2 = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert torch.isfinite(out2).all() and out2[0].item() != out[0].item()


def test_frozen_backbone_skips_encoder_gradients(b2u, cuda_device):
    dev = cuda_device
    C = 21
    params = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=6)
    _, _, grads_ref = O.train_step(params, imgs, pngs, torch.ones(C), C, dice=False)
    model = b2u.Unet(num_classes=C)
    model.load_state_dict(params)
    model = model.to(dev).train()
    model.freeze_backbone()                                  # nets/unet.py:80-86
    loss = b2u.CE_Loss(model(imgs.to(dev)), pngs.to(dev), torch.ones(C, device=dev), num_classes=C)
    loss.backward()
    for k, p in model.named_parameters():
        if k.startswith("vgg."):
            assert p.grad is None
        else:
            assert p.grad is not None
    dec = {k: p.grad for k, p in model.named_parameters() if not k.startswith("vgg.")}
    assert _global_rel(dec, {k: grads_ref[k] for k in dec}) <= 1e-2


def test_eval_forward_is_deterministic_and_repeatable(b2u, cuda_device):
    dev = cuda_device
    model = b2u.Unet(num_classes=21)
    model.load_state_dict(O.make_params(21))
    model = model.to(dev).eval()
    imgs, _ = O.make_inputs(1, 21, 64, 64, seed=9)
    with torch.no_grad():
        a = model(imgs.to(dev)); b = model(imgs.to(dev))
    assert torch.equal(a, b)


@pytest.mark.parametrize("model,C", [("unet_vgg", 21), ("traditional", 4), ("unet_resnet50", 21)])
def test_fused_upsample_equals_separate_pass(b2u, cuda_device, monkeypatch, model, C):
    """nets/unet.py:16-18 in one kernel: the decoder conv that interpolates its low-resolution source itself
    (EngineBase.fuse_upsample: 1 = the stages where it pays, the default; patched to 2 = every stage) gives BIT-identical
    logits, loss and gradients to the separate b2u_upsample2x_fwd pass (patched to 0 = no stage); a fused stage needs no
    upsample launch, and in inference it allocates no up-sampled tensor."""
    from unet_pytorch_b200._engine_base import EngineBase
    dev = cuda_device
    imgs, pngs = O.make_inputs(2, C, 96, 64, seed=5)
    runs = {}
    for fuse, rule in ((2, lambda self, cout_p: True), (1, None), (0, lambda self, cout_p: False)):
        with monkeypatch.context() as m:
            if rule is not None:
                m.setattr(EngineBase, "fuse_upsample", rule)
            tr = b2u.UnetTrainer(model=model, num_classes=C, device=dev, lr=0.0) if model != "unet_vgg" else \
                b2u.UnetTrainer(num_classes=C, device=dev, lr=0.0, state_dict=O.make_params(C, seed=11))
            # inference first, on the initial state (a training step of the BatchNorm nets moves the running statistics by the
            # summation order of the per-tile sums, which differs between the two kernels' tilings)
            logits = tr.engine.forward(imgs.to(dev), tr.tensors, save=False, training=False).clone()
            b2u.ops.lib().b2u_reset_launch_count()
            out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
            torch.cuda.synchronize()
            launches = b2u.ops.lib().b2u_launch_count()
            runs[fuse] = (out, {k: v.clone() for k, v in tr.grads.items()}, logits, launches)
            if fuse == 2:
                tr.engine.release()
                tr.engine.forward(imgs.to(dev), tr.tensors, save=False, training=False)
                lazy = getattr(tr.engine, "_lazy_up", None)       # GraphEngine: the up-sampled tensors read by decoder convs
                ups = [k for k in tr.engine._bufs if (k in lazy if lazy is not None else re.fullmatch(r"up\d+", k))]
                assert not ups, "inference must not materialise the up-sampled tensors"
    for fuse in (2, 1):
        assert torch.equal(runs[fuse][2], runs[0][2])            # inference logits: bit-identical for every family
        if model == "traditional":
            # BatchNorm statistics come from the conv epilogue's per-tile sums; the two kernels tile the image differently, so
            # mean / invstd differ in their last fp32 bits and a few bf16 roundings downstream flip
            assert torch.allclose(runs[fuse][0], runs[0][0], rtol=1e-4, atol=1e-6)
            assert _global_rel(runs[fuse][1], {k: v.cpu() for k, v in runs[0][1].items()}) <= 1e-2
        else:
            assert torch.equal(runs[fuse][0], runs[0][0])
            for k in runs[0][1]:
                assert torch.equal(runs[fuse][1][k], runs[0][1][k]), k
    n_dec = 3 if model == "traditional" else 4
    wide = {"unet_vgg": 3, "traditional": 1, "unet_resnet50": 3}[model]      # stages with >= 128 output channels
    assert runs[0][3] - runs[2][3] == n_dec          # one launch less per fused decoder stage
    assert runs[0][3] - runs[1][3] == wide


def test_relu_bit_masks_and_dgrad_bias_sums_change_nothing(b2u, cuda_device, monkeypatch):
    """Three round-2 traffic savers of the plain conv + ReLU nets -- ReLU backward from bit masks (UNetEngine.relu_bit_masks),
    bias gradients from the producing data gradient's column sums (UNetEngine.bias_from_dgrad), weight gradients on a second
    stream (single-stream while ops.timing_active()) -- against the straightforward order: the loss and the data path are
    bit-identical, bias gradients agree to fp32 summation order."""
    from unet_pytorch_b200.engine import UNetEngine
    dev, C = cuda_device, 21
    imgs, pngs = O.make_inputs(2, C, 96, 64, seed=8)
    runs = []
    for on in (True, False):
        with monkeypatch.context() as m:
            if not on:
                m.setattr(UNetEngine, "relu_bit_masks", lambda self, save: False)
                m.setattr(UNetEngine, "bias_from_dgrad", lambda self, c: False)
                m.setattr(b2u.ops, "timing_active", lambda: True)
            tr = b2u.UnetTrainer(num_classes=C, device=dev, lr=0.0, state_dict=O.make_params(C, seed=11))
            out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
            torch.cuda.synchronize()
            runs.append((out, {k: v.clone() for k, v in tr.grads.items()}))
    assert torch.equal(runs[0][0], runs[1][0])
    for k, g in runs[1][1].items():
        if k.endswith(".weight"):
            assert torch.equal(runs[0][1][k], g), k
        else:
            assert torch.allclose(runs[0][1][k], g, rtol=1e-4, atol=1e-6 * g.abs().max().item() + 1e-12), k


def test_full_size_step_properties(b2u, cuda_device):
    """BASELINE config-2 tile sizes (512x512, 21 classes) at batch 2: parity against the same restatement executed
    by torch on the GPU in fp32 (TF32 off) -- the CPU oracle needs minutes at this size -- plus finite loss."""
    dev = cuda_device
    C, n = 21, 2
    params = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(n, C, 512, 512, seed=3)
    pd = {k: v.to(dev) for k, v in params.items()}
    loss_ref, logits_ref, grads_ref = O.train_step(pd, imgs.to(dev), pngs.to(dev), torch.ones(C, device=dev), C, dice=True)
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=params, lr=0.0)
    out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert abs(out[0].item() - loss_ref.item()) <= 1e-2 * abs(loss_ref.item())
    logits = tr.engine.forward(imgs.to(dev), tr.params, save=False)
    assert rel(logits, logits_ref) <= 1e-2
    gr = {k: v.cpu() for k, v in grads_ref.items()}
    assert _global_rel(tr.grads, gr) <= 1e-2


# ------------------------------------------------------------------------------------------------ TraditionalUnet
# conv -> BatchNorm(train) -> ReLU nets amplify bf16 rounding: rounding only the *stored* tensors of the fp32 oracle
# (oracle.trad_train_step(bf16_storage=True)) already moves logits by ~5e-2 and gradients by 2e-1 .. 3e-1 on these
# fixtures, whatever the input statistics (BatchNorm subtracts a mean that dominates the bf16 ulp of z and of dy).
# The CUDA path is therefore held to (a) tight per-kernel BatchNorm tests (tests/test_kernels_gpu.py), (b) the
# bf16-storage model as yardstick here, (c) exact agreement of everything that is not rounding-limited: running
# statistics, loss value, eval-mode logits.
TRAD_BOUNDS = {"nc4_focaldice": (7e-2, 3e-1), "nc21_cedice": (7e-2, 3.5e-1)}      # (logits, gradients) vs the fp32 oracle, absolute
TRAD_CASES = [("nc4_focaldice", 4, 2, 64, 64, 3, [1, 15, 1.5, 2], True, True), ("nc21_cedice", 21, 2, 32, 64, 4, [1] * 21, True, False)]


@pytest.mark.parametrize("tag,C,n,h,w,seed,cw,dice,focal", TRAD_CASES)
def test_traditional_unet_dropin(b2u, cuda_device, golden_dir, tag, C, n, h, w, seed, cw, dice, focal):
    dev = cuda_device
    sd = O.make_trad_params(C, seed=11)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
    weights = torch.tensor(cw, dtype=torch.float32)
    l32, z32, g32, s32 = O.trad_train_step(sd, imgs, pngs, weights, C, dice=dice, focal=focal)
    lbf, zbf, gbf, sbf = O.trad_train_step(sd, imgs, pngs, weights, C, dice=dice, focal=focal, bf16_storage=True)
    model = b2u.TraditionalUnet(in_channels=3, num_classes=C)
    model.load_state_dict(sd)
    model = model.train().to(dev)
    outputs = model(imgs.to(dev))
    labels = O.one_hot(pngs, C).to(dev)
    loss = (b2u.Focal_Loss if focal else b2u.CE_Loss)(outputs, pngs.to(dev), weights.to(dev), num_classes=C)
    if dice:
        loss = loss + b2u.Dice_loss(outputs, labels)
    loss.backward()
    noise_z, noise_g = rel(zbf, z32), _global_rel(gbf, g32)
    assert rel(outputs, z32) <= 1.5 * noise_z and rel(outputs, zbf) <= noise_z
    assert abs(loss.item() - l32.item()) <= 2e-2 * abs(l32.item())
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert all(v is not None and torch.isfinite(v).all() for v in grads.values())
    assert _global_rel(grads, g32) <= 1.5 * noise_g and _global_rel(grads, gbf) <= 1.2 * noise_g
    _direct("traditional " + tag, outputs, z32, grads, g32, *TRAD_BOUNDS[tag])
    # BatchNorm buffers after one training step (fp32 statistics of bf16 pre-activations)
    for name, b in model.named_buffers():
        want = s32[name]
        if name.endswith("num_batches_tracked"):
            assert int(b.item()) == int(want.item()) == 1
        else:
            assert rel(b, want) <= 2e-2, name
    # the same quantities recorded from the UNMODIFIED reference
    g = np.load(os.path.join(golden_dir, f"traditional_{tag}.npz"))
    assert rel(outputs, torch.from_numpy(g["logits"])) <= 1.5 * noise_z
    assert abs(loss.item() - float(g["loss"])) <= 2e-2 * abs(float(g["loss"]))
    # eval mode uses the running statistics: no batch-mean cancellation, so this is a plain bf16 comparison
    model.eval()
    with torch.no_grad():
        ev = model(imgs.to(dev))
    sd_after = dict(sd); sd_after.update({k: v.cpu() for k, v in model.named_buffers()})
    with torch.no_grad():
        ev_ref, _ = O.trad_forward(sd_after, imgs, training=False)
    assert rel(ev, ev_ref) <= 2e-2


def test_traditional_trainer_step(b2u, cuda_device):
    """UnetTrainer(model='traditional'): fused step with BatchNorm, reproducible, loss decreases over a few steps."""
    dev = cuda_device
    C = 4
    sd = O.make_trad_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=3)
    lbf, zbf, gbf, _ = O.trad_train_step(sd, imgs, pngs, torch.ones(C), C, dice=True, bf16_storage=True)
    l32, z32, g32, _ = O.trad_train_step(sd, imgs, pngs, torch.ones(C), C, dice=True)
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0, model="traditional")
    out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert abs(out[0].item() - l32.item()) <= 2e-2 * abs(l32.item())
    assert _global_rel(tr.grads, g32) <= 1.5 * _global_rel(gbf, g32)
    g1 = {k: v.clone() for k, v in tr.grads.items()}
    tr2 = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0, model="traditional")
    tr2.train_step(imgs.to(dev), pngs.to(dev))
    assert all(torch.equal(g1[k], tr2.grads[k]) for k in g1)
    tr3 = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=1e-3, model="traditional")
    losses = [tr3.train_step(imgs.to(dev), pngs.to(dev))[0].item() for _ in range(8)]
    assert losses[-1] < losses[0]


# ------------------------------------------------------------------------------------------------ Unet-ResNet50
def test_resnet50_unet_dropin(b2u, cuda_device, golden_dir):
    """BASELINE configs[2]: Unet(backbone='resnet50'), train-mode BatchNorm, CE + Dice.  Same yardstick policy as
    TraditionalUnet (BatchNorm nets amplify bf16 storage rounding in the gradients); forward quantities are tight."""
    dev = cuda_device
    C, n, h, w, seed = 21, 2, 64, 64, 7
    sd = O.make_resnet_unet_params(C, seed=11)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
    weights = torch.ones(C)
    l32, z32, g32, s32 = O.resnet_unet_train_step(sd, imgs, pngs, weights, C, dice=True)
    lbf, zbf, gbf, sbf = O.resnet_unet_train_step(sd, imgs, pngs, weights, C, dice=True, bf16_storage=True)
    model = b2u.Unet(num_classes=C, pretrained=False, backbone="resnet50")
    model.load_state_dict(sd)
    model = model.train().to(dev)
    outputs = model(imgs.to(dev))
    loss = b2u.CE_Loss(outputs, pngs.to(dev), weights.to(dev), num_classes=C) + b2u.Dice_loss(outputs, O.one_hot(pngs, C).to(dev))
    loss.backward()
    noise_z, noise_g = rel(zbf, z32), _global_rel(gbf, g32)
    assert outputs.shape == z32.shape
    assert rel(outputs, z32) <= max(1.5 * noise_z, 1e-2)
    assert abs(loss.item() - l32.item()) <= 1e-2 * abs(l32.item())
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert all(v is not None and torch.isfinite(v).all() for v in grads.values())
    assert _global_rel(grads, g32) <= 1.5 * noise_g and _global_rel(grads, gbf) <= 1.2 * noise_g
    _direct("unet_resnet50 nc21", outputs, z32, grads, g32, 1e-2, 2e-1)
    # decoder-side tensors are not behind a BatchNorm backward: plain bf16 accuracy
    for k in ("final.weight", "final.bias", "up_conv.3.weight", "up_conv.1.weight", "up_concat1.conv2.weight"):
        assert rel(grads[k], g32[k]) <= 2e-2, k
    for name, b in model.named_buffers():
        # statistics of bf16 activations ~50 layers deep: the per-channel means are small against the activations' spread
        # (layer4 sees 2x2 maps: 8 samples per channel); each buffer is judged against the bf16-storage model's own
        # distance from fp32 for that buffer
        if name.endswith("running_mean"):
            assert rel(b, s32[name]) <= max(6e-2, 1.5 * rel(sbf[name], s32[name])), name
        elif name.endswith("running_var"):
            assert rel(b, s32[name]) <= max(2e-2, 1.5 * rel(sbf[name], s32[name])), name
    g = np.load(os.path.join(golden_dir, "unet_resnet50_nc21_cedice.npz"))
    assert rel(outputs, torch.from_numpy(g["logits"])) <= max(1.5 * noise_z, 1e-2)
    assert abs(loss.item() - float(g["loss"])) <= 1e-2 * abs(float(g["loss"]))
    model.eval()
    with torch.no_grad():
        ev = model(imgs.to(dev))
    sd_after = dict(sd); sd_after.update({k: v.cpu() for k, v in model.named_buffers()})
    with torch.no_grad():
        ev_ref, _ = O.resnet_unet_forward(sd_after, imgs, training=False)
    assert rel(ev, ev_ref) <= 2e-2


def test_resnet50_frozen_backbone_and_trainer(b2u, cuda_device):
    dev = cuda_device
    C = 4
    sd = O.make_resnet_unet_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=8)
    l32, z32, g32, _ = O.resnet_unet_train_step(sd, imgs, pngs, torch.ones(C), C, dice=True)
    lbf, zbf, gbf, _ = O.resnet_unet_train_step(sd, imgs, pngs, torch.ones(C), C, dice=True, bf16_storage=True)
    model = b2u.Unet(num_classes=C, backbone="resnet50")
    model.load_state_dict(sd)
    model = model.to(dev).train()
    model.freeze_backbone()
    out = model(imgs.to(dev))
    loss = b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C) + b2u.Dice_loss(out, O.one_hot(pngs, C).to(dev))
    loss.backward()
    dec = {k: p.grad for k, p in model.named_parameters() if not k.startswith("resnet.")}
    assert all(p.grad is None for k, p in model.named_parameters() if k.startswith("resnet."))
    assert _global_rel(dec, {k: g32[k] for k in dec}) <= 2e-2          # decoder gradients do not cross a BatchNorm backward
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0, model="unet_resnet50")
    o = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert abs(o[0].item() - l32.item()) <= 1e-2 * abs(l32.item())
    assert _global_rel(tr.grads, g32) <= 1.5 * _global_rel(gbf, g32)
    tr3 = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=1e-3, model="unet_resnet50")
    losses = [tr3.train_step(imgs.to(dev), pngs.to(dev))[0].item() for _ in range(6)]
    assert losses[-1] < losses[0]


# ------------------------------------------------------------------------------------------------ UltraLightweightUnet family
ULU_CASES = [("ultralight", "UltraLightweightUnet", "nc21_cedice"), ("ultralight_large", "UltraLightweightUnet_large", "nc4_focaldice"),
             ("ultralight_large_optimized", "UltraLightweightUnet_large_optimized", "nc21_cedice")]


ULU_BOUNDS = {"ultralight": (3e-2, 1.2e-1), "ultralight_large": (5e-2, 2e-1), "ultralight_large_optimized": (8e-2, 3e-1)}   # (logits, gradients), absolute


@pytest.mark.parametrize("variant,cls,tag", ULU_CASES)
def test_ultralight_unet_dropin(b2u, cuda_device, golden_dir, variant, cls, tag):
    """nets/UltraLightweightUnet*.py drop-ins against the reference's golden forward/backward (train-mode BatchNorm,
    depthwise-separable blocks, SE, the reference's own Dropout2d mask replayed).  Every conv sits in front of a BatchNorm,
    so gradients are judged against the bf16-storage model's own distance from fp32 (same policy as TraditionalUnet)."""
    import importlib
    dev = cuda_device
    g = np.load(os.path.join(golden_dir, f"{variant}_{tag}.npz"))
    C, n, h, w, seed, dice, focal = [int(v) for v in g["meta"]]
    sd = O.make_ulu_params(C, variant, seed=11)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
    weights = torch.from_numpy(g["cls_w"])
    mask = torch.from_numpy(g["drop_mask"]) if "drop_mask" in g.files else None
    l32, z32, g32, s32 = O.ulu_train_step(sd, imgs, pngs, weights, C, variant, dice=bool(dice), focal=bool(focal), drop_mask=mask)
    lbf, zbf, gbf, sbf = O.ulu_train_step(sd, imgs, pngs, weights, C, variant, dice=bool(dice), focal=bool(focal), drop_mask=mask,
                                          bf16_storage=True)
    Net = getattr(importlib.import_module(f"unet_pytorch_b200.nets.{cls}"), cls)
    model = Net(num_classes=C)
    assert list(model.state_dict().keys()) == list(sd.keys())
    model.load_state_dict(sd)
    model = model.train().to(dev)
    model._engine_for(dev).dropout_override = mask
    outputs = model(imgs.to(dev))
    lossf = b2u.Focal_Loss if focal else b2u.CE_Loss
    loss = lossf(outputs, pngs.to(dev), weights.to(dev), num_classes=C)
    if dice:
        loss = loss + b2u.Dice_loss(outputs, O.one_hot(pngs, C).to(dev))
    loss.backward()
    noise_z, noise_g = rel(zbf, z32), _global_rel(gbf, g32)
    ref = torch.from_numpy(g["logits"])
    assert outputs.shape == ref.shape
    assert rel(outputs, ref) <= max(1.5 * noise_z, 1e-2)
    assert rel(outputs, zbf) <= max(noise_z, 5e-3)
    assert abs(loss.item() - float(g["loss"])) <= 1e-2 * abs(float(g["loss"]))
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert all(v is not None and torch.isfinite(v).all() for v in grads.values())
    live = {k: v for k, v in grads.items() if not (k.endswith(".conv.0.bias") or k.endswith("wise.bias"))}    # zero-gradient biases
    assert _global_rel(live, {k: g32[k] for k in live}) <= 1.5 * noise_g
    assert _global_rel(live, {k: gbf[k] for k in live}) <= 1.2 * noise_g
    _direct(f"{variant} {tag}", outputs, z32, live, {k: g32[k] for k in live}, *ULU_BOUNDS[variant])
    for k in ("final.weight", "final.bias"):      # no BatchNorm backward in between: bounded by the head input's forward noise
        assert rel(grads[k], g32[k]) <= max(2e-2, 2 * noise_z), k
    for name, b in model.named_buffers():
        if name.endswith("running_mean"):
            assert rel(b, s32[name]) <= max(2e-2, 2 * noise_z), name
        elif name.endswith("running_var"):
            assert rel(b, s32[name]) <= max(2e-2, 2 * noise_z), name
        elif name.endswith("num_batches_tracked"):
            assert int(b) == 1
    model.eval()
    with torch.no_grad():
        ev = model(imgs.to(dev))
    sd_after = dict(sd); sd_after.update({k: v.cpu() for k, v in model.named_buffers()})
    with torch.no_grad():
        ev_ref, _ = O.ulu_forward(sd_after, imgs, variant, training=False)
    assert rel(ev, ev_ref) <= max(3e-2, 2 * noise_z)


def test_ultralight_trainer_and_dropout(b2u, cuda_device):
    dev = cuda_device
    C, variant = 4, "ultralight_large_optimized"
    sd = O.make_ulu_params(C, variant, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=12)
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=1e-3, model=variant)
    losses = [tr.train_step(imgs.to(dev), pngs.to(dev))[0].item() for _ in range(8)]
    assert all(np.isfinite(losses)) and min(losses[-3:]) < losses[0]
    # Dropout2d: training draws a fresh per-(sample, channel) mask, eval is deterministic
    from unet_pytorch_b200.nets.UltraLightweightUnet_large import UltraLightweightUnet_large
    model = UltraLightweightUnet_large(num_classes=C)
    model.load_state_dict(O.make_ulu_params(C, "ultralight_large", seed=11))
    model = model.to(dev).train()
    with torch.no_grad():
        a, b = model(imgs.to(dev)), model(imgs.to(dev))
    assert not torch.equal(a, b)
    model.eval()
    with torch.no_grad():
        a, b = model(imgs.to(dev)), model(imgs.to(dev))
    assert torch.equal(a, b)


def test_light_block_subnetwork_at_stated_tolerance(b2u, cuda_device):
    """The full UltraLightweightUnet stacks 18 BatchNorms, which amplify bf16 storage rounding beyond the 1e-2 the VGG path
    meets.  A two-level sub-network with every op of the family (padded 3/44/88-channel 1x1 convs, BN, depthwise, SE, pool,
    upsample + virtual concat, head) is shallow enough to be checked directly against fp32 autograd: the bf16-storage model of
    this sub-network sits at 8.3e-3 (logits) / 8.4e-3 (all gradients) / 1.9e-2 (worst tensor); bounds are 1.5e-2 / 2e-2 / 5e-2."""
    from unet_pytorch_b200.graph import GraphEngine, light_conv_block_ops
    dev = cuda_device
    C, c1_, c2_ = 5, 44, 88
    P, convs = [dict(op="input", out="x", c=3)], {}
    e1 = light_conv_block_ops(P, convs, "enc1", "x", 3, c1_, 16)
    P.append(dict(op="se", out="se1.out", x=e1, se="se1", c=c1_, r=11))
    P.append(dict(op="pool2", out="p2", x="se1.out"))
    e2 = light_conv_block_ops(P, convs, "enc2", "p2", c1_, c2_, 16)
    P.append(dict(op="up", out="up1", x=e2))
    d1 = light_conv_block_ops(P, convs, "dec1", "up1", c2_, c1_, 16, x1="se1.out", c1=c1_)
    P.append(dict(op="head", out="logits", x=d1, w="final.weight", bias="final.bias", cin=c1_))
    eng = GraphEngine(P, convs, C, device=dev)
    sd = {}
    for k, (name, shape) in enumerate(eng.param_shapes().items()):
        g = torch.Generator().manual_seed(900 + k)
        is_bn = ".conv.1." in name or ".conv.4." in name
        if name.endswith("depthwise.weight"):
            sd[name] = (1.0 / 3.0) * (1.0 + 0.5 * torch.randn(shape, generator=g))
        elif len(shape) == 4:
            sd[name] = torch.randn(shape, generator=g) * ((0.5 if name == "final.weight" else 1.0) * (2.0 / shape[1]) ** 0.5)
        elif len(shape) == 2:
            sd[name] = torch.randn(shape, generator=g) * (1.0 / shape[1]) ** 0.5
        elif is_bn:
            sd[name] = (1.0 if name.endswith("weight") else 0.5) + 0.05 * torch.randn(shape, generator=g)
        else:
            sd[name] = 0.05 * torch.randn(shape, generator=g)
    for name, shape in eng.buffer_shapes().items():
        sd[name] = torch.ones(shape) if name.endswith("var") else (torch.zeros(shape) if shape else torch.tensor(0))
    imgs, pngs = O.make_inputs(4, C, 64, 64, seed=21)
    imgs = imgs - 0.5

    def ref_forward(p):
        stats = {k: v.clone() for k, v in sd.items() if "running_" in k or "num_batches" in k}
        a = O._ulu_se(p, "se1", O._ulu_block(p, stats, "enc1", imgs, True, False), False)
        b_ = O._ulu_block(p, stats, "enc2", F.max_pool2d(a, 2, 2), True, False)
        up = F.interpolate(b_, scale_factor=2, mode="bilinear", align_corners=True)
        d = O._ulu_block(p, stats, "dec1", torch.cat([up, a], 1), True, False)
        return F.conv2d(d, p["final.weight"], p["final.bias"])

    names = list(eng.param_shapes().keys())
    p = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
    z_ref = ref_forward(p)
    loss_ref = O.ce_loss(z_ref, pngs, torch.ones(C), C) + O.dice_loss(z_ref, O.one_hot(pngs, C))
    g_ref = dict(zip(names, torch.autograd.grad(loss_ref, [p[k] for k in names])))
    params = {k: v.to(dev).contiguous() for k, v in sd.items()}
    logits = eng.forward(imgs.to(dev), params, save=True, training=True)
    assert rel(logits, z_ref.detach()) <= 1.5e-2
    lg = logits.detach().clone().requires_grad_(True)
    loss = b2u.CE_Loss(lg, pngs.to(dev), torch.ones(C, device=dev), num_classes=C) + b2u.Dice_loss(lg, O.one_hot(pngs, C).to(dev))
    loss.backward()
    grads = {k: torch.empty_like(params[k]) for k in names}
    eng.backward(lg.grad, params, grads)
    live = [k for k in names if not (k.endswith(".conv.0.bias") or k.endswith("wise.bias"))]
    assert _global_rel({k: grads[k] for k in live}, {k: g_ref[k] for k in live}) <= 2e-2
    for k in live:
        assert rel(grads[k], g_ref[k]) <= 5e-2, k


def test_ultralight_trained_checkpoint_eval(b2u, cuda_device, golden_dir):
    """The reference's own trained checkpoint (Submit_result/model.pth, UltraLightweightUnet_large_optimized, 4 classes) in
    eval mode: trained BatchNorm statistics keep bf16 rounding from being amplified, so the drop-in is held to 1.5e-2 of
    the reference's fp32 logits (the bf16-storage model itself sits at 1.1e-2) and 99.5 % identical class decisions."""
    from unet_pytorch_b200.nets.UltraLightweightUnet_large_optimized import UltraLightweightUnet_large_optimized
    g = np.load(os.path.join(golden_dir, "ultralight_large_optimized_checkpoint_eval.npz"))
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd:")}
    C, n, h, w, seed = [int(v) for v in g["meta"]]
    imgs, _ = O.make_inputs(n, C, h, w, seed=seed)
    ref = torch.from_numpy(g["logits"])
    model = UltraLightweightUnet_large_optimized(num_classes=C)
    model.load_state_dict(sd)
    model = model.to(cuda_device).eval()
    with torch.no_grad():
        out = model(imgs.to(cuda_device))
        again = model(imgs.to(cuda_device))
    assert torch.equal(out, again)
    assert rel(out, ref) <= 1.5e-2
    agree_all, agree_confident = _argmax_agreement(out, ref)
    assert agree_all >= 0.995 and agree_confident >= 0.999


# ------------------------------------------------------------------------------------------------ LightweightUnet
@pytest.mark.parametrize("tag", ["nc4_focaldice", "nc21_cedice"])
def test_lightweight_unet_dropin(b2u, cuda_device, golden_dir, tag):
    """nets/LightWeightUnet.py drop-in against the reference's golden forward/backward: half-resolution logits, the
    losses' bilinear resize, SE residual blocks, the reference's ten Dropout2d draws replayed.  34 BatchNorms: gradients are
    judged against the bf16-storage model's own distance from fp32 (same policy as the other BatchNorm nets)."""
    dev = cuda_device
    g = np.load(os.path.join(golden_dir, f"lightweight_{tag}.npz"))
    C, n, h, w, seed, dice, focal = [int(v) for v in g["meta"]]
    sd = O.make_lw_params(C, seed=11)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
    weights = torch.from_numpy(g["cls_w"])
    masks = {k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("drop:")}
    l32, z32, g32, s32 = O.lw_train_step(sd, imgs, pngs, weights, C, dice=bool(dice), focal=bool(focal), drop_masks=masks)
    lbf, zbf, gbf, sbf = O.lw_train_step(sd, imgs, pngs, weights, C, dice=bool(dice), focal=bool(focal), drop_masks=masks,
                                         bf16_storage=True)
    model = b2u.LightweightUnet(num_classes=C)
    assert list(model.state_dict().keys()) == list(sd.keys())
    model.load_state_dict(sd)
    model = model.train().to(dev)
    model._engine_for(dev).dropout_override = masks
    outputs = model(imgs.to(dev))
    assert tuple(outputs.shape) == (n, C, h // 2, w // 2)
    lossf = b2u.Focal_Loss if focal else b2u.CE_Loss
    loss = lossf(outputs, pngs.to(dev), weights.to(dev), num_classes=C)
    if dice:
        loss = loss + b2u.Dice_loss(outputs, O.one_hot(pngs, C).to(dev))
    loss.backward()
    noise_z, noise_g = rel(zbf, z32), _global_rel(gbf, g32)
    ref = torch.from_numpy(g["logits"])
    assert rel(outputs, ref) <= max(1.5 * noise_z, 1e-2)
    assert rel(outputs, zbf) <= max(noise_z, 5e-3)
    assert abs(loss.item() - float(g["loss"])) <= 1e-2 * abs(float(g["loss"]))
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert all(v is not None and torch.isfinite(v).all() for v in grads.values())

    def pre_bn_bias(k):
        base = k.rsplit(".", 1)[0]
        return k.endswith(".bias") and (base.endswith(".conv.0") or base.endswith(".conv1") or base.endswith(".conv2"))
    live = {k: v for k, v in grads.items() if not pre_bn_bias(k)}
    assert all(grads[k].abs().max().item() == 0 for k in grads if pre_bn_bias(k))      # exact zero by the BN identity
    assert _global_rel(live, {k: g32[k] for k in live}) <= 1.5 * noise_g
    assert _global_rel(live, {k: gbf[k] for k in live}) <= 1.2 * noise_g
    _direct("lightweight " + tag, outputs, z32, live, {k: g32[k] for k in live}, 4e-2, 2.2e-1)
    for k in ("final_conv.3.weight", "final_conv.3.bias"):
        assert rel(grads[k], g32[k]) <= max(2e-2, 2 * noise_z), k
    model.eval()
    with torch.no_grad():
        ev = model(imgs.to(dev))
    sd_after = dict(sd); sd_after.update({k: v.cpu() for k, v in model.named_buffers()})
    with torch.no_grad():
        ev_ref, _ = O.lw_forward(sd_after, imgs, training=False)
    assert rel(ev, ev_ref) <= max(3e-2, 2 * noise_z)


def test_lightweight_trainer_and_freeze(b2u, cuda_device):
    dev = cuda_device
    C = 4
    sd = O.make_lw_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=14)
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=1e-3, model="lightweight")
    losses = [tr.train_step(imgs.to(dev), pngs.to(dev))[0].item() for _ in range(8)]
    assert all(np.isfinite(losses)) and min(losses[-3:]) < losses[0]
    ev = tr.eval_step(imgs.to(dev), pngs.to(dev))
    assert torch.isfinite(ev).all()
    model = b2u.LightweightUnet(num_classes=C)
    model.load_state_dict(sd)
    model = model.to(dev).train()
    model.freeze_backbone()
    out = model(imgs.to(dev))
    b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C).backward()
    assert all(p.grad is None for k, p in model.named_parameters() if k.startswith("backbone."))
    assert all(p.grad is not None for k, p in model.named_parameters() if not k.startswith("backbone."))
    with pytest.raises(ValueError):
        b2u.LightweightUnet(num_classes=C, backbone="vgg")


def test_predictor_class_against_reference(b2u, cuda_device, golden_dir):
    """unet.py::Unet drop-in (detect_image / get_miou_png / get_FPS) against the mask the reference's own predictor class
    produced for the same image and weights.  Agreement is scored on pixels whose reference top-2 probability margin
    exceeds 0.02 (77 % of the image; >= 99.9 % must match) and overall (>= 97 %)."""
    from PIL import Image
    from unet_pytorch_b200.unet import Unet as Predictor
    g = np.load(os.path.join(golden_dir, "predictor_vgg_nc21.npz"))
    C, ih, iw = [int(v) for v in g["meta"]]
    pred = Predictor(state_dict=O.make_predictor_params(C, seed=11), num_classes=C, backbone="vgg", input_shape=[ih, iw], mix_type=1)
    image = Image.fromarray(g["image"])
    mask = np.array(pred.get_miou_png(image))
    assert mask.shape == g["mask"].shape and mask.dtype == np.uint8
    agree = mask == g["mask"]
    margin = g["margin"].astype(np.float32)
    assert agree[margin > 0.02].mean() >= 0.999
    assert agree.mean() >= 0.97
    seg = np.array(pred.detect_image(image))
    assert seg.shape == g["seg"].shape
    assert (seg == g["seg"]).all(axis=-1)[margin > 0.02].mean() >= 0.999
    # batched evaluation without the PNG round trip: device-resident masks folded into one confusion matrix
    gt = g["mask"].copy(); gt[:10] = 255                               # some ignored pixels
    hist, ious, recall, precision = pred.get_miou([image, image], [gt, Image.fromarray(gt)])
    ref_hist = 2 * O.fast_hist(gt.reshape(-1), mask.reshape(-1), C)
    assert np.array_equal(hist, ref_hist) and hist.sum() == 2 * (gt != 255).sum()
    assert np.allclose(ious, O.per_class_iu(ref_hist))
    pred.mix_type = 0
    assert pred.detect_image(image).size == image.size
    assert pred.get_FPS(image, 3) > 0
    with pytest.raises(RuntimeError):
        Predictor(state_dict=O.make_params(C, seed=11), num_classes=C, cuda=False)


def test_device_input_pipeline_uint8(b2u, cuda_device):
    """Raw uint8 NHWC images + uint8 label maps staged from pinned host memory give the same step as the fp32 NCHW / int64
    batches the reference's dataloader would have produced from them on the host (utils/dataloader.py:41-43)."""
    from unet_pytorch_b200 import ops
    dev = cuda_device
    C = 4
    sd = O.make_params(C, seed=11)
    g = torch.Generator().manual_seed(3)
    raw = torch.randint(0, 256, (2, 64, 96, 3), generator=g, dtype=torch.uint8)
    lab = torch.randint(0, C + 1, (2, 64, 96), generator=g).to(torch.uint8)
    imgs = (raw.float() / 255.0).permute(0, 3, 1, 2).contiguous()           # preprocess_input + transpose on the host
    conv = ops.u8hwc_to_nchw_f32(raw.to(dev))
    assert torch.allclose(conv.cpu(), imgs, rtol=0, atol=1e-7)
    assert torch.equal(ops.u8_to_i64(lab.to(dev)).cpu(), lab.long())
    a = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0)
    b = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0)
    ra = a.train_step(imgs.to(dev), lab.long().to(dev)).cpu()
    b.stage(raw.pin_memory(), lab.pin_memory())
    rb = b.train_step().cpu()
    assert torch.allclose(ra, rb, rtol=2e-3, atol=1e-5)
    # x * (1/255) on the device vs round(x * 255) / 255 on the host differ by one fp32 ulp, which the two-term image split now
    # carries into the network; the step amplifies it like any other 1-ulp difference
    assert _global_rel(b.grads, {k: v.cpu() for k, v in a.grads.items()}) <= 1e-2


def test_reference_training_wrappers(b2u, cuda_device):
    """The wrappers the reference's train.py puts around the model keep working with the drop-in: autocast + GradScaler
    (utils_fit.py:65-94), DistributedDataParallel(find_unused_parameters=True) (train.py:346) -- one rank here -- and a
    torch optimizer over model.parameters() (train.py:402-405)."""
    import torch.distributed as dist
    dev = cuda_device
    C = 4
    sd = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=5)
    l32, _, g32 = O.train_step(sd, imgs, pngs, torch.ones(C), C, dice=True)
    model = b2u.Unet(num_classes=C, backbone="vgg")
    model.load_state_dict(sd)
    model = model.to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    scaler = torch.amp.GradScaler("cuda")
    with torch.autocast("cuda", dtype=torch.float16):
        out = model(imgs.to(dev))
        loss = b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C) + b2u.Dice_loss(out, O.one_hot(pngs, C).to(dev))
    scaler.scale(loss).backward()
    scaler.unscale_(opt)
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert abs(loss.item() - l32.item()) <= 1e-2 * abs(l32.item())
    assert _global_rel(grads, g32) <= 1e-2
    scaler.step(opt); scaler.update()
    created = False
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1"); os.environ.setdefault("MASTER_PORT", "29577")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
        created = True
    try:
        m2 = b2u.Unet(num_classes=C, backbone="vgg")
        m2.load_state_dict(sd)
        ddp = torch.nn.parallel.DistributedDataParallel(m2.to(dev).train(), device_ids=[dev.index or 0], find_unused_parameters=True)
        out = ddp(imgs.to(dev))
        loss = b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C) + b2u.Dice_loss(out, O.one_hot(pngs, C).to(dev))
        loss.backward()
        assert _global_rel({k: p.grad for k, p in m2.named_parameters()}, g32) <= 1e-2
    finally:
        if created:
            dist.destroy_process_group()


def test_dataparallel_two_gpus(b2u, cuda_device):
    """train.py:348 wraps the model in nn.DataParallel when it is not running distributed: replicas on two GPUs (one engine
    per device, shared through the module's engine table) must give the single-GPU result on the concatenated batch."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    dev = cuda_device
    C = 4
    sd = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(4, C, 64, 64, seed=6)
    l32, z32, g32 = O.train_step(sd, imgs, pngs, torch.ones(C), C, dice=True)
    model = b2u.Unet(num_classes=C, backbone="vgg")
    model.load_state_dict(sd)
    dp = torch.nn.DataParallel(model.to(dev).train(), device_ids=[0, 1])
    out = dp(imgs.to(dev))
    assert out.shape == z32.shape and rel(out, z32) <= 1e-2
    loss = b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C) + b2u.Dice_loss(out, O.one_hot(pngs, C).to(dev))
    loss.backward()
    assert abs(loss.item() - l32.item()) <= 1e-2 * abs(l32.item())
    assert _global_rel({k: p.grad for k, p in model.named_parameters()}, g32) <= 1e-2
    assert len(model._engines) == 2


def _syncbn_worker(rank, world, port, sd, imgs, pngs, C, out):
    import torch.distributed as dist
    import unet_pytorch_b200 as b2u
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        solo = [dist.new_group([r]) for r in range(world)][rank]
        ref = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0, model="traditional", dice_loss=False, process_group=solo)
        r_ref = ref.train_step(imgs.to(dev), pngs.to(dev)).cpu()                       # full batch on one GPU
        tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0, model="traditional", dice_loss=False, sync_bn=True)
        n = imgs.shape[0] // world
        r_sync = tr.train_step(imgs[rank * n:(rank + 1) * n].to(dev), pngs[rank * n:(rank + 1) * n].to(dev))
        loss = r_sync[0].clone()
        dist.all_reduce(loss)
        # the flat gradient buffer holds the SUM over ranks (the 1/world factor is applied inside the optimizer kernel)
        num = sum((tr.grads[k] / world - ref.grads[k]).double().pow(2).sum().item() for k in ref.grads)
        den = sum(ref.grads[k].double().pow(2).sum().item() for k in ref.grads)
        rm_err = max((tr.buffers[k] - ref.buffers[k]).abs().max().item() for k in ref.buffers if k.endswith("running_mean"))
        worst = sorted(((((tr.grads[k] / world - ref.grads[k]).norm() / (ref.grads[k].norm() + 1e-20)).item(), k) for k in ref.grads), reverse=True)[:6]
        if os.environ.get("B2U_TEST_VERBOSE"):
            print(f"[rank {rank}] worst tensors: {worst}", flush=True)
        near = {k: ((tr.grads[k] / world - ref.grads[k]).norm() / (ref.grads[k].norm() + 1e-20)).item()
                for k in ("outc.weight", "outc.bias", "up3.conv.double_conv.4.weight", "up3.conv.double_conv.3.weight")}
        if os.environ.get("B2U_TEST_VERBOSE"):
            print(f"[rank {rank}] near-output tensors: {near}", flush=True)
        out[rank] = (loss.item() / world, r_ref[0].item(), (num / den) ** 0.5, rm_err, max(near.values()))
    finally:
        dist.destroy_process_group()


def test_sync_batchnorm_two_gpus(cuda_device):
    """UnetTrainer(sync_bn=True) on two ranks holding half a batch each = one GPU on the whole batch (CE without ignored
    pixels is a plain mean, so the mean of the shard losses and the averaged gradients must match): BatchNorm statistics,
    running averages and the data gradient see all ranks (train.py:335-336, nn.SyncBatchNorm)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    C = 4
    sd = O.make_trad_params(C)
    imgs, pngs = O.make_inputs(4, C, 64, 64, seed=9)
    pngs = pngs.clamp(max=C - 1)                      # no ignored pixels: equal normalisers on every shard
    out = mp.Manager().dict()
    mp.spawn(_syncbn_worker, args=(2, 29651, sd, imgs, pngs, C, out), nprocs=2, join=True)
    for rank in (0, 1):
        loss_sync, loss_ref, gerr, rm_err, near = out[rank]
        assert abs(loss_sync - loss_ref) <= 2e-3 * abs(loss_ref)
        assert rm_err <= 1e-3
        # two bf16 runs with different summation orders: the tensors next to the output agree closely; through the 14
        # BatchNorm backward passes the difference is amplified like any other bf16 rounding (see DESIGN.md section 5)
        assert near <= 2e-2 and gerr <= 0.15


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _syncbn_gloo_worker(rank, world, port, z, dy, residual, gamma, beta, rm, rv, out_dir):
    import torch.distributed as dist
    import unet_pytorch_b200 as b2u
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        dev = torch.device("cuda:0")
        n = z.shape[0] // world
        mine = slice(rank * n, (rank + 1) * n)
        zr, dyr, g, bt = z[mine].to(dev), dy[mine].to(dev), gamma.to(dev), beta.to(dev)
        res = {}
        for tag, rr in (("plain", None), ("residual", residual[mine].to(dev))):
            rmr, rvr = rm.to(dev), rv.to(dev)
            y, mean, invstd = b2u.ops.bn_fwd_train_sync(zr, g, bt, rmr, rvr, dist.group.WORLD, residual=rr)
            gout = torch.empty_like(zr)
            dz, dgam, dbet = b2u.ops.bn_bwd_sync(dyr, y if rr is not None else None, zr, g, mean, invstd, dist.group.WORLD,
                                                 gout=gout, beta=bt)
            res[tag] = {k: v.cpu() for k, v in dict(y=y, mean=mean, invstd=invstd, rm=rmr, rv=rvr, dz=dz, gout=gout,
                                                     dgamma=dgam, dbeta=dbet).items()}
        torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_sync_batchnorm_wrappers_gloo_one_gpu(b2u, cuda_device, tmp_path):
    """ops.bn_fwd_train_sync / ops.bn_bwd_sync in a two-process gloo group whose ranks share cuda:0, half a batch each:
    the collectives of the wrappers (all-gather of the moments, all-reduce of the backward sums, CUDA tensors through
    gloo) give what ops.bn_fwd_train / ops.bn_bwd give on the whole batch, both held to fp64 BatchNorm with the bounds of
    test_kernels_at_scale_gpu.py, at channel means up to 64 standard deviations."""
    import torch.multiprocessing as mp
    from test_kernels_at_scale_gpu import _bn_data, _bn_fwd_ref, _bn_stat_errors, check_bf16, check_sum
    dev = cuda_device
    N, H, W, C = 8, 64, 64, 128
    P = N * H * W
    z, ratio = _bn_data(dev, N, H, W, C, 19)
    g = torch.Generator(device=dev).manual_seed(20)
    gamma = (1 + 0.2 * torch.randn((C,), generator=g, device=dev)) * torch.where(torch.arange(C, device=dev) % 3 == 2, -1.0, 1.0)
    beta = 0.1 * torch.randn((C,), generator=g, device=dev)
    rm0, rv0 = 0.1 * torch.randn((C,), generator=g, device=dev), torch.rand((C,), generator=g, device=dev) + 0.5
    residual = torch.randn((N, H, W, C), generator=g, device=dev).to(torch.bfloat16)
    dy = torch.randn((N, H, W, C), generator=g, device=dev).to(torch.bfloat16)
    mp.spawn(_syncbn_gloo_worker, args=(2, _free_port(), z.cpu(), dy.cpu(), residual.cpu(), gamma.cpu(), beta.cpu(), rm0.cpu(),
                                        rv0.cpu(), str(tmp_path)), nprocs=2, join=True)
    ranks = [torch.load(tmp_path / f"rank{r}.pt") for r in range(2)]
    zd = z.double().permute(0, 3, 1, 2)
    sh = (-1, 1, 1)
    for tag, res in (("plain", None), ("residual", residual)):
        got = {k: [ranks[r][tag][k].to(dev) for r in range(2)] for k in ranks[0][tag]}
        for k in ("mean", "invstd", "rm", "rv"):
            assert torch.equal(got[k][0], got[k][1]), f"{tag}: {k} differs between the ranks"
        rm, rv = rm0.clone(), rv0.clone()
        y1, mean1, invstd1 = b2u.ops.bn_fwd_train(z, gamma, beta, rm, rv, residual=res)
        m_ref, v_ref = _bn_stat_errors(f"gloo sync bn {tag}", got["mean"][0], got["invstd"][0], z, ratio)
        _bn_stat_errors(f"one GPU bn {tag}", mean1, invstd1, z, ratio)
        want_rv = 0.9 * rv0.double() + 0.1 * v_ref * P / (P - 1)
        for r_v in (got["rv"][0], rv):
            assert ((r_v.double() - want_rv).abs() / want_rv).max().item() <= 2e-6
        for r_m in (got["rm"][0], rm):
            assert torch.allclose(r_m.double(), 0.9 * rm0.double() + 0.1 * m_ref, rtol=1e-6, atol=1e-6 * v_ref.sqrt().max().item())
        ref_y, A_y = _bn_fwd_ref(zd, m_ref, (v_ref + 1e-5).rsqrt(), gamma, beta, res)
        y_sync = torch.cat(got["y"])
        check_bf16(f"gloo sync bn {tag} y", y_sync, ref_y, A_y)
        check_bf16(f"one GPU bn {tag} y", y1, ref_y, A_y)
        # backward from each path's own forward (ReLU mask from z without a residual, from y with one)
        gout1 = torch.empty_like(z)
        dz1, dg1, db1 = b2u.ops.bn_bwd(dy, y1 if res is not None else None, z, gamma, mean1, invstd1, gout=gout1, beta=beta)
        for name, y_, dz_, gout_, mean_, invstd_ in (("gloo sync", y_sync, torch.cat(got["dz"]), torch.cat(got["gout"]),
                                                      got["mean"][0], got["invstd"][0]),
                                                     ("one GPU", y1, dz1, gout1, mean1, invstd1)):
            assert torch.equal(gout_, dy * (y_ > 0)), f"{name} {tag}: gout"
            gm = dy.double().permute(0, 3, 1, 2) * (y_ > 0).permute(0, 3, 1, 2)
            xk = (zd - mean_.double().view(sh)) * invstd_.double().view(sh)
            ref_db, ref_dg = gm.sum((0, 2, 3)), (gm * xk).sum((0, 2, 3))
            a = (gamma.double() * invstd_.double()).view(sh)
            ref_dz = a * (gm - (ref_db / P).view(sh) - xk * (ref_dg / P).view(sh))
            A_dz = a.abs() * (gm.abs() + (ref_db.abs() / P).view(sh) + xk.abs() * (ref_dg.abs() / P).view(sh))
            check_bf16(f"{name} bn {tag} dz", dz_, ref_dz, A_dz)
            if name == "one GPU":
                check_sum(f"one GPU bn {tag} dbeta", db1, ref_db, gm.abs().sum((0, 2, 3)))
                check_sum(f"one GPU bn {tag} dgamma", dg1, ref_dg, (gm * xk).abs().sum((0, 2, 3)))
            else:       # the affine gradients stay local to each rank, like nn.SyncBatchNorm's
                for r in range(2):
                    part = slice(r * N // 2, (r + 1) * N // 2)
                    check_sum(f"gloo sync bn {tag} rank {r} dbeta", got["dbeta"][r], gm[part].sum((0, 2, 3)), gm[part].abs().sum((0, 2, 3)))
                    check_sum(f"gloo sync bn {tag} rank {r} dgamma", got["dgamma"][r], (gm * xk)[part].sum((0, 2, 3)),
                              (gm * xk)[part].abs().sum((0, 2, 3)))


def _dp_trainer_worker(rank, world, port, sd, imgs, pngs, C, out):
    import torch.distributed as dist
    import unet_pytorch_b200 as b2u
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        n = imgs.shape[0] // world
        xs, ys = imgs[rank * n:(rank + 1) * n].to(dev), pngs[rank * n:(rank + 1) * n].to(dev)
        # rank 1 starts from DIFFERENT weights: the constructor's broadcast (DDP semantics, train.py:346) must overwrite them
        start = sd if rank == 0 else {k: v + 0.01 for k, v in sd.items()}
        tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=start, lr=1e-4, bucket_mb=1)
        res = tr.train_step(xs, ys).cpu()
        grads = {k: (v / world).cpu() for k, v in tr.grads.items()}       # the flat buffer holds the SUM over ranks
        for _ in range(2):
            tr.train_step(xs, ys)
        ref_p = tr.flat_param.clone()
        dist.broadcast(ref_p, src=0)
        diff = (tr.flat_param - ref_p).abs().max().reshape(1)
        dist.all_reduce(diff, op=dist.ReduceOp.MAX)
        out[rank] = (res.tolist(), grads if rank == 0 else None, float(diff.item()), len(tr.layout.buckets))
    finally:
        dist.destroy_process_group()


def test_data_parallel_trainer_two_gpus_vs_mean_of_shards(cuda_device):
    """UnetTrainer on two NCCL ranks, 2 images each: the synchronised gradient is the MEAN of the per-shard gradients (each
    shard normalises CE / Dice over itself, utils_fit.py:70-81 -- NOT the gradient of the global batch), per the fp32 oracle;
    after three Adam steps both ranks hold bit-identical parameters."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    C = 21
    sd = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(4, C, 64, 64, seed=13)
    w = torch.ones(C)
    shard = [O.train_step(sd, imgs[r * 2:(r + 1) * 2], pngs[r * 2:(r + 1) * 2], w, C, dice=True) for r in range(2)]
    mean = {k: (shard[0][2][k] + shard[1][2][k]) / 2 for k in sd}
    whole = O.train_step(sd, imgs, pngs, w, C, dice=True)[2]
    out = mp.Manager().dict()
    mp.spawn(_dp_trainer_worker, args=(2, 29653, sd, imgs, pngs, C, out), nprocs=2, join=True)
    (res0, grads, diff0, nb), (res1, _, diff1, _) = out[0], out[1]
    assert nb >= 4                                            # several buckets were in flight
    assert diff0 == 0.0 and diff1 == 0.0                      # replicas stay bit-identical
    for r, res in ((0, res0), (1, res1)):                     # every rank reports ITS shard's loss
        assert abs(res[0] - shard[r][0].item()) <= 1e-2 * abs(shard[r][0].item())
    gerr = _global_rel(grads, mean)
    assert gerr <= 1e-2
    # and it is measurably not the single-global-batch gradient where the two differ
    gap = _global_rel(mean, whole)
    print(f"\n[dp2] grad vs mean-of-shards oracle {gerr:.2e}; mean-of-shards vs global-batch gradient {gap:.2e}")


# ------------------------------------------------------------------------------------------------ bf16 on the pinned branch
def _bn_family(b2u, golden_dir, family):
    """(model, state dict, inputs, label map, class weights, oracle step, zero-gradient-bias predicate, dropout override)."""
    import importlib
    if family == "traditional":
        C, n, h, w, seed = 4, 2, 64, 64, 3
        sd = O.make_trad_params(C, seed=11)
        imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
        wts = torch.tensor([1, 15, 1.5, 2], dtype=torch.float32)
        step = lambda p, x, ww: O.trad_train_step(p, x, pngs, ww, C, dice=True, focal=True)
        return (b2u.TraditionalUnet(in_channels=3, num_classes=C), sd, imgs, pngs, wts, step, True, True,
                lambda k: k.endswith(".double_conv.0.bias") or k.endswith(".double_conv.3.bias"), None)
    if family == "resnet50":
        C, n, h, w, seed = 21, 2, 64, 64, 7
        sd = O.make_resnet_unet_params(C, seed=11)
        imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
        wts = torch.ones(C)
        step = lambda p, x, ww: O.resnet_unet_train_step(p, x, pngs, ww, C, dice=True)
        return b2u.Unet(num_classes=C, backbone="resnet50"), sd, imgs, pngs, wts, step, True, False, lambda k: False, None
    if family == "lightweight":
        g = np.load(os.path.join(golden_dir, "lightweight_nc21_cedice.npz"))
        C, n, h, w, seed, dice, focal = [int(v) for v in g["meta"]]
        sd = O.make_lw_params(C, seed=11)
        imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
        wts = torch.from_numpy(g["cls_w"])
        masks = {k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("drop:")}
        step = lambda p, x, ww: O.lw_train_step(p, x, pngs, ww, C, dice=bool(dice), focal=bool(focal), drop_masks=masks)

        def pre_bn_bias(k):
            base = k.rsplit(".", 1)[0]
            return k.endswith(".bias") and (base.endswith(".conv.0") or base.endswith(".conv1") or base.endswith(".conv2"))
        return b2u.LightweightUnet(num_classes=C), sd, imgs, pngs, wts, step, bool(dice), bool(focal), pre_bn_bias, masks
    variant, cls, tag = {"ultralight": ("ultralight", "UltraLightweightUnet", "nc21_cedice"),
                         "ultralight_large": ("ultralight_large", "UltraLightweightUnet_large", "nc4_focaldice"),
                         "ultralight_large_optimized": ("ultralight_large_optimized", "UltraLightweightUnet_large_optimized", "nc21_cedice")}[family]
    g = np.load(os.path.join(golden_dir, f"{variant}_{tag}.npz"))
    C, n, h, w, seed, dice, focal = [int(v) for v in g["meta"]]
    sd = O.make_ulu_params(C, variant, seed=11)
    imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
    wts = torch.from_numpy(g["cls_w"])
    mask = torch.from_numpy(g["drop_mask"]) if "drop_mask" in g.files else None
    step = lambda p, x, ww: O.ulu_train_step(p, x, pngs, ww, C, variant, dice=bool(dice), focal=bool(focal), drop_mask=mask)
    Net = getattr(importlib.import_module(f"unet_pytorch_b200.nets.{cls}"), cls)
    return (Net(num_classes=C), sd, imgs, pngs, wts, step, bool(dice), bool(focal),
            lambda k: k.endswith(".conv.0.bias") or k.endswith("wise.bias"), mask)


@pytest.mark.parametrize("family", ["traditional", "resnet50", "lightweight", "ultralight", "ultralight_large", "ultralight_large_optimized"])
def test_batchnorm_families_bf16_on_pinned_branch(b2u, cuda_device, golden_dir, family):
    """The product (bf16) path of every BatchNorm family against the float64 oracle evaluated on the branch the CUDA run took
    (its ReLU masks and max-pool winners, tests/branch_util.py).  Against the fp32 reference on ITS branch these nets' bf16
    gradients differ by 9-16 % (tests above); this test separates the two causes -- sign/winner flips of ~0 pre-activations,
    which bf16 storage makes by the thousand (0.3-2 % of all sites), and rounding proper -- by removing the first.  Measured
    (profiles/r1_fp32_validation.txt): 2.2e-2 ... 7.7e-2 on the branch, i.e. flips account for one half to three quarters of the
    9-16 %, and what remains is bf16 storage rounding amplified by the BatchNorm chain (the oracle's bf16-storage model shows
    the same 3.4e-2 for TraditionalUnet on its own pinned branch); the fp32 validation build on the same fixtures is at
    1.5e-6 ... 4e-5 (tests/test_fp32_validation_gpu.py), so the engines' logic is not part of it."""
    from branch_util import compare_on_branch
    dev = cuda_device
    model, sd, imgs, pngs, wts, step, dice, focal, zero_bias, drop = _bn_family(b2u, golden_dir, family)
    C = wts.numel()
    model.load_state_dict(sd)
    model = model.train().to(dev)
    eng = model._engine_for(dev)
    if drop is not None:
        eng.dropout_override = drop
    outputs = model(imgs.to(dev))
    loss = (b2u.Focal_Loss if focal else b2u.CE_Loss)(outputs, pngs.to(dev), wts.to(dev), num_classes=C)
    if dice:
        loss = loss + b2u.Dice_loss(outputs, O.one_hot(pngs, C).to(dev))
    loss.backward()
    grads = {k: p.grad for k, p in model.named_parameters()}
    d = compare_on_branch(family + " bf16", step, sd, imgs, wts, grads, eng, skip=zero_bias)
    zrel = rel(outputs, d["z64"])
    print(f"{family} bf16: logits vs float64 on the branch {zrel:.2e}, loss {loss.item():.6f} vs {d['l64'].item():.6f}")
    assert zrel <= 8e-2 and d["ours"] <= 1.2e-1        # ~1.5x the measured values: a regression guard, not a precision claim
