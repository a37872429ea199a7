"""GPU: the gradient with respect to the input image (x.grad) of every drop-in model, against torch.autograd.grad of the
float64 oracle.  The BatchNorm families are compared on the branch the CUDA run took (tests/branch_util.py: its ReLU masks
and max-pool winners replayed in the oracle), so what is measured is the arithmetic, not sign flips of ~0 pre-activations.
Also: the new kernels alone at training scale, frozen parameters, composition with a trainable module in front, and that
nothing changes (bit for bit, and no new launches) when the input needs no gradient."""
import contextlib
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import unet_oracle as O
from branch_util import engine_branch, rel

pytestmark = pytest.mark.gpu

NEW_KERNELS = ("first_conv_dgrad_input", "stem_dgrad_input", "nhwc_bf16_padded_to_nchw_f32")


@pytest.fixture()
def fp32_build(b2u, cuda_device):
    b2u.ops.set_validation_fp32(True)
    try:
        yield b2u
    finally:
        b2u.ops.set_validation_fp32(False)


def _family(b2u, golden_dir, family, training=True, in_channels=3):
    """(model, state dict, images, labels, oracle forward (sd, x) -> logits, dropout override, pin the branch?)"""
    if family == "vgg":
        C = 4
        imgs, pngs = O.make_inputs(2, C, 64, 64, seed=2)
        return (b2u.Unet(num_classes=C), O.make_params(C, seed=11), imgs, pngs,
                lambda sd, x, bf=False: (O.unet_forward_bf16_storage if bf else O.unet_forward)(sd, x), None, False)
    if family == "traditional":
        C = 4
        imgs, pngs = O.make_inputs(2, C, 64, 64, seed=3)
        if in_channels != 3:
            imgs = torch.randn(2, in_channels, 64, 64, generator=torch.Generator().manual_seed(5))
        return (b2u.TraditionalUnet(in_channels=in_channels, num_classes=C), O.make_trad_params(C, seed=11, in_channels=in_channels),
                imgs, pngs, lambda sd, x, bf=False: O.trad_forward(sd, x, training=training, bf16_storage=bf)[0], None, True)
    if family == "resnet50":
        C = 21
        imgs, pngs = O.make_inputs(2, C, 64, 64, seed=7)
        return (b2u.Unet(num_classes=C, backbone="resnet50"), O.make_resnet_unet_params(C, seed=11), imgs, pngs,
                lambda sd, x, bf=False: O.resnet_unet_forward(sd, x, training=training, bf16_storage=bf)[0], None, True)
    if family == "lightweight":
        g = np.load(os.path.join(golden_dir, "lightweight_nc21_cedice.npz"))
        C, n, h, w, seed = [int(v) for v in g["meta"]][:5]
        masks = {k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("drop:")} if training else None
        imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
        if in_channels != 3:
            imgs = torch.randn(n, in_channels, h, w, generator=torch.Generator().manual_seed(5))
        torch.manual_seed(3)
        model = b2u.LightweightUnet(num_classes=C, in_channels=in_channels)
        sd = O.make_lw_params(C, seed=11) if in_channels == 3 else {k: v.detach().clone() for k, v in model.state_dict().items()}
        return (model, sd, imgs, pngs, lambda s, x, bf=False: O.lw_forward(s, x, training=training, bf16_storage=bf, drop_masks=masks)[0],
                masks, True)
    if family.startswith("ultralight"):
        cls, tag = {"ultralight": ("UltraLightweightUnet", "nc21_cedice"), "ultralight_large": ("UltraLightweightUnet_large", "nc4_focaldice"),
                    "ultralight_large_optimized": ("UltraLightweightUnet_large_optimized", "nc21_cedice")}[family]
        g = np.load(os.path.join(golden_dir, f"{family}_{tag}.npz"))
        C, n, h, w, seed = [int(v) for v in g["meta"]][:5]
        mask = torch.from_numpy(g["drop_mask"]) if ("drop_mask" in g.files and training) else None
        imgs, pngs = O.make_inputs(n, C, h, w, seed=seed)
        import importlib
        Net = getattr(importlib.import_module(f"unet_pytorch_b200.nets.{cls}"), cls)
        return (Net(num_classes=C), O.make_ulu_params(C, family, seed=11), imgs, pngs,
                lambda sd, x, bf=False: O.ulu_forward(sd, x, family, training=training, bf16_storage=bf, drop_mask=mask)[0], mask, True)
    assert family in ("isn", "isn_deploy")
    C = 4
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=9)
    torch.manual_seed(0)
    model = b2u.ImprovedSegNet(num_classes=C)
    if family == "isn_deploy":
        model.switch_to_deploy()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    deploy = family == "isn_deploy"
    return (model, sd, imgs, pngs, lambda s, x, bf=False: None if bf else O.isn_forward(s, x, training=training, deploy=deploy)[0],
            torch.ones(2, 704) if training else None, True)


def _loss(logits, pngs, C):
    if logits.shape[-2:] != pngs.shape[-2:]:
        logits = O.resize_logits(logits, pngs.shape[1], pngs.shape[2])
    w = torch.ones(C, dtype=logits.dtype)
    return O.ce_loss(logits, pngs, w, C) + O.dice_loss(logits, O.one_hot(pngs, C).to(logits.dtype))


def _oracle_xgrad(fwd, sd, imgs, pngs, C, pin=None, dtype=torch.float64, pre=None, bf=False):
    """torch.autograd.grad(loss, x) of the oracle in `dtype`, on the pinned branch when pin is given.  pre: (a, b) of a
    per-channel affine applied to x first; then their gradients are returned too."""
    sdt = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd.items()}
    x = imgs.to(dtype).requires_grad_(True)
    leaves = [x]
    inp = x
    if pre is not None:
        a, b = (t.to(dtype).requires_grad_(True) for t in pre)
        leaves += [a, b]
        inp = x * a.view(1, -1, 1, 1) + b.view(1, -1, 1, 1)
    with (O.branch(pin=pin) if pin is not None else contextlib.nullcontext()):
        logits = fwd(sdt, inp, bf)
    if logits is None:
        return None
    return torch.autograd.grad(_loss(logits, pngs, C), leaves)


def _pin(eng, fwd, sd, imgs):
    own = {}
    with O.branch(record=own):
        fwd({k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}, imgs.double())
    # sites the oracle keys (ImprovedSegNet's residual / deploy ReLUs are plain F.relu there and stay unpinned)
    return {k: v[:, :own[k].shape[1]].contiguous() for k, v in engine_branch(eng).items() if k in own}


def cos(a, b):
    a, b = a.double().cpu().reshape(-1), b.double().cpu().reshape(-1)
    return (a @ b / (a.norm() * b.norm() + 1e-300)).item()


# Where bf16 storage alone moves x.grad by more than its own norm (Unet-ResNet50, ImprovedSegNet) a rel-L2 bound is above 1
# and would accept x.grad == 0; every product-build result must also point the way float64's does
COS_MIN = 0.5


def _check_close(tag, grad, g64, lim):
    r, c = rel(grad, g64), cos(grad, g64)
    print(f"\n[{tag}] x.grad vs float64: rel-L2 {r:.2e} (bound {lim:.2e}), cosine {c:.4f}")
    assert r <= lim, (tag, r, lim)
    if lim >= 1e-3:
        assert c >= COS_MIN, (tag, c)


def _limit(fwd, sd, imgs, pngs, C, pin, g64, pre=None):
    """Bound for the product build: rel-L2 1e-2 against float64, or 1.5x what bf16 storage alone costs where that is more --
    the oracle's bf16-storage model (fp32 math, rounded to bf16 where the engine stores a bf16 tensor) on the same branch.
    The input gradient is the end of the longest chain of the backward: in these nets bf16 storage alone moves it by
    2e-2 .. 1e-1 at these sizes.  Returns (limit, the model's distance or None where the oracle has no such model)."""
    gb = _oracle_xgrad(fwd, sd, imgs, pngs, C, pin, dtype=torch.float32, pre=pre, bf=True)
    model = rel(gb[0], g64) if gb is not None else None
    return max(1e-2, 1.5 * model) if model is not None else 1e-2, model


# ImprovedSegNet has no bf16-storage model in the oracle.  Its input gradient is the worst conditioned of all families here
# (torch fp32 vs float64: 2.6e-4 training form, 8.6e-5 deploy form, against ~1e-6 for most others), and bf16 measured
# 7.4e-1 (training form) and 5.5e-1 (deploy form) on one B200: the bound below is ~1.5x the larger, a regression guard and
# not a precision claim; the fp32 build checks the same path to fp32 round-off (test_input_grad_fp32_build)
NO_MODEL_GUARD = {"isn": 1.1, "isn_deploy": 1.1}


def _run(b2u, dev, model, sd, imgs, pngs, drop, training=True, params_grad=True, pre=None):
    model.load_state_dict(sd)
    model = model.to(dev).train(training)
    for p in model.parameters():
        p.requires_grad_(params_grad)
    eng = model._engine_for(dev)
    if drop is not None:
        eng.dropout_override = drop
    x = imgs.to(dev).requires_grad_(True)
    inp = x
    if pre is not None:
        inp = x * pre[0].view(1, -1, 1, 1) + pre[1].view(1, -1, 1, 1)
    out = model(inp)
    C = out.shape[1]
    loss = b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C) + b2u.Dice_loss(out, O.one_hot(pngs, C).to(dev))
    loss.backward()
    return model, eng, x, out


FAMILIES = ["vgg", "traditional", "resnet50", "lightweight", "ultralight", "ultralight_large", "ultralight_large_optimized",
            "isn", "isn_deploy"]


def _check_family(b2u, dev, golden_dir, family, in_channels=3, fp32=False):
    model, sd, imgs, pngs, fwd, drop, pinned = _family(b2u, golden_dir, family, in_channels=in_channels)
    model, eng, x, out = _run(b2u, dev, model, sd, imgs, pngs, drop)
    C = out.shape[1]
    pin = _pin(eng, fwd, sd, imgs) if pinned else None
    g64 = _oracle_xgrad(fwd, sd, imgs, pngs, C, pin)[0]
    g32 = _oracle_xgrad(fwd, sd, imgs, pngs, C, pin, dtype=torch.float32)[0]
    ours, ref32 = rel(x.grad, g64), rel(g32, g64)
    lim, model_d = (max(1e-5, 2 * ref32), None) if fp32 else _limit(fwd, sd, imgs, pngs, C, pin, g64)
    if model_d is None and not fp32:
        lim = NO_MODEL_GUARD[family]
    print(f"\n[x.grad {family} cin={in_channels} {'fp32 build' if fp32 else 'bf16'}] vs float64 {ours:.2e}; torch fp32 {ref32:.2e}; "
          f"bf16-storage model {model_d}")
    assert x.grad.shape == imgs.shape and x.grad.dtype == torch.float32
    _check_close(f"{family} cin={in_channels}", x.grad, g64, lim)
    for p in model.parameters():            # the parameter gradients are still there
        assert p.grad is not None


@pytest.mark.parametrize("family", FAMILIES)
def test_input_grad_matches_oracle(b2u, cuda_device, golden_dir, family):
    _check_family(b2u, cuda_device, golden_dir, family)


@pytest.mark.parametrize("family", FAMILIES)
def test_input_grad_fp32_build(fp32_build, cuda_device, golden_dir, family):
    _check_family(fp32_build, cuda_device, golden_dir, family, fp32=True)


@pytest.mark.parametrize("family,cin", [("traditional", 5), ("lightweight", 40)])
def test_input_grad_without_image_split(b2u, cuda_device, golden_dir, family, cin):
    """9 Cin > 32 (TraditionalUnet) and 2 Cin > 64 (LightweightUnet): the image enters without its lo half."""
    _check_family(b2u, cuda_device, golden_dir, family, in_channels=cin)


@pytest.mark.parametrize("family", ["vgg", "traditional", "ultralight_large"])
def test_only_input_requires_grad_eval(b2u, cuda_device, golden_dir, family):
    """Saliency / FGSM on a trained model: eval(), every parameter frozen, only x requires grad."""
    dev = cuda_device
    model, sd, imgs, pngs, fwd, _, pinned = _family(b2u, golden_dir, family, training=False)
    model, eng, x, out = _run(b2u, dev, model, sd, imgs, pngs, None, training=False, params_grad=False)
    pin = _pin(eng, fwd, sd, imgs) if pinned else None
    g64 = _oracle_xgrad(fwd, sd, imgs, pngs, out.shape[1], pin)[0]
    lim, model_d = _limit(fwd, sd, imgs, pngs, out.shape[1], pin, g64)
    print(f"\n[x.grad {family} eval, parameters frozen] vs float64 {rel(x.grad, g64):.2e}; bf16-storage model {model_d}")
    _check_close(f"{family} eval", x.grad, g64, lim)
    assert all(p.grad is None for p in model.parameters())


@pytest.mark.parametrize("build", ["bf16", "fp32"])
@pytest.mark.parametrize("family,prefix", [("vgg", "vgg."), ("resnet50", "resnet.")])
def test_frozen_backbone_still_reaches_the_image(b2u, cuda_device, golden_dir, family, prefix, build):
    dev = cuda_device
    if build == "fp32":
        b2u.ops.set_validation_fp32(True)
    try:
        _frozen_backbone(b2u, dev, golden_dir, family, prefix, build == "fp32")
    finally:
        b2u.ops.set_validation_fp32(False)


def _frozen_backbone(b2u, dev, golden_dir, family, prefix, fp32):
    model, sd, imgs, pngs, fwd, drop, pinned = _family(b2u, golden_dir, family)
    model.load_state_dict(sd)
    model = model.to(dev).train()
    model.freeze_backbone()
    eng = model._engine_for(dev)
    x = imgs.to(dev).requires_grad_(True)
    out = model(x)
    C = out.shape[1]
    loss = b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C) + b2u.Dice_loss(out, O.one_hot(pngs, C).to(dev))
    loss.backward()
    pin = _pin(eng, fwd, sd, imgs) if pinned else None
    g64 = _oracle_xgrad(fwd, sd, imgs, pngs, C, pin)[0]
    if fp32:
        lim = max(1e-5, 2 * rel(_oracle_xgrad(fwd, sd, imgs, pngs, C, pin, dtype=torch.float32)[0], g64))
    else:
        lim = _limit(fwd, sd, imgs, pngs, C, pin, g64)[0]
    _check_close(f"{family} frozen backbone, {'fp32 build' if fp32 else 'bf16'}", x.grad, g64, lim)
    for k, p in model.named_parameters():
        assert (p.grad is None) == k.startswith(prefix), k


def test_trainable_affine_in_front_gets_its_gradient(b2u, cuda_device, golden_dir):
    """A learnable per-channel input normalisation in front of the UNet learns: its gradient is the oracle's."""
    dev = cuda_device
    model, sd, imgs, pngs, fwd, drop, _ = _family(b2u, golden_dir, "vgg")
    a = torch.tensor([0.9, 1.1, 1.3], device=dev, requires_grad=True)
    b = torch.tensor([0.05, -0.1, 0.2], device=dev, requires_grad=True)
    model, eng, x, out = _run(b2u, dev, model, sd, imgs, pngs, drop, pre=(a, b))
    gx, ga, gb = _oracle_xgrad(fwd, sd, imgs, pngs, out.shape[1], pre=(a.detach().cpu(), b.detach().cpu()))
    pre = (a.detach().cpu(), b.detach().cpu())
    lim, model_d = _limit(fwd, sd, imgs, pngs, out.shape[1], None, gx, pre=pre)
    print(f"\n[affine in front] a.grad {rel(a.grad, ga):.2e}, b.grad {rel(b.grad, gb):.2e}, x.grad {rel(x.grad, gx):.2e}; "
          f"bf16-storage model {model_d}")
    assert rel(a.grad, ga) <= 1e-2 and rel(b.grad, gb) <= 1e-2 and rel(x.grad, gx) <= lim


def _step(b2u, model, sd, imgs, pngs, x_grad):
    model.load_state_dict(sd)           # the same running statistics (training centres BatchNorm inputs on them) every step
    for p in model.parameters():
        p.grad = None
    x = imgs.clone().requires_grad_(x_grad)
    out = model(x)
    C = out.shape[1]
    loss = b2u.CE_Loss(out, pngs, torch.ones(C, device=imgs.device), num_classes=C)
    loss.backward()
    return out.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters()}


@pytest.mark.parametrize("family", ["vgg", "ultralight"])
def test_nothing_changes_without_input_grad(b2u, cuda_device, golden_dir, family):
    dev = cuda_device
    model, sd, imgs, pngs, _, _, _ = _family(b2u, golden_dir, family)
    model.load_state_dict(sd)
    model = model.to(dev).train()
    imgs, pngs = imgs.to(dev), pngs.to(dev)
    z0, g0 = _step(b2u, model, sd, imgs, pngs, False)
    z1, g1 = _step(b2u, model, sd, imgs, pngs, True)
    assert torch.equal(z0, z1)
    for k in g0:
        assert torch.equal(g0[k], g1[k]), k
    from torch.profiler import ProfilerActivity, profile
    names = {}
    for x_grad in (False, True):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _step(b2u, model, sd, imgs, pngs, x_grad)
            torch.cuda.synchronize()
        names[x_grad] = [e.key for e in prof.key_averages()]
    assert not [n for n in names[False] if any(k in n for k in NEW_KERNELS)], names[False]
    assert [n for n in names[True] if any(k in n for k in NEW_KERNELS)], names[True]


def test_kernels_at_training_scale(b2u, cuda_device):
    """Batch 16 at 512 x 512 (stem dz at 256 x 256): many tiles per launch; two images of the batch against
    torch.nn.grad.conv2d_input in float64 on the CPU (dz is bf16, so the reference sees exactly the operands)."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator(device="cpu").manual_seed(0)
    N, H, W = 16, 512, 512
    check = [0, 15]
    for cin, cout in ((3, 64), (3, 32), (7, 64)):       # Unet-VGG16, TraditionalUnet (32 real of 64), widest first layer
        dz = torch.randn(N, H, W, 64, generator=g).to(torch.bfloat16)
        dz[..., cout:] = 0
        w = torch.randn(cout, cin, 3, 3, generator=g) * 0.1
        dx = ops.first_conv_dgrad_input(dz.to(dev), w.to(dev)).cpu()
        ref = torch.nn.grad.conv2d_input((len(check), cin, H, W), w.double(), dz[check, :, :, :cout].double().permute(0, 3, 1, 2), padding=1)
        assert rel(dx[check], ref) <= 1e-5, (cin, cout)
    dz = torch.randn(N, H // 2, W // 2, 64, generator=g).to(torch.bfloat16)
    w = torch.randn(64, 3, 7, 7, generator=g) * 0.05
    dx = ops.stem_dgrad_input(dz.to(dev), w.to(dev), H, W).cpu()
    ref = torch.nn.grad.conv2d_input((len(check), 3, H, W), w.double(), dz[check].double().permute(0, 3, 1, 2), stride=2, padding=3)
    assert rel(dx[check], ref) <= 1e-5
    x = torch.randn(N, H, W, 64, generator=g).to(torch.bfloat16)
    for c in (3, 40):
        y = ops.nhwc_padded_to_nchw_f32(x.to(dev), c).cpu()
        assert torch.equal(y, x[..., :c].float().permute(0, 3, 1, 2))


def test_kernels_at_odd_sizes_and_offset_outputs(b2u, cuda_device):
    """Partial tiles and odd widths (the stem's im2col takes any H, W), an output view whose start is not 16-byte aligned (the
    kernels then store element by element and give the same result), and a misaligned dz, which is refused."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator(device="cpu").manual_seed(1)
    N = 3
    for H, W in ((63, 65), (64, 33), (5, 3)):
        Ho, Wo = (H + 1) // 2, (W + 1) // 2
        dz = torch.randn(N, Ho, Wo, 64, generator=g).to(torch.bfloat16)
        w = torch.randn(64, 3, 7, 7, generator=g) * 0.05
        dx = ops.stem_dgrad_input(dz.to(dev), w.to(dev), H, W).cpu()
        ref = torch.nn.grad.conv2d_input((N, 3, H, W), w.double(), dz.double().permute(0, 3, 1, 2), stride=2, padding=3)
        assert rel(dx, ref) <= 1e-5, (H, W)
    for H, W, cin in ((37, 45, 3), (19, 66, 5), (3, 1, 7)):
        dz = torch.randn(N, H, W, 64, generator=g).to(torch.bfloat16)
        w = torch.randn(64, cin, 3, 3, generator=g) * 0.1
        dx = ops.first_conv_dgrad_input(dz.to(dev), w.to(dev)).cpu()
        ref = torch.nn.grad.conv2d_input((N, cin, H, W), w.double(), dz.double().permute(0, 3, 1, 2), padding=1)
        assert rel(dx, ref) <= 1e-5, (H, W, cin)
    H, W = 64, 64
    dz = torch.randn(N, H, W, 64, generator=g).to(torch.bfloat16).to(dev)
    w3 = (torch.randn(64, 3, 3, 3, generator=g) * 0.1).to(dev)
    w7 = (torch.randn(64, 3, 7, 7, generator=g) * 0.05).to(dev)
    dzs = dz[:, :H // 2, :W // 2].contiguous()

    def offset(shape, dtype, k):          # a contiguous tensor starting k elements into its storage
        n = int(np.prod(shape))
        return torch.empty(n + k, dtype=dtype, device=dev)[k:].view(shape)
    for fn in (lambda out: ops.first_conv_dgrad_input(dz, w3, out=out), lambda out: ops.stem_dgrad_input(dzs, w7, H, W, out=out),
               lambda out: ops.nhwc_padded_to_nchw_f32(dz, 3, out=out)):
        want = fn(None)
        got = fn(offset((N, 3, H, W), torch.float32, 1))
        assert got.data_ptr() % 16 == 4 and torch.equal(got, want)
    bad = offset(tuple(dz.shape), torch.bfloat16, 1)
    bad.copy_(dz)
    with pytest.raises(b2u._lib.B2UError, match="aligned"):
        ops.first_conv_dgrad_input(bad, w3)
    with pytest.raises(b2u._lib.B2UError, match="aligned"):
        ops.nhwc_padded_to_nchw_f32(bad, 3)


def test_improved_segnet_deploy_parameter_grads_fp32_build(fp32_build, cuda_device, golden_dir):
    """Training ImprovedSegNet after switch_to_deploy(): its SE blocks and bridge Dropout2d read fused-ReLU conv outputs, and
    the gradient they send back must be masked by that ReLU.  Parameter gradients of the fp32 build against float64
    autograd of the oracle's deploy form, on the CUDA run's branch."""
    b2u, dev = fp32_build, cuda_device
    model, sd, imgs, pngs, fwd, drop, _ = _family(b2u, golden_dir, "isn_deploy")
    model.load_state_dict(sd)
    model = model.to(dev).train()
    eng = model._engine_for(dev)
    eng.dropout_override = drop
    out = model(imgs.to(dev))
    C = out.shape[1]
    loss = b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C) + b2u.Dice_loss(out, O.one_hot(pngs, C).to(dev))
    loss.backward()
    pin = _pin(eng, fwd, sd, imgs)
    names = [k for k, _ in model.named_parameters()]
    ref = {}
    for dtype in (torch.float64, torch.float32):
        sdt = {k: (v.to(dtype).requires_grad_(k in names) if v.is_floating_point() else v) for k, v in sd.items()}
        with O.branch(pin=pin):
            lg = fwd(sdt, imgs.to(dtype))
        gs = torch.autograd.grad(_loss(lg, pngs, C), [sdt[k] for k in names], allow_unused=True)
        ref[dtype] = {k: gk for k, gk in zip(names, gs) if gk is not None}
    g64, g32 = ref[torch.float64], ref[torch.float32]
    ours = {k: p.grad for k, p in model.named_parameters() if k in g64}
    assert len(ours) > 40 and any(k.endswith("reparam_conv.weight") for k in ours)
    num = sum((ours[k].double().cpu() - g64[k]).pow(2).sum().item() for k in ours)
    num32 = sum((g32[k].double() - g64[k]).pow(2).sum().item() for k in ours)
    den = sum(g64[k].pow(2).sum().item() for k in ours)
    d, d32 = (num / den) ** 0.5, (num32 / den) ** 0.5
    print(f"\n[ImprovedSegNet deploy, fp32 build] parameter gradients vs float64 {d:.2e}; torch fp32 {d32:.2e}")
    assert d <= max(1e-5, 2 * d32)


def test_dataparallel_two_gpus_input_grad(b2u, cuda_device, golden_dir):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    dev = cuda_device
    model, sd, imgs, pngs, _, _, _ = _family(b2u, golden_dir, "vgg")
    model.load_state_dict(sd)
    model = model.to(dev).train()
    grads = []
    for m in (model, torch.nn.DataParallel(model, device_ids=[0, 1])):
        x = imgs.to(dev).requires_grad_(True)
        out = m(x)
        C = out.shape[1]
        b2u.CE_Loss(out, pngs.to(dev), torch.ones(C, device=dev), num_classes=C).backward()
        grads.append(x.grad.clone())
    assert rel(grads[1], grads[0]) <= 1e-5
