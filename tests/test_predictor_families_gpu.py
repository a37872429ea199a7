"""GPU: the predictor for every model family (`Unet(model=...)`) against the per-image host path bit for bit, and
detect_images' device rendering (csrc/render.cu) against the host rendering it replaced, byte for byte."""
import os

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import render as R
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu

FAMILIES = ["traditional", "lightweight", "ultralight", "ultralight_large", "ultralight_large_optimized", "improved_segnet"]


def _image(w, h, seed, mode="RGB"):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 255 // max(w - 1, 1)), (yy * 255 // max(h - 1, 1)), ((xx + yy) * 7) % 256], -1)
    img = Image.fromarray(np.clip(base + rng.integers(-40, 41, (h, w, 3)), 0, 255).astype(np.uint8))
    if mode == "P":
        return img.quantize(colors=64)
    return img.convert(mode) if mode != "RGB" else img


def _eval_images(n, seed):
    rng = np.random.default_rng(seed)
    modes = ["RGB"] * 6 + ["L", "RGBA", "P"]
    return [_image(int(rng.integers(40, 400)), int(rng.integers(40, 400)), seed * 100 + i, modes[i % len(modes)]) for i in range(n)]


def _state_dict(model, C, seed=0):
    """He-normal weights for the family's module (synthetic.random_state_dict), running statistics perturbed so the
    folded eval BatchNorm is not an identity."""
    from unet_pytorch_b200.synthetic import random_state_dict
    from unet_pytorch_b200.unet import FAMILIES as F
    m = F[model](num_classes=C)
    sd = random_state_dict({k: tuple(v.shape) for k, v in m.named_parameters()},
                           {k: tuple(v.shape) for k, v in m.named_buffers()}, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    for k in sd:
        if k.endswith("running_mean"):
            sd[k] = 0.05 * torch.randn(sd[k].shape, generator=g)
        elif k.endswith("running_var"):
            sd[k] = 1.0 + 0.2 * torch.rand(sd[k].shape, generator=g)
    return sd


def _predictor(model, C, shape=(192, 256)):
    """A predictor whose classifier bias is shifted by minus each class's mean logit over a few images: random weights
    otherwise let one class win everywhere, and the masks would not test the tail."""
    from unet_pytorch_b200.unet import Unet as Predictor
    sd = _state_dict(model, C)
    head = [k for k, v in sd.items() if k.endswith(".weight") and v.dim() == 4 and v.shape[0] == C and v.shape[2] == 1][-1]
    pred = Predictor(model=model, state_dict=sd, num_classes=C, input_shape=list(shape))
    with torch.no_grad():
        calib = [_image(300, 200, 1000 + i) for i in range(4)]
        pred._run_batch([pred._prepare(im) for im in calib])
        z = pred._forward(pred._input[:len(calib)])
        pred.net._by_name(head[:-len("weight")] + "bias").data -= z.mean((0, 2, 3))
        pred.net.invalidate()
    return pred


def _host_path(pred, im, dev):
    """Host letterbox -> batch-1 forward -> resize of smaller logits -> single-image tail."""
    from unet_pytorch_b200 import ops
    _, data, nw, nh, oh, ow = pred._letterbox(im)
    logits = pred.net(data.to(dev))
    if logits.shape[-2:] != data.shape[-2:]:
        logits = ops.resize_bilinear(logits, tuple(data.shape[-2:]))
    return ops.softmax_resize_argmax_u8(logits, pred._crop(nw, nh), (oh, ow))[0].cpu().numpy()


@pytest.mark.parametrize("model,C", [(m, c) for m in FAMILIES for c in (4, 21)] + [("lightweight", 150)])
def test_family_predict_masks_equal_host_path(b2u, cuda_device, model, C):
    """predict_masks at batch 1, 3 and 16 over 19 images of mixed sizes and modes equals the per-image host path; the
    batched forward gives every image its batch-1 logits bit for bit; get_miou equals fast_hist over those masks."""
    pred = _predictor(model, C)
    imgs = _eval_images(19, seed=7 + C)
    with torch.no_grad():
        host = [_host_path(pred, im, cuda_device) for im in imgs]
    for bs in (1, 3, 16):
        got = pred.predict_masks(imgs, batch_size=bs)
        for i, (g, m) in enumerate(zip(got, host)):
            assert g.shape == (imgs[i].size[1], imgs[i].size[0]) and np.array_equal(g, m), f"batch {bs}, image {i}"
    assert len(np.unique(np.concatenate([m.reshape(-1) for m in host]))) >= 2
    with torch.no_grad():
        pred._run_batch([pred._prepare(im) for im in imgs[:16]])
        x = pred._input[:16].clone()
        batched = pred.net(x).clone()
        for i in range(16):
            assert torch.equal(batched[i:i + 1], pred.net(x[i:i + 1].contiguous())), f"image {i}"
    rng = np.random.default_rng(C)
    gts = [np.where(rng.random(m.shape) < 0.6, m, rng.integers(0, C, m.shape)).astype(np.uint8) for m in host]
    for gt in gts[::3]:
        gt[:3] = 255
    want = sum(O.fast_hist(gt.reshape(-1), m.reshape(-1), C) for gt, m in zip(gts, host))
    assert np.array_equal(pred.get_miou(imgs, gts, batch_size=16)[0], want)


def test_trained_ultralight_checkpoint(b2u, cuda_device, golden_dir):
    """The reference's trained UltraLightweightUnet_large_optimized (4 classes) at the reference's 256x256 inference
    size: confident, multi-class masks that equal the host path."""
    from unet_pytorch_b200.unet import Unet as Predictor
    g = np.load(os.path.join(golden_dir, "ultralight_large_optimized_checkpoint_eval.npz"))
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd:")}
    C, n, h, w, seed = [int(v) for v in g["meta"]]
    x, _ = O.make_inputs(n, C, h, w, seed=seed)
    imgs = [Image.fromarray(np.round(x[i].permute(1, 2, 0).numpy() * 255).astype(np.uint8)) for i in range(n)]
    imgs += [im.resize((300, 200)) for im in imgs] + [im.resize((180, 330)) for im in imgs]
    pred = Predictor(model="ultralight_large_optimized", state_dict=sd, num_classes=C, input_shape=[256, 256])
    got = pred.predict_masks(imgs, batch_size=16)
    with torch.no_grad():
        for im, m in zip(imgs, got):
            assert np.array_equal(m, _host_path(pred, im, cuda_device))
        prob = torch.softmax(pred.net(pred._letterbox(imgs[0])[1].to(cuda_device)), 1).max(1).values
    classes = np.unique(np.concatenate([m.reshape(-1) for m in got]))
    print(f"trained ULU: classes {classes.tolist()}, median top-1 probability {prob.median().item():.4f}, "
          f"share above 0.9 {(prob > 0.9).float().mean().item():.4f}")
    assert len(classes) >= 2
    assert prob.median().item() >= 0.9


def test_improved_segnet_after_switch_to_deploy(b2u, cuda_device):
    """switch_to_deploy() on the predictor's network: the engines are rebuilt and the masks still equal the host path;
    against the training form they differ only by the bf16 rounding of the folded weights and of the activations.
    Measured on a B200 with these weights, whose balanced classes leave many near ties: logits 3.4e-2 apart in relative
    L2, 6.2 % of the logits' argmax pixels and 3.1 % of the mask pixels; the bounds leave 1.5x."""
    from unet_pytorch_b200 import ops
    C = 21
    pred = _predictor("improved_segnet", C)
    imgs = _eval_images(12, seed=31)
    before = pred.predict_masks(imgs)
    with torch.no_grad():
        pred._run_batch([pred._prepare(im) for im in imgs])
        x = pred._input[:len(imgs)].clone()
        z0 = pred.net(x).clone()
        pred.net.switch_to_deploy()
        z1 = pred.net(x).clone()
        after = pred.predict_masks(imgs)
        for im, m in zip(imgs, after):
            assert np.array_equal(m, _host_path(pred, im, cuda_device))
    rel = ((z1 - z0).norm() / z0.norm()).item()
    differ = float(np.mean(np.concatenate([(a != b).reshape(-1) for a, b in zip(before, after)])))
    argmax_differ = (ops.argmax_u8(z0) != ops.argmax_u8(z1)).float().mean().item()
    print(f"ImprovedSegNet deploy vs training form: logits rel-L2 {rel:.2e}, mask pixels differing {differ:.2e}, "
          f"logit argmax differing {argmax_differ:.2e}")
    assert 0 < rel <= 5e-2
    assert differ <= 5e-2 and argmax_differ <= 9e-2


def _host_render(pred, image, pr):
    """The host rendering detect_image ran before (palette lookup, Image.blend, np.where)."""
    old_img = image if np.asarray(image).ndim == 3 and np.asarray(image).shape[2] == 3 else image.convert("RGB")
    if pred.mix_type not in (0, 1, 2):
        return old_img
    if pred.mix_type == 2:
        return Image.fromarray(np.where((pr != 0)[..., None], np.asarray(old_img), 0).astype(np.uint8))
    seg = Image.fromarray(np.asarray(pred.colors, np.uint8)[pr])
    return Image.blend(old_img, seg, 0.7) if pred.mix_type == 0 else seg


@pytest.mark.parametrize("C", [21, 150])
def test_detect_images_equal_host_rendering(b2u, cuda_device, C):
    """mix_type 0, 1 and 2 (VOC palette at 21 classes, HSV at 150) over mixed sizes -- a 1920x1080 frame, 1x1, sizes
    whose pixel count is not a multiple of four -- and modes, at batch sizes 1 and 4: byte for byte the host rendering of
    the same masks; counts equal np.bincount; detect_image is a batch of one with 1-D counts."""
    from unet_pytorch_b200.unet import Unet as Predictor
    pred = Predictor(state_dict=O.make_predictor_params(C, seed=11), num_classes=C, backbone="vgg", input_shape=[128, 160])
    imgs = [_image(1920, 1080, 1), _image(1, 1, 2), _image(3, 5, 3), _image(333, 250, 4, "L"), _image(250, 333, 5, "P"),
            _image(640, 427, 6, "RGBA"), _image(97, 61, 7)]
    masks = pred.predict_masks(imgs)
    assert len(np.unique(np.concatenate([m.reshape(-1) for m in masks]))) > 3
    for mix in (0, 1, 2, 3):
        pred.mix_type = mix
        want = [np.asarray(_host_render(pred, im, m)) for im, m in zip(imgs, masks)]
        for bs in (1, 4):
            got = pred.detect_images(imgs, batch_size=bs, count=True)
            for i, (g, w) in enumerate(zip(got, want)):
                assert g.mode == "RGB" and np.array_equal(np.asarray(g), w), f"mix {mix}, batch {bs}, image {i}"
            assert pred.last_counts.dtype == np.int64 and pred.last_counts.shape == (len(imgs), C)
            for c, m in zip(pred.last_counts, masks):
                assert np.array_equal(c, np.bincount(m.reshape(-1), minlength=C))
        one = pred.detect_image(imgs[3], count=True)
        assert np.array_equal(np.asarray(one), want[3])
        assert np.array_equal(pred.last_counts, np.bincount(masks[3].reshape(-1), minlength=C))
        assert np.array_equal(np.asarray(R.render(np.asarray(imgs[0]), masks[0], mix, C)), want[0])
    pred.last_counts = None
    assert len(pred.detect_images(imgs[:2])) == 2 and pred.last_counts is None
    assert pred.detect_images([], count=True) == [] and pred.last_counts.shape == (0, C)
    with pytest.raises(ValueError):
        pred.detect_images(imgs, batch_size=0)


def test_render_kernel_unaligned_pointers(b2u, cuda_device):
    """b2u_render_batch straight from tensors at odd addresses (the per-pixel path) against the numpy rendering."""
    ops, dev = b2u.ops, cuda_device
    C, h, w = 21, 37, 53
    rng = np.random.default_rng(0)
    src = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    mask = rng.integers(0, C, (h, w)).astype(np.uint8)
    sbuf = torch.from_numpy(np.concatenate([[0], src.reshape(-1)]).astype(np.uint8)).to(dev)
    mbuf = torch.from_numpy(np.concatenate([[0, 0, 0], mask.reshape(-1)]).astype(np.uint8)).to(dev)
    pal = torch.from_numpy(R.palette(C)[:C].reshape(-1).copy()).to(dev)
    for mix in (0, 1, 2):
        out = torch.zeros(16 + 1 + 3 * h * w, dtype=torch.uint8, device=dev)
        table, offs, _ = ops.render_table([(sbuf.data_ptr() + 1, mbuf.data_ptr() + 3, h, w)], start=0)
        ops.render_batch(torch.frombuffer(bytearray(table), dtype=torch.uint8).to(dev), 1, pal, C, mix, out[1:], None, h * w)
        got = out[1 + offs[0]:1 + offs[0] + 3 * h * w].cpu().numpy().reshape(h, w, 3)
        assert np.array_equal(got, R.render(src, mask, mix, C)), f"mix {mix}"
