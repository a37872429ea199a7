"""GPU: the batched predictor -- the device letterbox (csrc/letterbox.cu) against the host letterbox bit for bit, the
batched tail against the single-image tail bit for bit, predict_masks / get_miou against the per-image path, and the
error cases."""
import types

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import pil_bicubic as B
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu


def _image(w, h, seed, mode="RGB"):
    """Smooth colour gradients plus noise (resampling must get both right); converted to `mode`."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 255 // max(w - 1, 1)), (yy * 255 // max(h - 1, 1)), ((xx + yy) * 7) % 256], -1)
    arr = np.clip(base + rng.integers(-40, 41, (h, w, 3)), 0, 255).astype(np.uint8)
    img = Image.fromarray(arr)
    if mode == "P":
        return img.quantize(colors=64)
    return img.convert(mode) if mode != "RGB" else img


def _mixed_images():
    sizes = [(500, 375), (375, 500), (4000, 3000), (512, 512), (256, 256), (1024, 1024), (640, 480), (480, 640), (1, 1),
             (3, 5), (5, 3), (1920, 1080), (1080, 1920), (513, 511), (511, 513), (200, 1200), (1200, 200), (300, 300),
             (777, 333), (333, 777), (512, 100), (100, 512), (64, 48), (48, 64), (1000, 999), (2, 700), (700, 2),
             (512, 384), (384, 512), (127, 129), (10, 1200), (6, 700)]
    imgs = [_image(w, h, seed=i) for i, (w, h) in enumerate(sizes)]
    imgs += [_image(333, 250, 91, "L"), _image(250, 333, 92, "P"), _image(640, 427, 93, "RGBA")]
    return imgs


def _device_letterbox(b2u, prepared, H, W, dev):
    ops = b2u.ops
    srcs = [torch.from_numpy(arr.copy()).to(dev) for _, arr, _ in prepared]
    table, ws_bytes = ops.letterbox_plan([(s.data_ptr(), *geo) for s, (_, _, geo) in zip(srcs, prepared)], H, W)
    tdev = torch.frombuffer(bytearray(table), dtype=torch.uint8).to(dev)
    out = torch.full((len(prepared) + 1, 3, H, W), float("nan"), device=dev)
    ops.letterbox_bicubic(tdev, len(prepared), out, torch.empty(ws_bytes, dtype=torch.uint8, device=dev))
    torch.cuda.synchronize()
    assert torch.isnan(out[-1]).all()                                  # nothing past the batch is written
    return out[:-1].cpu()


@pytest.mark.parametrize("shape", [(512, 512), (384, 640)])
def test_letterbox_kernel_equals_host_letterbox(b2u, cuda_device, shape):
    """35 images of mixed sizes in one launch -- a 4000x3000 source (33-tap filters), an exact 512x512 fit without bars,
    1x1, upscales and downscales, images more than 100 times taller than wide (PIL resamples them vertically first),
    'L' / 'P' / 'RGBA' inputs -- equal the host `_letterbox` tensor (PIL BICUBIC + np.float32 / 255) bit for bit."""
    from unet_pytorch_b200.unet import Unet as Predictor
    H, W = shape
    fake = types.SimpleNamespace(input_shape=[H, W])
    imgs = _mixed_images()
    prepared = [Predictor._prepare(fake, im) for im in imgs]
    got = _device_letterbox(b2u, prepared, H, W, cuda_device)
    for i, im in enumerate(imgs):
        _, ref, nw, nh, oh, ow = Predictor._letterbox(fake, im)
        assert prepared[i][2] == (oh, ow, nh, nw, (H - nh) // 2, (W - nw) // 2)
        assert torch.equal(got[i], ref[0]), f"image {i} ({im.size}, {im.mode})"
    if shape == (512, 512):
        assert torch.equal(got[3], torch.from_numpy(np.asarray(imgs[3], np.float32).transpose(2, 0, 1) / np.float32(255)))
        assert np.array_equal(got[0].numpy(), B.letterbox(np.asarray(imgs[0]), W, H))


@pytest.mark.parametrize("C", [21, 150])
def test_batched_tail_equals_single_image_kernel(b2u, cuda_device, C):
    """b2u_softmax_resize_argmax_u8_batch: per-image crops and output sizes (up- and down-scaled, 1x1, one axis unchanged),
    ragged 16-byte aligned masks in one buffer; every mask equals the single-image kernel's bit for bit and nothing
    between the masks is written."""
    ops, dev = b2u.ops, cuda_device
    H, W = 96, 128
    g = torch.Generator().manual_seed(C)
    crops = [(12, 0, 72, 128), (0, 0, 96, 128), (0, 40, 96, 48), (30, 7, 1, 1), (5, 3, 90, 100), (0, 0, 96, 128)]
    sizes = [(75, 133), (96, 128), (301, 150), (7, 9), (45, 50), (1, 1)]
    logits = (torch.randn(len(crops), C, H, W, generator=g) * 3).to(dev)
    logits[1, :, :10] = 0.0                                            # exact ties: the lowest class wins in both kernels
    table, offs, total = ops.tail_table(crops, sizes, H, W)
    masks = torch.full((total + 16,), 255, dtype=torch.uint8, device=dev)
    ops.softmax_resize_argmax_u8_batch(logits, torch.frombuffer(bytearray(table), dtype=torch.uint8).to(dev), len(crops),
                                       masks, max(s[0] for s in sizes), max(s[1] for s in sizes))
    m = masks.cpu()
    covered = torch.zeros_like(m, dtype=torch.bool)
    for i, (crop, (oh, ow)) in enumerate(zip(crops, sizes)):
        ref = ops.softmax_resize_argmax_u8(logits[i:i + 1].contiguous(), crop, (oh, ow))[0].cpu()
        assert torch.equal(m[offs[i]:offs[i] + oh * ow].view(oh, ow), ref), f"image {i}"
        covered[offs[i]:offs[i] + oh * ow] = True
    assert (m[~covered] == 255).all()
    assert int(m[covered].max()) < C


def _predictor(b2u, backbone, C, shape):
    from unet_pytorch_b200.unet import Unet as Predictor
    if backbone == "vgg":
        sd = O.make_predictor_params(C, seed=11)
    else:
        sd = O.make_resnet_unet_params(C, seed=11)
        sd["final.weight"] = sd["final.weight"] * 150.0               # confident, multi-class maps (see make_predictor_params)
    return Predictor(state_dict=sd, num_classes=C, backbone=backbone, input_shape=list(shape))


def _eval_images(n, seed):
    rng = np.random.default_rng(seed)
    modes = ["RGB"] * 6 + ["L", "RGBA", "P"]
    return [_image(int(rng.integers(40, 400)), int(rng.integers(40, 400)), seed * 100 + i, modes[i % len(modes)]) for i in range(n)]


@pytest.mark.parametrize("backbone", ["vgg", "resnet50"])
def test_predict_masks_equals_per_image_path(b2u, cuda_device, backbone):
    """predict_masks at batch 1, 3 and 16 over 19 images (partial last batches) equals get_miou_png per image, and the
    per-image result equals the host-letterbox path (PIL letterbox -> batch-1 forward -> single-image tail); the
    batched forward gives every image the logits of its batch-1 forward, bit for bit."""
    from unet_pytorch_b200 import ops
    C, shape = 21, (192, 256)
    pred = _predictor(b2u, backbone, C, shape)
    imgs = _eval_images(19, seed=3 if backbone == "vgg" else 4)
    per_image = [np.asarray(pred.get_miou_png(im)) for im in imgs]
    with torch.no_grad():
        for im, m in zip(imgs[:5], per_image):
            _, data, nw, nh, oh, ow = pred._letterbox(im)
            host_path = ops.softmax_resize_argmax_u8(pred.net(data.to(cuda_device)), pred._crop(nw, nh), (oh, ow))[0]
            assert np.array_equal(host_path.cpu().numpy(), m)
    for bs in (1, 3, 16):
        got = pred.predict_masks(imgs, batch_size=bs)
        assert len(got) == len(imgs)
        for i, (g, m) in enumerate(zip(got, per_image)):
            assert g.dtype == np.uint8 and g.shape == (imgs[i].size[1], imgs[i].size[0])
            assert np.array_equal(g, m), f"batch {bs}, image {i}"
    assert len(np.unique(np.concatenate([m.reshape(-1) for m in per_image]))) > 3
    # logits of a batch of 5 against batch-1 forwards of the same device inputs
    with torch.no_grad():
        prepared = [pred._prepare(im) for im in imgs[:5]]
        pred._run_batch(prepared)
        x = pred._input[:5].clone()
        batched = pred.net(x).clone()
        for i in range(5):
            assert torch.equal(batched[i:i + 1], pred.net(x[i:i + 1].contiguous())), f"image {i}"


def test_get_miou_batched(b2u, cuda_device):
    """get_miou's confusion matrix is identical at batch sizes 1, 4 and 16 and equals numpy fast_hist over the per-image
    masks; ignored gt pixels (255) and a size-mismatched pair (skipped) are included."""
    C = 21
    pred = _predictor(b2u, "vgg", C, (128, 160))
    imgs = _eval_images(11, seed=5)
    rng = np.random.default_rng(0)
    masks = [pred.predict_mask(im)[1] for im in imgs]
    gts = []
    for i, m in enumerate(masks):
        gt = np.where(rng.random(m.shape) < 0.7, m, rng.integers(0, C, m.shape)).astype(np.uint8)
        gt[: m.shape[0] // 5] = 255
        gts.append(Image.fromarray(gt) if i % 2 else gt)
    gts[4] = np.zeros((masks[4].shape[0] + 1, masks[4].shape[1]), np.uint8)       # size mismatch: skipped
    want = sum(O.fast_hist(np.asarray(g).reshape(-1), m.reshape(-1), C) for i, (g, m) in enumerate(zip(gts, masks)) if i != 4)
    hists = [pred.get_miou(imgs, gts, batch_size=bs) for bs in (1, 4, 16)]
    for h, ious, recall, precision in hists:
        assert np.array_equal(h, want)
        assert np.allclose(ious, O.per_class_iu(want), equal_nan=True)
    assert want.sum() == sum((np.asarray(g) != 255).sum() for i, g in enumerate(gts) if i != 4)
    assert pred.get_miou(iter(imgs[:3]), iter(gts[:3]))[0].sum() > 0           # any iterables, not only lists


def test_batched_predictor_errors(b2u, cuda_device):
    """Empty images, bad batch sizes, crops outside the logits and short tables are refused; the C entry points check
    their scalar arguments before touching the GPU."""
    ops, lib = b2u.ops, b2u._lib.lib()
    pred = _predictor(b2u, "vgg", 21, (64, 64))
    with pytest.raises(ValueError):
        pred.predict_masks([Image.new("RGB", (0, 0))])
    with pytest.raises(ValueError):
        pred.predict_mask(Image.new("RGB", (10, 0)))
    with pytest.raises(ValueError):
        pred.predict_masks([Image.new("RGB", (8, 8))], batch_size=0)
    with pytest.raises(ValueError):
        pred.get_miou([Image.new("RGB", (8, 8))], [np.zeros((8, 8), np.uint8)], batch_size=0)
    assert pred.predict_masks([]) == []
    logits = torch.zeros(1, 21, 64, 64, device=cuda_device)
    with pytest.raises(ValueError):
        ops.softmax_resize_argmax_u8_batch(logits, torch.zeros(32, dtype=torch.uint8, device=cuda_device), 2,
                                           torch.zeros(64, dtype=torch.uint8, device=cuda_device), 8, 8)
    with pytest.raises(ValueError):
        ops.letterbox_bicubic(torch.zeros(64, dtype=torch.uint8, device=cuda_device), 1,
                              torch.zeros(1, 4, 8, 8, device=cuda_device), torch.zeros(16, dtype=torch.uint8, device=cuda_device))
    assert lib.b2u_softmax_resize_argmax_u8_batch(None, None, 0, 21, 8, 8, None, 8, 8, None) == 1
    assert b"softmax_resize_argmax_batch" in lib.b2u_last_error()
    assert lib.b2u_letterbox_bicubic(None, 0, None, 8, 8, None, 0, None) == 1
    assert b"letterbox_bicubic" in lib.b2u_last_error()
    # the predictor's own results still hold after an error, and predict_mask_device returns a tensor it does not reuse
    im = _image(90, 70, 1)
    a = pred.predict_mask_device(im)
    pred.predict_masks([_image(50, 50, 2)] * 3)
    assert torch.equal(a.cpu(), torch.from_numpy(pred.predict_mask(im)[1]))
