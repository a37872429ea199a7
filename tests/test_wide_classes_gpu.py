"""GPU: heads with more than 32 classes (up to 255) and confusion matrices with more than 64 classes (up to 256).

ADE20K (150 classes), Pascal-Context (59) and COCO-Stuff (171) need these.  Every kernel of the wide paths is checked
against the same references and bounds that tests/test_kernels_gpu.py and tests/test_model_gpu.py use for C <= 32."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _global_rel(grads, ref):
    num = sum((grads[k].float().cpu() - ref[k]).double().pow(2).sum().item() for k in ref)
    den = sum(ref[k].double().pow(2).sum().item() for k in ref)
    return (num / den) ** 0.5


def nhwc(x, dev):
    return x.permute(0, 2, 3, 1).contiguous().to(BF).to(dev)


def nchw(x):
    return x.float().permute(0, 3, 1, 2).contiguous().cpu()


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("N,H,W,C", [(2, 16, 32, 33), (1, 24, 40, 64), (2, 8, 16, 65), (1, 5, 7, 150), (2, 16, 24, 150),
                                     (1, 5, 7, 255), (1, 16, 16, 255)])
def test_wide_head_forward_on_tensor_cores(b2u, cuda_device, N, H, W, C):
    """G = ceil(C / 32) groups of [hi | lo] columns, widest N tile, ragged last tile: against fp32 torch on the same bf16
    activations and against the SIMT head."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(C + H)
    x = torch.randn(N, 64, H, W, generator=g).to(BF).float()
    w = torch.randn(C, 64, generator=g) * 0.2
    b = torch.randn(C, generator=g)
    ref = F.conv2d(x, w[:, :, None, None], b)
    xd = nhwc(x, dev)
    wf = ops.pack_head_fprop(w.to(dev))
    assert tuple(wf.shape) == (64 * ops.head_groups(C), 64)
    out = ops.head_fwd_tc(xd, wf, b.to(dev), C)
    assert tuple(out.shape) == (N, C, H, W)
    assert rel(out, ref) <= 2e-5
    simt = ops.head_fwd(xd, w.to(dev), b.to(dev))
    assert rel(simt, ref) <= 2e-5
    assert rel(out, simt) <= 2e-5


@pytest.mark.parametrize("C,use_onehot", [(33, False), (33, True), (150, False), (150, True), (255, False), (255, True)])
def test_wide_head_and_losses_against_oracle(b2u, cuda_device, C, use_onehot):
    """CE / Focal / Dice / f_score and their gradients, the split bf16 dlogits of the tensor-core head backward, the dgrad
    operand and the SIMT head backward at C > 32; class weights with zeros; ignore label = C."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(C + int(use_onehot))
    N, H, W = 2, 24, 40
    xb = nhwc(torch.randn(N, 64, H, W, generator=g).relu(), dev)
    xr = nchw(xb).requires_grad_(True)
    w = (torch.randn(C, 64, 1, 1, generator=g) / 8).requires_grad_(True)
    b = torch.randn(C, generator=g).requires_grad_(True)
    logits = ops.head_fwd(xb, w.detach().reshape(C, 64).contiguous().to(dev), b.detach().to(dev))
    ref = F.conv2d(xr, w, b)
    assert rel(logits, ref) <= 1e-5
    png = torch.randint(0, C + 1, (N, H, W), generator=g)
    # blob-structured labels (as in real masks) in one image, random in the other
    png[0] = torch.randint(0, C + 1, (1, H // 8, W // 8), generator=g).repeat_interleave(8, 1).repeat_interleave(8, 2)[0]
    oh = O.one_hot(png, C)
    weights = 0.5 + torch.rand(C, generator=g) * 2
    weights[::7] = 0
    ce, fo = O.ce_loss(ref, png, weights, C), O.focal_loss(ref, png, weights, C)
    di, fs = O.dice_loss(ref, oh), O.f_score(ref, oh)
    fin = ops.loss_fwd(logits, target=png.to(dev), onehot=oh.to(dev) if use_onehot else None, cls_w=weights.to(dev)).cpu()
    for got, want in zip(fin[:4], (ce, fo, di, fs)):
        assert abs(got.item() - want.item()) <= 2e-5 * max(abs(want.item()), 1e-3)
    for gs, loss in (([1, 0, 0], ce), ([0, 1, 0], fo), ([0, 0, 1], di), ([1, 0, 1], ce + di)):
        gl, = torch.autograd.grad(loss, ref, retain_graph=True)
        dl = ops.loss_bwd(logits, fin.to(dev), torch.tensor(gs, dtype=torch.float32, device=dev), target=png.to(dev),
                          onehot=oh.to(dev) if use_onehot else None, cls_w=weights.to(dev))
        assert rel(dl, gl) <= 2e-4
    gs = torch.tensor([1, 0, 1], dtype=torch.float32, device=dev)
    gl, = torch.autograd.grad(ce + di, ref, retain_graph=True)
    G = ops.head_groups(C)
    d64 = ops.loss_bwd(logits, fin.to(dev), gs, target=png.to(dev), onehot=oh.to(dev) if use_onehot else None,
                       cls_w=weights.to(dev), nhwc64=True).float().cpu()
    assert d64.shape == (N, H, W, 64 * G)
    grp = d64.reshape(N, H, W, G, 2, 32)
    recon = (grp[..., 0, :] + grp[..., 1, :]).reshape(N, H, W, 32 * G)
    assert rel(recon[..., :C].permute(0, 3, 1, 2), gl) <= 2e-5
    assert grp[..., G - 1, :, C - 32 * (G - 1):].abs().sum() == 0          # padded classes of the last group: exact zeros
    wd = ops.pack_head_dgrad(w.detach().reshape(C, 64).contiguous().to(dev)).float().cpu()
    assert tuple(wd.shape) == (64, 64 * G)
    wdg = wd.reshape(64, G, 2, 32)
    want = torch.zeros(64, 32 * G)
    want[:, :C] = w.detach().reshape(C, 64).to(BF).float().t()
    assert torch.equal(wdg[:, :, 0].reshape(64, 32 * G), want) and torch.equal(wdg[:, :, 1], wdg[:, :, 0])
    (ce + di).backward()
    dx, dw, db = ops.head_bwd(gl.contiguous().to(dev), xb, w.detach().reshape(C, 64).contiguous().to(dev))
    assert rel(nchw(dx), xr.grad * (xr > 0)) <= 4e-3
    assert rel(dw, w.grad) <= 1e-4 and rel(db, b.grad) <= 1e-4
    assert torch.equal(ops.argmax_u8(logits).cpu().long(), logits.cpu().argmax(1))


def test_wide_loss_is_deterministic(b2u, cuda_device):
    """Two runs of the wide statistics and backward kernels on the same inputs are bitwise equal."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(3)
    C = 150
    logits = torch.randn(2, C, 64, 96, generator=g).to(dev)
    png = torch.randint(0, C + 1, (2, 64, 96), generator=g).to(dev)
    gs = torch.tensor([1, 1, 1], dtype=torch.float32, device=dev)
    runs = []
    for _ in range(2):
        fin = ops.loss_fwd(logits, target=png, alpha=0.5)
        runs.append((fin, ops.loss_bwd(logits, fin, gs, target=png, nhwc64=True)))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])


@pytest.mark.parametrize("C,H,W,crop,out", [(33, 24, 24, (2, 3, 20, 18), (61, 47)), (150, 64, 64, (8, 0, 48, 64), (90, 120)),
                                            (255, 32, 48, (0, 6, 32, 36), (17, 19))])
def test_wide_softmax_resize_argmax_kernel(b2u, cuda_device, C, H, W, crop, out):
    ops = b2u.ops
    g = torch.Generator().manual_seed(C + H)
    logits = torch.randn(2, C, H, W, generator=g) * 3
    cy, cx, ch, cw = crop
    got = ops.softmax_resize_argmax_u8(logits.to(cuda_device), crop, out).cpu().numpy()
    for n in range(2):
        pr = torch.softmax(logits[n].permute(1, 2, 0), dim=-1).numpy()[cy:cy + ch, cx:cx + cw]
        ref = O.resize_linear_cv2(pr, out[0], out[1])
        top2 = np.sort(ref, axis=-1)[..., -2:]
        confident = (top2[..., 1] - top2[..., 0]) > 1e-4
        assert (got[n] == ref.argmax(-1))[confident].all()
        assert (got[n] == ref.argmax(-1)).mean() >= 0.999


@pytest.mark.parametrize("n", [65, 150, 241, 242, 255, 256])
def test_wide_fast_hist_exact(b2u, cuda_device, n):
    """32-bit shared counters (n <= 241) and 16-bit counters with bounded flushes (n >= 242): uint8 / int32 / int64 inputs,
    ragged lengths, one bin hammered by many pixels, ignored labels, out-of-range predictions -> numpy's ValueError."""
    rng = np.random.default_rng(n)
    L = 512 * 512 * 3 + 13
    a = rng.integers(0, n, size=L)
    b = rng.integers(0, n, size=L)
    a[rng.random(L) < 0.05] = 255 if n < 256 else 300     # ignored ground truth (>= n)
    a[:5000] = 1 % n
    b[:5000] = 0
    a[200000:300000] = n - 1                          # one bin takes 1e5 pixels: > 2^16 in one block for the 16-bit table
    b[200000:300000] = n - 1
    if n < 256:
        au8, bu8 = a.astype(np.uint8), b.astype(np.uint8)
        assert np.array_equal(b2u.fast_hist(au8, bu8, n), O.fast_hist(au8, bu8, n))
    for dt in (np.int32, np.int64):
        ad, bd = a.astype(dt), b.astype(dt)
        ad[17] = -1                                   # negative ground truth is ignored
        assert np.array_equal(b2u.fast_hist(ad, bd, n), O.fast_hist(ad, bd, n))
    a_ok, b_bad = a.astype(np.int64), b.astype(np.int64)
    a_ok[L // 2], b_bad[L // 2] = n - 1, n                # n * a + b == n * n: past the last bin
    hist = b2u.fast_hist_device(a_ok, b_bad, n).cpu().numpy()
    assert hist[-1] == 1
    with pytest.raises(ValueError):
        b2u.fast_hist(a_ok, b_bad, n)


@pytest.mark.parametrize("n", [150, 255])
def test_wide_fast_hist_batch_and_argmax_hist(b2u, cuda_device, n):
    ops, dev = b2u.ops, cuda_device
    rng = np.random.default_rng(7 + n)
    sizes = [512 * 512, 16 * 33 + 9, 16, 100003, 512 * 384]
    pairs, ref = [], np.zeros((n, n), np.int64)
    for i, sz in enumerate(sizes):
        ga = rng.integers(0, n, size=sz).astype(np.uint8)
        ga[rng.random(sz) < (1.0 if i == 2 else 0.03)] = 255
        pb = rng.integers(0, n, size=sz).astype(np.uint8)
        ref += O.fast_hist(ga, pb, n)
        pairs.append((torch.from_numpy(ga).to(dev), torch.from_numpy(pb).to(dev)))
    got = ops.fast_hist_batch(pairs, n, torch.zeros(n * n + 1, dtype=torch.int64, device=dev)).cpu().numpy()
    assert got[-1] == 0 and np.array_equal(got[:-1].reshape(n, n), ref)
    C = n
    g = torch.Generator().manual_seed(C)
    logits = torch.randn(3, C, 64, 96, generator=g)
    logits[0, :, :8] = 0.25                              # ties: class 0 must win
    logits[1, 1, 5:9] = logits[1, 0, 5:9]
    gt = torch.randint(0, n, (3, 64, 96), generator=g, dtype=torch.uint8)
    gt[torch.rand(3, 64, 96, generator=g) < 0.05] = 255
    hist, pred = ops.argmax_hist(logits.to(dev), gt.to(dev), n, want_pred=True)
    want_pred = logits.numpy().argmax(1).astype(np.uint8)
    assert np.array_equal(pred.cpu().numpy(), want_pred)
    h = hist.cpu().numpy()
    assert h[-1] == 0 and np.array_equal(h[:-1].reshape(n, n), O.fast_hist(gt.numpy().reshape(-1), want_pred.reshape(-1), n))


# ------------------------------------------------------------------------------------------------ models
def test_wide_vgg_dropin_matches_oracle(b2u, cuda_device):
    """Unet-VGG16 drop-in at 150 classes (SIMT head backward through autograd) against the fp32 oracle, CASES bounds."""
    dev = cuda_device
    C = 150
    params = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=1)
    weights = torch.ones(C)
    loss_ref, logits_ref, grads_ref = O.train_step(params, imgs, pngs, weights, C, dice=True)
    model = b2u.Unet(num_classes=C, pretrained=False, backbone="vgg")
    model.load_state_dict(params)
    model = model.train().to(dev)
    outputs = model(imgs.to(dev))
    loss = b2u.CE_Loss(outputs, pngs.to(dev), weights.to(dev), num_classes=C) + b2u.Dice_loss(outputs, O.one_hot(pngs, C).to(dev))
    loss.backward()
    assert outputs.shape == logits_ref.shape
    assert rel(outputs, logits_ref) <= 1e-2
    assert abs(loss.item() - loss_ref.item()) <= 1e-2 * abs(loss_ref.item())
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert _global_rel(grads, grads_ref) <= 1e-2


def test_wide_trainer_matches_bf16_storage_model(b2u, cuda_device):
    """UnetTrainer at 150 classes: tensor-core head forward / backward over 5 groups, fused losses; against the bf16-storage
    model, and gradients bitwise reproducible."""
    dev = cuda_device
    C = 150
    params = O.make_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=5)
    lbf, zbf, gbf = O.train_step_bf16_storage(params, imgs, pngs, torch.ones(C), C, dice=True)
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=params, lr=0.0)
    out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert abs(out[0].item() - lbf.item()) <= 1e-4 * abs(lbf.item())
    assert _global_rel(tr.grads, gbf) <= 3e-3
    g1 = {k: v.clone() for k, v in tr.grads.items()}
    tr.train_step(imgs.to(dev), pngs.to(dev))
    assert all(torch.equal(g1[k], tr.grads[k]) for k in g1)


def test_wide_traditional_unet_dropin(b2u, cuda_device):
    """TraditionalUnet (head input 32 channels, padded to 64) at 150 classes, judged like tests/test_model_gpu.py."""
    dev = cuda_device
    C = 150
    sd = O.make_trad_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 32, 64, seed=4)
    weights = torch.ones(C)
    l32, z32, g32, _ = O.trad_train_step(sd, imgs, pngs, weights, C, dice=True)
    lbf, zbf, gbf, _ = O.trad_train_step(sd, imgs, pngs, weights, C, dice=True, bf16_storage=True)
    model = b2u.TraditionalUnet(in_channels=3, num_classes=C)
    model.load_state_dict(sd)
    model = model.train().to(dev)
    outputs = model(imgs.to(dev))
    loss = b2u.CE_Loss(outputs, pngs.to(dev), weights.to(dev), num_classes=C) + b2u.Dice_loss(outputs, O.one_hot(pngs, C).to(dev))
    loss.backward()
    noise_z, noise_g = rel(zbf, z32), _global_rel(gbf, g32)
    assert rel(outputs, z32) <= 1.5 * noise_z and rel(outputs, zbf) <= noise_z
    assert abs(loss.item() - l32.item()) <= 2e-2 * abs(l32.item())
    grads = {k: p.grad for k, p in model.named_parameters()}
    assert _global_rel(grads, g32) <= 1.5 * noise_g and _global_rel(grads, gbf) <= 1.2 * noise_g
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0, model="traditional")
    out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert abs(out[0].item() - l32.item()) <= 2e-2 * abs(l32.item())
    assert _global_rel(tr.grads, g32) <= 1.5 * noise_g


def test_wide_lightweight_unet_dropin(b2u, cuda_device):
    """LightweightUnet at 150 classes: half-resolution logits resized inside the loss, SIMT head backward (fp32 dlogits);
    Dropout2d off on both sides; bounds of tests/test_model_gpu.py::test_lightweight_unet_dropin."""
    dev = cuda_device
    C = 150
    sd = O.make_lw_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=14)
    weights = torch.ones(C)
    l32, z32, g32, _ = O.lw_train_step(sd, imgs, pngs, weights, C, dice=True)
    lbf, zbf, gbf, _ = O.lw_train_step(sd, imgs, pngs, weights, C, dice=True, bf16_storage=True)
    model = b2u.LightweightUnet(num_classes=C)
    model.load_state_dict(sd)
    model = model.train().to(dev)
    for ins in model._engine_for(dev).program:
        if ins["op"] == "drop":
            ins["p"] = 0.0
    outputs = model(imgs.to(dev))
    assert tuple(outputs.shape) == (2, C, 32, 32)
    loss = b2u.CE_Loss(outputs, pngs.to(dev), weights.to(dev), num_classes=C) + b2u.Dice_loss(outputs, O.one_hot(pngs, C).to(dev))
    loss.backward()
    noise_z, noise_g = rel(zbf, z32), _global_rel(gbf, g32)
    assert rel(outputs, z32) <= max(1.5 * noise_z, 1e-2)
    assert abs(loss.item() - l32.item()) <= 1e-2 * abs(l32.item())
    grads = {k: p.grad for k, p in model.named_parameters()}

    def pre_bn_bias(k):
        base = k.rsplit(".", 1)[0]
        return k.endswith(".bias") and (base.endswith(".conv.0") or base.endswith(".conv1") or base.endswith(".conv2"))
    live = {k: v for k, v in grads.items() if not pre_bn_bias(k)}
    assert _global_rel(live, {k: g32[k] for k in live}) <= 1.5 * noise_g
    for k in ("final_conv.3.weight", "final_conv.3.bias"):
        assert rel(grads[k], g32[k]) <= max(2e-2, 2 * noise_z), k


def test_wide_resnet50_trainer(b2u, cuda_device):
    """A GraphEngine BatchNorm family (Unet-ResNet50) at 150 classes through the trainer, with the checks of
    tests/test_model_gpu.py::test_resnet50_frozen_backbone_and_trainer."""
    dev = cuda_device
    C = 150
    sd = O.make_resnet_unet_params(C, seed=11)
    imgs, pngs = O.make_inputs(2, C, 64, 64, seed=2)
    l32, _, g32, _ = O.resnet_unet_train_step(sd, imgs, pngs, torch.ones(C), C, dice=True)
    _, _, gbf, _ = O.resnet_unet_train_step(sd, imgs, pngs, torch.ones(C), C, dice=True, bf16_storage=True)
    tr = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=0.0, model="unet_resnet50")
    out = tr.train_step(imgs.to(dev), pngs.to(dev)).cpu()
    assert abs(out[0].item() - l32.item()) <= 1e-2 * abs(l32.item())
    assert _global_rel(tr.grads, g32) <= 1.5 * _global_rel(gbf, g32)
    tr3 = b2u.UnetTrainer(num_classes=C, device=dev, state_dict=sd, lr=1e-3, model="unet_resnet50")
    losses = [tr3.train_step(imgs.to(dev), pngs.to(dev))[0].item() for _ in range(6)]
    assert losses[-1] < losses[0]


def test_wide_predictor_get_miou(b2u, cuda_device):
    """Predictor at 150 classes: get_miou's device confusion matrix equals numpy's over the same predicted masks."""
    from PIL import Image
    from unet_pytorch_b200.unet import Unet as Predictor
    C = 150
    pred = Predictor(state_dict=O.make_predictor_params(C, seed=11), num_classes=C, backbone="vgg", input_shape=[96, 128])
    rng = np.random.default_rng(0)
    images = [Image.fromarray(rng.integers(0, 256, (70 + 9 * i, 110 - 7 * i, 3), dtype=np.uint8)) for i in range(3)]
    gts = []
    for im in images:
        gt = rng.integers(0, C, (im.size[1], im.size[0])).astype(np.uint8)
        gt[:5] = 255
        gts.append(gt)
    h, ious, _, _ = pred.get_miou(images, gts)
    want = sum(O.fast_hist(gt.reshape(-1), pred.predict_mask_device(im).cpu().numpy().reshape(-1), C) for im, gt in zip(images, gts))
    assert np.array_equal(h, want)
    assert np.asarray(pred.get_miou_png(images[0])).max() < C
    assert pred.detect_image(images[0]) is not None


def test_wide_fp32_validation_build(b2u, cuda_device):
    """The fp32 validation build at 150 classes: Unet-VGG16 logits and gradients within 1e-5 of the oracle."""
    dev = cuda_device
    C = 150
    b2u.ops.set_validation_fp32(True)
    try:
        params = O.make_params(C, seed=11)
        imgs, pngs = O.make_inputs(2, C, 32, 32, seed=1)
        weights = torch.ones(C)
        loss_ref, logits_ref, grads_ref = O.train_step(params, imgs, pngs, weights, C, dice=True)
        model = b2u.Unet(num_classes=C, pretrained=False, backbone="vgg")
        model.load_state_dict(params)
        model = model.train().to(dev)
        outputs = model(imgs.to(dev))
        loss = b2u.CE_Loss(outputs, pngs.to(dev), weights.to(dev), num_classes=C) + b2u.Dice_loss(outputs, O.one_hot(pngs, C).to(dev))
        loss.backward()
        assert rel(outputs, logits_ref) <= 1e-5
        assert abs(loss.item() - loss_ref.item()) <= 1e-5 * abs(loss_ref.item())
        assert _global_rel({k: p.grad for k, p in model.named_parameters()}, grads_ref) <= 1e-5
    finally:
        b2u.ops.set_validation_fp32(False)
