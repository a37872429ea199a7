"""CPU oracle of the UNet hot path -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module;
the product path (unet-pytorch_b200/) never does and fails loudly without its CUDA library.

It restates, function by function, what clolckliang/unet-pytorch computes on this path.  The arithmetic itself
lives in a third-party dependency of the reference that is not vendored in it -- PyTorch (requirements.txt:1,
this image: torch 2.11.0) -- so the restatement is written directly against torch.nn.functional's published
semantics (conv2d cross-correlation with zero padding, max_pool2d, bilinear interpolate with
align_corners=True, cross_entropy with weight/ignore_index, softmax) on fp32 CPU tensors, plus closed forms for
the losses and numpy for the integer histogram.

Parity pin: the reference ships no tests or golden vectors for this path (SURVEY.md 8c), so the oracle is
pinned against outputs of the reference itself: oracle/make_golden.py imports /root/reference, runs its
nets.unet.Unet / nets.unet_training losses / utils.utils_metrics functions on seeded inputs and commits the
results under tests/golden/; tests/test_oracle.py checks this module against those files (<= 1e-5, integers exact).
"""
import numpy as np
import torch
import torch.nn.functional as F

# nets/vgg.py:62-64 cfgs['D'] (the trailing 'M' is dropped by VGG.forward's features[23:-1], nets/vgg.py:30)
VGG_CFG = [64, 64, "M", 128, 128, "M", 256, 256, 256, "M", 512, 512, 512, "M", 512, 512, 512]
VGG_CONV_IDX = [0, 2, 5, 7, 10, 12, 14, 17, 19, 21, 24, 26, 28]
# features[:4], [4:9], [9:16], [16:23], [23:-1]  (nets/vgg.py:26-30): index of the last conv of each slice
FEAT_AFTER = {2: 0, 7: 1, 14: 2, 21: 3, 28: 4}


def param_shapes(num_classes, in_channels=3):
    """state_dict names/shapes of nets/unet.py::Unet(backbone='vgg') in order (44 tensors)."""
    shapes = {}
    cin = in_channels
    it = iter(VGG_CONV_IDX)
    for v in VGG_CFG:
        if v == "M":
            continue
        i = next(it)
        shapes[f"vgg.features.{i}.weight"] = (v, cin, 3, 3)
        shapes[f"vgg.features.{i}.bias"] = (v,)
        cin = v
    in_filters = [192, 384, 768, 1024]      # nets/unet.py:29
    out_filters = [64, 128, 256, 512]       # nets/unet.py:35
    for k in (4, 3, 2, 1):
        shapes[f"up_concat{k}.conv1.weight"] = (out_filters[k - 1], in_filters[k - 1], 3, 3)
        shapes[f"up_concat{k}.conv1.bias"] = (out_filters[k - 1],)
        shapes[f"up_concat{k}.conv2.weight"] = (out_filters[k - 1], out_filters[k - 1], 3, 3)
        shapes[f"up_concat{k}.conv2.bias"] = (out_filters[k - 1],)
    shapes["final.weight"] = (num_classes, 64, 1, 1)
    shapes["final.bias"] = (num_classes,)
    return shapes


def make_params(num_classes, seed=11, in_channels=3, gain=0.5):
    """Deterministic synthetic weights (no checkpoint is shipped for this model, SURVEY.md section 2): tensor k of
    the state_dict is drawn from its own generator seeded seed*1000+k, std = gain * sqrt(2 / fan_in).  gain 0.5 is
    the scale of torch's default Conv2d init (what the reference's decoder starts from); gain 1.0 (full He) keeps
    activations O(1) through all 23 layers and is the harsh case for bf16 (DESIGN.md 5)."""
    params = {}
    for k, (name, shape) in enumerate(param_shapes(num_classes, in_channels).items()):
        g = torch.Generator().manual_seed(seed * 1000 + k)
        if len(shape) == 4:
            fan_in = shape[1] * shape[2] * shape[3]
            params[name] = torch.randn(shape, generator=g) * (gain * (2.0 / fan_in) ** 0.5)
        else:
            params[name] = torch.randn(shape, generator=g) * 0.05
    return params


def make_inputs(n, num_classes, h, w, seed=0, medical=False):
    """Structured synthetic batch (SURVEY.md 8d): low-frequency image field, labels correlated with it, ~2 %
    ignore pixels (= num_classes) unless `medical` (grey image replicated to RGB, binary labels, no ignore)."""
    g = torch.Generator().manual_seed(seed)
    if medical:
        base = F.interpolate(torch.rand(n, 1, max(h // 64, 2), max(w // 64, 2), generator=g), size=(h, w), mode="bilinear",
                             align_corners=True)
        img = (base + 0.1 * torch.rand(n, 1, h, w, generator=g)).clamp(0, 1)
        img = torch.round(img * 255) / 255
        png = (base[:, 0] > 0.5).long()
        return img.repeat(1, 3, 1, 1).contiguous(), png
    fields = F.interpolate(torch.rand(n, num_classes, max(h // 32, 2), max(w // 32, 2), generator=g), size=(h, w),
                           mode="bilinear", align_corners=True)
    png = fields.argmax(1)
    img = torch.stack([fields[:, k % num_classes] for k in range(3)], 1) * 0.7 + 0.3 * torch.rand(n, 3, h, w, generator=g)
    img = torch.round(img.clamp(0, 1) * 255) / 255
    ign = torch.rand(n, h, w, generator=g) < 0.02
    png = torch.where(ign, torch.full_like(png, num_classes), png)
    return img.contiguous(), png.contiguous()


# ----------------------------------------------------------------------------------------------- model
def vgg_features(params, x):
    """VGG.forward (nets/vgg.py:21-31): 13 x [conv3x3 p1 + bias + ReLU] (nets/vgg.py:53-57), MaxPool2d(2,2) (:51)."""
    feats = [None] * 5
    it = iter(VGG_CONV_IDX)
    for v in VGG_CFG:
        if v == "M":
            x = F.max_pool2d(x, kernel_size=2, stride=2)
            continue
        i = next(it)
        x = F.relu(F.conv2d(x, params[f"vgg.features.{i}.weight"], params[f"vgg.features.{i}.bias"], padding=1))
        if i in FEAT_AFTER:
            feats[FEAT_AFTER[i]] = x
    return feats


def unet_up(params, name, skip, low):
    """unetUp.forward (nets/unet.py:16-22): cat([skip, UpsamplingBilinear2d(2)(low)], 1) -> conv+ReLU -> conv+ReLU."""
    up = F.interpolate(low, scale_factor=2, mode="bilinear", align_corners=True)   # nets/unet.py:13
    x = torch.cat([skip, up], 1)                                                    # nets/unet.py:17
    x = F.relu(F.conv2d(x, params[name + ".conv1.weight"], params[name + ".conv1.bias"], padding=1))
    x = F.relu(F.conv2d(x, params[name + ".conv2.weight"], params[name + ".conv2.bias"], padding=1))
    return x


def unet_forward(params, x):
    """Unet.forward, backbone='vgg' (nets/unet.py:62-78)."""
    f1, f2, f3, f4, f5 = vgg_features(params, x)
    up4 = unet_up(params, "up_concat4", f4, f5)
    up3 = unet_up(params, "up_concat3", f3, up4)
    up2 = unet_up(params, "up_concat2", f2, up3)
    up1 = unet_up(params, "up_concat1", f1, up2)
    return F.conv2d(up1, params["final.weight"], params["final.bias"])             # nets/unet.py:58,76


# ----------------------------------------------------------------------------------------------- losses
def ce_loss(logits, target, cls_weights, num_classes):
    """CE_Loss (nets/unet_training.py:9-19): weighted mean NLL over pixels with target != num_classes."""
    n, c, h, w = logits.shape
    z = logits.permute(0, 2, 3, 1).reshape(-1, c)
    y = target.reshape(-1)
    valid = y != num_classes
    lsm = z - torch.logsumexp(z, dim=1, keepdim=True)
    yy = torch.where(valid, y, torch.zeros_like(y))
    wy = cls_weights[yy] * valid
    return -(wy * lsm.gather(1, yy[:, None])[:, 0]).sum() / wy.sum()


def focal_loss(logits, target, cls_weights, num_classes, alpha=0.5, gamma=2):
    """Focal_Loss (nets/unet_training.py:21-36): logpt = -w[y] nll (0 where ignored), mean over ALL pixels."""
    n, c, h, w = logits.shape
    z = logits.permute(0, 2, 3, 1).reshape(-1, c)
    y = target.reshape(-1)
    valid = y != num_classes
    lsm = z - torch.logsumexp(z, dim=1, keepdim=True)
    yy = torch.where(valid, y, torch.zeros_like(y))
    logpt = cls_weights[yy] * valid * lsm.gather(1, yy[:, None])[:, 0]
    pt = torch.exp(logpt)
    if alpha is not None:
        logpt = logpt * alpha
    return (-((1 - pt) ** gamma) * logpt).mean()


def _tp_fp_fn(prob, onehot):
    t = onehot[..., :-1]
    tp = (t * prob).sum((0, 1))
    return tp, prob.sum((0, 1)) - tp, t.sum((0, 1)) - tp


def dice_loss(logits, onehot, beta=1, smooth=1e-5):
    """Dice_loss (nets/unet_training.py:38-56); onehot: (N,H,W,C+1) fp32, last channel = ignore."""
    n, c, h, w = logits.shape
    p = torch.softmax(logits.permute(0, 2, 3, 1).reshape(n, -1, c), -1)
    tp, fp, fn = _tp_fp_fn(p, onehot.reshape(n, -1, c + 1))
    score = ((1 + beta ** 2) * tp + smooth) / ((1 + beta ** 2) * tp + beta ** 2 * fn + fp + smooth)
    return 1 - score.mean()


def f_score(logits, onehot, beta=1, smooth=1e-5, threhold=0.5):
    """f_score (utils/utils_metrics.py:12-31)."""
    n, c, h, w = logits.shape
    p = torch.softmax(logits.permute(0, 2, 3, 1).reshape(n, -1, c), -1)
    p = (p > threhold).float()
    tp, fp, fn = _tp_fp_fn(p, onehot.reshape(n, -1, c + 1))
    score = ((1 + beta ** 2) * tp + smooth) / ((1 + beta ** 2) * tp + beta ** 2 * fn + fp + smooth)
    return score.mean()


def one_hot(png, num_classes):
    """np.eye(num_classes + 1)[png] (utils/dataloader.py:49-50)."""
    return torch.eye(num_classes + 1, device=png.device)[png]


def train_step(params, imgs, pngs, cls_weights, num_classes, dice=True, focal=False):
    """One iteration of fit_one_epoch without the optimizer (utils/utils_fit.py:66-92): forward, CE|Focal (+Dice),
    backward.  Returns (loss, logits, grads dict)."""
    p = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    logits = unet_forward(p, imgs)
    loss = focal_loss(logits, pngs, cls_weights, num_classes) if focal else ce_loss(logits, pngs, cls_weights, num_classes)
    if dice:
        loss = loss + dice_loss(logits, one_hot(pngs, num_classes))
    grads = torch.autograd.grad(loss, list(p.values()))
    return loss.detach(), logits.detach(), dict(zip(p.keys(), grads))


# ----------------------------------------------------------------------------------------------- metrics
def fast_hist(a, b, n):
    """fast_hist (utils/utils_metrics.py:34-43) on flat integer numpy arrays."""
    a = np.asarray(a)
    b = np.asarray(b)
    k = (a >= 0) & (a < n)
    return np.bincount(n * a[k].astype(int) + b[k], minlength=n ** 2).reshape(n, n)


def per_class_iu(hist):
    """utils/utils_metrics.py:45-46"""
    return np.diag(hist) / np.maximum((hist.sum(1) + hist.sum(0) - np.diag(hist)), 1)


def per_class_PA_Recall(hist):
    """utils/utils_metrics.py:48-49"""
    return np.diag(hist) / np.maximum(hist.sum(1), 1)


def per_class_Precision(hist):
    """utils/utils_metrics.py:51-52"""
    return np.diag(hist) / np.maximum(hist.sum(0), 1)


def make_masks(n_masks, n, h=512, w=512, seed=0):
    """Config-5 masks (SURVEY.md 8d): gt = randint(0,n) with 3 % = 255, pred = gt with 20 % re-drawn."""
    rng = np.random.default_rng(seed)
    gt = rng.integers(0, n, size=(n_masks, h, w), dtype=np.uint8)
    pred = gt.copy()
    redraw = rng.random((n_masks, h, w)) < 0.2
    pred[redraw] = rng.integers(0, n, size=int(redraw.sum()), dtype=np.uint8)
    gt[rng.random((n_masks, h, w)) < 0.03] = 255
    return gt, pred


# ----------------------------------------------------------------------------------------------- bf16 storage model
class _RoundBF16(torch.autograd.Function):
    """y = bf16(x) in forward (if `fwd`), g = bf16(g) in backward: models a tensor that is STORED in bf16 in both
    directions.  Used only to separate "bf16 storage noise" from "bug" when judging the CUDA path (DESIGN.md 5)."""

    @staticmethod
    def forward(ctx, x, fwd):
        return x.to(torch.bfloat16).to(x.dtype) if fwd else x.clone()

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(g.dtype), None


def _r(x, fwd=True):
    return _RoundBF16.apply(x, fwd)


def unet_forward_bf16_storage(params, x):
    """unet_forward with every activation / activation-gradient tensor rounded to bf16 where the CUDA path stores
    it in bf16 and weights rounded to bf16 for the convolutions (fp32 accumulation everywhere, fp32 head + loss)."""
    def wq(name):
        w = params[name]
        return w + (w.to(torch.bfloat16).to(w.dtype) - w).detach()     # bf16 value, straight-through gradient

    def conv(x, name):
        return _r(F.relu(F.conv2d(_r(x, fwd=False), wq(name + ".weight"), params[name + ".bias"], padding=1)))

    # the image itself is NOT rounded: the product path feeds it as a two-term bf16 split (hi + lo im2col columns)
    feats = [None] * 5
    it = iter(VGG_CONV_IDX)
    for v in VGG_CFG:
        if v == "M":
            x = F.max_pool2d(x, kernel_size=2, stride=2)
            continue
        i = next(it)
        x = conv(x, f"vgg.features.{i}")
        if i in FEAT_AFTER:
            feats[FEAT_AFTER[i]] = x
    low = feats[4]
    for k in (4, 3, 2, 1):
        up = _r(F.interpolate(low, scale_factor=2, mode="bilinear", align_corners=True))
        low = conv(torch.cat([feats[k - 1], up], 1), f"up_concat{k}.conv1")
        low = conv(low, f"up_concat{k}.conv2")
    return F.conv2d(low, params["final.weight"], params["final.bias"])


def train_step_bf16_storage(params, imgs, pngs, cls_weights, num_classes, dice=True, focal=False):
    p = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    logits = unet_forward_bf16_storage(p, imgs)
    loss = focal_loss(logits, pngs, cls_weights, num_classes) if focal else ce_loss(logits, pngs, cls_weights, num_classes)
    if dice:
        loss = loss + dice_loss(logits, one_hot(pngs, num_classes))
    grads = torch.autograd.grad(loss, list(p.values()))
    return loss.detach(), logits.detach(), dict(zip(p.keys(), grads))


# ----------------------------------------------------------------------------------------------- TraditionalUnet
# nets/TraditionalUnet.py:45-66: DoubleConv prefixes in execution order, with (Cin, Cout)
TRAD_ENC = [("inc", None, 32), ("down1.maxpool_conv.1", 32, 64), ("down2.maxpool_conv.1", 64, 128),
            ("down3.maxpool_conv.1", 128, 256)]
TRAD_DEC = [("up1.conv", 384, 128), ("up2.conv", 192, 64), ("up3.conv", 96, 32)]


def trad_param_shapes(num_classes, in_channels=3):
    """Parameters (not buffers) of TraditionalUnet in state_dict order."""
    shapes = {}
    for prefix, cin, cout in TRAD_ENC + TRAD_DEC:
        cin = in_channels if cin is None else cin
        for idx, ci in ((0, cin), (3, cout)):
            shapes[f"{prefix}.double_conv.{idx}.weight"] = (cout, ci, 3, 3)
            shapes[f"{prefix}.double_conv.{idx}.bias"] = (cout,)
            shapes[f"{prefix}.double_conv.{idx + 1}.weight"] = (cout,)
            shapes[f"{prefix}.double_conv.{idx + 1}.bias"] = (cout,)
    shapes["outc.weight"] = (num_classes, 32, 1, 1)
    shapes["outc.bias"] = (num_classes,)
    return shapes


def make_trad_params(num_classes, seed=11, in_channels=3, gain=1.0):
    """Deterministic synthetic state_dict of TraditionalUnet: convs He-scaled (BatchNorm re-normalises, so the harsh
    full-He scale is harmless here), BN weight 1 + 0.1 N(0,1), BN bias 0.05 N(0,1), fresh running statistics."""
    sd = {}
    for k, (name, shape) in enumerate(trad_param_shapes(num_classes, in_channels).items()):
        g = torch.Generator().manual_seed(seed * 1000 + 500 + k)
        if len(shape) == 4:
            fan_in = shape[1] * shape[2] * shape[3]
            sd[name] = torch.randn(shape, generator=g) * (gain * (2.0 / fan_in) ** 0.5)
        elif ".double_conv.1." in name or ".double_conv.4." in name:
            r = torch.randn(shape, generator=g)
            sd[name] = 1.0 + 0.1 * r if name.endswith("weight") else 0.05 * r
        else:
            sd[name] = torch.randn(shape, generator=g) * 0.05
    for prefix, _, cout in TRAD_ENC + TRAD_DEC:
        for idx in (1, 4):
            sd[f"{prefix}.double_conv.{idx}.running_mean"] = torch.zeros(cout)
            sd[f"{prefix}.double_conv.{idx}.running_var"] = torch.ones(cout)
            sd[f"{prefix}.double_conv.{idx}.num_batches_tracked"] = torch.tensor(0, dtype=torch.long)
    return sd


_BRANCH = {"pin": None, "record": None}


class branch:
    """Context manager (test aid): inside it every ReLU / max-pool site of the BatchNorm families replays the decisions in `pin`
    ({site: bool mask | arg-max indices}) and / or stores its own in `record`.  Sites are keyed by the BatchNorm name (conv -> BN
    -> ReLU), the conv weight name (conv -> ReLU), the residual block's "<prefix>.out" (join + ReLU) and "p<i>" / "pool<k>" /
    "pool" for the max-pools, i.e. the tensor names of the CUDA engine's program.  Pinning removes the only discontinuities of
    the loss, so two precisions can be compared on one smooth branch."""

    def __init__(self, pin=None, record=None):
        self.new = {"pin": pin, "record": record}

    def __enter__(self):
        self.old = dict(_BRANCH)
        _BRANCH.update(self.new)
        return self

    def __exit__(self, *exc):
        _BRANCH.update(self.old)


def _pinned_relu(y, key, pin=None, record=None):
    """F.relu(y); pin (test aid): {key: bool mask} keeps exactly these elements instead, record receives this run's own mask."""
    pin = _BRANCH["pin"] if pin is None else pin
    record = _BRANCH["record"] if record is None else record
    if record is not None:
        record[key] = (y > 0).detach()
    return F.relu(y) if pin is None else y * pin[key].to(y.dtype)


def _pinned_max_pool(x, key, pool_indices=None, record=None, kernel=2, stride=2, ceil_mode=False):
    """F.max_pool2d(x, kernel, stride, ceil_mode=...); pool_indices (test aid, like relu_masks): {key: flat arg-max indices from
    return_indices=True} pins which element of each window passes (two precisions may order a near-tie differently)."""
    pool_indices = _BRANCH["pin"] if pool_indices is None else pool_indices
    record = _BRANCH["record"] if record is None else record
    if pool_indices is None:
        y, idx = F.max_pool2d(x, kernel, stride, ceil_mode=ceil_mode, return_indices=True)
    else:
        idx = pool_indices[key]
        y = x.flatten(2).gather(2, idx.flatten(2)).view(idx.shape)
    if record is not None:
        record[key] = idx.detach()
    return y


def _double_conv(sd, prefix, x, training, stats, bf16):
    """DoubleConv.forward (nets/TraditionalUnet.py:5-18); BatchNorm2d with torch defaults (eps 1e-5, momentum 0.1).
    The ReLU sites are keyed by their BatchNorm's name for oracle.branch."""
    for idx in (0, 3):
        w, b = sd[f"{prefix}.double_conv.{idx}.weight"], sd[f"{prefix}.double_conv.{idx}.bias"]
        bn = f"{prefix}.double_conv.{idx + 1}"
        if bf16:
            w = w + (w.to(torch.bfloat16).to(w.dtype) - w).detach()
            x = _r(x, fwd=False)
        z = F.conv2d(x, w, b, padding=1)
        if bf16:
            c = stats[bn + ".running_mean"].detach().clone().view(1, -1, 1, 1) if training else 0.0      # see _center
            z = _r(z - c) + c
        rm, rv = stats[bn + ".running_mean"], stats[bn + ".running_var"]
        y = F.batch_norm(z, rm, rv, sd[bn + ".weight"], sd[bn + ".bias"], training, 0.1, 1e-5)
        if training:
            stats[bn + ".num_batches_tracked"] = stats[bn + ".num_batches_tracked"] + 1
        x = _pinned_relu(y, bn)
        if bf16:
            x = _r(x)
    return x


def trad_forward(sd, x, training=True, stats=None, bf16_storage=False):
    """TraditionalUnet.forward (nets/TraditionalUnet.py:79-93).  stats: dict of BN buffers, updated in place when
    training (defaults to clones of the buffers in sd)."""
    if stats is None:
        stats = {k: v.clone() for k, v in sd.items() if "running_" in k or "num_batches" in k}
    feats = []          # (the image is not rounded: two-term bf16 split in the product path)
    for i, (prefix, _, _) in enumerate(TRAD_ENC):
        if i > 0:
            x = _pinned_max_pool(x, f"pool{i}")                                  # Down, :24-27
        x = _double_conv(sd, prefix, x, training, stats, bf16_storage)
        feats.append(x)
    for i, (prefix, _, _) in enumerate(TRAD_DEC):
        up = F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True)   # Up.up, :36
        if bf16_storage:
            up = _r(up)
        x = _double_conv(sd, prefix, torch.cat([feats[2 - i], up], 1), training, stats, bf16_storage)   # :40-42
    return F.conv2d(x, sd["outc.weight"], sd["outc.bias"]), stats                # :66, :92


def trad_train_step(sd, imgs, pngs, cls_weights, num_classes, dice=True, focal=False, bf16_storage=False):
    """One iteration of the TraditionalUnet_Train.py loop without the optimizer: returns (loss, logits, grads, stats)."""
    p = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.clone())
         for k, v in sd.items()}
    logits, stats = trad_forward(p, imgs, training=True, bf16_storage=bf16_storage)
    loss = focal_loss(logits, pngs, cls_weights, num_classes) if focal else ce_loss(logits, pngs, cls_weights, num_classes)
    if dice:
        loss = loss + dice_loss(logits, one_hot(pngs, num_classes))
    names = [k for k, v in p.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [p[k] for k in names])
    return loss.detach(), logits.detach(), dict(zip(names, grads)), stats


# ----------------------------------------------------------------------------------------------- Unet-ResNet50
RESNET_LAYERS = [(64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)]     # planes, blocks, stride (nets/resnet.py:115-121)


def resnet_unet_param_shapes(num_classes):
    """Parameters of Unet(backbone='resnet50') in state_dict order (181 tensors, 43,934,101 elements at 21 classes)."""
    sh = {"resnet.conv1.weight": (64, 3, 7, 7), "resnet.bn1.weight": (64,), "resnet.bn1.bias": (64,)}
    inpl = 64
    for li, (planes, blocks, stride) in enumerate(RESNET_LAYERS, start=1):
        for b in range(blocks):
            p = f"resnet.layer{li}.{b}"
            sh[p + ".conv1.weight"] = (planes, inpl, 1, 1)
            sh[p + ".bn1.weight"] = (planes,); sh[p + ".bn1.bias"] = (planes,)
            sh[p + ".conv2.weight"] = (planes, planes, 3, 3)
            sh[p + ".bn2.weight"] = (planes,); sh[p + ".bn2.bias"] = (planes,)
            sh[p + ".conv3.weight"] = (planes * 4, planes, 1, 1)
            sh[p + ".bn3.weight"] = (planes * 4,); sh[p + ".bn3.bias"] = (planes * 4,)
            if b == 0:
                sh[p + ".downsample.0.weight"] = (planes * 4, inpl, 1, 1)
                sh[p + ".downsample.1.weight"] = (planes * 4,); sh[p + ".downsample.1.bias"] = (planes * 4,)
            inpl = planes * 4
    in_filters, out_filters = [192, 512, 1024, 3072], [64, 128, 256, 512]      # nets/unet.py:31-35
    for k in (4, 3, 2, 1):
        sh[f"up_concat{k}.conv1.weight"] = (out_filters[k - 1], in_filters[k - 1], 3, 3)
        sh[f"up_concat{k}.conv1.bias"] = (out_filters[k - 1],)
        sh[f"up_concat{k}.conv2.weight"] = (out_filters[k - 1], out_filters[k - 1], 3, 3)
        sh[f"up_concat{k}.conv2.bias"] = (out_filters[k - 1],)
    for i in (1, 3):
        sh[f"up_conv.{i}.weight"] = (64, 64, 3, 3); sh[f"up_conv.{i}.bias"] = (64,)
    sh["final.weight"] = (num_classes, 64, 1, 1); sh["final.bias"] = (num_classes,)
    return sh


def make_resnet_unet_params(num_classes, seed=11, gain=1.0, dec_gain=0.5):
    """Deterministic synthetic state_dict: encoder convs He-scaled (BatchNorm follows), BN weight 1 + 0.1 N, bias 0.05 N,
    decoder convs at the default-init scale (gain 0.5), fresh running statistics."""
    sd = {}
    for k, (name, shape) in enumerate(resnet_unet_param_shapes(num_classes).items()):
        g = torch.Generator().manual_seed(seed * 1000 + 2000 + k)
        if len(shape) == 4:
            fan_in = shape[1] * shape[2] * shape[3]
            gn = gain if name.startswith("resnet.") else dec_gain
            sd[name] = torch.randn(shape, generator=g) * (gn * (2.0 / fan_in) ** 0.5)
        elif name.startswith("resnet.") and name.endswith(".weight"):
            sd[name] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:
            sd[name] = 0.05 * torch.randn(shape, generator=g)
    for name, shape in list(resnet_unet_param_shapes(num_classes).items()):
        if name.startswith("resnet.") and len(shape) == 1 and name.endswith(".weight"):
            base = name[:-len(".weight")]
            sd[base + ".running_mean"] = torch.zeros(shape)
            sd[base + ".running_var"] = torch.ones(shape)
            sd[base + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)
    return sd


def _rn_bn(sd, stats, name, z, training, relu, res=None, bf16=False):
    y = F.batch_norm(z, stats[name + ".running_mean"], stats[name + ".running_var"], sd[name + ".weight"], sd[name + ".bias"],
                     training, 0.1, 1e-5)
    if training:
        stats[name + ".num_batches_tracked"] = stats[name + ".num_batches_tracked"] + 1
    if res is not None:
        y = y + res
    if relu:
        y = _pinned_relu(y, name)
    return _r(y) if bf16 else y


def _center(stats, bn, training):
    """Storage model of the product path: in training a conv output read only by a BatchNorm is stored as
    bf16(z - running_mean) (the shift rides in the conv bias in fp32; BatchNorm is shift-invariant)."""
    return stats[bn + ".running_mean"].detach().clone().view(1, -1, 1, 1) if training else None


def _rn_conv(sd, name, x, stride=1, padding=0, bias=None, bf16=False, center=None):
    w = sd[name]
    if bf16:
        w = w + (w.to(torch.bfloat16).to(w.dtype) - w).detach()
        x = _r(x, fwd=False)
    z = F.conv2d(x, w, bias, stride=stride, padding=padding)
    if bf16 and center is not None:
        return _r(z - center) + center
    return _r(z) if bf16 else z


def resnet_unet_forward(sd, x, training=True, stats=None, bf16_storage=False):
    """Unet.forward with backbone='resnet50' (nets/unet.py:62-78, nets/resnet.py:151-176, 77-97).  For oracle.branch the ReLU
    sites are keyed by BatchNorm name (encoder) or conv weight name (decoder), the stem max-pool by "pool"."""
    b = bf16_storage
    if stats is None:
        stats = {k: v.clone() for k, v in sd.items() if "running_" in k or "num_batches" in k}
    if b:
        x = _r(x)
    z = _rn_conv(sd, "resnet.conv1.weight", x, stride=2, padding=3, bf16=b, center=_center(stats, "resnet.bn1", training))   # resnet.py:166
    feat1 = _rn_bn(sd, stats, "resnet.bn1", z, training, True, bf16=b)
    x = _pinned_max_pool(feat1, "pool", kernel=3, stride=2, ceil_mode=True)                         # resnet.py:113,170
    feats = [feat1]
    for li, (planes, blocks, stride) in enumerate(RESNET_LAYERS, start=1):
        for bi in range(blocks):
            p = f"resnet.layer{li}.{bi}"
            s = stride if bi == 0 else 1
            out = _rn_bn(sd, stats, p + ".bn1", _rn_conv(sd, p + ".conv1.weight", x, bf16=b, center=_center(stats, p + ".bn1", training)), training, True, bf16=b)
            out = _rn_bn(sd, stats, p + ".bn2", _rn_conv(sd, p + ".conv2.weight", out, stride=s, padding=1, bf16=b, center=_center(stats, p + ".bn2", training)), training, True, bf16=b)
            z3 = _rn_conv(sd, p + ".conv3.weight", out, bf16=b, center=_center(stats, p + ".bn3", training))
            idn = x
            if bi == 0:
                idn = _rn_bn(sd, stats, p + ".downsample.1", _rn_conv(sd, p + ".downsample.0.weight", x, stride=s, bf16=b, center=_center(stats, p + ".downsample.1", training)),
                             training, False, bf16=b)
            x = _rn_bn(sd, stats, p + ".bn3", z3, training, True, res=idn, bf16=b)            # resnet.py:89-95
        feats.append(x)

    def up_stage(name, skip, low):
        up = F.interpolate(low, scale_factor=2, mode="bilinear", align_corners=True)
        if b:
            up = _r(up)
        y = torch.cat([skip, up], 1)
        for cv in ("conv1", "conv2"):
            y = _pinned_relu(
                _rn_conv(sd, f"{name}.{cv}.weight", y, padding=1, bias=sd[f"{name}.{cv}.bias"], bf16=False) if not b else
                F.conv2d(_r(y, fwd=False), sd[f"{name}.{cv}.weight"] + (sd[f"{name}.{cv}.weight"].to(torch.bfloat16).float() - sd[f"{name}.{cv}.weight"]).detach(),
                         sd[f"{name}.{cv}.bias"], padding=1), f"{name}.{cv}.weight")
            if b:
                y = _r(y)
        return y
    up4 = up_stage("up_concat4", feats[3], feats[4])
    up3 = up_stage("up_concat3", feats[2], up4)
    up2 = up_stage("up_concat2", feats[1], up3)
    up1 = up_stage("up_concat1", feats[0], up2)
    y = F.interpolate(up1, scale_factor=2, mode="bilinear", align_corners=True)                     # up_conv, unet.py:48-54
    if b:
        y = _r(y)
    for i in (1, 3):
        w = sd[f"up_conv.{i}.weight"]
        if b:
            w = w + (w.to(torch.bfloat16).float() - w).detach()
            y = _r(y, fwd=False)
        y = _pinned_relu(F.conv2d(y, w, sd[f"up_conv.{i}.bias"], padding=1), f"up_conv.{i}.weight")
        if b:
            y = _r(y)
    return F.conv2d(y, sd["final.weight"], sd["final.bias"]), stats


def resnet_unet_train_step(sd, imgs, pngs, cls_weights, num_classes, dice=True, focal=False, bf16_storage=False):
    p = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.clone())
         for k, v in sd.items()}
    logits, stats = resnet_unet_forward(p, imgs, training=True, bf16_storage=bf16_storage)
    loss = focal_loss(logits, pngs, cls_weights, num_classes) if focal else ce_loss(logits, pngs, cls_weights, num_classes)
    if dice:
        loss = loss + dice_loss(logits, one_hot(pngs, num_classes))
    names = [k for k, v in p.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [p[k] for k in names])
    return loss.detach(), logits.detach(), dict(zip(names, grads)), stats


# ----------------------------------------------------------------------------------------------- UltraLightweightUnet family
# name: (stage widths, minimum mid channels, SE reduced-channel rule or None, bridge Dropout2d p)
ULU_VARIANTS = {
    "ultralight": ((32, 64, 128, 256, 512), 8, None, 0.0),                                   # nets/UltraLightweightUnet.py:57-108
    "ultralight_large": ((64, 128, 256, 512, 1024), 16, lambda c: max(8, c // 4), 0.2),      # nets/UltraLightweightUnet_large.py:55-113
    "ultralight_large_optimized": ((44, 88, 176, 352, 704), 16, lambda c: max(8, c // 4), 0.15),   # ..._large_optimized.py:51-109
}


def ulu_param_shapes(num_classes, variant):
    """state_dict-ordered trainable tensors (module registration order: enc1-4, bridge, dec4-1, final, se1-4)."""
    widths, mid_min, se_rule, _ = ULU_VARIANTS[variant]
    sh = {}

    def block(p, cin, cout):            # LightConvBlock, nets/UltraLightweightUnet_large.py:19-33
        mid = max(mid_min, cout // 2)
        sh[p + ".conv.0.weight"] = (mid, cin, 1, 1); sh[p + ".conv.0.bias"] = (mid,)
        sh[p + ".conv.1.weight"] = (mid,); sh[p + ".conv.1.bias"] = (mid,)
        sh[p + ".conv.3.depthwise.weight"] = (mid, 1, 3, 3); sh[p + ".conv.3.depthwise.bias"] = (mid,)
        sh[p + ".conv.3.pointwise.weight"] = (cout, mid, 1, 1); sh[p + ".conv.3.pointwise.bias"] = (cout,)
        sh[p + ".conv.4.weight"] = (cout,); sh[p + ".conv.4.bias"] = (cout,)

    cin = 3
    for i in range(4):
        block(f"enc{i + 1}", cin, widths[i]); cin = widths[i]
    block("bridge", widths[3], widths[4])
    for k in (4, 3, 2, 1):
        block(f"dec{k}", widths[k] + widths[k - 1], widths[k - 1])
    sh["final.weight"] = (num_classes, widths[0], 1, 1); sh["final.bias"] = (num_classes,)
    if se_rule is not None:
        for i in range(4):
            c, r = widths[i], se_rule(widths[i])
            sh[f"se{i + 1}.fc.0.weight"] = (r, c); sh[f"se{i + 1}.fc.0.bias"] = (r,)
            sh[f"se{i + 1}.fc.2.weight"] = (c, r); sh[f"se{i + 1}.fc.2.bias"] = (c,)
    return sh


def make_ulu_params(num_classes, variant, seed=11):
    """Deterministic synthetic state_dict: He-scaled 1x1 convs (BatchNorm follows each), depthwise taps 1/3 (1 + 0.5 N),
    BN weight 1 + 0.1 N and bias 0.5 + 0.05 N, other biases 0.05 N, SE linears at 1/sqrt(fan_in), fresh running statistics."""
    sd = {}
    shapes = ulu_param_shapes(num_classes, variant)
    for k, (name, shape) in enumerate(shapes.items()):
        g = torch.Generator().manual_seed(seed * 1000 + 5000 + k)
        is_bn = (".conv.1." in name or ".conv.4." in name)
        if name.endswith("depthwise.weight"):
            # smoothing-like filters (positive mean): random-sign 3x3 taps act as high-pass filters on the smooth feature
            # maps and amplify bf16 storage rounding ~4x, which would only loosen the parity tolerances
            sd[name] = (1.0 / 3.0) * (1.0 + 0.5 * torch.randn(shape, generator=g))
        elif len(shape) == 4:
            fan_in = shape[1] * shape[2] * shape[3]
            gn = 0.5 if name == "final.weight" else 1.0
            sd[name] = torch.randn(shape, generator=g) * (gn * (2.0 / fan_in) ** 0.5)
        elif len(shape) == 2:
            sd[name] = torch.randn(shape, generator=g) * (1.0 / shape[1]) ** 0.5
        elif is_bn and name.endswith(".weight"):
            sd[name] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        elif is_bn:
            sd[name] = 0.5 + 0.05 * torch.randn(shape, generator=g)      # beta > 0: most units stay alive after the ReLU
        else:
            sd[name] = 0.05 * torch.randn(shape, generator=g)
        if is_bn and name.endswith(".bias"):
            base = name[:-len(".bias")]
            sd[base + ".running_mean"] = torch.zeros(shape)
            sd[base + ".running_var"] = torch.ones(shape)
            sd[base + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)
    return sd


def _ulu_block(sd, stats, p, x, training, b):
    """LightConvBlock: 1x1 conv, BN, ReLU, depthwise 3x3 (+bias), 1x1 conv, BN, ReLU.  bf16 storage model: the CUDA path
    stores conv outputs, BN outputs and the depthwise output in bf16, weights of the tensor-core 1x1 convs in bf16; the
    depthwise weights stay fp32."""
    z = _rn_conv(sd, p + ".conv.0.weight", x, bias=sd[p + ".conv.0.bias"], bf16=b, center=_center(stats, p + ".conv.1", training))
    y = _rn_bn(sd, stats, p + ".conv.1", z, training, True, bf16=b)
    wdw = sd[p + ".conv.3.depthwise.weight"]
    d = F.conv2d(_r(y, fwd=False) if b else y, wdw, sd[p + ".conv.3.depthwise.bias"], padding=1, groups=wdw.shape[0])
    if b:
        d = _r(d)
    z = _rn_conv(sd, p + ".conv.3.pointwise.weight", d, bias=sd[p + ".conv.3.pointwise.bias"], bf16=b, center=_center(stats, p + ".conv.4", training))
    return _rn_bn(sd, stats, p + ".conv.4", z, training, True, bf16=b)


def _ulu_se(sd, name, x, b):
    """LightSEBlock (nets/UltraLightweightUnet_large.py:36-52): x * sigmoid(fc2(relu(fc1(avgpool(x)))))."""
    y = x.mean(dim=(2, 3))
    y = F.relu(F.linear(y, sd[name + ".fc.0.weight"], sd[name + ".fc.0.bias"]))
    y = torch.sigmoid(F.linear(y, sd[name + ".fc.2.weight"], sd[name + ".fc.2.bias"]))
    out = x * y[:, :, None, None]
    return _r(out) if b else out


def ulu_forward(sd, x, variant, training=True, stats=None, bf16_storage=False, drop_mask=None):
    """forward() of the three UltraLightweightUnet modules.  drop_mask: the [N, C_bridge] Dropout2d multiplier (already
    divided by 1-p) to apply in training; None = no dropout (eval, or the base variant, whose forward never calls it)."""
    widths, _, se_rule, p_drop = ULU_VARIANTS[variant]
    b = bf16_storage
    if stats is None:
        stats = {k: v.clone() for k, v in sd.items() if "running_" in k or "num_batches" in k}
    skips = []          # (the image is not rounded: two-term bf16 split in the product path)
    for i in range(1, 5):
        if i > 1:
            x = _pinned_max_pool(x, f"p{i}")
        x = _ulu_block(sd, stats, f"enc{i}", x, training, b)
        if se_rule is not None:
            x = _ulu_se(sd, f"se{i}", x, b)
        skips.append(x)
    x = _ulu_block(sd, stats, "bridge", _pinned_max_pool(x, "p5"), training, b)
    if training and p_drop > 0 and drop_mask is not None:
        x = x * drop_mask[:, :, None, None]
        if b:
            x = _r(x)
    for k in (4, 3, 2, 1):
        skip = skips[k - 1]
        up = F.interpolate(x, size=skip.shape[2:], mode="bilinear", align_corners=True)
        if b:
            up = _r(up)
        x = _ulu_block(sd, stats, f"dec{k}", torch.cat([up, skip], 1), training, b)
    logits = F.conv2d(x, sd["final.weight"], sd["final.bias"])
    return logits, stats        # the trailing interpolate to the input size is the identity (same size, align_corners)


def ulu_train_step(sd, imgs, pngs, cls_weights, num_classes, variant, dice=True, focal=False, bf16_storage=False, drop_mask=None):
    p = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.clone())
         for k, v in sd.items()}
    logits, stats = ulu_forward(p, imgs, variant, training=True, bf16_storage=bf16_storage, drop_mask=drop_mask)
    loss = focal_loss(logits, pngs, cls_weights, num_classes) if focal else ce_loss(logits, pngs, cls_weights, num_classes)
    if dice:
        loss = loss + dice_loss(logits, one_hot(pngs, num_classes))
    names = [k for k, v in p.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [p[k] for k in names])
    return loss.detach(), logits.detach(), dict(zip(names, grads)), stats


# ----------------------------------------------------------------------------------------------- ImprovedSegNet (RepVGG_Unet)
def _isn_block(sd, stats, p, x, training, deploy):
    """LightweightConvBlock(use_repvgg=True) (nets/RepVGG_Unet.py): 1x1 conv (+bias), BN, ReLU, then RepVGGBlock(mid -> out).
    Training form: relu(bn1(conv3x3(y)) + bn2(conv1x1(y))), both convs bias-free (no identity branch: mid != out in every
    block); deploy form: relu(reparam_conv(y))."""
    y = _rn_bn(sd, stats, p + ".conv.1", F.conv2d(x, sd[p + ".conv.0.weight"], sd[p + ".conv.0.bias"]), training, True)
    r = p + ".conv.3"
    if deploy:
        return F.relu(F.conv2d(y, sd[r + ".reparam_conv.weight"], sd[r + ".reparam_conv.bias"], padding=1))
    b3 = _rn_bn(sd, stats, r + ".bn1", F.conv2d(y, sd[r + ".conv1.weight"], padding=1), training, False)
    b1 = _rn_bn(sd, stats, r + ".bn2", F.conv2d(y, sd[r + ".conv2.weight"]), training, False)
    return F.relu(b3 + b1)


def isn_forward(sd, x, training=True, stats=None, deploy=False):
    """ImprovedSegNet(use_repvgg=True).forward without Dropout: the topology of UltraLightweightUnet_large_optimized
    (ulu_forward: widths 44-88-176-352-704, SE after each encoder stage, cat[upsampled, skip]) with LightweightConvBlock in
    place of LightConvBlock.  deploy=True runs the re-parameterised blocks (isn_deploy_params)."""
    if stats is None:
        stats = {k: v.clone() for k, v in sd.items() if "running_" in k or "num_batches" in k}
    skips = []
    for i in range(1, 5):
        if i > 1:
            x = _pinned_max_pool(x, f"p{i}")
        x = _ulu_se(sd, f"se{i}", _isn_block(sd, stats, f"enc{i}", x, training, deploy), False)
        skips.append(x)
    x = _isn_block(sd, stats, "bridge", _pinned_max_pool(x, "p5"), training, deploy)
    for k in (4, 3, 2, 1):
        skip = skips[k - 1]
        up = F.interpolate(x, size=skip.shape[2:], mode="bilinear", align_corners=True)
        x = _isn_block(sd, stats, f"dec{k}", torch.cat([up, skip], 1), training, deploy)
    return F.conv2d(x, sd["final.weight"], sd["final.bias"]), stats


def isn_deploy_params(sd, eps=1e-5):
    """switch_to_deploy (nets/RepVGG_Unet.py): every RepVGGBlock's conv3x3 + BN and conv1x1 + BN branches, the BatchNorms in
    eval form, become one conv3x3 with bias (`reparam_conv`); the 1x1 kernel sits at the centre tap.  The training-form
    tensors stay in the state_dict."""
    out = dict(sd)
    for key in [k for k in sd if k.endswith(".conv.3.conv1.weight")]:
        r = key[:-len(".conv1.weight")]
        folded = []
        for conv, bn in ((".conv1", ".bn1"), (".conv2", ".bn2")):
            scale = sd[r + bn + ".weight"] / torch.sqrt(sd[r + bn + ".running_var"] + eps)
            w = sd[r + conv + ".weight"] * scale.view(-1, 1, 1, 1)
            folded.append((F.pad(w, (1, 1, 1, 1)) if w.shape[-1] == 1 else w, sd[r + bn + ".bias"] - sd[r + bn + ".running_mean"] * scale))
        out[r + ".reparam_conv.weight"] = folded[0][0] + folded[1][0]
        out[r + ".reparam_conv.bias"] = folded[0][1] + folded[1][1]
    return out


# ----------------------------------------------------------------------------------------------- LightweightUnet
LW_WIDTHS = (24, 48, 96, 192, 384)                     # nets/LightWeightUnet.py:62-90


def resize_logits(logits, ht, wt):
    """The losses' `if h != ht and w != wt: F.interpolate(..., align_corners=True)` (nets/unet_training.py:12-13, 24-25, 41-42)."""
    if logits.shape[2] != ht and logits.shape[3] != wt:
        return F.interpolate(logits, size=(ht, wt), mode="bilinear", align_corners=True)
    return logits


def lw_param_shapes(num_classes, in_channels=3):
    sh = {}

    def conv_block(p, cin, cout):
        sh[p + ".conv.0.weight"] = (cout, cin, 3, 3); sh[p + ".conv.0.bias"] = (cout,)
        sh[p + ".conv.1.weight"] = (cout,); sh[p + ".conv.1.bias"] = (cout,)

    def res_block(p, c):
        for i in ("1", "2"):
            sh[f"{p}.conv{i}.weight"] = (c, c, 3, 3); sh[f"{p}.conv{i}.bias"] = (c,)
            sh[f"{p}.bn{i}.weight"] = (c,); sh[f"{p}.bn{i}.bias"] = (c,)
        # registration order in the reference: conv1, bn1, conv2, bn2, se
        sh[p + ".se.fc.0.weight"] = (c // 4, c); sh[p + ".se.fc.0.bias"] = (c // 4,)
        sh[p + ".se.fc.2.weight"] = (c, c // 4); sh[p + ".se.fc.2.bias"] = (c,)

    cin = in_channels
    for k, w in enumerate(LW_WIDTHS, start=1):
        conv_block(f"backbone.stage{k}.0", cin, w); res_block(f"backbone.stage{k}.1", w); cin = w
    for k, (cin, cout) in zip((4, 3, 2, 1), ((576, 192), (288, 96), (144, 48), (72, 24))):
        conv_block(f"up_concat{k}.conv.0", cin, cout); res_block(f"up_concat{k}.conv.1", cout)
    conv_block("final_conv.0", 24, 24); res_block("final_conv.2", 24)
    sh["final_conv.3.weight"] = (num_classes, 24, 1, 1); sh["final_conv.3.bias"] = (num_classes,)
    # state_dict order inside a ResidualBlock is conv1, bn1, conv2, bn2 (weights and biases interleaved per module)
    ordered = {}
    for name in sh:
        ordered[name] = sh[name]
    return _lw_reorder(ordered)


def _lw_reorder(sh):
    """conv1.{w,b}, bn1.{w,b}, conv2.{w,b}, bn2.{w,b}, se.* -- the per-module order nn.Module.state_dict() yields."""
    out, done = {}, set()
    names = list(sh)
    for n in names:
        if n in done:
            continue
        if ".conv1.weight" in n:
            p = n[:-len(".conv1.weight")]
            for k in ("conv1.weight", "conv1.bias", "bn1.weight", "bn1.bias", "conv2.weight", "conv2.bias", "bn2.weight", "bn2.bias",
                      "se.fc.0.weight", "se.fc.0.bias", "se.fc.2.weight", "se.fc.2.bias"):
                out[p + "." + k] = sh[p + "." + k]; done.add(p + "." + k)
        else:
            out[n] = sh[n]; done.add(n)
    return out


def make_lw_params(num_classes, seed=11):
    """Deterministic synthetic state_dict: He-scaled 3x3 convs (a BatchNorm follows each), BN weight 1 + 0.1 N and bias
    0.5 + 0.05 N (0.05 N for bn2, whose output feeds the residual sum), conv biases 0.05 N, SE linears at 1/sqrt(fan_in),
    head at half the He scale, fresh running statistics."""
    sd = {}
    for k, (name, shape) in enumerate(lw_param_shapes(num_classes).items()):
        g = torch.Generator().manual_seed(seed * 1000 + 7000 + k)
        base_ = name.rsplit(".", 1)[0]
        is_bn = base_.endswith(".conv.1") or base_.endswith(".bn1") or base_.endswith(".bn2")
        if len(shape) == 4:
            fan_in = shape[1] * shape[2] * shape[3]
            sd[name] = torch.randn(shape, generator=g) * ((0.5 if name.startswith("final_conv.3") else 1.0) * (2.0 / fan_in) ** 0.5)
        elif len(shape) == 2:
            sd[name] = torch.randn(shape, generator=g) * (1.0 / shape[1]) ** 0.5
        elif is_bn and name.endswith(".weight"):
            sd[name] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        elif is_bn:
            sd[name] = (0.0 if ".bn2." in name else 0.5) + 0.05 * torch.randn(shape, generator=g)
        else:
            sd[name] = 0.05 * torch.randn(shape, generator=g)
        if is_bn and name.endswith(".bias"):
            base = name[:-len(".bias")]
            sd[base + ".running_mean"] = torch.zeros(shape)
            sd[base + ".running_var"] = torch.ones(shape)
            sd[base + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)
    return sd


def _lw_conv_block(sd, stats, p, x, training, b):
    z = _rn_conv(sd, p + ".conv.0.weight", x, padding=1, bias=sd[p + ".conv.0.bias"], bf16=b, center=_center(stats, p + ".conv.1", training))
    return _rn_bn(sd, stats, p + ".conv.1", z, training, True, bf16=b)


def _lw_res_block(sd, stats, p, x, training, b):
    """ResidualBlock.forward (nets/LightWeightUnet.py:45-55)."""
    y = _rn_bn(sd, stats, p + ".bn1", _rn_conv(sd, p + ".conv1.weight", x, padding=1, bias=sd[p + ".conv1.bias"], bf16=b, center=_center(stats, p + ".bn1", training)), training, True, bf16=b)
    y = _rn_bn(sd, stats, p + ".bn2", _rn_conv(sd, p + ".conv2.weight", y, padding=1, bias=sd[p + ".conv2.bias"], bf16=b, center=_center(stats, p + ".bn2", training)), training, False, bf16=b)
    y = _ulu_se(sd, p + ".se", y, b)
    y = _pinned_relu(y + x, p + ".out")
    return _r(y) if b else y


def lw_forward(sd, x, training=True, stats=None, bf16_storage=False, drop_masks=None):
    """LightweightUnet.forward (nets/LightWeightUnet.py:160-169, 92-110, 117-122).  drop_masks: {site: [N, C] multiplier} for
    the ten Dropout2d sites (feat1..5, up_concat4..1.drop, final_conv.1) in training; missing sites = no dropout."""
    b = bf16_storage
    drop_masks = drop_masks or {}
    if stats is None:
        stats = {k: v.clone() for k, v in sd.items() if "running_" in k or "num_batches" in k}

    def drop(site, t):
        m = drop_masks.get(site) if training else None
        if m is None:
            return t
        t = t * m[:, :, None, None]
        return _r(t) if b else t

    feats = []          # (the image is not rounded: two-term bf16 split in the product path)
    for k in range(1, 6):
        x = _lw_conv_block(sd, stats, f"backbone.stage{k}.0", x, training, b)
        x = _lw_res_block(sd, stats, f"backbone.stage{k}.1", x, training, b)
        x = drop(f"feat{k}", _pinned_max_pool(x, f"pool{k}"))
        feats.append(x)
    low = feats[4]
    for k in (4, 3, 2, 1):
        up = F.interpolate(low, scale_factor=2, mode="bilinear", align_corners=True)
        if b:
            up = _r(up)
        y = _lw_conv_block(sd, stats, f"up_concat{k}.conv.0", torch.cat([feats[k - 1], up], 1), training, b)
        y = _lw_res_block(sd, stats, f"up_concat{k}.conv.1", y, training, b)
        low = drop(f"up_concat{k}.drop", y)
    y = _lw_conv_block(sd, stats, "final_conv.0", low, training, b)
    y = drop("final_conv.1", y)
    y = _lw_res_block(sd, stats, "final_conv.2", y, training, b)
    return F.conv2d(y, sd["final_conv.3.weight"], sd["final_conv.3.bias"]), stats


def lw_train_step(sd, imgs, pngs, cls_weights, num_classes, dice=True, focal=False, bf16_storage=False, drop_masks=None):
    p = {k: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.clone())
         for k, v in sd.items()}
    logits, stats = lw_forward(p, imgs, training=True, bf16_storage=bf16_storage, drop_masks=drop_masks)
    full = resize_logits(logits, pngs.shape[1], pngs.shape[2])
    loss = focal_loss(full, pngs, cls_weights, num_classes) if focal else ce_loss(full, pngs, cls_weights, num_classes)
    if dice:
        loss = loss + dice_loss(full, one_hot(pngs, num_classes))
    names = [k for k, v in p.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [p[k] for k in names])
    return loss.detach(), logits.detach(), dict(zip(names, grads)), stats


# ----------------------------------------------------------------------------------------------- predictor (unet.py)
def make_predictor_params(num_classes, seed=11):
    """make_params with the classifier scaled x150: random-init logits are all ~0 (every class at 1/C), which would make the
    predictor's argmax a coin flip; the scaled head yields confident, multi-class maps (77 % of pixels with a top-2
    probability margin > 0.02 on the fixture image)."""
    p = make_params(num_classes, seed=seed)
    p["final.weight"] = p["final.weight"] * 150.0
    return p


def letterbox(img_u8, input_shape):
    """cvtColor + resize_image (utils/utils.py:12-34): BICUBIC resize that keeps the aspect ratio, pasted on a grey canvas.
    img_u8: H x W x 3 uint8.  Returns (float32 1x3xHxW in [0,1], nw, nh)."""
    from PIL import Image
    image = Image.fromarray(img_u8)
    iw, ih = image.size
    h, w = input_shape
    scale = min(w / iw, h / ih)
    nw, nh = int(iw * scale), int(ih * scale)
    canvas = Image.new("RGB", (w, h), (128, 128, 128))
    canvas.paste(image.resize((nw, nh), Image.BICUBIC), ((w - nw) // 2, (h - nh) // 2))
    data = np.transpose(np.array(canvas, np.float32) / 255.0, (2, 0, 1))[None]
    return torch.from_numpy(data), nw, nh


def resize_linear_cv2(pr, out_h, out_w):
    """cv2.resize(pr, (out_w, out_h), interpolation=cv2.INTER_LINEAR) for float32 H x W x C (unet.py:144, 336):
    f = (d + 0.5) * in / out - 0.5, s = floor(f), f -= s; s < 0 -> (0, 0); s >= in - 1 -> (in - 1, 0)."""
    pr = np.asarray(pr, np.float32)
    ih, iw = pr.shape[:2]

    def taps(n_out, n_in):
        f = (np.arange(n_out, dtype=np.float32) + np.float32(0.5)) * np.float32(n_in / n_out) - np.float32(0.5)
        s = np.floor(f).astype(np.int64)
        f = (f - s).astype(np.float32)
        lo = s < 0
        s[lo] = 0; f[lo] = 0
        hi = s >= n_in - 1
        s[hi] = n_in - 1; f[hi] = 0
        return s, np.minimum(s + 1, n_in - 1), f
    y0, y1, fy = taps(out_h, ih)
    x0, x1, fx = taps(out_w, iw)
    fy = fy[:, None, None]; fx = fx[None, :, None]
    top = pr[y0][:, x0] * (1 - fx) + pr[y0][:, x1] * fx
    bot = pr[y1][:, x0] * (1 - fx) + pr[y1][:, x1] * fx
    return top * (1 - fy) + bot * fy


def predictor_mask(params, img_u8, input_shape):
    """Unet.get_miou_png (unet.py:298-344): the class map at the original image size."""
    oh, ow = img_u8.shape[:2]
    data, nw, nh = letterbox(img_u8, input_shape)
    with torch.no_grad():
        pr = torch.softmax(unet_forward(params, data)[0].permute(1, 2, 0), dim=-1).numpy()
    top, left = (input_shape[0] - nh) // 2, (input_shape[1] - nw) // 2
    pr = resize_linear_cv2(pr[top:top + nh, left:left + nw], oh, ow)
    return pr.argmax(-1).astype(np.uint8), pr
