"""Drop-ins for the loss functions of the reference's nets/unet_training.py (lines 9-56) plus its small host
helpers (weights_init :58-76, get_lr_scheduler :78-108, set_optimizer_lr :110-113).

CE_Loss / Focal_Loss / Dice_loss keep the reference signatures and run the fused CUDA loss kernels
(csrc/head_loss.cu); `ce_dice_loss` is the one-pass combination the training loop uses (utils_fit.py:74-81)."""
import math
from functools import partial

import torch

from .. import ops


class _ResizeBilinear(torch.autograd.Function):
    """F.interpolate(x, size=(ht, wt), mode="bilinear", align_corners=True) on the CUDA resize kernels."""

    @staticmethod
    def forward(ctx, x, ht, wt):
        ctx.size_in = tuple(x.shape[2:])
        return ops.resize_bilinear(x, (ht, wt))

    @staticmethod
    def backward(ctx, g):
        return ops.resize_bilinear_bwd(g.contiguous(), ctx.size_in), None, None


def _prep_logits(inputs, ht, wt):
    n, c, h, w = inputs.shape
    if not inputs.is_cuda:
        raise RuntimeError("B200 loss kernels need CUDA tensors (no CPU fallback)")
    x = inputs
    if x.dtype != torch.float32:
        x = x.float()
    x = x.contiguous()
    if h != ht and w != wt:   # same (and-) condition as the reference, nets/unet_training.py:12 (LightweightUnet: H/2 logits)
        x = _ResizeBilinear.apply(x, ht, wt)
    elif h != ht or w != wt:
        raise ValueError("logits and labels differ in exactly one spatial dimension (the reference would fail in view())")
    return x


class _LossFunction(torch.autograd.Function):
    """out = w_ce * CE + w_focal * Focal + w_dice * Dice, one stats pass; backward = one dlogits pass."""

    @staticmethod
    def forward(ctx, logits, target, onehot, cls_w, w_ce, w_focal, w_dice, beta, smooth, alpha, gamma):
        # (alpha = 0 zeroes the focal term exactly; the kernel then skips its powf / expf -- only Focal_Loss asks for it)
        fin = ops.loss_fwd(logits, target=target, onehot=onehot, cls_w=cls_w, beta=beta, smooth=smooth,
                           alpha=alpha if w_focal != 0.0 else 0.0, gamma=gamma)
        ctx.save_for_backward(logits, target, onehot, cls_w, fin)
        ctx.cfg = (w_ce, w_focal, w_dice, alpha, gamma)
        # only the requested terms: an unrequested CE is 0/0 = nan when no label map was given
        terms = [wt * fin[i] for i, wt in enumerate((w_ce, w_focal, w_dice)) if wt != 0.0]
        return sum(terms[1:], terms[0])

    @staticmethod
    def backward(ctx, gout):
        logits, target, onehot, cls_w, fin = ctx.saved_tensors
        w_ce, w_focal, w_dice, alpha, gamma = ctx.cfg
        gscale = gout.reshape(1).to(torch.float32) * torch.tensor([w_ce, w_focal, w_dice], dtype=torch.float32,
                                                                  device=logits.device)
        d = ops.loss_bwd(logits, fin, gscale, target=target, onehot=onehot, cls_w=cls_w, alpha=alpha, gamma=gamma)
        return (d,) + (None,) * 10


def _target_map(target, num_classes):
    t = target
    if t.dtype != torch.int64:
        t = t.long()
    return t.contiguous()


def CE_Loss(inputs, target, cls_weights, num_classes=21):
    nt, ht, wt = target.size()
    x = _prep_logits(inputs, ht, wt)
    cw = None if cls_weights is None else cls_weights.to(device=x.device, dtype=torch.float32).contiguous()
    if x.shape[1] != num_classes:
        raise ValueError("CE_Loss: ignore_index == num_classes requires logits with num_classes channels")
    return _LossFunction.apply(x, _target_map(target, num_classes), None, cw, 1.0, 0.0, 0.0, 1.0, 1e-5, 0.5, 2.0)


def Focal_Loss(inputs, target, cls_weights, num_classes=21, alpha=0.5, gamma=2):
    nt, ht, wt = target.size()
    x = _prep_logits(inputs, ht, wt)
    cw = None if cls_weights is None else cls_weights.to(device=x.device, dtype=torch.float32).contiguous()
    a = 1.0 if alpha is None else float(alpha)   # reference: `if alpha is not None: logpt *= alpha`
    return _LossFunction.apply(x, _target_map(target, num_classes), None, cw, 0.0, 1.0, 0.0, 1.0, 1e-5, a, float(gamma))


def Dice_loss(inputs, target, beta=1, smooth=1e-5):
    nt, ht, wt, ct = target.size()
    x = _prep_logits(inputs, ht, wt)
    if ct != x.shape[1] + 1:
        raise ValueError("Dice_loss: target must be one-hot with num_classes + 1 channels")
    oh = target.to(device=x.device, dtype=torch.float32).contiguous()
    return _LossFunction.apply(x, None, oh, None, 0.0, 0.0, 1.0, float(beta), float(smooth), 0.5, 2.0)


def ce_dice_loss(inputs, target, cls_weights, num_classes=21, dice=True, focal=False, beta=1, smooth=1e-5, alpha=0.5,
                 gamma=2):
    """CE (or Focal) + Dice exactly as utils_fit.py:74-81 combines them, from the integer label map alone:
    the fp32 one-hot tensor the reference feeds Dice_loss is np.eye(C+1)[png] (dataloader.py:49-50), so it is
    implied by `target`."""
    nt, ht, wt = target.size()
    x = _prep_logits(inputs, ht, wt)
    cw = None if cls_weights is None else cls_weights.to(device=x.device, dtype=torch.float32).contiguous()
    a = 1.0 if alpha is None else float(alpha)
    return _LossFunction.apply(x, _target_map(target, num_classes), None, cw, 0.0 if focal else 1.0,
                               1.0 if focal else 0.0, 1.0 if dice else 0.0, float(beta), float(smooth), a, float(gamma))


# ---------------------------------------------------------------------------------------- host helpers
# weights_init / get_lr_scheduler / set_optimizer_lr (nets/unet_training.py:58-113): host-side helpers outside the hot
# path, restated with the reference's signatures and arithmetic so that the training scripts can import them from here.
def weights_init(net, init_type="normal", init_gain=0.02):
    """Every module whose class name contains 'Conv' and that has a weight: N(0, init_gain) (or the named init);
    BatchNorm2d: weight N(1, 0.02), bias 0."""
    def init_func(m):
        classname = m.__class__.__name__
        if hasattr(m, "weight") and classname.find("Conv") != -1:
            if init_type == "normal":
                torch.nn.init.normal_(m.weight.data, 0.0, init_gain)
            elif init_type == "xavier":
                torch.nn.init.xavier_normal_(m.weight.data, gain=init_gain)
            elif init_type == "kaiming":
                torch.nn.init.kaiming_normal_(m.weight.data, a=0, mode="fan_in")
            elif init_type == "orthogonal":
                torch.nn.init.orthogonal_(m.weight.data, gain=init_gain)
            else:
                raise NotImplementedError("initialization method [%s] is not implemented" % init_type)
        elif classname.find("BatchNorm2d") != -1:
            torch.nn.init.normal_(m.weight.data, 1.0, 0.02)
            torch.nn.init.constant_(m.bias.data, 0.0)
    print("initialize network with %s type" % init_type)
    net.apply(init_func)


def get_lr_scheduler(lr_decay_type, lr, min_lr, total_iters, warmup_iters_ratio=0.05, warmup_lr_ratio=0.1,
                     no_aug_iter_ratio=0.05, step_num=10):
    """epoch -> learning rate.  "cos": quadratic warm-up, cosine decay, min_lr for the last epochs; otherwise step decay
    from lr to min_lr in step_num steps."""
    def yolox_warm_cos_lr(lr, min_lr, total_iters, warmup_total_iters, warmup_lr_start, no_aug_iter, iters):
        if iters <= warmup_total_iters:
            lr = (lr - warmup_lr_start) * pow(iters / float(warmup_total_iters), 2) + warmup_lr_start
        elif iters >= total_iters - no_aug_iter:
            lr = min_lr
        else:
            lr = min_lr + 0.5 * (lr - min_lr) * (
                1.0 + math.cos(math.pi * (iters - warmup_total_iters) / (total_iters - warmup_total_iters - no_aug_iter)))
        return lr

    def step_lr(lr, decay_rate, step_size, iters):
        if step_size < 1:
            raise ValueError("step_size must above 1.")
        n = iters // step_size
        return lr * decay_rate ** n

    if lr_decay_type == "cos":
        warmup_total_iters = min(max(warmup_iters_ratio * total_iters, 1), 3)
        warmup_lr_start = max(warmup_lr_ratio * lr, 1e-6)
        no_aug_iter = min(max(no_aug_iter_ratio * total_iters, 1), 15)
        return partial(yolox_warm_cos_lr, lr, min_lr, total_iters, warmup_total_iters, warmup_lr_start, no_aug_iter)
    decay_rate = (min_lr / lr) ** (1 / (step_num - 1))
    step_size = total_iters / step_num
    return partial(step_lr, lr, decay_rate, step_size)


def set_optimizer_lr(optimizer, lr_scheduler_func, epoch):
    lr = lr_scheduler_func(epoch)
    for param_group in optimizer.param_groups:
        param_group["lr"] = lr
