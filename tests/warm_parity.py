"""Warm, structured 512x512 parity fixtures (VERDICT r1 item 1, SURVEY.md 8c(5) / section 7 hard part 6).

For one model family: build the REFERENCE model (the oracle's restatement of the reference, oracle/unet_oracle.py, which
tests/test_oracle.py pins to the reference's own outputs stored under tests/golden/) on the GPU in fp32 (TF32 off), train it for a few hundred Adam steps on structured
synthetic batches so the logits have margins (a mid-training state instead of near-tied random init), then on one held-out
structured batch compare, against the reference evaluated in FLOAT64 on the same weights:

    ours        the product bf16 path (drop-in nn.Module + CE_Loss + Dice_loss, loss.backward())
    ref_fp32    the reference in fp32 on the GPU (cuDNN, TF32 off) -- how far fp32 itself is from float64
    autocast    the reference under torch.autocast(bfloat16)     -- the same-precision library peer

Quantities: logits rel-L2, global (concatenated) gradient rel-L2, per-tensor gradient rel-L2 (median / worst), arg-max
agreement over ALL pixels.  Used by tests/test_parity_512_gpu.py (asserts) and scripts/parity_512.py (report).
TEST INFRASTRUCTURE: nothing under unet-pytorch_b200/ imports this.
"""
import copy
import os
import sys
import time
import types

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import unet_oracle as O  # noqa: E402

# family -> (ctor kwargs builder, class name of the reference module and of its drop-in)
FAMILIES = {
    "unet_vgg": (lambda C: dict(num_classes=C, pretrained=False, backbone="vgg"), "Unet"),
    "unet_resnet50": (lambda C: dict(num_classes=C, pretrained=False, backbone="resnet50"), "Unet"),
    "traditional": (lambda C: dict(in_channels=3, num_classes=C), "TraditionalUnet"),
    "lightweight": (lambda C: dict(num_classes=C), "LightweightUnet"),
    "ultralight": (lambda C: dict(num_classes=C), "UltraLightweightUnet"),
    "ultralight_large": (lambda C: dict(num_classes=C), "UltraLightweightUnet_large"),
    "ultralight_large_optimized": (lambda C: dict(num_classes=C), "UltraLightweightUnet_large_optimized"),
}


def _oracle_forward(family):
    """(state_dict, x, training, stats) -> (logits, stats): the oracle's forward of the family."""
    if family == "unet_vgg":
        return lambda sd, x, training, stats: (O.unet_forward(sd, x), stats)
    if family.startswith("ultralight"):
        return lambda sd, x, training, stats: O.ulu_forward(sd, x, family, training=training, stats=stats)
    fwd = {"unet_resnet50": O.resnet_unet_forward, "traditional": O.trad_forward, "lightweight": O.lw_forward}[family]
    return lambda sd, x, training, stats: fwd(sd, x, training=training, stats=stats)


class OracleReference(torch.nn.Module):
    """One model family of the reference as the oracle computes it, without Dropout: the trainable tensors of its state_dict
    are parameters, the BatchNorm statistics buffers (updated in training mode like torch's BatchNorm2d)."""

    def __init__(self, family, state_dict):
        super().__init__()
        self.fwd = _oracle_forward(family)
        self.names = [k for k, v in state_dict.items() if v.is_floating_point() and "running_" not in k]
        self.buffer_names = [k for k in state_dict if k not in self.names]
        self.weights = torch.nn.ParameterList(torch.nn.Parameter(state_dict[k].clone()) for k in self.names)
        for i, k in enumerate(self.buffer_names):
            self.register_buffer(f"stat{i}", state_dict[k].clone())

    def reference_state_dict(self):
        """The state_dict of the reference module (its own key names)."""
        sd = dict(zip(self.names, self.weights))
        sd.update((k, getattr(self, f"stat{i}")) for i, k in enumerate(self.buffer_names))
        return sd

    def forward(self, x):
        sd = self.reference_state_dict()
        logits, stats = self.fwd(sd, x, self.training, {k: sd[k] for k in self.buffer_names})
        with torch.no_grad():
            for i, k in enumerate(self.buffer_names):
                if stats[k] is not sd[k]:           # num_batches_tracked is replaced, the running statistics update in place
                    getattr(self, f"stat{i}").copy_(stats[k])
        return logits

    def grads(self):
        return {k: p.grad.detach() for k, p in zip(self.names, self.weights) if p.grad is not None}


# CE_Loss / Dice_loss (nets/unet_training.py) as the oracle restates them, logits resized to the label size first
ORACLE_LOSSES = types.SimpleNamespace(
    CE_Loss=lambda inputs, target, cls_weights, num_classes=21: O.ce_loss(
        O.resize_logits(inputs, target.shape[1], target.shape[2]), target, cls_weights, num_classes),
    Dice_loss=lambda inputs, target: O.dice_loss(O.resize_logits(inputs, target.shape[1], target.shape[2]), target))


def build_reference(family, C, seed=11):
    """The reference model (OracleReference) and its loss functions.  Its initial weights are those the module's own
    constructor draws after torch.manual_seed(seed); the drop-in module keeps the reference's module tree and init."""
    import unet_pytorch_b200 as b2u
    kw, cls = FAMILIES[family]
    torch.manual_seed(seed)
    sd = getattr(b2u, cls)(**kw(C)).state_dict()
    return OracleReference(family, sd), ORACLE_LOSSES


def make_batch(n, C, hw, seed, medical=False, device="cpu"):
    imgs, pngs = O.make_inputs(n, C, hw, hw, seed=seed, medical=medical)
    return imgs.to(device), pngs.to(device)


def loss_of(T, logits, pngs, C, weights, dice=True):
    labels = F.one_hot(pngs, C + 1).to(logits.dtype)
    loss = T.CE_Loss(logits, pngs, weights.to(logits.dtype), num_classes=C)
    if dice:
        loss = loss + T.Dice_loss(logits, labels)
    return loss


def warm_up(model, T, C, hw, batch, steps, device, lr=1e-3, medical=False, nbatches=4, log=None):
    """A few hundred fp32 Adam steps of the reference on structured batches (seeds 1000..): returns the final loss."""
    model.train()
    torch.backends.cudnn.allow_tf32 = True          # the warm-up only has to produce plausible mid-training weights
    torch.backends.cuda.matmul.allow_tf32 = True
    # ask for reproducible kernels so every run (and box) trains towards the same fixture; ops without a deterministic
    # implementation only warn
    det = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark, torch.are_deterministic_algorithms_enabled())
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    torch.use_deterministic_algorithms(True, warn_only=True)
    opt = torch.optim.Adam(model.parameters(), lr=lr)
    w = torch.ones(C, device=device)
    data = [make_batch(batch, C, hw, 1000 + i, medical, device) for i in range(nbatches)]
    last = None
    for it in range(steps):
        imgs, pngs = data[it % nbatches]
        opt.zero_grad(set_to_none=True)
        loss = loss_of(T, model(imgs), pngs, C, w)
        loss.backward()
        opt.step()
        if it == 0 or it == steps - 1 or (log and (it + 1) % 50 == 0):
            last = loss.item()
            if log:
                log(f"    warm step {it + 1}/{steps}: loss {last:.4f}")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = det[0], det[1]
    torch.use_deterministic_algorithms(det[2])
    return last


def _rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / (b.norm() + 1e-300)).item()


def compare(grads, logits, ref_grads, ref_logits):
    names = list(ref_grads.keys())
    num = sum((grads[k].double() - ref_grads[k].double()).pow(2).sum().item() for k in names)
    den = sum(ref_grads[k].double().pow(2).sum().item() for k in names)
    # per-tensor distances; tensors whose true gradient is identically zero (a conv bias in front of a BatchNorm: float64
    # returns 1e-20 residue) carry no relative error
    per = sorted(((_rel(grads[k], ref_grads[k]), k) for k in names if ref_grads[k].double().norm().item() > 1e-9 * den ** 0.5),
                 reverse=True)
    vals = [p[0] for p in per]
    agree = (logits.argmax(1) == ref_logits.argmax(1)).double().mean().item()
    return {"logits": _rel(logits, ref_logits), "grad_global": (num / den) ** 0.5, "grad_worst": per[0][0], "grad_worst_name": per[0][1],
            "grad_median": vals[len(vals) // 2], "argmax_all": agree}


def run_reference(model, T, imgs, pngs, C, dtype, autocast=False):
    """logits + gradients of the reference in `dtype` (float64 / float32), or fp32 weights under bf16 autocast."""
    m = copy.deepcopy(model).to(dtype).train()
    for p in m.parameters():
        p.grad = None
    w = torch.ones(C, device=imgs.device, dtype=dtype)
    x = imgs.to(dtype)
    if autocast:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            logits = m(x)
        logits = logits.float()
    else:
        logits = m(x)
    loss = loss_of(T, logits, pngs, C, w)
    loss.backward()
    return logits.detach(), m.grads(), loss.item()


def run_product(b2u, family, state_dict, imgs, pngs, C):
    """The product bf16 path through the drop-in module API (the calls of utils_fit.py:70-92)."""
    kw, cls = FAMILIES[family]
    model = getattr(b2u, cls)(**kw(C))
    model.load_state_dict(state_dict)
    model = model.train().to(imgs.device)
    for eng_owner in (model,):
        eng = eng_owner._engine_for(imgs.device)
        for ins in getattr(eng, "program", []):          # Dropout disabled, like the reference side
            if ins["op"] == "drop":
                ins["p"] = 0.0
    w = torch.ones(C, device=imgs.device)
    logits = model(imgs)
    labels = F.one_hot(pngs, C + 1).float()
    loss = b2u.CE_Loss(logits, pngs, w, num_classes=C) + b2u.Dice_loss(logits, labels)
    loss.backward()
    grads = {k: p.grad.detach() for k, p in model.named_parameters() if p.grad is not None}
    out = logits.detach().clone()
    for e in model._engines.values():
        e.release()
    return out, grads, loss.item()


def measure(b2u, family, C, hw=512, batch=8, warm_steps=200, warm_batch=4, device="cuda:0", medical=False, log=None,
            with_autocast=True, cache_dir=None):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device(device)
    t0 = time.time()
    model, T = build_reference(family, C)
    model = model.to(dev)
    cache = os.path.join(cache_dir, f"warm_{family}_nc{C}_{hw}_{warm_steps}.pt") if cache_dir else None
    if cache and os.path.exists(cache):
        model.load_state_dict(torch.load(cache, map_location=dev))
        warm_loss = None
    else:
        warm_loss = warm_up(model, T, C, hw, warm_batch, warm_steps, dev, medical=medical, log=log)
        if cache:
            os.makedirs(cache_dir, exist_ok=True)
            torch.save(model.state_dict(), cache)
    sd = {k: v.detach().clone() for k, v in model.reference_state_dict().items()}
    imgs, pngs = make_batch(batch, C, hw, 7, medical, dev)
    z64, g64, l64 = run_reference(model, T, imgs, pngs, C, torch.float64)
    out = {"family": family, "classes": C, "hw": hw, "batch": batch, "warm_steps": warm_steps, "warm_loss": warm_loss, "loss_fp64": l64}
    z32, g32, _ = run_reference(model, T, imgs, pngs, C, torch.float32)
    out["ref_fp32"] = compare(g32, z32, g64, z64)
    del z32, g32
    if with_autocast:
        za, ga, _ = run_reference(model, T, imgs, pngs, C, torch.float32, autocast=True)
        out["autocast_bf16"] = compare(ga, za, g64, z64)
        del za, ga
    del model
    torch.cuda.empty_cache()
    zo, go, lo = run_product(b2u, family, sd, imgs, pngs, C)
    out["ours_bf16"] = compare(go, zo, g64, z64)
    out["loss_ours"] = lo
    out["seconds"] = time.time() - t0
    return out
