#!/usr/bin/env python
"""Which bf16 rounding site costs what?  The staged reference model, evaluated in float64 on the warm 512x512 fixture of
tests/warm_parity.py, with ONE class of tensors rounded to bf16 at a time (straight-through: the rounding perturbs the
value, the gradient passes unchanged unless the site is a gradient site):

    weights   every conv / linear weight                    image    the input image
    act       the input of every conv (stored activations)  prebn    the output of every conv that feeds a BatchNorm
    act_inner the same without the first conv (whose input is the image)
    grad      the gradient flowing back through every conv output
    all       everything above (a bf16-storage model of the product path)

Prints logits / global-gradient rel-L2 against the unrounded float64 run.  Diagnostic for DESIGN.md section 5."""
import argparse
import copy
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


class RoundFwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return g


class RoundBwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.clone()

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(g.dtype)


# family -> module and class of the reference (the rounding sites are hooked on its nn.Conv2d / nn.Linear modules)
REFERENCE_CLASSES = {"unet_vgg": ("nets.unet", "Unet"), "unet_resnet50": ("nets.unet", "Unet"),
                     "traditional": ("nets.TraditionalUnet", "TraditionalUnet"), "lightweight": ("nets.LightWeightUnet", "LightweightUnet"),
                     "ultralight": ("nets.UltraLightweightUnet", "UltraLightweightUnet"),
                     "ultralight_large": ("nets.UltraLightweightUnet_large", "UltraLightweightUnet_large"),
                     "ultralight_large_optimized": ("nets.UltraLightweightUnet_large_optimized", "UltraLightweightUnet_large_optimized")}


def build_reference(fam, C, WP, seed=11):
    """The unmodified reference module staged under baseline/_ref (baseline/stage_ref.py), Dropout disabled, and its losses."""
    from baseline import stage_ref
    mod, cls = REFERENCE_CLASSES[fam]
    torch.manual_seed(seed)
    model = getattr(stage_ref.import_reference(mod), cls)(**WP.FAMILIES[fam][0](C))
    for m in model.modules():
        if isinstance(m, (torch.nn.Dropout, torch.nn.Dropout2d)):
            m.p = 0.0
    return model, stage_ref.import_reference("nets.unet_training")


def run(model, T, imgs, pngs, C, sites, WP):
    m = copy.deepcopy(model).double().train()
    convs = [mod for mod in m.modules() if isinstance(mod, torch.nn.Conv2d)]
    # convs followed by a BatchNorm: by module order inside the reference's Sequentials / blocks
    mods = list(m.modules())
    prebn = set()
    for a, b in zip(mods[:-1], mods[1:]):
        if isinstance(a, torch.nn.Conv2d) and isinstance(b, torch.nn.BatchNorm2d):
            prebn.add(a)
    handles = []
    if "weights" in sites:
        with torch.no_grad():
            for mod in m.modules():
                if isinstance(mod, (torch.nn.Conv2d, torch.nn.Linear)):
                    mod.weight.copy_(mod.weight.to(torch.bfloat16).double())
    x = imgs.double()
    if "image" in sites:
        x = x.to(torch.bfloat16).double()
    for cv in convs:
        if "act" in sites or ("act_inner" in sites and cv.in_channels != 3):
            handles.append(cv.register_forward_pre_hook(lambda mod, inp: (RoundFwd.apply(inp[0]),)))
        if "prebn" in sites or "grad" in sites:
            def hook(mod, inp, out, _pb=(cv in prebn)):
                if "prebn" in sites and _pb:
                    out = RoundFwd.apply(out)
                if "grad" in sites:
                    out = RoundBwd.apply(out)
                return out
            handles.append(cv.register_forward_hook(hook))
    w = torch.ones(C, device=imgs.device, dtype=torch.float64)
    logits = m(x)
    loss = WP.loss_of(T, logits, pngs, C, w)
    loss.backward()
    grads = {k: p.grad.detach() for k, p in m.named_parameters() if p.grad is not None}
    for h in handles:
        h.remove()
    return logits.detach(), grads


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--families", default="traditional:21,ultralight_large:2,ultralight:21,lightweight:2,unet_resnet50:21,unet_vgg:21")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--hw", type=int, default=512)
    ap.add_argument("--warm", type=int, default=200)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "precision_sites.json"))
    args = ap.parse_args()
    import warm_parity as WP
    dev = torch.device("cuda:0")
    rows = []
    for item in args.families.split(","):
        fam, C = item.split(":")
        C = int(C)
        medical = C == 2
        model, T = build_reference(fam, C, WP)
        model = model.to(dev)
        WP.warm_up(model, T, C, args.hw, 4, args.warm, dev, lr=args.lr, medical=medical)
        imgs, pngs = WP.make_batch(args.batch, C, args.hw, 7, medical, dev)
        z0, g0 = run(model, T, imgs, pngs, C, (), WP)
        print(f"== {fam} nc={C} warm {args.warm} steps lr {args.lr}", flush=True)
        for sites in (("weights",), ("image",), ("act_inner",), ("prebn",), ("grad",), ("weights", "act_inner"), ("weights", "act_inner", "grad"),
                      ("weights", "image", "act", "prebn", "grad")):
            z, g = run(model, T, imgs, pngs, C, sites, WP)
            c = WP.compare(g, z, g0, z0)
            print(f"  {'+'.join(sites):32s} logits {c['logits']:.2e}  grad global {c['grad_global']:.2e}  median {c['grad_median']:.2e}  "
                  f"worst {c['grad_worst']:.2e}  argmax {100 * c['argmax_all']:.3f} %", flush=True)
            rows.append({"family": fam, "classes": C, "sites": list(sites), **c})
        del model
        torch.cuda.empty_cache()
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        json.dump(rows, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
