"""Cost of the gradient wrt the input image (x.grad) on the GPU -> profiles/r4_input_grad.json.

  kernels  the three new entry points alone at batch 16, 512 x 512 (stem dz at 256 x 256), CUDA events over `reps` launches;
           dz is 512 MB, larger than L2, so every launch reads it from HBM
  steps    fwd + loss + bwd of the drop-in module (train mode, CE + Dice) with and without x.requires_grad, alternated in
           the same process, for Unet-VGG16 and UltraLightweightUnet_large
  delta    where the step's extra time goes: one torch.profiler run of each variant after the timed ones, the per-kernel CUDA
           time summed by name, and the kernels whose total differs by more than 20 us (the timed steps run without it)

Usage: python scripts/input_grad_bench.py [--batch 16] [--size 512] [--steps 20] [--out profiles/r4_input_grad.json]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _events(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def _kernel_delta(step):
    from torch.profiler import ProfilerActivity, profile
    per = {}
    for xg in (False, True):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(xg)
            torch.cuda.synchronize()
        per[xg] = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t > 0:
                per[xg][e.key] = t / 1e3
    keys = set(per[False]) | set(per[True])
    delta = {k: per[True].get(k, 0.0) - per[False].get(k, 0.0) for k in keys}
    out = {k[:120]: round(v, 4) for k, v in sorted(delta.items(), key=lambda kv: -abs(kv[1])) if abs(v) > 0.02}
    out["total_kernel_ms_without"] = round(sum(per[False].values()), 4)
    out["total_kernel_ms_with"] = round(sum(per[True].values()), 4)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_input_grad.json"))
    a = ap.parse_args()
    import unet_pytorch_b200 as b2u
    ops = b2u.ops
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    N, S = a.batch, a.size
    res = {"gpu": smi[0] if smi else "unknown", "batch": N, "size": S, "kernels_ms": {}, "steps_ms": {}}
    g = torch.Generator(device=dev).manual_seed(0)
    dz = torch.randn(N, S, S, 64, device=dev, generator=g).to(torch.bfloat16)
    w3 = torch.randn(64, 3, 3, 3, device=dev, generator=g) * 0.1
    dx = torch.empty(N, 3, S, S, device=dev)
    res["kernels_ms"]["first_conv_dgrad_input (Cin 3, Cout 64)"] = _events(lambda: ops.first_conv_dgrad_input(dz, w3, out=dx), 50)
    res["kernels_ms"]["nhwc_bf16_padded_to_nchw_f32 (C 3 of 64)"] = _events(lambda: ops.nhwc_padded_to_nchw_f32(dz, 3, out=dx), 50)
    dzs = dz[:, : S // 2, : S // 2].contiguous()
    w7 = torch.randn(64, 3, 7, 7, device=dev, generator=g) * 0.05
    res["kernels_ms"]["stem_dgrad_input (Cin 3, Cout 64, dz at half size)"] = _events(lambda: ops.stem_dgrad_input(dzs, w7, S, S, out=dx), 50)
    # the bytes each kernel has to move at least (dz read once, dx written once), for a bandwidth figure
    res["kernels_min_bytes"] = {"first_conv_dgrad_input": dz.numel() * 2 + dx.numel() * 4,
                                "stem_dgrad_input": dzs.numel() * 2 + dx.numel() * 4,
                                "nhwc_bf16_padded_to_nchw_f32": N * S * S * 16 + dx.numel() * 4}
    del dz, dzs

    C = 21
    imgs = torch.rand(N, 3, S, S, device=dev, generator=g)
    pngs = torch.randint(0, C, (N, S, S), device=dev, generator=g)
    onehot = torch.nn.functional.one_hot(pngs, C + 1).float()
    wts = torch.ones(C, device=dev)
    from unet_pytorch_b200.nets.UltraLightweightUnet_large import UltraLightweightUnet_large
    for name, model in (("Unet-VGG16", b2u.Unet(num_classes=C)), ("UltraLightweightUnet_large", UltraLightweightUnet_large(num_classes=C))):
        model = model.to(dev).train()

        def step(x_grad):
            x = imgs.detach().requires_grad_(x_grad)
            out = model(x)
            loss = b2u.CE_Loss(out, pngs, wts, num_classes=C) + b2u.Dice_loss(out, onehot)
            loss.backward()
            model.zero_grad(set_to_none=True)

        for xg in (False, True, False, True):       # warm-up: both shapes of the saved state
            step(xg)
        times = {False: [], True: []}
        for i in range(2 * a.steps):                # alternate the two variants
            xg = bool(i % 2)
            times[xg].append(_events(lambda: step(xg), 1))
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        res["steps_ms"][name] = {"without_x_grad_median": med[False], "with_x_grad_median": med[True],
                                 "without_x_grad_all": times[False], "with_x_grad_all": times[True]}
        res["steps_ms"][name]["kernel_ms_delta"] = _kernel_delta(step)
        del model
        torch.cuda.empty_cache()
    print(json.dumps({k: v for k, v in res.items() if k != "steps_ms"}, indent=1))
    for k, v in res["steps_ms"].items():
        print(k, f"{v['without_x_grad_median']:.2f} ms without x.grad, {v['with_x_grad_median']:.2f} ms with;",
              "kernel time delta:", json.dumps(v["kernel_ms_delta"]))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
