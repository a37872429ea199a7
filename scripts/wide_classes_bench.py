"""Heads with more than 32 classes: Unet-VGG16 training step (batch 16, 512x512) at C in {21, 59, 150, 255}, and the
per-kernel time and achieved GB/s of the wide paths at C = 150 (n = 150 for the histogram, 1000 masks of 512x512).

GB/s counts ALGORITHMIC bytes (each tensor the kernel must read or write, once), computed from shapes below; a kernel that
re-reads its input from L2 or HBM shows up as a lower rate, not as more bytes.  Byte model of the step at C = 150 (not
measured): fp32 logits are 2.5 GB; the head writes them, the loss reads them twice; the split bf16 dlogits (2.7 GB) are
written once and read twice: ~10 GB more HBM traffic than C = 21, ~2 ms per step at 5 TB/s.

usage: python scripts/wide_classes_bench.py [out.json]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import unet_pytorch_b200 as b2u
from unet_pytorch_b200 import ops
import bench


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:           # the numbers stay valid; the record says the query failed
        info["power_limit_w"] = f"unavailable: {e}"
    return info


def rate(ms, nbytes):
    return {"ms": round(ms, 4), "GB": round(nbytes / 1e9, 4), "GBps": round(nbytes / 1e9 / ms * 1e3, 1)}


def main():
    dev = torch.device("cuda:0")
    res = {"card": card(), "steps": {}, "kernels_c150": {}}
    N, H, W = 16, 512, 512
    P = N * H * W
    g = torch.Generator(device=dev).manual_seed(0)
    imgs = torch.rand((N, 3, H, W), device=dev, generator=g)
    for C in (21, 59, 150, 255):
        pngs = torch.randint(0, C + 1, (N, H, W), device=dev, generator=g)
        tr = b2u.UnetTrainer(num_classes=C, device=dev, lr=1e-4)
        ms = bench._ev_ms(lambda: tr.train_step(imgs, pngs), 10, 3)
        res["steps"][f"C{C}"] = {"ms_per_step": round(ms, 3), "img_per_s": round(N / ms * 1e3, 1)}
        del tr
        torch.cuda.empty_cache()

    C, G = 150, ops.head_groups(150)
    k = res["kernels_c150"]
    x = (torch.randn((N, H, W, 64), device=dev, generator=g).relu()).to(torch.bfloat16)
    w = torch.randn((C, 64), device=dev, generator=g) * 0.1
    bias = torch.randn((C,), device=dev, generator=g)
    wf = ops.pack_head_fprop(w)
    logits = torch.empty((N, C, H, W), device=dev)
    k["head_fwd_tc"] = rate(bench._ev_ms(lambda: ops.head_fwd_tc(x, wf, bias, C, out=logits), 20, 3), 2 * 64 * P + 4 * C * P)
    pngs = torch.randint(0, C + 1, (N, H, W), device=dev, generator=g)
    ws = torch.empty(ops.lib().b2u_loss_workspace(C), dtype=torch.uint8, device=dev)
    k["loss_fwd"] = rate(bench._ev_ms(lambda: ops.loss_fwd(logits, target=pngs, ws=ws), 20, 3), 4 * C * P + 8 * P)
    fin = ops.loss_fwd(logits, target=pngs, ws=ws)
    gs = torch.tensor([1.0, 0.0, 1.0], device=dev)
    d64 = torch.empty((N, H, W, 64 * G), dtype=torch.bfloat16, device=dev)
    k["loss_bwd_nhwc64"] = rate(bench._ev_ms(lambda: ops.loss_bwd(logits, fin, gs, target=pngs, out=d64, nhwc64=True), 20, 3),
                                4 * C * P + 8 * P + 2 * 64 * G * P)
    wd = ops.pack_head_dgrad(w)
    dx = torch.empty_like(x)
    k["head_dgrad_tc"] = rate(bench._ev_ms(lambda: ops.conv_dgrad(d64, wd, 64, taps=1, mask=x, out0=dx), 20, 3),
                              2 * 64 * G * P + 2 * 2 * 64 * P)
    dw = torch.empty((64 * G, 64, 1, 1), device=dev)
    db = torch.empty((64 * G,), device=dev)
    k["head_wgrad_tc"] = rate(bench._ev_ms(lambda: ops.conv_wgrad(x, d64, taps=1, dw=dw, db=db), 20, 3), 2 * 64 * G * P + 2 * 64 * P)
    mask = torch.empty((N, H, W), dtype=torch.uint8, device=dev)
    k["softmax_resize_argmax"] = rate(bench._ev_ms(lambda: ops.softmax_resize_argmax_u8(logits, (0, 0, H, W), (H, W), out=mask), 10, 2),
                                      4 * C * P + P)
    del x, dx, d64, logits
    torch.cuda.empty_cache()
    n, M = 150, 1000
    gt = torch.randint(0, n, (M, H, W), dtype=torch.uint8, device=dev, generator=g)
    pred = torch.where(torch.rand((M, H, W), device=dev, generator=g) < 0.2,
                       torch.randint(0, n, (M, H, W), dtype=torch.uint8, device=dev, generator=g), gt)
    hist = torch.zeros(n * n + 1, dtype=torch.int64, device=dev)
    table = ops.HistTable([(gt[i].reshape(-1), pred[i].reshape(-1)) for i in range(M)], dev)
    k["fast_hist_batch_n150_1000x512x512"] = rate(bench._ev_ms(lambda: ops.fast_hist_batch(table, n, hist), 5, 2), 2 * M * H * W)
    k["fast_hist_n150_one_call"] = rate(bench._ev_ms(lambda: ops.fast_hist_accumulate(gt.reshape(-1), pred.reshape(-1), n, hist), 5, 2),
                                        2 * M * H * W)
    out = json.dumps(res, indent=1)
    print(out)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
