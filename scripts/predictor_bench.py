"""Predictor evaluation throughput: `Unet.get_miou` images/s over a seeded synthetic set (512 RGB images, sides drawn from
200 to 1200, uint8 ground truths, n = 21, Unet-VGG16 at 512x512), batched path (device letterbox, batch forward, batched
tail; batch 16 and 64) against the per-image loop of the previous predictor (host PIL letterbox, batch-1 forward,
single-image tail), restated below.  The paths run alternately in one call and must give the same confusion matrix.

Host time is split out per image: the batched path's `_prepare` (cvtColor + the image bytes + geometry) against the old
loop's host letterbox (PIL BICUBIC resize + paste + float32 / 255 + transpose).

usage: python scripts/predictor_bench.py [out.json] [--images N] [--rounds R]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from PIL import Image

from unet_pytorch_b200 import ops
from unet_pytorch_b200.nets.unet import Unet as UnetNet
from unet_pytorch_b200.unet import Unet as Predictor


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:           # the numbers stay valid; the record says the query failed
        info["power_limit_w"] = f"unavailable: {e}"
    return info


def per_image_get_miou(pred, images, gts):
    """The previous get_miou: host letterbox, batch-1 forward and single-image tail per image, pairs folded every 256."""
    n = pred.num_classes
    hist = torch.zeros(n * n + 1, dtype=torch.int64, device=pred.device)
    pairs = []
    for image, gt in zip(images, gts):
        _, data, nw, nh, oh, ow = pred._letterbox(image)
        with torch.no_grad():
            logits = pred.net(data.to(pred.device, non_blocking=True))
            mask = ops.softmax_resize_argmax_u8(logits, pred._crop(nw, nh), (oh, ow))[0]
        g = torch.from_numpy(np.ascontiguousarray(np.array(gt, dtype=np.uint8))).to(pred.device, non_blocking=True)
        if g.numel() != mask.numel():
            continue
        pairs.append((g.reshape(-1), mask.reshape(-1).contiguous()))
        if len(pairs) == 256:
            ops.fast_hist_batch(pairs, n, hist)
            pairs.clear()
    if pairs:
        ops.fast_hist_batch(pairs, n, hist)
    return hist.cpu().numpy()[:-1].reshape(n, n)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?")
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()
    torch.manual_seed(0)
    C = 21
    pred = Predictor(state_dict=UnetNet(num_classes=C, backbone="vgg").state_dict(), num_classes=C, backbone="vgg",
                     input_shape=[512, 512])
    rng = np.random.default_rng(0)
    images, gts = [], []
    for _ in range(args.images):
        w, h = (int(v) for v in rng.integers(200, 1201, 2))
        images.append(Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)))
        gts.append(rng.integers(0, C, (h, w), dtype=np.uint8))
    px = float(np.mean([im.size[0] * im.size[1] for im in images]))

    paths = {"per_image": lambda ims, gs: per_image_get_miou(pred, ims, gs),
             "batched_16": lambda ims, gs: pred.get_miou(ims, gs, batch_size=16)[0],
             "batched_64": lambda ims, gs: pred.get_miou(ims, gs, batch_size=64)[0]}
    for fn in paths.values():                       # warm-up: every batch shape the timed passes use
        fn(images[:64], gts[:64])
        fn(images[:1], gts[:1])
    times = {k: [] for k in paths}
    hists = {}
    for _ in range(args.rounds):
        for k, fn in paths.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            hists[k] = fn(images, gts)               # ends with the read-back of the confusion matrix
            times[k].append(time.perf_counter() - t0)
    same = all(np.array_equal(hists["per_image"], h) for h in hists.values())

    # host share per image
    t0 = time.perf_counter()
    for im in images:
        pred._prepare(im)
    prep_ms = (time.perf_counter() - t0) * 1e3 / len(images)
    t0 = time.perf_counter()
    for im in images[:128]:
        pred._letterbox(im)
    host_lb_ms = (time.perf_counter() - t0) * 1e3 / 128

    # device time per batch of 64 (CUDA events, 10 launches each): letterbox kernels, forward, batched tail
    prepared = [pred._prepare(im) for im in images[:64]]
    dev_ms = {}
    with torch.no_grad():
        masks, layout, nbytes, _, _ = pred._run_batch(prepared)        # leaves this batch's tables in the device staging buffer
        tail_at = ops.pad16(64 * ops.LETTERBOX_ITEM.size)
        x = pred._input[:64]
        logits = pred.net(x)
        sizes = [(h, w) for _, h, w in layout]
        steps = {"letterbox": lambda: ops.letterbox_bicubic(pred._dev_stage[:tail_at], 64, x, pred._lb_ws),
                 "forward": lambda: pred.net(x),
                 "tail": lambda: ops.softmax_resize_argmax_u8_batch(logits, pred._dev_stage[tail_at:], 64, masks,
                                                                    max(h for h, _ in sizes), max(w for _, w in sizes))}
        for k, fn in steps.items():
            fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                fn()
            e1.record()
            torch.cuda.synchronize()
            dev_ms[k] = round(e0.elapsed_time(e1) / 10, 3)

    res = {"card": card(), "config": {"images": args.images, "sides": [200, 1200], "mean_pixels": round(px),
                                      "num_classes": C, "model": "Unet-VGG16", "input_shape": [512, 512],
                                      "rounds": args.rounds},
           "same_hist_all_paths": bool(same), "images_per_s": {}, "seconds": {},
           "host_ms_per_image": {"batched_prepare": round(prep_ms, 3), "per_image_host_letterbox": round(host_lb_ms, 3)},
           "batch64_device_ms": dev_ms,
           "device_ms_per_image_batch64": round(sum(dev_ms.values()) / 64, 3)}
    for k, ts in times.items():
        res["seconds"][k] = [round(t, 3) for t in ts]
        res["images_per_s"][k] = round(args.images / min(ts), 1)
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")
    if not same:
        sys.exit("the batched and per-image paths gave different confusion matrices")


if __name__ == "__main__":
    main()
