"""Predictor throughput for every model family, and detect_image's rendering on the host against the device.

1. `Unet.get_FPS` at batch 1 (forward [+ resize] + per-pixel class + crop, result on the host) for every family, at the
   reference's protocol (4 classes, 256x256 input; its Submit_result reports 82.75 FPS for TraditionalUnet and 105.41 FPS
   for UltraLightweightUnet_large_optimized on hardware it does not name) and at 21 classes, 512x512.
2. `Unet.get_miou` images/s at batch 16 per family over the seeded synthetic set of scripts/predictor_bench.py (RGB
   images with sides from 200 to 1200, uint8 ground truths, 21 classes, 512x512 input).
3. 1920x1080 frames, mix_type 0 and 2: the previous detect_image (device mask read back, then palette lookup,
   Image.blend / np.where on the host; restated below) against detect_image / detect_images rendering on the device.  The
   two run alternately in one call and must give the same bytes.  The render launch's own device time comes from CUDA
   events around each C-ABI call (_lib.CallProfile) in a separate pass.

Weights are seeded He-normal (synthetic.random_state_dict): throughput does not depend on their values.

usage: python scripts/predictor_families_bench.py [out.json] [--images N] [--frames N] [--fps-frames N]"""
import argparse
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np
import torch
from PIL import Image

from predictor_bench import card
from unet_pytorch_b200 import _lib
from unet_pytorch_b200.nets.unet import Unet as UnetNet
from unet_pytorch_b200.synthetic import random_state_dict
from unet_pytorch_b200.unet import FAMILIES, Unet as Predictor

MODELS = [("unet", "vgg"), ("unet", "resnet50")] + [(m, None) for m in FAMILIES]
PUBLISHED_FPS_NC4_256 = {"traditional": 82.75, "ultralight_large_optimized": 105.41}


def name(model, backbone):
    return f"unet_{backbone}" if model == "unet" else model


def predictor(model, backbone, C, size):
    m = UnetNet(num_classes=C, backbone=backbone) if model == "unet" else FAMILIES[model](num_classes=C)
    sd = random_state_dict({k: tuple(v.shape) for k, v in m.named_parameters()},
                           {k: tuple(v.shape) for k, v in m.named_buffers()}, seed=0)
    return Predictor(model=model, backbone=backbone or "vgg", state_dict=sd, num_classes=C, input_shape=[size, size])


def host_detect_image(pred, image):
    """The previous detect_image: the mask read back, rendered on the host."""
    old_img, pr = pred.predict_mask(image)
    if pred.mix_type == 2:
        return Image.fromarray(np.where((pr != 0)[..., None], np.asarray(old_img), 0).astype(np.uint8))
    seg = Image.fromarray(np.asarray(pred.colors, np.uint8)[pr])
    return Image.blend(old_img, seg, 0.7) if pred.mix_type == 0 else seg


def host_render_only(pred, image, pr):
    if pred.mix_type == 2:
        return Image.fromarray(np.where((pr != 0)[..., None], np.asarray(image), 0).astype(np.uint8))
    return Image.blend(image, Image.fromarray(np.asarray(pred.colors, np.uint8)[pr]), 0.7)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?")
    ap.add_argument("--images", type=int, default=512)
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--fps-frames", type=int, default=100)
    args = ap.parse_args()
    rng = np.random.default_rng(0)
    res = {"card": card(), "get_fps": {}, "get_miou_batch16": {}, "render_1920x1080": {}}

    # 1. get_FPS, batch 1
    fps_image = Image.fromarray(rng.integers(0, 256, (375, 500, 3), dtype=np.uint8))
    for C, size in ((4, 256), (21, 512)):
        key = f"nc{C}_{size}x{size}"
        res["get_fps"][key] = {}
        for model, bb in MODELS:
            pred = predictor(model, bb, C, size)
            pred.get_FPS(fps_image, 10)                                      # warm-up
            secs = [pred.get_FPS(fps_image, args.fps_frames) for _ in range(2)]
            rec = {"fps": round(1.0 / min(secs), 1), "ms_per_frame": [round(s * 1e3, 3) for s in secs]}
            if C == 4 and model in PUBLISHED_FPS_NC4_256:
                rec["reference_published_fps"] = PUBLISHED_FPS_NC4_256[model]
                rec["reference_hardware"] = "unknown (Submit_result does not name it)"
            res["get_fps"][key][name(model, bb)] = rec
            del pred
    res["get_fps"]["config"] = {"test_interval": args.fps_frames, "image": [500, 375], "rounds": 2, "best_of_rounds": True}

    # 2. get_miou, batch 16
    C = 21
    images, gts = [], []
    for _ in range(args.images):
        w, h = (int(v) for v in rng.integers(200, 1201, 2))
        images.append(Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)))
        gts.append(rng.integers(0, C, (h, w), dtype=np.uint8))
    for model, bb in MODELS:
        pred = predictor(model, bb, C, 512)
        pred.get_miou(images[:32], gts[:32], batch_size=16)                # warm-up
        secs = [timed(lambda: pred.get_miou(images, gts, batch_size=16))[0] for _ in range(2)]
        res["get_miou_batch16"][name(model, bb)] = {"images_per_s": round(args.images / min(secs), 1),
                                                    "seconds": [round(s, 3) for s in secs]}
        del pred
    res["get_miou_batch16"]["config"] = {"images": args.images, "sides": [200, 1200], "num_classes": C,
                                         "input_shape": [512, 512], "rounds": 2, "best_of_rounds": True}

    # 3. rendering of 1920x1080 frames
    pred = predictor("unet", "vgg", 21, 512)
    frames = [Image.fromarray(rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8)) for _ in range(args.frames)]
    for mix in (0, 2):
        pred.mix_type = mix
        paths = {"host_rendering_batch1": lambda: [host_detect_image(pred, f) for f in frames],
                 "device_rendering_batch1": lambda: [pred.detect_image(f) for f in frames],
                 "device_rendering_batch16": lambda: pred.detect_images(frames, batch_size=16)}
        for fn in paths.values():
            fn()
        secs, outs = {k: [] for k in paths}, {}
        for _ in range(2):
            for k, fn in paths.items():
                t, outs[k] = timed(fn)
                secs[k].append(t)
        same = all(np.array_equal(np.asarray(a), np.asarray(b)) for k in paths for a, b in zip(outs[k], outs["host_rendering_batch1"]))
        masks = [pred.predict_mask(f)[1] for f in frames[:8]]
        t0 = time.perf_counter()
        for f, m in zip(frames[:8], masks):
            host_render_only(pred, f, m)
        render_host_ms = (time.perf_counter() - t0) * 1e3 / 8
        with _lib.CallProfile() as prof:
            pred.detect_images(frames, batch_size=16)
        rk = prof.read().get("b2u_render_batch", {"launches": 0, "ms": float("nan")})
        res["render_1920x1080"][f"mix_type_{mix}"] = {
            "same_bytes_all_paths": bool(same),
            "ms_per_frame": {k: round(min(v) * 1e3 / len(frames), 3) for k, v in secs.items()},
            "host_rendering_only_ms_per_frame": round(render_host_ms, 3),
            "device_render_kernel_ms_per_frame": round(rk["ms"] / len(frames), 4),
            "device_render_launches": rk["launches"]}
        if not same:
            sys.exit(f"mix_type {mix}: the device rendering differs from the host rendering")
    res["render_1920x1080"]["config"] = {"frames": args.frames, "model": "Unet-VGG16", "num_classes": 21,
                                         "input_shape": [512, 512], "rounds": 2, "best_of_rounds": True}
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
