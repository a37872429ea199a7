"""Restatement of Pillow's BICUBIC resize of 8-bit RGB images (Resample.c: precompute_coeffs, normalize_coeffs_8bpc,
ImagingResampleHorizontal_8bpc / Vertical_8bpc, ImagingResampleInner) and of the predictor's letterbox
(utils/utils.py:22-34 resize_image + preprocess_input + transpose) in numpy.  Test infrastructure only: the product
computes the same bytes in csrc/letterbox.cu.

Per axis with scale = in / out, fs = max(scale, 1), support = 2 fs, ksize = 2 ceil(support) + 1, and for output o:
center = (o + 0.5) scale, xmin = max(int(center - support + 0.5), 0), n = min(int(center + support + 0.5), in) - xmin,
w[k] = bicubic((k + xmin - center + 0.5) * (1 / fs)), normalised by their sequential double sum, then quantised to
22 fractional bits with round-half-away-from-zero.  Each pass sums 2^21 + sum(src * w) in int32 and stores
clamp(acc >> 22, 0, 255); horizontal pass first (vertical first when Image.resize takes its two-call path for an image
more than 100 times taller than wide whose height shrinks), and an axis whose size does not change is skipped."""
import math

import numpy as np

PRECISION_BITS = 22


def bicubic_filter(x):
    a = -0.5
    if x < 0.0:
        x = -x
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def ksize(inp, out):
    fs = max(inp / out, 1.0)
    return int(math.ceil(2.0 * fs)) * 2 + 1


def coeffs(inp, out):
    """(xmin int32 [out], n int32 [out], k int32 [out, ksize]) exactly as Pillow's 8-bit path uses them."""
    scale = inp / out
    fs = max(scale, 1.0)
    support = 2.0 * fs
    K = int(math.ceil(support)) * 2 + 1
    ss = 1.0 / fs
    xmin = np.zeros(out, np.int32)
    cnt = np.zeros(out, np.int32)
    kk = np.zeros((out, K), np.int32)
    for o in range(out):
        center = (o + 0.5) * scale
        lo = max(int(center - support + 0.5), 0)
        n = min(int(center + support + 0.5), inp) - lo
        w = [bicubic_filter((x + lo - center + 0.5) * ss) for x in range(n)]
        ww = 0.0
        for v in w:
            ww += v
        for x, v in enumerate(w):
            v = v / ww if ww != 0.0 else v
            kk[o, x] = int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS))
        xmin[o], cnt[o] = lo, n
    return xmin, cnt, kk


def _pass(src, inp, out, axis):
    """One 8-bit resampling pass of a uint8 HWC image along axis 1 (horizontal) or 0 (vertical)."""
    xmin, cnt, kk = coeffs(inp, out)
    s = np.moveaxis(src, axis, 0).astype(np.int64)                 # [in, other, 3]
    dst = np.empty((out,) + s.shape[1:], np.uint8)
    for o in range(out):
        taps = s[xmin[o]:xmin[o] + cnt[o]]
        acc = (1 << (PRECISION_BITS - 1)) + np.tensordot(kk[o, :cnt[o]].astype(np.int64), taps, axes=(0, 0))
        dst[o] = np.clip(acc >> PRECISION_BITS, 0, 255)
    return np.moveaxis(dst, 0, axis)


def resize_bicubic(src, size):
    """Image.fromarray(src).resize(size, Image.BICUBIC) for a uint8 [H, W, 3] array; size = (w, h)."""
    src = np.asarray(src, np.uint8)
    w, h = size
    ih, iw = src.shape[:2]
    out = src
    if ih > 100 * iw and h < ih:            # Image.resize: tall images shrinking in height go vertical first
        out = _pass(out, ih, h, 0)
        if w != iw:
            out = _pass(out, iw, w, 1)
        return np.ascontiguousarray(out)
    if w != iw:
        out = _pass(out, iw, w, 1)
    if h != ih:
        out = _pass(out, ih, h, 0)
    return np.ascontiguousarray(out)


def letterbox_geometry(iw, ih, w, h):
    """resize_image's (nw, nh, dx, dy) for an iw x ih image boxed into w x h."""
    scale = min(w / iw, h / ih)
    nw, nh = int(iw * scale), int(ih * scale)
    return nw, nh, (w - nw) // 2, (h - nh) // 2


def letterbox(src, w, h):
    """The predictor's network input for a uint8 [H, W, 3] image: fp32 [3, h, w], grey (128) bars, / 255."""
    ih, iw = src.shape[:2]
    nw, nh, dx, dy = letterbox_geometry(iw, ih, w, h)
    canvas = np.full((h, w, 3), 128, np.uint8)
    canvas[dy:dy + nh, dx:dx + nw] = resize_bicubic(src, (nw, nh))
    return np.transpose(canvas.astype(np.float32) / 255.0, (2, 0, 1))
