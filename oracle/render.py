"""numpy restatement of the predictor's rendering (the reference's detect_image, unet.py:150-203), the yardstick of the
device rendering (csrc/render.cu).

Image.blend(a, b, alpha) computes, per byte, (UINT8)((int)a + alpha * ((int)b - (int)a)) with a C float alpha (Pillow's
Blend.c): float32 products and sums, no fused multiply-add, truncated towards zero.  numpy's float32 arithmetic rounds
each operation the same way; float64 differs on a few byte pairs."""
import colorsys

import numpy as np


def blend(a, b, alpha=0.7):
    """Image.blend of two uint8 arrays of one shape."""
    a = np.asarray(a, np.uint8)
    d = (np.asarray(b, np.int32) - a.astype(np.int32)).astype(np.float32)
    return (a.astype(np.float32) + np.float32(alpha) * d).astype(np.uint8)


def voc_palette(n):
    """The PASCAL VOC colour of class i: the bits of i spread over the top bits of r, g and b."""
    out = np.zeros((n, 3), np.uint8)
    for i in range(n):
        c, rgb = i, [0, 0, 0]
        for j in range(8):
            for k in range(3):
                rgb[k] |= ((c >> k) & 1) << (7 - j)
            c >>= 3
        out[i] = rgb
    return out


def palette(num_classes):
    """detect_image's table: the VOC colours up to 21 classes, evenly spaced hues beyond."""
    if num_classes <= 21:
        return voc_palette(22)
    return np.array([[int(v * 255) for v in colorsys.hsv_to_rgb(x / num_classes, 1.0, 1.0)] for x in range(num_classes)],
                    np.uint8)


def render(image, mask, mix_type, num_classes):
    """detect_image's output for an RGB uint8 image [h, w, 3] and its class mask [h, w]."""
    seg = palette(num_classes)[mask]
    if mix_type == 0:
        return blend(image, seg)
    if mix_type == 1:
        return seg
    if mix_type == 2:
        return np.where((mask != 0)[..., None], image, 0).astype(np.uint8)
    return np.asarray(image)
