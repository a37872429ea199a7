"""CPU: the numpy restatement of detect_image's rendering (oracle/render.py) against Pillow and against the expressions the
host predictor used, the item table of the device rendering, and the predictor's model names."""
import colorsys

import numpy as np
import pytest
from PIL import Image

from oracle import render as R


def test_blend_restatement_equals_pillow_on_every_byte_pair():
    """All 65536 (a, b) byte pairs: a in the rows, b in the columns of two RGB images."""
    a = np.repeat(np.arange(256, dtype=np.uint8)[:, None], 256, 1)
    b = a.T.copy()
    ia, ib = (Image.fromarray(np.stack([x] * 3, -1)) for x in (a, b))
    ref = np.asarray(Image.blend(ia, ib, 0.7))[..., 0]
    assert np.array_equal(R.blend(a, b), ref)
    f64 = (a + 0.7 * (b.astype(np.float64) - a)).astype(np.uint8)      # double arithmetic is not Pillow's
    assert (f64 != ref).sum() > 0


@pytest.mark.parametrize("h,w,seed", [(1, 1, 0), (37, 53, 1), (480, 640, 2)])
def test_blend_restatement_equals_pillow_on_images(h, w, seed):
    rng = np.random.default_rng(seed)
    a, b = (rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for _ in range(2))
    assert np.array_equal(R.blend(a, b), np.asarray(Image.blend(Image.fromarray(a), Image.fromarray(b), 0.7)))


@pytest.mark.parametrize("C", [2, 21, 150])
def test_palette_and_keep_equal_the_host_expressions(b2u, C):
    """mix_type 1 and 2 of oracle.render against the numpy expressions the host detect_image evaluated, with the
    predictor's own palette rule (VOC up to 21 classes, HSV beyond)."""
    from unet_pytorch_b200.unet import _voc_palette
    colors = _voc_palette(22) if C <= 21 else \
        [tuple(int(v * 255) for v in colorsys.hsv_to_rgb(x / C, 1.0, 1.0)) for x in range(C)]
    assert np.array_equal(R.palette(C), np.asarray(colors, np.uint8))
    rng = np.random.default_rng(C)
    img = rng.integers(0, 256, (31, 45, 3), dtype=np.uint8)
    pr = rng.integers(0, C, (31, 45)).astype(np.uint8)
    pr[:4] = 0
    seg = np.asarray(colors, np.uint8)[pr]
    assert np.array_equal(R.render(img, pr, 1, C), seg)
    assert np.array_equal(R.render(img, pr, 2, C), np.where((pr != 0)[..., None], img, 0).astype(np.uint8))
    blended = np.asarray(Image.blend(Image.fromarray(img), Image.fromarray(seg), 0.7))
    assert np.array_equal(R.render(img, pr, 0, C), blended)
    assert np.array_equal(R.render(img, pr, 5, C), img)


def test_render_table_layout(b2u):
    """One 32-byte item per image; rendered images at 16-byte aligned offsets after `start`, without overlap."""
    ops = b2u.ops
    items = [(0x1000, 0x9000, 3, 5), (0x2000, 0x9100, 1080, 1920), (0x3000, 0x9200, 1, 1)]
    table, offs, end = ops.render_table(items, start=8 * 3 * 21)
    assert len(table) == 32 * len(items) and offs[0] == ops.pad16(8 * 3 * 21)
    prev = offs[0]
    for i, (src, mask, h, w) in enumerate(items):
        assert ops.RENDER_ITEM.unpack_from(table, 32 * i) == (src, mask, offs[i], h, w)
        assert offs[i] % 16 == 0 and offs[i] >= prev
        prev = offs[i] + 3 * h * w
    assert end == ops.pad16(prev)
    with pytest.raises(ValueError):
        ops.render_table([(0x1000, 0x9000, 0, 5)])
    lib = b2u._lib.lib()
    assert lib.b2u_render_batch(None, 1, None, 21, 0, None, None, 100, None) == 1
    assert b"render_batch" in lib.b2u_last_error()
    assert lib.b2u_render_batch(None, 1, None, 21, 3, None, None, 100, None) != 0


def test_unknown_model_is_refused(b2u):
    from unet_pytorch_b200.unet import FAMILIES, Unet as Predictor
    with pytest.raises(ValueError, match="unknown model"):
        Predictor(model="segnet", state_dict={})
    assert sorted(FAMILIES) == sorted(set(b2u.UnetTrainer.ENGINES) - {"unet_vgg", "unet_resnet50"})
