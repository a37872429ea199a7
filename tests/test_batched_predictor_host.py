"""CPU: the batched predictor's host pieces -- the numpy restatement of PIL's BICUBIC resize (oracle/pil_bicubic.py) against
Pillow itself, the letterbox geometry, the item tables of the device letterbox and of the batched tail, and the 16-byte
mask-offset layout that lets the ragged masks go straight to fast_hist_batch."""
import types

import numpy as np
import pytest
from PIL import Image

from oracle import pil_bicubic as B


def _rand(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


_GRID = [((1, 1), (1, 1)), ((1, 1), (5, 3)), ((1, 9), (4, 36)), ((9, 1), (36, 4)), ((1, 40), (1, 10)), ((40, 1), (10, 1)),
         ((7, 13), (7, 52)), ((7, 13), (28, 13)), ((16, 16), (4, 4)), ((16, 16), (64, 64)), ((30, 20), (8, 80)),
         ((33, 47), (132, 12)), ((64, 48), (16, 191)), ((100, 37), (25, 148)), ((5, 3), (512, 307)),
         ((257, 129), (65, 33)), ((200, 300), (150, 120)), ((700, 2), (512, 1)), ((250, 2), (100, 2)), ((1000, 3), (999, 2))]


@pytest.mark.parametrize("src,dst", _GRID)
def test_oracle_equals_pil_bicubic(src, dst):
    """Up and down by up to 4x per axis, 1xN, Nx1, 1x1, one axis unchanged, and images more than 100 times taller than
    wide (Image.resize runs their vertical pass first): byte for byte what Pillow produces."""
    a = _rand(*src, seed=src[0] * 1000 + src[1])
    ref = np.asarray(Image.fromarray(a).resize((dst[1], dst[0]), Image.BICUBIC))
    got = B.resize_bicubic(a, (dst[1], dst[0]))
    assert got.shape == ref.shape and np.array_equal(got, ref)


def test_oracle_coefficients_are_pillows_rules():
    """Weights sum to ~2^22 per output, support follows max(scale, 1), and an unchanged axis is an identity filter."""
    for inp, out in [(1920, 512), (512, 1920), (3, 307), (17, 17)]:
        xmin, n, k = B.coeffs(inp, out)
        assert k.shape == (out, B.ksize(inp, out)) and (n <= k.shape[1]).all() and (xmin + n <= inp).all()
        assert np.abs(k.sum(1) - (1 << 22)).max() <= n.max()
    xmin, n, k = B.coeffs(9, 9)
    assert all(k[o, o - xmin[o]] == 1 << 22 and k[o].sum() == 1 << 22 for o in range(9))


def test_oracle_letterbox_equals_resize_image(b2u):
    """oracle.letterbox is the predictor's host letterbox (resize_image + preprocess_input + transpose) for RGB images."""
    from unet_pytorch_b200.unet import Unet as Predictor
    fake = types.SimpleNamespace(input_shape=[96, 128])
    for h, w in [(50, 70), (300, 120), (96, 128), (1, 3)]:
        img = Image.fromarray(_rand(h, w, seed=h + w))
        _, data, nw, nh, oh, ow = Predictor._letterbox(fake, img)
        assert (oh, ow) == (h, w) and (nw, nh) == B.letterbox_geometry(w, h, 128, 96)[:2]
        assert np.array_equal(data[0].numpy(), B.letterbox(np.asarray(img), 128, 96))


def test_prepare_geometry_and_conversion(b2u):
    """Predictor._prepare: cvtColor's rule (3-channel images as they are, others converted to RGB), resize_image's
    (nh, nw, dy, dx), and ValueError for an empty image or one that letterboxes to zero pixels."""
    from unet_pytorch_b200.unet import Unet as Predictor, resize_image
    fake = types.SimpleNamespace(input_shape=[512, 512])
    for size, mode in [((500, 375), "RGB"), ((375, 500), "L"), ((512, 512), "P"), ((4000, 3000), "RGBA"), ((3, 900), "RGB")]:
        img = Image.new(mode, size)
        conv, arr, (ih, iw, nh, nw, dy, dx) = Predictor._prepare(fake, img)
        assert conv.mode == "RGB" and arr.shape == (size[1], size[0], 3) and arr.dtype == np.uint8 and arr.flags.c_contiguous
        _, rnw, rnh = resize_image(conv, (512, 512))
        assert (ih, iw, nh, nw) == (size[1], size[0], rnh, rnw)
        assert (dy, dx) == ((512 - nh) // 2, (512 - nw) // 2)
    assert Predictor._prepare(fake, Image.new("RGB", (512, 512)))[2] == (512, 512, 512, 512, 0, 0)   # exact fit, no bars
    with pytest.raises(ValueError):
        Predictor._prepare(fake, Image.new("RGB", (0, 0)))
    with pytest.raises(ValueError):
        Predictor._prepare(fake, Image.new("RGB", (1, 1000)))        # 1 * 0.512 -> zero columns


def test_letterbox_plan_fills_the_item_table(b2u):
    """b2u_letterbox_workspace (host-only): taps per axis as Pillow's ksize, 0 for an unchanged axis, 16-byte aligned,
    non-overlapping workspace regions; items that do not fit the canvas are refused."""
    ops = b2u.ops
    geo = [(0x1000, 375, 500, 384, 512, 64, 0), (0x2000, 512, 512, 512, 512, 0, 0), (0x3000, 3000, 4000, 384, 512, 64, 0),
           (0x4000, 9, 3, 512, 170, 0, 171), (0x5000, 300, 512, 300, 512, 106, 0)]
    table, ws = ops.letterbox_plan(geo, 512, 512)
    assert len(table) == 64 * len(geo)
    end = 0
    for i, (_, ih, iw, nh, nw, dy, dx) in enumerate(geo):
        f = ops.LETTERBOX_ITEM.unpack_from(table, 64 * i)
        assert f[1:7] == (ih, iw, nh, nw, dy, dx)
        kx, ky, cx, cy, tmp = f[7:]
        assert kx == (B.ksize(iw, nw) if nw != iw else 0) and ky == (B.ksize(ih, nh) if nh != ih else 0)
        assert cx % 16 == 0 and cy % 16 == 0 and tmp % 16 == 0 and cx >= end
        assert cy >= cx + (nw * (8 + 4 * kx) if kx else 0) and tmp >= cy + (nh * (8 + 4 * ky) if ky else 0)
        end = tmp + (ih * nw * 3 if kx else 0)
    assert ws >= end
    assert dict(zip(("kx", "ky"), ops.LETTERBOX_ITEM.unpack_from(table, 128)[7:9])) == {"kx": 33, "ky": 33}
    with pytest.raises(ValueError):
        ops.letterbox_plan([(0x1000, 375, 500, 384, 512, 129, 0)], 512, 512)      # one row past the canvas
    with pytest.raises(ValueError):
        ops.letterbox_plan([(0, 375, 500, 384, 512, 64, 0)], 512, 512)            # no source
    with pytest.raises(ValueError):
        ops.letterbox_plan([], 512, 512)


def test_tail_table_mask_offsets(b2u):
    """Ragged masks: each offset is a multiple of 16 and the previous mask ends at or before it; crops outside the
    logits are refused."""
    ops = b2u.ops
    sizes = [(375, 500), (1, 1), (17, 3), (512, 512), (333, 777)]
    crops = [(64, 0, 384, 512), (0, 0, 512, 512), (0, 170, 512, 170), (0, 0, 512, 512), (138, 0, 236, 512)]
    table, offs, total = ops.tail_table(crops, sizes, 512, 512)
    assert len(table) == 32 * len(sizes)
    prev_end = 0
    for i, ((cy, cx, ch, cw), (oh, ow)) in enumerate(zip(crops, sizes)):
        assert ops.TAIL_ITEM.unpack_from(table, 32 * i) == (cy, cx, ch, cw, oh, ow, offs[i])
        assert offs[i] % 16 == 0 and offs[i] >= prev_end and offs[i] - prev_end < 16
        prev_end = offs[i] + oh * ow
    assert total == ops.pad16(prev_end)
    with pytest.raises(ValueError):
        ops.tail_table([(1, 0, 512, 512)], [(10, 10)], 512, 512)
    with pytest.raises(ValueError):
        ops.tail_table([(0, 0, 512, 512)], [(0, 10)], 512, 512)
