"""GPU: every CUDA kernel behind the C ABI against fp32 CPU references on the same seeded inputs.
bf16 kernels: rel-L2 <= 6e-3 against the fp32 result of the same bf16-rounded operands (output rounding only);
fp32 kernels (head, losses, wgrad accumulation): <= 1e-4; integer kernels: exact."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def nhwc(x, dev):
    return x.permute(0, 2, 3, 1).contiguous().to(BF).to(dev)


def nchw(x):
    return x.float().permute(0, 3, 1, 2).contiguous().cpu()


CONV_CASES = [
    # N, H, W, C0, C1, Cout, taps, relu
    (1, 8, 16, 64, 0, 64, 9, True),        # exactly one tile
    (2, 24, 40, 64, 0, 64, 9, True),       # Cout = 64 with ragged tiles in both directions (swapped-role wgrad)
    (3, 5, 7, 128, 64, 64, 9, False),      # Cout = 64, image smaller than a tile, two sources, three cin blocks
    (2, 32, 48, 64, 0, 64, 9, True),       # exactly one stack of four M tiles
    (1, 72, 40, 64, 64, 64, 9, True),      # four-tile stacks with a ragged last stack (72 = 2 x 32 + 8) and two sources
    (2, 24, 40, 128, 0, 128, 9, True),     # ragged tiles in both directions
    (1, 16, 16, 256, 0, 256, 9, False),
    (1, 16, 16, 512, 0, 512, 9, True),
    (1, 16, 32, 64, 128, 64, 9, True),     # virtual concat; dgrad N tile 192 split 64|128
    (1, 16, 16, 512, 512, 512, 9, True),   # up_concat4.conv1 shape
    (1, 4, 4, 512, 0, 512, 9, True),       # image smaller than the 8x16 tile
    (2, 16, 16, 64, 0, 128, 1, False),     # 1x1
    (1, 64, 64, 128, 256, 128, 9, True),   # dgrad 384 = 2 x 192
]


@pytest.mark.parametrize("N,H,W,C0,C1,Cout,taps,relu", CONV_CASES)
def test_conv_fprop_dgrad_wgrad(b2u, cuda_device, N, H, W, C0, C1, Cout, taps, relu):
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(1)
    k = 3 if taps == 9 else 1
    x = torch.randn(N, C0 + C1, H, W, generator=g)
    w = torch.randn(Cout, C0 + C1, k, k, generator=g) / ((C0 + C1) * taps) ** 0.5
    b = torch.randn(Cout, generator=g)
    xb = nhwc(x, dev); xr = nchw(xb)
    wr = w.to(BF).float()
    wf, wd = ops.pack_weights(w.to(dev))
    x0 = xb[..., :C0].contiguous(); x1 = xb[..., C0:].contiguous() if C1 else None
    ref = F.conv2d(xr, wr, b, padding=k // 2)
    ref = ref.relu() if relu else ref
    # every tiling the launcher can pick: default, one M tile per CTA step (bit 16), each legal N tile
    # bit 17: at most two stacked M tiles (the unmasked N = 64 layers default to four when H >= 32)
    variants = [0, 1 << 16, 2 << 16] + [bn for bn in (64, 128, 192, 256) if Cout % bn == 0] + [(1 << 16) | 64, (2 << 16) | 64]
    for bn in variants:
        y = ops.conv_fprop(x0, wf, b.to(dev), Cout, taps=taps, relu=relu, x1=x1, bn=bn)
        assert rel(nchw(y), ref) <= 6e-3, f"tiling variant {bn:#x}"
    dz = torch.randn(N, Cout, H, W, generator=g)
    dzb = nhwc(dz, dev); dzr = nchw(dzb)
    ref_dx = F.conv_transpose2d(dzr, wr, padding=k // 2)
    if C1:
        d0, d1 = ops.conv_dgrad(dzb, wd, C0, taps=taps, C1=C1)
        assert rel(torch.cat([nchw(d0), nchw(d1)], 1), ref_dx) <= 6e-3
    else:
        mask = nhwc(torch.randn(N, C0, H, W, generator=g), dev)
        d0 = ops.conv_dgrad(dzb, wd, C0, taps=taps, mask=mask)
        assert rel(nchw(d0), ref_dx * (nchw(mask) > 0)) <= 6e-3
        # the same launch leaving the column sums of what it stores: the bias gradient of the conv below without a pass over dz
        rows = ops.conv_dgrad_stat_rows(N, H, W, C0, taps, masked=True)
        st = torch.full((rows * 2 * C0,), float("nan"), device=dev)
        d0s = ops.conv_dgrad(dzb, wd, C0, taps=taps, mask=mask, stats=st)
        assert torch.equal(d0s.view(torch.int16), d0.view(torch.int16))
        assert rel(ops.bias_from_stats(st, rows, C0), nchw(d0).double().sum((0, 2, 3))) <= 1e-5
    ref_dw = torch.nn.grad.conv2d_weight(xr, w.shape, dzr, padding=k // 2)
    dw, db = ops.conv_wgrad(x0, dzb, taps=taps, x1=x1, want_db=True)
    assert rel(dw, ref_dw) <= 1e-4
    assert rel(db, dzr.sum((0, 2, 3))) <= 1e-4      # bias gradient fused into the wgrad kernel
    # without db: Cout = 64 3x3 layers take the swapped-role kernel (x as the M operand, three shifted dz boxes as N);
    # flags bit 1 forces the generic kernel
    assert rel(ops.conv_wgrad(x0, dzb, taps=taps, x1=x1), ref_dw) <= 1e-4
    assert rel(ops.conv_wgrad(x0, dzb, taps=taps, x1=x1, flags=2), ref_dw) <= 1e-4
    assert rel(ops.bias_grad(dzb), dzr.sum((0, 2, 3))) <= 1e-4


def _bits_of(y):
    """(y > 0) packed like the kernels do: int64 [N, H, W, C // 64], bit c % 64 of word c // 64."""
    N, H, W, C = y.shape
    b = (y.float() > 0).view(N, H, W, C // 64, 64).to(torch.int64)
    sh = torch.arange(64, device=y.device, dtype=torch.int64)
    return (b << sh).sum(-1)          # bit 63 wraps into the sign bit: exactly the two's-complement word


@pytest.mark.parametrize("N,H,W,C0,C1,Cout,taps", [(1, 8, 16, 64, 0, 64, 9), (2, 40, 24, 64, 0, 64, 9), (1, 72, 40, 64, 64, 64, 9),
                                                     (2, 24, 40, 128, 0, 128, 9), (1, 16, 16, 256, 0, 512, 9), (2, 16, 24, 64, 0, 64, 1),
                                                     (1, 16, 32, 64, 128, 192, 9)])
def test_relu_bit_masks(b2u, cuda_device, N, H, W, C0, C1, Cout, taps):
    """ReLU backward from bit masks: b2u_conv_fprop_relu_bits writes (y > 0) as one bit per channel next to a bit-identical y,
    and b2u_conv_dgrad_bits masks with those bits exactly like b2u_conv_dgrad does with y itself (bit-identical dx, same
    column sums), while tiling like an unmasked launch."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(23)
    k = 3 if taps == 9 else 1
    x = nhwc(torch.randn(N, C0 + C1, H, W, generator=g), dev)
    w = torch.randn(Cout, C0 + C1, k, k, generator=g) / ((C0 + C1) * taps) ** 0.5
    b = torch.randn(Cout, generator=g).to(dev)
    wf, _ = ops.pack_weights(w.to(dev))
    x0 = x[..., :C0].contiguous(); x1 = x[..., C0:].contiguous() if C1 else None
    y = ops.conv_fprop(x0, wf, b, Cout, taps=taps, relu=True, x1=x1)
    bits = torch.zeros(N, H, W, Cout // 64, dtype=torch.int64, device=dev)
    yb = ops.conv_fprop_relu_bits(x0, wf, b, Cout, bits, taps=taps, x1=x1)
    assert torch.equal(yb.view(torch.int16), y.view(torch.int16))
    assert torch.equal(bits, _bits_of(y))
    assert 0.2 < (y > 0).float().mean().item() < 0.8                      # a real mask, not all ones / zeros
    # the backward of a conv that READS y: dz has Cz channels, dx has Cout (= y's) channels
    Cz = 128
    wn = torch.randn(Cz, Cout, k, k, generator=g) / (Cout * taps) ** 0.5
    _, wd = ops.pack_weights(wn.to(dev))
    dz = nhwc(torch.randn(N, Cz, H, W, generator=g), dev)
    ref = ops.conv_dgrad(dz, wd, Cout, taps=taps, mask=y)
    got = ops.conv_dgrad_bits(dz, wd, Cout, bits, taps=taps)
    assert torch.equal(got.view(torch.int16), ref.view(torch.int16))
    rows = ops.conv_dgrad_stat_rows(N, H, W, Cout, taps, masked=False)
    st = torch.full((rows * 2 * Cout,), float("nan"), device=dev)
    got2 = ops.conv_dgrad_bits(dz, wd, Cout, bits, taps=taps, stats=st)
    assert torch.equal(got2.view(torch.int16), ref.view(torch.int16))
    assert rel(ops.bias_from_stats(st, rows, Cout), nchw(ref).double().sum((0, 2, 3))) <= 1e-5


def test_relu_bit_masks_decoder_conv(b2u, cuda_device):
    """The decoder conv (fused up-sampling) writes the same bit mask as the plain conv over the materialised up-sampled tensor."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(29)
    N, H, W, C0, C1, Cout = 2, 40, 24, 64, 128, 128
    skip = nhwc(torch.randn(N, C0, H, W, generator=g), dev)
    low = nhwc(torch.randn(N, C1, H // 2, W // 2, generator=g), dev)
    w = torch.randn(Cout, C0 + C1, 3, 3, generator=g) / ((C0 + C1) * 9) ** 0.5
    b = torch.randn(Cout, generator=g).to(dev)
    wf, _ = ops.pack_weights(w.to(dev))
    up = ops.upsample2x(low)
    y = ops.conv_fprop(skip, wf, b, Cout, relu=True, x1=up)
    bits = torch.zeros(N, H, W, Cout // 64, dtype=torch.int64, device=dev)
    up_out = torch.empty_like(up)
    yb = ops.conv_fprop_relu_bits(skip, wf, b, Cout, bits, low=low, up_out=up_out)
    assert torch.equal(yb.view(torch.int16), y.view(torch.int16)) and torch.equal(up_out.view(torch.int16), up.view(torch.int16))
    assert torch.equal(bits, _bits_of(y))


DECODER_CASES = [
    # N, H, W, C0 (skip), C1 (low), Cout -- H, W of the conv (the low tensor is H/2 x W/2)
    (1, 8, 16, 64, 64, 64),        # one tile, one M tile per step
    (2, 16, 32, 64, 128, 64),      # up_concat1.conv1 proportions, two stacked M tiles
    (1, 48, 40, 64, 128, 64),      # exactly one stack of three M tiles
    (1, 104, 36, 128, 64, 64),     # three-tile stacks, ragged in both directions, two skip blocks
    (2, 24, 40, 128, 256, 128),    # N tile 128, ragged
    (1, 8, 8, 64, 64, 128),        # N tile 128, one M tile
    (1, 16, 16, 256, 512, 256),    # up_concat3.conv1 proportions, N tile 256
    (1, 4, 4, 512, 512, 512),      # image smaller than a tile: the 2x2 low tensor, two N tiles
    (1, 12, 20, 64, 64, 192),      # N tile 192
    (3, 6, 10, 64, 64, 64),        # odd low-resolution sizes (3 x 5)
    (8, 128, 256, 64, 64, 64),     # 512 / 1024 / 2048 tiles: every CTA of the persistent grid walks several tiles (slot hand-off phases)
    (4, 64, 128, 64, 128, 256),    # the same for the wide N tiles (256 tiles; 512 with N tile 128; 1024 with N tile 64)
]


@pytest.mark.parametrize("N,H,W,C0,C1,Cout", DECODER_CASES)
def test_decoder_conv_fused_upsample(b2u, cuda_device, N, H, W, C0, C1, Cout):
    """b2u_decoder_conv_fprop (bilinear 2x up-sampling + concat folded into the conv's operand load, nets/unet.py:16-18)
    against the two-kernel path it replaces: BIT-identical outputs, the by-product up-sampled tensor bit-identical to
    b2u_upsample2x_fwd, and both within 6e-3 of torch's fp32 upsample + cat + conv on the same bf16 operands."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(17)
    skip = nhwc(torch.randn(N, C0, H, W, generator=g), dev)
    low = nhwc(torch.randn(N, C1, H // 2, W // 2, generator=g), dev)
    w = torch.randn(Cout, C0 + C1, 3, 3, generator=g) / ((C0 + C1) * 9) ** 0.5
    b = torch.randn(Cout, generator=g).to(dev)
    wf, _ = ops.pack_weights(w.to(dev))
    up = ops.upsample2x(low)
    variants = [0, 1 << 16, 2 << 16] + [bn for bn in (64, 128, 192, 256) if Cout % bn == 0] + [(1 << 16) | 64, (2 << 16) | 64]
    ref = F.conv2d(torch.cat([nchw(skip), F.interpolate(nchw(low), scale_factor=2, mode="bilinear", align_corners=True)], 1),
                   w.to(BF).float(), b.cpu(), padding=1).relu()
    for bn in variants:
        two = ops.conv_fprop(skip, wf, b, Cout, relu=True, x1=up, bn=bn)
        up_out = torch.full_like(up, float("nan"))
        one = ops.decoder_conv_fprop(skip, low, wf, b, Cout, relu=True, up_out=up_out, bn=bn)
        assert torch.equal(one.view(torch.int16), two.view(torch.int16)), f"tiling variant {bn:#x}"
        assert torch.equal(up_out.view(torch.int16), up.view(torch.int16)), f"by-product, tiling variant {bn:#x}"
        assert rel(nchw(one), ref) <= 6e-3
        # inference form: no by-product
        assert torch.equal(ops.decoder_conv_fprop(skip, low, wf, b, Cout, relu=True, bn=bn).view(torch.int16), two.view(torch.int16))
    # BatchNorm statistics from the epilogue and the folded eval-mode BatchNorm ride on the same kernel
    rows2, rows1 = ops.conv_stat_rows(N, H, W, Cout), ops.conv_stat_rows(N, H, W, Cout, bn=1 << 18)     # bit 18: the decoder conv's tiles
    st1 = torch.zeros(rows1 * 2 * Cout, device=dev); st2 = torch.zeros(rows2 * 2 * Cout, device=dev)
    z2 = ops.conv_fprop(skip, wf, b, Cout, relu=False, x1=up, stats=st2)
    z1 = ops.decoder_conv_fprop(skip, low, wf, b, Cout, relu=False, stats=st1)
    assert torch.equal(z1.view(torch.int16), z2.view(torch.int16))
    # the two kernels cut the image into different tiles: the per-tile sums differ, their totals agree to fp32 summation order
    t1, t2 = st1.view(rows1, 2, Cout).double().sum(0), st2.view(rows2, 2, Cout).double().sum(0)
    assert torch.allclose(t1, t2, rtol=1e-5, atol=1e-3)
    sc = (torch.rand(Cout, generator=g) + 0.5).to(dev)
    y2 = ops.conv_fprop_scaled(skip, wf, sc, b, Cout, relu=True, x1=up)
    y1 = ops.decoder_conv_fprop(skip, low, wf, b, Cout, relu=True, scale=sc)
    assert torch.equal(y1.view(torch.int16), y2.view(torch.int16))


def test_first_layer_im2col_conv(b2u, cuda_device):
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(2)
    x = torch.rand(2, 3, 32, 48, generator=g)
    w = torch.randn(64, 3, 3, 3, generator=g) / 27 ** 0.5
    b = torch.randn(64, generator=g)
    col = ops.im2col_first(x.to(dev))
    y = ops.conv_fprop(col, ops.pack_weights_first(w.to(dev)), b.to(dev), 64, taps=1, relu=True)
    ref = F.conv2d(x, w.to(BF).float(), b, padding=1).relu()          # x itself: the image is a two-term bf16 split
    assert rel(nchw(y), ref) <= 6e-3
    dzb = nhwc(torch.randn(2, 64, 32, 48, generator=g), dev)
    dw = ops.conv_wgrad(col, dzb, taps=1, first_cin=3)
    # the image enters as a two-term bf16 split (hi + lo columns of the im2col row): the weight gradient sees x itself
    ref_dw = torch.nn.grad.conv2d_weight(x, w.shape, nchw(dzb), padding=1)
    assert rel(dw, ref_dw) <= 1e-4


@pytest.mark.parametrize("N,H,W,C", [(2, 16, 32, 64), (1, 8, 8, 128), (1, 2, 2, 512), (3, 6, 10, 8)])
def test_pool_and_upsample(b2u, cuda_device, N, H, W, C):
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(3)
    xb = nhwc(torch.randn(N, C, H, W, generator=g).relu(), dev)
    xr = nchw(xb).requires_grad_(True)
    ref = F.max_pool2d(xr, 2, 2)
    assert torch.equal(nchw(ops.maxpool2x2(xb)), ref.detach())
    dp = nhwc(torch.randn(N, C, H // 2, W // 2, generator=g), dev)
    dsk = nhwc(torch.randn(N, C, H, W, generator=g), dev)
    ref.backward(nchw(dp))
    want = (xr.grad + nchw(dsk)) * (xr > 0)
    assert rel(nchw(ops.maxpool2x2_bwd(dp, xb, dskip=dsk, relu_mask=True)), want) <= 4e-3
    xr2 = nchw(xb).requires_grad_(True)
    refu = F.interpolate(xr2, scale_factor=2, mode="bilinear", align_corners=True)   # nets/unet.py:13
    assert rel(nchw(ops.upsample2x(xb)), refu.detach()) <= 4e-3
    du = nhwc(torch.randn(N, C, 2 * H, 2 * W, generator=g), dev)
    refu.backward(nchw(du))
    assert rel(nchw(ops.upsample2x_bwd(du, ylow=xb)), xr2.grad * (xr2 > 0)) <= 4e-3


@pytest.mark.parametrize("C,use_onehot,cw", [(21, False, None), (4, True, [1, 15, 1.5, 2]), (2, True, [1, 1]), (4, False, [1, 15, 0, 0])])
def test_head_and_losses_against_oracle(b2u, cuda_device, C, use_onehot, cw):
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(4)
    N, H, W = 2, 32, 48
    xb = nhwc(torch.randn(N, 64, H, W, generator=g).relu(), dev)
    xr = nchw(xb).requires_grad_(True)
    w = (torch.randn(C, 64, 1, 1, generator=g) / 8).requires_grad_(True)
    b = torch.randn(C, generator=g).requires_grad_(True)
    logits = ops.head_fwd(xb, w.detach().reshape(C, 64).contiguous().to(dev), b.detach().to(dev))
    ref = F.conv2d(xr, w, b)
    assert rel(logits, ref) <= 1e-5
    png = torch.randint(0, C + 1, (N, H, W), generator=g)
    oh = O.one_hot(png, C)
    weights = torch.ones(C) if cw is None else torch.tensor(cw, dtype=torch.float32)
    ce, fo = O.ce_loss(ref, png, weights, C), O.focal_loss(ref, png, weights, C)
    di, fs = O.dice_loss(ref, oh), O.f_score(ref, oh)
    fin = ops.loss_fwd(logits, target=png.to(dev), onehot=oh.to(dev) if use_onehot else None, cls_w=weights.to(dev)).cpu()
    for got, want in zip(fin[:4], (ce, fo, di, fs)):
        assert abs(got.item() - want.item()) <= 2e-5 * max(abs(want.item()), 1e-3)
    for gs, loss in (([1, 0, 0], ce), ([0, 1, 0], fo), ([0, 0, 1], di), ([1, 0, 1], ce + di)):
        gl, = torch.autograd.grad(loss, ref, retain_graph=True)
        dl = ops.loss_bwd(logits, fin.to(dev), torch.tensor(gs, dtype=torch.float32, device=dev), target=png.to(dev),
                          onehot=oh.to(dev) if use_onehot else None, cls_w=weights.to(dev))
        assert rel(dl, gl) <= 2e-4
    # tensor-core head backward operands: dlogits as a two-term bf16 split [hi(32) | lo(32)] in NHWC64
    gs = torch.tensor([1, 0, 1], dtype=torch.float32, device=dev)
    gl, = torch.autograd.grad(ce + di, ref, retain_graph=True)
    d64 = ops.loss_bwd(logits, fin.to(dev), gs, target=png.to(dev), onehot=oh.to(dev) if use_onehot else None,
                       cls_w=weights.to(dev), nhwc64=True).float().cpu()
    assert d64.shape == (N, H, W, 64)
    recon = (d64[..., :C] + d64[..., 32:32 + C]).permute(0, 3, 1, 2)
    assert rel(recon, gl) <= 2e-5
    assert d64[..., C:32].abs().max() == 0 and d64[..., 32 + C:].abs().max() == 0
    wd = ops.pack_head_dgrad(w.detach().reshape(C, 64).contiguous().to(dev)).float().cpu()
    assert torch.equal(wd[:, :C], w.detach().reshape(C, 64).to(BF).float().t()) and torch.equal(wd[:, 32:32 + C], wd[:, :C])
    (ce + di).backward()
    dx, dw, db = ops.head_bwd(gl.contiguous().to(dev), xb, w.detach().reshape(C, 64).contiguous().to(dev))
    assert rel(nchw(dx), xr.grad * (xr > 0)) <= 4e-3
    assert rel(dw, w.grad) <= 1e-4 and rel(db, b.grad) <= 1e-4
    assert torch.equal(ops.argmax_u8(logits).cpu().long(), logits.cpu().argmax(1))


def test_losses_against_reference_golden(b2u, cuda_device, golden_dir):
    """Drop-in CE_Loss / Focal_Loss / Dice_loss / f_score against values the reference itself produced."""
    dev = cuda_device
    g = np.load(os.path.join(golden_dir, "losses.npz"))
    for C in (21, 4, 2):
        logits = torch.from_numpy(g[f"C{C}:logits"]).to(dev).requires_grad_(True)
        png = torch.from_numpy(g[f"C{C}:png"]).to(dev)
        w = torch.from_numpy(g[f"C{C}:w"]).to(dev)
        oh = O.one_hot(torch.from_numpy(g[f"C{C}:png"]), C).to(dev)
        ce = b2u.CE_Loss(logits, png, w, num_classes=C)
        fo = b2u.Focal_Loss(logits, png, w, num_classes=C)
        di = b2u.Dice_loss(logits, oh)
        fs = b2u.f_score(logits, oh)
        for got, want in zip((ce, fo, di, fs), g[f"C{C}:vals"]):
            assert abs(got.item() - want) <= 2e-5 * max(abs(want), 1e-3)
        for loss, key in ((ce, "g_ce"), (fo, "g_focal"), (di, "g_dice")):
            gr, = torch.autograd.grad(loss, logits, retain_graph=True)
            assert rel(gr, torch.from_numpy(g[f"C{C}:{key}"])) <= 2e-4


@pytest.mark.parametrize("n", [2, 4, 21])
def test_fast_hist_bit_exact(b2u, cuda_device, golden_dir, n):
    g = np.load(os.path.join(golden_dir, "fast_hist.npz"))
    gt, pred = O.make_masks(3, n, h=64, w=96, seed=n)
    hist = np.zeros((n, n))
    for i in range(3):
        hist += b2u.fast_hist(gt[i].flatten(), pred[i].flatten(), n)       # the compute_mIoU loop, utils_metrics.py:95
    assert np.array_equal(hist.astype(np.int64), g[f"n{n}:hist"])
    assert np.array_equal(b2u.per_class_iu(hist), g[f"n{n}:iou"])
    assert np.nanmean(b2u.per_class_iu(hist)) == float(g[f"n{n}:miou"])
    # other integer dtypes, ragged lengths, negative labels
    rng = np.random.default_rng(n)
    a = rng.integers(-2, n + 2, size=100003).astype(np.int64)
    b = rng.integers(0, n, size=100003).astype(np.int64)
    assert np.array_equal(b2u.fast_hist(a, b, n), O.fast_hist(a, b, n))
    a32, b32 = a.astype(np.int32), b.astype(np.int32)
    assert np.array_equal(b2u.fast_hist(a32, b32, n), O.fast_hist(a32, b32, n))


def test_fast_hist_edge_cases(b2u, cuda_device, golden_dir):
    g = np.load(os.path.join(golden_dir, "fast_hist.npz"))
    assert np.array_equal(b2u.fast_hist(np.full(1000, 255, np.uint8), np.zeros(1000, np.uint8), 21), g["allignore:hist"])
    assert np.array_equal(b2u.fast_hist(np.full(1000, 3, np.uint8), np.full(1000, 3, np.uint8), 21), g["single:hist"])
    assert np.array_equal(b2u.fast_hist(np.zeros(0, np.uint8), np.zeros(0, np.uint8), 4), g["empty:hist"])
    with pytest.raises(ValueError):
        b2u.fast_hist(np.array([1], np.uint8), np.array([200], np.uint8), 2)
    # unaligned device views take the scalar path
    a = torch.randint(0, 21, (4099,), dtype=torch.uint8); b = torch.randint(0, 21, (4099,), dtype=torch.uint8)
    got = b2u.fast_hist(a.cuda()[3:], b.cuda()[3:], 21)
    assert np.array_equal(got, O.fast_hist(a[3:].numpy(), b[3:].numpy(), 21))


@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 21, 32, 45, 64])
def test_fast_hist_all_kernel_variants(b2u, cuda_device, n):
    """vote kernel (n*n <= 32), lane-private byte counters (up to ~75 bins x 75), shared-atomic fallback; lengths that
    force byte-counter folds; out-of-range predictions land in the overflow counter exactly like numpy's failure."""
    rng = np.random.default_rng(100 + n)
    L = 16 * 256 * 148 * 3 + 7                       # several rounds per lane + a ragged tail
    a = rng.integers(0, n, size=L).astype(np.uint8)
    a[rng.random(L) < 0.05] = 255
    a[:5000] = 1 % n                                  # one lane hammers a single bin: exercises the 240-increment fold
    b = rng.integers(0, n, size=L).astype(np.uint8)
    b[:5000] = 0
    assert np.array_equal(b2u.fast_hist(a, b, n), O.fast_hist(a, b, n))
    b_bad = b.copy()
    b_bad[L // 2] = 255                               # pushes n*a+b past n*n unless that pixel is ignored
    a_ok = a.copy(); a_ok[L // 2] = n - 1
    hist = b2u.fast_hist_device(a_ok, b_bad, n).cpu().numpy()
    assert hist[-1] == 1
    with pytest.raises(ValueError):
        b2u.fast_hist(a_ok, b_bad, n)


def test_fast_hist_full_size_properties(b2u, cuda_device):
    """BASELINE config 5 size (512x512 masks): exact against numpy on 50 masks; sum of per-mask histograms ==
    histogram of the concatenation; total count == number of non-ignored pixels."""
    n = 21
    gt, pred = O.make_masks(50, n, seed=0)
    dev_hist = None
    for i in range(gt.shape[0]):
        dev_hist = b2u.fast_hist_device(gt[i], pred[i], n, hist=dev_hist)
    acc = dev_hist.cpu().numpy()
    assert acc[-1] == 0
    whole = b2u.fast_hist(gt.reshape(-1), pred.reshape(-1), n)
    assert np.array_equal(acc[:-1].reshape(n, n), whole)
    assert np.array_equal(whole, O.fast_hist(gt.reshape(-1), pred.reshape(-1), n))
    assert whole.sum() == int((gt < n).sum())


@pytest.mark.parametrize("n", [2, 4, 21, 30])
def test_fast_hist_lanes_kernel_wraps_and_batches(b2u, cuda_device, n):
    """The lane-private byte counters wrap (255 -> 0) into the per-warp 32-bit table: a mask that sends > 255 pixels of ONE bin
    through every lane must stay exact; the batched entry point (pointer table, one launch) equals the per-mask loop,
    including ragged lengths and all-ignored masks."""
    ops, dev = b2u.ops, cuda_device
    L = 148 * 384 * 16 * 20 + 5                        # ~320 pixels per lane, all in one bin
    a = torch.full((L,), n - 1, dtype=torch.uint8, device=dev)
    b = torch.full((L,), n - 1, dtype=torch.uint8, device=dev)
    a[7::1001] = 255                                    # a few ignored pixels
    hist = ops.fast_hist_accumulate(a, b, n, torch.zeros(n * n + 1, dtype=torch.int64, device=dev)).cpu().numpy()
    want = np.zeros(n * n + 1, np.int64)
    want[n * n - 1] = int((a != 255).sum().item())
    assert np.array_equal(hist, want)
    rng = np.random.default_rng(5 + n)
    sizes = [512 * 512, 16 * 33 + 9, 0 + 16, 100003, 512 * 384]
    pairs, ref = [], np.zeros((n, n), np.int64)
    for i, sz in enumerate(sizes):
        ga = rng.integers(0, n, size=sz).astype(np.uint8)
        ga[rng.random(sz) < (1.0 if i == 2 else 0.03)] = 255
        pb = rng.integers(0, n, size=sz).astype(np.uint8)
        ref += O.fast_hist(ga, pb, n)
        pairs.append((torch.from_numpy(ga).to(dev), torch.from_numpy(pb).to(dev)))
    got = ops.fast_hist_batch(pairs, n, torch.zeros(n * n + 1, dtype=torch.int64, device=dev)).cpu().numpy()
    assert got[-1] == 0 and np.array_equal(got[:-1].reshape(n, n), ref)
    loop = torch.zeros(n * n + 1, dtype=torch.int64, device=dev)
    for ga, pb in pairs:
        ops.fast_hist_accumulate(ga, pb, n, loop)
    assert np.array_equal(loop.cpu().numpy(), got)


@pytest.mark.parametrize("C,n", [(21, 21), (2, 2), (4, 4)])
def test_argmax_hist_fused(b2u, cuda_device, C, n):
    """logits -> class mask + confusion matrix in one pass == numpy argmax (lowest index on ties) + the reference's bincount
    formulation (utils/utils_metrics.py:34-43), exactly."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(C)
    logits = torch.randn(3, C, 64, 96, generator=g)
    logits[0, :, :8] = 0.25                              # ties everywhere: class 0 must win
    logits[1, 1, 5:9] = logits[1, 0, 5:9]                # two-way ties
    gt = torch.randint(0, n, (3, 64, 96), generator=g, dtype=torch.uint8)
    gt[torch.rand(3, 64, 96, generator=g) < 0.05] = 255
    hist, pred = ops.argmax_hist(logits.to(dev), gt.to(dev), n, want_pred=True)
    want_pred = logits.numpy().argmax(1).astype(np.uint8)
    assert np.array_equal(pred.cpu().numpy(), want_pred)
    assert np.array_equal(pred.cpu().numpy(), ops.argmax_u8(logits.to(dev)).cpu().numpy())
    h = hist.cpu().numpy()
    assert h[-1] == 0 and np.array_equal(h[:-1].reshape(n, n), O.fast_hist(gt.numpy().reshape(-1), want_pred.reshape(-1), n))
    _, only_mask = ops.argmax_hist(logits.to(dev), want_pred=True)
    assert np.array_equal(only_mask.cpu().numpy(), want_pred)


def test_optimizer_steps_match_torch(b2u, cuda_device):
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(6)
    n = 4096 * 3
    p0 = torch.randn(n, generator=g)
    grads = [torch.randn(n, generator=g) for _ in range(3)]
    for kind in ("adam", "sgd"):
        p_ref = p0.clone().requires_grad_(True)
        opt = torch.optim.Adam([p_ref], lr=1e-3) if kind == "adam" else torch.optim.SGD([p_ref], lr=1e-2, momentum=0.9, nesterov=True)
        p = p0.clone().to(dev); m = torch.zeros_like(p); v = torch.zeros_like(p)
        for step, gr in enumerate(grads, 1):
            p_ref.grad = gr.clone(); opt.step()
            if kind == "adam":
                ops.adam_step(p, gr.to(dev), m, v, step, 1e-3)
            else:
                ops.sgd_step(p, gr.to(dev), m, 1e-2, momentum=0.9, nesterov=True, first_step=(step == 1))
        assert rel(p, p_ref.detach()) <= 1e-6


@pytest.mark.parametrize("N,H,W,C,relu", [(2, 16, 24, 64, True), (1, 8, 8, 256, True), (3, 5, 7, 8, False), (2, 32, 32, 128, True)])
def test_batchnorm_kernels(b2u, cuda_device, N, H, W, C, relu):
    """nn.BatchNorm2d (+ReLU) train forward (batch statistics, running-stat update), eval forward and backward against
    torch on the same bf16-rounded pre-activations."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(8)
    z = torch.randn(N, C, H, W, generator=g) * 1.5 + torch.randn(1, C, 1, 1, generator=g)
    zb = nhwc(z, dev); zr = nchw(zb).requires_grad_(True)
    gamma = (1 + 0.2 * torch.randn(C, generator=g)).requires_grad_(True)
    beta = (0.1 * torch.randn(C, generator=g)).requires_grad_(True)
    rm0, rv0 = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
    rm_ref, rv_ref = rm0.clone(), rv0.clone()
    ref = F.batch_norm(zr, rm_ref, rv_ref, gamma, beta, True, 0.1, 1e-5)
    ref_y = ref.relu() if relu else ref
    rm, rv = rm0.clone().to(dev), rv0.clone().to(dev)
    y, mean, invstd = ops.bn_fwd_train(zb, gamma.detach().to(dev), beta.detach().to(dev), rm, rv, relu=relu)
    assert rel(nchw(y), ref_y.detach()) <= 6e-3
    assert torch.allclose(rm.cpu(), rm_ref, rtol=1e-5, atol=1e-6) and torch.allclose(rv.cpu(), rv_ref, rtol=1e-5, atol=1e-6)
    assert torch.allclose(mean.cpu(), zr.detach().mean((0, 2, 3)), rtol=1e-5, atol=1e-6)
    # backward
    dy = torch.randn(N, C, H, W, generator=g)
    dyb = nhwc(dy, dev)
    ref_y.backward(nchw(dyb))
    dz, dgam, dbet = ops.bn_bwd(dyb, y, zb, gamma.detach().to(dev), mean, invstd, relu=relu)
    # same gradients with the ReLU mask recomputed from z instead of read from y (bit-identical by construction)
    dz2, dgam2, dbet2 = ops.bn_bwd(dyb, None, zb, gamma.detach().to(dev), mean, invstd, relu=relu, beta=beta.detach().to(dev))
    assert torch.equal(dz2, dz) and torch.equal(dgam2, dgam) and torch.equal(dbet2, dbet)
    # the kernel masks with its own bf16 y (> 0); where torch's fp32 y differs in sign the elements are ~0 anyway
    assert rel(nchw(dz), zr.grad) <= 1e-2
    assert rel(dgam, gamma.grad) <= 2e-3 and rel(dbet, beta.grad) <= 2e-3
    # eval mode
    ye = ops.bn_fwd_eval(zb, gamma.detach().to(dev), beta.detach().to(dev), rm, rv, relu=relu)
    ref_e = F.batch_norm(zr.detach(), rm_ref, rv_ref, gamma.detach(), beta.detach(), False, 0.1, 1e-5)
    ref_e = ref_e.relu() if relu else ref_e
    assert rel(nchw(ye), ref_e) <= 6e-3


def test_resnet_helper_kernels(b2u, cuda_device):
    """7x7 stride-2 stem as im2col GEMM (+ its wgrad), stride-2 helpers, ceil-mode 3x3 max-pool fwd/bwd, residual
    BatchNorm tail, bf16 add -- nets/resnet.py:109-113, 77-97."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(9)
    # stem
    x = torch.rand(2, 3, 64, 96, generator=g)
    w = torch.randn(64, 3, 7, 7, generator=g) / 147 ** 0.5
    col = ops.im2col_stem(x.to(dev))
    wf = ops.pack_weights_im2col(w.to(dev), 192)
    z = ops.conv_fprop(col, wf, None, 64, taps=1, relu=False)
    ref = F.conv2d(x.to(BF).float(), w.to(BF).float(), None, stride=2, padding=3)
    assert rel(nchw(z), ref) <= 6e-3
    dz = nhwc(torch.randn(2, 64, 32, 48, generator=g), dev)
    dw = ops.conv_wgrad_im2col(col, dz, 3, 49)
    ref_dw = torch.nn.grad.conv2d_weight(x.to(BF).float(), w.shape, nchw(dz), stride=2, padding=3)
    assert rel(dw, ref_dw) <= 1e-4
    # stride-2 3x3 conv = stride-1 conv + subsample; its backward through zero_insert
    xb = nhwc(torch.randn(2, 64, 16, 24, generator=g), dev)
    full = nchw(xb)
    sub = ops.subsample2(xb)
    assert torch.equal(nchw(sub), full[:, :, ::2, ::2])
    back = ops.zero_insert2(sub, 16, 24)
    want = torch.zeros_like(full); want[:, :, ::2, ::2] = full[:, :, ::2, ::2]
    assert torch.equal(nchw(back), want)
    w3 = torch.randn(128, 64, 3, 3, generator=g) / 24
    wf3, wd3 = ops.pack_weights(w3.to(dev))
    y2 = ops.subsample2(ops.conv_fprop(xb, wf3, None, 128, taps=9, relu=False))
    assert rel(nchw(y2), F.conv2d(full, w3.to(BF).float(), None, stride=2, padding=1)) <= 6e-3
    # ceil-mode pool, odd and even sizes
    for (H, W) in ((16, 24), (15, 9), (3, 3)):
        xp = nhwc(torch.randn(2, 16, H, W, generator=g), dev)
        xr = nchw(xp).requires_grad_(True)
        refp = F.max_pool2d(xr, 3, 2, 0, ceil_mode=True)
        yp = ops.maxpool3x3s2(xp)
        assert torch.equal(nchw(yp), refp.detach())
        dyp = nhwc(torch.randn(refp.shape, generator=g), dev)
        refp.backward(nchw(dyp))
        assert rel(nchw(ops.maxpool3x3s2_bwd(dyp, xp)), xr.grad) <= 4e-3
    # add
    a, b_ = nhwc(torch.randn(2, 64, 8, 8, generator=g), dev), nhwc(torch.randn(2, 64, 8, 8, generator=g), dev)
    assert rel(ops.add_bf16(a, b_), a.float() + b_.float()) <= 4e-3
    # residual BatchNorm tail: y = relu(bn(z) + identity)
    C = 64
    zt = torch.randn(2, C, 8, 12, generator=g); idn = torch.randn(2, C, 8, 12, generator=g)
    zb, ib = nhwc(zt, dev), nhwc(idn, dev)
    zr, ir = nchw(zb).requires_grad_(True), nchw(ib).requires_grad_(True)
    gamma = (1 + 0.2 * torch.randn(C, generator=g)).requires_grad_(True); beta = (0.1 * torch.randn(C, generator=g)).requires_grad_(True)
    refy = (F.batch_norm(zr, None, None, gamma, beta, True, 0.1, 1e-5) + ir).relu()
    rm, rv = torch.zeros(C, device=dev), torch.ones(C, device=dev)
    y, mean, invstd = ops.bn_fwd_train(zb, gamma.detach().to(dev), beta.detach().to(dev), rm, rv, relu=True, residual=ib)
    assert rel(nchw(y), refy.detach()) <= 6e-3
    dy = nhwc(torch.randn(2, C, 8, 12, generator=g), dev)
    refy.backward(nchw(dy))
    gout = torch.empty_like(zb)
    dzb, dgam, dbet = ops.bn_bwd(dy, y, zb, gamma.detach().to(dev), mean, invstd, relu=True, gout=gout)
    assert rel(nchw(dzb), zr.grad) <= 1e-2 and rel(nchw(gout), ir.grad) <= 6e-3
    assert rel(dgam, gamma.grad) <= 3e-3 and rel(dbet, beta.grad) <= 3e-3


def test_conv_large_channel_counts(b2u, cuda_device):
    """ResNet50 decoder shapes: 3072 -> 512 over a virtual concat (1024 | 2048), 1x1 2048-wide GEMMs."""
    ops, dev = b2u.ops, cuda_device
    g = torch.Generator().manual_seed(10)
    x0 = nhwc(torch.randn(1, 1024, 8, 8, generator=g), dev); x1 = nhwc(torch.randn(1, 2048, 8, 8, generator=g), dev)
    w = torch.randn(512, 3072, 3, 3, generator=g) / (3072 * 9) ** 0.5
    b = torch.randn(512, generator=g)
    wf, wd = ops.pack_weights(w.to(dev))
    y = ops.conv_fprop(x0, wf, b.to(dev), 512, taps=9, relu=True, x1=x1)
    xr = torch.cat([nchw(x0), nchw(x1)], 1)
    assert rel(nchw(y), F.conv2d(xr, w.to(BF).float(), b, padding=1).relu()) <= 6e-3
    dz = nhwc(torch.randn(1, 512, 8, 8, generator=g), dev)
    d0, d1 = ops.conv_dgrad(dz, wd, 1024, taps=9, C1=2048)
    ref_dx = F.conv_transpose2d(nchw(dz), w.to(BF).float(), padding=1)
    assert rel(torch.cat([nchw(d0), nchw(d1)], 1), ref_dx) <= 6e-3
    assert rel(ops.conv_wgrad(x0, dz, taps=9, x1=x1), torch.nn.grad.conv2d_weight(xr, w.shape, nchw(dz), padding=1)) <= 1e-4
    w1 = torch.randn(2048, 512, 1, 1, generator=g) / 512 ** 0.5
    wf1, wd1 = ops.pack_weights(w1.to(dev))
    xs = nhwc(torch.randn(2, 512, 8, 8, generator=g), dev)
    y1 = ops.conv_fprop(xs, wf1, None, 2048, taps=1, relu=False)
    assert rel(nchw(y1), F.conv2d(nchw(xs), w1.to(BF).float())) <= 6e-3
    dz1 = nhwc(torch.randn(2, 2048, 8, 8, generator=g), dev)
    assert rel(nchw(ops.conv_dgrad(dz1, wd1, 512, taps=1)), F.conv_transpose2d(nchw(dz1), w1.to(BF).float())) <= 6e-3
    assert rel(ops.conv_wgrad(xs, dz1, taps=1), torch.nn.grad.conv2d_weight(nchw(xs), w1.shape, nchw(dz1))) <= 1e-4


# ------------------------------------------------------------------------------ depthwise conv / squeeze-excite / padding
@pytest.mark.parametrize("N,H,W,C", [(2, 16, 24, 64), (1, 7, 9, 128), (3, 32, 32, 64), (1, 2, 2, 512)])
def test_depthwise_conv_kernels(b2u, cuda_device, N, H, W, C):
    from unet_pytorch_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(N * 100 + C)
    x = torch.randn(N, C, H, W, generator=g).to(BF).float()
    w = torch.randn(C, 1, 3, 3, generator=g) * 0.3
    b = torch.randn(C, generator=g) * 0.1
    dy = torch.randn(N, C, H, W, generator=g).to(BF).float()
    xr = x.clone().requires_grad_(True); wr = w.clone().requires_grad_(True); br = b.clone().requires_grad_(True)
    y_ref = F.conv2d(xr, wr, br, padding=1, groups=C)
    y_ref.backward(dy)
    xd, dyd, wd = nhwc(x, dev), nhwc(dy, dev), w.reshape(C, 9).contiguous().to(dev)
    y = ops.dwconv3x3(xd, wd, b.to(dev))
    assert rel(nchw(y), y_ref.detach()) <= 6e-3
    dx = ops.dwconv3x3(dyd, wd, None, flip=True)
    assert rel(nchw(dx), xr.grad) <= 6e-3
    dw, db = ops.dwconv3x3_wgrad(xd, dyd)
    assert rel(dw.reshape(C, 1, 3, 3), wr.grad) <= 1e-4
    assert rel(db, br.grad) <= 1e-4


@pytest.mark.parametrize("N,H,W,C,Cp,R", [(2, 16, 16, 64, 64, 16), (3, 8, 8, 44, 64, 11), (2, 4, 4, 512, 512, 128), (1, 32, 32, 176, 192, 44)])
def test_squeeze_excite_kernels(b2u, cuda_device, N, H, W, C, Cp, R):
    """spatial_reduce -> se_fc_fwd -> scale_nc and the matching backward against autograd of the module's math
    (nets/UltraLightweightUnet_large.py:36-52); channels C..Cp are zero padding and must stay zero."""
    from unet_pytorch_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(C + R)
    x = torch.zeros(N, Cp, H, W); x[:, :C] = torch.randn(N, C, H, W, generator=g).to(BF).float()
    dy = torch.zeros(N, Cp, H, W); dy[:, :C] = torch.randn(N, C, H, W, generator=g).to(BF).float()
    w1 = (torch.randn(R, C, generator=g) / C ** 0.5); b1 = torch.randn(R, generator=g) * 0.1
    w2 = (torch.randn(C, R, generator=g) / R ** 0.5); b2 = torch.randn(C, generator=g) * 0.1
    xr = x[:, :C].clone().requires_grad_(True)
    ps = [t.clone().requires_grad_(True) for t in (w1, b1, w2, b2)]
    s_ref = torch.sigmoid(F.linear(F.relu(F.linear(xr.mean(dim=(2, 3)), ps[0], ps[1])), ps[2], ps[3]))
    y_ref = xr * s_ref[:, :, None, None]
    y_ref.backward(dy[:, :C])
    xd, dyd = nhwc(x, dev), nhwc(dy, dev)
    pooled = ops.spatial_reduce(xd, scale=1.0 / (H * W))
    assert rel(pooled[:, :C], x[:, :C].mean(dim=(2, 3))) <= 1e-5
    hidden, sc = ops.se_fc_fwd(pooled, w1.to(dev), b1.to(dev), w2.to(dev), b2.to(dev), C)
    assert rel(sc[:, :C], s_ref.detach()) <= 1e-5
    y = ops.scale_nc(xd, sc)
    assert rel(nchw(y)[:, :C], y_ref.detach()) <= 6e-3
    assert nchw(y)[:, C:].abs().max().item() == 0 if Cp > C else True
    dscale = ops.spatial_reduce(dyd, xd)
    grads = [torch.empty_like(t, device=dev) for t in (w1, b1, w2, b2)]
    dpooled = ops.se_fc_bwd(dscale, pooled, hidden, sc, w1.to(dev), w2.to(dev), C, 1.0 / (H * W), dw1=grads[0], db1=grads[1],
                            dw2=grads[2], db2=grads[3])
    for got, p in zip(grads, ps):
        assert rel(got, p.grad) <= 1e-4
    dx = ops.scale_nc(dyd, sc, add=dpooled)
    assert rel(nchw(dx)[:, :C], xr.grad) <= 6e-3
    if Cp > C:
        assert nchw(dx)[:, C:].abs().max().item() == 0


def test_padded_channel_convs(b2u, cuda_device):
    """Channel counts that are not multiples of 64 (UltraLightweightUnet_large_optimized: 44/88/176/352/704, mids 22..352)
    run on the tensor-core kernels with zero-padded operands: pack_weights_multi pads, the conv sees pad64 channels."""
    import struct
    from unet_pytorch_b200 import ops
    from unet_pytorch_b200._engine_base import pad64
    dev = cuda_device
    g = torch.Generator().manual_seed(5)
    for (cout, c0, c1, taps) in ((22, 3, 0, 1), (44, 22, 0, 1), (176, 352, 176, 1), (88, 44, 0, 9), (352, 704, 352, 1)):
        k = 3 if taps == 9 else 1
        w = (torch.randn(cout, c0 + c1, k, k, generator=g) / ((c0 + c1) * k * k) ** 0.5).to(dev)
        c0p, c1p, coutp = pad64(c0), (pad64(c1) if c1 else 0), pad64(cout)
        wf = torch.zeros((coutp, taps * (c0p + c1p)), dtype=BF, device=dev)
        wd = torch.zeros((c0p + c1p, taps * coutp), dtype=BF, device=dev)
        blob = struct.pack("<QQQqiiiiiiii", w.data_ptr(), wf.data_ptr(), wd.data_ptr(), 0, cout, c0 + c1, taps, 0, c0, c0p, c0p + c1p, coutp)
        count = ((cout + 31) // 32) * ((c0 + c1 + 31) // 32)
        table = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)
        ops.check(ops.lib().b2u_pack_weights_multi(table.data_ptr(), 1, count, ops.stream_ptr()))
        N, H, W = 2, 16, 16
        x0 = torch.zeros(N, c0p, H, W); x0[:, :c0] = torch.randn(N, c0, H, W, generator=g).to(BF).float()
        x1 = None
        if c1:
            x1 = torch.zeros(N, c1p, H, W); x1[:, :c1] = torch.randn(N, c1, H, W, generator=g).to(BF).float()
        bias = torch.zeros(coutp); bias[:cout] = torch.randn(cout, generator=g) * 0.1
        xin = x0[:, :c0] if x1 is None else torch.cat([x0[:, :c0], x1[:, :c1]], 1)
        wr = w.cpu().to(BF).float()
        y_ref = F.conv2d(xin, wr, bias[:cout], padding=k // 2)
        y = ops.conv_fprop(nhwc(x0, dev), wf, bias.to(dev), coutp, taps=taps, relu=False, x1=nhwc(x1, dev) if c1 else None)
        yh = nchw(y)
        assert rel(yh[:, :cout], y_ref) <= 6e-3, (cout, c0, c1)
        if coutp > cout:
            assert yh[:, cout:].abs().max().item() == 0
        dz = torch.zeros(N, coutp, H, W); dz[:, :cout] = torch.randn(N, cout, H, W, generator=g).to(BF).float()
        dx_ref = F.conv_transpose2d(dz[:, :cout], wr, padding=k // 2)
        if c1:
            d0, d1 = ops.conv_dgrad(nhwc(dz, dev), wd, c0p, taps=taps, C1=c1p)
            assert rel(nchw(d0)[:, :c0], dx_ref[:, :c0]) <= 6e-3 and rel(nchw(d1)[:, :c1], dx_ref[:, c0:]) <= 6e-3
            assert nchw(d0)[:, c0:].abs().max().item() == 0 if c0p > c0 else True
        else:
            d0 = ops.conv_dgrad(nhwc(dz, dev), wd, c0p, taps=taps)
            d0 = d0[0] if isinstance(d0, tuple) else d0
            assert rel(nchw(d0)[:, :c0], dx_ref) <= 6e-3
        # weight gradient of the padded problem: real rows/columns match, padding rows/columns are exactly zero
        dwp = ops.conv_wgrad(nhwc(x0, dev), nhwc(dz, dev), taps=taps, x1=nhwc(x1, dev) if c1 else None)
        dwp = (dwp[0] if isinstance(dwp, tuple) else dwp).cpu()
        xr = xin.clone().requires_grad_(True)
        wr_ = wr.clone().requires_grad_(True)
        F.conv2d(xr, wr_, None, padding=k // 2).backward(dz[:, :cout])
        got = dwp[:cout, :c0] if not c1 else torch.cat([dwp[:cout, :c0], dwp[:cout, c0p:c0p + c1]], 1)
        assert rel(got, wr_.grad) <= 1e-4, (cout, c0, c1)
        assert dwp[cout:].abs().max().item() == 0 if coutp > cout else True


def test_padded_input_conversion(b2u, cuda_device):
    from unet_pytorch_b200 import ops
    x = torch.randn(2, 3, 16, 32)
    y = ops.nchw_to_nhwc_bf16_padded(x.to(cuda_device), 64)
    assert tuple(y.shape) == (2, 16, 32, 64)
    hi = x.permute(0, 2, 3, 1).to(BF)
    assert torch.equal(y[..., :3].cpu(), hi) and y[..., 6:].abs().max().item() == 0
    # channels [C, 2C): the second term of the two-term bf16 split of the image (the first conv's weights repeat there)
    assert torch.equal(y[..., 3:6].cpu(), (x.permute(0, 2, 3, 1) - hi.float()).to(BF))


def test_residual_join_and_resize_kernels(b2u, cuda_device, golden_dir):
    """relu(a + b) and its gradient mask; F.interpolate(bilinear, align_corners=True) of fp32 NCHW logits and its adjoint
    (the losses' resize for half-resolution logits) against torch, including non-2x sizes."""
    from unet_pytorch_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(31)
    a = torch.randn(2, 12, 20, 64, generator=g).to(BF); b = torch.randn(2, 12, 20, 64, generator=g).to(BF)
    y = ops.add_relu(a.to(dev), b.to(dev))
    assert torch.equal(y.cpu(), (a.float() + b.float()).relu().to(BF))
    dy = torch.randn(2, 12, 20, 64, generator=g).to(BF)
    dx = ops.relu_bwd(dy.to(dev), y)
    assert torch.equal(dx.cpu(), torch.where(y.cpu().float() > 0, dy.float(), torch.zeros(())).to(BF))
    for (hi, wi, ho, wo) in ((16, 24, 32, 48), (7, 5, 20, 11), (1, 1, 4, 4), (32, 32, 64, 64), (9, 9, 9, 17)):
        x = torch.randn(2, 5, hi, wi, generator=g)
        xr = x.clone().requires_grad_(True)
        ref = F.interpolate(xr, size=(ho, wo), mode="bilinear", align_corners=True)
        out = ops.resize_bilinear(x.to(dev), (ho, wo))
        assert torch.allclose(out.cpu(), ref.detach(), rtol=1e-5, atol=1e-6), (hi, wi, ho, wo)
        gy = torch.randn(2, 5, ho, wo, generator=g)
        ref.backward(gy)
        gx = ops.resize_bilinear_bwd(gy.to(dev), (hi, wi))
        assert torch.allclose(gx.cpu(), xr.grad, rtol=1e-4, atol=1e-5), (hi, wi, ho, wo)
    # the loss wrappers resize exactly like the reference's (golden values of CE/Dice/f_score on half-resolution logits)
    gl = np.load(os.path.join(golden_dir, "lightweight_nc4_focaldice.npz"))
    C, n, h, w, seed, dice, focal = [int(v) for v in gl["meta"]]
    _, pngs = O.make_inputs(n, C, h, w, seed=seed)
    lg = torch.from_numpy(gl["logits"]).to(dev).requires_grad_(True)
    cw = torch.from_numpy(gl["cls_w"]).to(dev)
    loss = b2u.Focal_Loss(lg, pngs.to(dev), cw, num_classes=C) + b2u.Dice_loss(lg, O.one_hot(pngs, C).to(dev))
    assert abs(loss.item() - float(gl["loss"])) <= 1e-5 * abs(float(gl["loss"]))
    assert abs(b2u.f_score(lg.detach(), O.one_hot(pngs, C).to(dev)).item() - float(gl["f_score"])) <= 1e-5
    loss.backward()
    lref = torch.from_numpy(gl["logits"]).requires_grad_(True)
    full = O.resize_logits(lref, h, w)
    (O.focal_loss(full, pngs, cw.cpu(), C) + O.dice_loss(full, O.one_hot(pngs, C))).backward()
    assert rel(lg.grad, lref.grad) <= 1e-4


@pytest.mark.parametrize("N,H,W,C", [(2, 16, 32, 21), (1, 24, 40, 2), (3, 8, 16, 32), (1, 5, 7, 4)])
def test_head_forward_on_tensor_cores(b2u, cuda_device, N, H, W, C):
    """The 1x1 classifier through the conv kernel's head epilogue ([hi | lo] bf16 split of the fp32 weights, fp32 NCHW
    logits) against fp32 torch on the same bf16 activations and against the SIMT head."""
    from unet_pytorch_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(C)
    x = torch.randn(N, 64, H, W, generator=g).to(BF).float()
    w = torch.randn(C, 64, generator=g) * 0.2
    b = torch.randn(C, generator=g)
    ref = F.conv2d(x, w[:, :, None, None], b)
    xd = nhwc(x, dev)
    out = ops.head_fwd_tc(xd, ops.pack_head_fprop(w.to(dev)), b.to(dev), C)
    assert tuple(out.shape) == (N, C, H, W)
    assert rel(out, ref) <= 2e-5          # fp32 accumulation of bf16 x (exact products) and ~2^-17 weights
    simt = ops.head_fwd(xd, w.to(dev), b.to(dev))
    assert rel(out, simt) <= 2e-5


@pytest.mark.parametrize("C,H,W,crop,out", [(21, 64, 64, (8, 0, 48, 64), (90, 120)), (2, 32, 48, (0, 6, 32, 36), (17, 19)),
                                            (4, 16, 16, (0, 0, 16, 16), (16, 16)), (32, 24, 24, (2, 3, 20, 18), (61, 47))])
def test_softmax_resize_argmax_kernel(b2u, cuda_device, C, H, W, crop, out):
    """softmax -> crop -> cv2-style INTER_LINEAR resize -> argmax in one kernel against the oracle's numpy restatement
    (itself pinned to cv2 through the reference predictor's golden mask)."""
    from unet_pytorch_b200 import ops
    g = torch.Generator().manual_seed(C + H)
    logits = torch.randn(2, C, H, W, generator=g) * 3
    cy, cx, ch, cw = crop
    got = ops.softmax_resize_argmax_u8(logits.to(cuda_device), crop, out).cpu().numpy()
    for n in range(2):
        pr = torch.softmax(logits[n].permute(1, 2, 0), dim=-1).numpy()[cy:cy + ch, cx:cx + cw]
        ref = O.resize_linear_cv2(pr, out[0], out[1])
        top2 = np.sort(ref, axis=-1)[..., -2:]
        confident = (top2[..., 1] - top2[..., 0]) > 1e-4
        assert (got[n] == ref.argmax(-1))[confident].all()
        assert (got[n] == ref.argmax(-1)).mean() >= 0.999


@pytest.mark.parametrize("N,H,W,C0,C1,Cout,taps", [(2, 24, 40, 64, 0, 64, 9), (2, 40, 40, 64, 0, 64, 9), (1, 16, 16, 128, 0, 256, 9), (2, 32, 32, 64, 64, 128, 9),
                                                    (2, 16, 48, 64, 0, 64, 1), (1, 8, 8, 256, 0, 512, 1), (3, 5, 7, 64, 0, 192, 1),
                                                    (1, 40, 24, 64, 0, 128, 1)])
def test_conv_epilogue_batchnorm_statistics(b2u, cuda_device, N, H, W, C0, C1, Cout, taps):
    """conv_fprop(stats=...) emits per-tile sums of z and z^2 of the stored bf16 output; BatchNorm driven by them must equal
    BatchNorm driven by its own statistics pass over the same z (ragged tiles, stacked tiles, virtual concat, 1x1)."""
    from unet_pytorch_b200 import ops
    dev = cuda_device
    g = torch.Generator().manual_seed(Cout + H)
    k = 3 if taps == 9 else 1
    x0 = nhwc(torch.randn(N, C0, H, W, generator=g), dev)
    x1 = nhwc(torch.randn(N, C1, H, W, generator=g), dev) if C1 else None
    w = torch.randn(Cout, C0 + C1, k, k, generator=g) / ((C0 + C1) * k * k) ** 0.5
    wf, _ = ops.pack_weights(w.to(dev))
    bias = (torch.randn(Cout, generator=g) * 0.5).to(dev)
    rows = ops.conv_stat_rows(N, H, W, Cout, taps)
    stats = torch.full((rows, 2, Cout), float("nan"), dtype=torch.float32, device=dev)
    z = ops.conv_fprop(x0, wf, bias, Cout, taps=taps, relu=False, x1=x1, stats=stats)
    z_plain = ops.conv_fprop(x0, wf, bias, Cout, taps=taps, relu=False, x1=x1)
    assert torch.equal(z, z_plain)
    assert torch.isfinite(stats).all()
    zf = z.float().reshape(-1, Cout)
    tot = stats.double().sum(0).cpu()
    assert torch.allclose(tot[0], zf.double().sum(0).cpu(), rtol=1e-5, atol=1e-3)
    assert torch.allclose(tot[1], (zf.double() ** 2).sum(0).cpu(), rtol=1e-5, atol=1e-3)
    gamma = (1 + 0.1 * torch.randn(Cout, generator=g)).to(dev); beta = (0.1 * torch.randn(Cout, generator=g)).to(dev)
    rm_a, rv_a = torch.zeros(Cout, device=dev), torch.ones(Cout, device=dev)
    rm_b, rv_b = torch.zeros(Cout, device=dev), torch.ones(Cout, device=dev)
    ya, ma, ia = ops.bn_fwd_train(z, gamma, beta, rm_a, rv_a)
    yb, mb, ib = ops.bn_fwd_train(z, gamma, beta, rm_b, rv_b, stats=stats, stat_rows=rows)
    assert torch.allclose(ma, mb, rtol=1e-5, atol=1e-6) and torch.allclose(ia, ib, rtol=1e-4, atol=1e-6)
    assert torch.allclose(rm_a, rm_b, rtol=1e-5, atol=1e-6) and torch.allclose(rv_a, rv_b, rtol=1e-4, atol=1e-6)
    assert rel(yb, ya) <= 1e-3
