"""GPU: the layers that read the image, at full training resolution, against exact host layouts and float64 references.

These launches are the largest of each step and hold the project's least common code: the first 3x3 conv of Unet-VGG16
and TraditionalUnet over im2col_first rows (the image enters as a two-term bf16 split, hi = bf16(x) in columns
[0, 9 Cin) and lo = bf16(x - hi) in [9 Cin, 18 Cin) when 18 Cin <= 64; the packed weights repeat over the lo columns and
the weight gradient folds the lo partial sums back), every first-layer width the engines accept (Cin = 1..7), the
ResNet-50 stem (7x7 stride-2 im2col, 147 of 192 columns, a 1x1 GEMM with K = 192 and its split-K weight gradient), the
ceil-mode 3x3 stride-2 max-pool whose backward decides "first maximum in scan order" per window, and the exact copies
around them (subsample2 / zero_insert2, nchw_to_nhwc_bf16_padded).

Layouts are compared bit for bit.  Arithmetic uses the bounds of test_kernels_at_scale_gpu.py: |y - ref| <= 2^-8 |ref|
+ c A for bf16 outputs, c' A for fp32 sums, A the same computation over absolute values.  Calibration, one NVIDIA B200
(148 SMs) at a 1000 W power limit: the largest err / bound seen per case is noted next to each case list.
"""
import pytest
import torch
import torch.nn.functional as F

from test_kernels_at_scale_gpu import C_BF16, C_WGRAD, _bf, _gen, _note, _sms, check_bf16, check_sum, conv_ref, wgrad_ref, wgrad_plan

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
F64 = torch.float64


def _bits(t):
    return t.view(torch.int16)


def _split(x):
    """Two-term bf16 split of fp32 x: hi = bf16(x), lo = bf16(x - hi)."""
    hi = x.to(BF)
    return hi, (x - hi.float()).to(BF)


def _first_cols(img):
    """3x3 'same' im2col of NCHW img -> [N, H, W, 9 Cin] in the kernels' column order k = tap * Cin + c (values as fp32)."""
    N, Cin, H, W = img.shape
    u = F.unfold(img.float(), 3, padding=1)                    # [N, Cin * 9, H W], c slowest
    return u.view(N, Cin, 9, H, W).permute(0, 3, 4, 2, 1).reshape(N, H, W, 9 * Cin)


def _first_weights(w):
    """OIHW [Cout, Cin, 3, 3] -> bf16 [Cout, 9 Cin], column k = tap * Cin + c."""
    return w.to(BF).permute(0, 2, 3, 1).reshape(w.shape[0], -1)


def _packed_first(w):
    """The first layer's fprop operand [Cout, 64]: [w | w | 0] when the image is split (18 Cin <= 64), else [w | 0]."""
    K = 9 * w.shape[1]
    wk = _first_weights(w)
    want = torch.zeros((w.shape[0], 64), dtype=BF, device=w.device)
    want[:, :K] = wk
    if 2 * K <= 64:
        want[:, K:2 * K] = wk
    return want


def _nhwc(img):
    return img.permute(0, 2, 3, 1)


# ------------------------------------------------------------------------------------------------- exact layouts
# N, Cin, H, W: Cin = 3 has its own kernel; 1, 2 take the generic one with the split, 4..7 without it; 5 and 7 leave an
# odd column count (the pad column of the last 32-bit pair).  W = 383: the last 64-pixel segment holds 63 pixels.
IM2COL_CASES = [(16, 3, 512, 512), (16, 7, 512, 512)] + [(3, c, 37, 383) for c in range(1, 8)]


@pytest.mark.parametrize("N,Cin,H,W", IM2COL_CASES)
def test_im2col_first_layout(b2u, cuda_device, N, Cin, H, W):
    """im2col_first against a host unfold: hi in [0, 9 Cin), lo = bf16(x - hi) in [9 Cin, 18 Cin) when split, zeros after,
    zero padding at the image border."""
    ops, dev = b2u.ops, cuda_device
    x = torch.randn((N, Cin, H, W), generator=_gen(dev, 20 + Cin), device=dev)
    K = 9 * Cin
    hi, lo = _split(x)
    want = torch.zeros((N, H, W, 64), dtype=BF, device=dev)
    want[..., :K] = _first_cols(hi).to(BF)
    if 2 * K <= 64:
        want[..., K:2 * K] = _first_cols(lo).to(BF)
        assert (want[..., K:2 * K] != 0).float().mean().item() > 0.9        # the lo columns carry data
    col = ops.im2col_first(x)
    assert torch.equal(_bits(col), _bits(want)), f"Cin={Cin}: {(col != want).sum().item()} values differ"


def _pack_multi_first(ops, ws, couts_p):
    """b2u_pack_weights_multi over first-layer records only: w [Cout, Cin, 3, 3] -> zeroed [Cout_pad, 64] operands."""
    import struct
    blob, start, outs = b"", 0, []
    for w, cout_p in zip(ws, couts_p):
        cout, cin = w.shape[:2]
        wf = torch.zeros((cout_p, 64), dtype=BF, device=w.device)
        blob += struct.pack("<QQQqiiiiiiii", w.data_ptr(), wf.data_ptr(), 0, start, cout, cin, 1, 1, cin, 64, 64, cout_p)
        start += (cout + 31) // 32
        outs.append(wf)
    table = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(ws[0].device)
    ops.check(ops.lib().b2u_pack_weights_multi(table.data_ptr(), len(ws), start, ops.stream_ptr()))
    return outs


def test_pack_weights_first_layout(b2u, cuda_device):
    """pack_weights_first and the first-layer records of pack_weights_multi, Cin = 1..7, Cout = 64 and Cout = 32 on a
    64-row operand (TraditionalUnet's first conv: rows 32..63 stay zero), all records in one table."""
    ops, dev = b2u.ops, cuda_device
    g = _gen(dev, 30)
    ws, couts_p = [], []
    for cin in range(1, 8):
        for cout in (64, 32):
            ws.append(torch.randn((cout, cin, 3, 3), generator=g, device=dev))
            couts_p.append(64)
    for w in ws:
        assert torch.equal(_bits(ops.pack_weights_first(w)), _bits(_packed_first(w))), tuple(w.shape)
    for w, wf in zip(ws, _pack_multi_first(ops, ws, couts_p)):
        cout = w.shape[0]
        assert torch.equal(_bits(wf[:cout]), _bits(_packed_first(w))), f"pack_weights_multi first {tuple(w.shape)}"
        assert not wf[cout:].any(), f"pack_weights_multi first {tuple(w.shape)}: padding rows written"


def _stem_cols(xb):
    """7x7 stride-2 pad-3 im2col of NCHW bf16 xb -> [N, Ho, Wo, 49 Cin], k = tap * Cin + c (values as fp32)."""
    N, Cin, H, W = xb.shape
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    u = F.unfold(xb.float(), 7, stride=2, padding=3)
    return u.view(N, Cin, 49, Ho, Wo).permute(0, 3, 4, 2, 1).reshape(N, Ho, Wo, 49 * Cin)


# N, Cin, H, W.  383 x 509: Ho = 192, Wo = 255 (the last 32-pixel segment holds 31 pixels).
STEM_LAYOUT_CASES = [(16, 3, 512, 512), (3, 3, 383, 509), (2, 1, 383, 509)]


@pytest.mark.parametrize("N,Cin,H,W", STEM_LAYOUT_CASES)
def test_im2col_stem_layout(b2u, cuda_device, N, Cin, H, W):
    ops, dev = b2u.ops, cuda_device
    x = torch.randn((N, Cin, H, W), generator=_gen(dev, 31), device=dev)
    col = ops.im2col_stem(x)
    want = torch.zeros((N, (H + 1) // 2, (W + 1) // 2, 192), dtype=BF, device=dev)
    want[..., :49 * Cin] = _stem_cols(x.to(BF)).to(BF)
    assert torch.equal(_bits(col), _bits(want)), f"{(col != want).sum().item()} values differ"


@pytest.mark.parametrize("Cout,Cin,k,Kpad", [(64, 3, 7, 192), (128, 1, 7, 64), (64, 3, 3, 64)])
def test_pack_weights_im2col_layout(b2u, cuda_device, Cout, Cin, k, Kpad):
    ops, dev = b2u.ops, cuda_device
    w = torch.randn((Cout, Cin, k, k), generator=_gen(dev, 32), device=dev)
    want = torch.zeros((Cout, Kpad), dtype=BF, device=dev)
    want[:, :k * k * Cin] = w.to(BF).permute(0, 2, 3, 1).reshape(Cout, -1)
    assert torch.equal(_bits(ops.pack_weights_im2col(w, Kpad)), _bits(want))


@pytest.mark.parametrize("N,H,W,C", [(16, 256, 256, 64), (3, 37, 51, 24), (2, 36, 51, 8), (5, 1, 3, 8)])
def test_subsample2_zero_insert2_exact(b2u, cuda_device, N, H, W, C):
    ops, dev = b2u.ops, cuda_device
    x = _bf((N, H, W, C), _gen(dev, 33), dev)
    sub = ops.subsample2(x)
    assert torch.equal(_bits(sub), _bits(x[:, ::2, ::2].contiguous()))
    want = torch.zeros_like(x)
    want[:, ::2, ::2] = sub
    assert torch.equal(_bits(ops.zero_insert2(sub, H, W)), _bits(want))


# C = 1, 3, 32: channels [C, 2C) hold lo = bf16(x - hi); C = 40: no room for the split.  383 x 37 pixels: a ragged last block.
@pytest.mark.parametrize("N,C,H,W", [(16, c, 512, 512) for c in (1, 3, 32, 40)] + [(3, c, 37, 383) for c in (3, 40)])
def test_nchw_to_nhwc_padded_exact(b2u, cuda_device, N, C, H, W):
    ops, dev = b2u.ops, cuda_device
    x = torch.randn((N, C, H, W), generator=_gen(dev, 34), device=dev)
    hi, lo = _split(x)
    want = torch.zeros((N, H, W, 64), dtype=BF, device=dev)
    want[..., :C] = _nhwc(hi)
    if 2 * C <= 64:
        want[..., C:2 * C] = _nhwc(lo)
    assert torch.equal(_bits(ops.nchw_to_nhwc_bf16_padded(x, 64)), _bits(want))


# ------------------------------------------------------------------------------------------------- first conv
# Observed err / bound: y 0.990-0.992 (bf16 rounding) with and without ReLU; against the conv of x itself 0.986-0.989,
# where the hi-only conv of the same data scores 64 (Cin = 3) and 84 (Cin = 1).
FIRST_CONV_CIN = [1, 3, 7]


@pytest.mark.parametrize("Cin", FIRST_CONV_CIN)
def test_first_conv_fprop_at_scale(b2u, cuda_device, Cin):
    """conv_fprop(im2col_first(x), pack_weights_first(w), b) at 16 x 512 x 512 with and without ReLU, against the fp64
    conv over hi + lo (split) or hi (no split).  With the split, the result must also sit within the bound of the fp64
    conv of the fp32 image itself, where the hi-only conv of the same data lies many bounds away."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    N, H, W, Cout = 16, 512, 512, 64
    g = _gen(dev, 40 + Cin)
    x = torch.randn((N, Cin, H, W), generator=g, device=dev)
    w = torch.randn((Cout, Cin, 3, 3), generator=g, device=dev) / (9 * Cin) ** 0.5
    b = torch.randn((Cout,), generator=g, device=dev) * 0.1
    split = 18 * Cin <= 64
    assert ops.conv_stat_rows(N, H, W, Cout, 1) >= 3 * sms
    col = ops.im2col_first(x)
    wf = ops.pack_weights_first(w)
    hi, lo = _split(x)
    xs = hi.double() + lo.double() if split else hi.double()
    xa = hi.double().abs() + lo.double().abs() if split else hi.double().abs()
    wb = w.to(BF)
    ref = conv_ref(_nhwc(xs), wb, b)
    A = conv_ref(_nhwc(xa), wb, b, absolute=True)
    del xs, xa
    tag = f"first conv {N}x{H}x{W} Cin={Cin}"
    for relu in (False, True):
        y = ops.conv_fprop(col, wf, b, Cout, taps=1, relu=relu)
        check_bf16(f"{tag} relu={relu}", y, ref.relu() if relu else ref, A)
    if not split:
        return
    # the split is really there: against the conv of x itself (|x - hi - lo| <= 2^-16 |x| adds up to C_BF16 A), on four
    # images of the batch
    n = 4
    y = ops.conv_fprop(col, wf, b, Cout, taps=1, relu=False)[:n]
    ref_x = conv_ref(_nhwc(x[:n]), wb, b)
    bound = 2.0 ** -8 * ref_x.abs() + 2 * C_BF16 * A[:n]
    r_kernel = ((y.permute(0, 3, 1, 2).double() - ref_x).abs() / bound).max().item()
    r_hi = ((conv_ref(_nhwc(hi[:n]), wb, b) - ref_x).abs() / bound).max().item()
    _note(f"{tag} against conv(x)", r_kernel)
    _note(f"{tag} hi-only conv against conv(x)", r_hi)
    assert r_kernel <= 1.0, f"{tag}: err / bound against conv(x) = {r_kernel:.3g}"
    assert r_hi >= 8.0, f"{tag}: the fixture cannot tell the split from hi alone ({r_hi:.3g})"


# Observed (444 splits): err / bound (c' = 2^-20) dw 0.028-0.033, db <= 0.0012; with the split, |dw - ref| is 0.0064 of
# the lo columns' contribution.
FIRST_WGRAD_CIN = [1, 3, 4, 7]


@pytest.mark.parametrize("Cin", FIRST_WGRAD_CIN)
def test_first_conv_wgrad_at_scale(b2u, cuda_device, Cin):
    """conv_wgrad(col, dz, taps=1, first_cin=Cin) with and without the bias gradient at 16 x 512 x 512: hundreds of
    split-K units folded by wgrad_reduce_kernel (mode 2 folds the lo columns into the same weight, mode 1 has none)."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    N, H, W, Cout = 16, 512, 512, 64
    g = _gen(dev, 50 + Cin)
    x = torch.randn((N, Cin, H, W), generator=g, device=dev)
    dz = _bf((N, H, W, Cout), g, dev)
    split = 18 * Cin <= 64
    splits, units = wgrad_plan(N, H, W, 64, Cout, 1, sms, False)
    assert units >= 3 * sms, f"{units} work units"
    col = ops.im2col_first(x)
    hi, lo = _split(x)
    xs = hi.double() + lo.double() if split else hi.double()
    xa = hi.double().abs() + lo.double().abs() if split else hi.double().abs()
    ref = wgrad_ref(_nhwc(xs), dz, 3)
    A = wgrad_ref(_nhwc(xa), dz, 3, absolute=True)
    del xs, xa
    ref_db, A_db = dz.double().sum((0, 1, 2)), dz.double().abs().sum((0, 1, 2))
    tag = f"first wgrad {N}x{H}x{W} Cin={Cin} splits={splits} mode={2 if split else 1}"
    for want_db in (False, True):
        out = ops.conv_wgrad(col, dz, taps=1, first_cin=Cin, want_db=want_db)
        dw, db = out if want_db else (out, None)
        check_sum(f"{tag} db={want_db}", dw, ref, A, c=C_WGRAD)
        if db is not None:
            check_sum(f"{tag} db", db, ref_db, A_db, c=C_WGRAD)
    if split:
        # the lo partial sums are folded in: the kernel's distance from the hi + lo gradient is a small fraction of the
        # lo columns' whole contribution
        r = ((dw.double() - ref).norm() / (wgrad_ref(_nhwc(hi), dz, 3) - ref).norm()).item()
        _note(f"{tag} |dw - ref| / |lo contribution|", r)
        assert r <= 0.1, f"{tag}: the lo columns' contribution is missing ({r:.3g})"


# ------------------------------------------------------------------------------------------------- ResNet-50 stem
def _stem_ref(xb, w, b, dz):
    """fp64 stride-2 7x7 conv of NCHW bf16 xb (+ b) -> NCHW, its weight gradient against NHWC dz, and both over absolute
    values, one image at a time (unfold + DGEMM)."""
    N, Cin, H, W = xb.shape
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    Cout = w.shape[0]
    wm = w.double().reshape(Cout, -1)
    y = torch.empty((N, Cout, Ho, Wo), dtype=F64, device=xb.device)
    Ay = torch.empty_like(y)
    dw = torch.zeros((Cout, Cin * 49), dtype=F64, device=xb.device)
    Adw = torch.zeros_like(dw)
    for n in range(N):
        cols = F.unfold(xb[n:n + 1].double(), 7, stride=2, padding=3)[0]        # [Cin * 49, Ho Wo]
        y[n] = (wm @ cols).view(Cout, Ho, Wo)
        Ay[n] = (wm.abs() @ cols.abs()).view(Cout, Ho, Wo)
        d = dz[n].reshape(-1, Cout).double()
        dw += d.t() @ cols.t()
        Adw += d.abs().t() @ cols.abs().t()
    y += b.double().view(-1, 1, 1)
    Ay += b.double().abs().view(-1, 1, 1)
    return y, Ay, dw.view(Cout, Cin, 7, 7), Adw.view(Cout, Cin, 7, 7)


# N, H, W of the image.  Observed err / bound: y 0.985-0.986 (bf16 rounding); dw 0.051 and 0.028 (148 splits).
STEM_CASES = [(16, 512, 512), (8, 383, 509)]


@pytest.mark.parametrize("N,H,W", STEM_CASES)
def test_stem_at_scale(b2u, cuda_device, N, H, W):
    """conv_fprop(im2col_stem(x), pack_weights_im2col(w, 192), b, 64, taps=1) and conv_wgrad_im2col(col, dz, 3, 49): the
    split-K kernel with Cout = 64 (half of a 128-row M block) over three 64-column K blocks, then the mode-1 reduce over
    49 taps."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    Ho, Wo, Cout = (H + 1) // 2, (W + 1) // 2, 64
    g = _gen(dev, 60)
    x = torch.randn((N, 3, H, W), generator=g, device=dev)
    w = torch.randn((Cout, 3, 7, 7), generator=g, device=dev) / 147 ** 0.5
    b = torch.randn((Cout,), generator=g, device=dev) * 0.1
    dz = _bf((N, Ho, Wo, Cout), g, dev)
    assert ops.conv_stat_rows(N, Ho, Wo, Cout, 1) >= 3 * sms
    splits, units = wgrad_plan(N, Ho, Wo, 192, Cout, 1, sms, False)
    assert units >= 3 * sms, f"{units} work units"
    col = ops.im2col_stem(x)
    wf = ops.pack_weights_im2col(w, 192)
    ref, A, ref_dw, A_dw = _stem_ref(x.to(BF), w.to(BF), b, dz)
    tag = f"stem {N}x{H}x{W}"
    for relu in (False, True):
        y = ops.conv_fprop(col, wf, b, Cout, taps=1, relu=relu)
        check_bf16(f"{tag} fprop relu={relu}", y, ref.relu() if relu else ref, A)
    check_sum(f"{tag} wgrad splits={splits}", ops.conv_wgrad_im2col(col, dz, 3, 49), ref_dw, A_dw, c=C_WGRAD)


# ------------------------------------------------------------------------------------------------- ceil-mode max-pool
def _pool_input(kind, shape, g, dev):
    """NHWC bf16 input whose windows often hold their maximum more than once.  relu: a post-ReLU tensor, ~84 % zeros;
    grid: values on a 0.5 grid, positive ties at the window maximum.  + 0.0 turns every -0.0 into +0.0, so that the
    forward can be compared bit for bit."""
    z = torch.randn(shape, generator=g, device=dev)
    v = (z - 1.0).clamp_min(0.0) if kind == "relu" else torch.round(2.0 * z) / 2.0
    return (v + 0.0).to(BF)


def _pool_ref(x):
    """fp64 nn.MaxPool2d(3, 2, ceil_mode=True) of NHWC x: pooled NCHW values, flat arg-max indices, and the fraction of
    windows whose maximum occurs more than once."""
    xd = x.permute(0, 3, 1, 2).double()
    N, C = xd.shape[:2]
    y, idx = F.max_pool2d(xd, 3, 2, ceil_mode=True, return_indices=True)
    # ATen keeps the first maximum in row-major scan order; the same on the CPU for two images
    y_cpu, idx_cpu = F.max_pool2d(xd[:2].cpu(), 3, 2, ceil_mode=True, return_indices=True)
    assert torch.equal(idx[:2].cpu(), idx_cpu) and torch.equal(y[:2].cpu(), y_cpu)
    # windows: a partial last window reaches one pixel past the edge, padded with -inf
    win = F.unfold(F.pad(xd, (0, 1, 0, 1), value=float("-inf")), 3, stride=2).view(N, C, 9, -1)
    ties = ((win == y.view(N, C, 1, -1)).sum(2) >= 2).double().mean().item()
    return y, idx, ties


# N, H, W, C: the stem's output, then 3 (one window), 4 (ceil mode's partial last window: H - 3 odd), 5 (whole windows)
# and odd x even.  Observed: ties in 0.199-0.350 of the windows; backward err / bound <= 0.992 (bf16 rounding of up to four dy;
# 0 at 3 x 3, where every pixel lies in one window).
POOL_CASES = [(16, 256, 256, 64), (16, 3, 3, 16), (16, 4, 4, 16), (16, 5, 5, 8), (8, 37, 64, 24), (8, 64, 37, 8)]


@pytest.mark.parametrize("kind", ["relu", "grid"])
@pytest.mark.parametrize("N,H,W,C", POOL_CASES)
def test_maxpool3x3s2_ceil_ties(b2u, cuda_device, N, H, W, C, kind):
    """maxpool3x3s2 bit for bit and maxpool3x3s2_bwd element by element against F.max_pool2d(ceil_mode=True) in fp64, with
    dy scattered through ATen's arg-max indices, on inputs where a tenth or more of the windows are tied."""
    ops, dev = b2u.ops, cuda_device
    g = _gen(dev, 70)
    x = _pool_input(kind, (N, H, W, C), g, dev)
    y_ref, idx, ties = _pool_ref(x)
    tag = f"maxpool3x3s2 {N}x{H}x{W}x{C} {kind}"
    print(f"[ties] {tag}: {ties:.3f} of the windows")
    assert ties >= 0.1, f"{tag}: only {ties:.3f} of the windows hold a tie"
    y = ops.maxpool3x3s2(x)
    assert torch.equal(_bits(y), _bits(y_ref.to(BF).permute(0, 2, 3, 1).contiguous())), f"{tag}: forward differs"
    Ho, Wo = y_ref.shape[2:]
    dy = _bf((N, Ho, Wo, C), g, dev)
    dyd = dy.permute(0, 3, 1, 2).double().reshape(N, C, -1)
    flat = idx.view(N, C, -1)
    ref = torch.zeros((N, C, H * W), dtype=F64, device=dev).scatter_add_(2, flat, dyd).view(N, C, H, W)
    A = torch.zeros((N, C, H * W), dtype=F64, device=dev).scatter_add_(2, flat, dyd.abs()).view(N, C, H, W)
    check_bf16(f"{tag} bwd", ops.maxpool3x3s2_bwd(dy, x), ref, A)
