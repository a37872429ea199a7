"""GPU: the hot kernels at training-scale shapes, where every CTA of a persistent or fixed-size grid takes several tiles,
work units or grid-stride passes, against float64 references of the same bf16 operands the kernels read.

The kernel tests in test_kernels_gpu.py mostly run shapes where each CTA gets one tile.  The state that matters only from
a CTA's second tile on (tile-id queue, double-buffered accumulator, bias parity, cross-tile mask prefetch, split-K units,
the second grid-stride pass, the reduction tail) is checked here, element by element:

  bf16 outputs   |y - ref| <= 2^-8 |ref| + c A,   A = conv(|x|, |w|) + |b|  (the magnitude the fp32 accumulation handled)
  fp32 sums      |s - ref| <= c' A_s,            A_s = the same sum over absolute values

A wrong tile, a dropped K chunk or split, or one element off by 1.0 breaks these bounds by orders of magnitude, while
rel-L2 over a tensor of 10^7 elements may not notice.  Each case also asserts the regime it claims to exercise (at
least three tiles or units per SM), so a change of the tiling rules cannot quietly shrink it.

Calibration, one NVIDIA B200 (148 SMs): the largest err / bound seen per case is noted next to each case list.
"""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
F64 = torch.float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Calibrated on one NVIDIA B200 at a 1000 W power limit.  The bf16 bounds are tight by design (round to nearest
# alone reaches ~0.99 of 2^-8 |ref|); the fp32 constants leave >= 3x headroom over the largest err / bound observed.
C_BF16 = 2.0 ** -16        # fp32 accumulation term of the bf16-output bound
C_SUM = 2.0 ** -18         # fp32 sums: statistics rows, grid-stride reductions, head and losses
C_WGRAD = 2.0 ** -20       # split-K weight gradients: tight enough that one partial off by 1.0 fails every case


def _gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def _bf(shape, g, dev, scale=1.0):
    return (torch.randn(shape, generator=g, device=dev) * scale).to(BF)


def _sms(b2u):
    return b2u.ops.lib().b2u_num_sms()


def _note(name, ratio):
    print(f"[err/bound] {name}: {ratio:.3g}")


def check_bf16(name, y_nhwc, ref, A, c=C_BF16):
    """y: bf16 NHWC kernel output; ref, A: fp64 NCHW."""
    y = y_nhwc.permute(0, 3, 1, 2).double()
    err = (y - ref).abs()
    bound = 2.0 ** -8 * ref.abs() + c * A
    ratio = (err / (bound + 1e-300)).max().item()
    _note(name, ratio)
    assert ratio <= 1.0, f"{name}: err / bound = {ratio:.3g}"
    assert ((y - ref).norm() / ref.norm()).item() <= 6e-3, name


def check_sum(name, got, ref, A, c=C_SUM):
    err = (got.double() - ref).abs()
    ratio = (err / (c * A + 1e-300)).max().item()
    _note(name, ratio)
    assert ratio <= 1.0, f"{name}: err / bound = {ratio:.3g}"
    assert ((got.double() - ref).norm() / ref.norm()).item() <= 1e-4, name


def conv_ref(x, w, b=None, absolute=False):
    """fp64 cross-correlation, 'same' padding, of NHWC x with OIHW w -> NCHW, one image at a time (unfold + DGEMM).
    absolute: the same over |x| and |w| (+ |b|)."""
    N, H, W, _ = x.shape
    k = w.shape[-1]
    wm = w.double().reshape(w.shape[0], -1)
    if absolute:
        wm = wm.abs()
    out = torch.empty((N, w.shape[0], H, W), dtype=F64, device=x.device)
    for n in range(N):
        xn = x[n:n + 1].permute(0, 3, 1, 2).double()
        cols = F.unfold(xn.abs() if absolute else xn, k, padding=k // 2)[0]
        out[n] = (wm @ cols).view(-1, H, W)
    if b is not None:
        out += (b.double().abs() if absolute else b.double()).view(1, -1, 1, 1)
    return out


def wgrad_ref(x, dz, k, absolute=False):
    """fp64 weight gradient [Cout, Cin, k, k] of the 'same' conv: sum over pixels of dz (x) im2col(x)."""
    N, H, W, Cin = x.shape
    acc = torch.zeros((dz.shape[-1], Cin * k * k), dtype=F64, device=x.device)
    for n in range(N):
        xn = x[n:n + 1].permute(0, 3, 1, 2).double()
        cols = F.unfold(xn.abs() if absolute else xn, k, padding=k // 2)[0]
        dn = dz[n].reshape(H * W, -1).double()
        acc += (dn.abs() if absolute else dn).t() @ cols.t()
    return acc.view(-1, Cin, k, k)


def dgrad_weight(w):
    """OIHW weight of the data gradient as a forward conv: transpose in/out channels, rotate the taps."""
    return w.transpose(0, 1).flip(2, 3)


def default_bn(Cout):
    return 256 if Cout % 256 == 0 else 192 if Cout % 192 == 0 else 128 if Cout % 128 == 0 else 64


def tile_sums(z, rows, tile_w=16, tile_h=8):
    """fp64 per-M-tile column sums (sum z, sum z^2, and the same over |z|) in the kernels' tile order
    m = (n * tiles_h + th) * tiles_w + tw; the stacked tile height follows from the row count."""
    N, H, W, C = z.shape
    tw = -(-W // tile_w)
    th = rows // (N * tw)
    assert th * N * tw == rows
    hh = next(tile_h * m for m in (1, 2, 4) if -(-H // (tile_h * m)) == th)
    zp = torch.zeros((N, th * hh, tw * tile_w, C), dtype=F64, device=z.device)
    zp[:, :H, :W] = z.double()
    zp = zp.view(N, th, hh, tw, tile_w, C)
    s = zp.sum((2, 4)).reshape(rows, C)
    q = (zp * zp).sum((2, 4)).reshape(rows, C)
    a = zp.abs().sum((2, 4)).reshape(rows, C)
    return s, q, a


# ------------------------------------------------------------------------------------------------- conv forward
CONV_CASES = [
    # N, H, W, C0, C1, Cout, taps.  Observed err / bound: y, z and the scaled y 0.96-0.99 (bf16 rounding), statistics
    # rows <= 0.056, totals <= 5e-4.
    (8, 256, 256, 64, 0, 64, 9),        # 1024 tiles with four stacked M tiles, 4096 with one
    (8, 128, 128, 128, 128, 128, 9),    # two sources; N tile 128 and 64 (two N tiles: bias parity)
    (8, 64, 64, 512, 0, 512, 9),        # N tiles 256 / 128 / 64: 2..8 N tiles per M tile
    (24, 100, 92, 64, 0, 64, 9),        # ragged in both directions (100 = 3 x 32 + 4, 92 = 5 x 16 + 12)
    (8, 128, 128, 64, 0, 128, 1),       # 1x1
]


def _conv_case(b2u, dev, N, H, W, C0, C1, Cout, taps, seed):
    g = _gen(dev, seed)
    k = 3 if taps == 9 else 1
    x = _bf((N, H, W, C0 + C1), g, dev)
    w = torch.randn((Cout, C0 + C1, k, k), generator=g, device=dev) / ((C0 + C1) * taps) ** 0.5
    b = torch.randn((Cout,), generator=g, device=dev)
    wf, wd = b2u.ops.pack_weights(w)
    x0 = x[..., :C0].contiguous()
    x1 = x[..., C0:].contiguous() if C1 else None
    return x, x0, x1, w.to(BF), b, wf, wd


def _folded_bn_coeffs(C, dev, seed):
    """Per-channel scale s (|s| in [0.5, 1.5], both signs) and shift b' of a folded eval-mode BatchNorm."""
    g = _gen(dev, seed)
    s = (torch.rand((C,), generator=g, device=dev) + 0.5) * torch.where(torch.arange(C, device=dev) % 2 == 1, -1.0, 1.0)
    return s, torch.randn((C,), generator=g, device=dev)


def _scaled_ref(conv, A, s, bp):
    """fp64 relu(s conv + b') of an NCHW conv result and its magnitude bound |s| A + |b'|."""
    sh = (-1, 1, 1)
    return (s.double().view(sh) * conv + bp.double().view(sh)).relu(), s.double().abs().view(sh) * A + bp.double().abs().view(sh)


@pytest.mark.parametrize("N,H,W,C0,C1,Cout,taps", CONV_CASES)
def test_conv_fprop_at_scale(b2u, cuda_device, N, H, W, C0, C1, Cout, taps):
    """conv + bias + ReLU in every tiling variant the launcher can pick, and the statistics epilogue (per-tile rows)."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    x, x0, x1, wb, b, wf, _ = _conv_case(b2u, dev, N, H, W, C0, C1, Cout, taps, 1)
    ref_z = conv_ref(x, wb, b)
    A = conv_ref(x, wb, b, absolute=True)
    ref = ref_z.relu()
    variants = [0, 1 << 16, 2 << 16] + [bn for bn in (64, 128, 192, 256) if Cout % bn == 0]
    for bn in variants:
        n_tiles = Cout // ((bn & 0xffff) or default_bn(Cout))
        assert ops.conv_stat_rows(N, H, W, Cout, taps, bn) * n_tiles >= 3 * sms, f"variant {bn:#x} is not multi-tile"
        y = ops.conv_fprop(x0, wf, b, Cout, taps=taps, relu=True, x1=x1, bn=bn)
        check_bf16(f"fprop {N}x{H}x{W} {C0}+{C1}->{Cout} t{taps} bn={bn:#x}", y, ref, A)
    # folded eval-mode BatchNorm in the epilogue: y = relu(s conv(x) + b'), s of both signs (a ReLU taken before the
    # scale would pass every channel with s > 0)
    s, bp = _folded_bn_coeffs(Cout, dev, 16)
    ref_s, A_s = _scaled_ref(ref_z - b.double().view(-1, 1, 1), A, s, bp)
    for bn in variants:
        y = ops.conv_fprop_scaled(x0, wf, s, bp, Cout, taps=taps, relu=True, x1=x1, bn=bn)
        check_bf16(f"fprop scaled {N}x{H}x{W} {C0}+{C1}->{Cout} t{taps} bn={bn:#x}", y, ref_s, A_s)
    del ref_s, A_s
    for bn in (0, 1 << 16):
        rows = ops.conv_stat_rows(N, H, W, Cout, taps, bn)
        st = torch.full((rows * 2 * Cout,), float("nan"), device=dev)
        z = ops.conv_fprop(x0, wf, b, Cout, taps=taps, relu=False, x1=x1, bn=bn, stats=st)
        assert torch.equal(z.view(torch.int16), ops.conv_fprop(x0, wf, b, Cout, taps=taps, relu=False, x1=x1, bn=bn).view(torch.int16))
        name = f"fprop stats {N}x{H}x{W} {C0}+{C1}->{Cout} t{taps} bn={bn:#x}"
        check_bf16(name, z, ref_z, A)
        # every M tile's row holds that tile's sums of the bf16 values as stored, whichever CTA computed it
        s, q, a = tile_sums(z, rows)
        got = st.view(rows, 2, Cout)
        check_sum(name + " rows sum", got[:, 0], s, a)
        check_sum(name + " rows sumsq", got[:, 1], q, q)
        check_sum(name + " total", got.double().sum(0)[0], s.sum(0), a.sum(0))


def test_decoder_conv_scaled_at_scale(b2u, cuda_device):
    """b2u_decoder_conv_fprop with a folded eval-mode BatchNorm (scale=...), the inference form of every BatchNorm decoder
    stage: relu(s conv([skip, upsample2x(low)]) + b') against fp64 on the up-sampled bf16 operand the kernel interpolates
    (bit-identical to b2u_upsample2x_fwd), s of both signs, in every N tile and M-tile stacking of a multi-tile launch.
    Observed err / bound: <= 0.98 (bf16 rounding)."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    N, H, W, C0, C1, Cout = 8, 128, 128, 128, 128, 128
    g = _gen(dev, 17)
    skip = _bf((N, H, W, C0), g, dev)
    low = _bf((N, H // 2, W // 2, C1), g, dev)
    w = torch.randn((Cout, C0 + C1, 3, 3), generator=g, device=dev) / ((C0 + C1) * 9) ** 0.5
    wf, _ = ops.pack_weights(w)
    x = torch.cat([skip, ops.upsample2x(low)], -1)
    wb = w.to(BF)
    s, bp = _folded_bn_coeffs(Cout, dev, 18)
    ref_s, A_s = _scaled_ref(conv_ref(x, wb), conv_ref(x, wb, absolute=True), s, bp)
    for bn in (0, 1 << 16, 64, (1 << 16) | 64):
        units = ops.conv_stat_rows(N, H, W, Cout, 9, bn | (1 << 18)) * (Cout // ((bn & 0xffff) or default_bn(Cout)))
        assert units >= 3 * sms, f"variant {bn:#x} is not multi-tile"
        y = ops.decoder_conv_fprop(skip, low, wf, bp, Cout, relu=True, scale=s, bn=bn)
        check_bf16(f"decoder scaled {N}x{H}x{W} {C0}+{C1}->{Cout} bn={bn:#x}", y, ref_s, A_s)


# ------------------------------------------------------------------------------------------------- conv data gradient
DGRAD_CASES = [
    # N, H, W, C0, C1, Cz: dx has C0 + C1 channels (split in two outputs when C1 > 0), dz has Cz.
    # Observed err / bound: dx 0.97-0.98 (bf16 rounding), column sums <= 3.3e-4.
    (8, 256, 256, 64, 0, 64),           # masked N tile 64: the cp.async mask stream prefetches across tiles (static order)
    (8, 128, 128, 128, 128, 128),       # two outputs; masked / bit-masked over 256 channels (N tile 256, dynamic order)
]


@pytest.mark.parametrize("N,H,W,C0,C1,Cz", DGRAD_CASES)
def test_conv_dgrad_at_scale(b2u, cuda_device, N, H, W, C0, C1, Cz):
    """dgrad masked by a bf16 tensor, by the relu bit mask conv_fprop_relu_bits wrote (bit-identical to y > 0 at scale),
    with the column-sum epilogue (bias_from_stats), and split into two outputs."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    g = _gen(dev, 2)
    Cm = C0 + C1
    # the layer whose output is masked: a multi-tile forward conv + ReLU writing y and its bit mask
    xin = _bf((N, H, W, 64), g, dev)
    wy = torch.randn((Cm, 64, 3, 3), generator=g, device=dev) / 24.0
    by = torch.randn((Cm,), generator=g, device=dev) * 0.5
    wfy, _ = ops.pack_weights(wy)
    y = ops.conv_fprop(xin, wfy, by, Cm, relu=True)
    bits = torch.zeros((N, H, W, Cm // 64), dtype=torch.int64, device=dev)
    yb = ops.conv_fprop_relu_bits(xin, wfy, by, Cm, bits)
    assert torch.equal(yb.view(torch.int16), y.view(torch.int16))
    want_bits = ((y > 0).view(N, H, W, Cm // 64, 64).to(torch.int64) << torch.arange(64, device=dev)).sum(-1)
    assert torch.equal(bits, want_bits)
    del want_bits
    # the conv whose data gradient is taken
    dz = _bf((N, H, W, Cz), g, dev)
    w = (torch.randn((Cz, Cm, 3, 3), generator=g, device=dev) / (Cm * 9) ** 0.5).to(BF)
    _, wd = ops.pack_weights(w.float())
    wt = dgrad_weight(w)
    ref = conv_ref(dz, wt)
    A = conv_ref(dz, wt, absolute=True)
    keep = (y > 0).permute(0, 3, 1, 2)
    tag = f"{N}x{H}x{W} {Cz}->{Cm}"
    for masked in (True, False):
        rows = ops.conv_dgrad_stat_rows(N, H, W, Cm, 9, masked=masked)
        assert rows * (Cm // default_bn(Cm)) >= 3 * sms
    d = ops.conv_dgrad(dz, wd, Cm, mask=y)
    check_bf16(f"dgrad mask {tag}", d, ref * keep, A)
    db = ops.conv_dgrad_bits(dz, wd, Cm, bits)
    assert torch.equal(db.view(torch.int16), d.view(torch.int16))
    col = d.double().sum((0, 1, 2))
    col_abs = d.double().abs().sum((0, 1, 2))
    for masked in (True, False):
        rows = ops.conv_dgrad_stat_rows(N, H, W, Cm, 9, masked=masked)
        st = torch.full((rows * 2 * Cm,), float("nan"), device=dev)
        ds = ops.conv_dgrad(dz, wd, Cm, mask=y, stats=st) if masked else ops.conv_dgrad_bits(dz, wd, Cm, bits, stats=st)
        assert torch.equal(ds.view(torch.int16), d.view(torch.int16))
        check_sum(f"dgrad {'mask' if masked else 'bits'} stats {tag}", ops.bias_from_stats(st, rows, Cm), col, col_abs)
    if C1:
        d0, d1 = ops.conv_dgrad(dz, wd, C0, C1=C1)
        check_bf16(f"dgrad two outputs {tag}", torch.cat([d0, d1], -1), ref, A)


# ------------------------------------------------------------------------------------------------- conv weight gradient
def _choose_splits(base, kblocks, sms):
    """conv_wgrad.cu choose_splits: the split count giving 3..8 units per SM that wastes the fewest slots of the last round."""
    lo, hi = -(-3 * sms // base), -(-8 * sms // base)
    cap = max(kblocks // 8, 1)
    lo, hi = max(min(lo, cap), 1), min(hi, cap)
    best, best_waste = lo, 1e30
    for sp in range(lo, hi + 1):
        units = base * sp
        waste = -(-units // sms) * sms / units
        if waste < best_waste - 1e-9:
            best, best_waste = sp, waste
    return best


def wgrad_plan(N, H, W, Cin, Cout, taps, sms, swapped):
    """(splits, units) of plan_wgrad / plan_wgrad64 (16 x 8 pixel K blocks)."""
    kblocks = N * -(-H // 8) * -(-W // 16)
    base = Cin // 64 if swapped else -(-Cout // 128) * (Cin // 64) * (3 if taps == 9 else 1)
    sp = _choose_splits(base, kblocks, sms)
    return sp, base * sp


WGRAD_CASES = [
    # N, H, W, Cin, Cout, taps.  Observed err / bound (c' = 2^-20): dw 0.037, 0.20, 0.023, 0.012 in this order; db <= 0.0031.
    (8, 128, 128, 128, 128, 9),         # 74 splits (74 % 4 = 2: the reduction tail runs)
    (4, 64, 64, 512, 512, 9),           # four M blocks of 128 output channels, 6 splits (tail again)
    (8, 256, 256, 128, 128, 1),         # 1x1: the generic reduction, hundreds of splits
    (8, 256, 256, 64, 64, 9),           # Cout = 64: swapped-role kernel (444 splits) and the generic one (flags bit 1)
]


@pytest.mark.parametrize("N,H,W,Cin,Cout,taps", WGRAD_CASES)
def test_conv_wgrad_at_scale(b2u, cuda_device, N, H, W, Cin, Cout, taps):
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    g = _gen(dev, 3)
    k = 3 if taps == 9 else 1
    x = _bf((N, H, W, Cin), g, dev)
    dz = _bf((N, H, W, Cout), g, dev)
    ref = wgrad_ref(x, dz, k)
    A = wgrad_ref(x, dz, k, absolute=True)
    ref_db, A_db = dz.double().sum((0, 1, 2)), dz.double().abs().sum((0, 1, 2))
    tag = f"{N}x{H}x{W} {Cin}->{Cout} t{taps}"
    swapped_shape = Cout == 64 and taps == 9
    runs = [(0, True), (0, False)] + ([(2, False), (2, True)] if swapped_shape else [])      # (flags, want_db)
    for flags, want_db in runs:
        swapped = swapped_shape and not flags & 2
        splits, units = wgrad_plan(N, H, W, Cin, Cout, taps, sms, swapped)
        assert units >= 3 * sms, f"flags {flags}: {units} work units"
        out = ops.conv_wgrad(x, dz, taps=taps, flags=flags, want_db=want_db)
        dw, db = out if want_db else (out, None)
        name = f"wgrad {tag} flags={flags} db={want_db} splits={splits}"
        check_sum(name, dw, ref, A, c=C_WGRAD)
        if db is not None:
            check_sum(name + " db", db, ref_db, A_db, c=C_WGRAD)


def test_wgrad_cases_cover_the_reduction_tail(b2u, cuda_device):
    sms = _sms(b2u)
    tails = [c for c in WGRAD_CASES if c[5] == 9 and wgrad_plan(*c, sms, False)[0] % 4 != 0]
    assert tails, "no 3x3 wgrad case leaves a remainder for wgrad_reduce9_kernel's tail loop"


# ------------------------------------------------------------------------------------------------- BatchNorm
BN_SHIFTS = (0, 4, -4, 16, -16, 32, -32, 64, -64)       # channel mean / std


def _bn_data(dev, N, H, W, C, seed, shifts=BN_SHIFTS):
    g = _gen(dev, seed)
    std = torch.linspace(0.25, 1.0, C, device=dev)
    ratio = torch.tensor([shifts[c % len(shifts)] for c in range(C)], dtype=torch.float32, device=dev)
    z = (torch.randn((N, H, W, C), generator=g, device=dev) * std + ratio * std).to(BF)
    return z, ratio


def _bn_ref_stats(z):
    zd = z.double().reshape(-1, z.shape[-1])
    mean = zd.mean(0)
    var = ((zd - mean) ** 2).mean(0)           # two-pass
    return mean, var


# P = 4.19 M (the benchmark's full-resolution layer); C8 = 256.  Observed: var rel <= 4.0e-6, invstd rel <= 2.0e-6 at every
# shift (1.2e-2 and 6.1e-3 at mean = 64 std before the column sums were taken about a pivot); err / bound y, dz <= 0.992
# (bf16 rounding), dgamma, dbeta <= 1.7e-3.
BN_CASES = [(16, 512, 512, 64), (8, 32, 32, 2048)]


@pytest.mark.parametrize("N,H,W,C", BN_CASES)
def test_batchnorm_train_at_scale(b2u, cuda_device, N, H, W, C):
    """Batch statistics over the grid-stride column sums: mean, var, invstd and the running statistics to 2e-5 relative at
    channel means up to 64 standard deviations; y, and the backward (dgamma, dbeta, dz), element by element."""
    ops, dev = b2u.ops, cuda_device
    z, ratio = _bn_data(dev, N, H, W, C, 4)
    P = N * H * W
    g = _gen(dev, 5)
    gamma = 1 + 0.2 * torch.randn((C,), generator=g, device=dev)
    beta = 0.1 * torch.randn((C,), generator=g, device=dev)
    rm0, rv0 = 0.1 * torch.randn((C,), generator=g, device=dev), torch.rand((C,), generator=g, device=dev) + 0.5
    rm, rv = rm0.clone(), rv0.clone()
    y, mean, invstd = ops.bn_fwd_train(z, gamma, beta, rm, rv, relu=True)
    m_ref, v_ref = _bn_ref_stats(z)
    is_ref = (v_ref + 1e-5).rsqrt()
    std_ref = v_ref.sqrt()
    e_mean = ((mean.double() - m_ref).abs() / std_ref)
    e_var = (invstd.double() ** -2 - 1e-5 - v_ref).abs() / v_ref          # the variance the kernel normalised with
    e_is = (invstd.double() - is_ref).abs() / is_ref
    for r in sorted(set(ratio.tolist())):
        sel = ratio == r
        print(f"[bn] P={P} C={C} mean/std={r:+.0f}: mean err/std {e_mean[sel].max().item():.2e}  "
              f"var rel {e_var[sel].max().item():.2e}  invstd rel {e_is[sel].max().item():.2e}")
    assert e_mean.max().item() <= 2e-5
    assert e_var.max().item() <= 2e-5 and e_is.max().item() <= 2e-5
    want_rv = 0.9 * rv0.double() + 0.1 * v_ref * P / (P - 1)
    assert ((rv.double() - want_rv).abs() / want_rv).max().item() <= 2e-6
    assert torch.allclose(rm.double(), 0.9 * rm0.double() + 0.1 * m_ref, rtol=1e-6, atol=1e-6 * std_ref.max().item())
    # y = relu(gamma (z - mean) invstd + beta): the apply pass in fp32 from the kernel's saved statistics
    zd = z.double().permute(0, 3, 1, 2)
    sh = (-1, 1, 1)
    xhat = (zd - m_ref.view(sh)) * is_ref.view(sh)
    ref_y = (gamma.double().view(sh) * xhat + beta.double().view(sh)).relu()
    A_y = (gamma.double().abs().view(sh) * (zd.abs() + m_ref.abs().view(sh)) * is_ref.view(sh) + beta.double().abs().view(sh))
    check_bf16(f"bn fwd P={P} C={C}", y, ref_y, A_y)
    # eval forward with the updated running statistics
    ye = ops.bn_fwd_eval(z, gamma, beta, rm, rv, relu=True)
    ise = (rv.double() + 1e-5).rsqrt().view(sh)
    ref_e = (gamma.double().view(sh) * (zd - rm.double().view(sh)) * ise + beta.double().view(sh)).relu()
    A_e = gamma.double().abs().view(sh) * (zd.abs() + rm.double().abs().view(sh)) * ise + beta.double().abs().view(sh)
    check_bf16(f"bn eval P={P} C={C}", ye, ref_e, A_e)
    del ref_e, A_e, ye
    # backward with the kernel's own ReLU decisions (a tie at y = 0 is the kernel's to make)
    dy = _bf((N, H, W, C), g, dev)
    gm = dy.double().permute(0, 3, 1, 2) * (y > 0).permute(0, 3, 1, 2)
    dz, dgam, dbet = ops.bn_bwd(dy, None, z, gamma, mean, invstd, relu=True, beta=beta)
    xk = (zd - mean.double().view(sh)) * invstd.double().view(sh)
    ref_db, ref_dg = gm.sum((0, 2, 3)), (gm * xk).sum((0, 2, 3))
    check_sum(f"bn bwd dbeta P={P} C={C}", dbet, ref_db, gm.abs().sum((0, 2, 3)))
    check_sum(f"bn bwd dgamma P={P} C={C}", dgam, ref_dg, (gm * xk).abs().sum((0, 2, 3)))
    a = (gamma.double() * invstd.double()).view(sh)
    ref_dz = a * (gm - (ref_db / P).view(sh) - xk * (ref_dg / P).view(sh))
    A_dz = a.abs() * (gm.abs() + (ref_db.abs() / P).view(sh) + xk.abs() * (ref_dg.abs() / P).view(sh))
    check_bf16(f"bn bwd dz P={P} C={C}", dz, ref_dz, A_dz)


def test_batchnorm_centered_running_mean(b2u, cuda_device):
    """centered: z holds conv - running_mean; the statistics are of the stored tensor, the running mean sees the true one."""
    ops, dev = b2u.ops, cuda_device
    N, H, W, C = 16, 512, 512, 64
    z, _ = _bn_data(dev, N, H, W, C, 6, shifts=(0, 1, -2, 3))
    P = N * H * W
    rm0 = torch.linspace(-40, 40, C, device=dev)
    rv0 = torch.ones(C, device=dev)
    rm, rv = rm0.clone(), rv0.clone()
    _, mean, invstd = ops.bn_fwd_train(z, None, None, rm, rv, relu=False, centered=True)
    m_ref, v_ref = _bn_ref_stats(z)
    assert ((mean.double() - m_ref).abs() / v_ref.sqrt()).max().item() <= 2e-5
    assert ((invstd.double() - (v_ref + 1e-5).rsqrt()).abs() * (v_ref + 1e-5).sqrt()).max().item() <= 2e-5
    want_rm = 0.9 * rm0.double() + 0.1 * (m_ref + rm0.double())
    assert ((rm.double() - want_rm).abs() <= 1e-5 * (want_rm.abs() + 1)).all()
    want_rv = 0.9 + 0.1 * v_ref * P / (P - 1)
    assert ((rv.double() - want_rv).abs() / want_rv).max().item() <= 2e-5


def test_batchnorm_epilogue_statistics_at_scale(b2u, cuda_device):
    """bn_fwd_train_stats from the per-tile sums of a multi-tile 1x1 conv whose bias shifts each channel by up to 64 of its
    standard deviations.  Each row sums one tile (256 pixels) in fp32, so E[z^2] - mean^2 loses ~2^-24 (mean / std)^2 of
    the variance (observed: var rel 3.7e-4 at 64 std, 3.2e-5 at 16, 1.4e-6 at 4).  The centred mode is the remedy: with
    the running mean folded into the conv's bias the same channels meet 2e-5."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    N, H, W, C = 16, 512, 512, 64
    P = N * H * W
    g = _gen(dev, 7)
    x = _bf((N, H, W, C), g, dev)
    std = torch.linspace(0.25, 1.0, C, device=dev)
    ratio = torch.tensor([BN_SHIFTS[c % len(BN_SHIFTS)] for c in range(C)], dtype=torch.float32, device=dev)
    wf, _ = ops.pack_weights(torch.diag(std).view(C, C, 1, 1))
    rows = ops.conv_stat_rows(N, H, W, C, 1)
    assert rows >= 3 * sms
    for centered in (False, True):
        rm = ratio * std if centered else torch.zeros(C, device=dev)       # a running mean that has converged
        st = torch.empty((rows * 2 * C,), device=dev)
        z = ops.conv_fprop(x, wf, ratio * std - rm, C, taps=1, relu=False, stats=st)
        rv = torch.ones(C, device=dev)
        _, mean, invstd = ops.bn_fwd_train(z, None, None, rm, rv, relu=False, stats=st, stat_rows=rows, centered=centered)
        m_ref, v_ref = _bn_ref_stats(z)
        e_mean = (mean.double() - m_ref).abs() / v_ref.sqrt()
        e_var = (invstd.double() ** -2 - 1e-5 - v_ref).abs() / v_ref
        for r in sorted(set(ratio.tolist())):
            sel = ratio == r
            print(f"[bn stats epilogue] centered={centered} mean/std={r:+.0f}: mean err/std {e_mean[sel].max().item():.2e}  "
                  f"var rel {e_var[sel].max().item():.2e}")
        assert e_mean.max().item() <= 2e-5
        allowed = 2e-5 + (0.0 if centered else 2e-7) * ratio.double() ** 2
        assert (e_var <= allowed).all(), (e_var / allowed).max().item()
        assert ((rv.double() - (0.9 + 0.1 * v_ref * P / (P - 1))).abs() <= 0.1 * allowed * v_ref + 2e-6).all()


# ------------------------------------------------------------------------------------------------- SyncBatchNorm
BN_BLOCKS = 296            # bn.cu kBnBlocks: the column-sum grid (2 blocks of 256 threads per SM of a B200)


def _colsum_passes(P, C, unroll):
    """Grid-stride passes of the last, least loaded block of bn_colsum_kernel over P rows (0: some blocks get no row).
    unroll: kBnUnroll, 8 for the forward statistics, 4 for the backward sums."""
    rows = 256 // min(C // 8, 256)
    first = (BN_BLOCKS - 1) * rows
    return 0 if first >= P else -(-(P - first) // (unroll * BN_BLOCKS * rows))


def _bn_ws(ops, C, dev):
    return torch.empty(ops.lib().b2u_bn_workspace(C), dtype=torch.uint8, device=dev)


def _sync_bn_fwd(ops, z, R, gamma, beta, rm0, rv0, residual=None):
    """SyncBatchNorm forward on R emulated ranks holding one shard of whole images each: every rank's moments land in its
    slot of one [R][2][C] buffer (what the all-gather delivers), then every rank applies with its own running statistics.
    Returns the stitched y and, per rank, (save_mean, save_invstd, running_mean, running_var)."""
    lib, ptr, check, sp = ops.lib(), ops.ptr, ops.check, ops.stream_ptr()
    C = z.shape[-1]
    zs = z.view(R, -1, C)
    res = residual.view(R, -1, C) if residual is not None else [None] * R
    Pr = zs.shape[1]
    ws = _bn_ws(ops, C, z.device)
    moments = torch.full((R, 2, C), float("nan"), device=z.device)
    for r in range(R):
        check(lib.b2u_bn_moments(ptr(zs[r]), ptr(moments[r]), ptr(ws), ws.numel(), Pr, C, sp))
    y = torch.empty_like(z)
    ys = y.view(R, -1, C)
    per_rank = []
    for r in range(R):
        mean, invstd = torch.empty(C, device=z.device), torch.empty(C, device=z.device)
        rm, rv = rm0.clone(), rv0.clone()
        check(lib.b2u_bn_fwd_train_moments(ptr(zs[r]), ptr(res[r]), ptr(ys[r]), ptr(gamma), ptr(beta), ptr(rm), ptr(rv), ptr(mean),
                                           ptr(invstd), ptr(moments), R, ptr(ws), ws.numel(), Pr, C, 1e-5, 0.1, 1, sp))
        per_rank.append((mean, invstd, rm, rv))
    return y, per_rank


def _sync_bn_bwd(ops, dy, y, z, R, gamma, beta, mean, invstd):
    """SyncBatchNorm backward on R emulated ranks: each rank's (sum g, sum g xhat), their sum (the all-reduce), then each
    rank's dz and gout.  y=None recomputes the ReLU mask from z.  Returns (dz, gout, per-rank sums [R][2][C])."""
    lib, ptr, check, sp = ops.lib(), ops.ptr, ops.check, ops.stream_ptr()
    C = z.shape[-1]
    dys, zs = dy.view(R, -1, C), z.view(R, -1, C)
    yv = y.view(R, -1, C) if y is not None else [None] * R
    Pr = zs.shape[1]
    ws = _bn_ws(ops, C, z.device)
    sums = torch.full((R, 2, C), float("nan"), device=z.device)
    for r in range(R):
        check(lib.b2u_bn_bwd_sums(ptr(dys[r]), ptr(yv[r]), ptr(zs[r]), ptr(gamma), ptr(beta), ptr(mean), ptr(invstd), ptr(sums[r]),
                                  ptr(ws), ws.numel(), Pr, C, 1, sp))
    total = sums.sum(0)
    dz, gout = torch.full_like(z, float("nan")), torch.full_like(z, float("nan"))
    dzs, gs = dz.view(R, -1, C), gout.view(R, -1, C)
    for r in range(R):
        check(lib.b2u_bn_bwd_apply_sums(ptr(dys[r]), ptr(yv[r]), ptr(zs[r]), ptr(gamma), ptr(beta), ptr(mean), ptr(invstd), ptr(dzs[r]),
                                        ptr(gs[r]), ptr(total), R * Pr, ptr(ws), ws.numel(), Pr, C, 1, sp))
    return dz, gout, sums


def _bn_stat_errors(tag, mean, invstd, z, ratio):
    """Per-shift errors of the statistics a BatchNorm normalised with (mean in standard deviations, var and invstd relative),
    printed; asserted against the one-GPU bounds."""
    m_ref, v_ref = _bn_ref_stats(z)
    e_mean = (mean.double() - m_ref).abs() / v_ref.sqrt()
    e_var = (invstd.double() ** -2 - 1e-5 - v_ref).abs() / v_ref
    is_ref = (v_ref + 1e-5).rsqrt()
    e_is = (invstd.double() - is_ref).abs() / is_ref
    for r in sorted(set(ratio.tolist())):
        sel = ratio == r
        print(f"[{tag}] mean/std={r:+.0f}: mean err/std {e_mean[sel].max().item():.2e}  var rel {e_var[sel].max().item():.2e}  "
              f"invstd rel {e_is[sel].max().item():.2e}")
    assert e_mean.max().item() <= 2e-5, f"{tag}: mean err / std {e_mean.max().item():.3g}"
    assert e_var.max().item() <= 2e-5 and e_is.max().item() <= 2e-5, f"{tag}: var rel {e_var.max().item():.3g}"
    return m_ref, v_ref


def _bn_fwd_ref(zd, mean, invstd, gamma, beta, residual=None):
    """fp64 y = relu(gamma (z - mean) invstd + beta [+ residual]) of NCHW zd, and the magnitude A of its fp32 evaluation."""
    sh = (-1, 1, 1)
    m, s = mean.double().view(sh), invstd.double().view(sh)
    gd, bd = gamma.double().view(sh), beta.double().view(sh)
    v = gd * (zd - m) * s + bd
    A = gd.abs() * (zd.abs() + m.abs()) * s + bd.abs()
    if residual is not None:
        rd = residual.double().permute(0, 3, 1, 2)
        v, A = v + rd, A + rd.abs()
    return v.relu(), A


def _bn_bwd_check(tag, dz, gout, sums, dy, y, z, R, gamma, mean, invstd):
    """dz and gout of the whole batch element by element (ReLU decisions: the kernel's own y > 0), and each rank's
    (dbeta, dgamma) against fp64 sums over that rank's shard."""
    N, C = z.shape[0], z.shape[-1]
    P = z.numel() // C
    sh = (-1, 1, 1)
    keep = (y > 0).permute(0, 3, 1, 2)
    gm = dy.double().permute(0, 3, 1, 2) * keep
    assert torch.equal(gout, dy * (y > 0)), f"{tag}: gout is not the ReLU-masked dy"
    xk = (z.double().permute(0, 3, 1, 2) - mean.double().view(sh)) * invstd.double().view(sh)
    gx = gm * xk
    n = N // R
    for r in range(R):
        part = slice(r * n, (r + 1) * n)
        check_sum(f"{tag} rank {r} dbeta", sums[r, 0], gm[part].sum((0, 2, 3)), gm[part].abs().sum((0, 2, 3)))
        check_sum(f"{tag} rank {r} dgamma", sums[r, 1], gx[part].sum((0, 2, 3)), gx[part].abs().sum((0, 2, 3)))
    ref_db, ref_dg = gm.sum((0, 2, 3)), gx.sum((0, 2, 3))
    a = (gamma.double() * invstd.double()).view(sh)
    ref_dz = a * (gm - (ref_db / P).view(sh) - xk * (ref_dg / P).view(sh))
    A_dz = a.abs() * (gm.abs() + (ref_db.abs() / P).view(sh) + xk.abs() * (ref_dg.abs() / P).view(sh))
    check_bf16(f"{tag} dz", dz, ref_dz, A_dz)


# N, H, W, C, R emulated ranks, least grid-stride passes per block of both column-sum kernels (0: a regime of idle blocks).
# Observed err / bound: y, dz <= 0.992 (bf16 rounding); per-rank dgamma <= 0.031, dbeta <= 0.0038.  Statistics at every
# shift and R: mean err <= 4.9e-6 std, var rel <= 8.0e-7, invstd rel <= 4.0e-7 (all-reduced raw fp32 sums, the earlier
# design: var rel 1.2e-2 at 64 std with R = 1, 3.5e-4..8.6e-4 with R = 2..8).
SYNC_BN_CASES = [
    (16, 512, 512, 64, 1, 2),
    (16, 512, 512, 64, 2, 2),
    (16, 512, 512, 64, 8, 2),
    (12, 256, 256, 256, 3, 2),
    (8, 32, 32, 2048, 2, 2),          # one row per block and pass: the forward's last block takes exactly two passes
    (8, 3, 5, 2560, 8, 0),            # 15 rows per rank: 281 of 296 blocks idle; C/8 = 320, a second channel chunk of 64
]


@pytest.mark.parametrize("N,H,W,C,R,passes", SYNC_BN_CASES)
def test_sync_batchnorm_emulated_ranks(b2u, cuda_device, N, H, W, C, R, passes):
    """SyncBatchNorm's four entry points on R ranks emulated on one GPU (shards of whole images), stitched together,
    against fp64 BatchNorm over the whole batch: the statistics to the one-GPU bounds at channel means up to 64 standard
    deviations, bit-identical on every rank; the running statistics with the unbiased factor of the global row count;
    y with and without a residual; dz and gout element by element with the ReLU mask read from y and recomputed from z;
    each rank's local dgamma / dbeta."""
    ops, dev = b2u.ops, cuda_device
    assert N % R == 0
    P, Pr = N * H * W, N // R * H * W
    if passes:
        assert min(_colsum_passes(Pr, C, 8), _colsum_passes(Pr, C, 4)) >= passes
    else:
        assert Pr < BN_BLOCKS and C // 8 > 256 and (C // 8) % 256 != 0
    z, ratio = _bn_data(dev, N, H, W, C, 11)
    g = _gen(dev, 12)
    sign = torch.where(torch.arange(C, device=dev) % 3 == 2, -1.0, 1.0)
    gamma = (1 + 0.2 * torch.randn((C,), generator=g, device=dev)) * sign
    beta = 0.1 * torch.randn((C,), generator=g, device=dev)
    rm0, rv0 = 0.1 * torch.randn((C,), generator=g, device=dev), torch.rand((C,), generator=g, device=dev) + 0.5
    residual = _bf((N, H, W, C), g, dev)
    dy = _bf((N, H, W, C), g, dev)
    tag = f"sync bn {N}x{H}x{W}x{C} R={R}"
    y, ranks = _sync_bn_fwd(ops, z, R, gamma, beta, rm0, rv0)
    mean, invstd, rm, rv = ranks[0]
    for r, t in enumerate(ranks[1:], 1):
        for a, b, what in zip(t, ranks[0], ("save_mean", "save_invstd", "running_mean", "running_var")):
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"{tag}: {what} of rank {r} differs from rank 0"
    m_ref, v_ref = _bn_stat_errors(tag, mean, invstd, z, ratio)
    want_rv = 0.9 * rv0.double() + 0.1 * v_ref * P / (P - 1)
    assert ((rv.double() - want_rv).abs() / want_rv).max().item() <= 2e-6
    assert torch.allclose(rm.double(), 0.9 * rm0.double() + 0.1 * m_ref, rtol=1e-6, atol=1e-6 * v_ref.sqrt().max().item())
    zd = z.double().permute(0, 3, 1, 2)
    ref_y, A_y = _bn_fwd_ref(zd, m_ref, (v_ref + 1e-5).rsqrt(), gamma, beta)
    check_bf16(f"{tag} y", y, ref_y, A_y)
    del ref_y, A_y
    y_res, ranks_res = _sync_bn_fwd(ops, z, R, gamma, beta, rm0, rv0, residual=residual)
    assert torch.equal(ranks_res[0][1], invstd)
    ref_y, A_y = _bn_fwd_ref(zd, m_ref, (v_ref + 1e-5).rsqrt(), gamma, beta, residual)
    check_bf16(f"{tag} y residual", y_res, ref_y, A_y)
    del ref_y, A_y, zd
    # backward: ReLU mask recomputed from z (no residual), then read from y (residual added before the ReLU)
    dz, gout, sums = _sync_bn_bwd(ops, dy, None, z, R, gamma, beta, mean, invstd)
    _bn_bwd_check(f"{tag} bwd", dz, gout, sums, dy, y, z, R, gamma, mean, invstd)
    dz, gout, sums = _sync_bn_bwd(ops, dy, y_res, z, R, gamma, beta, mean, invstd)
    _bn_bwd_check(f"{tag} bwd residual", dz, gout, sums, dy, y_res, z, R, gamma, mean, invstd)


# ------------------------------------------------------------------------------------------------- eval-mode BatchNorm
# Observed err / bound: y, dz <= 0.992 (bf16 rounding); dgamma <= 0.0025, dbeta <= 8e-4.
@pytest.mark.parametrize("N,H,W,C", BN_CASES)
def test_batchnorm_eval_backward_at_scale(b2u, cuda_device, N, H, W, C):
    """model.eval() + backward: y = relu(bn(z) [+ residual]) from the running statistics, then ops.bn_bwd_eval against
    dz = gamma / sqrt(rv + eps) g (no batch-mean terms), dbeta = sum g, dgamma = sum g (z - rm) / sqrt(rv + eps), with g
    the ReLU-masked dy; every fifth channel has rv = 1e-4, where eps moves invstd by 5 %."""
    ops, dev = b2u.ops, cuda_device
    z, _ = _bn_data(dev, N, H, W, C, 13)
    g = _gen(dev, 14)
    m_ref, v_ref = _bn_ref_stats(z)
    gamma = (1 + 0.2 * torch.randn((C,), generator=g, device=dev)) * torch.where(torch.arange(C, device=dev) % 3 == 2, -1.0, 1.0)
    beta = 0.1 * torch.randn((C,), generator=g, device=dev)
    rm = (m_ref + 0.2 * v_ref.sqrt() * torch.randn((C,), generator=g, device=dev, dtype=F64)).float()
    rv = (v_ref * (torch.rand((C,), generator=g, device=dev, dtype=F64) + 0.5)).float()
    rv[::5] = 1e-4
    residual = _bf((N, H, W, C), g, dev)
    dy = _bf((N, H, W, C), g, dev)
    sh = (-1, 1, 1)
    is_ref = (rv.double() + 1e-5).rsqrt()
    for res in (None, residual):
        tag = f"bn eval bwd {N}x{H}x{W}x{C} residual={res is not None}"
        y = ops.bn_fwd_eval(z, gamma, beta, rm, rv, relu=True, residual=res)
        ref_y, A_y = _bn_fwd_ref(z.double().permute(0, 3, 1, 2), rm, is_ref, gamma, beta, res)
        check_bf16(tag + " y", y, ref_y, A_y)
        del ref_y, A_y
        gout = torch.full_like(z, float("nan")) if res is not None else None
        dz, dgam, dbet = ops.bn_bwd_eval(dy, y, z, gamma, beta, rm, rv, relu=True, gout=gout)
        gm = dy.double().permute(0, 3, 1, 2) * (y > 0).permute(0, 3, 1, 2)
        if gout is not None:
            assert torch.equal(gout, dy * (y > 0)), f"{tag}: gout is not the ReLU-masked dy"
        a = (gamma.double() * is_ref).view(sh)
        check_bf16(tag + " dz", dz, a * gm, a.abs() * gm.abs())
        gx = gm * (z.double().permute(0, 3, 1, 2) - rm.double().view(sh)) * is_ref.view(sh)
        check_sum(tag + " dbeta", dbet, gm.sum((0, 2, 3)), gm.abs().sum((0, 2, 3)))
        check_sum(tag + " dgamma", dgam, gx.sum((0, 2, 3)), gx.abs().sum((0, 2, 3)))
        del gm, gx


def test_bn_fold_against_float64(b2u, cuda_device):
    """b2u_bn_fold (eval BatchNorm folded into the conv before it): scale = gamma / sqrt(rv + eps) and
    bias = (conv_bias - rm) scale + beta to fp32 rounding, with gamma of both signs, rv from 1e-6 (eps dominates) to 10, and
    each of gamma / beta / conv_bias absent.  Observed err / bound <= 0.52."""
    ops, dev = b2u.ops, cuda_device
    C = 1000                                  # not a multiple of the 128-thread block
    g = _gen(dev, 15)
    gamma = torch.randn((C,), generator=g, device=dev)
    beta = torch.randn((C,), generator=g, device=dev)
    rm = 3 * torch.randn((C,), generator=g, device=dev)
    rv = 10 ** (7 * torch.rand((C,), generator=g, device=dev) - 6)
    rv[:4] = torch.tensor([1e-6, 2e-6, 1e-5, 1e-4])
    cb = torch.randn((C,), generator=g, device=dev)
    assert (gamma < 0).any() and (rv < 1e-5).sum() >= 20
    for drop in (None, "gamma", "beta", "conv_bias"):
        ga, bt, b0 = (None if drop == "gamma" else gamma), (None if drop == "beta" else beta), (None if drop == "conv_bias" else cb)
        s, b = ops.bn_fold(ga, bt, rm, rv, b0)
        gd = ga.double() if ga is not None else torch.ones(C, dtype=F64, device=dev)
        bd = bt.double() if bt is not None else torch.zeros(C, dtype=F64, device=dev)
        cd = b0.double() if b0 is not None else torch.zeros(C, dtype=F64, device=dev)
        ref_s = gd / (rv.double() + 1e-5).sqrt()
        ref_b = (cd - rm.double()) * ref_s + bd
        e_s = ((s.double() - ref_s).abs() / (2.0 ** -21 * ref_s.abs() + 1e-300)).max().item()
        e_b = ((b.double() - ref_b).abs() / (2.0 ** -21 * ((cd - rm.double()).abs() * ref_s.abs() + bd.abs()) + 1e-300)).max().item()
        _note(f"bn_fold without {drop} scale", e_s)
        _note(f"bn_fold without {drop} bias", e_b)
        assert e_s <= 1.0 and e_b <= 1.0, drop


# ------------------------------------------------------------------------------------------------- grid-stride reductions
def test_grid_stride_reductions_at_scale(b2u, cuda_device):
    """bias_grad, the depthwise 3x3 weight gradient and spatial_reduce over 4.19 M pixels of 64 channels."""
    ops, dev = b2u.ops, cuda_device
    N, H, W, C = 16, 512, 512, 64
    g = _gen(dev, 8)
    dz = _bf((N, H, W, C), g, dev)
    dz[..., ::2] = (dz[..., ::2].float() + 3.0).to(BF)      # channels with a large mean: no cancellation to hide behind
    zd = dz.double()
    check_sum("bias_grad", ops.bias_grad(dz), zd.sum((0, 1, 2)), zd.abs().sum((0, 1, 2)))
    pooled = ops.spatial_reduce(dz, scale=1.0)
    check_sum("spatial_reduce", pooled, zd.sum((1, 2)), zd.abs().sum((1, 2)))
    x = _bf((N, H, W, C), g, dev)
    pooled2 = ops.spatial_reduce(dz, x, scale=0.5)
    prod = zd * x.double()
    check_sum("spatial_reduce product", pooled2, 0.5 * prod.sum((1, 2)), 0.5 * prod.abs().sum((1, 2)))
    del prod, pooled2
    dw, db = ops.dwconv3x3_wgrad(x, dz)
    xp = torch.zeros((N, H + 2, W + 2, C), dtype=F64, device=dev)
    xp[:, 1:-1, 1:-1] = x.double()
    ref = torch.empty((C, 9), dtype=F64, device=dev)
    A = torch.empty((C, 9), dtype=F64, device=dev)
    for t in range(9):
        tap = xp[:, t // 3:t // 3 + H, t % 3:t % 3 + W] * zd
        ref[:, t] = tap.sum((0, 1, 2))
        A[:, t] = tap.abs().sum((0, 1, 2))
    check_sum("dwconv3x3_wgrad dw", dw.view(C, 9), ref, A)
    check_sum("dwconv3x3_wgrad db", db, zd.sum((0, 1, 2)), zd.abs().sum((0, 1, 2)))


# ------------------------------------------------------------------------------------------------- head and losses
@pytest.mark.parametrize("C", [21, 150])
def test_head_and_losses_at_scale(b2u, cuda_device, C):
    """1x1 classifier (SIMT and tensor-core forward, backward dx / dw / db) and the four losses with their gradients at
    8 x 512 x 512, ~5 % ignored pixels: the kLossBlocks and head-wgrad grid-stride loops, fp64 partials."""
    ops, dev = b2u.ops, cuda_device
    N, H, W = 8, 512, 512
    g = _gen(dev, 9 + C)
    x = _bf((N, H, W, 64), g, dev).relu()
    w = torch.randn((C, 64), generator=g, device=dev) / 8
    b = torch.randn((C,), generator=g, device=dev)
    xd = x.double().permute(0, 3, 1, 2)
    ref = torch.einsum("nkhw,ck->nchw", xd, w.double()) + b.double().view(1, -1, 1, 1)
    A = torch.einsum("nkhw,ck->nchw", xd.abs(), w.double().abs()) + b.double().abs().view(1, -1, 1, 1)
    logits = ops.head_fwd(x, w, b)
    check_sum(f"head fwd C={C}", logits, ref, A)
    logits_tc = ops.head_fwd_tc(x, ops.pack_head_fprop(w), b, C)
    check_sum(f"head fwd tc C={C}", logits_tc, ref, A, c=2.0 ** -15)      # w enters as a two-term bf16 split
    del A
    png = torch.randint(0, C, (N, H, W), generator=g, device=dev)
    png[torch.rand((N, H, W), generator=g, device=dev) < 0.05] = C
    cw = torch.rand((C,), generator=g, device=dev) + 0.5
    oh = O.one_hot(png, C) if C <= 32 else None
    fin = ops.loss_fwd(logits, target=png, onehot=oh, cls_w=cw)
    lr = logits.double().requires_grad_(True)
    ohd = O.one_hot(png, C).double() if oh is None else oh.double()
    ce, fo = O.ce_loss(lr, png, cw.double(), C), O.focal_loss(lr, png, cw.double(), C)
    di, fs = O.dice_loss(lr, ohd), O.f_score(lr.detach(), ohd)
    del ohd
    for name, got, want in zip(("ce", "focal", "dice", "f_score"), fin[:4].tolist(), (ce, fo, di, fs)):
        assert abs(got - want.item()) <= 2e-5 * max(abs(want.item()), 1e-3), f"{name} C={C}: {got} vs {want.item()}"
    for gs, loss in (([1, 0, 1], ce + di), ([0, 1, 0], fo)):
        gl, = torch.autograd.grad(loss, lr, retain_graph=True)
        dl = ops.loss_bwd(logits, fin, torch.tensor(gs, dtype=torch.float32, device=dev), target=png, onehot=oh, cls_w=cw)
        scale = gl.abs().mean().item()
        err = ((dl.double() - gl).abs() / (1e-4 * (gl.abs() + scale))).max().item()
        _note(f"loss bwd {gs} C={C}", err)
        assert err <= 1.0
    gl = gl.float().contiguous()
    dx, dw, dbias = ops.head_bwd(gl, x, w)
    gd = gl.double()
    ref_dw = torch.einsum("nchw,nkhw->ck", gd, xd)
    A_dw = torch.einsum("nchw,nkhw->ck", gd.abs(), xd)
    check_sum(f"head bwd dw C={C}", dw.view(C, 64), ref_dw, A_dw)
    check_sum(f"head bwd db C={C}", dbias, gd.sum((0, 2, 3)), gd.abs().sum((0, 2, 3)))
    ref_dx = torch.einsum("nchw,ck->nkhw", gd, w.double()) * (xd > 0)
    A_dx = torch.einsum("nchw,ck->nkhw", gd.abs(), w.double().abs())
    check_bf16(f"head bwd dx C={C}", dx, ref_dx, A_dx)


# ------------------------------------------------------------------------------------------------- tile scheduler
def _sched_inputs(b2u, dev):
    g = _gen(dev, 10)
    N, H, W, C = 8, 128, 128, 128
    x = _bf((N, H, W, C), g, dev)
    w = torch.randn((C, C, 3, 3), generator=g, device=dev) / (C * 9) ** 0.5
    b = torch.randn((C,), generator=g, device=dev)
    dz = _bf((N, H, W, C), g, dev)
    mask = _bf((N, H, W, C), g, dev)
    return dict(x=x, w=w, b=b, dz=dz, mask=mask)


def _sched_outputs(ops, t):
    """Multi-tile launches on the dynamic scheduler: forward + ReLU, forward with statistics, masked dgrad, two-output dgrad."""
    N, H, W, C = t["x"].shape
    wf, wd = ops.pack_weights(t["w"])
    rows = ops.conv_stat_rows(N, H, W, C)
    st = torch.full((rows * 2 * C,), float("nan"), device=t["x"].device)
    drows = ops.conv_dgrad_stat_rows(N, H, W, C, masked=True)
    dst = torch.full((drows * 2 * C,), float("nan"), device=t["x"].device)
    out = dict(y=ops.conv_fprop(t["x"], wf, t["b"], C, relu=True),
               z=ops.conv_fprop(t["x"], wf, t["b"], C, relu=False, stats=st), st=st,
               dm=ops.conv_dgrad(t["dz"], wd, C, mask=t["mask"], stats=dst), dst=dst)
    out["d0"], out["d1"] = ops.conv_dgrad(t["dz"], wd, 64, C1=C - 64)
    return out


_STATIC_CHILD = """
import sys, torch
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[2])
from unet_pytorch_b200 import ops
from test_kernels_at_scale_gpu import _sched_outputs
torch.backends.cudnn.allow_tf32 = False
t = torch.load(sys.argv[3])
torch.save({k: v.cpu() for k, v in _sched_outputs(ops, {k: v.cuda() for k, v in t.items()}).items()}, sys.argv[4])
"""


def test_static_and_dynamic_tile_order_bitwise(b2u, cuda_device, tmp_path):
    """Each tile is computed whole by one CTA, so the order in which CTAs take tiles must not change a bit: the dynamic
    scheduler here against B2U_STATIC_TILES=1 (static round robin) in a child process, statistics rows included."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    t = _sched_inputs(b2u, dev)
    N, H, W, C = t["x"].shape
    assert ops.conv_stat_rows(N, H, W, C) >= 3 * sms and ops.conv_dgrad_stat_rows(N, H, W, C, masked=True) >= 3 * sms
    dyn = _sched_outputs(ops, t)
    torch.cuda.synchronize()
    src, dst = tmp_path / "in.pt", tmp_path / "out.pt"
    torch.save({k: v.cpu() for k, v in t.items()}, src)
    script = tmp_path / "child.py"
    script.write_text(_STATIC_CHILD)
    env = dict(os.environ, B2U_STATIC_TILES="1")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [str(script), ROOT, os.path.dirname(__file__), str(src), str(dst)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    stat = torch.load(dst)
    for k, v in dyn.items():
        a, s = v.cpu(), stat[k]
        same = torch.equal(a.view(torch.int16), s.view(torch.int16)) if a.dtype == BF else torch.equal(a.view(torch.int32), s.view(torch.int32))
        print(f"[static vs dynamic] {k}: {'bitwise equal' if same else 'DIFFERENT'}")
        assert same, f"{k}: static and dynamic tile order differ"


def test_scheduler_slot_ring_reuse(b2u, cuda_device):
    """520 = 2 x 256 scheduler slots + 8 back-to-back multi-tile launches on one stream, alternating forward-with-statistics
    and masked dgrad: every slot is re-armed by the last CTA of its previous launch, so each launch reproduces the first."""
    ops, dev, sms = b2u.ops, cuda_device, _sms(b2u)
    t = _sched_inputs(b2u, dev)
    N, H, W, C = t["x"].shape
    wf, wd = ops.pack_weights(t["w"])
    rows, drows = ops.conv_stat_rows(N, H, W, C), ops.conv_dgrad_stat_rows(N, H, W, C, masked=True)
    assert rows >= 3 * sms and drows >= 3 * sms
    st, dst = torch.empty((rows * 2 * C,), device=dev), torch.empty((drows * 2 * C,), device=dev)
    z, d = torch.empty_like(t["x"]), torch.empty_like(t["x"])
    bad = torch.zeros((), dtype=torch.int64, device=dev)
    first = None
    for i in range(260):
        ops.conv_fprop(t["x"], wf, t["b"], C, relu=False, stats=st, out=z)
        ops.conv_dgrad(t["dz"], wd, C, mask=t["mask"], stats=dst, out0=d)
        if first is None:
            first = [v.clone() for v in (z, st, d, dst)]
            continue
        for a, f in zip((z, st, d, dst), first):
            bad += (a.view(torch.int16) != f.view(torch.int16)).any() if a.dtype == BF else (a.view(torch.int32) != f.view(torch.int32)).any()
    assert bad.item() == 0, f"{bad.item()} launches differ from the first"
