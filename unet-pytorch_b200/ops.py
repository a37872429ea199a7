"""Tensor-level wrappers over the C ABI (include/b2u.h).

Activations are NHWC bf16 CUDA tensors ([N, H, W, C], contiguous); parameters and logits keep the reference's
fp32 OIHW / NCHW layouts.  Every function launches on torch's current stream and allocates its outputs and
workspaces with torch's caching allocator; none of them has a CPU or PyTorch fallback.
"""
import ctypes
import struct

import torch

from . import _lib
from ._lib import check, lib, ptr, stream_ptr

# dtype of every activation / gradient / packed-operand tensor ("void*" in include/b2u.h): bf16 on the product path, fp32
# when the process runs the fp32 validation build (csrc/validation_fp32.cu)
ACT = torch.float32 if _lib.validation_fp32() else torch.bfloat16


def act_dtype():
    return ACT


def set_validation_fp32(on):
    """Switches the process between the product library (bf16 NHWC tensors, tcgen05 kernels) and the fp32 validation build
    of the same ABI (BASELINE.json: rel-L2 <= 1e-5 against the fp32 reference).  Build engines / modules after the call."""
    global ACT
    _lib.set_validation_fp32(on)
    ACT = torch.float32 if on else torch.bfloat16


def _req(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (the hot path has no CPU fallback)")
    if t.dtype != dtype:
        raise ValueError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous tensor")


class KernelTimer:
    """CUDA-event timer around individual launches of the tensor-core kernels (bench.py's roofline leg).
    Events are recorded on the launching (current) stream; read() synchronises once at the end."""

    def __init__(self):
        self.records = {}       # tag -> [(start, end, flops)]

    def add(self, tag, start, end, flops):
        self.records.setdefault(tag, []).append((start, end, flops))

    def read(self):
        torch.cuda.synchronize()
        out = {}
        for tag, recs in self.records.items():
            ms = sum(a.elapsed_time(b) for a, b, _ in recs)
            out[tag] = {"launches": len(recs), "ms": ms, "flops": float(sum(f for _, _, f in recs))}
        return out


_TIMER = None


def set_timer(timer):
    global _TIMER
    _TIMER = timer


def timing_active():
    """True while a KernelTimer brackets individual launches with events: the engines then keep every launch on one stream,
    so that an event pair measures that kernel alone."""
    return _TIMER is not None


class _timed:
    def __init__(self, tag, flops):
        self.tag, self.flops = tag, flops

    def __enter__(self):
        if _TIMER is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if _TIMER is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            _TIMER.add(self.tag, self.a, b, self.flops)


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


# ---------------------------------------------------------------------------------------------- layout
def im2col_first(x_nchw):
    _req(x_nchw, torch.float32, "x")
    N, C, H, W = x_nchw.shape
    col = torch.empty((N, H, W, 64), dtype=ACT, device=x_nchw.device)
    check(lib().b2u_im2col_first(ptr(x_nchw), ptr(col), N, C, H, W, stream_ptr()))
    return col


def pack_weights(w, want_dgrad=True, wf=None, wd=None):
    """OIHW fp32 -> (wf [Cout, taps*Cin], wd [Cin, taps*Cout]) bf16."""
    _req(w, torch.float32, "weight")
    Cout, Cin, kh, kw = w.shape
    taps = kh * kw
    if wf is None:
        wf = torch.empty((Cout, taps * Cin), dtype=ACT, device=w.device)
    if want_dgrad and wd is None:
        wd = torch.empty((Cin, taps * Cout), dtype=ACT, device=w.device)
    check(lib().b2u_pack_weights(ptr(w), ptr(wf), ptr(wd) if want_dgrad else None, Cout, Cin, taps, stream_ptr()))
    return wf, (wd if want_dgrad else None)


def pack_weights_first(w, wf=None):
    _req(w, torch.float32, "weight")
    Cout, Cin, kh, kw = w.shape
    assert kh == 3 and kw == 3
    if wf is None:
        wf = torch.empty((Cout, 64), dtype=ACT, device=w.device)
    check(lib().b2u_pack_weights_first(ptr(w), ptr(wf), Cout, Cin, stream_ptr()))
    return wf


def nhwc_to_nchw_f32(x):
    _req(x, ACT, "x")
    N, H, W, C = x.shape
    y = torch.empty((N, C, H, W), dtype=torch.float32, device=x.device)
    check(lib().b2u_nhwc_bf16_to_nchw_f32(ptr(x), ptr(y), N, C, H, W, stream_ptr()))
    return y


def nchw_to_nhwc_bf16(x):
    _req(x, torch.float32, "x")
    N, C, H, W = x.shape
    y = torch.empty((N, H, W, C), dtype=ACT, device=x.device)
    check(lib().b2u_nchw_f32_to_nhwc_bf16(ptr(x), ptr(y), N, C, H, W, stream_ptr()))
    return y


def u8hwc_to_nchw_f32(x, scale=1.0 / 255.0, out=None):
    """uint8 [N, H, W, C] image batch -> fp32 [N, C, H, W] * scale (the dataloader's preprocess_input + transpose)."""
    _req(x, torch.uint8, "x")
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty((N, C, H, W), dtype=torch.float32, device=x.device)
    check(lib().b2u_u8hwc_to_nchw_f32(ptr(x), ptr(out), N, H, W, C, scale, stream_ptr()))
    return out


def u8_to_i64(x, out=None):
    _req(x, torch.uint8, "x")
    if out is None:
        out = torch.empty(x.shape, dtype=torch.int64, device=x.device)
    check(lib().b2u_u8_to_i64(ptr(x), ptr(out), x.numel(), stream_ptr()))
    return out


def nchw_to_nhwc_bf16_padded(x, cpad, out=None):
    _req(x, torch.float32, "x")
    N, C, H, W = x.shape
    if out is None:
        out = torch.empty((N, H, W, cpad), dtype=ACT, device=x.device)
    check(lib().b2u_nchw_f32_to_nhwc_bf16_padded(ptr(x), ptr(out), N, C, H, W, cpad, stream_ptr()))
    return out


# ---------------------------------------------------------------------------------------------- gradient wrt the image
def _image_grad_out(out, shape, device):
    if out is None:
        return torch.empty(shape, dtype=torch.float32, device=device)
    _req(out, torch.float32, "dx")
    if tuple(out.shape) != tuple(shape):
        raise ValueError(f"dx: expected shape {tuple(shape)}, got {tuple(out.shape)}")
    return out


def first_conv_dgrad_input(dz, w, out=None):
    """Gradient wrt the NCHW fp32 image of the first 3x3 conv (the one over im2col_first rows): dz [N,H,W,Cz] (gradient wrt
    its output), w fp32 OIHW [Cout, Cin, 3, 3] -> dx [N, Cin, H, W] fp32."""
    N, H, W, Cz = dz.shape
    Cout, Cin, kh, kw = w.shape
    if (kh, kw) != (3, 3):
        raise ValueError("first_conv_dgrad_input: expected a 3x3 weight")
    _req(dz, ACT, "dz"); _req(w, torch.float32, "weight")
    out = _image_grad_out(out, (N, Cin, H, W), dz.device)
    check(lib().b2u_first_conv_dgrad_input(ptr(dz), Cz, ptr(w), ptr(out), N, Cin, H, W, Cout, stream_ptr()))
    return out


def stem_dgrad_input(dz, w, H, W, out=None):
    """Gradient wrt the H x W NCHW fp32 image of the 7x7 stride-2 stem: dz [N, ceil(H/2), ceil(W/2), Cz], w fp32
    [Cout, Cin, 7, 7] -> dx [N, Cin, H, W] fp32."""
    N, Ho, Wo, Cz = dz.shape
    Cout, Cin, kh, kw = w.shape
    if (kh, kw) != (7, 7) or (Ho, Wo) != ((H + 1) // 2, (W + 1) // 2):
        raise ValueError("stem_dgrad_input: expected a 7x7 weight and dz at half the image size")
    _req(dz, ACT, "dz"); _req(w, torch.float32, "weight")
    out = _image_grad_out(out, (N, Cin, H, W), dz.device)
    check(lib().b2u_stem_dgrad_input(ptr(dz), Cz, ptr(w), ptr(out), N, Cin, H, W, Cout, stream_ptr()))
    return out


def nhwc_padded_to_nchw_f32(x, C, out=None):
    """Channels [0, C) of NHWC x [N,H,W,Cpad] -> NCHW fp32 [N, C, H, W] (the gradient wrt an image that entered through
    nchw_to_nhwc_bf16_padded)."""
    N, H, W, Cpad = x.shape
    if not 0 < C <= Cpad:
        raise ValueError(f"nhwc_padded_to_nchw_f32: C = {C} must be in [1, {Cpad}]")
    _req(x, ACT, "x")
    out = _image_grad_out(out, (N, C, H, W), x.device)
    check(lib().b2u_nhwc_bf16_padded_to_nchw_f32(ptr(x), ptr(out), N, C, H, W, Cpad, stream_ptr()))
    return out


# ---------------------------------------------------------------------------------------------- convs
def conv_fprop(x0, wf, bias, Cout, taps=9, relu=True, x1=None, out=None, bn=0, stats=None):
    """stats: optional fp32 buffer [>= conv_stat_rows(...)][2][Cout]; the conv then also writes the per-tile sums of z and
    z^2 of its output (BatchNorm statistics, consumed by bn_fwd_train(stats=...))."""
    _req(x0, ACT, "x0"); _req(x1, ACT, "x1"); _req(wf, ACT, "wf"); _req(bias, torch.float32, "bias")
    N, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else x1.shape[3]
    if out is None:
        out = torch.empty((N, H, W, Cout), dtype=ACT, device=x0.device)
    with _timed(f"conv_igemm|fprop|{N}x{H}x{W}|{C0}+{C1}->{Cout}|t{taps}", 2.0 * N * H * W * Cout * (C0 + C1) * taps):
        if stats is None:
            check(lib().b2u_conv_fprop(ptr(x0), C0, ptr(x1), C1, ptr(wf), ptr(bias), ptr(out), N, H, W, Cout, taps,
                                       1 if relu else 0, bn, stream_ptr()))
        else:
            _req(stats, torch.float32, "stats")
            check(lib().b2u_conv_fprop_stats(ptr(x0), C0, ptr(x1), C1, ptr(wf), ptr(bias), ptr(out), N, H, W, Cout, taps,
                                             1 if relu else 0, bn, ptr(stats), stats.numel() // (2 * Cout), stream_ptr()))
    return out


def conv_fprop_scaled(x0, wf, scale, bias, Cout, taps=9, relu=True, x1=None, out=None, bn=0):
    """y = [relu](conv(x) * scale[c] + bias[c]): conv + eval-mode BatchNorm (+ReLU) in one kernel (scale/bias from bn_fold)."""
    _req(x0, ACT, "x0"); _req(x1, ACT, "x1"); _req(wf, ACT, "wf"); _req(bias, torch.float32, "bias"); _req(scale, torch.float32, "scale")
    N, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else x1.shape[3]
    if out is None:
        out = torch.empty((N, H, W, Cout), dtype=ACT, device=x0.device)
    check(lib().b2u_conv_fprop_scaled(ptr(x0), C0, ptr(x1), C1, ptr(wf), ptr(scale), ptr(bias), ptr(out), N, H, W, Cout, taps,
                                      1 if relu else 0, bn, stream_ptr()))
    return out


def decoder_conv_fprop(skip, low, wf, bias, Cout, relu=True, out=None, up_out=None, scale=None, stats=None, bn=0):
    """conv3x3(cat([skip, upsample2x(low)])) with the bilinear up-sampling done by the conv's producer warps (nets/unet.py:16-18).
    low: [N, H/2, W/2, C1].  up_out (optional [N,H,W,C1]): by-product copy of the up-sampled tensor for the weight gradient.
    scale: folded eval-mode BatchNorm; stats: per-tile BatchNorm sums as in conv_fprop."""
    _req(skip, ACT, "skip"); _req(low, ACT, "low"); _req(wf, ACT, "wf"); _req(bias, torch.float32, "bias")
    _req(scale, torch.float32, "scale"); _req(stats, torch.float32, "stats"); _req(up_out, ACT, "up_out")
    N, H, W, C0 = skip.shape
    Nl, HL, WL, C1 = low.shape
    if Nl != N or 2 * HL != H or 2 * WL != W:
        raise ValueError(f"decoder_conv_fprop: low {tuple(low.shape)} is not half the resolution of skip {tuple(skip.shape)}")
    if up_out is not None and tuple(up_out.shape) != (N, H, W, C1):
        raise ValueError("decoder_conv_fprop: up_out must be [N, H, W, C1]")
    if out is None:
        out = torch.empty((N, H, W, Cout), dtype=ACT, device=skip.device)
    with _timed(f"conv_igemm|fprop|{N}x{H}x{W}|{C0}+{C1}->{Cout}|t9", 2.0 * N * H * W * Cout * (C0 + C1) * 9):
        check(lib().b2u_decoder_conv_fprop(ptr(skip), C0, ptr(low), C1, ptr(wf), ptr(scale), ptr(bias), ptr(out), ptr(up_out),
                                           N, H, W, Cout, 1 if relu else 0, bn, ptr(stats),
                                           0 if stats is None else stats.numel() // (2 * Cout), stream_ptr()))
    return out


def bn_fold(gamma, beta, running_mean, running_var, conv_bias, eps=1e-5, scale=None, bias=None):
    C = running_mean.numel()
    if scale is None:
        scale = torch.empty((C,), dtype=torch.float32, device=running_mean.device)
    if bias is None:
        bias = torch.empty((C,), dtype=torch.float32, device=running_mean.device)
    check(lib().b2u_bn_fold(ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var), ptr(conv_bias), ptr(scale), ptr(bias), C, eps,
                            stream_ptr()))
    return scale, bias


def conv_stat_rows(N, H, W, Cout, taps=9, bn=0):
    return lib().b2u_conv_stat_rows(N, H, W, Cout, taps, bn)


def conv_dgrad(dz, wd, C0, taps=9, C1=0, mask=None, out0=None, out1=None, bn=0, stats=None):
    """stats: optional fp32 buffer of conv_dgrad_stat_rows(...) x 2 x (C0 + C1) floats; the launch then also leaves the per-tile
    column sums of the (masked) gradient it stores -- the bias gradient of the conv below, see bias_from_stats."""
    _req(dz, ACT, "dz"); _req(wd, ACT, "wd"); _req(mask, ACT, "mask"); _req(stats, torch.float32, "stats")
    N, H, W, Cz = dz.shape
    if out0 is None:
        out0 = torch.empty((N, H, W, C0), dtype=ACT, device=dz.device)
    if C1 > 0 and out1 is None:
        out1 = torch.empty((N, H, W, C1), dtype=ACT, device=dz.device)
    with _timed(f"conv_igemm|dgrad|{N}x{H}x{W}|{Cz}->{C0}+{C1}|t{taps}", 2.0 * N * H * W * Cz * (C0 + C1) * taps):
        if stats is None:
            check(lib().b2u_conv_dgrad(ptr(dz), Cz, ptr(wd), ptr(out0), C0, ptr(out1) if C1 > 0 else None, C1, ptr(mask),
                                       N, H, W, taps, bn, stream_ptr()))
        else:
            check(lib().b2u_conv_dgrad_stats(ptr(dz), Cz, ptr(wd), ptr(out0), C0, ptr(out1) if C1 > 0 else None, C1, ptr(mask),
                                             N, H, W, taps, bn, ptr(stats), stats.numel() // (2 * (C0 + C1)), stream_ptr()))
    return (out0, out1) if C1 > 0 else out0


def conv_fprop_relu_bits(x0, wf, bias, Cout, bits, taps=9, x1=None, low=None, up_out=None, out=None, bn=0):
    """conv + bias + ReLU that also writes the ReLU decisions as a bit mask: bits int64 [N, H, W, Cout // 64], bit c % 64 of
    word c // 64 = (y > 0).  low: the decoder form (second source = upsample2x(low), see decoder_conv_fprop)."""
    _req(x0, ACT, "x0"); _req(x1, ACT, "x1"); _req(low, ACT, "low"); _req(wf, ACT, "wf"); _req(bias, torch.float32, "bias")
    _req(bits, torch.int64, "bits"); _req(up_out, ACT, "up_out")
    N, H, W, C0 = x0.shape
    C1 = x1.shape[3] if x1 is not None else (low.shape[3] if low is not None else 0)
    if tuple(bits.shape) != (N, H, W, Cout // 64):
        raise ValueError("conv_fprop_relu_bits: bits must be int64 [N, H, W, Cout // 64]")
    if out is None:
        out = torch.empty((N, H, W, Cout), dtype=ACT, device=x0.device)
    with _timed(f"conv_igemm|fprop|{N}x{H}x{W}|{C0}+{C1}->{Cout}|t{taps}", 2.0 * N * H * W * Cout * (C0 + C1) * taps):
        check(lib().b2u_conv_fprop_relu_bits(ptr(x0), C0, ptr(x1), C1, ptr(low), ptr(wf), ptr(bias), ptr(out), ptr(up_out), ptr(bits),
                                             N, H, W, Cout, taps, bn, stream_ptr()))
    return out


def conv_dgrad_bits(dz, wd, C0, bits, taps=9, out0=None, bn=0, stats=None):
    """conv_dgrad (one output) with the ReLU mask given as the bit mask conv_fprop_relu_bits wrote for the tensor that fed the
    conv; stats as in conv_dgrad (rows from conv_dgrad_stat_rows(masked=False))."""
    _req(dz, ACT, "dz"); _req(wd, ACT, "wd"); _req(bits, torch.int64, "bits"); _req(stats, torch.float32, "stats")
    N, H, W, Cz = dz.shape
    if tuple(bits.shape) != (N, H, W, C0 // 64):
        raise ValueError("conv_dgrad_bits: bits must be int64 [N, H, W, C0 // 64]")
    if out0 is None:
        out0 = torch.empty((N, H, W, C0), dtype=ACT, device=dz.device)
    with _timed(f"conv_igemm|dgrad|{N}x{H}x{W}|{Cz}->{C0}+0|t{taps}", 2.0 * N * H * W * Cz * C0 * taps):
        check(lib().b2u_conv_dgrad_bits(ptr(dz), Cz, ptr(wd), ptr(out0), C0, ptr(bits), N, H, W, taps, bn, ptr(stats),
                                        0 if stats is None else stats.numel() // (2 * C0), stream_ptr()))
    return out0


def conv_dgrad_stat_rows(N, H, W, Ctot, taps=9, bn=0, masked=False):
    return lib().b2u_conv_dgrad_stat_rows(N, H, W, Ctot, taps, bn, 1 if masked else 0)


def bias_from_stats(stats, rows, C, db=None):
    """db[c] = column sums recorded by conv_dgrad(stats=...) folded over the tiles (deterministic order)."""
    _req(stats, torch.float32, "stats")
    if db is None:
        db = torch.empty((C,), dtype=torch.float32, device=stats.device)
    check(lib().b2u_bias_from_stats(ptr(stats), rows, C, ptr(db), stream_ptr()))
    return db


def conv_wgrad(x0, dz, taps=9, x1=None, first_cin=0, dw=None, ws=None, flags=0, db=None, want_db=False):
    """Returns dw, or (dw, db) when the bias gradient is requested (db tensor given or want_db)."""
    _req(x0, ACT, "x0"); _req(x1, ACT, "x1"); _req(dz, ACT, "dz")
    N, H, W, C0 = x0.shape
    C1 = 0 if x1 is None else x1.shape[3]
    Cout = dz.shape[3]
    need = lib().b2u_conv_wgrad_workspace(N, H, W, C0 + C1, Cout, taps)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, x0.device)
    if dw is None:
        if first_cin > 0:
            dw = torch.empty((Cout, first_cin, 3, 3), dtype=torch.float32, device=x0.device)
        else:
            k = 3 if taps == 9 else 1
            dw = torch.empty((Cout, C0 + C1, k, k), dtype=torch.float32, device=x0.device)
    if want_db and db is None:
        db = torch.empty((Cout,), dtype=torch.float32, device=x0.device)
    with _timed(f"conv_wgrad|wgrad|{N}x{H}x{W}|{C0}+{C1}->{Cout}|t{taps}", 2.0 * N * H * W * Cout * (C0 + C1) * taps):
        check(lib().b2u_conv_wgrad(ptr(x0), C0, ptr(x1), C1, ptr(dz), Cout, ptr(dw), ptr(db), ptr(ws),
                                   ws.numel() * ws.element_size(), N, H, W, taps, first_cin, flags, stream_ptr()))
    return (dw, db) if db is not None else dw


def bias_grad(dz, db=None, ws=None):
    _req(dz, ACT, "dz")
    C = dz.shape[-1]
    P = dz.numel() // C
    need = lib().b2u_bias_grad_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, dz.device)
    if db is None:
        db = torch.empty((C,), dtype=torch.float32, device=dz.device)
    check(lib().b2u_bias_grad(ptr(dz), ptr(db), ptr(ws), ws.numel() * ws.element_size(), P, C, stream_ptr()))
    return db


# ---------------------------------------------------------------------------------------------- pool / upsample
def maxpool2x2(x, out=None):
    _req(x, ACT, "x")
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty((N, H // 2, W // 2, C), dtype=ACT, device=x.device)
    check(lib().b2u_maxpool2x2_fwd(ptr(x), ptr(out), N, H, W, C, stream_ptr()))
    return out


def maxpool2x2_bwd(dpool, y, dskip=None, relu_mask=True, out=None):
    _req(dpool, ACT, "dpool"); _req(y, ACT, "y"); _req(dskip, ACT, "dskip")
    N, H, W, C = y.shape
    if out is None:
        out = torch.empty_like(y)
    check(lib().b2u_maxpool2x2_bwd(ptr(dpool), ptr(dskip), ptr(y), ptr(out), N, H, W, C, 1 if relu_mask else 0,
                                   stream_ptr()))
    return out


def upsample2x(x, out=None):
    _req(x, ACT, "x")
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty((N, 2 * H, 2 * W, C), dtype=ACT, device=x.device)
    check(lib().b2u_upsample2x_fwd(ptr(x), ptr(out), N, H, W, C, stream_ptr()))
    return out


def upsample2x_bwd(dup, ylow=None, out=None):
    _req(dup, ACT, "dup"); _req(ylow, ACT, "ylow")
    N, H2, W2, C = dup.shape
    H, W = H2 // 2, W2 // 2
    if out is None:
        out = torch.empty((N, H, W, C), dtype=ACT, device=dup.device)
    check(lib().b2u_upsample2x_bwd(ptr(dup), ptr(ylow), ptr(out), N, H, W, C, stream_ptr()))
    return out


# ---------------------------------------------------------------------------------------------- batch norm
def bn_fwd_train(z, gamma, beta, running_mean, running_var, eps=1e-5, momentum=0.1, relu=True, out=None, ws=None,
                 residual=None, stats=None, stat_rows=0, centered=False):
    """Returns (y, save_mean, save_invstd); running statistics are updated in place (torch semantics).
    stats/stat_rows: per-tile column sums written by conv_fprop(stats=...) -- skips the statistics pass over z.
    centered: z holds conv(x) + bias - running_mean (the producing conv folded the shift into its bias, so the bf16 rounding of
    z is relative to the channel's spread, not its mean); only the running-mean update needs to know."""
    rflag = (1 if relu else 0) | (2 if centered else 0)
    _req(z, ACT, "z")
    C = z.shape[-1]
    P = z.numel() // C
    need = lib().b2u_bn_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, z.device)
    if out is None:
        out = torch.empty_like(z)
    mean = torch.empty((C,), dtype=torch.float32, device=z.device)
    invstd = torch.empty((C,), dtype=torch.float32, device=z.device)
    if stats is None:
        check(lib().b2u_bn_fwd_train(ptr(z), ptr(residual), ptr(out), ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var), ptr(mean),
                                     ptr(invstd), ptr(ws), ws.numel() * ws.element_size(), P, C, eps, momentum, rflag,
                                     stream_ptr()))
    else:
        check(lib().b2u_bn_fwd_train_stats(ptr(z), ptr(residual), ptr(out), ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
                                           ptr(mean), ptr(invstd), ptr(stats), stat_rows, ptr(ws), ws.numel() * ws.element_size(), P, C,
                                           eps, momentum, rflag, stream_ptr()))
    return out, mean, invstd


def bn_fwd_train_sync(z, gamma, beta, running_mean, running_var, group, eps=1e-5, momentum=0.1, relu=True, out=None, ws=None,
                      residual=None, centered=False):
    """SyncBatchNorm forward (train.py:335-336): this rank's (mean, biased var), one all-gather of 2C floats per rank over
    `group`, apply with the combined statistics.  Every rank is assumed to hold the same number of rows (DistributedSampler
    batches)."""
    import torch.distributed as dist
    _req(z, ACT, "z")
    C = z.shape[-1]
    P = z.numel() // C
    need = lib().b2u_bn_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, z.device)
    if out is None:
        out = torch.empty_like(z)
    mine = torch.empty((2, C), dtype=torch.float32, device=z.device)
    check(lib().b2u_bn_moments(ptr(z), ptr(mine), ptr(ws), ws.numel() * ws.element_size(), P, C, stream_ptr()))
    world = dist.get_world_size(group)
    moments = torch.empty((world, 2, C), dtype=torch.float32, device=z.device)
    dist.all_gather(list(moments.unbind(0)), mine, group=group)
    mean = torch.empty((C,), dtype=torch.float32, device=z.device)
    invstd = torch.empty((C,), dtype=torch.float32, device=z.device)
    check(lib().b2u_bn_fwd_train_moments(ptr(z), ptr(residual), ptr(out), ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
                                         ptr(mean), ptr(invstd), ptr(moments), world, ptr(ws), ws.numel() * ws.element_size(), P, C,
                                         eps, momentum, (1 if relu else 0) | (2 if centered else 0), stream_ptr()))
    return out, mean, invstd


def bn_bwd_sync(dy, y, z, gamma, mean, invstd, group, relu=True, out=None, dgamma=None, dbeta=None, ws=None, gout=None, beta=None):
    """SyncBatchNorm backward: local (sum g, sum g xhat) = this rank's (dbeta, dgamma), all-reduced only for dz."""
    import torch.distributed as dist
    _req(dy, ACT, "dy"); _req(y, ACT, "y"); _req(z, ACT, "z")
    if y is None and relu and beta is None:
        raise ValueError("bn_bwd_sync: y=None needs beta to recompute the ReLU mask")
    C = z.shape[-1]
    P = z.numel() // C
    need = lib().b2u_bn_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, z.device)
    if out is None:
        out = torch.empty_like(z)
    sums = torch.empty((2, C), dtype=torch.float32, device=z.device)
    check(lib().b2u_bn_bwd_sums(ptr(dy), ptr(y), ptr(z), ptr(gamma), ptr(beta), ptr(mean), ptr(invstd), ptr(sums), ptr(ws),
                                ws.numel() * ws.element_size(), P, C, 1 if relu else 0, stream_ptr()))
    if dbeta is not None:
        dbeta.copy_(sums[0])
    if dgamma is not None:
        dgamma.copy_(sums[1])
    local = sums.clone()
    dist.all_reduce(sums, group=group)
    world = dist.get_world_size(group)
    check(lib().b2u_bn_bwd_apply_sums(ptr(dy), ptr(y), ptr(z), ptr(gamma), ptr(beta), ptr(mean), ptr(invstd), ptr(out), ptr(gout),
                                      ptr(sums), P * world, ptr(ws), ws.numel() * ws.element_size(), P, C, 1 if relu else 0,
                                      stream_ptr()))
    return out, local[1], local[0]


def bn_fwd_eval(z, gamma, beta, running_mean, running_var, eps=1e-5, relu=True, out=None, ws=None, residual=None):
    _req(z, ACT, "z")
    C = z.shape[-1]
    P = z.numel() // C
    need = lib().b2u_bn_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, z.device)
    if out is None:
        out = torch.empty_like(z)
    check(lib().b2u_bn_fwd_eval(ptr(z), ptr(residual), ptr(out), ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var), ptr(ws),
                                ws.numel() * ws.element_size(), P, C, eps, 1 if relu else 0, stream_ptr()))
    return out


def bn_bwd(dy, y, z, gamma, mean, invstd, relu=True, out=None, dgamma=None, dbeta=None, ws=None, gout=None, beta=None):
    """Returns (dz, dgamma, dbeta); gout (optional tensor) receives the ReLU-masked dy (residual-branch gradient).
    y=None (allowed when no residual was added before the ReLU; needs beta) recomputes the ReLU mask from z."""
    _req(dy, ACT, "dy"); _req(y, ACT, "y"); _req(z, ACT, "z")
    if y is None and relu and beta is None:
        raise ValueError("bn_bwd: y=None needs beta to recompute the ReLU mask")
    C = z.shape[-1]
    P = z.numel() // C
    need = lib().b2u_bn_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, z.device)
    if out is None:
        out = torch.empty_like(z)
    if dgamma is None:
        dgamma = torch.empty((C,), dtype=torch.float32, device=z.device)
    if dbeta is None:
        dbeta = torch.empty((C,), dtype=torch.float32, device=z.device)
    check(lib().b2u_bn_bwd(ptr(dy), ptr(y), ptr(z), ptr(gamma), ptr(beta), ptr(mean), ptr(invstd), ptr(out), ptr(gout), ptr(dgamma),
                           ptr(dbeta), ptr(ws), ws.numel() * ws.element_size(), P, C, 1 if relu else 0, stream_ptr()))
    return out, dgamma, dbeta


def bn_bwd_eval(dy, y, z, gamma, beta, running_mean, running_var, eps=1e-5, relu=True, out=None, dgamma=None, dbeta=None, ws=None,
                gout=None):
    """Backward of an eval-mode BatchNorm (+ReLU) -- `model.eval()` followed by `loss.backward()` (frozen-statistics
    fine-tuning): the statistics are constants, so dz = gamma / sqrt(rv + eps) * g with g = dy * (y > 0), dbeta = sum g,
    dgamma = sum g * xhat.  Runs the SyncBatchNorm pair of kernels with the batch sums set to zero (no mean terms)."""
    _req(dy, ACT, "dy"); _req(y, ACT, "y"); _req(z, ACT, "z")
    if relu and y is None:
        raise ValueError("bn_bwd_eval: the ReLU mask is taken from y")
    C = z.shape[-1]
    P = z.numel() // C
    need = lib().b2u_bn_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, z.device)
    if out is None:
        out = torch.empty_like(z)
    invstd = torch.rsqrt(running_var + eps)
    sums = torch.empty((2, C), dtype=torch.float32, device=z.device)
    check(lib().b2u_bn_bwd_sums(ptr(dy), ptr(y), ptr(z), ptr(gamma), ptr(beta), ptr(running_mean), ptr(invstd), ptr(sums), ptr(ws),
                                ws.numel() * ws.element_size(), P, C, 1 if relu else 0, stream_ptr()))
    if dbeta is not None:
        dbeta.copy_(sums[0])
    if dgamma is not None:
        dgamma.copy_(sums[1])
    local = sums.clone()
    sums.zero_()
    check(lib().b2u_bn_bwd_apply_sums(ptr(dy), ptr(y), ptr(z), ptr(gamma), ptr(beta), ptr(running_mean), ptr(invstd), ptr(out), ptr(gout),
                                      ptr(sums), P, ptr(ws), ws.numel() * ws.element_size(), P, C, 1 if relu else 0,
                                      stream_ptr()))
    return out, local[1], local[0]


# ---------------------------------------------------------------------------------------------- ResNet helpers
def im2col_stem(x_nchw, out=None):
    _req(x_nchw, torch.float32, "x")
    N, C, H, W = x_nchw.shape
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    if out is None:
        out = torch.empty((N, Ho, Wo, 192), dtype=ACT, device=x_nchw.device)
    check(lib().b2u_im2col_stem(ptr(x_nchw), ptr(out), N, C, H, W, stream_ptr()))
    return out


def pack_weights_im2col(w, kpad, wf=None):
    _req(w, torch.float32, "weight")
    Cout, Cin, kh, kw = w.shape
    if wf is None:
        wf = torch.empty((Cout, kpad), dtype=ACT, device=w.device)
    check(lib().b2u_pack_weights_im2col(ptr(w), ptr(wf), Cout, Cin, kh * kw, kpad, stream_ptr()))
    return wf


def conv_wgrad_im2col(col, dz, cin, taps, dw=None, ws=None):
    """wgrad of a conv executed as a 1x1 GEMM over im2col rows; dw: [Cout, cin, k, k] with k*k = taps."""
    _req(col, ACT, "col"); _req(dz, ACT, "dz")
    N, H, W, Kpad = col.shape
    Cout = dz.shape[3]
    need = lib().b2u_conv_wgrad_workspace(N, H, W, Kpad, Cout, 1)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, col.device)
    if dw is None:
        k = int(round(taps ** 0.5))
        dw = torch.empty((Cout, cin, k, k), dtype=torch.float32, device=col.device)
    with _timed(f"conv_wgrad|wgrad|{N}x{H}x{W}|{Kpad}+0->{Cout}|t1", 2.0 * N * H * W * Cout * Kpad):
        check(lib().b2u_conv_wgrad_im2col(ptr(col), Kpad, ptr(dz), Cout, ptr(dw), ptr(ws), ws.numel() * ws.element_size(),
                                          N, H, W, cin, taps, stream_ptr()))
    return dw


def subsample2(x, out=None):
    _req(x, ACT, "x")
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty((N, (H + 1) // 2, (W + 1) // 2, C), dtype=ACT, device=x.device)
    check(lib().b2u_subsample2(ptr(x), ptr(out), N, H, W, C, stream_ptr()))
    return out


def zero_insert2(y, H, W, out=None):
    _req(y, ACT, "y")
    N, _, _, C = y.shape
    if out is None:
        out = torch.empty((N, H, W, C), dtype=ACT, device=y.device)
    check(lib().b2u_zero_insert2(ptr(y), ptr(out), N, H, W, C, stream_ptr()))
    return out


def maxpool3x3s2(x, out=None):
    _req(x, ACT, "x")
    N, H, W, C = x.shape
    Ho, Wo = (H - 2) // 2 + 1, (W - 2) // 2 + 1
    if out is None:
        out = torch.empty((N, Ho, Wo, C), dtype=ACT, device=x.device)
    check(lib().b2u_maxpool3x3s2_fwd(ptr(x), ptr(out), N, H, W, C, stream_ptr()))
    return out


def maxpool3x3s2_bwd(dy, x, out=None):
    _req(dy, ACT, "dy"); _req(x, ACT, "x")
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    check(lib().b2u_maxpool3x3s2_bwd(ptr(dy), ptr(x), ptr(out), N, H, W, C, stream_ptr()))
    return out


def add_bf16(a, b, out=None):
    _req(a, ACT, "a"); _req(b, ACT, "b")
    if out is None:
        out = torch.empty_like(a)
    check(lib().b2u_add_bf16(ptr(a), ptr(b), ptr(out), a.numel(), stream_ptr()))
    return out


def add_relu(a, b, out=None):
    """relu(a + b), bf16 (the residual join of nets/LightWeightUnet.py:52-53)."""
    _req(a, ACT, "a"); _req(b, ACT, "b")
    if out is None:
        out = torch.empty_like(a)
    check(lib().b2u_add_relu_bf16(ptr(a), ptr(b), ptr(out), a.numel(), stream_ptr()))
    return out


def relu_bwd(dy, y, out=None):
    _req(dy, ACT, "dy"); _req(y, ACT, "y")
    if out is None:
        out = torch.empty_like(dy)
    check(lib().b2u_relu_bwd_bf16(ptr(dy), ptr(y), ptr(out), dy.numel(), stream_ptr()))
    return out


def resize_bilinear(x, size, out=None):
    """F.interpolate(x, size, mode='bilinear', align_corners=True) for fp32 NCHW."""
    _req(x, torch.float32, "x")
    N, C, Hi, Wi = x.shape
    Ho, Wo = size
    if out is None:
        out = torch.empty((N, C, Ho, Wo), dtype=torch.float32, device=x.device)
    check(lib().b2u_resize_bilinear_f32_fwd(ptr(x), ptr(out), N * C, Hi, Wi, Ho, Wo, stream_ptr()))
    return out


def resize_bilinear_bwd(dy, size_in, out=None):
    _req(dy, torch.float32, "dy")
    N, C, Ho, Wo = dy.shape
    Hi, Wi = size_in
    if out is None:
        out = torch.empty((N, C, Hi, Wi), dtype=torch.float32, device=dy.device)
    check(lib().b2u_resize_bilinear_f32_bwd(ptr(dy), ptr(out), N * C, Hi, Wi, Ho, Wo, stream_ptr()))
    return out


# ---------------------------------------------------------------------------------------------- depthwise / SE
def dwconv3x3(x, w, bias=None, flip=False, out=None):
    """w: fp32 [C, 9] (or [C,1,3,3]); flip=True is the data gradient."""
    _req(x, ACT, "x"); _req(w, torch.float32, "w")
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    check(lib().b2u_dwconv3x3_fwd(ptr(x), ptr(w), ptr(bias), ptr(out), N, H, W, C, 1 if flip else 0, stream_ptr()))
    return out


def dwconv3x3_wgrad(x, dy, dw=None, db=None, ws=None):
    _req(x, ACT, "x"); _req(dy, ACT, "dy")
    N, H, W, C = x.shape
    need = lib().b2u_dwconv3x3_wgrad_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, x.device)
    if dw is None:
        dw = torch.empty((C, 9), dtype=torch.float32, device=x.device)
    if db is None:
        db = torch.empty((C,), dtype=torch.float32, device=x.device)
    check(lib().b2u_dwconv3x3_wgrad(ptr(x), ptr(dy), ptr(dw), ptr(db), ptr(ws), ws.numel() * ws.element_size(), N, H, W, C,
                                    stream_ptr()))
    return dw, db


def spatial_reduce(a, b=None, scale=1.0, out=None, ws=None):
    """[N, C] fp32: scale * sum over H*W of a (or a*b)."""
    _req(a, ACT, "a"); _req(b, ACT, "b")
    N, H, W, C = a.shape
    need = lib().b2u_spatial_reduce_workspace_floats(N, C) * 4
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, a.device)
    if out is None:
        out = torch.empty((N, C), dtype=torch.float32, device=a.device)
    check(lib().b2u_spatial_reduce(ptr(a), ptr(b), ptr(out), ptr(ws), ws.numel() * ws.element_size(), N, H * W, C, scale,
                                   stream_ptr()))
    return out


def scale_nc(x, s, add=None, out=None):
    _req(x, ACT, "x"); _req(s, torch.float32, "s"); _req(add, torch.float32, "add")
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty_like(x)
    check(lib().b2u_scale_nc(ptr(x), ptr(s), ptr(add), ptr(out), N, H * W, C, stream_ptr()))
    return out


def se_fc_fwd(pooled, w1, b1, w2, b2, C):
    N, Cp = pooled.shape
    R = w1.shape[0]
    hidden = torch.empty((N, R), dtype=torch.float32, device=pooled.device)
    scale = torch.empty((N, Cp), dtype=torch.float32, device=pooled.device)
    check(lib().b2u_se_fc_fwd(ptr(pooled), ptr(w1), ptr(b1), ptr(w2), ptr(b2), ptr(hidden), ptr(scale), N, C, Cp, R, stream_ptr()))
    return hidden, scale


def se_fc_bwd(dscale, pooled, hidden, scale, w1, w2, C, dp_scale, dw1=None, db1=None, dw2=None, db2=None):
    N, Cp = pooled.shape
    R = w1.shape[0]
    dpooled = torch.empty((N, Cp), dtype=torch.float32, device=pooled.device)
    scratch = torch.empty((N * (C + R),), dtype=torch.float32, device=pooled.device)
    check(lib().b2u_se_fc_bwd(ptr(dscale), ptr(pooled), ptr(hidden), ptr(scale), ptr(w1), ptr(w2), ptr(dpooled), ptr(dw1),
                              ptr(db1), ptr(dw2), ptr(db2), ptr(scratch), N, C, Cp, R, dp_scale, stream_ptr()))
    return dpooled


# ---------------------------------------------------------------------------------------------- head
def head_fwd(x, w, b, out=None):
    _req(x, ACT, "x"); _req(w, torch.float32, "w"); _req(b, torch.float32, "b")
    N, H, W, Cin = x.shape
    ncls = w.shape[0]
    if out is None:
        out = torch.empty((N, ncls, H, W), dtype=torch.float32, device=x.device)
    check(lib().b2u_head_fwd(ptr(x), ptr(w), ptr(b), ptr(out), N, H, W, Cin, ncls, stream_ptr()))
    return out


def head_bwd(dlogits, x, w, need_dx=True, need_dw=True, relu_mask=True, dx=None, dw=None, db=None, ws=None):
    _req(dlogits, torch.float32, "dlogits"); _req(x, ACT, "x"); _req(w, torch.float32, "w")
    N, H, W, Cin = x.shape
    ncls = w.shape[0]
    need = lib().b2u_head_bwd_workspace_cls(ncls)
    if need_dw and (ws is None or ws.numel() * ws.element_size() < need):
        ws = _ws(need, x.device)
    if need_dx and dx is None:
        dx = torch.empty_like(x)
    if need_dw:
        if dw is None:
            dw = torch.empty((ncls, Cin, 1, 1), dtype=torch.float32, device=x.device)
        if db is None:
            db = torch.empty((ncls,), dtype=torch.float32, device=x.device)
    check(lib().b2u_head_bwd(ptr(dlogits), ptr(x), ptr(w), ptr(dx) if need_dx else None,
                             ptr(dw) if need_dw else None, ptr(db) if need_dw else None, ptr(ws) if need_dw else None,
                             0 if not need_dw else ws.numel() * ws.element_size(), N, H, W, Cin, ncls,
                             1 if relu_mask else 0, stream_ptr()))
    return dx, dw, db


# ---------------------------------------------------------------------------------------------- loss / metrics
def loss_fwd(logits, target=None, onehot=None, cls_w=None, beta=1.0, smooth=1e-5, alpha=0.5, gamma=2.0, thr=0.5,
             ws=None):
    """Returns the device vector [CE, Focal, Dice, f_score, backward coefficients...]."""
    _req(logits, torch.float32, "logits"); _req(target, torch.int64, "target")
    _req(onehot, torch.float32, "onehot"); _req(cls_w, torch.float32, "cls_weights")
    N, C, H, W = logits.shape
    need = lib().b2u_loss_workspace(C)
    if ws is None or ws.numel() * ws.element_size() < need:
        ws = _ws(need, logits.device)
    out = torch.empty((lib().b2u_loss_out_len(C),), dtype=torch.float32, device=logits.device)
    check(lib().b2u_loss_fwd(ptr(logits), ptr(target), ptr(onehot), ptr(cls_w), ptr(out), None, ptr(ws),
                             ws.numel() * ws.element_size(), N, C, H, W, beta, smooth,
                             0.0 if alpha is None else alpha, gamma, thr, stream_ptr()))
    return out


def loss_bwd(logits, fin, gscale, target=None, onehot=None, cls_w=None, alpha=0.5, gamma=2.0, out=None, nhwc64=False):
    """dlogits as fp32 NCHW, or (nhwc64) as bf16 [N, H, W, 64 G] zero padded for the tensor-core head backward
    (G = head_groups(C) groups [hi(32) | lo(32)] of 32 classes)."""
    _req(logits, torch.float32, "logits"); _req(gscale, torch.float32, "gscale")
    N, C, H, W = logits.shape
    if out is None:
        out = (torch.empty((N, H, W, 64 * head_groups(C)), dtype=ACT, device=logits.device) if nhwc64
               else torch.empty_like(logits))
    check(lib().b2u_loss_bwd(ptr(logits), ptr(target), ptr(onehot), ptr(cls_w), ptr(fin), ptr(gscale), ptr(out),
                             1 if nhwc64 else 0, N, C, H, W, 0.0 if alpha is None else alpha, gamma, stream_ptr()))
    return out


def head_groups(ncls):
    """Column groups of the tensor-core head: group g = [hi(32) | lo(32)] of classes 32g .. 32g + 31."""
    return (ncls + 31) // 32


def fold_head_groups(t, C, cin, out):
    """out[c] = t[64g + r] + t[64g + 32 + r] for class c = 32g + r: the per-class sum of the hi and lo halves of a [64 G, ...]
    gradient of the tensor-core head (cin: leading input channels kept along dim 1, when t has one)."""
    for g in range(head_groups(C)):
        c0, cn = 32 * g, min(32, C - 32 * g)
        hi, lo = t[64 * g:64 * g + cn], t[64 * g + 32:64 * g + 32 + cn]
        if t.dim() > 1:
            hi, lo = hi[:, :cin], lo[:, :cin]
        torch.add(hi, lo, out=out[c0:c0 + cn])
    return out


def pack_head_dgrad(w, wd=None):
    _req(w, torch.float32, "final.weight")
    ncls = w.shape[0]
    if wd is None:
        wd = torch.empty((64, 64 * head_groups(ncls)), dtype=ACT, device=w.device)
    check(lib().b2u_pack_head_dgrad(ptr(w), ptr(wd), ncls, stream_ptr()))
    return wd


def pack_head_fprop(w, wf=None):
    _req(w, torch.float32, "final.weight")
    ncls = w.shape[0]
    if wf is None:
        wf = torch.empty((64 * head_groups(ncls), 64), dtype=ACT, device=w.device)
    check(lib().b2u_pack_head_fprop(ptr(w), ptr(wf), ncls, stream_ptr()))
    return wf


def head_fwd_tc(x, wf, b, ncls, out=None):
    """The 1x1 classifier on the tensor cores (wf from pack_head_fprop): fp32 NCHW logits."""
    _req(x, ACT, "x"); _req(wf, ACT, "wf"); _req(b, torch.float32, "b")
    N, H, W, Cin = x.shape
    if Cin != 64:
        raise ValueError("head_fwd_tc: the head input must have 64 (padded) channels")
    if out is None:
        out = torch.empty((N, ncls, H, W), dtype=torch.float32, device=x.device)
    check(lib().b2u_head_fwd_tc(ptr(x), ptr(wf), ptr(b), ptr(out), N, H, W, ncls, stream_ptr()))
    return out


def argmax_u8(logits, out=None):
    _req(logits, torch.float32, "logits")
    N, C, H, W = logits.shape
    if out is None:
        out = torch.empty((N, H, W), dtype=torch.uint8, device=logits.device)
    check(lib().b2u_argmax_u8(ptr(logits), ptr(out), N, C, H, W, stream_ptr()))
    return out


def softmax_resize_argmax_u8(logits, crop, out_size, out=None):
    """argmax(cv2.resize(softmax(logits)[crop], out_size, INTER_LINEAR)) as a uint8 mask; crop = (y, x, h, w)."""
    _req(logits, torch.float32, "logits")
    N, C, H, W = logits.shape
    cy, cx, ch, cw = crop
    oh, ow = out_size
    if out is None:
        out = torch.empty((N, oh, ow), dtype=torch.uint8, device=logits.device)
    check(lib().b2u_softmax_resize_argmax_u8(ptr(logits), ptr(out), N, C, H, W, cy, cx, ch, cw, oh, ow, stream_ptr()))
    return out


def pad16(nbytes):
    """Byte offsets of the batched predictor's ragged buffers are multiples of 16 (fast_hist_batch reads 16-byte vectors)."""
    return (int(nbytes) + 15) & ~15


LETTERBOX_ITEM = struct.Struct("<Q8i3q")     # include/b2u.h: src; ih, iw, nh, nw, dy, dx, kx, ky; coef_x, coef_y, tmp
TAIL_ITEM = struct.Struct("<6iq")            # include/b2u.h: cy, cx, ch, cw, oh, ow; mask_off


def letterbox_plan(items, H, W):
    """Host half of the batched letterbox.  items: (src device address of a uint8 [ih, iw, 3] image, ih, iw, nh, nw, dy, dx)
    per image, with resize_image's geometry.  Returns (item table as bytes, workspace bytes) for letterbox_bicubic."""
    if not items:
        raise ValueError("letterbox: empty batch")
    blob = bytearray(b"".join(LETTERBOX_ITEM.pack(int(p), *map(int, g), 0, 0, 0, 0, 0) for p, *g in items))
    buf = (ctypes.c_char * len(blob)).from_buffer(blob)
    ws = lib().b2u_letterbox_workspace(ctypes.addressof(buf), len(items), H, W)
    del buf
    if ws == 0:
        msg = lib().b2u_last_error()
        raise ValueError(f"b2u: {msg.decode() if msg else 'letterbox_workspace failed'}")
    return bytes(blob), ws


def letterbox_bicubic(table, count, out, ws):
    """PIL BICUBIC letterbox of `count` images into fp32 NCHW out[:count] ([>= count, 3, H, W]), bit-exact with
    resize_image + np.float32 / 255; table: letterbox_plan's bytes in a uint8 CUDA tensor, ws: uint8 CUDA workspace."""
    _req(table, torch.uint8, "table"); _req(out, torch.float32, "out"); _req(ws, torch.uint8, "ws")
    if out.dim() != 4 or out.shape[0] < count or out.shape[1] != 3 or table.numel() < count * LETTERBOX_ITEM.size:
        raise ValueError("letterbox: out must be [>= count, 3, H, W] and the table must hold count items")
    check(lib().b2u_letterbox_bicubic(ptr(table), count, ptr(out), out.shape[2], out.shape[3], ptr(ws), ws.numel(),
                                      stream_ptr()))
    return out


def tail_table(crops, sizes, H, W):
    """Item table of softmax_resize_argmax_u8_batch: crop (y, x, h, w) inside H x W and output size (oh, ow) per image.
    Returns (bytes, mask byte offsets (16-byte aligned), total mask bytes)."""
    blob, offs, off = [], [], 0
    for (cy, cx, ch, cw), (oh, ow) in zip(crops, sizes):
        if cy < 0 or cx < 0 or ch <= 0 or cw <= 0 or cy + ch > H or cx + cw > W or oh <= 0 or ow <= 0:
            raise ValueError(f"softmax_resize_argmax_batch: crop {(cy, cx, ch, cw)} / size {(oh, ow)} outside {H}x{W}")
        blob.append(TAIL_ITEM.pack(cy, cx, ch, cw, oh, ow, off))
        offs.append(off)
        off = pad16(off + oh * ow)
    return b"".join(blob), offs, off


def softmax_resize_argmax_u8_batch(logits, table, count, masks, max_oh, max_ow):
    """softmax_resize_argmax_u8 with one crop and output size per image: image i's mask goes to the flat uint8 `masks` at
    the offset tail_table gave it; table: tail_table's bytes in a uint8 CUDA tensor."""
    _req(logits, torch.float32, "logits"); _req(table, torch.uint8, "table"); _req(masks, torch.uint8, "masks")
    N, C, H, W = logits.shape
    if count > N or table.numel() < count * TAIL_ITEM.size:
        raise ValueError("softmax_resize_argmax_batch: more items than logits or table entries")
    check(lib().b2u_softmax_resize_argmax_u8_batch(ptr(logits), ptr(table), count, C, H, W, ptr(masks), max_oh, max_ow,
                                                   stream_ptr()))
    return masks


RENDER_ITEM = struct.Struct("<QQq2i")       # include/b2u.h: src, mask; out_off; ih, iw


def render_table(items, start=0):
    """Item table of render_batch from (src address, mask address, ih, iw) per image; each rendered [ih, iw, 3] image gets a
    16-byte aligned offset from `start` on.  Returns (bytes, image offsets, end offset)."""
    blob, offs, off = [], [], pad16(start)
    for src, mask, ih, iw in items:
        if ih <= 0 or iw <= 0 or not src or not mask:
            raise ValueError(f"render_batch: bad item ({ih}x{iw})")
        blob.append(RENDER_ITEM.pack(src, mask, off, ih, iw))
        offs.append(off)
        off = pad16(off + 3 * ih * iw)
    return b"".join(blob), offs, off


def render_batch(table, count, palette, C, mix_type, out, counts, max_pixels):
    """detect_image's rendering of `count` images in one launch (mix_type 0: blend with 0.7, 1: palette, 2: keep the
    non-background pixels, -1: counts only): table is render_table's bytes in a uint8 CUDA tensor, palette a uint8 CUDA
    tensor of >= 3 C bytes, out the flat uint8 buffer the offsets point into, counts (optional) int64 [>= count * C]."""
    _req(table, torch.uint8, "table"); _req(palette, torch.uint8, "palette"); _req(out, torch.uint8, "out")
    _req(counts, torch.int64, "counts")
    if table.numel() < count * RENDER_ITEM.size or (palette is not None and palette.numel() < 3 * C) or \
            (counts is not None and counts.numel() < count * C):
        raise ValueError("render_batch: the table, palette or counts hold fewer entries than count / C")
    check(lib().b2u_render_batch(ptr(table), count, ptr(palette), C, mix_type, ptr(out), ptr(counts), max_pixels,
                                 stream_ptr()))
    return out


_HIST_DTYPES = {torch.uint8: 0, torch.int32: 1, torch.int64: 2}


def fast_hist_accumulate(a, b, n, hist):
    """hist (uint64 as int64 tensor, n*n+1) += histogram of (a, b); a, b flat CUDA tensors of one dtype."""
    if a.dtype != b.dtype or a.dtype not in _HIST_DTYPES:
        raise ValueError("fast_hist: a and b must both be uint8, int32 or int64")
    _req(a, a.dtype, "a"); _req(b, b.dtype, "b"); _req(hist, torch.int64, "hist")
    if a.numel() != b.numel():
        raise ValueError("fast_hist: a and b must have the same number of elements")
    check(lib().b2u_fast_hist(ptr(a), ptr(b), a.numel(), n, _HIST_DTYPES[a.dtype], ptr(hist), stream_ptr()))
    return hist


def hist_items(pairs):
    """Item table of fast_hist_batch from (a address, b address, length) per uint8 mask pair, both 16-byte aligned.
    Returns (table bytes, total chunks)."""
    blob, chunks = [], 0
    chunk_fn = lib().b2u_fast_hist_chunks
    for a, b, n in pairs:
        if a % 16 or b % 16:
            raise ValueError("fast_hist_batch: masks must be 16-byte aligned")
        blob.append(struct.pack("<QQqq", a, b, n, chunks))
        chunks += chunk_fn(n)
    return b"".join(blob), chunks


class HistTable:
    """Device-resident pointer table of (a, b) uint8 CUDA mask pairs for fast_hist_batch (keeps the masks alive)."""

    def __init__(self, pairs, device):
        for a, b in pairs:
            _req(a, torch.uint8, "a"); _req(b, torch.uint8, "b")
            if a.numel() != b.numel():
                raise ValueError("fast_hist_batch: a and b must have the same number of elements")
        blob, chunks = hist_items([(a.data_ptr(), b.data_ptr(), a.numel()) for a, b in pairs])
        self.pairs, self.count, self.chunks = list(pairs), len(pairs), chunks
        self.table = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(device) if blob else None


def fast_hist_batch(pairs, n, hist):
    """hist += confusion matrices of many (a, b) uint8 CUDA mask pairs in ONE launch.  pairs: list of (a, b) or a HistTable."""
    _req(hist, torch.int64, "hist")
    tab = pairs if isinstance(pairs, HistTable) else HistTable(pairs, hist.device)
    if tab.count:
        check(lib().b2u_fast_hist_batch(ptr(tab.table), tab.count, tab.chunks, n, ptr(hist), stream_ptr()))
    return hist


def fast_hist_batch_items(table, count, chunks, n, hist):
    """fast_hist_batch over an item table already in device memory (hist_items' bytes in a uint8 CUDA tensor); the caller
    keeps the masks alive until the launch has run."""
    _req(table, torch.uint8, "table"); _req(hist, torch.int64, "hist")
    if table.numel() < 32 * count:
        raise ValueError("fast_hist_batch: the table holds fewer than count items")
    if count:
        check(lib().b2u_fast_hist_batch(ptr(table), count, chunks, n, ptr(hist), stream_ptr()))
    return hist


def argmax_hist(logits, gt=None, n=0, hist=None, pred=None, want_pred=False):
    """Per-pixel class decision of fp32 NCHW logits (+ optional uint8 mask) fused with fast_hist against `gt` (uint8 [N, H, W]).
    Returns (hist, pred)."""
    _req(logits, torch.float32, "logits"); _req(gt, torch.uint8, "gt"); _req(hist, torch.int64, "hist"); _req(pred, torch.uint8, "pred")
    N, C, H, W = logits.shape
    if want_pred and pred is None:
        pred = torch.empty((N, H, W), dtype=torch.uint8, device=logits.device)
    if gt is not None and hist is None:
        hist = torch.zeros(n * n + 1, dtype=torch.int64, device=logits.device)
    check(lib().b2u_argmax_hist(ptr(logits), ptr(gt), ptr(pred), N, C, H, W, n, ptr(hist), stream_ptr()))
    return hist, pred


# ---------------------------------------------------------------------------------------------- optimizer
def adam_step(param, grad, m, v, step, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, grad_scale=1.0):
    for t, nme in ((param, "param"), (grad, "grad"), (m, "exp_avg"), (v, "exp_avg_sq")):
        _req(t, torch.float32, nme)
    check(lib().b2u_adam_step(ptr(param), ptr(grad), ptr(m), ptr(v), param.numel(), lr, betas[0], betas[1], eps,
                              weight_decay, step, grad_scale, stream_ptr()))


def sgd_step(param, grad, buf, lr, momentum=0.0, weight_decay=0.0, nesterov=False, first_step=False, grad_scale=1.0):
    check(lib().b2u_sgd_step(ptr(param), ptr(grad), ptr(buf), param.numel(), lr, momentum, weight_decay,
                             1 if nesterov else 0, 1 if first_step else 0, grad_scale, stream_ptr()))
