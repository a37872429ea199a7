"""ctypes binding of libb200unet.so (include/b2u.h).  No fallback: a missing library is a hard error."""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_longlong, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# B2U_LIB_PATH: an alternative build of the SAME library (A/B runs of two kernel generations on one box); there still is no
# fallback -- the named file must exist and export the whole ABI
LIB_PATH = os.environ.get("B2U_LIB_PATH") or os.path.join(_HERE, "libb200unet.so")
# fp32 VALIDATION build of the same ABI (csrc/validation_fp32.cu): NHWC fp32 tensors, CUDA-core contractions; covers the
# entry points UNetEngine uses.  Selected by set_validation_fp32(True) or B2U_FP32_VALIDATION=1; never the product path.
LIB_PATH_FP32 = os.path.join(_HERE, "libb200unet_fp32.so")

P, I, F, LL, SZ = c_void_p, c_int, c_float, c_longlong, c_size_t

# name -> (restype, argtypes); must list every symbol include/b2u.h declares (tests/test_abi.py checks this)
SIGNATURES = {
    "b2u_last_error": (c_char_p, []),
    "b2u_version": (I, []),
    "b2u_num_sms": (I, []),
    "b2u_launch_count": (LL, []),
    "b2u_reset_launch_count": (None, []),
    "b2u_im2col_first": (I, [P, P, I, I, I, I, P]),
    "b2u_pack_weights": (I, [P, P, P, I, I, I, P]),
    "b2u_pack_weights_first": (I, [P, P, I, I, P]),
    "b2u_pack_weights_multi": (I, [P, I, LL, P]),
    "b2u_nhwc_bf16_to_nchw_f32": (I, [P, P, I, I, I, I, P]),
    "b2u_nchw_f32_to_nhwc_bf16": (I, [P, P, I, I, I, I, P]),
    "b2u_nchw_f32_to_nhwc_bf16_padded": (I, [P, P, I, I, I, I, I, P]),
    "b2u_u8hwc_to_nchw_f32": (I, [P, P, I, I, I, I, F, P]),
    "b2u_u8_to_i64": (I, [P, P, LL, P]),
    "b2u_letterbox_workspace": (SZ, [P, I, I, I]),
    "b2u_letterbox_bicubic": (I, [P, I, P, I, I, P, SZ, P]),
    "b2u_conv_fprop": (I, [P, I, P, I, P, P, P, I, I, I, I, I, I, I, P]),
    "b2u_bn_moments": (I, [P, P, P, SZ, LL, I, P]),
    "b2u_bn_fwd_train_moments": (I, [P, P, P, P, P, P, P, P, P, P, I, P, SZ, LL, I, F, F, I, P]),
    "b2u_bn_bwd_sums": (I, [P, P, P, P, P, P, P, P, P, SZ, LL, I, I, P]),
    "b2u_bn_bwd_apply_sums": (I, [P, P, P, P, P, P, P, P, P, P, LL, P, SZ, LL, I, I, P]),
    "b2u_bn_fold": (I, [P, P, P, P, P, P, P, I, F, P]),
    "b2u_conv_fprop_scaled": (I, [P, I, P, I, P, P, P, P, I, I, I, I, I, I, I, P]),
    "b2u_conv_stat_rows": (I, [I, I, I, I, I, I]),
    "b2u_conv_fprop_stats": (I, [P, I, P, I, P, P, P, I, I, I, I, I, I, I, P, I, P]),
    "b2u_bn_fwd_train_stats": (I, [P, P, P, P, P, P, P, P, P, P, I, P, SZ, LL, I, F, F, I, P]),
    "b2u_decoder_conv_fprop": (I, [P, I, P, I, P, P, P, P, P, I, I, I, I, I, I, P, I, P]),
    "b2u_conv_dgrad": (I, [P, I, P, P, I, P, I, P, I, I, I, I, I, P]),
    "b2u_conv_fprop_relu_bits": (I, [P, I, P, I, P, P, P, P, P, P, I, I, I, I, I, I, P]),
    "b2u_conv_dgrad_bits": (I, [P, I, P, P, I, P, I, I, I, I, I, P, I, P]),
    "b2u_conv_dgrad_stat_rows": (I, [I, I, I, I, I, I, I]),
    "b2u_conv_dgrad_stats": (I, [P, I, P, P, I, P, I, P, I, I, I, I, I, P, I, P]),
    "b2u_bias_from_stats": (I, [P, I, I, P, P]),
    "b2u_conv_wgrad_workspace": (SZ, [I, I, I, I, I, I]),
    "b2u_conv_wgrad": (I, [P, I, P, I, P, I, P, P, P, SZ, I, I, I, I, I, I, P]),
    "b2u_bias_grad_workspace": (SZ, [I]),
    "b2u_bias_grad": (I, [P, P, P, SZ, LL, I, P]),
    "b2u_first_conv_dgrad_input": (I, [P, I, P, P, I, I, I, I, I, P]),
    "b2u_stem_dgrad_input": (I, [P, I, P, P, I, I, I, I, I, P]),
    "b2u_nhwc_bf16_padded_to_nchw_f32": (I, [P, P, I, I, I, I, I, P]),
    "b2u_maxpool2x2_fwd": (I, [P, P, I, I, I, I, P]),
    "b2u_maxpool2x2_bwd": (I, [P, P, P, P, I, I, I, I, I, P]),
    "b2u_upsample2x_fwd": (I, [P, P, I, I, I, I, P]),
    "b2u_upsample2x_bwd": (I, [P, P, P, I, I, I, I, P]),
    "b2u_bn_workspace": (SZ, [I]),
    "b2u_bn_fwd_train": (I, [P, P, P, P, P, P, P, P, P, P, SZ, LL, I, F, F, I, P]),
    "b2u_bn_fwd_eval": (I, [P, P, P, P, P, P, P, P, SZ, LL, I, F, I, P]),
    "b2u_bn_bwd": (I, [P, P, P, P, P, P, P, P, P, P, P, P, SZ, LL, I, I, P]),
    "b2u_im2col_stem": (I, [P, P, I, I, I, I, P]),
    "b2u_pack_weights_im2col": (I, [P, P, I, I, I, I, P]),
    "b2u_conv_wgrad_im2col": (I, [P, I, P, I, P, P, SZ, I, I, I, I, I, P]),
    "b2u_subsample2": (I, [P, P, I, I, I, I, P]),
    "b2u_zero_insert2": (I, [P, P, I, I, I, I, P]),
    "b2u_maxpool3x3s2_fwd": (I, [P, P, I, I, I, I, P]),
    "b2u_maxpool3x3s2_bwd": (I, [P, P, P, I, I, I, I, P]),
    "b2u_add_bf16": (I, [P, P, P, LL, P]),
    "b2u_add_relu_bf16": (I, [P, P, P, LL, P]),
    "b2u_relu_bwd_bf16": (I, [P, P, P, LL, P]),
    "b2u_resize_bilinear_f32_fwd": (I, [P, P, LL, I, I, I, I, P]),
    "b2u_resize_bilinear_f32_bwd": (I, [P, P, LL, I, I, I, I, P]),
    "b2u_dwconv3x3_fwd": (I, [P, P, P, P, I, I, I, I, I, P]),
    "b2u_dwconv3x3_wgrad_workspace": (SZ, [I]),
    "b2u_dwconv3x3_wgrad": (I, [P, P, P, P, P, SZ, I, I, I, I, P]),
    "b2u_spatial_reduce_workspace_floats": (I, [I, I]),
    "b2u_spatial_reduce": (I, [P, P, P, P, SZ, I, LL, I, F, P]),
    "b2u_scale_nc": (I, [P, P, P, P, I, LL, I, P]),
    "b2u_se_fc_fwd": (I, [P, P, P, P, P, P, P, I, I, I, I, P]),
    "b2u_se_fc_bwd": (I, [P, P, P, P, P, P, P, P, P, P, P, P, I, I, I, I, F, P]),
    "b2u_head_fwd": (I, [P, P, P, P, I, I, I, I, I, P]),
    "b2u_head_bwd_workspace": (SZ, []),
    "b2u_head_bwd_workspace_cls": (SZ, [I]),
    "b2u_head_bwd": (I, [P, P, P, P, P, P, P, SZ, I, I, I, I, I, I, P]),
    "b2u_loss_workspace": (SZ, [I]),
    "b2u_loss_out_len": (I, [I]),
    "b2u_loss_fwd": (I, [P, P, P, P, P, P, P, SZ, I, I, I, I, F, F, F, F, F, P]),
    "b2u_loss_bwd": (I, [P, P, P, P, P, P, P, I, I, I, I, I, F, F, P]),
    "b2u_pack_head_dgrad": (I, [P, P, I, P]),
    "b2u_pack_head_fprop": (I, [P, P, I, P]),
    "b2u_head_fwd_tc": (I, [P, P, P, P, I, I, I, I, P]),
    "b2u_argmax_u8": (I, [P, P, I, I, I, I, P]),
    "b2u_softmax_resize_argmax_u8": (I, [P, P, I, I, I, I, I, I, I, I, I, I, P]),
    "b2u_softmax_resize_argmax_u8_batch": (I, [P, P, I, I, I, I, P, I, I, P]),
    "b2u_render_batch": (I, [P, I, P, I, I, P, P, LL, P]),
    "b2u_fast_hist": (I, [P, P, LL, I, I, P, P]),
    "b2u_fast_hist_batch": (I, [P, I, LL, I, P, P]),
    "b2u_fast_hist_chunks": (LL, [LL]),
    "b2u_argmax_hist": (I, [P, P, P, I, I, I, I, I, P, P]),
    "b2u_adam_step": (I, [P, P, P, P, LL, F, F, F, F, F, I, F, P]),
    "b2u_sgd_step": (I, [P, P, P, LL, F, F, F, I, I, F, P]),
}

_lib = None
_handles = {}                     # library path -> loaded handle
_validation = os.environ.get("B2U_FP32_VALIDATION", "0") not in ("", "0")


class B2UError(RuntimeError):
    pass


class _ValidationLib:
    """The fp32 validation library exports a subset of the ABI; anything else fails loudly instead of silently running bf16."""

    def __init__(self, handle):
        self._h = handle

    def __getattr__(self, name):
        try:
            fn = getattr(self._h, name)
        except AttributeError:
            raise B2UError(f"{name} is not part of the fp32 validation build (libb200unet_fp32.so)") from None
        setattr(self, name, fn)
        return fn


def _load(path, validation):
    if not os.path.exists(path):
        raise B2UError(
            f"{path} is missing: build it with `python unet-pytorch_b200/build.py` "
            "(there is no CPU or PyTorch fallback for the hot path)")
    h = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        if validation and not hasattr(h, name):
            continue
        fn = getattr(h, name)
        fn.restype = res
        fn.argtypes = args
    return _ValidationLib(h) if validation else h


def lib():
    """Loads the CUDA library; raises if it has not been built (python unet-pytorch_b200/build.py)."""
    global _lib
    if _lib is None:
        path = LIB_PATH_FP32 if _validation else LIB_PATH
        if path not in _handles:
            _handles[path] = _load(path, _validation)
        _lib = _handles[path]
    return _lib


def validation_fp32():
    return _validation


def set_validation_fp32(on):
    """Routes every C-ABI call of this process to the fp32 validation build (True) or back to the product library (False).
    Engines / modules must be constructed after the switch: their buffers and packed operands take the activation dtype
    (ops.act_dtype()) of the library they were built for."""
    global _lib, _validation
    _validation = bool(on)
    _lib = None


class CallProfile:
    """Measurement aid (scripts/variants_bench.py): while active, every C-ABI call made through lib() is bracketed with CUDA
    events on the current stream.  read() -> {entry point: {"launches", "ms"}}.  Not used on the product path."""

    def __init__(self, by_shape=False):
        self.records = {}
        self.by_shape = by_shape

    def __enter__(self):
        import torch
        real, rec, by_shape = lib(), self.records, self.by_shape

        class _Proxy:
            def __getattr__(self, name):
                fn = getattr(real, name)
                if not name.startswith("b2u_") or not SIGNATURES.get(name, (None, []))[1] or SIGNATURES[name][1][-1] is not ctypes.c_void_p:
                    return fn

                def timed(*a):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); rc = fn(*a); e1.record()
                    key = name if not by_shape else name + str(tuple(x for x in a if isinstance(x, int) and 0 <= x < (1 << 24)))
                    rec.setdefault(key, []).append((e0, e1))
                    return rc
                return timed
        global _lib
        self._real = real
        _lib = _Proxy()
        return self

    def __exit__(self, *exc):
        global _lib
        _lib = self._real

    def read(self):
        import torch
        torch.cuda.synchronize()
        return {k: {"launches": len(v), "ms": sum(a.elapsed_time(b) for a, b in v)} for k, v in self.records.items()}


def check(rc):
    if rc != 0:
        msg = lib().b2u_last_error()
        msg = msg.decode() if msg else ""
        if rc == 1:
            raise ValueError(f"b2u: {msg}")
        raise B2UError(f"b2u error {rc}: {msg}")


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return None if t is None else t.data_ptr()
