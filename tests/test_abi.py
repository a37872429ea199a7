"""CPU: the C-ABI library builds, loads and exports exactly what include/b2u.h declares; the product path has no
CPU fallback."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "b2u.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b2u_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(b2u):
    names = _declared()
    assert len(names) >= 30
    h = ctypes.CDLL(b2u._lib.LIB_PATH)
    for n in names:
        assert hasattr(h, n), f"{n} declared in include/b2u.h but not exported"


def test_ctypes_signatures_cover_the_header(b2u):
    assert sorted(b2u._lib.SIGNATURES.keys()) == _declared()


def test_version_and_error_channel_without_gpu(b2u):
    lib = b2u._lib.lib()
    assert lib.b2u_version() >= 100
    # argument validation happens before any CUDA call: a bad shape reports through the error channel
    rc = lib.b2u_fast_hist(None, None, 10, 0, 0, None, None)
    assert rc == 1 and b"fast_hist" in lib.b2u_last_error()
    rc = lib.b2u_conv_fprop(None, 60, None, 0, None, None, None, 1, 8, 8, 64, 9, 1, 0, None)
    assert rc == 1 and b"multiples of 64" in lib.b2u_last_error()
    assert lib.b2u_conv_wgrad_workspace(16, 512, 512, 64, 64, 9) > 0


def test_conv_wgrad_rejects_undefined_flags(b2u):
    """b2u_conv_wgrad defines flags bit 1 only (force the generic kernel); the product and the fp32 validation library both
    reject any other bit before touching the GPU."""
    fp32 = ctypes.CDLL(b2u._lib.LIB_PATH_FP32)
    fp32.b2u_last_error.restype = ctypes.c_char_p
    for lib in (b2u._lib.lib(), fp32):
        for flags in (1, 3, 4):
            rc = lib.b2u_conv_wgrad(None, 64, None, 0, None, 64, None, None, None, 0, 1, 8, 16, 9, 0, flags, None)
            assert rc == 5 and b"flags" in lib.b2u_last_error(), (lib, flags)       # B2U_ERR_ARG


def test_product_path_has_no_cpu_fallback(b2u):
    m = b2u.Unet(num_classes=2)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 32, 32))
    with pytest.raises(ValueError):
        b2u.ops.maxpool2x2(torch.zeros(1, 4, 4, 8, dtype=torch.bfloat16))
    with pytest.raises(RuntimeError):
        b2u.CE_Loss(torch.zeros(1, 2, 4, 4), torch.zeros(1, 4, 4, dtype=torch.long), torch.ones(2), num_classes=2)


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "unet-pytorch_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                assert "oracle" not in open(os.path.join(dirpath, f)).read(), f"{f} mentions the oracle"


def test_missing_library_is_a_hard_error(b2u, monkeypatch):
    monkeypatch.setattr(b2u._lib, "_lib", None)
    monkeypatch.setattr(b2u._lib, "LIB_PATH", "/nonexistent/libb200unet.so")
    with pytest.raises(b2u._lib.B2UError):
        b2u._lib.lib()


def test_fp32_validation_library_exports_its_subset(b2u):
    """libb200unet_fp32.so (csrc/validation_fp32.cu): the same ABI names for the entry points UNetEngine uses, and nothing
    undeclared except its identification symbol; selected explicitly, never by default."""
    h = ctypes.CDLL(b2u._lib.LIB_PATH_FP32)
    need = ["b2u_im2col_first", "b2u_pack_weights_multi", "b2u_conv_fprop", "b2u_conv_fprop_stats", "b2u_conv_fprop_scaled",
            "b2u_conv_dgrad", "b2u_conv_wgrad", "b2u_conv_wgrad_workspace", "b2u_bias_grad", "b2u_maxpool2x2_fwd",
            "b2u_maxpool2x2_bwd", "b2u_upsample2x_fwd", "b2u_upsample2x_bwd", "b2u_head_fwd", "b2u_head_bwd", "b2u_bn_fwd_train",
            "b2u_bn_fwd_train_stats", "b2u_bn_fwd_eval", "b2u_bn_bwd", "b2u_bn_fold", "b2u_loss_fwd", "b2u_loss_bwd",
            "b2u_fast_hist", "b2u_adam_step", "b2u_sgd_step", "b2u_last_error", "b2u_launch_count"]
    for n in need:
        assert hasattr(h, n) and n in b2u._lib.SIGNATURES, n
    assert h.b2u_validation_fp32() == 1
    assert not hasattr(ctypes.CDLL(b2u._lib.LIB_PATH), "b2u_validation_fp32")
    assert not b2u._lib.validation_fp32() and b2u.ops.act_dtype() == torch.bfloat16      # the default is the product library
    h.b2u_conv_fprop.restype = ctypes.c_int
    rc = h.b2u_conv_fprop(None, 60, None, 0, None, None, None, 1, 8, 8, 64, 9, 1, 0, None)
    assert rc == 1


def test_validation_switch_routes_and_restores(b2u):
    """ops.set_validation_fp32: the process-wide switch between the product library and the fp32 validation build; entry
    points the validation build lacks raise instead of falling through to another precision."""
    ops, _lib = b2u.ops, b2u._lib
    try:
        ops.set_validation_fp32(True)
        assert _lib.validation_fp32() and ops.act_dtype() == torch.float32
        v = _lib.lib()
        assert v.b2u_validation_fp32() == 1 and v.b2u_version() >= 100
        with pytest.raises(_lib.B2UError):
            v.b2u_head_fwd_tc
        with pytest.raises(_lib.B2UError):
            v.b2u_bn_moments                # SyncBatchNorm building blocks are product-only
    finally:
        ops.set_validation_fp32(False)
    assert not _lib.validation_fp32() and ops.act_dtype() == torch.bfloat16
    assert not hasattr(_lib.lib(), "b2u_validation_fp32")
