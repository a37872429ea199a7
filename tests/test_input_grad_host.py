"""CPU: the entry points of the gradient wrt the input image are exported by both libraries with the header's signatures,
validate their arguments before touching the GPU, and compile without register spills."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["b2u_first_conv_dgrad_input", "b2u_stem_dgrad_input", "b2u_nhwc_bf16_padded_to_nchw_f32"]


def _libs(b2u):
    out = []
    for path in (b2u._lib.LIB_PATH, b2u._lib.LIB_PATH_FP32):
        h = ctypes.CDLL(path)
        for n in NAMES + ["b2u_last_error"]:
            res, args = b2u._lib.SIGNATURES[n]
            getattr(h, n).restype, getattr(h, n).argtypes = res, args
        out.append(h)
    return out


def test_both_libraries_export_the_input_grad_entry_points(b2u):
    for h in _libs(b2u):
        for n in NAMES:
            assert hasattr(h, n), n


def test_bad_shapes_are_refused_without_a_gpu(b2u):
    for h in _libs(b2u):
        # 9 Cin > 64, Cout > Cz, Cz not a multiple of 16
        for args in ((64, 8, 64), (64, 3, 128), (40, 3, 40)):
            cz, cin, cout = args
            assert h.b2u_first_conv_dgrad_input(None, cz, None, None, 1, cin, 8, 8, cout, None) == 1
            assert b"first_conv_dgrad_input" in h.b2u_last_error()
        assert h.b2u_stem_dgrad_input(None, 64, None, None, 1, 4, 8, 8, 64, None) == 1      # 49 Cin > 192
        assert b"stem_dgrad_input" in h.b2u_last_error()
        assert h.b2u_nhwc_bf16_padded_to_nchw_f32(None, None, 1, 65, 8, 8, 64, None) == 1  # C > Cpad
        assert b"padded_to_nchw" in h.b2u_last_error()
        # a dz / x that is not 16-byte aligned is refused (B2U_ERR_ARG), before any launch
        assert h.b2u_first_conv_dgrad_input(8, 64, None, None, 1, 3, 8, 8, 64, None) == 5
        assert b"aligned" in h.b2u_last_error()
        assert h.b2u_stem_dgrad_input(8, 64, None, None, 1, 3, 8, 8, 64, None) == 5
        assert h.b2u_nhwc_bf16_padded_to_nchw_f32(8, None, 1, 3, 8, 8, 64, None) == 5


def test_ops_wrappers_check_their_arguments(b2u):
    """Shape errors are reported before the device checks (so they show on CPU tensors); CPU tensors of the right shape are
    refused as such -- there is no CPU fallback."""
    import torch
    dz = torch.zeros(1, 8, 8, 64, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="3x3"):
        b2u.ops.first_conv_dgrad_input(dz, torch.zeros(64, 3, 7, 7))
    with pytest.raises(ValueError, match="7x7"):
        b2u.ops.stem_dgrad_input(dz, torch.zeros(64, 3, 3, 3), 16, 16)
    with pytest.raises(ValueError, match="half the image size"):
        b2u.ops.stem_dgrad_input(dz, torch.zeros(64, 3, 7, 7), 18, 16)
    with pytest.raises(ValueError, match="must be in"):
        b2u.ops.nhwc_padded_to_nchw_f32(dz, 65)
    with pytest.raises(ValueError, match="CUDA"):
        b2u.ops.first_conv_dgrad_input(dz, torch.zeros(64, 3, 3, 3))
    with pytest.raises(ValueError, match="CUDA"):
        b2u.ops.stem_dgrad_input(dz, torch.zeros(64, 3, 7, 7), 16, 15)      # odd widths are accepted shapes
    with pytest.raises(ValueError, match="CUDA"):
        b2u.ops.nhwc_padded_to_nchw_f32(dz, 3)


def test_new_kernels_do_not_spill(b2u):
    log = os.path.join(ROOT, "unet-pytorch_b200", "build", "ptxas.log")
    if not os.path.exists(log):
        pytest.skip("no ptxas log: the libraries were not built in this tree")
    text = open(log).read()
    blocks = re.findall(r"Compiling entry function '([^']+)'.*?\n(.*?bytes spill loads)", text, flags=re.S)
    ours = [(k, s) for k, s in blocks if any(n in k for n in ("dgrad_input", "padded_to_nchw"))]
    assert len(ours) >= 9, [k for k, _ in ours]
    for k, s in ours:
        assert "0 bytes spill stores, 0 bytes spill loads" in s, k
