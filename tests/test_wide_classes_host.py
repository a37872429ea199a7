"""CPU: the host side of heads with up to 255 classes -- state_dict shapes of every family, the class-count bounds, the
ABI's shape errors past them, and the class-dependent workspace of the SIMT head backward."""
import pytest
import torch

from oracle import unet_oracle as O


@pytest.mark.parametrize("C", [150, 255])
def test_wide_state_dict_shapes_every_family(b2u, C):
    import importlib
    m = b2u.Unet(num_classes=C, pretrained=False, backbone="vgg")
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == O.param_shapes(C)
    m.load_state_dict(O.make_params(C))
    r = b2u.Unet(num_classes=C, backbone="resnet50")
    assert {n: tuple(p.shape) for n, p in r.named_parameters()} == O.resnet_unet_param_shapes(C)
    t = b2u.TraditionalUnet(in_channels=3, num_classes=C)
    assert {n: tuple(p.shape) for n, p in t.named_parameters()} == O.trad_param_shapes(C)
    lw = b2u.LightweightUnet(num_classes=C)
    sd = O.make_lw_params(C)
    assert {k: tuple(v.shape) for k, v in lw.state_dict().items()} == {k: tuple(v.shape) for k, v in sd.items()}
    for variant, cls in (("ultralight", "UltraLightweightUnet"), ("ultralight_large", "UltraLightweightUnet_large"),
                         ("ultralight_large_optimized", "UltraLightweightUnet_large_optimized")):
        Net = getattr(importlib.import_module(f"unet_pytorch_b200.nets.{cls}"), cls)
        u = Net(num_classes=C)
        ref = O.make_ulu_params(C, variant)
        assert {k: tuple(v.shape) for k, v in u.state_dict().items()} == {k: tuple(v.shape) for k, v in ref.items()}
    from unet_pytorch_b200.nets.RepVGG_Unet import ImprovedSegNet
    isn = ImprovedSegNet(num_classes=C)
    heads = [v for k, v in isn.state_dict().items() if v.dim() == 4 and v.shape[0] == C]
    assert heads


@pytest.mark.parametrize("C", [0, 256])
def test_class_count_bounds(b2u, C):
    from unet_pytorch_b200.graph import (ImprovedSegNetEngine, LightweightUnetEngine, ResNet50UnetEngine,
                                         UltraLightUnetEngine)
    from unet_pytorch_b200.engine import UNetEngine, traditional_unet_config, vgg_unet_config
    for make in (lambda: UNetEngine(vgg_unet_config(C)), lambda: UNetEngine(traditional_unet_config(C)),
                 lambda: ResNet50UnetEngine(C), lambda: UltraLightUnetEngine(C),
                 lambda: LightweightUnetEngine(C), lambda: ImprovedSegNetEngine(C)):
        with pytest.raises(ValueError):
            make()


def test_wide_engines_accept_255(b2u):
    from unet_pytorch_b200.graph import LightweightUnetEngine, ResNet50UnetEngine
    from unet_pytorch_b200.engine import UNetEngine, traditional_unet_config, vgg_unet_config
    for make in (lambda: UNetEngine(vgg_unet_config(255)), lambda: UNetEngine(traditional_unet_config(255)),
                 lambda: ResNet50UnetEngine(255), lambda: LightweightUnetEngine(255)):
        make()


def test_wide_abi_shape_errors(b2u):
    """Argument checks run before any CUDA call: one past the supported range reports through the error channel."""
    lib = b2u._lib.lib()
    assert lib.b2u_head_fwd(None, None, None, None, 1, 8, 8, 64, 256, None) == 1 and b"255" in lib.b2u_last_error()
    assert lib.b2u_head_fwd_tc(None, None, None, None, 1, 8, 8, 256, None) == 1
    assert lib.b2u_pack_head_fprop(None, None, 256, None) == 1 and lib.b2u_pack_head_dgrad(None, None, 256, None) == 1
    assert lib.b2u_loss_bwd(None, None, None, None, None, None, None, 0, 1, 256, 8, 8, 0.5, 2.0, None) == 1
    assert lib.b2u_softmax_resize_argmax_u8(None, None, 1, 256, 8, 8, 0, 0, 8, 8, 8, 8, None) == 1
    assert lib.b2u_fast_hist(None, None, 10, 257, 0, None, None) == 1 and b"256" in lib.b2u_last_error()
    assert lib.b2u_fast_hist_batch(None, 1, 1, 257, None, None) == 1
    assert lib.b2u_argmax_hist(None, b"\0", None, 1, 4, 8, 8, 257, None, None) != 0 and b"argmax_hist" in lib.b2u_last_error()


def test_head_bwd_workspace_by_class_count(b2u):
    lib = b2u._lib.lib()
    old = lib.b2u_head_bwd_workspace()
    assert all(lib.b2u_head_bwd_workspace_cls(c) == old for c in (1, 2, 21, 32))
    sizes = [lib.b2u_head_bwd_workspace_cls(c) for c in (33, 64, 65, 150, 255)]
    assert sizes == sorted(sizes) and sizes[0] > old and sizes[-1] == 8 * old
    assert b2u.ops.head_groups(32) == 1 and b2u.ops.head_groups(33) == 2 and b2u.ops.head_groups(255) == 8


def test_fold_head_groups(b2u):
    """[64 G, ...] tensor-core head gradients fold to [C, ...]: row 64g + r (hi) plus row 64g + 32 + r (lo) -> class 32g + r."""
    C, G = 70, 3
    t = torch.randn(64 * G, 64, 1, 1)
    out = torch.empty(C, 48, 1, 1)
    b2u.ops.fold_head_groups(t, C, 48, out)
    for c in (0, 31, 32, 63, 64, 69):
        g, r = divmod(c, 32)
        assert torch.equal(out[c], t[64 * g + r, :48] + t[64 * g + 32 + r, :48])
    tb = torch.randn(64 * G)
    ob = b2u.ops.fold_head_groups(tb, C, 48, torch.empty(C))
    assert torch.equal(ob[69], tb[64 * 2 + 5] + tb[64 * 2 + 32 + 5])
