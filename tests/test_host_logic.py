"""CPU: host-side mirror of the reference interface -- module tree / state_dict contract, freeze semantics,
LR schedule, flat-buffer layout and bucket planning."""
import math

import numpy as np
import pytest
import torch

from oracle import unet_oracle as O


def test_state_dict_contract(b2u):
    m = b2u.Unet(num_classes=21, pretrained=False, backbone="vgg")
    shapes = O.param_shapes(21)
    sd = m.state_dict()
    assert list(sd.keys()) == list(shapes.keys())            # 44 tensors, reference order (SURVEY.md section 5)
    assert all(tuple(sd[k].shape) == shapes[k] and sd[k].dtype == torch.float32 for k in sd)
    assert sum(v.numel() for v in sd.values()) == 24_892_437
    m.load_state_dict(O.make_params(21))
    assert m.backbone == "vgg" and m.up_conv is None and hasattr(m, "vgg") and hasattr(m, "final")


def test_backbone_errors(b2u):
    with pytest.raises(ValueError):
        b2u.Unet(num_classes=2, backbone="mobilenet")          # nets/unet.py:34


def test_resnet50_and_traditional_state_dict_contract(b2u):
    m = b2u.Unet(num_classes=21, backbone="resnet50")
    shapes = O.resnet_unet_param_shapes(21)
    assert [n for n, _ in m.named_parameters()] == list(shapes.keys())
    assert all(tuple(p.shape) == shapes[n] for n, p in m.named_parameters())
    assert sum(p.numel() for p in m.parameters()) == 43_934_101       # SURVEY.md section 2
    assert m.up_conv is not None and hasattr(m, "resnet")
    m.load_state_dict(O.make_resnet_unet_params(21))
    m.freeze_backbone()
    assert all(not p.requires_grad for p in m.resnet.parameters()) and m.final.weight.requires_grad
    t = b2u.TraditionalUnet(in_channels=3, num_classes=21)
    assert [n for n, _ in t.named_parameters()] == list(O.trad_param_shapes(21).keys())
    assert sum(p.numel() for p in t.parameters()) == 1_950_357        # Submit_result figure quoted in BASELINE.md
    t.load_state_dict(O.make_trad_params(21))
    t.freeze_encoder()
    assert not t.inc.double_conv[0].weight.requires_grad and t.outc.weight.requires_grad


def test_freeze_unfreeze(b2u):
    m = b2u.Unet(num_classes=2)
    m.freeze_backbone()
    assert all(not p.requires_grad for p in m.vgg.parameters())
    assert all(p.requires_grad for n, p in m.named_parameters() if not n.startswith("vgg."))
    m.unfreeze_backbone()
    assert all(p.requires_grad for p in m.parameters())


def test_weights_init_matches_class_name_rule(b2u):
    from unet_pytorch_b200.nets.unet_training import weights_init
    m = b2u.Unet(num_classes=2)
    torch.manual_seed(0)
    weights_init(m)
    w = m.up_concat1.conv1.weight
    assert abs(w.std().item() - 0.02) < 2e-3 and abs(w.mean().item()) < 1e-3


def test_lr_scheduler_closed_forms(b2u):
    from unet_pytorch_b200.nets.unet_training import get_lr_scheduler
    f = get_lr_scheduler("cos", 1e-4, 1e-6, 100)
    assert f(0) == pytest.approx(1e-5)                        # warm-up start = max(0.1 * lr, 1e-6)
    assert f(3) == pytest.approx(1e-4)
    assert f(99) == pytest.approx(1e-6)
    mid = 1e-6 + 0.5 * (1e-4 - 1e-6) * (1 + math.cos(math.pi * (50 - 3) / (100 - 3 - 5)))
    assert f(50) == pytest.approx(mid)
    s = get_lr_scheduler("step", 1e-4, 1e-6, 100)
    assert s(0) == pytest.approx(1e-4) and s(99) == pytest.approx(1e-6)


def test_flat_layout_and_buckets(b2u):
    from unet_pytorch_b200.trainer import FlatBuckets, _backward_order
    shapes = b2u.vgg_unet_param_shapes(21)
    order = _backward_order(list(shapes))
    assert order[0] == "final.weight" and order[-1] == "vgg.features.0.bias"
    assert order.index("up_concat1.conv2.weight") < order.index("up_concat1.conv1.weight") < order.index("up_concat2.conv2.weight")
    lay = FlatBuckets(shapes, order, torch.device("cpu"), bucket_bytes=16 << 20)
    assert lay.total % 4 == 0 and lay.total >= 24_892_437
    covered = 0
    for s, e, names in lay.buckets:
        assert s == covered and e > s
        covered = e
    assert covered == lay.total
    flat = lay.new_buffer()
    views = lay.views(flat)
    views["final.bias"].fill_(3.0)
    o, n, _ = lay.offsets["final.bias"]
    assert flat[o:o + n].eq(3.0).all() and flat.sum().item() == 3.0 * n
    for k, v in views.items():
        assert v.data_ptr() % 16 == 0


def test_per_class_metrics_match_oracle(b2u):
    rng = np.random.default_rng(0)
    hist = rng.integers(0, 1000, size=(21, 21)).astype(np.float64)
    assert np.array_equal(b2u.per_class_iu(hist), O.per_class_iu(hist))
    assert np.array_equal(b2u.per_class_PA_Recall(hist), O.per_class_PA_Recall(hist))
    assert np.array_equal(b2u.per_class_Precision(hist), O.per_class_Precision(hist))


ULU = [("ultralight", "UltraLightweightUnet", 449_810), ("ultralight_large", "UltraLightweightUnet_large", 1_946_322),
       ("ultralight_large_optimized", "UltraLightweightUnet_large_optimized", 926_257)]


@pytest.mark.parametrize("variant,cls,nparams", ULU)
def test_ultralight_state_dict_and_program_contract(b2u, variant, cls, nparams):
    """Module tree, state_dict order and parameter counts of the three UltraLightweightUnet files (2 classes), and the
    static program behind them: every parameter appears exactly once in the backward order, narrow mids are pixel-packed."""
    import importlib
    from unet_pytorch_b200.graph import UltraLightUnetEngine
    Net = getattr(importlib.import_module(f"unet_pytorch_b200.nets.{cls}"), cls)
    m = Net(num_classes=2)
    sd = O.make_ulu_params(2, variant)
    assert list(m.state_dict().keys()) == list(sd.keys())
    assert all(tuple(m.state_dict()[k].shape) == tuple(sd[k].shape) for k in sd)
    assert sum(p.numel() for p in m.parameters()) == nparams
    m.load_state_dict(sd)
    eng = UltraLightUnetEngine(2, variant)
    shapes = eng.param_shapes()
    assert set(shapes) == set(n for n, _ in m.named_parameters())
    assert all(tuple(shapes[n]) == tuple(p.shape) for n, p in m.named_parameters())
    order = eng.backward_param_order()
    assert sorted(order) == sorted(shapes) and len(set(order)) == len(order)
    assert set(eng.buffer_shapes()) == set(n for n, _ in m.named_buffers())
    packed = {i["w"]: i["pix"] for i in eng.pk.values()}
    mids = {"ultralight": {"enc1": 4, "enc2": 2, "dec1": 4, "dec2": 2}, "ultralight_large": {"enc1": 2, "dec1": 2},
            "ultralight_large_optimized": {"enc1": 2, "dec1": 2}}[variant]
    assert packed == {f"{blk}.conv.{sfx}.weight": f for blk, f in mids.items() for sfx in ("0", "3.pointwise")}
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 64, 64))          # CPU tensors: no fallback


def test_lightweight_state_dict_and_program_contract(b2u):
    from unet_pytorch_b200.graph import LightweightUnetEngine
    m = b2u.LightweightUnet(num_classes=21)
    sd = O.make_lw_params(21)
    assert list(m.state_dict().keys()) == list(sd.keys())
    assert sum(p.numel() for p in m.parameters()) == 6_770_756 + (21 - 2) * 25     # SURVEY.md 8(a) a6 counts the 2-class model
    m.load_state_dict(sd)
    m.freeze_backbone()
    assert all(not p.requires_grad for p in m.backbone.parameters()) and m.final_conv[3].weight.requires_grad
    m.unfreeze_backbone()
    assert all(p.requires_grad for p in m.parameters())
    eng = LightweightUnetEngine(21)
    assert sorted(eng.backward_param_order()) == sorted(eng.param_shapes())
    assert sum(1 for i in eng.program if i["op"] == "drop") == 10 and eng.logit_stride == 2
    assert sum(1 for i in eng.program if i["op"] == "se") == 5 + 4 + 1
    with pytest.raises(ValueError):
        b2u.LightweightUnet(num_classes=2, backbone="resnet50")


def test_fused_upsample_planning(b2u):
    """Which "up" instructions the graph engines leave to the decoder conv (b2u_decoder_conv_fprop): only up-sampled tensors read
    exactly once, as the SECOND source of a stride-1 3x3 conv (unetUp, nets/unet.py:16-18) -- Unet-ResNet50's four decoder
    stages and LightweightUnet's (nets/LightWeightUnet.py concatenates [skip, up] too); the UltraLightweight family concatenates
    [up, skip] (up-sampled tensor first) and keeps the separate pass.  Host logic only."""
    from unet_pytorch_b200.graph import LightweightUnetEngine, ResNet50UnetEngine, UltraLightUnetEngine
    from unet_pytorch_b200.engine import VGGUnetEngine
    eng = ResNet50UnetEngine(21)
    assert eng._lazy_up == {"up4": 512, "up3": 256, "up2": 128, "up1": 64}          # name -> padded output channels of the reader
    assert "upc" not in eng._lazy_up                                                # up_conv reads it as its FIRST source
    assert LightweightUnetEngine(2)._lazy_up == {"up4": 192, "up3": 128, "up2": 64, "up1": 64}
    assert not UltraLightUnetEngine(2, variant="ultralight_large")._lazy_up
    # the rule: fuse where the decoder conv has >= 128 output channels
    v = VGGUnetEngine(21)
    assert [v.fuse_upsample(c1.cout_p) for c1, _ in v.dec] == [True, True, True, False]
    assert [eng.fuse_upsample(c) for c in eng._lazy_up.values()] == [True, True, True, False]


def test_conv_tile_count_helper(b2u):
    """b2u_conv_stat_rows (host-only arithmetic): plain convs use M tiles of 16 (w) x 8 (h) pixels, two stacked per step for
    the small-N configs (four for the unmasked N = 64 tiles from 32 rows on); the decoder conv (bit 18 of bn_override) uses
    8 (w) x 16 (h) tiles, stacks of two, or three from 48 rows on."""
    lib = b2u._lib.lib()
    assert lib.b2u_conv_stat_rows(2, 24, 40, 256, 9, 0) == 2 * 3 * 3
    assert lib.b2u_conv_stat_rows(2, 24, 40, 64, 9, 0) == 2 * 2 * 3            # tall: 16-row steps
    assert lib.b2u_conv_stat_rows(2, 100, 40, 64, 9, 0) == 2 * 4 * 3           # 32-row steps
    assert lib.b2u_conv_stat_rows(2, 100, 40, 64, 9, 2 << 16) == 2 * 7 * 3     # bit 17: at most two stacked tiles
    assert lib.b2u_conv_stat_rows(1, 8, 16, 64, 9, 0) == 1                     # H <= 8: one tile per step
    assert lib.b2u_conv_stat_rows(3, 5, 7, 64, 1, 0) == 3                      # 1x1, N tile 64: always two stacked tiles
    assert lib.b2u_conv_stat_rows(3, 5, 7, 192, 1, 0) == 3
    assert lib.b2u_conv_stat_rows(0, 5, 7, 192, 1, 0) == 0
    dec = 1 << 18
    assert lib.b2u_conv_stat_rows(2, 24, 40, 256, 9, dec) == 2 * 2 * 5
    assert lib.b2u_conv_stat_rows(2, 24, 40, 64, 9, dec) == 2 * 1 * 5          # 32-row steps
    assert lib.b2u_conv_stat_rows(2, 100, 40, 64, 9, dec) == 2 * 3 * 5         # 48-row steps
    assert lib.b2u_conv_stat_rows(2, 100, 40, 64, 9, dec | (2 << 16)) == 2 * 4 * 5
    assert lib.b2u_conv_stat_rows(1, 8, 16, 64, 9, dec) == 2


def test_predictor_host_helpers(b2u):
    """Letterbox geometry of the predictor (utils/utils.py:22-34) and its refusal to run without CUDA."""
    from PIL import Image
    from unet_pytorch_b200.unet import Unet as Predictor, resize_image, cvtColor
    img = Image.fromarray(np.zeros((300, 420, 3), np.uint8))
    boxed, nw, nh = resize_image(img, (256, 256))
    assert boxed.size == (256, 256) and (nw, nh) == (256, 182)
    assert np.array(boxed)[0, 0].tolist() == [128, 128, 128]                  # grey bars above/below
    assert cvtColor(Image.fromarray(np.zeros((8, 8), np.uint8))).mode == "RGB"
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            Predictor(state_dict={}, num_classes=2)
