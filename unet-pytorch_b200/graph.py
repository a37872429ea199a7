"""Static-program executor for the networks that are not a plain conv chain: the ResNet50-backbone Unet
(nets/unet.py:24-78 with backbone='resnet50' + nets/resnet.py:55-176 of the reference).

A network is a list of instructions over named tensors (NHWC bf16, channels multiples of 64).  forward() interprets
the list and keeps what backward needs; backward() walks it in reverse, accumulating gradients at tensors that have
several consumers (residual identities, skip connections) with the add kernel.  Every instruction maps to kernels
of libb200unet.so (the conv, BatchNorm and head launches through EngineBase, _engine_base.py, shared with UNetEngine):

  stem      7x7 stride-2 conv as im2col rows (K = 147 -> 192) + 1x1 tensor-core GEMM           nets/resnet.py:109
  conv      1x1 / 3x3, stride 1 or 2 (3x3 s2 = stride-1 conv -> keep even pixels; 1x1 s2 = keep even pixels -> conv),
            bias-free (encoder) or bias + fused ReLU (decoder), optional second source (virtual concat)
  bn        BatchNorm (+ residual add) (+ ReLU), train or eval                                  nets/resnet.py:77-97
  pool3     MaxPool2d(3, 2, 0, ceil_mode=True)                                                  nets/resnet.py:113
  up        UpsamplingBilinear2d(2)                                                             nets/unet.py:13,49
  head      final 1x1 conv -> logits NCHW fp32                                                  nets/unet.py:58,76
  input     NCHW fp32 image -> NHWC bf16, channels zero-padded to 64 (nets that start with a 1x1 conv)
  dw        depthwise 3x3 conv + bias                                         nets/UltraLightweightUnet_large.py:9-10
  se        squeeze-excite: global mean, Linear-ReLU-Linear-Sigmoid, channel scaling              ...:36-52
  drop      nn.Dropout2d (per-(image, channel) mask)                                              ...:78,97
  pool2     MaxPool2d(2, 2)

Channel counts that are not multiples of 64 are zero-padded in the activation buffers and operands (padded channels
stay exactly zero in both directions); parameters and their gradients keep the reference's unpadded shapes.

ReLU handling: a tensor produced by a conv with fused ReLU is marked `fused_relu`; whoever sends a gradient to it
applies the mask (y > 0) on the way (dgrad epilogue / upsample adjoint / head dgrad), so its gradient is always wrt
the pre-activation.  BatchNorm outputs are plain: the bn instruction's own backward applies its ReLU mask.
"""
import torch

from . import ops
from ._engine_base import EngineBase, pad64


class _T:
    __slots__ = ("data", "grad", "fused_relu", "needs_grad", "aux", "stats", "folded", "centered", "low")

    def __init__(self, data, fused_relu=False, needs_grad=False):
        self.data, self.grad, self.fused_relu, self.needs_grad, self.aux = data, None, fused_relu, needs_grad, None
        self.stats = None      # (fp32 per-tile column sums, rows) when the producing conv emitted BatchNorm statistics
        self.folded = False    # eval mode: this conv output already is the BatchNorm (+ReLU) output
        self.centered = False  # training: stored as z - running_mean of the BatchNorm that reads it
        self.low = None        # an "up" output not materialised yet: the low-resolution tensor the reading conv interpolates itself


def resnet50_unet_program(num_classes):
    """Instruction list + conv table of Unet(backbone='resnet50')."""
    P = []
    convs = {}       # weight name -> (cout, cin, taps)

    def conv(out, x, w, cin, cout, taps, stride=1, bias=None, relu=False, x1=None, c1=0):
        convs[w] = (cout, cin, c1, taps)
        P.append(dict(op="conv", out=out, x=x, x1=x1, w=w, bias=bias, cin=cin, c1=c1, cout=cout, taps=taps, stride=stride,
                      relu=relu))

    def bn(out, z, name, c, relu=True, res=None):
        P.append(dict(op="bn", out=out, z=z, bn=name, c=c, relu=relu, res=res))

    P.append(dict(op="stem", out="stem.z", w="resnet.conv1.weight", cout=64))
    bn("feat1", "stem.z", "resnet.bn1", 64)
    P.append(dict(op="pool3", out="pool", x="feat1"))
    x, inplanes = "pool", 64
    feats = ["feat1"]
    for li, (planes, blocks, stride) in enumerate([(64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)], start=1):
        for b in range(blocks):
            pre = f"resnet.layer{li}.{b}"
            s = stride if b == 0 else 1
            conv(pre + ".z1", x, pre + ".conv1.weight", inplanes, planes, 1)
            bn(pre + ".y1", pre + ".z1", pre + ".bn1", planes)
            conv(pre + ".z2", pre + ".y1", pre + ".conv2.weight", planes, planes, 9, stride=s)
            bn(pre + ".y2", pre + ".z2", pre + ".bn2", planes)
            conv(pre + ".z3", pre + ".y2", pre + ".conv3.weight", planes, planes * 4, 1)
            idn = x
            if b == 0:      # downsample branch (nets/resnet.py:134-141): 1x1 conv (stride s) + BN, no ReLU
                conv(pre + ".zd", x, pre + ".downsample.0.weight", inplanes, planes * 4, 1, stride=s)
                bn(pre + ".yd", pre + ".zd", pre + ".downsample.1", planes * 4, relu=False)
                idn = pre + ".yd"
            bn(pre + ".out", pre + ".z3", pre + ".bn3", planes * 4, relu=True, res=idn)
            x, inplanes = pre + ".out", planes * 4
        feats.append(x)
    # decoder: in_filters [192, 512, 1024, 3072], out_filters [64, 128, 256, 512] (nets/unet.py:31-45)
    chans = {"feat1": 64, feats[1]: 256, feats[2]: 512, feats[3]: 1024, feats[4]: 2048}
    low, clow = feats[4], 2048
    for k, co in ((4, 512), (3, 256), (2, 128), (1, 64)):
        skip = feats[k - 1]
        P.append(dict(op="up", out=f"up{k}", x=low))
        conv(f"d{k}a", skip, f"up_concat{k}.conv1.weight", chans[skip], co, 9, bias=f"up_concat{k}.conv1.bias", relu=True,
             x1=f"up{k}", c1=clow)
        conv(f"d{k}b", f"d{k}a", f"up_concat{k}.conv2.weight", co, co, 9, bias=f"up_concat{k}.conv2.bias", relu=True)
        low, clow = f"d{k}b", co
    # up_conv (nets/unet.py:47-54): upsample, conv+ReLU, conv+ReLU at full resolution
    P.append(dict(op="up", out="upc", x=low))
    conv("uc1", "upc", "up_conv.1.weight", 64, 64, 9, bias="up_conv.1.bias", relu=True)
    conv("uc2", "uc1", "up_conv.3.weight", 64, 64, 9, bias="up_conv.3.bias", relu=True)
    P.append(dict(op="head", out="logits", x="uc2", w="final.weight", bias="final.bias"))
    return P, convs


def light_conv_block_ops(P, convs, prefix, x, cin, cout, mid_min, x1=None, c1=0, pack_mid=True):
    """Appends one LightConvBlock (1x1 conv, BN, ReLU, depthwise 3x3, 1x1 conv, BN, ReLU) reading x (and x1: virtual concat).

    pack_mid: a mid width of at most 32 channels is stored at 16 or 32 channels ([N,H,W,64/f], not zero-padded to 64) and the two 1x1 convs
    around it see it as [N,H,W/f,64] with f = 64/mid pixels per row and block-diagonal weights (kron(I_f, W)): the GEMM does
    f x the multiply-adds on zeros, but these layers are HBM-bound and every pass over the mid tensors (conv out, BN
    statistics/apply, depthwise, and all their gradients) moves 1/f of the bytes."""
    def conv(out, xin, w, ci, co, bias, x1=None, c1=0, pk=None, pix=1):
        convs[w] = (co, ci, c1, 1)
        P.append(dict(op="conv", out=out, x=xin, x1=x1, w=w, bias=bias, cin=ci, c1=c1, cout=co, taps=1, stride=1, relu=False,
                      pk=pk, pix=pix))

    mid = max(mid_min, cout // 2)
    if pack_mid and mid <= 32:
        f = 4 if mid <= 16 else 2        # stored width 64 / f (16 or 32 channels; e.g. 22 real channels are padded to 32)
        conv(prefix + ".z1", x, prefix + ".conv.0.weight", cin, mid, prefix + ".conv.0.bias", x1=x1, c1=c1, pk="to", pix=f)
        P.append(dict(op="bn", out=prefix + ".y1", z=prefix + ".z1", bn=prefix + ".conv.1", c=mid, relu=True, res=None))
        P.append(dict(op="dw", out=prefix + ".d", x=prefix + ".y1", w=prefix + ".conv.3.depthwise.weight",
                      bias=prefix + ".conv.3.depthwise.bias", c=mid))
        conv(prefix + ".z2", prefix + ".d", prefix + ".conv.3.pointwise.weight", mid, cout, prefix + ".conv.3.pointwise.bias",
             pk="from", pix=f)
        P.append(dict(op="bn", out=prefix + ".out", z=prefix + ".z2", bn=prefix + ".conv.4", c=cout, relu=True, res=None))
        return prefix + ".out"
    conv(prefix + ".z1", x, prefix + ".conv.0.weight", cin, mid, prefix + ".conv.0.bias", x1=x1, c1=c1)
    P.append(dict(op="bn", out=prefix + ".y1", z=prefix + ".z1", bn=prefix + ".conv.1", c=mid, relu=True, res=None))
    P.append(dict(op="dw", out=prefix + ".d", x=prefix + ".y1", w=prefix + ".conv.3.depthwise.weight",
                  bias=prefix + ".conv.3.depthwise.bias", c=mid))
    conv(prefix + ".z2", prefix + ".d", prefix + ".conv.3.pointwise.weight", mid, cout, prefix + ".conv.3.pointwise.bias")
    P.append(dict(op="bn", out=prefix + ".out", z=prefix + ".z2", bn=prefix + ".conv.4", c=cout, relu=True, res=None))
    return prefix + ".out"


def ultralight_unet_program(num_classes, widths, mid_min, se_rule=None, dropout_p=0.0):
    """UltraLightweightUnet / _large / _large_optimized (nets/UltraLightweightUnet*.py): LightConvBlock stages; optional SE
    after each encoder block; Dropout2d on the bridge; decoder input = cat[upsampled, skip] (upsampled FIRST); 1x1 head.
    se_rule: channels -> reduced channels, or None."""
    P, convs = [], {}

    def block(prefix, x, cin, cout, x1=None, c1=0):
        return light_conv_block_ops(P, convs, prefix, x, cin, cout, mid_min, x1=x1, c1=c1)

    P.append(dict(op="input", out="x", c=3))
    x, cin, skips = "x", 3, []
    for i, w_ in enumerate(widths[:4], start=1):
        if i > 1:
            P.append(dict(op="pool2", out=f"p{i}", x=x))
            x = f"p{i}"
        x = block(f"enc{i}", x, cin, w_)
        if se_rule is not None:
            P.append(dict(op="se", out=f"se{i}.out", x=x, se=f"se{i}", c=w_, r=se_rule(w_)))
            x = f"se{i}.out"
        skips.append((x, w_))
        cin = w_
    P.append(dict(op="pool2", out="p5", x=x))
    x = block("bridge", "p5", cin, widths[4])
    if dropout_p > 0:
        P.append(dict(op="drop", out="bridge.drop", x=x, p=dropout_p))
        x = "bridge.drop"
    clow = widths[4]
    for k in (4, 3, 2, 1):
        skip, cs = skips[k - 1]
        P.append(dict(op="up", out=f"up{k}", x=x))
        x = block(f"dec{k}", f"up{k}", clow, cs, x1=skip, c1=cs)      # cat([up, skip]): nets/UltraLightweightUnet_large.py:100-107
        clow = cs
    P.append(dict(op="head", out="logits", x=x, w="final.weight", bias="final.bias", cin=widths[0]))
    return P, convs


def lightweight_unet_program(num_classes, in_channels=3):
    """LightweightUnet (nets/LightWeightUnet.py:125-177): five stages of ConvBlock (conv3x3+bias, BN, ReLU) + ResidualBlock
    (conv-BN-ReLU-conv-BN-SE, + input, ReLU) + maxpool + Dropout2d(0.1); four decoder stages cat[skip, up2x(low)] ->
    ConvBlock -> ResidualBlock -> Dropout2d; final_conv = ConvBlock, Dropout2d, ResidualBlock, 1x1 conv.  The logits are at
    H/2 x W/2 (every stage, including the first, ends in a maxpool)."""
    P, convs = [], {}
    p_drop = 0.1

    def conv3(out, x, w, cin, cout, bias, x1=None, c1=0):
        convs[w] = (cout, cin, c1, 9)
        P.append(dict(op="conv", out=out, x=x, x1=x1, w=w, bias=bias, cin=cin, c1=c1, cout=cout, taps=9, stride=1, relu=False))

    def conv_block(prefix, x, cin, cout, x1=None, c1=0):
        conv3(prefix + ".z", x, prefix + ".conv.0.weight", cin, cout, prefix + ".conv.0.bias", x1=x1, c1=c1)
        P.append(dict(op="bn", out=prefix + ".y", z=prefix + ".z", bn=prefix + ".conv.1", c=cout, relu=True, res=None))
        return prefix + ".y"

    def res_block(prefix, x, c):
        conv3(prefix + ".z1", x, prefix + ".conv1.weight", c, c, prefix + ".conv1.bias")
        P.append(dict(op="bn", out=prefix + ".y1", z=prefix + ".z1", bn=prefix + ".bn1", c=c, relu=True, res=None))
        conv3(prefix + ".z2", prefix + ".y1", prefix + ".conv2.weight", c, c, prefix + ".conv2.bias")
        P.append(dict(op="bn", out=prefix + ".y2", z=prefix + ".z2", bn=prefix + ".bn2", c=c, relu=False, res=None))
        P.append(dict(op="se", out=prefix + ".s", x=prefix + ".y2", se=prefix + ".se", c=c, r=c // 4))
        P.append(dict(op="addrelu", out=prefix + ".out", a=prefix + ".s", b=x))
        return prefix + ".out"

    def drop(name, x):
        P.append(dict(op="drop", out=name, x=x, p=p_drop))
        return name

    P.append(dict(op="input", out="x", c=in_channels))
    x, cin, feats = "x", in_channels, []
    for k, w_ in enumerate((24, 48, 96, 192, 384), start=1):
        x = conv_block(f"backbone.stage{k}.0", x, cin, w_)
        x = res_block(f"backbone.stage{k}.1", x, w_)
        P.append(dict(op="pool2", out=f"pool{k}", x=x))
        x = drop(f"feat{k}", f"pool{k}")
        feats.append((x, w_))
        cin = w_
    low, clow = feats[4]
    for k in (4, 3, 2, 1):
        skip, cs = feats[k - 1]
        P.append(dict(op="up", out=f"up{k}", x=low))
        x = conv_block(f"up_concat{k}.conv.0", skip, cs, cs, x1=f"up{k}", c1=clow)      # cat([skip, up]): LightWeightUnet.py:120
        x = res_block(f"up_concat{k}.conv.1", x, cs)
        low, clow = drop(f"up_concat{k}.drop", x), cs
    x = conv_block("final_conv.0", low, 24, 24)
    x = drop("final_conv.1", x)
    x = res_block("final_conv.2", x, 24)
    P.append(dict(op="head", out="logits", x=x, w="final_conv.3.weight", bias="final_conv.3.bias", cin=24))
    return P, convs


def improved_segnet_program(num_classes, deploy=False):
    """ImprovedSegNet(use_repvgg=True) of nets/RepVGG_Unet.py:149-206 (8(f) rank 4, "RepVGG deploy re-param"): the topology of
    UltraLightweightUnet_large_optimized (widths 44-88-176-352-704, SE after the encoder stages, Dropout2d(0.15) on the bridge,
    cat[upsampled, skip]) with LightweightConvBlock = 1x1 conv (+bias) -> BN -> ReLU -> RepVGGBlock(mid -> out), mid = max(16, out // 2).
    RepVGGBlock (training form, :25-60): relu(bn1(conv3x3(x)) + bn2(conv1x1(x))) -- both convs bias-free; the identity branch only
    exists when mid == out, which none of these blocks has.  Deploy form (:67-73): one conv3x3 + bias + ReLU (`reparam_conv`)."""
    widths = (44, 88, 176, 352, 704)
    P, convs = [], {}

    def conv(out, x, w, ci, co, taps, bias=None, relu=False, x1=None, c1=0):
        convs[w] = (co, ci, c1, taps)
        P.append(dict(op="conv", out=out, x=x, x1=x1, w=w, bias=bias, cin=ci, c1=c1, cout=co, taps=taps, stride=1, relu=relu))

    def bn(out, z, name, c, relu=True, res=None):
        P.append(dict(op="bn", out=out, z=z, bn=name, c=c, relu=relu, res=res))

    def block(p, x, cin, cout, x1=None, c1=0):
        mid = max(16, cout // 2)
        if mid == cout:
            raise NotImplementedError("RepVGGBlock identity branch (in == out channels) is not used by ImprovedSegNet")
        conv(p + ".z0", x, p + ".conv.0.weight", cin, mid, 1, bias=p + ".conv.0.bias", x1=x1, c1=c1)
        bn(p + ".y0", p + ".z0", p + ".conv.1", mid)
        rep = p + ".conv.3"
        if deploy:
            conv(p + ".out", p + ".y0", rep + ".reparam_conv.weight", mid, cout, 9, bias=rep + ".reparam_conv.bias", relu=True)
            return p + ".out"
        conv(p + ".z1", p + ".y0", rep + ".conv2.weight", mid, cout, 1)                 # 1x1 branch
        bn(p + ".y1", p + ".z1", rep + ".bn2", cout, relu=False)
        conv(p + ".z3", p + ".y0", rep + ".conv1.weight", mid, cout, 9)                 # 3x3 branch
        bn(p + ".out", p + ".z3", rep + ".bn1", cout, relu=True, res=p + ".y1")         # relu(bn1(.) + bn2(.))
        return p + ".out"

    P.append(dict(op="input", out="x", c=3))
    x, cin, skips = "x", 3, []
    for i, w_ in enumerate(widths[:4], start=1):
        if i > 1:
            P.append(dict(op="pool2", out=f"p{i}", x=x))
            x = f"p{i}"
        x = block(f"enc{i}", x, cin, w_)
        P.append(dict(op="se", out=f"se{i}.out", x=x, se=f"se{i}", c=w_, r=max(8, w_ // 4)))
        x = f"se{i}.out"
        skips.append((x, w_))
        cin = w_
    P.append(dict(op="pool2", out="p5", x=x))
    x = block("bridge", "p5", cin, widths[4])
    P.append(dict(op="drop", out="bridge.drop", x=x, p=0.15))
    x, clow = "bridge.drop", widths[4]
    for k in (4, 3, 2, 1):
        skip, cs = skips[k - 1]
        P.append(dict(op="up", out=f"up{k}", x=x))
        x = block(f"dec{k}", f"up{k}", clow, cs, x1=skip, c1=cs)
        clow = cs
    P.append(dict(op="head", out="logits", x=x, w="final.weight", bias="final.bias", cin=widths[0]))
    return P, convs


ULU_VARIANTS = {
    # name: (widths, minimum mid channels, SE reduction rule, bridge dropout)
    "ultralight": ((32, 64, 128, 256, 512), 8, None, 0.0),                                     # UltraLightweightUnet.py
    "ultralight_large": ((64, 128, 256, 512, 1024), 16, lambda c: max(8, c // 4), 0.2),        # ..._large.py
    "ultralight_large_optimized": ((44, 88, 176, 352, 704), 16, lambda c: max(8, c // 4), 0.15),   # ..._large_optimized.py
}


class GraphEngine(EngineBase):
    def __init__(self, program, convs, num_classes, device=None, first_trainable_prefix=None):
        super().__init__(device)
        self.program, self.convs, self.num_classes = program, convs, num_classes
        self._packed = {}            # weight name -> (wf, wd)
        self.has_stem = any(i["op"] == "stem" for i in program)
        self.in_channels = next((i["c"] for i in program if i["op"] == "input"), 3)      # the stem (ResNet) takes RGB
        self.pk = {i["w"]: i for i in program if i["op"] == "conv" and i.get("pk")}     # pixel-packed 1x1 convs
        # convs that read the image: the input instruction stores the image as a two-term bf16 split (hi in channels [0, C),
        # lo = x - hi in [C, 2C)), so their weights are repeated over the second channel range and the MMA sees the image
        # to ~2^-17 (a single bf16 rounding of the image alone costs these nets 5e-2 of gradient accuracy)
        inputs = {i["out"]: i["c"] for i in program if i["op"] == "input"}
        self.image_convs = {i["w"]: inputs[i["x"]] for i in program if i["op"] == "conv" and i["x"] in inputs and 2 * inputs[i["x"]] <= 64}
        self.dropout_override = None
        readers = {}
        for i in program:
            for key in ("x", "x1", "z", "res", "a", "b"):
                if i.get(key):
                    readers.setdefault(i[key], []).append(i["op"] if key == "z" else "other")
        self._pre_bn = {name for name, ops_ in readers.items() if ops_ == ["bn"]}      # tensors read only as a BN input
        # eval-mode folding: conv output -> the BatchNorm (without residual) that is its only reader
        self._fold_bn = {i["z"]: i for i in program if i["op"] == "bn" and i["z"] in self._pre_bn and not i["res"]}
        self._bn_reader = {i["z"]: i for i in program if i["op"] == "bn" and i["z"] in self._pre_bn}      # conv output -> its BatchNorm
        # "up" outputs read exactly once, as the SECOND source of a stride-1 3x3 conv (unetUp, nets/unet.py:16-18) -> padded
        # output channels of that conv: where fuse_upsample() says so, the conv interpolates the low-resolution tensor in its
        # producer warps (b2u_decoder_conv_fprop) and the "up" instruction launches nothing
        ups = {i["out"] for i in program if i["op"] == "up"}
        self._lazy_up = {i["x1"]: pad64(i["cout"]) for i in program if i["op"] == "conv" and i.get("x1") in ups
                         and len(readers.get(i["x1"], [])) == 1 and i["taps"] == 9 and i["stride"] == 1 and not i.get("pk")}

    # ------------------------------------------------------------------ static description
    def param_shapes(self):
        shapes = {}
        for ins in self.program:
            op = ins["op"]
            if op == "stem":
                shapes[ins["w"]] = (ins["cout"], 3, 7, 7)
            elif op == "conv":
                k = 3 if ins["taps"] == 9 else 1
                shapes[ins["w"]] = (ins["cout"], ins["cin"] + ins["c1"], k, k)
                if ins["bias"]:
                    shapes[ins["bias"]] = (ins["cout"],)
            elif op == "bn":
                shapes[ins["bn"] + ".weight"] = (ins["c"],)
                shapes[ins["bn"] + ".bias"] = (ins["c"],)
            elif op == "dw":
                shapes[ins["w"]] = (ins["c"], 1, 3, 3)
                shapes[ins["bias"]] = (ins["c"],)
            elif op == "se":
                shapes[ins["se"] + ".fc.0.weight"] = (ins["r"], ins["c"])
                shapes[ins["se"] + ".fc.0.bias"] = (ins["r"],)
                shapes[ins["se"] + ".fc.2.weight"] = (ins["c"], ins["r"])
                shapes[ins["se"] + ".fc.2.bias"] = (ins["c"],)
            elif op == "head":
                shapes[ins["w"]] = (self.num_classes, ins.get("cin", 64), 1, 1)
                shapes[ins["bias"]] = (self.num_classes,)
        return shapes

    def buffer_shapes(self):
        shapes = {}
        for ins in self.program:
            if ins["op"] == "bn":
                shapes[ins["bn"] + ".running_mean"] = (ins["c"],)
                shapes[ins["bn"] + ".running_var"] = (ins["c"],)
                shapes[ins["bn"] + ".num_batches_tracked"] = ()
        return shapes

    def backward_param_order(self):
        out = []
        for ins in reversed(self.program):
            op = ins["op"]
            if op == "head":
                out += [ins["w"], ins["bias"]]
            elif op == "conv":
                out += [ins["w"]] + ([ins["bias"]] if ins["bias"] else [])
            elif op == "bn":
                out += [ins["bn"] + ".weight", ins["bn"] + ".bias"]
            elif op == "dw":
                out += [ins["w"], ins["bias"]]
            elif op == "se":
                out += [ins["se"] + ".fc.0.weight", ins["se"] + ".fc.0.bias", ins["se"] + ".fc.2.weight", ins["se"] + ".fc.2.bias"]
            elif op == "stem":
                out += [ins["w"]]
        return out

    # ------------------------------------------------------------------ buffers
    def _center_shift(self, ins, params, training, width):
        """Padded running mean of the BatchNorm that is the only reader of this conv's output (training, bf16 path), or None."""
        bn_ins = self._bn_reader.get(ins["out"])
        if bn_ins is None or not self.center_pre_bn(training):
            return None
        return self._padded("rm:" + bn_ins["bn"], params[bn_ins["bn"] + ".running_mean"], (width,))

    def _tiled(self, key, t, width, f):
        """fp32 vector zero-padded to `width` and repeated f times (bias of a pixel-packed conv)."""
        b = self._bufs.get(key)
        if b is None or b.numel() != width * f:
            b = torch.zeros((f, width), dtype=torch.float32, device=self.device)
            self._bufs[key] = b
        b[:, :t.numel()].copy_(t.reshape(1, -1).expand(f, -1))
        return b.view(-1)

    # ------------------------------------------------------------------ weights
    def pack(self, params, need_dgrad=True):
        names = list(self.convs.keys())
        key = tuple(params[n].data_ptr() for n in names) + (need_dgrad,)
        versions = tuple(params[n]._version for n in names)
        if self.has_stem:
            versions += (params["resnet.conv1.weight"]._version,)
        if self._pack_key == key and self._pack_versions == versions:
            return
        dev = params[names[0]].device
        if self._pack_key != key:
            layers = []
            for n in names:
                cout, c0, c1, taps = self.convs[n]
                c0p, c1p, coutp = pad64(c0), (pad64(c1) if c1 else 0), pad64(cout)
                src = params[n]
                if n in self.image_convs and n not in self.pk:      # [w | w] over the hi / lo halves of the image split
                    ci = self.image_convs[n]
                    k = 3 if taps == 9 else 1
                    src = self._bufs.get("w2:" + n)
                    if src is None or tuple(src.shape) != (cout, 2 * ci, k, k):
                        src = torch.zeros((cout, 2 * ci, k, k), dtype=torch.float32, device=dev)
                        self._bufs["w2:" + n] = src
                    c0 = 2 * ci
                if n in self.pk:            # the view problem: block-diagonal weights over f pixels (built below)
                    f, kind = self.pk[n]["pix"], self.pk[n]["pk"]
                    if kind == "to":        # dense 64-padded inputs -> packed `cout` (= mid) channels
                        cout, c0, c1 = 64, f * c0p, f * c1p
                    else:                   # packed `c0` (= mid) channels -> dense 64-padded outputs
                        cout, c0, c1 = f * coutp, 64, 0
                    c0p, c1p, coutp = c0, c1, cout
                    src = self._bufs.get("w2:" + n)
                    if src is None or tuple(src.shape) != (cout, c0 + c1, 1, 1):
                        src = torch.zeros((cout, c0 + c1, 1, 1), dtype=torch.float32, device=dev)
                        self._bufs["w2:" + n] = src
                wf, wd = self._packed.get(n, (None, None))
                if wf is None:
                    wf = torch.zeros((coutp, taps * (c0p + c1p)), dtype=ops.act_dtype(), device=dev)
                if need_dgrad and wd is None:
                    wd = torch.zeros((c0p + c1p, taps * coutp), dtype=ops.act_dtype(), device=dev)
                self._packed[n] = (wf, wd)
                layers.append((src, wf, wd if need_dgrad else None, cout, c0 + c1, taps, False, c0, c0p, c0p + c1p, coutp))
            self._set_pack_table(layers, dev)
            self._pack_key = key
        for n, ci in self.image_convs.items():   # refresh [w | w]
            if n not in self.pk:
                w2, w = self._bufs["w2:" + n], params[n]
                w2[:, :ci].copy_(w); w2[:, ci:].copy_(w)
        for n, ins in self.pk.items():          # refresh the block-diagonal fp32 weights kron(I_f, W) of the packed convs
            f, w2, w = ins["pix"], self._bufs["w2:" + n], params[n]
            midp = 64 // f
            if ins["pk"] == "to":
                mid, c0r, c1r = ins["cout"], ins["cin"], ins["c1"]
                c0p, c1p = pad64(c0r), (pad64(c1r) if c1r else 0)
                for k in range(f):
                    w2[k * midp:k * midp + mid, k * c0p:k * c0p + c0r].copy_(w[:, :c0r])
                    if n in self.image_convs:      # lo half of the image split: same weights
                        w2[k * midp:k * midp + mid, k * c0p + c0r:k * c0p + 2 * c0r].copy_(w[:, :c0r])
                    if c1r:
                        w2[k * midp:k * midp + mid, f * c0p + k * c1p:f * c0p + k * c1p + c1r].copy_(w[:, c0r:])
            else:
                mid, co, cop = ins["cin"], ins["cout"], pad64(ins["cout"])
                for k in range(f):
                    w2[k * cop:k * cop + co, k * midp:k * midp + mid].copy_(w)
        self._launch_pack()
        if self.has_stem:
            self._stem_wf = ops.pack_weights_im2col(params["resnet.conv1.weight"], 192, wf=getattr(self, "_stem_wf", None))
        self._pack_versions = versions

    # ------------------------------------------------------------------ forward
    def forward(self, x, params, save=True, training=None, trainable=None, input_grad=False):
        """input_grad: backward() will be asked for the gradient wrt x, so the image (the input instruction's tensor, or
        the stem's output) needs a gradient and every layer between it and the loss runs its data gradient."""
        if not x.is_cuda:
            raise ValueError("GraphEngine.forward: input must be a CUDA tensor (no CPU fallback)")
        x = x.float().contiguous() if x.dtype != torch.float32 else x.contiguous()
        N, C, H, W = x.shape
        if C != self.in_channels or H % 32 or W % 32:
            raise ValueError(f"expected a {self.in_channels}-channel image with height and width multiples of 32")
        if training is None:
            training = save
        if trainable is None:
            trainable = set(self.param_shapes().keys())
        self.device = x.device
        self.pack(params, need_dgrad=save)
        T = {}
        logits = None
        for ins in self.program:
            op = ins["op"]
            if op == "stem":
                col = ops.im2col_stem(x, out=self._buf("stem.col", (N, H // 2, W // 2, 192)))
                z = self._buf(ins["out"], (N, H // 2, W // 2, 64))
                shift = self._center_shift(ins, params, training, 64)
                sbias = torch.neg(shift, out=self._buf("bc:" + ins["w"], (64,), torch.float32)) if shift is not None else None
                ops.conv_fprop(col, self._stem_wf, sbias, 64, taps=1, relu=False, out=z)
                t = _T(z, needs_grad=ins["w"] in trainable or input_grad)
                t.centered = shift is not None
                t.aux = col
                T[ins["out"]] = t
            elif op == "input":
                T[ins["out"]] = _T(ops.nchw_to_nhwc_bf16_padded(x, 64, out=self._buf("x", (N, H, W, 64))),      # hi | lo split when 2C <= 64
                                   needs_grad=input_grad)
            elif op == "conv":
                xin = T[ins["x"]]
                x1 = T[ins["x1"]] if ins["x1"] else None
                wf, _ = self._packed[ins["w"]]
                n, h, w, _ = xin.data.shape
                ng = xin.needs_grad or (x1 is not None and x1.needs_grad) or ins["w"] in trainable or (ins["bias"] in trainable)
                # folding is for pure inference: an eval-mode forward that will be back-propagated (model.eval() +
                # loss.backward()) keeps z and runs the BatchNorm instruction so its backward has what it needs
                fold = self._fold_bn.get(ins["out"]) if (not training and not save) else None
                scale, relu = None, ins["relu"]
                if ins.get("pk"):           # pixel-packed 1x1 conv: every tensor is viewed with f pixels per row
                    f = ins["pix"]
                    if ins["pk"] == "to":
                        z = self._buf(ins["out"], (n, h, w, 64 // f))               # 16 or 32 stored channels
                        bias = self._tiled("b2:" + ins["w"], params[ins["bias"]], 64 // f, f)
                    else:
                        z = self._buf(ins["out"], (n, h, w, pad64(ins["cout"])))
                        bias = self._tiled("b2:" + ins["w"], params[ins["bias"]], pad64(ins["cout"]), f)
                    shift = self._center_shift(ins, params, training, z.shape[3])
                    if shift is not None:
                        bias = torch.sub(bias, self._tiled("c2:" + ins["w"], shift, z.shape[3], f), out=self._buf("bc:" + ins["w"], (bias.numel(),), torch.float32))
                    if fold is not None:        # eval: BatchNorm (+ReLU) folded into the epilogue, vectors tiled like the bias
                        sc, bs = self._folded_bn(fold["bn"], params, params[ins["bias"]], z.shape[3])
                        scale = self._tiled("fs2:" + ins["w"], sc, z.shape[3], f)
                        bias = self._tiled("fb2:" + ins["w"], bs, z.shape[3], f)
                        relu = fold["relu"]
                    self._conv_fwd(xin.data.view(n, h, w // f, -1), wf, bias, z.shape[3] * f, 1, relu, z.view(n, h, w // f, -1),
                                   x1=x1.data.view(n, h, w // f, -1) if x1 else None, scale=scale)
                    t = _T(z, needs_grad=ng)
                    t.folded = fold is not None
                    t.centered = shift is not None
                    T[ins["out"]] = t
                    continue
                coutp = pad64(ins["cout"])
                bias = self._padded("b:" + ins["w"], params[ins["bias"]], (coutp,)) if ins["bias"] else None
                low = up_out = None
                if x1 is not None and x1.data is None:
                    # second source = upsample2x(low), interpolated inside the conv; the up-sampled tensor is written (as a
                    # by-product) only when a backward pass needs it as the weight gradient's operand
                    low = x1.low
                    if save or ops.act_dtype() == torch.float32:
                        up_out = self._buf(ins["x1"], (n, h, w, low.shape[3]))
                    if bias is None:
                        bias = self._bufs.get("b0:" + ins["w"])
                        if bias is None or bias.numel() != coutp:
                            bias = self._bufs["b0:" + ins["w"]] = torch.zeros((coutp,), dtype=torch.float32, device=self.device)
                shift = self._center_shift(ins, params, training, coutp)
                if shift is not None:
                    cb = self._buf("bc:" + ins["w"], (coutp,), torch.float32)
                    bias = torch.sub(bias, shift, out=cb) if bias is not None else torch.neg(shift, out=cb)
                if fold is not None:
                    # eval mode: y = [relu](acc * s + b') straight from the conv epilogue; the BatchNorm instruction passes it on
                    scale, bias = self._folded_bn(fold["bn"], params, params[ins["bias"]] if ins["bias"] else None, coutp)
                    relu = fold["relu"]
                aux = stats = None
                if ins["stride"] == 1:
                    z = self._buf(ins["out"], (n, h, w, coutp))
                    kdim = ins["taps"] * (xin.data.shape[3] + (low.shape[3] if low is not None else x1.data.shape[3] if x1 else 0))
                    if ins["out"] in self._pre_bn and self.fuse_bn_stats(training, kdim, coutp):
                        # the BatchNorm that reads this output takes its statistics from this conv's epilogue (no pass over
                        # z); one buffer per conv output: another conv may run before that BatchNorm (downsample branches)
                        stats = self._bn_stats("bnstat:" + ins["out"], n, h, w, coutp, ins["taps"], decoder=low is not None)
                    self._conv_fwd(xin.data, wf, bias, coutp, ins["taps"], relu, z, x1=x1.data if x1 else None, low=low,
                                   up_out=up_out, scale=scale, stats=stats)
                    if low is not None:
                        x1.data = up_out
                elif ins["taps"] == 9:      # 3x3 stride 2 = stride-1 conv, keep even pixels
                    full = self._buf(ins["out"] + ":full", (n, h, w, coutp))
                    self._conv_fwd(xin.data, wf, bias, coutp, 9, relu, full, scale=scale)
                    z = ops.subsample2(full, out=self._buf(ins["out"], (n, h // 2, w // 2, coutp)))
                else:                        # 1x1 stride 2 = keep even pixels, then conv
                    aux = ops.subsample2(xin.data, out=self._buf(ins["out"] + ":xs", (n, h // 2, w // 2, xin.data.shape[3])))
                    z = self._buf(ins["out"], (n, h // 2, w // 2, coutp))
                    self._conv_fwd(aux, wf, bias, coutp, 1, relu, z, scale=scale)
                t = _T(z, fused_relu=ins["relu"], needs_grad=ng)
                t.aux = aux
                t.stats = stats
                t.folded = fold is not None
                t.centered = shift is not None
                T[ins["out"]] = t
            elif op == "bn":
                zt = T[ins["z"]]
                if zt.folded:            # eval mode: the producing conv already applied this BatchNorm (+ReLU)
                    T[ins["out"]] = _T(zt.data)
                    continue
                res = T[ins["res"]] if ins["res"] else None
                bnn = ins["bn"]
                y = self._buf(ins["out"], zt.data.shape)
                aux = self._bn_fwd(bnn, zt.data, params, training, ins["relu"], y, residual=res.data if res else None,
                                   stats=zt.stats, centered=zt.centered)
                ng = zt.needs_grad or (res is not None and res.needs_grad) or (bnn + ".weight") in trainable or (bnn + ".bias") in trainable
                t = _T(y, needs_grad=ng)
                t.aux = aux
                T[ins["out"]] = t
            elif op == "dw":
                xin = T[ins["x"]]
                c, cp = ins["c"], xin.data.shape[3]
                wdw = self._padded("dw:" + ins["w"], params[ins["w"]].reshape(c, 9), (cp, 9))
                bdw = self._padded("dwb:" + ins["w"], params[ins["bias"]], (cp,))
                y = ops.dwconv3x3(xin.data, wdw, bdw, out=self._buf(ins["out"], xin.data.shape))
                t = _T(y, needs_grad=xin.needs_grad or ins["w"] in trainable or ins["bias"] in trainable)
                t.aux = wdw
                T[ins["out"]] = t
            elif op == "se":
                xin = T[ins["x"]]
                n, h, w, cp = xin.data.shape
                se, c = ins["se"], ins["c"]
                ws = self._workspace("spatial", ops.lib().b2u_spatial_reduce_workspace_floats(n, cp) * 4)
                pooled = ops.spatial_reduce(xin.data, scale=1.0 / (h * w), ws=ws)
                hidden, sc = ops.se_fc_fwd(pooled, params[se + ".fc.0.weight"], params[se + ".fc.0.bias"],
                                           params[se + ".fc.2.weight"], params[se + ".fc.2.bias"], c)
                y = ops.scale_nc(xin.data, sc, out=self._buf(ins["out"], xin.data.shape))
                t = _T(y, needs_grad=xin.needs_grad or any((se + s_) in trainable for s_ in (".fc.0.weight", ".fc.0.bias", ".fc.2.weight", ".fc.2.bias")))
                t.aux = (pooled, hidden, sc)
                T[ins["out"]] = t
            elif op == "drop":
                xin = T[ins["x"]]
                if training and ins["p"] > 0:
                    n, h, w, cp = xin.data.shape
                    keep = 1.0 - ins["p"]
                    ov = self.dropout_override
                    if isinstance(ov, dict):
                        ov = ov.get(ins["out"])
                    if ov is not None:       # tests replay the multiplier the reference drew ([N, C])
                        mask = torch.zeros((n, cp), dtype=torch.float32, device=self.device)
                        mask[:, :ov.shape[1]] = ov.to(self.device)
                    else:
                        mask = torch.bernoulli(torch.full((n, cp), keep, dtype=torch.float32, device=self.device)) / keep
                    y = ops.scale_nc(xin.data, mask, out=self._buf(ins["out"], xin.data.shape))
                    t = _T(y, needs_grad=xin.needs_grad)
                    t.aux = mask
                else:
                    t = _T(xin.data, needs_grad=xin.needs_grad)
                    t.aux = None
                T[ins["out"]] = t
            elif op == "addrelu":
                a, b = T[ins["a"]], T[ins["b"]]
                y = ops.add_relu(a.data, b.data, out=self._buf(ins["out"], a.data.shape))
                T[ins["out"]] = _T(y, needs_grad=a.needs_grad or b.needs_grad)
            elif op == "pool3":
                xin = T[ins["x"]]
                n, h, w, c = xin.data.shape
                y = ops.maxpool3x3s2(xin.data, out=self._buf(ins["out"], (n, (h - 2) // 2 + 1, (w - 2) // 2 + 1, c)))
                T[ins["out"]] = _T(y, needs_grad=xin.needs_grad)
            elif op == "pool2":
                xin = T[ins["x"]]
                n, h, w, c = xin.data.shape
                y = ops.maxpool2x2(xin.data, out=self._buf(ins["out"], (n, h // 2, w // 2, c)))
                T[ins["out"]] = _T(y, needs_grad=xin.needs_grad)
            elif op == "up":
                xin = T[ins["x"]]
                n, h, w, c = xin.data.shape
                if ins["out"] in self._lazy_up and self.fuse_upsample(self._lazy_up[ins["out"]]):
                    t = _T(None, needs_grad=xin.needs_grad)          # the reading conv interpolates xin itself
                    t.low = xin.data
                    T[ins["out"]] = t
                    continue
                y = ops.upsample2x(xin.data, out=self._buf(ins["out"], (n, 2 * h, 2 * w, c)))
                T[ins["out"]] = _T(y, needs_grad=xin.needs_grad)
            elif op == "head":
                logits = self._head_fwd(T[ins["x"]].data, params, ins["w"], ins["bias"], ins.get("cin", 64))
        if save:
            self.saved = (T, (N, H, W), set(trainable), input_grad)
        return logits

    # ------------------------------------------------------------------ backward
    def _acc(self, t, g):
        if t.grad is None:
            t.grad = g
        else:
            ops.add_bf16(t.grad, g, out=t.grad)

    def backward(self, dlogits, params, grads, trainable=None, on_grads_ready=None, dx=None):
        """grads: name -> fp32 tensor to overwrite (missing / not in `trainable`: skipped).  dx (optional, needs a forward
        with input_grad=True): NCHW fp32 buffer shaped like the input, receives the gradient wrt the image."""
        if self.saved is None:
            raise RuntimeError("backward() without a saved forward()")
        T, (N, H, W), fwd_trainable, input_grad = self.saved
        if dx is not None and not input_grad:
            raise RuntimeError("backward(dx=...) needs a forward(input_grad=True)")
        if trainable is None:
            trainable = set(grads.keys())
        for t in T.values():
            t.grad = None

        def has(n):
            return n is not None and n in trainable and n in grads

        def ready(*names):
            if on_grads_ready is not None:
                on_grads_ready([n for n in names if n in grads])

        dx_written = False
        for ins in reversed(self.program):
            op = ins["op"]
            if op == "head":
                xin = T[ins["x"]]
                g = self._buf("g:" + ins["x"], xin.data.shape) if xin.needs_grad else None
                self._head_bwd(dlogits, xin.data, params, grads, has, ins["w"], ins["bias"], ins.get("cin", 64), g,
                               xin.data if xin.fused_relu else None)
                if g is not None:
                    self._acc(xin, g)
                ready(ins["w"], ins["bias"])
            elif op == "up":
                t, xin = T[ins["out"]], T[ins["x"]]
                if t.grad is None or not xin.needs_grad:
                    continue
                g = self._buf("g:" + ins["out"] + ">", xin.data.shape)
                ops.upsample2x_bwd(t.grad, ylow=xin.data if xin.fused_relu else None, out=g)
                self._acc(xin, g)
            elif op == "addrelu":
                t, a, b = T[ins["out"]], T[ins["a"]], T[ins["b"]]
                if t.grad is None:
                    continue
                # both inputs receive dy * (y > 0).  They may share this buffer: `a` (the SE output) is consumed by the
                # next backward instruction, before anything accumulates into `b` (the block input) in place.
                g = ops.relu_bwd(t.grad, t.data, out=self._buf("g:" + ins["out"] + ">", t.data.shape))
                if a.needs_grad:
                    self._acc(a, g)
                if b.needs_grad:
                    self._acc(b, g)
            elif op == "pool3":
                t, xin = T[ins["out"]], T[ins["x"]]
                if t.grad is None or not xin.needs_grad:
                    continue
                g = ops.maxpool3x3s2_bwd(t.grad, xin.data, out=self._buf("g:" + ins["out"] + ">", xin.data.shape))
                self._acc(xin, g)
            elif op == "pool2":
                t, xin = T[ins["out"]], T[ins["x"]]
                if t.grad is None or not xin.needs_grad:
                    continue
                # the gradient already accumulated at the pooled tensor (its skip consumer) is added in the same pass
                g = ops.maxpool2x2_bwd(t.grad, xin.data, dskip=xin.grad, relu_mask=xin.fused_relu,
                                       out=self._buf("g:" + ins["out"] + ">", xin.data.shape))
                xin.grad = g
            elif op == "drop":
                t, xin = T[ins["out"]], T[ins["x"]]
                if t.grad is None or not xin.needs_grad:
                    continue
                if t.aux is None:
                    g = t.grad
                else:
                    g = ops.scale_nc(t.grad, t.aux, out=self._buf("g:" + ins["out"] + ">", xin.data.shape))
                self._acc(xin, self._relu_mask(xin, g, ins["out"]))
            elif op == "se":
                t, xin = T[ins["out"]], T[ins["x"]]
                if t.grad is None:
                    continue
                se, c = ins["se"], ins["c"]
                pooled, hidden, sc = t.aux
                n, h, w, cp = xin.data.shape
                ws = self._workspace("spatial", ops.lib().b2u_spatial_reduce_workspace_floats(n, cp) * 4)
                dscale = ops.spatial_reduce(t.grad, xin.data, ws=ws)
                names = [se + ".fc.0.weight", se + ".fc.0.bias", se + ".fc.2.weight", se + ".fc.2.bias"]
                dpooled = ops.se_fc_bwd(dscale, pooled, hidden, sc, params[names[0]], params[names[2]], c, 1.0 / (h * w),
                                        dw1=grads[names[0]] if has(names[0]) else None, db1=grads[names[1]] if has(names[1]) else None,
                                        dw2=grads[names[2]] if has(names[2]) else None, db2=grads[names[3]] if has(names[3]) else None)
                ready(*names)
                if xin.needs_grad:
                    g = ops.scale_nc(t.grad, sc, add=dpooled, out=self._buf("g:" + ins["out"] + ">", xin.data.shape))
                    self._acc(xin, self._relu_mask(xin, g, ins["out"]))
            elif op == "dw":
                t, xin = T[ins["out"]], T[ins["x"]]
                if t.grad is None:
                    continue
                c, cp = ins["c"], xin.data.shape[3]
                if has(ins["w"]) or has(ins["bias"]):
                    dwp = self._buf("dwg:" + ins["w"], (cp, 9), torch.float32)
                    dbp = self._buf("dwgb:" + ins["w"], (cp,), torch.float32)
                    ops.dwconv3x3_wgrad(xin.data, t.grad, dw=dwp, db=dbp,
                                        ws=self._workspace("dwgrad", ops.lib().b2u_dwconv3x3_wgrad_workspace(cp)))
                    if has(ins["w"]):
                        grads[ins["w"]].copy_(dwp[:c].reshape(c, 1, 3, 3))
                    if has(ins["bias"]):
                        grads[ins["bias"]].copy_(dbp[:c])
                ready(ins["w"], ins["bias"])
                if xin.needs_grad:
                    g = ops.dwconv3x3(t.grad, t.aux, None, flip=True, out=self._buf("g:" + ins["out"] + ">", xin.data.shape))
                    self._acc(xin, g)
            elif op == "bn":
                t, zt = T[ins["out"]], T[ins["z"]]
                res = T[ins["res"]] if ins["res"] else None
                if t.grad is None:
                    continue
                bnn = ins["bn"]
                need_res = res is not None and res.needs_grad
                gout = self._buf("g:" + ins["out"] + ">res", t.data.shape) if need_res else None
                dz = self._buf("g:" + ins["z"], zt.data.shape)
                self._bn_bwd(t.grad, t.data, zt.data, t.aux, ins["relu"], dz, grads, has, bnn, ins["c"], residual=res is not None,
                             gout=gout)
                ready(bnn + ".weight", bnn + ".bias")
                if zt.needs_grad:
                    self._acc(zt, dz)
                if need_res:
                    self._acc(res, gout)
            elif op == "conv":
                t, xin = T[ins["out"]], T[ins["x"]]
                x1 = T[ins["x1"]] if ins["x1"] else None
                if t.grad is None:
                    continue
                dz = t.grad
                wf, wd = self._packed[ins["w"]]
                n, h, w, _ = xin.data.shape
                taps, cout, c0r, c1r = ins["taps"], ins["cout"], ins["cin"], ins["c1"]
                if ins.get("pk"):
                    # pixel-packed 1x1 conv: wgrad / dgrad of the view problem (f pixels per row, block-diagonal weights);
                    # the real weight gradient is the sum of the f diagonal blocks
                    f = ins["pix"]
                    xv = xin.data.view(n, h, w // f, -1)
                    x1v = x1.data.view(n, h, w // f, -1) if x1 else None
                    dzv = dz.view(n, h, w // f, -1)
                    cin_v = xv.shape[3] + (x1v.shape[3] if x1 else 0)
                    if has(ins["w"]):
                        need = ops.lib().b2u_conv_wgrad_workspace(n, h, w // f, cin_v, dzv.shape[3], 1)
                        tmp = self._buf("dw:" + ins["w"], (dzv.shape[3], cin_v, 1, 1), torch.float32)
                        ops.conv_wgrad(xv, dzv, taps=1, x1=x1v, dw=tmp, ws=self._workspace("wgrad", need))
                        gw = grads[ins["w"]]
                        midp = 64 // f
                        if ins["pk"] == "to":
                            mid, c0p = cout, xin.data.shape[3]
                            c1p = x1.data.shape[3] if x1 else 0
                            for k in range(f):
                                blk = tmp[k * midp:k * midp + mid]
                                if k == 0:
                                    gw[:, :c0r].copy_(blk[:, k * c0p:k * c0p + c0r])
                                else:
                                    gw[:, :c0r].add_(blk[:, k * c0p:k * c0p + c0r])
                                if ins["w"] in self.image_convs:      # + the lo half of the image split
                                    gw[:, :c0r].add_(blk[:, k * c0p + c0r:k * c0p + 2 * c0r])
                                if c1r:
                                    src = blk[:, f * c0p + k * c1p:f * c0p + k * c1p + c1r]
                                    if k == 0:
                                        gw[:, c0r:].copy_(src)
                                    else:
                                        gw[:, c0r:].add_(src)
                        else:
                            mid, cop = c0r, dz.shape[3]
                            for k in range(f):
                                src = tmp[k * cop:k * cop + cout, k * midp:k * midp + mid]
                                if k == 0:
                                    gw.copy_(src)
                                else:
                                    gw.add_(src)
                    if has(ins["bias"]):
                        grads[ins["bias"]].zero_()          # both packed convs of a LightConvBlock sit in front of a BatchNorm
                    ready(ins["w"], ins["bias"])
                    need0, need1 = xin.needs_grad, (x1 is not None and x1.needs_grad)
                    if need0 or need1:
                        d0 = self._buf("g:" + ins["out"] + ">0", xin.data.shape)
                        if x1 is not None:
                            d1 = self._buf("g:" + ins["out"] + ">1", x1.data.shape)
                            ops.conv_dgrad(dzv, wd, xv.shape[3], taps=1, C1=x1v.shape[3], out0=d0.view(xv.shape), out1=d1.view(x1v.shape))
                            if need0:
                                self._acc_masked(xin, d0)
                            if need1:
                                self._acc_masked(x1, d1)
                        else:
                            ops.conv_dgrad(dzv, wd, xv.shape[3], taps=1, out0=d0.view(xv.shape))
                            self._acc(xin, d0)
                    continue
                coutp = pad64(cout)
                if ins["stride"] == 2 and taps == 9:
                    dz = ops.zero_insert2(dz, h, w, out=self._buf("g:" + ins["out"] + ":full", (n, h, w, coutp)))
                xw = t.aux if (ins["stride"] == 2 and taps == 1) else xin.data          # wgrad's activation operand
                c0p = xw.shape[3]
                c1p = x1.data.shape[3] if x1 else 0
                self._conv_param_grads(xw, dz, grads, has, ins["w"], ins["bias"], cout, c0r, c1r, x1=x1.data if x1 else None,
                                       taps=taps, pre_bn=ins["out"] in self._pre_bn, lo_half=ins["w"] in self.image_convs)
                ready(ins["w"], ins["bias"])
                need0, need1 = xin.needs_grad, (x1 is not None and x1.needs_grad)
                if not (need0 or need1):
                    continue
                if x1 is not None:
                    if need0:
                        d0 = self._buf("g:" + ins["out"] + ">0", xin.data.shape)
                        d1 = self._buf("g:" + ins["out"] + ">1", x1.data.shape)
                        ops.conv_dgrad(dz, wd, c0p, taps=taps, C1=c1p, out0=d0, out1=d1)
                        self._acc_masked(xin, d0)
                        if need1:
                            self._acc_masked(x1, d1)
                    else:       # frozen first source: only the second half needs a gradient
                        d1 = self._buf("g:" + ins["out"] + ">1", x1.data.shape)
                        ops.conv_dgrad(dz, wd[c0p:], c1p, taps=taps, mask=x1.data if x1.fused_relu else None, out0=d1)
                        self._acc(x1, d1)
                else:
                    d0 = self._buf("g:" + ins["out"] + ">0", xw.shape)
                    ops.conv_dgrad(dz, wd, c0p, taps=taps, mask=xin.data if (xin.fused_relu and xw is xin.data) else None, out0=d0)
                    if ins["stride"] == 2 and taps == 1:
                        d0 = ops.zero_insert2(d0, h, w, out=self._buf("g:" + ins["out"] + ">0:full", xin.data.shape))
                    self._acc(xin, d0)
            elif op == "stem":
                t = T[ins["out"]]
                if t.grad is None:
                    continue
                if has(ins["w"]):
                    col = t.aux
                    need = ops.lib().b2u_conv_wgrad_workspace(col.shape[0], col.shape[1], col.shape[2], 192, 64, 1)
                    ops.conv_wgrad_im2col(col, t.grad, 3, 49, dw=grads[ins["w"]], ws=self._workspace("wgrad", need))
                    ready(ins["w"])
                if dx is not None:
                    ops.stem_dgrad_input(t.grad, params[ins["w"]], H, W, out=dx)
                    dx_written = True
            elif op == "input":
                t = T[ins["out"]]
                if dx is not None and t.grad is not None:
                    # channels [C, 2C) (the lo half of the image split) meet the same weights: their gradient equals [0, C)'s
                    ops.nhwc_padded_to_nchw_f32(t.grad, ins["c"], out=dx)
                    dx_written = True
        if dx is not None and not dx_written:
            dx.zero_()          # no path from the image reached the loss: its gradient is zero, not whatever dx held

    def _relu_mask(self, t, g, key):
        """g, a gradient for t, made wrt t's pre-activation when t is a fused-ReLU conv output (ImprovedSegNet's deploy form
        feeds those to SE and Dropout2d, which cannot mask in their own pass)."""
        if not t.fused_relu:
            return g
        return ops.relu_bwd(g, t.data, out=self._buf("g:" + key + ">relu", g.shape))

    def _acc_masked(self, t, g):
        """Gradient from a split (two-output) dgrad, which cannot mask in its epilogue."""
        if t.fused_relu:
            raise NotImplementedError("split dgrad into a fused-ReLU tensor needs a mask pass")
        self._acc(t, g)


class ResNet50UnetEngine(GraphEngine):
    def __init__(self, num_classes, device=None):
        if not 1 <= num_classes <= 255:
            raise ValueError("num_classes must be in [1, 255]")
        program, convs = resnet50_unet_program(num_classes)
        super().__init__(program, convs, num_classes, device=device)


class UltraLightUnetEngine(GraphEngine):
    def __init__(self, num_classes, variant="ultralight_large", device=None):
        if not 1 <= num_classes <= 255:
            raise ValueError("num_classes must be in [1, 255]")
        widths, mid_min, se_rule, p = ULU_VARIANTS[variant]
        program, convs = ultralight_unet_program(num_classes, widths, mid_min, se_rule, p)
        super().__init__(program, convs, num_classes, device=device)
        self.variant = variant


class LightweightUnetEngine(GraphEngine):
    def __init__(self, num_classes, in_channels=3, device=None):
        if not 1 <= num_classes <= 255:
            raise ValueError("num_classes must be in [1, 255]")
        if not 1 <= in_channels <= 64:
            raise ValueError("in_channels must be in [1, 64] (the image is zero-padded to one 64-channel block)")
        program, convs = lightweight_unet_program(num_classes, in_channels)
        super().__init__(program, convs, num_classes, device=device)
        self.logit_stride = 2       # logits are H/2 x W/2; the losses resize them (nets/unet_training.py:12-13)


class ImprovedSegNetEngine(GraphEngine):
    """nets/RepVGG_Unet.py::ImprovedSegNet(use_repvgg=True); deploy=True runs the re-parameterised single-conv blocks."""

    def __init__(self, num_classes, deploy=False, device=None):
        if not 1 <= num_classes <= 255:
            raise ValueError("num_classes must be in [1, 255]")
        program, convs = improved_segnet_program(num_classes, deploy=deploy)
        super().__init__(program, convs, num_classes, device=device)
        self.deploy = deploy
