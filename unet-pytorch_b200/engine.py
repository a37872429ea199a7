"""Execution engine of the UNet hot path: one configurable encoder/decoder schedule that runs both the
VGG16-backbone Unet (nets/unet.py:62-78 + nets/vgg.py:21-31 of the reference: conv+bias+ReLU) and the
conv+BatchNorm+ReLU family (nets/TraditionalUnet.py:5-93).

The engine owns the bf16 NHWC activation buffers and the packed bf16 weights and launches the CUDA kernels of
libb200unet.so in the order of the reference's forward, then the hand-derived backward:

  forward   im2col(first conv) -> encoder blocks of [conv3x3 (+bias) (+BN) +ReLU] separated by 2x2 max-pools ->
            decoder stages (upsample2x -> conv over the *virtual* concat [skip, up] -> conv) -> 1x1 head -> logits
  backward  head bwd -> per decoder stage: (BN bwd,) wgrad/dgrad conv2, wgrad conv1, split dgrad conv1 (d skip | d up),
            upsample adjoint -> per encoder block: wgrad, dgrad, pool bwd (+skip grad); ReLU masks are fused into the
            dgrad / pool / upsample kernels (plain nets) or applied by the BN backward kernel (BN nets)

The per-layer launches (conv forward, conv parameter gradients, BatchNorm, head) are EngineBase's (_engine_base.py), shared
with GraphEngine; this engine adds what only the plain conv + ReLU nets use: ReLU bit masks, bias gradients from the
dgrad epilogue and the weight-gradient side stream.

Channel counts that are not multiples of 64 (the 32-channel layers of TraditionalUnet) are zero-padded to 64 in the
activation buffers and operands; padded channels stay exactly zero in both directions.

backward(dx=...) also returns the gradient wrt the input image: every layer then runs its data gradient (weight gradients
still follow `trainable`), and the first conv's data gradient, b2u_first_conv_dgrad_input, writes it as NCHW fp32.

Gradients are written straight into caller-provided fp32 OIHW tensors (normally views of one flat buffer), and
`on_grads_ready(names)` is called after the launches that complete each layer's gradients so a data-parallel
trainer can start that bucket's all-reduce while the remaining dgrad/wgrad kernels still run.
"""
import contextlib

import torch

from . import ops
from ._engine_base import EngineBase, pad64

# (features index, Cin, Cout) and 'M' for nn.MaxPool2d(2,2): cfgs['D'] of nets/vgg.py:62-64 without the last pool
VGG16_CFG = [(0, 3, 64), (2, 64, 64), "M", (5, 64, 128), (7, 128, 128), "M", (10, 128, 256), (12, 256, 256),
             (14, 256, 256), "M", (17, 256, 512), (19, 512, 512), (21, 512, 512), "M", (24, 512, 512), (26, 512, 512),
             (28, 512, 512)]
# (module name, C_skip, C_up, C_out): in_filters [192, 384, 768, 1024], out_filters [64, 128, 256, 512] (nets/unet.py:28-45)
DECODER_CFG = [("up_concat4", 512, 512, 512), ("up_concat3", 256, 512, 256), ("up_concat2", 128, 256, 128),
               ("up_concat1", 64, 128, 64)]


def vgg_unet_param_shapes(num_classes, in_channels=3):
    """name -> shape, in the reference's state_dict order (44 tensors)."""
    shapes = {}
    for item in VGG16_CFG:
        if item == "M":
            continue
        i, cin, cout = item
        cin = in_channels if i == 0 else cin
        shapes[f"vgg.features.{i}.weight"] = (cout, cin, 3, 3)
        shapes[f"vgg.features.{i}.bias"] = (cout,)
    for name, cs, cu, co in DECODER_CFG:
        shapes[f"{name}.conv1.weight"] = (co, cs + cu, 3, 3)
        shapes[f"{name}.conv1.bias"] = (co,)
        shapes[f"{name}.conv2.weight"] = (co, co, 3, 3)
        shapes[f"{name}.conv2.bias"] = (co,)
    shapes["final.weight"] = (num_classes, 64, 1, 1)
    shapes["final.bias"] = (num_classes,)
    return shapes


class ConvSpec:
    """One conv3x3 (+BN) + ReLU layer.  name/bn: parameter-name prefixes; c0/c1: real channels of the two sources
    of a virtual concat (c1 = 0: single source)."""
    __slots__ = ("name", "bn", "cin", "cout", "first", "c0", "c1", "wf", "wd", "cout_p", "c0_p", "c1_p")

    def __init__(self, name, cin, cout, first=False, c0=None, c1=0, bn=None):
        self.name, self.bn, self.cin, self.cout, self.first = name, bn, cin, cout, first
        self.c0 = cin if c0 is None else c0
        self.c1 = c1
        self.cout_p = pad64(cout)
        self.c0_p = 64 if first else pad64(self.c0)
        self.c1_p = pad64(c1) if c1 else 0
        self.wf = self.wd = None

    @property
    def padded(self):
        return self.cout_p != self.cout or (not self.first and (self.c0_p != self.c0 or self.c1_p != self.c1))


class UNetConfig:
    """enc: list of blocks (lists of ConvSpec) separated by 2x2 max-pools; dec: list of (conv1, conv2) stages, stage i
    consumes the output of stage i-1 (or the last encoder block) upsampled 2x plus encoder block len(enc)-2-i as skip;
    head: (name, real input channels)."""

    def __init__(self, enc, dec, head, num_classes, in_channels=3):
        self.enc, self.dec, self.head, self.num_classes, self.in_channels = enc, dec, head, num_classes, in_channels
        self.bn = any(c.bn for b in enc for c in b)


def vgg_unet_config(num_classes, in_channels=3):
    enc, block = [], []
    for item in VGG16_CFG:
        if item == "M":
            enc.append(block)
            block = []
        else:
            i, cin, cout = item
            block.append(ConvSpec(f"vgg.features.{i}", in_channels if i == 0 else cin, cout, first=(i == 0)))
    enc.append(block)
    dec = [(ConvSpec(f"{name}.conv1", cs + cu, co, c0=cs, c1=cu), ConvSpec(f"{name}.conv2", co, co))
           for name, cs, cu, co in DECODER_CFG]
    return UNetConfig(enc, dec, ("final", 64), num_classes, in_channels)


def traditional_unet_config(num_classes, in_channels=3):
    """nets/TraditionalUnet.py:45-93: DoubleConv = (conv3x3+bias, BN, ReLU) x 2; widths 32-64-128-256; Up concatenates
    [skip, up] (:41) like unetUp."""
    def double(prefix, cin, cout, first=False, c0=None, c1=0):
        return [ConvSpec(f"{prefix}.double_conv.0", cin, cout, first=first, c0=c0, c1=c1, bn=f"{prefix}.double_conv.1"),
                ConvSpec(f"{prefix}.double_conv.3", cout, cout, bn=f"{prefix}.double_conv.4")]
    enc = [double("inc", in_channels, 32, first=True), double("down1.maxpool_conv.1", 32, 64),
           double("down2.maxpool_conv.1", 64, 128), double("down3.maxpool_conv.1", 128, 256)]
    dec = [tuple(double("up1.conv", 384, 128, c0=128, c1=256)), tuple(double("up2.conv", 192, 64, c0=64, c1=128)),
           tuple(double("up3.conv", 96, 32, c0=32, c1=64))]
    return UNetConfig(enc, dec, ("outc", 32), num_classes, in_channels)


class UNetEngine(EngineBase):
    def __init__(self, cfg, device=None):
        if cfg.in_channels * 9 > 64:
            raise ValueError("in_channels must be <= 7 (first-layer im2col is 64 columns wide)")
        if not 1 <= cfg.num_classes <= 255:
            raise ValueError("num_classes must be in [1, 255]")
        super().__init__(device)
        self.cfg = cfg
        self.num_classes = cfg.num_classes
        self.in_channels = cfg.in_channels
        self.enc, self.dec, self.bn = cfg.enc, cfg.dec, cfg.bn
        self.head_name, self.head_cin = cfg.head
        self.convs = [c for b in self.enc for c in b] + [c for pair in self.dec for c in pair]
        self._side = None

    # ------------------------------------------------------------------ policies of the plain conv + ReLU nets
    def relu_bit_masks(self, save):
        """ReLU backward from bit masks (training forward, bf16): every conv epilogue also writes (y > 0) as one bit per
        channel ([N,H,W,C/64] 64-bit words, 1/16 of the bytes of y) and the masked data gradients / the head backward read
        those 8 bytes per pixel and block instead of 128 bytes of y -- 2.8 GB less HBM traffic per headline step, and the
        HBM-bound 64-channel data gradients at 512 x 512 then tile like unmasked launches (four stacked M tiles, no cp.async
        mask stream).  Same-call A/B: 22.13 / 22.15 ms per step without, 21.77 / 21.73 with, results bit-identical
        (test_relu_bit_masks*).  The pool / upsample adjoints always read y."""
        return save and ops.act_dtype() == torch.bfloat16

    def bias_from_dgrad(self, c):
        """Bias gradient of a wide plain layer (one whose db does not come from the wgrad kernel, see fused_db) from the
        data-gradient launch that PRODUCES its dz: that epilogue leaves per-tile column sums of the masked gradient it stores
        (b2u_conv_dgrad_stats, the BatchNorm-statistics machinery) and b2u_bias_from_stats folds them, instead of
        b2u_bias_grad re-reading dz from HBM (1.2 GB per headline step).  Those dgrads have K >= 1152, long enough to hide the
        extra epilogue work.  Layers whose dz comes from the pool / upsample adjoints keep the separate pass."""
        return not self.bn and ops.act_dtype() == torch.bfloat16 and not c.padded and not c.first and not self.fused_db(c.cout_p)

    # ------------------------------------------------------------------ weights
    def pack(self, params, need_dgrad=True):
        """(Re)packs fp32 OIHW weights to bf16 operands when any of them changed: one launch for the whole model,
        driven by a device-resident table of (weight, operand) pointers that is rebuilt only if a pointer moved."""
        key = tuple(params[c.name + ".weight"].data_ptr() for c in self.convs) + (need_dgrad,)
        versions = tuple(params[c.name + ".weight"]._version for c in self.convs)
        if self._pack_key == key and self._pack_versions == versions:
            return
        dev = params[self.convs[0].name + ".weight"].device
        if self._pack_key != key:
            layers = []
            for c in self.convs:
                ctot_p = c.c0_p + c.c1_p
                if c.first:
                    if c.wf is None:
                        c.wf = torch.zeros((c.cout_p, 64), dtype=ops.act_dtype(), device=dev)
                else:
                    if c.wf is None:
                        c.wf = torch.zeros((c.cout_p, 9 * ctot_p), dtype=ops.act_dtype(), device=dev)
                    if need_dgrad and c.wd is None:
                        c.wd = torch.zeros((ctot_p, 9 * c.cout_p), dtype=ops.act_dtype(), device=dev)
                layers.append((params[c.name + ".weight"], c.wf, c.wd if need_dgrad else None, c.cout, c.cin,
                               1 if c.first else 9, c.first, c.c0, c.c0_p, ctot_p, c.cout_p))
            self._set_pack_table(layers, dev)
            self._pack_key = key
        self._launch_pack()
        self._pack_versions = versions

    def param_shapes(self):
        """name -> shape of every trainable tensor, in the reference module's state_dict order."""
        shapes = {}
        for c in self.convs:
            shapes[c.name + ".weight"] = (c.cout, c.cin, 3, 3)
            shapes[c.name + ".bias"] = (c.cout,)
            if c.bn:
                shapes[c.bn + ".weight"] = (c.cout,)
                shapes[c.bn + ".bias"] = (c.cout,)
        shapes[self.head_name + ".weight"] = (self.num_classes, self.head_cin, 1, 1)
        shapes[self.head_name + ".bias"] = (self.num_classes,)
        return shapes

    def buffer_shapes(self):
        """BatchNorm buffers (running statistics), state_dict names."""
        shapes = {}
        for c in self.convs:
            if c.bn:
                shapes[c.bn + ".running_mean"] = (c.cout,)
                shapes[c.bn + ".running_var"] = (c.cout,)
                shapes[c.bn + ".num_batches_tracked"] = ()
        return shapes

    def backward_param_order(self):
        """Parameter names in the order backward() completes their gradients (head first, first conv last)."""
        layers = []
        for si in range(len(self.dec) - 1, -1, -1):
            layers += [self.dec[si][1], self.dec[si][0]]
        for bi in range(len(self.enc) - 1, -1, -1):
            layers += list(reversed(self.enc[bi]))
        out = [self.head_name + ".weight", self.head_name + ".bias"]
        for c in layers:
            if c.bn:
                out += [c.bn + ".weight", c.bn + ".bias"]
            out += [c.name + ".weight", c.name + ".bias"]
        return out

    # ------------------------------------------------------------------ one conv (+BN) + ReLU layer, forward
    def _layer_fwd(self, c, x0, params, A, training, x1=None, save=True, low=None, up_out=None):
        """low (instead of x1): the second source is upsample2x(low), interpolated inside the conv kernel
        (ops.decoder_conv_fprop); up_out then optionally receives the up-sampled tensor as a by-product."""
        n, h, w, _ = x0.shape
        bias = self._padded("b:" + c.name, params[c.name + ".bias"], (c.cout_p,))
        taps = 1 if c.first else 9
        out = A[c.name] = self._buf(c.name, (n, h, w, c.cout_p))
        if not c.bn and self.relu_bit_masks(save):
            bits = A["bits:" + c.name] = self._buf("bits:" + c.name, (n, h, w, c.cout_p // 64), torch.int64)
            ops.conv_fprop_relu_bits(x0, c.wf, bias, c.cout_p, bits, taps=taps, x1=x1, low=low, up_out=up_out, out=out)
            return out
        if not c.bn or (not training and not save):
            # pure inference: BatchNorm is an affine map with fixed statistics, folded into the conv epilogue
            # (y = relu(acc * s + b')): no z tensor, no BatchNorm pass.  An eval-mode forward that will be back-propagated
            # (model.eval() + loss.backward()) takes the unfused path below so the BatchNorm backward has z
            scale = None
            if c.bn:
                scale, bias = self._folded_bn(c.bn, params, bias, c.cout_p)
            self._conv_fwd(x0, c.wf, bias, c.cout_p, taps, True, out, x1=x1, low=low, up_out=up_out, scale=scale)
            return out
        z = self._buf("z:" + c.name, (n, h, w, c.cout_p))
        centered = self.center_pre_bn(training)
        if centered:
            rmp = self._padded("rm:" + c.bn, params[c.bn + ".running_mean"], (c.cout_p,))
            bias = torch.sub(bias, rmp, out=self._buf("bc:" + c.name, (c.cout_p,), torch.float32))
        stats = None
        kdim = taps * (x0.shape[3] + (x1.shape[3] if x1 is not None else 0) + (low.shape[3] if low is not None else 0))
        if self.fuse_bn_stats(training, kdim, c.cout_p):
            stats = self._bn_stats("bnstat", n, h, w, c.cout_p, taps, decoder=low is not None)
        self._conv_fwd(x0, c.wf, bias, c.cout_p, taps, False, z, x1=x1, low=low, up_out=up_out, stats=stats)
        A["bn:" + c.name] = (z,) + self._bn_fwd(c.bn, z, params, training, True, out, stats=stats, centered=centered)
        return out

    # ------------------------------------------------------------------ forward
    def forward(self, x, params, save=True, training=None, trainable=None, input_grad=False):
        """x: NCHW fp32 CUDA [N, Cin, H, W] -> logits NCHW fp32.  training (BN nets): batch statistics + running-stat
        update (default: same as `save`).  trainable and input_grad are accepted for interface parity with GraphEngine
        (backward decides what to skip from the gradient names it is given, and whether to reach the image from its dx)."""
        if not x.is_cuda:
            raise ValueError("UNetEngine.forward: input must be a CUDA tensor (no CPU fallback)")
        if x.dtype != torch.float32:
            x = x.float()
        x = x.contiguous()
        N, C, H, W = x.shape
        if C != self.in_channels:
            raise ValueError(f"expected {self.in_channels} input channels, got {C}")
        div = 2 ** (len(self.enc) - 1)
        if H % div or W % div:
            raise ValueError(f"input height and width must be multiples of {div}")
        if training is None:
            training = save
        self.device = x.device
        self.pack(params, need_dgrad=save)
        A = {}
        col = self._buf("col", (N, H, W, 64))
        ops.check(ops.lib().b2u_im2col_first(x.data_ptr(), col.data_ptr(), N, C, H, W, ops.stream_ptr()))
        A["col"] = col
        cur = col
        h, w = H, W
        feats = []
        for bi, block in enumerate(self.enc):
            if bi > 0:
                pooled = self._buf(f"pool{bi}", (N, h // 2, w // 2, cur.shape[3]))
                ops.maxpool2x2(cur, out=pooled)
                A[f"pool{bi}"] = pooled
                cur = pooled
                h, w = h // 2, w // 2
            for c in block:
                cur = self._layer_fwd(c, cur, params, A, training, save=save)
            feats.append(cur)
        low = feats[-1]
        for si, (c1, c2) in enumerate(self.dec):
            skip = feats[len(self.enc) - 2 - si]
            _, hl, wl, cl = low.shape
            if self.fuse_upsample(c1.cout_p):
                # the decoder conv interpolates `low` inside its producer warps (nets/unet.py:16-18 in one kernel); the
                # up-sampled tensor is written only when a backward pass will need it as the weight gradient's operand
                # (the fp32 validation build always takes the buffer: it keeps the two steps apart)
                keep = save or ops.act_dtype() == torch.float32
                up = self._buf(f"up{si}", (N, 2 * hl, 2 * wl, cl)) if keep else None
                o1 = self._layer_fwd(c1, skip, params, A, training, save=save, low=low, up_out=up)
            else:
                up = self._buf(f"up{si}", (N, 2 * hl, 2 * wl, cl))
                ops.upsample2x(low, out=up)
                o1 = self._layer_fwd(c1, skip, params, A, training, x1=up, save=save)
            A[f"up{si}"] = up
            low = self._layer_fwd(c2, o1, params, A, training, save=save)
        logits = self._head_fwd(low, params, self.head_name + ".weight", self.head_name + ".bias", self.head_cin)
        if save:
            self.saved = (A, feats, (N, H, W))
        return logits

    # ------------------------------------------------------------------ backward
    def backward(self, dlogits, params, grads, trainable=None, on_grads_ready=None, dx=None):
        """dlogits: NCHW fp32, or bf16 [N,H,W,64] from ops.loss_bwd(nhwc64=True).  grads: name -> fp32 tensor to
        overwrite (missing / not in `trainable`: skipped).  dx (optional): NCHW fp32 buffer shaped like the input, which
        receives the gradient wrt the image (x.grad); every layer then runs its data gradient, frozen ones included, while
        weight gradients still follow `trainable`."""
        if self.saved is None:
            raise RuntimeError("backward() without a saved forward()")
        # Weight/bias gradients on a second stream (plain conv+ReLU nets): wgrad_L depends only on dz_L and the saved
        # activation, not on the dgrad chain, so its launches are queued on a side stream behind an event and the
        # HBM-bound glue of the main chain (pool / upsample adjoints, column-sum folds) shares the SMs with tensor-core-bound
        # kernels of the other stream instead of running alone.  Same-box A/B (bench.py --kernels-only, 12 steps, twice each,
        # round 2 final build): 21.79 / 21.67 ms per step with it, 22.05 / 21.87 without (-1 %; round 1 measured -0.9 %).
        # Per-launch CUDA-event times are not a kernel's own duration while two streams overlap, so the roofline pass of
        # bench.py (ops.KernelTimer) runs single-stream.
        side = None
        if not self.bn and dlogits.is_cuda and not ops.timing_active():
            if self._side is None or self._side.device != dlogits.device:
                self._side = torch.cuda.Stream(device=dlogits.device)
            side = self._side
            # size the shared workspaces before the side stream starts using them (a reallocation mid-backward would hand
            # the old block back to the allocator while a kernel of the other stream may still read it)
            A, _, (N, H, W) = self.saved
            need = 0
            for c in self.convs:
                t = A[c.name]
                need = max(need, ops.lib().b2u_conv_wgrad_workspace(t.shape[0], t.shape[1], t.shape[2],
                                                                     64 if c.first else c.c0_p + c.c1_p, c.cout_p, 1 if c.first else 9))
            need = max(need, ops.lib().b2u_conv_wgrad_workspace(N, H, W, 64, 64, 1))
            self._workspace("wgrad", need)
            self._workspace("bias", ops.lib().b2u_bias_grad_workspace(max(c.cout_p for c in self.convs)))
            side.wait_stream(torch.cuda.current_stream())
        try:
            self._backward(dlogits, params, grads, trainable, on_grads_ready, side, dx)
        finally:
            if side is not None:
                torch.cuda.current_stream().wait_stream(side)      # optimizer / next forward see every gradient

    def _backward(self, dlogits, params, grads, trainable, on_grads_ready, side, dx):
        A, feats, (N, H, W) = self.saved
        if trainable is None:
            trainable = set(grads.keys())
        bn = self.bn
        order = [c.name for c in self.convs] + [self.head_name]

        def wanted(c):
            names = [c.name + ".weight", c.name + ".bias"] + ([c.bn + ".weight", c.bn + ".bias"] if c.bn else [])
            return any(n in trainable for n in names)
        want = {c.name: wanted(c) for c in self.convs}
        want[self.head_name] = (self.head_name + ".weight") in trainable or (self.head_name + ".bias") in trainable
        # data gradients are needed down to the first (in execution order) trainable conv, or to the image
        first_trainable = -1 if dx is not None else next((i for i, n in enumerate(order) if want[n]), len(order))
        need_dx = {n: i > first_trainable for i, n in enumerate(order)}   # does layer n have to produce dx?
        n_enc = sum(len(b) for b in self.enc)
        enc_trainable = first_trainable < n_enc       # the encoder's features need their skip gradients

        def ready(*names):
            if on_grads_ready is not None:
                on_grads_ready([n for n in names if n in grads])

        def grad_stream():
            """Context for the launches that produce parameter gradients: the side stream, ordered after everything queued on
            the main stream so far (the dz they read), or a no-op."""
            if side is None:
                return contextlib.nullcontext()
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            side.wait_event(ev)
            return torch.cuda.stream(side)

        def has(n):
            return n in trainable and n in grads

        db_stats = {}      # conv name -> (per-tile column sums of its dz, rows), left behind by the dgrad that produced dz

        def dgrad_to(below, dz, wd, C0, mask, out0):
            """Masked data gradient that becomes `below`'s dz; also records dz's column sums when `below` wants a bias gradient
            that would otherwise need a pass over dz.  The ReLU mask is `below`'s bit mask when the forward left one."""
            bits = A.get("bits:" + below.name) if mask is not None else None
            stats = None
            if want[below.name] and has(below.name + ".bias") and self.bias_from_dgrad(below):
                n_, h_, w_, _ = out0.shape
                rows = ops.conv_dgrad_stat_rows(n_, h_, w_, C0, 9, masked=mask is not None and bits is None)
                nbytes = rows * 2 * C0 * 4
                stats = self._workspace("dbstat:" + below.name, nbytes)[:nbytes].view(torch.float32)
                db_stats[below.name] = (stats, rows)
            if bits is not None:
                ops.conv_dgrad_bits(dz, wd, C0, bits, out0=out0, stats=stats)
            else:
                ops.conv_dgrad(dz, wd, C0, mask=mask, out0=out0, stats=stats)

        def layer_bwd(c, x0, g, x1=None):
            """g: gradient wrt the layer's output (BN nets: wrt y, unmasked; plain nets: wrt the pre-activation, already
            masked).  Runs BN backward if any, wgrad, bias grad; returns dz (the conv's output gradient)."""
            if c.bn:
                z, *saved = A["bn:" + c.name]
                self._bn_bwd(g, A[c.name], z, saved, True, g, grads, has, c.bn, c.cout)
                ready(c.bn + ".weight", c.bn + ".bias")
            if want[c.name]:
                with grad_stream():
                    self._conv_param_grads(x0, g, grads, has, c.name + ".weight", c.name + ".bias", c.cout, c.c0, c.c1, x1=x1,
                                           taps=1 if c.first else 9, pre_bn=bool(c.bn), first_cin=c.cin if c.first else 0,
                                           db_stats=db_stats.pop(c.name, None))
                    ready(c.name + ".weight", c.name + ".bias")
            return g

        # ---- head
        hn = self.head_name
        last = A[self.dec[-1][1].name]
        g = self._buf("g:" + self.dec[-1][1].name, last.shape) if need_dx[hn] else None
        self._head_bwd(dlogits, last, params, grads, has, hn + ".weight", hn + ".bias", self.head_cin, g,
                       None if bn else last, bits=None if bn else A.get("bits:" + self.dec[-1][1].name), grad_stream=grad_stream)
        with grad_stream():          # (orders the side stream after the head's launches, whichever stream ran them)
            ready(hn + ".weight", hn + ".bias")
        if g is None:
            return

        # ---- decoder, last stage first
        n_dec = len(self.dec)
        dskips = [None] * (len(self.enc) - 1)     # gradient wrt the encoder features coming from the decoder
        for si in range(n_dec - 1, -1, -1):
            c1, c2 = self.dec[si]
            fi = len(self.enc) - 2 - si
            skip = feats[fi]
            up = A[f"up{si}"]
            o1 = A[c1.name]
            low = feats[-1] if si == 0 else A[self.dec[si - 1][1].name]
            dz = layer_bwd(c2, o1, g)
            if not need_dx[c2.name]:
                return
            g1 = self._buf("g:" + c1.name, o1.shape)
            dgrad_to(c1, dz, c2.wd, c2.c0_p, None if bn else o1, g1)
            dz1 = layer_bwd(c1, skip, g1, x1=up)
            if not need_dx[c1.name]:
                return
            dup = self._buf(f"g:up{si}", up.shape)
            if enc_trainable:
                dsk = self._buf(f"g:skip{fi}", skip.shape)
                ops.conv_dgrad(dz1, c1.wd, c1.c0_p, C1=c1.c1_p, out0=dsk, out1=dup)
                dskips[fi] = dsk
            else:
                # frozen encoder: only the up-sampled half of the concat needs a gradient
                ops.conv_dgrad(dz1, c1.wd[c1.c0_p:], c1.c1_p, out0=dup)
            if si == 0 and not enc_trainable:
                return
            g = self._buf("g:low" + str(si), low.shape)
            ops.upsample2x_bwd(dup, ylow=None if bn else low, out=g)

        # ---- encoder, deepest block first; g = gradient wrt the block's last conv output
        for bi in range(len(self.enc) - 1, -1, -1):
            block = self.enc[bi]
            for ci in range(len(block) - 1, -1, -1):
                c = block[ci]
                if ci > 0:
                    xin = A[block[ci - 1].name]
                elif bi > 0:
                    xin = A[f"pool{bi}"]
                else:
                    xin = A["col"]
                dz = layer_bwd(c, xin, g)
                if not need_dx[c.name]:
                    return
                if ci > 0:
                    nxt = self._buf("g:" + block[ci - 1].name, xin.shape)
                    dgrad_to(block[ci - 1], dz, c.wd, c.c0_p, None if bn else xin, nxt)
                    g = nxt
                elif bi == 0:
                    ops.first_conv_dgrad_input(dz, params[c.name + ".weight"], out=dx)
                else:
                    dpool = self._buf(f"g:pool{bi}", xin.shape)
                    ops.conv_dgrad(dz, c.wd, c.c0_p, out0=dpool)
                    y = feats[bi - 1]
                    nxt = self._buf(f"g:feat{bi - 1}", y.shape)
                    ops.maxpool2x2_bwd(dpool, y, dskip=dskips[bi - 1], relu_mask=not bn, out=nxt)
                    g = nxt


class VGGUnetEngine(UNetEngine):
    def __init__(self, num_classes, in_channels=3, device=None):
        super().__init__(vgg_unet_config(num_classes, in_channels), device=device)


class TraditionalUnetEngine(UNetEngine):
    def __init__(self, num_classes, in_channels=3, device=None):
        super().__init__(traditional_unet_config(num_classes, in_channels), device=device)
