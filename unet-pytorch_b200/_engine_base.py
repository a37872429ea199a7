"""What the two training engines share: UNetEngine (engine.py: Unet-VGG16 and TraditionalUnet) and GraphEngine (graph.py:
the other families).

  buffers    activation buffers, kernel workspaces and padded parameter vectors, cached by key across steps
  weights    the device table of b2u_pack_weights_multi (one record per conv) and its launch
  policies   which fused kernel variant runs where -- each decided by a B200 measurement (DESIGN.md)
  BatchNorm  forward (train / SyncBatchNorm / eval, padded running statistics) and backward (dgamma / dbeta included)
  convs      the choice among the forward conv launches, and a conv's weight and bias gradients
  head       the 1x1 classifier, forward and backward

Each engine decides WHICH of these a layer runs (its topology, its ReLU masks, its streams); the launches are written here once.
"""
import contextlib
import functools
import struct

import torch

from . import ops


def pad64(c):
    return (c + 63) // 64 * 64


class EngineBase:
    eps, momentum = 1e-5, 0.1           # nn.BatchNorm2d defaults (the reference never changes them)

    def __init__(self, device=None):
        self.device = device
        self.sync_bn_group = None       # torch.distributed group: BatchNorm statistics over all ranks (SyncBatchNorm)
        self.saved = None
        self._bufs, self._ws = {}, {}
        self._pack_key = self._pack_versions = self._pack_table = None
        self._pack_count = self._pack_total = 0

    # ------------------------------------------------------------------ policies
    def fuse_upsample(self, cout_p):
        """Bilinear 2x up-sampling folded into the operand load of the decoder conv that reads it (b2u_decoder_conv_fprop),
        for a conv of cout_p padded output channels.  Measured at the four unetUp shapes of the headline step
        (scripts/ab_fused_upsample.py, profiles/r2_fused_upsample.json): with N tiles of 128 / 256 output channels the fused
        conv beats upsample + conv (0.42 / 0.65 / 0.70 ms against 0.42 / 0.67 / 0.77); with the N = 64 tile (64+128 -> 64 at
        512 x 512) the five interpolation warps cannot keep up with a main loop that short (1.32 against 1.07 ms), so that
        stage keeps the separate pass.  Both ways are bit-identical (test_fused_upsample_equals_separate_pass)."""
        return cout_p >= 128

    def fuse_bn_stats(self, training, kdim, cout_p):
        """BatchNorm statistics from the producing conv's epilogue (one pass over z less), for a conv with reduction length
        kdim and cout_p padded output channels.  The extra epilogue work only hides behind the main loop when the reduction
        is long enough: it gains 0.8 ms on Unet-ResNet50 but loses 0.7-1.3 ms on the full-resolution, short-K layers of the
        other BatchNorm nets.  SyncBatchNorm sums over all ranks instead."""
        return training and self.sync_bn_group is None and (kdim >= 1024 or cout_p >= 256)

    def center_pre_bn(self, training):
        """Training: a tensor read only by a BatchNorm is stored CENTRED on that BatchNorm's running mean (the shift rides in
        the conv bias, in fp32, before the bf16 rounding; BatchNorm is shift-invariant; the running-mean update adds it back).
        Without it a channel with |mean| >> std loses |mean|/std * 2^-9 of relative accuracy in bf16 -- the dominant error
        site of the depthwise nets on warm weights (profiles/r2_precision_sites.txt).  At initialisation the running mean
        is 0: no change."""
        return training and ops.act_dtype() == torch.bfloat16

    def fused_db(self, cout_p):
        """A 3x3 conv's bias gradient from its weight-gradient launch (the kernel's bias warps sum the staged dz tiles) instead
        of a separate pass over dz: free for Cout = 64, where the swapped-role kernel runs.  For the wider layers an A/B on
        one B200 showed no gain (23.2-23.9 against 23.4-23.5 ms per step): the extra shared-memory reads slow the work units
        that own the bias."""
        return cout_p == 64

    # ------------------------------------------------------------------ buffers
    def _buf(self, key, shape, dtype=None):
        dtype = ops.act_dtype() if dtype is None else dtype      # bf16; fp32 under the fp32 validation build
        t = self._bufs.get(key)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            t = torch.empty(shape, dtype=dtype, device=self.device)
            self._bufs[key] = t
        return t

    def _workspace(self, key, nbytes):
        t = self._ws.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=self.device)
            self._ws[key] = t
        return t

    def _padded(self, key, t, shape, fill=0.0):
        """fp32 parameter padded with `fill` to `shape` (persistent buffer; the real part is refreshed every call)."""
        if tuple(t.shape) == tuple(shape):
            return t
        b = self._bufs.get(key)
        if b is None or tuple(b.shape) != tuple(shape):
            b = torch.full(shape, fill, dtype=torch.float32, device=self.device)
            self._bufs[key] = b
        b[tuple(slice(0, d) for d in t.shape)].copy_(t)
        return b

    def release(self):
        self._bufs.clear()
        self._ws.clear()
        self.saved = None

    # ------------------------------------------------------------------ weights
    def _set_pack_table(self, layers, dev):
        """layers: per conv (fp32 OIHW source, wf, wd or None, Cout, Cin, taps, first, C0, C0_pad, Ctot_pad, Cout_pad), the
        fields of one b2u_pack_weights_multi record (include/b2u.h) besides its first work block."""
        blob, start = b"", 0
        for src, wf, wd, cout, cin, taps, first, c0, c0_p, ctot_p, cout_p in layers:
            blob += struct.pack("<QQQqiiiiiiii", src.data_ptr(), wf.data_ptr(), 0 if wd is None else wd.data_ptr(), start,
                                cout, cin, taps, int(first), c0, c0_p, ctot_p, cout_p)
            start += (cout + 31) // 32 * (1 if first else (cin + 31) // 32)      # 32 x 32 work blocks (first layer: 32 rows)
        self._pack_table = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)
        self._pack_count, self._pack_total = len(layers), start

    def _launch_pack(self):
        ops.check(ops.lib().b2u_pack_weights_multi(self._pack_table.data_ptr(), self._pack_count, self._pack_total,
                                                   ops.stream_ptr()))

    def invalidate_packed_weights(self):
        """Call after writing parameters behind torch's back (raw-pointer optimizer kernels)."""
        self._pack_versions = None

    # ------------------------------------------------------------------ BatchNorm
    def _bn_stats(self, key, n, h, w, cout_p, taps, decoder=False):
        """Workspace for the BatchNorm statistics a conv epilogue emits: (fp32 per-tile column sums, rows)."""
        rows = ops.conv_stat_rows(n, h, w, cout_p, taps, bn=(1 << 18) if decoder else 0)      # bit 18: the decoder conv's tiles
        nbytes = rows * 2 * cout_p * 4
        return self._workspace(key, nbytes)[:nbytes].view(torch.float32), rows

    def _folded_bn(self, bn, params, conv_bias, cp):
        """(scale, bias) of `conv -> eval BatchNorm` as one affine map, padded to cp channels."""
        gamma = self._padded("g:" + bn, params[bn + ".weight"], (cp,), 1.0)
        beta = self._padded("bt:" + bn, params[bn + ".bias"], (cp,))
        rmp = self._padded("rm:" + bn, params[bn + ".running_mean"], (cp,))
        rvp = self._padded("rv:" + bn, params[bn + ".running_var"], (cp,), 1.0)
        cb = self._padded("b:" + bn, conv_bias, (cp,)) if conv_bias is not None else None
        return ops.bn_fold(gamma, beta, rmp, rvp, cb, self.eps, scale=self._buf("fs:" + bn, (cp,), torch.float32),
                           bias=self._buf("fb:" + bn, (cp,), torch.float32))

    def _bn_fwd(self, bn, z, params, training, relu, out, residual=None, stats=None, centered=False):
        """BatchNorm `bn` of z (channels padded to z.shape[3]) (+ residual) (+ ReLU) into out.  Training: batch statistics
        (over all ranks under SyncBatchNorm), running statistics and num_batches_tracked updated; eval: running statistics.
        stats: (per-tile column sums, rows) from the producing conv's epilogue; centered: z is stored minus the running mean.
        Returns (mean, invstd, gamma, beta) for _bn_bwd; eval mode: ((running mean, running var), None, gamma, beta)."""
        cp = z.shape[3]
        ws = self._workspace("bn", ops.lib().b2u_bn_workspace(cp))
        gamma = self._padded("g:" + bn, params[bn + ".weight"], (cp,), 1.0)
        beta = self._padded("bt:" + bn, params[bn + ".bias"], (cp,))
        rm, rv = params[bn + ".running_mean"], params[bn + ".running_var"]
        rmp, rvp = self._padded("rm:" + bn, rm, (cp,)), self._padded("rv:" + bn, rv, (cp,), 1.0)
        if not training:
            ops.bn_fwd_eval(z, gamma, beta, rmp, rvp, self.eps, relu, out=out, ws=ws, residual=residual)
            return (rmp, rvp), None, gamma, beta
        if self.sync_bn_group is not None:
            _, mean, invstd = ops.bn_fwd_train_sync(z, gamma, beta, rmp, rvp, self.sync_bn_group, self.eps, self.momentum, relu,
                                                    out=out, ws=ws, residual=residual, centered=centered)
        else:
            _, mean, invstd = ops.bn_fwd_train(z, gamma, beta, rmp, rvp, self.eps, self.momentum, relu, out=out, ws=ws,
                                               residual=residual, stats=stats[0] if stats else None,
                                               stat_rows=stats[1] if stats else 0, centered=centered)
        if rmp is not rm:
            rm.copy_(rmp[:rm.numel()]); rv.copy_(rvp[:rv.numel()])
        nbt = params.get(bn + ".num_batches_tracked")
        if nbt is not None:
            nbt.add_(1)
        return mean, invstd, gamma, beta

    def _bn_bwd(self, dy, y, z, saved, relu, out, grads, has, bn, c, residual=False, gout=None):
        """Backward of _bn_fwd (saved = what it returned) for BatchNorm `bn` of c real channels: dz into out, dgamma / dbeta
        into grads (through padded buffers when z's channels are padded); gout receives the ReLU-masked dy (the residual
        branch's gradient).  y is read in eval mode and where a residual was added before the ReLU; otherwise the mask is
        recomputed from z."""
        mean, invstd, gamma, beta = saved
        cp = z.shape[3]
        wn, bn_ = bn + ".weight", bn + ".bias"
        dgamma = grads[wn] if cp == c and has(wn) else self._buf("dg:" + bn, (cp,), torch.float32)
        dbeta = grads[bn_] if cp == c and has(bn_) else self._buf("db:" + bn, (cp,), torch.float32)
        ws = self._workspace("bn", ops.lib().b2u_bn_workspace(cp))
        if invstd is None:          # eval-mode forward (model.eval() + backward): the statistics are constants
            ops.bn_bwd_eval(dy, y, z, gamma, beta, mean[0], mean[1], self.eps, relu=relu, out=out, dgamma=dgamma, dbeta=dbeta,
                            ws=ws, gout=gout)
        else:
            bwd = ops.bn_bwd if self.sync_bn_group is None else functools.partial(ops.bn_bwd_sync, group=self.sync_bn_group)
            bwd(dy, y if residual else None, z, gamma, mean, invstd, relu=relu, out=out, dgamma=dgamma, dbeta=dbeta, beta=beta,
                ws=ws, gout=gout)
        if cp != c:
            if has(wn):
                grads[wn].copy_(dgamma[:c])
            if has(bn_):
                grads[bn_].copy_(dbeta[:c])

    # ------------------------------------------------------------------ convolutions
    def _conv_fwd(self, x0, wf, bias, cout_p, taps, relu, out, x1=None, low=None, up_out=None, scale=None, stats=None):
        """One conv launch into out: over x0 (+ x1, virtual concat), or over x0 + upsample2x(low) interpolated inside the
        kernel (up_out optionally receives the up-sampled tensor); scale: an eval-mode BatchNorm folded into the epilogue;
        stats: (per-tile column sums, rows) of _bn_stats, which the epilogue fills."""
        sums = stats[0] if stats else None
        if low is not None:
            return ops.decoder_conv_fprop(x0, low, wf, bias, cout_p, relu=relu, out=out, up_out=up_out, scale=scale, stats=sums)
        if scale is not None:
            return ops.conv_fprop_scaled(x0, wf, scale, bias, cout_p, taps=taps, relu=relu, x1=x1, out=out)
        return ops.conv_fprop(x0, wf, bias, cout_p, taps=taps, relu=relu, x1=x1, out=out, stats=sums)

    def _conv_param_grads(self, x0, dz, grads, has, w, b, cout, c0, c1=0, x1=None, taps=9, pre_bn=False, first_cin=0,
                          lo_half=False, db_stats=None):
        """Weight gradient grads[w] and bias gradient grads[b] of a stride-1 conv over x0 (+ x1) with output gradient dz (a
        stride-2 conv passes its stride-1 form: zero-inserted dz, or the subsampled x0 of a 1x1).  c0 / c1: real input channels of the two sources (x0 / x1 hold them zero-padded); cout: real output channels.
        first_cin: x0 is the im2col of a first_cin-channel image (UNetEngine's first layer); lo_half: x0's channels
        [c0, 2 c0) are the lo half of the image split and add to the same weights; pre_bn: a BatchNorm reads the output;
        db_stats: (column sums, rows) of dz that the dgrad producing it left behind (UNetEngine.bias_from_dgrad)."""
        cout_p, c0_p, c1_p = dz.shape[3], x0.shape[3], (x1.shape[3] if x1 is not None else 0)
        direct = cout_p == cout and (first_cin or (c0_p == c0 and c1_p == c1))
        fuse_b = has(w) and has(b) and direct and taps == 9 and not pre_bn and self.fused_db(cout_p)
        if has(w):
            need = ops.lib().b2u_conv_wgrad_workspace(dz.shape[0], dz.shape[1], dz.shape[2], c0_p + c1_p, cout_p, taps)
            ws = self._workspace("wgrad", need)
            if direct:
                ops.conv_wgrad(x0, dz, taps=taps, x1=x1, first_cin=first_cin, dw=grads[w], db=grads[b] if fuse_b else None,
                               ws=ws)
            else:       # padded operands: gradient of the padded weight, then keep the real rows / columns
                k = 3 if taps == 9 else 1
                tmp = self._buf("dw:" + w, (cout_p, first_cin, 3, 3) if first_cin else (cout_p, c0_p + c1_p, k, k),
                                torch.float32)
                ops.conv_wgrad(x0, dz, taps=taps, x1=x1, first_cin=first_cin, dw=tmp, ws=ws)
                gw = grads[w]
                if first_cin:
                    gw.copy_(tmp[:cout])
                else:
                    gw[:, :c0].copy_(tmp[:cout, :c0])
                    if lo_half:
                        gw[:, :c0].add_(tmp[:cout, c0:2 * c0])
                    if c1:
                        gw[:, c0:].copy_(tmp[:cout, c0_p:c0_p + c1])
        if has(b) and pre_bn:
            # a bias in front of BatchNorm: dz = a (g - mean(g) - xhat mean(g xhat)) sums to zero over the batch exactly,
            # so the gradient is 0 (the reference's autograd returns fp32 cancellation residue ~1e-8)
            grads[b].zero_()
        elif has(b) and not fuse_b and db_stats is not None:
            ops.bias_from_stats(db_stats[0], db_stats[1], cout_p, db=grads[b])
        elif has(b) and not fuse_b:
            ws = self._workspace("bias", ops.lib().b2u_bias_grad_workspace(cout_p))
            if cout_p == cout:
                ops.bias_grad(dz, db=grads[b], ws=ws)
            else:
                tb = ops.bias_grad(dz, db=self._buf("dbias:" + w, (cout_p,), torch.float32), ws=ws)
                grads[b].copy_(tb[:cout])

    # ------------------------------------------------------------------ classifier head
    def _head_weight(self, params, w, cin):
        return self._padded("head:w", params[w].reshape(self.num_classes, cin), (self.num_classes, 64))

    def _head_fwd(self, x, params, w, b, cin):
        """1x1 classifier -> fp32 NCHW logits: on the tensor cores ([hi | lo] bf16 split of the fp32 weights); the fp32
        validation build runs a plain fp32 1x1 conv."""
        wh = self._head_weight(params, w, cin)
        if ops.act_dtype() == torch.float32:
            return ops.head_fwd(x, wh, params[b])
        wf = ops.pack_head_fprop(wh, wf=self._buf("head:wf", (64 * ops.head_groups(self.num_classes), 64)))
        return ops.head_fwd_tc(x, wf, params[b], self.num_classes)

    def _head_bwd(self, dlogits, x, params, grads, has, w, b, cin, g, mask, bits=None, grad_stream=contextlib.nullcontext):
        """Backward of _head_fwd: the gradient wrt x into g (None: not needed), ReLU-masked by mask (= x) or by bits (x's bit
        mask) when given; grads[w] / grads[b] from weight-gradient launches run under grad_stream()."""
        C = self.num_classes
        wh = self._head_weight(params, w, cin)
        fw, fb = has(w), has(b)
        cz = 64 * ops.head_groups(C)
        if dlogits.dtype == torch.bfloat16 and dlogits.dim() == 4 and dlogits.shape[-1] == cz and ops.act_dtype() == torch.bfloat16:
            # [N,H,W,64 G] = per group of 32 classes, [hi | lo] split dlogits from loss_bwd(nhwc64=True): the head's backward
            # runs on the tensor cores as a 1x1 dgrad (+ReLU mask) and a 1x1 wgrad (+bias) over G x 2 x 32 padded classes
            dl = dlogits.contiguous()
            if g is not None:
                wd = ops.pack_head_dgrad(wh, wd=self._buf("head:wd", (64, cz)))
                if bits is not None:
                    ops.conv_dgrad_bits(dl, wd, 64, bits, taps=1, out0=g)
                else:
                    ops.conv_dgrad(dl, wd, 64, taps=1, mask=mask, out0=g)
            if fw or fb:
                dw64 = self._buf("head:dw", (cz, 64, 1, 1), torch.float32)
                db64 = self._buf("head:db", (cz,), torch.float32)
                need = ops.lib().b2u_conv_wgrad_workspace(dl.shape[0], dl.shape[1], dl.shape[2], 64, cz, 1)
                with grad_stream():
                    ops.conv_wgrad(x, dl, taps=1, dw=dw64, db=db64, ws=self._workspace("wgrad", need))
                    # in group g, rows 64g + [0,32) came from the hi half of dlogits, rows 64g + [32,64) from the lo half
                    if fw:
                        ops.fold_head_groups(dw64, C, cin, grads[w])
                    if fb:
                        ops.fold_head_groups(db64, C, cin, grads[b])
        else:
            dl = dlogits.float().contiguous() if dlogits.dtype != torch.float32 else dlogits.contiguous()
            dwt = None
            if fw:
                dwt = grads[w] if cin == 64 else self._buf("head:dwf", (C, 64, 1, 1), torch.float32)
            ops.head_bwd(dl, x, wh, need_dx=g is not None, need_dw=fw or fb, relu_mask=mask is not None, dx=g, dw=dwt,
                         db=grads[b] if fb else None, ws=self._workspace("head", ops.lib().b2u_head_bwd_workspace_cls(C)))
            if fw and cin != 64:
                grads[w].copy_(dwt[:, :cin])
