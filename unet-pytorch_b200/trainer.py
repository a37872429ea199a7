"""Data-parallel training step of the VGG16-UNet hot path: what one iteration of the reference's
`fit_one_epoch` does between the DataLoader and `loss.item()` (utils/utils_fit.py:26-97), with the model wrapped
as train.py:335-350 wraps it (one process per GPU, gradients averaged across ranks).

  train_step(imgs, pngs):  [H2D] -> forward -> CE|Focal (+Dice) (+f_score) -> backward -> bucketed all-reduce
                           (overlapped with the remaining wgrad/dgrad kernels) -> Adam/SGD step

All parameters, gradients and optimizer moments live in flat fp32 buffers laid out in *backward completion order*
(final, up_concat1.conv2, ..., vgg.features.0) so each all-reduce bucket is one contiguous slice that becomes
ready front to back, and one kernel launch updates every parameter.  Like DDP in the reference, every rank
normalises its loss over its own shard and the ranks' gradients are averaged (SURVEY.md 8e).
"""
import functools
import os

import torch
import torch.distributed as dist

from . import ops
from .engine import TraditionalUnetEngine, VGGUnetEngine, vgg_unet_param_shapes
from .graph import ImprovedSegNetEngine, LightweightUnetEngine, ResNet50UnetEngine, UltraLightUnetEngine


def _backward_order(names):
    """state_dict order -> order in which VGGUnetEngine.backward completes the gradients."""
    def layer(n):
        return n.rsplit(".", 1)[0]
    layers = []
    for n in names:
        if layer(n) not in layers:
            layers.append(layer(n))
    enc = [l for l in layers if l.startswith("vgg.")]
    dec = [l for l in layers if l.startswith("up_concat")]
    # decoder executes up_concat4 .. up_concat1 (conv1, conv2); backward walks it in reverse, then the encoder in reverse
    dec_exec = sorted(dec, key=lambda l: (-int(l[len("up_concat")]), l.endswith("conv2")))
    order = ["final"] + dec_exec[::-1] + enc[::-1]
    out = []
    for l in order:
        out += [l + ".weight", l + ".bias"]
    assert sorted(out) == sorted(names)
    return out


class FlatBuckets:
    """Flat fp32 storage for a set of named tensors + contiguous buckets for gradient all-reduce.
    Device-agnostic (the gloo tests run it on CPU)."""

    def __init__(self, shapes, order, device, bucket_bytes=16 << 20):
        self.order = list(order)
        self.offsets = {}
        off = 0
        for n in self.order:
            numel = 1
            for s in shapes[n]:
                numel *= s
            self.offsets[n] = (off, numel, tuple(shapes[n]))
            off += (numel + 3) // 4 * 4            # 16-byte aligned slices
        self.total = off
        self.device = device
        # buckets: consecutive parameters until bucket_bytes is reached
        self.buckets = []          # (start, end, [names])
        start, names = 0, []
        for n in self.order:
            o, numel, _ = self.offsets[n]
            names.append(n)
            end = o + (numel + 3) // 4 * 4
            if (end - start) * 4 >= bucket_bytes:
                self.buckets.append((start, end, names))
                start, names = end, []
        if names:
            self.buckets.append((start, self.total, names))
        self.bucket_of = {n: bi for bi, (_, _, ns) in enumerate(self.buckets) for n in ns}

    def new_buffer(self):
        return torch.zeros(self.total, dtype=torch.float32, device=self.device)

    def views(self, flat):
        return {n: flat[o:o + numel].view(shape) for n, (o, numel, shape) in self.offsets.items()}


class GradientSync:
    """Bucketed all-reduce (sum) of a flat gradient buffer on a side stream, fired as buckets complete."""

    def __init__(self, layout, flat_grad, group=None, enabled=None):
        self.layout = layout
        self.flat = flat_grad
        self.group = group
        self.world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        self.enabled = (self.world > 1) if enabled is None else enabled
        self.cuda = flat_grad.is_cuda
        self.stream = torch.cuda.Stream(device=flat_grad.device) if (self.cuda and self.enabled) else None
        # Wire format of the gradient buckets.  "fp32" (default) is what DistributedDataParallel sends for the reference
        # (train.py:346).  "bf16" halves the bytes on NVLink (49.8 MB instead of 99.6 MB for Unet-VGG16, the payload SURVEY.md
        # 8(d)/(e) plans with): each bucket is rounded to bf16 on the communication stream, summed by NCCL in bf16 and widened
        # back into the fp32 gradient buffer; every rank still receives bit-identical sums.  B2U_GRAD_WIRE=bf16 selects it.
        self.wire = os.environ.get("B2U_GRAD_WIRE", "fp32").lower()
        if self.wire not in ("fp32", "bf16"):
            raise ValueError("B2U_GRAD_WIRE must be fp32 or bf16")
        self._wire_bufs = {}
        self._pending = None
        self._handles = []
        self.reset()

    def reset(self, active=None):
        """active: names that will be reported ready this step (default: all)."""
        names = set(self.layout.order if active is None else active)
        self._pending = [sum(1 for n in ns if n in names) for (_, _, ns) in self.layout.buckets]
        self._handles = []

    def _fire(self, bi):
        s, e, _ = self.layout.buckets[bi]
        view = self.flat[s:e]
        if self.cuda:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self.stream.wait_event(ev)
            with torch.cuda.stream(self.stream):
                if self.wire == "bf16":
                    tmp = self._wire_bufs.get(bi)
                    if tmp is None:
                        tmp = self._wire_bufs[bi] = torch.empty(e - s, dtype=torch.bfloat16, device=self.flat.device)
                    tmp.copy_(view)
                    dist.all_reduce(tmp, op=dist.ReduceOp.SUM, group=self.group)
                    view.copy_(tmp)
                else:
                    dist.all_reduce(view, op=dist.ReduceOp.SUM, group=self.group)
        else:
            self._handles.append(dist.all_reduce(view, op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def ready(self, names):
        if not self.enabled:
            return
        for n in names:
            bi = self.layout.bucket_of[n]
            self._pending[bi] -= 1
            if self._pending[bi] == 0:
                self._fire(bi)

    def finish(self):
        """Makes the current stream wait for all fired buckets; returns the factor that turns the sum into a mean."""
        if not self.enabled:
            return 1.0
        if self.cuda:
            torch.cuda.current_stream().wait_stream(self.stream)
        else:
            for h in self._handles:
                h.wait()
        return 1.0 / self.world


class UnetTrainer:
    """model: "unet_vgg" / "unet_resnet50" (nets/unet.py::Unet with backbone 'vgg' / 'resnet50'), "traditional"
    (nets/TraditionalUnet.py) or "ultralight" / "ultralight_large" / "ultralight_large_optimized"
    (nets/UltraLightweightUnet*.py) or "lightweight" (nets/LightWeightUnet.py; logits at H/2, resized inside the loss) or
    "improved_segnet" (nets/RepVGG_Unet.py::ImprovedSegNet, RepVGG blocks in their training form)."""

    ENGINES = {"unet_vgg": VGGUnetEngine, "traditional": TraditionalUnetEngine, "unet_resnet50": ResNet50UnetEngine,
               "lightweight": LightweightUnetEngine, "improved_segnet": ImprovedSegNetEngine,
               "ultralight": functools.partial(UltraLightUnetEngine, variant="ultralight"),
               "ultralight_large": functools.partial(UltraLightUnetEngine, variant="ultralight_large"),
               "ultralight_large_optimized": functools.partial(UltraLightUnetEngine, variant="ultralight_large_optimized")}

    def __init__(self, num_classes=21, device=None, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0,
                 optimizer="adam", momentum=0.9, cls_weights=None, dice_loss=True, focal_loss=False,
                 state_dict=None, process_group=None, bucket_mb=16, compute_f_score=True, model="unet_vgg", sync_bn=False):
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("UnetTrainer needs a CUDA device (no CPU fallback)")
        if model not in self.ENGINES:
            raise ValueError(f"unknown model {model!r}; choose from {sorted(self.ENGINES)}")
        self.num_classes = num_classes
        self.engine = self.ENGINES[model](num_classes, device=self.device)
        shapes = self.engine.param_shapes()
        self.names = list(shapes.keys())                       # trainable tensors, state_dict order
        self.layout = FlatBuckets(shapes, self.engine.backward_param_order(), self.device, bucket_bytes=bucket_mb << 20)
        self.flat_param = self.layout.new_buffer()
        self.flat_grad = self.layout.new_buffer()
        self.params = self.layout.views(self.flat_param)
        self.grads = self.layout.views(self.flat_grad)
        # BatchNorm buffers: not optimised, kept beside the flat parameters (train.py's DDP broadcasts them from rank 0)
        self.buffers = {}
        for n, shp in self.engine.buffer_shapes().items():
            if n.endswith("running_var"):
                self.buffers[n] = torch.ones(shp, dtype=torch.float32, device=self.device)
            elif n.endswith("num_batches_tracked"):
                self.buffers[n] = torch.zeros(shp, dtype=torch.int64, device=self.device)
            else:
                self.buffers[n] = torch.zeros(shp, dtype=torch.float32, device=self.device)
        self.tensors = dict(self.params)
        self.tensors.update(self.buffers)
        self.opt_kind = optimizer
        self.lr, self.betas, self.eps, self.weight_decay, self.momentum = lr, betas, eps, weight_decay, momentum
        self.m = self.layout.new_buffer()
        self.v = self.layout.new_buffer() if optimizer == "adam" else None
        self.step_count = 0
        self.steps = {}                 # per-tensor optimizer step count (torch.optim keeps `state['step']` per parameter)
        self.dice, self.focal, self.compute_f_score = dice_loss, focal_loss, compute_f_score
        cw = torch.ones(num_classes) if cls_weights is None else torch.as_tensor(cls_weights, dtype=torch.float32)
        self.cls_w = cw.to(self.device).contiguous()
        self.sync = GradientSync(self.layout, self.flat_grad, group=process_group)
        if sync_bn and self.sync.world > 1:       # train.py:66, 335-336: BatchNorm statistics over all ranks
            self.engine.sync_bn_group = process_group if process_group is not None else dist.group.WORLD
        self.trainable = set(self.names)
        self.backbone_prefixes = {"unet_vgg": ("vgg.",), "unet_resnet50": ("resnet.",)}.get(
            model, ("backbone.",) if model == "lightweight" else ("enc", "se") if model.startswith("ultralight") else ("inc.", "down1.", "down2.", "down3."))
        self._gscale = torch.tensor([0.0 if focal_loss else 1.0, 1.0 if focal_loss else 0.0, 1.0 if dice_loss else 0.0],
                                    dtype=torch.float32, device=self.device)
        self._copy_stream = torch.cuda.Stream(device=self.device)
        self._staged = None
        self._slots = [None, None]
        self._stage_count = 0
        self.last = None
        if state_dict is None:       # random init (the reference's weights_init / _initialize_weights role)
            from .synthetic import random_state_dict
            state_dict = random_state_dict(shapes, self.engine.buffer_shapes(), seed=0)
        self.load_state_dict(state_dict)
        if self.sync.world > 1:
            dist.broadcast(self.flat_param, src=0, group=process_group)      # DDP ctor semantics (train.py:346)

    # ------------------------------------------------------------------ state
    def load_state_dict(self, sd):
        with torch.no_grad():
            for n in self.names:
                self.params[n].copy_(sd[n].to(self.device, dtype=torch.float32))
            for n, b in self.buffers.items():
                if n in sd:
                    b.copy_(sd[n].to(self.device, dtype=b.dtype))
        self.engine.invalidate_packed_weights()

    def state_dict(self):
        sd = {n: self.params[n].detach().clone() for n in self.names}
        sd.update({n: b.detach().clone() for n, b in self.buffers.items()})
        return sd

    def freeze_backbone(self):
        """nets/unet.py:80-86 / nets/TraditionalUnet.py:95-104 (freeze_encoder)"""
        self.trainable = {n for n in self.names if not n.startswith(self.backbone_prefixes)}

    def unfreeze_backbone(self):
        self.trainable = set(self.names)

    # ------------------------------------------------------------------ input staging
    def stage(self, imgs, pngs):
        """Asynchronous host->device copy of the next batch (pinned host tensors) on a copy stream into one of two
        persistent device slots, so the copy overlaps the current step's kernels and no allocation happens per step.
        A slot is overwritten only after the step that read it has consumed it (event recorded after its last read)."""
        slot = self._stage_count % 2
        self._stage_count += 1
        bufs = self._slots[slot]
        if (bufs is None or bufs[0].shape != imgs.shape or bufs[0].dtype != imgs.dtype or bufs[1].shape != pngs.shape
                or bufs[1].dtype != pngs.dtype):
            # fp32 NCHW images (what the reference's dataloader yields) or raw uint8 NHWC images (device input pipeline)
            bufs = [torch.empty(imgs.shape, dtype=torch.uint8 if imgs.dtype == torch.uint8 else torch.float32, device=self.device),
                    torch.empty(pngs.shape, dtype=pngs.dtype, device=self.device), None]
            self._slots[slot] = bufs
        with torch.cuda.stream(self._copy_stream):
            if bufs[2] is not None:
                self._copy_stream.wait_event(bufs[2])          # previous reader of this slot is done
            bufs[0].copy_(imgs, non_blocking=True)
            bufs[1].copy_(pngs, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        self._staged = (slot, ev)

    def _take(self, imgs, pngs):
        """Returns (imgs, pngs, slot): device tensors for this step; slot is None for caller-owned tensors."""
        if imgs is None:
            if self._staged is None:
                raise RuntimeError("train_step(None, None) needs a batch staged with stage()")
            slot, ev = self._staged
            self._staged = None
            torch.cuda.current_stream().wait_event(ev)
            imgs, pngs = self._device_preprocess(self._slots[slot][0], self._slots[slot][1])
            return imgs, pngs, slot
        if not imgs.is_cuda:
            imgs = imgs.to(self.device, non_blocking=True)
        if not pngs.is_cuda:
            pngs = pngs.to(self.device, non_blocking=True)
        imgs, pngs = self._device_preprocess(imgs, pngs)
        return imgs, pngs, None

    def _device_preprocess(self, imgs, pngs):
        """Raw uint8 inputs (NHWC image batch, uint8 label map) -> what the dataloader would have produced on the host
        (utils/dataloader.py:41-43): fp32 NCHW image / 255 and an int64 label map, on the device."""
        if imgs.dtype == torch.uint8:
            n, h, w, c = imgs.shape
            imgs = ops.u8hwc_to_nchw_f32(imgs.contiguous(), out=self.engine._buf("in:f32", (n, c, h, w), torch.float32))
        if pngs.dtype == torch.uint8:
            pngs = ops.u8_to_i64(pngs.contiguous(), out=self.engine._buf("in:i64", tuple(pngs.shape), torch.int64))
        return imgs, pngs

    def _consumed(self, slot):
        if slot is not None:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self._slots[slot][2] = ev

    # ------------------------------------------------------------------ the step
    def forward_loss(self, imgs, pngs, save=True):
        logits = self.engine.forward(imgs, self.tensors, save=save, trainable=self.trainable)
        if pngs.dtype != torch.int64:
            pngs = pngs.long()
        if logits.shape[2] != pngs.shape[1] and logits.shape[3] != pngs.shape[2]:
            # LightweightUnet: logits at H/2 x W/2 are resized to the label size inside the loss (unet_training.py:12-13)
            logits = ops.resize_bilinear(logits, tuple(pngs.shape[1:]))
        # alpha = 0 makes the focal term exactly zero and lets the kernel skip its powf / expf when the loop does not ask for it
        fin = ops.loss_fwd(logits, target=pngs.contiguous(), onehot=None, cls_w=self.cls_w, alpha=0.5 if self.focal else 0.0)
        return logits, pngs, fin

    def train_step(self, imgs=None, pngs=None):
        """Returns a device tensor [total loss, f_score]; `.item()`/`.tolist()` on it is the per-iteration sync of
        utils_fit.py:96-97."""
        imgs, pngs, slot = self._take(imgs, pngs)
        logits, pngs, fin = self.forward_loss(imgs, pngs, save=True)
        n, _, h, w = logits.shape
        stride = getattr(self.engine, "logit_stride", 1)
        if stride == 1 and ops.act_dtype() == torch.bfloat16:
            dlogits = ops.loss_bwd(logits, fin, self._gscale, target=pngs, onehot=None, cls_w=self.cls_w, nhwc64=True,
                                   out=self.engine._buf("g:logits64", (n, h, w, 64 * ops.head_groups(self.num_classes))))
        elif stride == 1:       # fp32 validation build: fp32 NCHW dlogits, plain fp32 head backward
            dlogits = ops.loss_bwd(logits, fin, self._gscale, target=pngs, onehot=None, cls_w=self.cls_w)
        else:       # gradient at label resolution (fp32), then the adjoint of the resize back to the logits' own size
            dfull = ops.loss_bwd(logits, fin, self._gscale, target=pngs, onehot=None, cls_w=self.cls_w)
            dlogits = ops.resize_bilinear_bwd(dfull, (h // stride, w // stride))
        self._consumed(slot)            # image and label map are not read after this point
        active = [n for n in self.layout.order if n in self.trainable]
        self.sync.reset(active)
        grads = {n: self.grads[n] for n in active}
        self.engine.backward(dlogits, self.tensors, grads, trainable=self.trainable, on_grads_ready=self.sync.ready)
        scale = self.sync.finish()
        self.optimizer_step(scale)
        loss = self._total(fin)
        self.last = torch.stack([loss, fin[3]])
        return self.last

    def _total(self, fin):
        """CE | Focal (+ Dice), utils_fit.py:74-81"""
        loss = fin[1] if self.focal else fin[0]
        return loss + fin[2] if self.dice else loss

    def _update_ranges(self):
        """Contiguous slices of the flat buffers to update this step, as (start, end, step count) -- torch.optim semantics for
        frozen parameters (train.py:382-383 flips requires_grad, so their .grad is None and the optimizer skips them: no
        update, no weight decay, no moment decay, and their per-parameter `step` only starts counting once they receive
        gradients).  The layout is in backward-completion order, so the decoder and the backbone are one or two slices each;
        neighbouring trainable tensors with the same step count are merged into one launch."""
        ranges = []
        for n in self.layout.order:
            if n not in self.trainable:
                continue
            o, numel, _ = self.layout.offsets[n]
            e = o + (numel + 3) // 4 * 4
            st = self.steps.get(n, 0) + 1
            self.steps[n] = st
            if ranges and ranges[-1][1] == o and ranges[-1][2] == st:
                ranges[-1][1] = e
            else:
                ranges.append([o, e, st])
        return ranges

    def optimizer_step(self, grad_scale=1.0):
        self.step_count += 1
        for s, e, st in self._update_ranges():
            if self.opt_kind == "adam":
                ops.adam_step(self.flat_param[s:e], self.flat_grad[s:e], self.m[s:e], self.v[s:e], st, self.lr, self.betas,
                              self.eps, self.weight_decay, grad_scale)
            else:
                ops.sgd_step(self.flat_param[s:e], self.flat_grad[s:e], self.m[s:e], self.lr, self.momentum, self.weight_decay,
                             True, st == 1, grad_scale)
        # the flat update wrote every parameter behind torch's back: invalidate the engine's packed-weight cache
        self.engine.invalidate_packed_weights()

    @torch.no_grad()
    def eval_step(self, imgs, pngs):
        """Validation iteration (utils_fit.py:111-151): forward + losses + f_score, no gradient."""
        imgs, pngs, slot = self._take(imgs, pngs)
        _, _, fin = self.forward_loss(imgs, pngs, save=False)
        self._consumed(slot)
        return torch.stack([self._total(fin), fin[3]])
