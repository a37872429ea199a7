"""Drop-in for the reference's predictor class `unet.py::Unet` (lines 19-357): same keyword configuration
(`model_path`, `num_classes`, `backbone`, `input_shape`, `mix_type`, `cuda`), same `detect_image`, `get_FPS`,
`get_miou_png` results -- with the per-frame work moved onto the GPU (SURVEY.md 8(f) rank 1) and batched.

Reference per frame: PIL BICUBIC letterbox with grey bars -> / 255 -> batch-1 forward -> softmax -> .cpu().numpy()
(H x W x C fp32, 22 MB at C = 21, 512^2) -> crop of the letterbox bars -> cv2.resize of the probabilities to the original
size -> argmax (utils/utils.py:22-34, unet.py:116-148).  Here, per batch of images of any sizes: the raw uint8 RGB bytes
go up in one pinned copy, `b2u_letterbox_bicubic` builds the network input (bit-exact with PIL's BICUBIC resize and
numpy's / 255), one forward runs the whole batch, and `b2u_softmax_resize_argmax_u8_batch` (softmax + crop +
INTER_LINEAR resize + argmax) writes every image's uint8 mask into one flat buffer, the only thing copied back.
`detect_images` renders on the device too (`b2u_render_batch`: palette, Pillow's 0.7 blend or the kept foreground, and
the per-class pixel counts), so only the rendered RGB images come back.  RGB conversion (`cvtColor`) stays on the host.

`model` selects the network: "unet" (nets/unet.py::Unet with `backbone`, the reference's default) or one of the other
families the trainer runs (FAMILIES).  LightweightUnet's logits are half the input size; they are resized to the input
size with the bilinear, align_corners=True resize its losses use, and the tail then runs as for every other family."""
import colorsys
import itertools
import time

import numpy as np
import torch
from PIL import Image

from . import ops
from .nets.LightWeightUnet import LightweightUnet
from .nets.RepVGG_Unet import ImprovedSegNet
from .nets.TraditionalUnet import TraditionalUnet
from .nets.UltraLightweightUnet import UltraLightweightUnet
from .nets.UltraLightweightUnet_large import UltraLightweightUnet_large
from .nets.UltraLightweightUnet_large_optimized import UltraLightweightUnet_large_optimized
from .nets.unet import Unet as unet

# the `model` names other than "unet", as UnetTrainer names the families
FAMILIES = {"traditional": TraditionalUnet, "lightweight": LightweightUnet, "ultralight": UltraLightweightUnet,
            "ultralight_large": UltraLightweightUnet_large, "ultralight_large_optimized": UltraLightweightUnet_large_optimized,
            "improved_segnet": ImprovedSegNet}

def _voc_palette(n):
    """The PASCAL VOC class palette (bit-interleaved colour code of the class index) -- the table of unet.py:59-63."""
    out = []
    for i in range(n):
        r = g = b = 0
        c = i
        for j in range(8):
            r |= ((c >> 0) & 1) << (7 - j)
            g |= ((c >> 1) & 1) << (7 - j)
            b |= ((c >> 2) & 1) << (7 - j)
            c >>= 3
        out.append((r, g, b))
    return out


def cvtColor(image):                                   # utils/utils.py:12-17
    if len(np.shape(image)) == 3 and np.shape(image)[2] == 3:
        return image
    return image.convert("RGB")


def resize_image(image, size):                         # utils/utils.py:22-34: undistorted resize onto a grey canvas
    iw, ih = image.size
    w, h = size
    scale = min(w / iw, h / ih)
    nw, nh = int(iw * scale), int(ih * scale)
    canvas = Image.new("RGB", size, (128, 128, 128))
    canvas.paste(image.resize((nw, nh), Image.BICUBIC), ((w - nw) // 2, (h - nh) // 2))
    return canvas, nw, nh


def _chunks(iterable, n):
    it = iter(iterable)
    while chunk := list(itertools.islice(it, n)):
        yield chunk


class Unet(object):
    _defaults = {
        "model": "unet",
        "model_path": "model_data/unet_vgg_voc.pth",
        "num_classes": 21,
        "backbone": "vgg",
        "input_shape": [512, 512],
        "mix_type": 0,
        "cuda": True,
    }

    def __init__(self, **kwargs):
        self.__dict__.update(self._defaults)
        self.state_dict = None                         # optional: weights passed in memory instead of model_path
        for name, value in kwargs.items():
            setattr(self, name, value)
        if self.num_classes <= 21:
            self.colors = _voc_palette(22)
        else:
            hsv = [(x / self.num_classes, 1.0, 1.0) for x in range(self.num_classes)]
            self.colors = [tuple(int(v * 255) for v in colorsys.hsv_to_rgb(*t)) for t in hsv]
        self.generate()

    def generate(self, onnx=False):                    # unet.py:86-98
        if self.model != "unet" and self.model not in FAMILIES:
            raise ValueError(f"unknown model {self.model!r}; choose 'unet' or one of {sorted(FAMILIES)}")
        if not self.cuda or not torch.cuda.is_available():
            raise RuntimeError("the B200 predictor needs CUDA (cuda=True and a visible GPU); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device())
        if self.model == "unet":
            self.net = unet(num_classes=self.num_classes, backbone=self.backbone)
        else:
            self.net = FAMILIES[self.model](num_classes=self.num_classes)
        sd = self.state_dict if self.state_dict is not None else torch.load(self.model_path, map_location="cpu")
        self.net.load_state_dict(sd)
        self.net = self.net.eval().to(self.device)

    # ------------------------------------------------------------------ shared pieces
    def _letterbox(self, image):
        """The host letterbox of the reference (PIL BICUBIC + numpy); the batched path computes the same tensor on the GPU."""
        image = cvtColor(image)
        oh, ow = np.array(image).shape[:2]
        boxed, nw, nh = resize_image(image, (self.input_shape[1], self.input_shape[0]))
        data = np.expand_dims(np.transpose(np.array(boxed, np.float32) / 255.0, (2, 0, 1)), 0)     # preprocess_input
        return image, torch.from_numpy(data), nw, nh, oh, ow

    def _forward(self, x):
        """Logits at the input size: smaller logits (LightweightUnet's H/2) are resized bilinearly, align_corners=True."""
        logits = self.net(x)
        if tuple(logits.shape[-2:]) != tuple(x.shape[-2:]):
            logits = ops.resize_bilinear(logits, tuple(x.shape[-2:]))
        return logits

    def _crop(self, nw, nh):
        return (int((self.input_shape[0] - nh) // 2), int((self.input_shape[1] - nw) // 2), nh, nw)

    def _prepare(self, image):
        """Host part of one image: cvtColor (the RGB view is returned for detect_image), its uint8 [h, w, 3] bytes and
        resize_image's geometry (ih, iw, nh, nw, dy, dx)."""
        arr = np.asarray(image)
        if not (arr.ndim == 3 and arr.shape[2] == 3):       # cvtColor's test, without converting the image twice
            image = image.convert("RGB")
            arr = np.asarray(image)
        ih, iw = arr.shape[:2]
        if ih == 0 or iw == 0:
            raise ValueError(f"predictor: empty image ({iw}x{ih})")
        h, w = self.input_shape
        scale = min(w / iw, h / ih)
        nw, nh = int(iw * scale), int(ih * scale)
        if nw == 0 or nh == 0:
            raise ValueError(f"predictor: a {iw}x{ih} image letterboxes to {nw}x{nh} pixels")
        return image, np.ascontiguousarray(arr, dtype=np.uint8), (ih, iw, nh, nw, (h - nh) // 2, (w - nw) // 2)

    def _buffer(self, name, nbytes, pinned=False):
        """Staging buffers reused across batches, grown on demand (uint8)."""
        buf = getattr(self, name, None)
        if buf is None or buf.numel() < nbytes:
            nbytes = max(int(nbytes * 1.25), 4096)
            buf = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True) if pinned else \
                torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            setattr(self, name, buf)
        return buf

    def _run_batch(self, prepared, gts=None, render=None, count=False):
        """One batch on the device: a single pinned host-to-device copy of [letterbox table | tail table | histogram table |
        render table | palette | images | ground truths], the letterbox kernels into the reused input buffer, one forward,
        the batched tail and, with `render` (a mix_type, or -1 for counts only), the rendering launch.
        Returns (flat uint8 mask buffer, per-image (offset, oh, ow), total mask bytes, histogram items, rendered) where the
        histogram items (device table, count, chunks) pair each ground truth of the image's size with its mask (None
        without gts) and rendered is (flat uint8 device buffer, image offsets, bytes to read back) -- with `count`, the
        buffer starts with the int64 [b, num_classes] class counts -- or None.  Must run under torch.no_grad()."""
        b = len(prepared)
        H, W = self.input_shape
        sizes = [(ih, iw) for _, _, (ih, iw, _, _, _, _) in prepared]
        crops = [(dy, dx, nh, nw) for _, _, (_, _, nh, nw, dy, dx) in prepared]
        tail, mask_offs, mask_bytes = ops.tail_table(crops, sizes, H, W)
        masks = self._buffer("_masks", mask_bytes)
        tail_at = ops.pad16(b * ops.LETTERBOX_ITEM.size)
        hist_at = tail_at + ops.pad16(len(tail))
        counted = [i for i, g in enumerate(gts or ()) if g.size == sizes[i][0] * sizes[i][1]]   # the others are skipped
        render_at = hist_at + ops.pad16(32 * len(counted))
        pal_at = render_at + (ops.pad16(b * ops.RENDER_ITEM.size) if render is not None else 0)
        palette = np.asarray(self.colors[:self.num_classes], np.uint8).tobytes() if render is not None else b""
        off = pal_at + ops.pad16(len(palette))
        src_offs, gt_offs = [], []
        for _, arr, _ in prepared:
            src_offs.append(off)
            off = ops.pad16(off + arr.nbytes)
        for g in gts or ():
            gt_offs.append(off)
            off = ops.pad16(off + g.nbytes)
        total = off
        if getattr(self, "_staged", None) is not None:
            self._staged.synchronize()                      # the previous batch's copy has left the pinned buffer
        host, dev = self._buffer("_host_stage", total, pinned=True), self._buffer("_dev_stage", total)
        base = dev.data_ptr()
        lb, ws_bytes = ops.letterbox_plan([(base + o, *geo) for o, (_, _, geo) in zip(src_offs, prepared)], H, W)
        hist_tab, chunks = ops.hist_items([(base + gt_offs[i], masks.data_ptr() + mask_offs[i], gts[i].size) for i in counted])
        rtab = b""
        if render is not None:
            cbytes = 8 * b * self.num_classes if count else 0
            rtab, out_offs, out_bytes = ops.render_table(
                [(base + s, masks.data_ptr() + m, h, w) for s, m, (h, w) in zip(src_offs, mask_offs, sizes)], start=cbytes)
            if render < 0:
                out_bytes = ops.pad16(cbytes)
        hn = host.numpy()
        for at, blob in ((0, lb), (tail_at, tail), (hist_at, hist_tab), (render_at, rtab), (pal_at, palette)):
            hn[at:at + len(blob)] = np.frombuffer(blob, np.uint8)
        for o, (_, arr, _) in zip(src_offs, prepared):
            hn[o:o + arr.nbytes] = arr.reshape(-1)
        for o, g in zip(gt_offs, gts or ()):
            hn[o:o + g.nbytes] = g.reshape(-1)
        dev[:total].copy_(host[:total], non_blocking=True)
        self._staged = torch.cuda.Event()
        self._staged.record()
        x = getattr(self, "_input", None)
        if x is None or x.shape[0] < b:
            x = self._input = torch.empty((b, 3, H, W), dtype=torch.float32, device=self.device)
        ws = self._buffer("_lb_ws", ws_bytes)
        ops.letterbox_bicubic(dev[:len(lb)], b, x, ws)
        logits = self._forward(x[:b])
        ops.softmax_resize_argmax_u8_batch(logits, dev[tail_at:tail_at + len(tail)], b, masks,
                                           max(h for h, _ in sizes), max(w for _, w in sizes))
        hist_items = (dev[hist_at:hist_at + max(len(hist_tab), 16)], len(counted), chunks) if gts is not None else None
        rendered = None
        if render is not None:
            out = self._buffer("_render_out", out_bytes)
            ops.render_batch(dev[render_at:render_at + len(rtab)], b, dev[pal_at:pal_at + len(palette)], self.num_classes,
                             render, out, out[:cbytes].view(torch.int64) if count else None, max(h * w for h, w in sizes))
            rendered = (out, out_offs, out_bytes)
        return masks, [(o, h, w) for o, (h, w) in zip(mask_offs, sizes)], mask_bytes, hist_items, rendered

    def predict_masks(self, images, batch_size=16):
        """uint8 class maps, one per image at the image's original size, each equal to predict_mask(image)[1]; the images
        run through the device letterbox, the forward and the tail `batch_size` at a time."""
        return [m for _, m in self._predict(images, batch_size)]

    def _predict(self, images, batch_size):
        if batch_size < 1:
            raise ValueError("predict_masks: batch_size must be >= 1")
        out = []
        for chunk in _chunks(images, batch_size):
            prepared = [self._prepare(im) for im in chunk]
            with torch.no_grad():
                masks, layout, nbytes, _, _ = self._run_batch(prepared)
            host = self._buffer("_host_masks", nbytes, pinned=True)
            host[:nbytes].copy_(masks[:nbytes], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            hn = host.numpy()
            out.extend((p[0], hn[o:o + h * w].reshape(h, w).copy()) for p, (o, h, w) in zip(prepared, layout))
        return out

    def predict_mask(self, image):
        """uint8 class map at the original image size (the `pr` of unet.py:148 / 340)."""
        return self._predict([image], 1)[0]

    def predict_mask_device(self, image):
        """The same class map, left on the device (uint8 [H, W] CUDA tensor)."""
        with torch.no_grad():
            masks, [(o, h, w)], _, _, _ = self._run_batch([self._prepare(image)])
        return masks[o:o + h * w].view(h, w).clone()

    def get_miou(self, images, gts, batch_size=16):
        """get_miou.py:45-65 + utils_metrics.compute_mIoU (:58-126) without the PNG round trip: the images run in batches
        of `batch_size` (device letterbox, forward, batched tail), and each batch's masks are folded with their ground
        truths into one device-resident confusion matrix (`fast_hist_batch`), read back once at the end.
        images: iterable of PIL images; gts: iterable of label maps (PIL 'L'/'P' images or uint8 arrays, 255 = ignore);
        a pair whose sizes differ is skipped (utils_metrics.py:88-93).
        Returns (hist int64 [n, n], IoUs, PA_Recall, Precision) like compute_mIoU."""
        from .utils.utils_metrics import per_class_iu, per_class_PA_Recall, per_class_Precision
        if batch_size < 1:
            raise ValueError("get_miou: batch_size must be >= 1")
        n = self.num_classes
        hist = torch.zeros(n * n + 1, dtype=torch.int64, device=self.device)
        for chunk in _chunks(zip(images, gts), batch_size):
            prepared = [self._prepare(im) for im, _ in chunk]
            garr = [np.ascontiguousarray(np.array(gt, dtype=np.uint8)) for _, gt in chunk]
            with torch.no_grad():
                _, _, _, (table, count, chunks), _ = self._run_batch(prepared, garr)
            ops.fast_hist_batch_items(table, count, chunks, n, hist)      # one launch per batch, no host synchronisation
        h = hist.cpu().numpy()
        if h[-1] != 0:
            raise ValueError("predictions outside [0, num_classes)")
        h = h[:-1].reshape(n, n)
        return h, per_class_iu(h), per_class_PA_Recall(h), per_class_Precision(h)

    # ------------------------------------------------------------------ reference API
    def detect_images(self, images, batch_size=16, count=False):
        """unet.py:100-203 for many images: the class maps rendered on the device with the reference's mix types (0: blend
        with the palette at 0.7, 1: the palette image, 2: the non-background pixels of the image; any other value returns
        the RGB image), `batch_size` images per launch, each batch read back in one copy.  Returns PIL RGB images; with
        `count`, `self.last_counts` is the int64 [n, num_classes] array of per-class pixel counts."""
        if batch_size < 1:
            raise ValueError("detect_images: batch_size must be >= 1")
        mode = self.mix_type if self.mix_type in (0, 1, 2) else -1
        n, out, counts = self.num_classes, [], []
        for chunk in _chunks(images, batch_size):
            prepared = [self._prepare(im) for im in chunk]
            if mode < 0 and not count:
                out.extend(p[0] for p in prepared)
                continue
            with torch.no_grad():
                *_, (dev, offs, nbytes) = self._run_batch(prepared, render=mode, count=count)
            host = self._buffer("_host_render", nbytes, pinned=True)
            host[:nbytes].copy_(dev[:nbytes], non_blocking=True)
            torch.cuda.current_stream().synchronize()
            hn = host.numpy()
            if count:
                counts.append(hn[:8 * n * len(prepared)].view(np.int64).reshape(len(prepared), n).copy())
            for (image, arr, _), o in zip(prepared, offs):     # Pillow copies RGB bytes into its own 4-byte pixels
                h, w = arr.shape[:2]
                out.append(image if mode < 0 else Image.fromarray(hn[o:o + 3 * h * w].reshape(h, w, 3)))
        if count:
            self.last_counts = np.concatenate(counts) if counts else np.zeros((0, n), np.int64)
        return out

    def detect_image(self, image, count=False, name_classes=None):
        """unet.py:100-203: detect_images for one image; `count` leaves its per-class pixel counts in `self.last_counts`
        (1-D; the reference prints them as a table)."""
        out = self.detect_images([image], 1, count)[0]
        if count:
            self.last_counts = self.last_counts[0]
        return out

    def get_FPS(self, image, test_interval):           # unet.py:205-258: forward [+ resize] + per-pixel class + crop, on the host
        _, data, nw, nh, _, _ = self._letterbox(image)
        cy, cx, ch, cw = self._crop(nw, nh)
        pinned = data.pin_memory()
        host = torch.empty((1, ch, cw), dtype=torch.uint8).pin_memory()

        def frame():
            with torch.no_grad():
                logits = self._forward(pinned.to(self.device, non_blocking=True))
                host.copy_(ops.argmax_u8(logits)[:, cy:cy + ch, cx:cx + cw], non_blocking=True)
            torch.cuda.current_stream().synchronize()
        frame()
        t1 = time.time()
        for _ in range(test_interval):
            frame()
        return (time.time() - t1) / test_interval

    def get_miou_png(self, image):                     # unet.py:298-344
        _, pr = self.predict_mask(image)
        return Image.fromarray(np.uint8(pr))
