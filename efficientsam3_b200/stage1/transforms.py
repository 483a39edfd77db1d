"""Input preprocessing on the device: decoded images in, the model's [B,3,S,S] fp32 input out.

Replaces the CPU work between decoding and the encoder:
  * stage-1 loaders (stage1/data/sa1b_dataset.py:68-69, 163-171, 216-227, coco_dataset.py:146-153): pil_to_tensor ->
    ResizeLongestSide.apply_image_torch (transforms.py:48-54, antialiased bilinear to the longest side) -> norm -> pad;
  * the interactive predictor's SAM2Transforms (sam3/sam3/model/utils/sam1_utils.py:17-41): ToTensor -> Resize((S,S))
    antialiased -> Normalize(0.5, 0.5).

`ImagePreprocessor` takes a list of uint8 or fp32 images, CHW or HWC, of any size, on the host or on the device, and runs
one es3_preprocess_images call for the whole list.  Host images are packed, with the image table, into one pinned staging
buffer and sent in one host-to-device copy; host tensors that are already pinned and contiguous are copied straight from
their memory (asynchronously: leave them unchanged until the stream has passed the call); CUDA images are read in place
through their strides.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from .. import ops

TABLE_FIELDS = 16
# Descriptor fields, in the order csrc/preprocess.cu reads them.
(F_PTR, F_SC, F_SH, F_SW, F_IN_H, F_IN_W, F_OUT_H, F_OUT_W, F_DTYPE, F_PLANES, F_XC, F_KX, F_KY, F_TAPX, F_TAPY) = range(15)
SLOT_ROW = 768        # bytes of one staged input row in the kernel's shared memory (PP_SLOT_ROW)
ALIGN = 256           # byte alignment of each image and of the table inside the staging buffer
_DTYPES = {torch.uint8: 0, torch.float32: 1}


def get_preprocess_shape(oldh: int, oldw: int, long_side_length: int) -> tuple[int, int]:
    """Output (h, w) with the longest side at `long_side_length`, rounded as the reference does (transforms.py:80-85)."""
    scale = long_side_length * 1.0 / max(oldh, oldw)
    newh, neww = oldh * scale, oldw * scale
    return int(newh + 0.5), int(neww + 0.5)


class ResizeLongestSide:
    """The image-size part of the reference's ResizeLongestSide (stage1/data/transforms.py): the resampling itself runs in
    ImagePreprocessor."""

    get_preprocess_shape = staticmethod(get_preprocess_shape)

    def __init__(self, target_length: int):
        self.target_length = int(target_length)

    def target_size(self, h: int, w: int) -> tuple[int, int]:
        return get_preprocess_shape(h, w, self.target_length)


def taps_per_output(in_size: int, out_size: int) -> int:
    """Tap-record width of one axis: torch's max_interp_size = ceil(support) * 2 + 1 with support = max(in / out, 1) in fp32."""
    scale = float(np.float32(in_size) / np.float32(out_size))
    return int(math.ceil(max(scale, 1.0))) * 2 + 1


def image_layout(shape, strides, hwc: bool):
    """(h, w, channel / row / column element strides) of a 3-channel image tensor."""
    if len(shape) != 3:
        raise ValueError(f"expected a 3-D image, got shape {tuple(shape)}")
    if hwc:
        (h, w, c), (sh, sw, sc) = shape, strides
    else:
        (c, h, w), (sc, sh, sw) = shape, strides
    if c != 3:
        raise ValueError(f"expected 3 channels ({'HWC' if hwc else 'CHW'}), got shape {tuple(shape)}")
    if h < 1 or w < 1 or sw < 1 or sc < 0 or sh < 0:
        raise ValueError(f"unsupported image shape / strides {tuple(shape)} / {tuple(strides)}")
    return h, w, sc, sh, sw


def describe(address: int, dtype_code: int, h: int, w: int, sc: int, sh: int, sw: int, out_hw) -> np.ndarray:
    """One descriptor row (tap offsets left at 0; build_table fills them)."""
    es = 1 if dtype_code == 0 else 4
    planes = 1 if sc < sw else 3             # interleaved channels share one staged span per row
    extra = 2 * sc if planes == 1 else 0
    room = (SLOT_ROW // planes - 15) // es   # elements of one staging slot, less the 16-byte alignment slack
    if room - 1 - extra < 0:
        raise ValueError(f"image strides {(sc, sh, sw)} are too wide to stage one column")
    oh, ow = out_hw
    if oh < 1 or ow < 1:
        raise ValueError(f"a {h}x{w} image resizes to {oh}x{ow}: nothing to sample")
    d = np.zeros(TABLE_FIELDS, dtype=np.int64)
    d[[F_PTR, F_SC, F_SH, F_SW, F_IN_H, F_IN_W, F_OUT_H, F_OUT_W, F_DTYPE, F_PLANES]] = (
        address, sc, sh, sw, h, w, oh, ow, dtype_code, planes)
    d[F_XC] = (room - 1 - extra) // sw + 1
    d[F_KX], d[F_KY] = taps_per_output(w, ow), taps_per_output(h, oh)
    return d


def build_table(rows) -> tuple[np.ndarray, int, int]:
    """Stack descriptor rows and lay their tap records out back to back: -> (table [B,16] int64, tap floats, largest output side)."""
    table = np.stack(rows).astype(np.int64)
    off = 0
    for d in table:
        d[F_TAPX] = off
        off += int(d[F_OUT_W]) * (int(d[F_KX]) + 2)
        d[F_TAPY] = off
        off += int(d[F_OUT_H]) * (int(d[F_KY]) + 2)
    return table, off, int(max(table[:, F_OUT_H].max(), table[:, F_OUT_W].max()))


def _dtype_code(t) -> int:
    return _DTYPES[t.dtype] if torch.is_tensor(t) else (0 if t.dtype == np.uint8 else 1)


def _align(n: int) -> int:
    return (n + ALIGN - 1) // ALIGN * ALIGN


class ImagePreprocessor:
    """Decoded images -> (x [B,3,S,S] fp32 CUDA, img_size_before_pad [(3, h, w), ...]).

    Each image is resized with torch's antialiased bilinear filter (align_corners=False) to the reference's longest-side size
    (`square=True`: to S x S, SAM2Transforms), normalised as (x - pixel_mean) / pixel_std, and zero padded to S x S.
    pixel_mean / pixel_std are in the units of uint8 images; fp32 images are multiplied by `float_scale` first (255 for
    ToTensor's [0, 1] float convention, 1 for float images on the 0-255 scale).

    Images: numpy arrays, PIL images or torch tensors, uint8 or fp32 (other float dtypes are converted to fp32), 3 channels.
    Layout: torch tensors are CHW unless their first dimension is not 3 (then HWC); numpy arrays and PIL images are HWC unless
    their last dimension is not 3 (then CHW).  `out=` takes a preallocated [B,3,S,S] fp32 CUDA buffer."""

    def __init__(self, img_size: int, pixel_mean=(123.675, 116.28, 103.53), pixel_std=(58.395, 57.12, 57.375),
                 square: bool = False, float_scale: float = 1.0, device=None):
        self.img_size, self.square = int(img_size), bool(square)
        mean, std = np.asarray(pixel_mean, dtype=np.float64), np.asarray(pixel_std, dtype=np.float64)
        assert mean.shape == (3,) and std.shape == (3,)
        self._affine = {0: np.concatenate([1.0 / std, -mean / std]).astype(np.float32),
                        1: np.concatenate([float_scale / std, -mean / std]).astype(np.float32)}
        self.device = torch.device(device) if device is not None else None
        self._pinned = [None, None]       # two staging buffers: packing batch i+1 overlaps batch i's copy
        self._copied = [None, None]
        self._slot = 0

    def output_size(self, h: int, w: int) -> tuple[int, int]:
        return (self.img_size, self.img_size) if self.square else get_preprocess_shape(h, w, self.img_size)

    @staticmethod
    def _as_tensor(img):
        """-> (tensor or ndarray, hwc)."""
        if torch.is_tensor(img):
            t = img if img.dtype in _DTYPES else img.float()
            return t, not (t.dim() == 3 and t.shape[0] == 3)
        a = np.asarray(img)
        if a.dtype != np.uint8 and a.dtype != np.float32:
            if not np.issubdtype(a.dtype, np.floating):
                raise TypeError(f"unsupported image dtype {a.dtype}")
            a = a.astype(np.float32)
        return a, not (a.ndim == 3 and a.shape[-1] != 3)

    def _staging(self, nbytes: int) -> torch.Tensor:
        i = self._slot
        if self._copied[i] is not None:
            self._copied[i].synchronize()   # the copy that last read this buffer has finished
        buf = self._pinned[i]
        if buf is None or buf.numel() < nbytes:
            buf = self._pinned[i] = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, pin_memory=True)
        return buf

    def __call__(self, images, out=None):
        images = list(images)
        if not images:
            raise ValueError("no images")
        S = self.img_size
        prepared = [self._as_tensor(im) for im in images]
        dev = self.device
        if dev is None:
            on_dev = [t.device for t, _ in prepared if torch.is_tensor(t) and t.is_cuda]
            dev = out.device if out is not None else (on_dev[0] if on_dev else torch.device("cuda", torch.cuda.current_device()))
        # device staging buffer: packed host images | table | affine | pinned host images.  The first three parts go through the
        # pinned staging buffer in one copy; a contiguous pinned host tensor is copied straight from its own memory.
        plan, off = [], 0
        for t, hwc in prepared:
            shape = tuple(t.shape)
            if torch.is_tensor(t) and t.is_cuda:
                if t.device != dev:
                    raise ValueError(f"image on {t.device}, expected {dev}")
                plan.append([t, hwc, shape, tuple(t.stride()), None, 0, False])
                continue
            n = int(np.prod(shape)) * (1 if _dtype_code(t) == 0 else 4)
            strides = tuple(int(np.prod(shape[k + 1:])) for k in range(3))      # contiguous in the device staging buffer
            direct = torch.is_tensor(t) and t.is_contiguous() and t.is_pinned()
            plan.append([t, hwc, shape, strides, None if direct else off, n, direct])
            if not direct:
                off = _align(off + n)
        B = len(plan)
        toff = off
        aoff = _align(toff + B * TABLE_FIELDS * 8)
        head = total = aoff + B * 6 * 4
        for p in plan:
            if p[6]:
                total = _align(total)
                p[4], total = total, total + p[5]
        staging = torch.empty(total, dtype=torch.uint8, device=dev)
        base = staging.data_ptr()
        rows, affine, sizes, in_bytes = [], np.empty((B, 6), dtype=np.float32), [], 0
        for i, (t, hwc, shape, strides, o, n, _) in enumerate(plan):
            code = _dtype_code(t)
            h, w, sc, sh, sw = image_layout(shape, strides, hwc)
            oh, ow = self.output_size(h, w)
            rows.append(describe(base + o if o is not None else t.data_ptr(), code, h, w, sc, sh, sw, (oh, ow)))
            affine[i] = self._affine[code]
            sizes.append((3, oh, ow))
            in_bytes += 3 * h * w * (1 if code == 0 else 4)
        table, taps_floats, max_out = build_table(rows)
        host = self._staging(head)
        for t, hwc, shape, strides, o, n, direct in plan:
            if o is None or direct:
                continue
            if torch.is_tensor(t):
                host[o:o + n].view(t.dtype).view(shape).copy_(t)
            else:
                np.copyto(host[o:o + n].numpy().view(t.dtype).reshape(shape), t)
        host[toff:toff + table.nbytes].numpy()[:] = table.view(np.uint8).reshape(-1)
        host[aoff:aoff + affine.nbytes].numpy()[:] = affine.view(np.uint8).reshape(-1)
        with torch.cuda.device(dev):
            staging[:head].copy_(host[:head], non_blocking=True)
            for t, _, _, _, o, n, direct in plan:
                if direct:
                    staging[o:o + n].copy_(t.reshape(-1).view(torch.uint8), non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            self._copied[self._slot] = ev
            self._slot ^= 1
            x = ops.preprocess_images(staging[toff:toff + table.nbytes].view(torch.int64).view(B, TABLE_FIELDS),
                                      staging[aoff:aoff + affine.nbytes].view(torch.float32).view(B, 6), S, max_out,
                                      taps_floats, in_bytes, out=out)
        return x, sizes
