"""The text-recognition test pipeline of mmocr 0.4 as one batched GPU step.

A recogniser config's ``test_pipeline`` (reference mmocr/datasets/pipelines/ocr_transforms.py:67-130 and mmdet's loading /
formatting transforms) is a list of per-image host transforms::

    [dict(type='LoadImageFromFile'),
     dict(type='ResizeOCR', height=32, min_width=32, max_width=128, keep_aspect_ratio=True),
     dict(type='ToTensorOCR'),
     dict(type='NormalizeOCR', mean=[0.5, 0.5, 0.5], std=[0.5, 0.5, 0.5]),
     dict(type='Collect', keys=['img'], meta_keys=['filename', 'ori_shape', 'img_shape', 'valid_ratio'])]

:class:`TestPipeline` takes that list unchanged.  The transforms registered here (registry ``PIPELINES``) hold the
reference's kwargs and the per-image host arithmetic (ResizeOCR's width rule); the pixel work -- resize, ``/255``,
mean/std normalisation and padding for the whole batch -- is one ``tpspp_ocr_prep`` launch over the packed uint8 images
(``functional.ocr_prep``), writing the [N, 3, height, max_width] fp32 tensor the recogniser reads.  Only that sequence
(Load, ResizeOCR, ToTensorOCR, NormalizeOCR, Collect) with the cv2 backend and a fixed ``max_width`` is supported, or the
rotation test-time augmentation of mmocr's attention recognisers around the last four::

    [dict(type='LoadImageFromFile'),
     dict(type='MultiRotateAugOCR', rotate_degrees=[0, 90, 270],
          transforms=[dict(type='ResizeOCR', ...), dict(type='ToTensorOCR'), dict(type='NormalizeOCR', ...),
                      dict(type='Collect', ...)])]

where each rotation of an image is one more descriptor over the same packed bytes, resampled rotated by the same launch.
"""
from __future__ import annotations

import math
import os
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import functional as TF
from .registry import PIPELINES


def _check_kwargs(name, given, allowed):
    bad = {k: v for k, v in given.items() if allowed.get(k, object()) != v}
    if bad:
        raise ValueError(f"tps_pp_b200.{name}: {bad} is not supported by the batched GPU pipeline (supported: {allowed})")


def check_image(img, index=0):
    """An input image must be a uint8 [H, W, 3] array with H, W >= 1, or a path."""
    if isinstance(img, (str, os.PathLike)):
        return
    if not isinstance(img, np.ndarray):
        raise ValueError(f"tps_pp_b200: image {index} must be a numpy array or a file path, got {type(img).__name__}")
    if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3 or img.shape[0] < 1 or img.shape[1] < 1:
        raise ValueError(f"tps_pp_b200: image {index} must be a uint8 [H, W, 3] array with H, W >= 1, got {img.dtype} {img.shape}")


@PIPELINES.register_module()
class LoadImageFromFile:
    """mmdet ``LoadImageFromFile``: ``cv2.imread(path, cv2.IMREAD_COLOR)``, i.e. uint8 BGR (mmcv's default channel order).
    Arrays passed to a pipeline that starts with it are taken as they are, as mmocr's ``model_inference`` does when it swaps
    in ``LoadImageFromNdarray``."""

    def __init__(self, **kwargs):
        _check_kwargs(type(self).__name__, kwargs, dict(to_float32=False, color_type="color", channel_order="bgr",
                                                        file_client_args=dict(backend="disk")))

    def load(self, item, index=0):
        """-> (uint8 [H, W, 3] image, filename or None)."""
        check_image(item, index)
        if isinstance(item, np.ndarray):
            return item, None
        import cv2                                # only files need OpenCV
        path = os.fspath(item)
        img = cv2.imread(path, cv2.IMREAD_COLOR)
        if img is None:
            raise ValueError(f"tps_pp_b200: could not read image file {path!r}")
        return img, path


@PIPELINES.register_module()
class LoadImageFromNdarray(LoadImageFromFile):
    """mmocr ``LoadImageFromNdarray``: the image is the uint8 array itself (no channel swap)."""


@PIPELINES.register_module()
class ResizeOCR:
    """mmocr 0.4 ``ResizeOCR`` with the cv2 backend, bilinear.  This checkout has no copy of ``ocr_transforms.py``; the
    restatement in tests/ocr_pipeline_restatement.py (``resize_width``) is the contract of :meth:`resize_width`:

    * ``keep_aspect_ratio=False``: the image is resized to (max_width, height), valid_ratio 1.0;
    * otherwise ``new_w = ceil(height / h * w)``; if ``new_w % d`` (``d = int(1 / width_downsample_ratio)``) it becomes
      ``round(new_w / d) * d`` (Python ``round``, half to even); then ``max(min_width, new_w)``; ``valid_ratio =
      min(1, new_w / max_width)``; the image is resized to ``min(max_width, new_w)`` and padded on the right to ``max_width``
      with ``img_pad_value``.

    A batch needs one width, so ``max_width`` is required."""

    def __init__(self, height, min_width=None, max_width=None, keep_aspect_ratio=True, img_pad_value=0,
                 width_downsample_ratio=1.0 / 16, backend=None):
        if backend not in (None, "cv2"):
            raise ValueError(f"tps_pp_b200.ResizeOCR: backend {backend!r} is not supported (None or 'cv2')")
        if max_width is None:
            raise ValueError("tps_pp_b200.ResizeOCR: max_width is required: a batch is one [N, 3, height, max_width] tensor")
        if isinstance(height, (tuple, list)) or int(height) != height or height < 1:
            raise ValueError(f"tps_pp_b200.ResizeOCR: height must be a positive int, got {height!r}")
        if int(max_width) != max_width or max_width < 1 or (min_width is not None and min_width < 1):
            raise ValueError(f"tps_pp_b200.ResizeOCR: max_width / min_width must be positive ints, got {max_width!r} / {min_width!r}")
        if not 0 < width_downsample_ratio <= 1:
            raise ValueError(f"tps_pp_b200.ResizeOCR: width_downsample_ratio must be in (0, 1], got {width_downsample_ratio!r}")
        if int(img_pad_value) != img_pad_value or not 0 <= img_pad_value <= 255:
            raise ValueError(f"tps_pp_b200.ResizeOCR: img_pad_value must be an int in [0, 255], got {img_pad_value!r}")
        self.height, self.min_width, self.max_width = int(height), min_width, int(max_width)
        self.keep_aspect_ratio = keep_aspect_ratio
        self.img_pad_value = int(img_pad_value)
        self.width_downsample_ratio = width_downsample_ratio
        self.backend = backend

    def resize_width(self, h: int, w: int):
        """(resize_w, valid_ratio) of an h x w image."""
        if not self.keep_aspect_ratio:
            return self.max_width, 1.0
        new_w = math.ceil(float(self.height) / h * w)
        d = int(1 / self.width_downsample_ratio)
        if new_w % d != 0:
            new_w = round(new_w / d) * d
        if self.min_width is not None:
            new_w = max(self.min_width, new_w)
        return min(self.max_width, new_w), min(1.0, 1.0 * new_w / self.max_width)


@PIPELINES.register_module()
class ToTensorOCR:
    """mmocr ``ToTensorOCR`` (torchvision ``to_tensor``: HWC uint8 -> CHW fp32 / 255)."""


@PIPELINES.register_module()
class NormalizeOCR:
    """mmocr ``NormalizeOCR`` (torchvision ``normalize``: ``(x - mean) / std`` per channel, in fp32)."""

    def __init__(self, mean, std):
        mean, std = [float(m) for m in mean], [float(s) for s in std]
        if len(mean) != 3 or len(std) != 3:
            raise ValueError(f"tps_pp_b200.NormalizeOCR: 3 means and 3 stds are needed, got {mean} / {std}")
        if any(s == 0 for s in std):
            raise ValueError(f"tps_pp_b200.NormalizeOCR: std evaluated to zero: {std}")
        self.mean, self.std = mean, std


META_KEYS = ("filename", "ori_filename", "ori_shape", "img_shape", "resize_shape", "pad_shape", "valid_ratio", "img_norm_cfg")


@PIPELINES.register_module()
class Collect:
    """mmdet ``Collect``: ``keys`` must be ``['img']``; ``meta_keys`` a subset of ``META_KEYS``."""

    def __init__(self, keys, meta_keys=("filename", "ori_shape", "img_shape", "valid_ratio")):
        if list(keys) != ["img"]:
            raise ValueError(f"tps_pp_b200.Collect: keys must be ['img'], got {keys!r}")
        unknown = [k for k in meta_keys if k not in META_KEYS]
        if unknown:
            raise ValueError(f"tps_pp_b200.Collect: meta_keys {unknown} are not produced by the pipeline (available: {META_KEYS})")
        self.keys, self.meta_keys = list(keys), list(meta_keys)


_ORDER = ((LoadImageFromFile, LoadImageFromNdarray), (ResizeOCR,), (ToTensorOCR,), (NormalizeOCR,), (Collect,))


def _build(t):
    if isinstance(t, dict):
        kind = t.get("type")
        if not isinstance(kind, str) or PIPELINES.get(kind) is None:
            raise ValueError(f"tps_pp_b200.TestPipeline: transform {kind!r} is not supported by the batched GPU pipeline "
                             f"(supported: {sorted(PIPELINES.module_dict)})")
        return PIPELINES.build(t)
    return t


class MultiRotateAugOCR:
    """mmocr 0.4 ``MultiRotateAugOCR`` (datasets/pipelines/test_time_aug.py): each image taller than it is wide (every image
    with ``force_rotate``) is read once per degree of ``rotate_degrees``, rotated counter-clockwise (``np.rot90(img, d //
    90)``); any other image once, unrotated.  ``rotate_degrees``: an int or a list of ints in [0, 360), multiples of 90; 0 is
    appended when missing; ``None`` is ``[0]``.  ``transforms`` must be ResizeOCR, ToTensorOCR, NormalizeOCR, Collect.

    It is not registered in ``PIPELINES``: :class:`TestPipeline` takes it, as a config dict or an instance, as the transform
    after the loader and runs the rotations inside its one ``tpspp_ocr_prep`` launch."""

    def __init__(self, transforms, rotate_degrees=None, force_rotate=False):
        if not isinstance(transforms, (list, tuple)) or len(transforms) == 0:
            raise ValueError(f"tps_pp_b200.MultiRotateAugOCR: transforms must be a non-empty list, got {transforms!r}")
        ts = []
        for i, t in enumerate(transforms):
            try:
                ts.append(_build(t))
            except (TypeError, ValueError) as e:
                raise ValueError(f"tps_pp_b200.MultiRotateAugOCR: transforms[{i}]: {e}") from e
        if len(ts) != len(_ORDER) - 1 or not all(isinstance(t, kinds) for t, kinds in zip(ts, _ORDER[1:])):
            raise ValueError(f"tps_pp_b200.MultiRotateAugOCR: transforms must be ResizeOCR, ToTensorOCR, NormalizeOCR, Collect; got "
                             f"{[type(t).__name__ for t in ts]}")
        if rotate_degrees is None:
            degrees = [0]
        else:
            degrees = list(rotate_degrees) if isinstance(rotate_degrees, list) else [rotate_degrees]
            for d in degrees:
                if isinstance(d, bool) or not isinstance(d, int) or not 0 <= d < 360 or d % 90 != 0:
                    raise ValueError(f"tps_pp_b200.MultiRotateAugOCR: rotate_degrees must be ints in [0, 360) that are multiples of "
                                     f"90, got {rotate_degrees!r}")
            if 0 not in degrees:
                degrees.append(0)
        self.transforms = ts
        self.rotate_degrees = degrees
        self.force_rotate = bool(force_rotate)
        # the reference iterates set(rotate_degrees); for these values (0, 90, 180, 270) CPython's set yields them ascending
        self._candidates = sorted(set(degrees))

    def degrees(self, h: int, w: int) -> List[int]:
        """The rotations, in degrees, that an h x w image is read in, in the reference's order."""
        return list(self._candidates) if self.force_rotate or h > w else [0]


def _is_rotate(t) -> bool:
    return isinstance(t, MultiRotateAugOCR) or (isinstance(t, dict) and t.get("type") == "MultiRotateAugOCR")


def _build_rotate(t) -> MultiRotateAugOCR:
    if isinstance(t, MultiRotateAugOCR):
        return t
    kw = {k: v for k, v in t.items() if k != "type"}
    unknown = sorted(set(kw) - {"transforms", "rotate_degrees", "force_rotate"})
    if unknown or "transforms" not in kw:
        raise ValueError(f"tps_pp_b200.MultiRotateAugOCR takes transforms, rotate_degrees and force_rotate; got {sorted(kw)}")
    return MultiRotateAugOCR(**kw)


class TestPipeline:
    """``test_pipeline`` config list -> a callable ``imgs -> (img [N, 3, height, max_width] fp32 on ``device``, img_metas)``.

    ``imgs`` is a non-empty list of uint8 [H, W, 3] arrays and/or image paths.  The images are packed, with their
    descriptors, into one pinned host buffer, copied to the device in one ``non_blocking`` copy, and turned into the batch
    tensor by one ``tpspp_ocr_prep`` launch on the current stream.  The pinned buffer is reused by the next call once the
    copy that reads it has completed.

    With :class:`MultiRotateAugOCR` (``self.rotate``) the batch holds every image's rotations, consecutively and in the
    reference's order, ``[N', 3, height, max_width]``, and ``img_metas`` is a list of N lists: one meta per rotation, as
    mmocr's aug test takes them.  Each image is still packed and uploaded once."""

    __test__ = False        # not a pytest test class despite its name

    def __init__(self, cfg_list: Sequence, device="cuda"):
        cfg_list = list(cfg_list)
        self.rotate: Optional[MultiRotateAugOCR] = None
        if any(_is_rotate(t) for t in cfg_list):
            if len(cfg_list) != 2 or _is_rotate(cfg_list[0]) or not _is_rotate(cfg_list[1]):
                raise ValueError("tps_pp_b200.TestPipeline: MultiRotateAugOCR must be the second and last transform, after "
                                 "LoadImageFromFile / LoadImageFromNdarray, and wrap ResizeOCR, ToTensorOCR, NormalizeOCR, Collect")
            self.rotate = _build_rotate(cfg_list[1])
            ts = [_build(cfg_list[0])] + self.rotate.transforms
        else:
            ts = [_build(t) for t in cfg_list]
        if len(ts) != len(_ORDER) or not all(isinstance(t, kinds) for t, kinds in zip(ts, _ORDER)):
            names = [type(t).__name__ for t in ts]
            raise ValueError(f"tps_pp_b200.TestPipeline: the pipeline must be LoadImageFromFile / LoadImageFromNdarray, ResizeOCR, "
                             f"ToTensorOCR, NormalizeOCR, Collect; got {names}")
        self.load, self.resize, _, self.normalize, self.collect = ts
        self.device = torch.device(device)
        self.out_h, self.out_w = self.resize.height, self.resize.max_width
        self._staging: Optional[torch.Tensor] = None
        self._copied: Optional[torch.cuda.Event] = None

    def _staging_buffer(self, nbytes: int) -> torch.Tensor:
        if self._copied is not None:
            self._copied.synchronize()            # the previous upload has read the buffer
        if self._staging is None or self._staging.numel() < nbytes:
            self._staging = torch.empty(max(nbytes, 1 << 20, 2 * (self._staging.numel() if self._staging is not None else 0)),
                                        dtype=torch.uint8, pin_memory=True)
        return self._staging

    def __call__(self, imgs: List):
        if isinstance(imgs, (np.ndarray, str, os.PathLike)) or len(imgs) == 0:
            raise ValueError("tps_pp_b200.TestPipeline takes a non-empty list of images")
        for i, x in enumerate(imgs):
            check_image(x, i)
        return self.prepare([self.load.load(x, i) for i, x in enumerate(imgs)])

    def _meta(self, img, fname, rw, ratio):
        meta = dict(filename=fname, ori_filename=fname, ori_shape=tuple(img.shape), img_shape=(self.out_h, rw, 3),
                    resize_shape=(self.out_h, rw, 3), pad_shape=(self.out_h, self.out_w, 3), valid_ratio=ratio,
                    img_norm_cfg=dict(mean=list(self.normalize.mean), std=list(self.normalize.std)))
        return {k: meta[k] for k in self.collect.meta_keys}

    def prepare(self, loaded: List):
        """The batch and metas of images already loaded: a list of ``(uint8 [H, W, 3] array, filename or None)``."""
        fields = 4 if self.rotate is None else 5
        rows, offsets, metas = [], [], []
        off = 0
        for img, fname in loaded:
            h, w = img.shape[:2]
            # every rotation of an image takes the width rule of the stored, unrotated image: this is the reference's
            # behaviour, since its ResizeOCR reads results['img_shape'], which MultiRotateAugOCR leaves unrotated when it
            # replaces results['img'].  The rotated pixels are then resized to (resize_w, height).
            rw, ratio = self.resize.resize_width(h, w)
            if self.rotate is None:
                rows.append((off, h, w, rw))
                metas.append(self._meta(img, fname, rw, ratio))
            else:
                degrees = self.rotate.degrees(h, w)
                rows += [(off, h, w, rw, d // 90) for d in degrees]
                metas.append([self._meta(img, fname, rw, ratio) for _ in degrees])
            offsets.append(off)
            off += h * w * 3
        n = len(rows)
        desc = np.array(rows, dtype=np.int64).reshape(n, fields)
        head = 8 * fields * n                      # [n, fields] int64 descriptors, then the pixels
        TF.check_ocr_desc(desc, off, self.out_w)
        staging = self._staging_buffer(head + off)
        host = staging.numpy()
        host[:head] = desc.view(np.uint8).reshape(-1)
        for (img, _), o in zip(loaded, offsets):
            h, w = img.shape[:2]
            host[head + o:head + o + h * w * 3].reshape(h, w, 3)[...] = img
        with torch.cuda.device(self.device):
            dev = staging[:head + off].to(self.device, non_blocking=True)
            self._copied = torch.cuda.Event()
            self._copied.record()
            out = TF.ocr_prep(dev[head:], desc, self.out_h, self.out_w, self.normalize.mean, self.normalize.std,
                              self.resize.img_pad_value, desc_dev=dev[:head].view(torch.int64).view(n, fields))
        return out, metas
