"""The mmocr 0.4 text-recognition test pipeline (LoadImage -> ResizeOCR -> ToTensorOCR -> NormalizeOCR -> Collect), restated
per image from its specification, independently of tps_pp_b200: ``cv2.resize`` (what ``mmcv.imresize`` calls for the cv2
backend), ``np.pad`` (``mmcv.impad`` on the right / bottom with a constant), torch ``float().div(255)`` (``to_tensor``), then
``sub`` and ``div`` (``normalize``).  ``resize_fixed_point`` is OpenCV's INTER_LINEAR arithmetic on uint8 written out in numpy,
the form the CUDA kernel implements."""
from __future__ import annotations

import math

import cv2
import numpy as np
import torch


def resize_width(h, w, height, min_width=None, max_width=None, keep_aspect_ratio=True, width_downsample_ratio=1.0 / 16):
    """mmocr 0.4 ``ResizeOCR.__call__``: (resize_w, valid_ratio) for an h x w image and a fixed ``max_width``."""
    if not keep_aspect_ratio:
        return max_width, 1.0
    new_w = math.ceil(float(height) / h * w)
    d = int(1 / width_downsample_ratio)
    if new_w % d != 0:
        new_w = round(new_w / d) * d
    if min_width is not None:
        new_w = max(min_width, new_w)
    return min(max_width, new_w), min(1.0, 1.0 * new_w / max_width)


def pipeline_one(img, height, max_width, min_width=None, keep_aspect_ratio=True, img_pad_value=0, width_downsample_ratio=1.0 / 16,
                 mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5)):
    """One uint8 HWC image -> ([3, height, max_width] fp32, metas)."""
    h, w = img.shape[:2]
    rw, ratio = resize_width(h, w, height, min_width, max_width, keep_aspect_ratio, width_downsample_ratio)
    r = cv2.resize(img, (rw, height), interpolation=cv2.INTER_LINEAR)
    resize_shape = r.shape
    if rw < max_width:
        r = np.pad(r, ((0, 0), (0, max_width - rw), (0, 0)), constant_values=img_pad_value)
    t = torch.from_numpy(np.ascontiguousarray(r.transpose(2, 0, 1))).float().div(255)
    t = t.sub(torch.tensor(mean, dtype=torch.float32).view(3, 1, 1)).div(torch.tensor(std, dtype=torch.float32).view(3, 1, 1))
    metas = dict(ori_shape=img.shape, img_shape=resize_shape, resize_shape=resize_shape, pad_shape=r.shape, valid_ratio=ratio)
    return t, metas


def pipeline_batch(imgs, **kw):
    """A list of images -> ([N, 3, height, max_width], [metas])."""
    outs = [pipeline_one(i, **kw) for i in imgs]
    return torch.stack([t for t, _ in outs]), [m for _, m in outs]


def _axis(s, d):
    """Per destination index along one axis: source index i0 and the fractional part f (float32)."""
    scale = 1.0 / (float(d) / s)
    f = ((np.arange(d, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    i0 = np.floor(f).astype(np.int64)
    f = (f - i0.astype(np.float32)).astype(np.float32)
    return i0, f


def _coef(f):
    """rint((1 - f) * 2048), rint(f * 2048) in float32, round half to even."""
    a0 = np.rint((np.float32(1.0) - f) * np.float32(2048)).astype(np.int64)
    a1 = np.rint(f * np.float32(2048)).astype(np.int64)
    return a0, a1


def resize_fixed_point(img, dw, dh):
    """``cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR)`` for uint8 [H, W] or [H, W, C], in OpenCV's fixed-point
    arithmetic (11-bit coefficients, horizontal pass in int32, vertical pass with its >> 4 / >> 16 / rounding shifts)."""
    src = img.astype(np.int64)
    if src.ndim == 2:
        src = src[:, :, None]
    h, w = src.shape[:2]
    ix, fx = _axis(w, dw)
    low, high = ix < 0, ix >= w - 1
    fx = np.where(low | high, np.float32(0), fx).astype(np.float32)
    ix = np.where(low, 0, np.where(high, w - 1, ix))
    a0, a1 = _coef(fx)
    iy, fy = _axis(h, dh)
    b0, b1 = _coef(fy)
    r0, r1 = np.clip(iy, 0, h - 1), np.clip(iy + 1, 0, h - 1)
    hor = src[:, ix, :] * a0[None, :, None] + src[:, np.minimum(ix + 1, w - 1), :] * a1[None, :, None]
    v = (((hor[r0] >> 4) * b0[:, None, None]) >> 16) + (((hor[r1] >> 4) * b1[:, None, None]) >> 16)
    out = np.clip((v + 2) >> 2, 0, 255).astype(np.uint8)
    return out[:, :, 0] if img.ndim == 2 else out
