"""mmocr 0.4's rotation test-time augmentation, restated per image from its specification, independently of tps_pp_b200:
``MultiRotateAugOCR`` (datasets/pipelines/test_time_aug.py) around the test pipeline of ocr_pipeline_restatement.py, and
``EncodeDecodeRecognizer.merge_aug_results`` (recognizer/encode_decode_recognizer.py).

* ``rotate_degrees``: an int or a list of ints in [0, 360), multiples of 90; 0 appended when missing; ``None`` is ``[0]``.
* An image is rotated only when ``ori_height > ori_width`` (or ``force_rotate``); its candidates come in the iteration order of
  ``set(rotate_degrees)``.  Degree d is ``np.rot90(img, d // 90)``.
* The wrapper replaces only ``img``, so ResizeOCR reads the unrotated ``img_shape``: every candidate of an image takes the
  ``resize_w`` / ``valid_ratio`` of the stored image, and the rotated pixels are resized to ``(resize_w, height)``.
* Merge: start at ``('', -1)``; a candidate's score is ``sum(score) / max(1, len(text))``; only a strictly greater score
  replaces the best; the result is ``[dict(text, score=<float>)]``."""
from __future__ import annotations

import cv2
import numpy as np
import torch

from ocr_pipeline_restatement import resize_width


def rotate_degrees(degrees):
    """``MultiRotateAugOCR.__init__``'s list of degrees."""
    if degrees is None:
        return [0]
    out = degrees if isinstance(degrees, list) else [degrees]
    out = list(out)
    assert all(isinstance(d, int) and 0 <= d < 360 and d % 90 == 0 for d in out)
    if 0 not in out:
        out.append(0)
    return out


def candidates(h, w, degrees, force_rotate=False):
    """``MultiRotateAugOCR.__call__``: the degrees, in order, that an h x w image is read in."""
    if not force_rotate and h <= w:
        return [0]
    return list(set(rotate_degrees(degrees)))


def candidate_one(img, degree, height, max_width, min_width=None, keep_aspect_ratio=True, img_pad_value=0,
                  width_downsample_ratio=1.0 / 16, mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5)):
    """One rotation of one uint8 HWC image -> ([3, height, max_width] fp32, metas)."""
    h, w = img.shape[:2]
    rw, ratio = resize_width(h, w, height, min_width, max_width, keep_aspect_ratio, width_downsample_ratio)   # unrotated shape
    rot = np.ascontiguousarray(np.rot90(img, degree // 90))
    r = cv2.resize(rot, (rw, height), interpolation=cv2.INTER_LINEAR)
    resize_shape = r.shape
    if rw < max_width:
        r = np.pad(r, ((0, 0), (0, max_width - rw), (0, 0)), constant_values=img_pad_value)
    t = torch.from_numpy(np.ascontiguousarray(r.transpose(2, 0, 1))).float().div(255)
    t = t.sub(torch.tensor(mean, dtype=torch.float32).view(3, 1, 1)).div(torch.tensor(std, dtype=torch.float32).view(3, 1, 1))
    metas = dict(ori_shape=img.shape, img_shape=resize_shape, resize_shape=resize_shape, pad_shape=r.shape, valid_ratio=ratio,
                 img_norm_cfg=dict(mean=list(mean), std=list(std)))
    return t, metas


def tta_batch(imgs, degrees, force_rotate=False, **kw):
    """A list of images -> ([N', 3, height, max_width] with each image's candidates consecutive, [[metas per candidate]])."""
    ts, metas = [], []
    for img in imgs:
        group = []
        for d in candidates(img.shape[0], img.shape[1], degrees, force_rotate):
            t, m = candidate_one(img, d, **kw)
            ts.append(t)
            group.append(m)
        metas.append(group)
    return torch.stack(ts), metas


def merge(results):
    """``merge_aug_results`` over one image's candidate results (``dict(text, score=[...])`` each)."""
    out_text, out_score = "", -1
    for r in results:
        score = sum(r["score"]) / max(1, len(r["text"]))
        if score > out_score:
            out_text, out_score = r["text"], score
    return [dict(text=out_text, score=out_score)]
