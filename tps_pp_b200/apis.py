"""Image-to-text entry points in the shape of mmocr's ``init_detector`` / ``model_inference`` (reference
mmocr/apis/inference.py:19-195): a recogniser from a config dict, and uint8 images or image files in, strings out.

    model = init_recognizer(dict(model=dict(type='NRTR', ...), test_pipeline=[...]), 'nrtr.pth')
    model_inference(model, ['word_1.png', crop_array])   # -> [dict(text=..., score=[...]), ...]

The test pipeline runs batched on the GPU (:class:`tps_pp_b200.pipeline.TestPipeline`), then ``simple_test``.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from .pipeline import TestPipeline, check_image
from .registry import build_recognizer


def init_recognizer(config, checkpoint=None, device="cuda"):
    """``config``: ``dict(model=<recogniser config>, test_pipeline=[<transform configs>])``.  ``checkpoint``: a path to (or
    the object of) a ``state_dict`` or ``{'state_dict': ...}``, loaded with ``strict=True``.  Returns the recogniser in eval
    mode on ``device`` with ``test_pipeline`` (and ``cfg``) attached."""
    if not isinstance(config, dict) or "model" not in config or "test_pipeline" not in config:
        raise ValueError("tps_pp_b200.init_recognizer: config must be a dict with 'model' and 'test_pipeline'")
    pipeline = TestPipeline(config["test_pipeline"], device)
    model = build_recognizer(config["model"])
    if checkpoint is not None:
        state = torch.load(checkpoint, map_location="cpu") if isinstance(checkpoint, (str, os.PathLike)) else checkpoint
        if isinstance(state, dict) and "state_dict" in state:
            state = state["state_dict"]
        model.load_state_dict(state, strict=True)
    model.cfg = config
    model.test_pipeline = pipeline
    return model.to(device).eval()


def model_inference(model, imgs, batch_size: int = 256):
    """One image (uint8 [H, W, 3] array or path) -> ``dict(text, score)``; a list of them -> a list of such dicts.  Works in
    chunks of at most ``batch_size`` images under ``torch.no_grad()``; every input is checked before the first chunk runs.

    With a ``MultiRotateAugOCR`` test pipeline, ``batch_size`` bounds the rotations a chunk holds: a chunk takes whole images
    while their rotations fit, so ``batch_size`` must be at least the number of distinct rotate degrees.  Each image's
    readings are merged by ``model.merge_aug_results`` into ``dict(text, score)`` with a float ``score``."""
    if int(batch_size) < 1:
        raise ValueError(f"tps_pp_b200.model_inference: batch_size must be >= 1, got {batch_size}")
    single = isinstance(imgs, (np.ndarray, str, os.PathLike))
    items = [imgs] if single else list(imgs)
    if not items:
        raise ValueError("tps_pp_b200.model_inference: no images")
    for i, x in enumerate(items):
        check_image(x, i)
    pipeline = getattr(model, "test_pipeline", None)
    if pipeline is None:
        raise ValueError("tps_pp_b200.model_inference: the model has no test_pipeline (build it with init_recognizer)")
    rotate = getattr(pipeline, "rotate", None)
    if rotate is not None and int(batch_size) < len(set(rotate.rotate_degrees)):
        raise ValueError(f"tps_pp_b200.model_inference: batch_size {batch_size} is smaller than the {len(set(rotate.rotate_degrees))} "
                         "rotations MultiRotateAugOCR reads a tall image in")
    results = []
    with torch.no_grad():
        if rotate is None:
            for s in range(0, len(items), int(batch_size)):
                img, metas = pipeline(items[s:s + int(batch_size)])
                results += model.simple_test(img, metas)
        else:
            chunk, rows = [], 0
            for i, x in enumerate(items):
                img, fname = pipeline.load.load(x, i)
                n = len(rotate.degrees(*img.shape[:2]))
                if rows + n > int(batch_size):
                    results += _aug_chunk(model, pipeline, chunk)
                    chunk, rows = [], 0
                chunk.append((img, fname))
                rows += n
            results += _aug_chunk(model, pipeline, chunk)
    return results[0] if single else results


def _aug_chunk(model, pipeline, loaded):
    """Whole images through the rotating pipeline and one ``simple_test``, then one merged result per image."""
    img, metas = pipeline.prepare(loaded)
    flat = model.simple_test(img, [m for group in metas for m in group])
    out, s = [], 0
    for group in metas:
        out += model.merge_aug_results(flat[s:s + len(group)])
        s += len(group)
    return out
