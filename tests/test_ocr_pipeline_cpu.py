"""CPU: OpenCV's INTER_LINEAR arithmetic as the CUDA kernel states it, against cv2.resize bit for bit; ResizeOCR's width rule;
the host-side descriptor checks of functional.ocr_prep; the registry and TestPipeline's config and input checks; the C layout
of tpspp_ocr_prep_cfg."""
import ctypes
import os
import shutil
import subprocess
import sys

import cv2
import numpy as np
import pytest
import torch

import tps_pp_b200 as T
from tps_pp_b200 import _native
from tps_pp_b200 import functional as TF
from tps_pp_b200.pipeline import ResizeOCR

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the restatement beside these tests
from ocr_pipeline_restatement import resize_fixed_point, resize_width  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pipeline_cfg(**resize):
    r = dict(type="ResizeOCR", height=32, min_width=32, max_width=128, keep_aspect_ratio=True)
    r.update(resize)
    return [dict(type="LoadImageFromFile"), r, dict(type="ToTensorOCR"),
            dict(type="NormalizeOCR", mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225]),
            dict(type="Collect", keys=["img"], meta_keys=["filename", "ori_shape", "img_shape", "valid_ratio"])]


def test_fixed_point_resize_is_cv2_bit_for_bit():
    rng = np.random.default_rng(1234)
    cases = []
    for _ in range(320):
        h, w = int(rng.integers(6, 151)), int(rng.integers(6, 501))
        cases.append(((h, w, 3) if rng.random() < 0.5 else (h, w), (int(rng.integers(8, 161)), 32)))
    for h, w in ((16, 64), (32, 128), (7, 9), (33, 65), (150, 500)):
        for c in ((h, w, 3), (h, w)):
            cases += [(c, (2 * w, 2 * h)), (c, (w, h)), (c, (max(1, w // 2), max(1, h // 2)))]
    cases += [((40, 37, 3), (131, 32)), ((6, 6, 3), (159, 32)), ((150, 6), (8, 32))]     # odd target widths, extreme ratios
    for shape, (dw, dh) in cases:
        img = rng.integers(0, 256, shape, dtype=np.uint8)
        want = cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR)
        got = resize_fixed_point(img, dw, dh)
        assert got.dtype == np.uint8 and np.array_equal(got, want), (shape, dw, dh)
    assert len(cases) >= 300


# (h, w, kwargs, resize_w, valid_ratio); height 32, max_width 128
WIDTHS = [
    (32, 100, {}, 96, 0.75),                                 # 100 -> round(6.25) * 16
    (32, 40, {}, 32, 0.25),                                  # 40 / 16 = 2.5 -> 2: half to even
    (32, 56, {}, 64, 0.5),                                   # 56 / 16 = 3.5 -> 4: half to even
    (32, 88, {}, 96, 0.75),                                  # 5.5 -> 6
    (48, 100, {}, 64, 0.5),                                  # ceil(66.67) = 67 -> 64
    (32, 10, {}, 16, 0.125),                                 # 0.625 -> 1
    (32, 10, dict(min_width=32), 32, 0.25),                  # min_width
    (32, 400, {}, 128, 1.0),                                 # clipped to max_width, valid_ratio 1
    (32, 136, {}, 128, 1.0),                                 # 136 % 16 = 8: 8.5 -> 8 -> 128
    (32, 152, {}, 128, 1.0),                                 # 9.5 -> 10 -> 160 -> clipped
    (32, 50, dict(width_downsample_ratio=0.25), 48, 0.375),  # d = 4: 12.5 -> 12
    (32, 54, dict(width_downsample_ratio=0.25), 56, 0.4375),  # 13.5 -> 14
    (16, 30, dict(width_downsample_ratio=0.25), 60, 0.46875),
    (37, 211, dict(min_width=32, width_downsample_ratio=0.25), 128, 1.0),
    (32, 100, dict(keep_aspect_ratio=False), 128, 1.0),
    (200, 20, dict(keep_aspect_ratio=False), 128, 1.0),
]


@pytest.mark.parametrize("h,w,kw,rw,ratio", WIDTHS)
def test_resize_ocr_width_rule(h, w, kw, rw, ratio):
    args = dict(height=32, max_width=128)
    args.update(kw)
    assert ResizeOCR(**args).resize_width(h, w) == (rw, ratio)
    assert resize_width(h, w, **args) == (rw, ratio)


def test_resize_ocr_width_rule_matches_the_restatement_on_random_sizes():
    rng = np.random.default_rng(7)
    for _ in range(500):
        h, w = int(rng.integers(1, 200)), int(rng.integers(1, 1000))
        kw = dict(height=int(rng.choice([32, 48, 64])), max_width=int(rng.choice([100, 128, 160])),
                  min_width=[None, 32][int(rng.integers(2))], keep_aspect_ratio=bool(rng.random() < 0.8),
                  width_downsample_ratio=float(rng.choice([1.0, 0.5, 0.25, 1.0 / 16])))
        assert ResizeOCR(**kw).resize_width(h, w) == resize_width(h, w, **kw)


def _packed(sizes):
    off, rows = 0, []
    for h, w in sizes:
        rows.append((off, h, w, 64))
        off += h * w * 3
    return torch.zeros(off, dtype=torch.uint8), np.array(rows, dtype=np.int64)


@pytest.mark.parametrize("col,val,what", [(1, 0, "h >= 1"), (2, -3, "w >= 1"), (3, 0, "resize_w"), (3, 129, "resize_w"),
                                          (0, -1, "offset")])
def test_ocr_prep_rejects_bad_descriptors_on_the_host(col, val, what):
    packed, desc = _packed([(10, 20), (5, 7)])
    TF.check_ocr_desc(desc, packed.numel(), 128)            # the valid rows pass
    desc[1, col] = val
    with pytest.raises(ValueError, match=what):
        TF.ocr_prep(packed, desc, 32, 128, [0.5] * 3, [0.5] * 3)           # a CPU `packed`: no device is touched first
    with pytest.raises(ValueError, match=what):
        TF.ocr_prep(packed, torch.from_numpy(desc), 32, 128, [0.5] * 3, [0.5] * 3)


def test_ocr_prep_rejects_an_image_past_the_end_of_the_buffer():
    packed, desc = _packed([(10, 20), (5, 7)])
    desc[1, 0] += 1
    with pytest.raises(ValueError, match="past the end"):
        TF.ocr_prep(packed, desc, 32, 128, [0.5] * 3, [0.5] * 3)
    with pytest.raises(ValueError, match="past the end"):
        TF.ocr_prep(packed[:-1], _packed([(10, 20), (5, 7)])[1], 32, 128, [0.5] * 3, [0.5] * 3)
    with pytest.raises(ValueError, match="int64"):
        TF.ocr_prep(packed, desc.astype(np.int32), 32, 128, [0.5] * 3, [0.5] * 3)
    with pytest.raises(ValueError, match="int64"):
        TF.ocr_prep(packed, desc[:0], 32, 128, [0.5] * 3, [0.5] * 3)
    with pytest.raises(RuntimeError, match="CUDA"):                          # valid descriptors: then the device check
        TF.ocr_prep(packed, _packed([(10, 20), (5, 7)])[1], 32, 128, [0.5] * 3, [0.5] * 3)


def test_registry_builds_the_pipeline_from_config_dicts():
    assert set(T.PIPELINES.module_dict) == {"LoadImageFromFile", "LoadImageFromNdarray", "ResizeOCR", "ToTensorOCR", "NormalizeOCR",
                                            "Collect"}
    p = T.TestPipeline(_pipeline_cfg(img_pad_value=7), "cuda")
    assert (p.out_h, p.out_w) == (32, 128)
    assert p.resize.img_pad_value == 7 and p.resize.min_width == 32
    assert p.normalize.mean == [0.485, 0.456, 0.406] and p.collect.meta_keys == ["filename", "ori_shape", "img_shape", "valid_ratio"]
    cfg = _pipeline_cfg()
    cfg[0] = dict(type="LoadImageFromNdarray")
    assert isinstance(T.TestPipeline(cfg).load, T.PIPELINES.get("LoadImageFromNdarray"))
    r = T.PIPELINES.build(dict(type="ResizeOCR", height=32, max_width=160, keep_aspect_ratio=False, backend="cv2"))
    assert r.resize_width(10, 1000) == (160, 1.0)


@pytest.mark.parametrize("change,match", [
    (lambda c: c.insert(1, dict(type="MultiRotateAugOCR", rotate_degrees=[0, 90, 270], transforms=[])), "MultiRotateAugOCR"),
    (lambda c: c[1].update(backend="pillow"), "backend"),
    (lambda c: c[1].update(max_width=None), "max_width"),
    (lambda c: c.__setitem__(slice(2, 4), c[3:1:-1]), "must be"),             # NormalizeOCR before ToTensorOCR
    (lambda c: c.pop(2), "must be"),
    (lambda c: c[3].update(std=[0.5, 0.0, 0.5]), "std"),
    (lambda c: c[3].update(mean=[0.5]), "3 means"),
    (lambda c: c[4].update(meta_keys=["scale_factor"]), "scale_factor"),
    (lambda c: c[4].update(keys=["img", "gt_label"]), "keys"),
    (lambda c: c[0].update(to_float32=True), "to_float32"),
    (lambda c: c[0].update(color_type="grayscale"), "color_type"),
    (lambda c: c[1].update(img_pad_value=300), "img_pad_value"),
])
def test_rejected_configs_raise(change, match):
    cfg = _pipeline_cfg()
    change(cfg)
    with pytest.raises(ValueError, match=match):
        T.TestPipeline(cfg)


@pytest.mark.parametrize("bad", [np.zeros((8, 8, 3), np.float32), np.zeros((8, 8), np.uint8), np.zeros((8, 8, 4), np.uint8),
                                 np.zeros((0, 8, 3), np.uint8), np.zeros((8, 0, 3), np.uint8), 3, None])
def test_rejected_inputs_raise_before_any_launch(bad):
    p = T.TestPipeline(_pipeline_cfg())
    good = np.zeros((8, 8, 3), np.uint8)
    with pytest.raises(ValueError):
        p([good, bad])

    class Model:                                            # model_inference checks every input before the first chunk
        test_pipeline = p

        def simple_test(self, *a, **k):
            raise AssertionError("no image may reach the model")
    with pytest.raises(ValueError):
        T.model_inference(Model(), [good] * 3 + [bad], batch_size=2)


def test_empty_inputs_raise():
    p = T.TestPipeline(_pipeline_cfg())
    with pytest.raises(ValueError):
        p([])
    with pytest.raises(ValueError):
        T.model_inference(type("M", (), dict(test_pipeline=p))(), [])
    with pytest.raises(ValueError):
        T.model_inference(type("M", (), dict(test_pipeline=p))(), [np.zeros((8, 8, 3), np.uint8)], batch_size=0)
    with pytest.raises(ValueError):
        T.init_recognizer(dict(model=dict(type="NRTR")))     # no test_pipeline


def test_unreadable_file_raises(tmp_path):
    p = T.TestPipeline(_pipeline_cfg())
    with pytest.raises(ValueError, match="could not read"):
        p([str(tmp_path / "missing.png")])


def test_ocr_prep_cfg_has_the_header_layout(tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    mirror = _native.OcrPrepCfg
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "tpspp.h"', "int main(void) {",
             '  printf("%zu", sizeof(tpspp_ocr_prep_cfg));']
    lines += [f'  printf(" %zu", offsetof(tpspp_ocr_prep_cfg, {f}));' for f, _ in mirror._fields_]
    lines += ['  printf("\\n");', "  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    vals = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == ctypes.sizeof(mirror)
    assert vals[1:] == [getattr(mirror, f).offset for f, _ in mirror._fields_]
    assert [f for f, _ in mirror._fields_] == ["n", "out_h", "out_w", "mean", "std", "pad_value", "flags", "packed_bytes"]
