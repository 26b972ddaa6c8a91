"""CPU: the rotation test-time augmentation -- MultiRotateAugOCR's candidate lists and NRTR.merge_aug_results against
hand-worked cases and the restatement, the configs TestPipeline takes and rejects, model_inference's chunking of whole images,
the [n, 5] descriptor checks, and TPSPP_OCR_FLAG_ROTATED in the header."""
import itertools
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

import tps_pp_b200 as T
from tps_pp_b200 import _native
from tps_pp_b200 import functional as TF
from tps_pp_b200.pipeline import MultiRotateAugOCR

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the restatement beside these tests
from ocr_tta_restatement import candidates, merge, rotate_degrees  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INNER = [dict(type="ResizeOCR", height=32, min_width=32, max_width=128, keep_aspect_ratio=True), dict(type="ToTensorOCR"),
         dict(type="NormalizeOCR", mean=[0.5, 0.5, 0.5], std=[0.5, 0.5, 0.5]),
         dict(type="Collect", keys=["img"], meta_keys=["filename", "ori_shape", "img_shape", "valid_ratio"])]

# mmocr 0.4 configs/_base_/recog_pipelines/nrtr_pipeline.py, test_pipeline, verbatim
IMG_NORM_CFG = dict(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])
NRTR_TEST_PIPELINE = [
    dict(type='LoadImageFromFile'),
    dict(
        type='MultiRotateAugOCR',
        rotate_degrees=[0, 90, 270],
        transforms=[
            dict(
                type='ResizeOCR',
                height=32,
                min_width=32,
                max_width=160,
                keep_aspect_ratio=True,
                width_downsample_ratio=0.25),
            dict(type='ToTensorOCR'),
            dict(type='NormalizeOCR', **IMG_NORM_CFG),
            dict(
                type='Collect',
                keys=['img'],
                meta_keys=[
                    'filename', 'ori_shape', 'img_shape', 'valid_ratio',
                    'resize_shape', 'img_norm_cfg', 'ori_filename'
                ]),
        ])
]


def _rotating(rotate_degrees=(0, 90, 270), force_rotate=False, inner=None):
    return [dict(type="LoadImageFromNdarray"),
            dict(type="MultiRotateAugOCR", rotate_degrees=list(rotate_degrees), force_rotate=force_rotate,
                 transforms=[dict(t) for t in (inner or INNER)])]


# (h, w, rotate_degrees, force_rotate, candidates)
CANDIDATES = [
    (10, 40, [0, 90, 270], False, [0]),                    # wide
    (20, 20, [0, 90, 270], False, [0]),                    # square: not taller than wide
    (21, 20, [0, 90, 270], False, [0, 90, 270]),           # tall
    (10, 40, [0, 90, 270], True, [0, 90, 270]),            # force_rotate
    (40, 10, [90, 270], False, [0, 90, 270]),              # 0 appended
    (40, 10, [270, 90, 90, 0, 270], False, [0, 90, 270]),  # duplicates
    (40, 10, [180, 90, 0, 270], False, [0, 90, 180, 270]),
    (40, 10, 180, False, [0, 180]),                        # an int
    (40, 10, None, True, [0]),                             # None is [0]
]


@pytest.mark.parametrize("h,w,degrees,force,want", CANDIDATES)
def test_candidates_match_hand_worked_cases(h, w, degrees, force, want):
    assert candidates(h, w, degrees, force) == want
    aug = MultiRotateAugOCR(transforms=INNER, rotate_degrees=degrees, force_rotate=force)
    assert aug.degrees(h, w) == want
    assert aug.rotate_degrees == rotate_degrees(degrees)


def test_candidate_order_is_the_reference_set_order_for_every_degree_list():
    for r in range(1, 5):
        for combo in itertools.permutations([0, 90, 180, 270], r):
            aug = MultiRotateAugOCR(transforms=INNER, rotate_degrees=list(combo))
            assert aug.degrees(9, 3) == candidates(9, 3, list(combo)), combo
            assert aug.degrees(3, 9) == [0]


def test_rotate_degrees_append_zero_like_the_reference():
    assert MultiRotateAugOCR(transforms=INNER, rotate_degrees=[90, 270]).rotate_degrees == [90, 270, 0]
    assert MultiRotateAugOCR(transforms=INNER).rotate_degrees == [0]
    assert MultiRotateAugOCR(transforms=INNER, rotate_degrees=90).rotate_degrees == [90, 0]


def _r(text, score):
    return dict(text=text, score=list(score))


MERGES = [
    ([_r("ab", [0.5, 0.5]), _r("cd", [0.25, 0.75])], "ab", 0.5),              # tie: the first wins
    ([_r("ab", [0.5, 0.5]), _r("xyz", [0.6, 0.6, 0.6])], "xyz", 0.6),         # strictly greater replaces
    ([_r("", []), _r("a", [0.0])], "", 0.0),                                  # empty text scores 0 / 1; 0 is not > 0
    ([_r("<UKN>", [0.9]), _r("ab", [0.3, 0.3])], "ab", 0.3),                  # <UKN> counts 5 characters: 0.18
    ([_r("<UKN>a", [0.9, 0.9]), _r("q", [0.29])], "<UKN>a", 0.3),
    ([_r("only", [0.1, 0.2, 0.3, 0.4])], "only", 0.25),
]


@pytest.mark.parametrize("results,text,score", MERGES)
def test_merge_aug_results_on_hand_written_results(results, text, score):
    want = [dict(text=text, score=pytest.approx(score))]
    assert merge(results) == want
    got = T.NRTR.merge_aug_results(results)
    assert got == merge(results) and isinstance(got[0]["score"], float)
    assert T.NRTR.merge_aug_results([[r] for r in results]) == got          # mmocr's per-augmentation result lists


def test_stock_nrtr_test_pipeline_builds():
    p = T.TestPipeline(NRTR_TEST_PIPELINE, "cuda")
    assert p.rotate is not None and p.rotate.rotate_degrees == [0, 90, 270] and not p.rotate.force_rotate
    assert (p.out_h, p.out_w) == (32, 160) and p.resize.width_downsample_ratio == 0.25
    assert p.normalize.mean == IMG_NORM_CFG["mean"]
    assert set(p.collect.meta_keys) == {"filename", "ori_shape", "img_shape", "valid_ratio", "resize_shape", "img_norm_cfg",
                                        "ori_filename"}
    assert p.rotate.degrees(40, 10) == [0, 90, 270]
    # an instance is taken as well, and the registry is unchanged
    aug = MultiRotateAugOCR(transforms=INNER, rotate_degrees=[0, 180], force_rotate=True)
    assert T.TestPipeline([dict(type="LoadImageFromNdarray"), aug]).rotate is aug
    assert "MultiRotateAugOCR" not in T.PIPELINES.module_dict


def _wrapper(cfg):
    return cfg[1]


@pytest.mark.parametrize("change", [
    lambda c: _wrapper(c).update(transforms=[]),
    lambda c: _wrapper(c).pop("transforms"),
    lambda c: _wrapper(c)["transforms"].pop(3),                                             # no Collect
    lambda c: _wrapper(c)["transforms"].reverse(),
    lambda c: _wrapper(c)["transforms"].insert(0, dict(type="LoadImageFromFile")),
    lambda c: _wrapper(c)["transforms"].append(dict(type="RandomRotate")),
    lambda c: _wrapper(c)["transforms"][0].update(max_width=None),
    lambda c: _wrapper(c).update(rotate_degrees=[0, 45]),
    lambda c: _wrapper(c).update(rotate_degrees=[0, 360]),
    lambda c: _wrapper(c).update(rotate_degrees=[0, -90]),
    lambda c: _wrapper(c).update(rotate_degrees=[0, 90.0]),
    lambda c: _wrapper(c).update(rotate_degrees=(0, 90)),
    lambda c: _wrapper(c).update(rotate_degrees=[True]),
    lambda c: _wrapper(c).update(flip=True),
    lambda c: c.append(dict(type="Collect", keys=["img"])),                                # the wrapper is not last
    lambda c: c.insert(0, c.pop(1)),                                                        # the wrapper before the loader
    lambda c: c.insert(1, dict(type="ResizeOCR", height=32, max_width=128)),                # the wrapper at position 2
    lambda c: c.__setitem__(0, dict(type="MultiRotateAugOCR", transforms=list(INNER))),     # two wrappers
])
def test_malformed_wrappers_raise(change):
    cfg = _rotating()
    change(cfg)
    with pytest.raises(ValueError, match="MultiRotateAugOCR"):
        T.TestPipeline(cfg)


def test_rotated_descriptors_are_checked_on_the_host():
    packed = torch.zeros(10 * 20 * 3 + 5 * 7 * 3, dtype=torch.uint8)
    desc = np.array([[0, 10, 20, 64, 0], [0, 10, 20, 64, 1], [600, 5, 7, 32, 3]], dtype=np.int64)
    TF.check_ocr_desc(desc, packed.numel(), 128)                # shared offsets and k in [0, 3] pass
    for k in (-1, 4, 5):
        bad = desc.copy()
        bad[2, 4] = k
        with pytest.raises(ValueError, match="k"):
            TF.ocr_prep(packed, bad, 32, 128, [0.5] * 3, [0.5] * 3)             # a CPU `packed`: no device is touched first
    with pytest.raises(ValueError, match=r"\[n, 5\]"):
        TF.ocr_prep(packed, np.zeros((3, 6), np.int64), 32, 128, [0.5] * 3, [0.5] * 3)
    bad = desc.copy()
    bad[2, 0] += 1
    with pytest.raises(ValueError, match="past the end"):
        TF.ocr_prep(packed, bad, 32, 128, [0.5] * 3, [0.5] * 3)
    with pytest.raises(RuntimeError, match="CUDA"):                          # valid descriptors: then the device check
        TF.ocr_prep(packed, desc, 32, 128, [0.5] * 3, [0.5] * 3)


class _FakePipeline(T.TestPipeline):
    """The rotating pipeline without the device step: row i of the batch holds its image's index (pixel [0, 0, 0])."""

    def prepare(self, loaded):
        metas = [[dict(image=int(img[0, 0, 0]), degree=d, ori_shape=img.shape)
                  for d in self.rotate.degrees(*img.shape[:2])] for img, _ in loaded]
        rows = [m["image"] for g in metas for m in g]
        return torch.tensor(rows, dtype=torch.float32).view(-1, 1), metas


def _fake_result(image, degree):
    """Seeded per (image, degree), from a few score values so that ties happen, some texts empty or with <UKN>."""
    rng = np.random.default_rng(1000 * image + degree)
    chars = [str(c) for c in rng.choice(list("ab") + ["<UKN>"], int(rng.integers(0, 4)))]
    return dict(text="".join(chars), score=[float(v) for v in rng.choice([0.25, 0.5, 1.0], len(chars))])


class _FakeModel:
    merge_aug_results = staticmethod(T.NRTR.merge_aug_results)

    def __init__(self, pipeline, batch_size):
        self.test_pipeline, self.batch_size, self.calls = pipeline, batch_size, []

    def simple_test(self, img, metas):
        assert img.shape[0] == len(metas) <= self.batch_size
        assert [int(v) for v in img[:, 0]] == [m["image"] for m in metas]
        self.calls.append([(m["image"], m["degree"]) for m in metas])
        return [_fake_result(m["image"], m["degree"]) for m in metas]


def _shapes(n, seed):
    rng = np.random.default_rng(seed)
    return [(int(rng.integers(1, 60)), int(rng.integers(1, 60))) for _ in range(n)]


@pytest.mark.parametrize("degrees,force,batch_size", [([0, 90, 270], False, 3), ([0, 90, 270], False, 4), ([0, 90, 270], False, 7),
                                                      ([90, 180, 0, 270], False, 5), ([0, 90, 270], True, 8),
                                                      ([0, 90, 270], False, 256), (None, False, 1)])
def test_model_inference_chunks_whole_images(degrees, force, batch_size):
    shapes = _shapes(60, seed=batch_size)
    imgs = []
    for i, (h, w) in enumerate(shapes):
        img = np.zeros((h, w, 3), np.uint8)
        img[0, 0, 0] = i
        imgs.append(img)
    cfg = _rotating(force_rotate=force)
    cfg[1]["rotate_degrees"] = degrees
    model = _FakeModel(_FakePipeline(cfg), batch_size)
    got = T.model_inference(model, imgs, batch_size=batch_size)
    # every image's candidates, in the reference's order, in one call; the images in order across calls
    want_rows = [(i, d) for i, (h, w) in enumerate(shapes) for d in candidates(h, w, degrees, force)]
    assert [r for call in model.calls for r in call] == want_rows
    for call in model.calls:
        for i in {img for img, _ in call}:
            assert [d for img, d in call if img == i] == candidates(*shapes[i], degrees, force)
    # a chunk closes only when the next image would not fit
    for call, nxt in zip(model.calls, model.calls[1:]):
        assert len(call) + len(candidates(*shapes[nxt[0][0]], degrees, force)) > batch_size
    want = [merge([_fake_result(i, d) for d in candidates(h, w, degrees, force)])[0] for i, (h, w) in enumerate(shapes)]
    assert got == want and all(isinstance(r["score"], float) for r in got)
    one = T.model_inference(model, imgs[5], batch_size=batch_size)
    assert one == want[5]


def test_model_inference_rejects_a_batch_smaller_than_the_rotations():
    class Model:
        test_pipeline = T.TestPipeline(_rotating([0, 90, 270]))

        def simple_test(self, *a, **k):
            raise AssertionError("no image may reach the model")
    wide = np.zeros((8, 16, 3), np.uint8)
    with pytest.raises(ValueError, match="batch_size"):
        T.model_inference(Model(), [wide] * 4, batch_size=2)
    with pytest.raises(ValueError):                       # and every input is still checked before the first chunk
        T.model_inference(Model(), [wide] * 4 + [np.zeros((8, 8), np.uint8)], batch_size=3)


def _nrtr():
    torch.manual_seed(0)
    return T.build_recognizer(dict(
        type="NRTR",
        backbone=dict(type="ResNetABI_v2_large", arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]),
        tpsnet=dict(type="TPS_PP"),
        encoder=dict(type="NRTREncoder"),
        decoder=dict(type="NRTRDecoder"),
        label_convertor=dict(type="AttnConvertor", dict_type="DICT90", with_unknown=True, max_seq_len=40))).eval()


def test_forward_rejects_malformed_aug_test_inputs():
    model = _nrtr()
    one = torch.zeros((1, 3, 32, 128))
    meta = [dict(valid_ratio=1.0)]
    for imgs, metas in (([one, torch.zeros((2, 3, 32, 128))], [meta, meta]),      # an entry whose batch is not 1
                        ([], []),
                        ([one, one], [meta]),                                       # one [meta] list per tensor
                        ([one], [dict(valid_ratio=1.0)]),
                        ([one], None)):
        with pytest.raises(ValueError, match="aug test"):
            model(imgs, metas, return_loss=False)


def test_ocr_flag_rotated_matches_the_header(tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "flag.c"
    src.write_text('#include <stdio.h>\n#include "tpspp.h"\nint main(void) { printf("%d\\n", (int)TPSPP_OCR_FLAG_ROTATED); return 0; }\n')
    exe = tmp_path / "flag"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    assert int(out) == _native.OCR_FLAG_ROTATED == 2
