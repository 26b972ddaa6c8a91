"""GPU: the rotation test-time augmentation on the device -- tpspp_ocr_prep with [n, 5] descriptors against cv2.resize of
np.rot90 bit for bit, the flag-less call against the k = 0 rows, TestPipeline with MultiRotateAugOCR against the per-image
restatement (images and nested metas, from arrays and files), and model_inference / NRTR.forward on the native recogniser
chain against simple_test on the restatement's candidate batch followed by the restated merge."""
import os
import sys

import cv2
import numpy as np
import pytest
import torch

import tps_pp_b200 as T
from tps_pp_b200 import functional as TF

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the restatements beside these tests
from ocr_tta_restatement import candidate_one, candidates, merge, tta_batch  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
META_KEYS = ["filename", "ori_filename", "ori_shape", "img_shape", "resize_shape", "pad_shape", "valid_ratio", "img_norm_cfg"]

# the four configurations of tests/test_ocr_pipeline_gpu.py
CONFIGS = {
    "default": dict(),
    "stretch": dict(keep_aspect_ratio=False, mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)),
    "pad127_h48_w160": dict(height=48, min_width=16, max_width=160, img_pad_value=127, width_downsample_ratio=0.25,
                            mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)),
    "odd_widths_pad255": dict(max_width=100, min_width=8, width_downsample_ratio=1.0, img_pad_value=255, mean=(0.1, 0.9, 0.3),
                              std=(2.0, 0.07, 1.0)),
}


def ref_kw(height=32, min_width=32, max_width=128, keep_aspect_ratio=True, img_pad_value=0, width_downsample_ratio=1.0 / 16,
           mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5)):
    return dict(height=height, min_width=min_width, max_width=max_width, keep_aspect_ratio=keep_aspect_ratio,
                img_pad_value=img_pad_value, width_downsample_ratio=width_downsample_ratio, mean=tuple(mean), std=tuple(std))


def rotating_config(kw, rotate_degrees=(0, 90, 270), force_rotate=False, loader="LoadImageFromNdarray"):
    resize = {k: v for k, v in kw.items() if k not in ("mean", "std")}
    return [dict(type=loader),
            dict(type="MultiRotateAugOCR", rotate_degrees=list(rotate_degrees), force_rotate=force_rotate,
                 transforms=[dict(type="ResizeOCR", **resize), dict(type="ToTensorOCR"),
                             dict(type="NormalizeOCR", mean=list(kw["mean"]), std=list(kw["std"])),
                             dict(type="Collect", keys=["img"], meta_keys=META_KEYS)])]


def crops(n, seed):
    """Seeded uint8 crops, a quarter of them tall: heights 8-120, aspect ratios 1-8, every fourth transposed; a few extremes
    (1 x 1, 1 x N, N x 1) up front; one smooth channel beside two noisy ones."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        h = int(rng.integers(8, 121))
        w = max(1, int(h * rng.uniform(1.0, 8.0)))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        img[:, :, 1] = np.linspace(0, 255, w, dtype=np.uint8)[None, :]
        out.append(np.ascontiguousarray(img.transpose(1, 0, 2)) if i % 4 == 3 else img)
    extremes = [(1, 1, 3), (1, 50, 3), (120, 3, 3), (200, 1, 3), (1, 300, 3), (7, 6, 3)]
    out[:len(extremes)] = [rng.integers(0, 256, s, dtype=np.uint8) for s in extremes][:n]
    return out


def _equal(got, want):
    bad = (got.cpu() != want).nonzero()
    assert len(bad) == 0, f"{len(bad)} values differ, first at {bad[0].tolist()}: {got.cpu()[tuple(bad[0])]} vs {want[tuple(bad[0])]}"


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_rotated_descriptors_match_cv2_of_rot90(native_lib, name):
    kw = ref_kw(**CONFIGS[name])
    resize = T.PIPELINES.build(dict(type="ResizeOCR", **{k: v for k, v in kw.items() if k not in ("mean", "std")}))
    imgs = crops(48, seed=100 + len(name))
    offsets = np.cumsum([0] + [i.size for i in imgs])
    packed = torch.from_numpy(np.concatenate([i.reshape(-1) for i in imgs])).to(DEV)
    # every image in all four rotations, rows shuffled so that rows sharing an offset are not neighbours
    rows = [(int(offsets[i]), *img.shape[:2], resize.resize_width(*img.shape[:2])[0], k) for i, img in enumerate(imgs) for k in range(4)]
    order = np.random.default_rng(3).permutation(len(rows))
    desc = np.array([rows[j] for j in order], dtype=np.int64)
    out = TF.ocr_prep(packed, desc, kw["height"], kw["max_width"], kw["mean"], kw["std"], kw["img_pad_value"])
    want = torch.stack([candidate_one(imgs[j // 4], 90 * (j % 4), **kw)[0] for j in order])
    assert out.shape == want.shape
    _equal(out, want)
    # the k = 0 rows are bit-identical to the flag-less call on the same images
    zero = np.flatnonzero(desc[:, 4] == 0)
    plain = TF.ocr_prep(packed, np.ascontiguousarray(desc[zero, :4]), kw["height"], kw["max_width"], kw["mean"], kw["std"],
                        kw["img_pad_value"])
    assert torch.equal(out[torch.from_numpy(zero).to(DEV)], plain)


def _check_pipeline(pipe, items, imgs, degrees, force, kw, filenames):
    out, metas = pipe(items)
    want, want_metas = tta_batch(imgs, degrees, force, **kw)
    assert out.shape == want.shape and out.dtype == torch.float32 and out.device.type == "cuda"
    _equal(out, want)
    for group, fname in zip(want_metas, filenames):
        for m in group:
            m.update(filename=fname, ori_filename=fname)
    assert metas == want_metas
    assert [len(g) for g in metas] == [len(candidates(*i.shape[:2], degrees, force)) for i in imgs]


@pytest.mark.parametrize("name,degrees,force", [("default", [0, 90, 270], False), ("pad127_h48_w160", [0, 90, 180, 270], False),
                                                ("odd_widths_pad255", [270, 90], True), ("stretch", [0, 180], False)])
def test_pipeline_with_rotation_matches_the_restatement(native_lib, name, degrees, force):
    kw = ref_kw(**CONFIGS[name])
    pipe = T.TestPipeline(rotating_config(kw, degrees, force), DEV)
    imgs = crops(96, seed=7 + len(name))
    _check_pipeline(pipe, imgs, imgs, degrees, force, kw, [None] * len(imgs))
    _check_pipeline(pipe, imgs[40:41], imgs[40:41], degrees, force, kw, [None])        # the staging buffer reused
    tall = next(i for i, im in enumerate(imgs) if im.shape[0] > im.shape[1])
    _check_pipeline(pipe, imgs[tall:tall + 1], imgs[tall:tall + 1], degrees, force, kw, [None])


def test_pipeline_with_rotation_from_files(native_lib, tmp_path):
    kw = ref_kw(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
    pipe = T.TestPipeline(rotating_config(kw, loader="LoadImageFromFile"), DEV)
    imgs = crops(24, seed=11)
    paths = []
    for i, img in enumerate(imgs):
        p = tmp_path / f"crop_{i}.png"
        assert cv2.imwrite(str(p), img)
        paths.append(str(p) if i % 2 else p)
    _check_pipeline(pipe, paths, imgs, [0, 90, 270], False, kw, [os.fspath(p) for p in paths])


def _recognizer(pipeline):
    torch.manual_seed(0)                            # the weights of tests/test_ocr_pipeline_gpu.py's model_inference test
    model = T.init_recognizer(dict(
        model=dict(type="NRTR",
                   backbone=dict(type="ResNetABI_v2_large", arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]),
                   tpsnet=dict(type="TPS_PP"),
                   encoder=dict(type="NRTREncoder"),
                   decoder=dict(type="NRTRDecoder"),
                   label_convertor=dict(type="AttnConvertor", dict_type="DICT90", with_unknown=True, max_seq_len=40)),
        test_pipeline=pipeline), device=DEV)
    with torch.no_grad():
        model.decoder.classifier.weight.mul_(8.0)
    return model


def test_model_inference_with_rotation_matches_simple_test_on_the_restatement(native_lib):
    kw = ref_kw(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
    degrees = [0, 90, 270]
    model = _recognizer(rotating_config(kw, degrees))
    imgs = crops(160, seed=21)
    batch_size = 96
    results = T.model_inference(model, imgs, batch_size=batch_size)
    assert model.backbone._last_stage_native and model.encoder.last_forward_native and model.decoder.last_test_native
    # the same chunks of whole images: an image joins the chunk while its candidates fit in batch_size rows
    chunks, chunk, rows = [], [], 0
    for img in imgs:
        n = len(candidates(*img.shape[:2], degrees))
        if rows + n > batch_size:
            chunks.append(chunk)
            chunk, rows = [], 0
        chunk.append(img)
        rows += n
    chunks.append(chunk)
    assert len(chunks) >= 2
    want = []
    with torch.no_grad():
        for chunk in chunks:
            ref, ref_metas = tta_batch(chunk, degrees, **kw)
            flat = model.simple_test(ref.to(DEV), [m for g in ref_metas for m in g])
            s = 0
            for g in ref_metas:
                want += merge(flat[s:s + len(g)])
                s += len(g)
    assert len(results) == len(imgs)
    assert results == want
    assert all(isinstance(r["score"], float) for r in results)
    tall = [i for i, im in enumerate(imgs) if im.shape[0] > im.shape[1]]
    assert len(tall) >= 30
    one = T.model_inference(model, imgs[tall[0]])
    with torch.no_grad():
        ref, ref_metas = tta_batch(imgs[tall[0]:tall[0] + 1], degrees, **kw)
        want_one = merge(model.simple_test(ref.to(DEV), ref_metas[0]))[0]
    assert isinstance(one, dict) and one == want_one
    print(f"model_inference with rotation: {len(imgs)} crops ({len(tall)} tall), texts {[r['text'] for r in results[:3]]}")


def test_forward_of_a_list_is_the_merged_aug_test(native_lib):
    kw = ref_kw(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
    model = _recognizer(rotating_config(kw, [0, 90, 180, 270]))
    imgs = crops(12, seed=5)
    tall = next(im for im in imgs[6:] if im.shape[0] > im.shape[1])
    out, metas = model.test_pipeline([tall])
    assert out.shape[0] == 4 and len(metas) == 1 and len(metas[0]) == 4
    img_list = [out[i:i + 1] for i in range(4)]
    meta_list = [[m] for m in metas[0]]
    with torch.no_grad():
        got = model(img_list, meta_list, return_loss=False)
        flat = model.simple_test(torch.cat(img_list), metas[0])
    assert got == model.merge_aug_results(flat) == merge(flat)
    assert len(got) == 1 and isinstance(got[0]["score"], float)
    with pytest.raises(ValueError, match="aug test"):
        model([out[:2]], [metas[0][:2]], return_loss=False)
