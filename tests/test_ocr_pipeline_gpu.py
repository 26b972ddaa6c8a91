"""GPU: TestPipeline (one tpspp_ocr_prep launch) against the per-image restatement of the mmocr test pipeline, bit for bit, with
its metas; the library's rejection of invalid configs; model_inference from uint8 arrays and image files to strings on the
native recogniser chain; init_recognizer's checkpoint loading."""
import os
import sys

import cv2
import numpy as np
import pytest
import torch

import tps_pp_b200 as T
from tps_pp_b200 import _native as N
from tps_pp_b200 import functional as TF

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the restatement beside these tests
from ocr_pipeline_restatement import pipeline_batch  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
META_KEYS = ["ori_shape", "img_shape", "resize_shape", "pad_shape", "valid_ratio"]


def crops(n, seed):
    """Seeded uint8 crops of mixed sizes: up- and down-scaled to a 32-high target, aspect ratios 0.3-8, a few extreme."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        h = int(rng.integers(8, 121))
        w = max(1, int(h * rng.uniform(0.3, 8.0)))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        img[:, :, 1] = np.linspace(0, 255, w, dtype=np.uint8)[None, :]          # one smooth channel beside two noisy ones
        out.append(img)
    out[:3] = [rng.integers(0, 256, s, dtype=np.uint8) for s in ((1, 1, 3), (1, 50, 3), (120, 3, 3))][:min(3, n)]
    return out


def config(height=32, min_width=32, max_width=128, keep_aspect_ratio=True, img_pad_value=0, width_downsample_ratio=1.0 / 16,
           mean=(0.5, 0.5, 0.5), std=(0.5, 0.5, 0.5)):
    resize = dict(height=height, min_width=min_width, max_width=max_width, keep_aspect_ratio=keep_aspect_ratio,
                  img_pad_value=img_pad_value, width_downsample_ratio=width_downsample_ratio)
    cfg = [dict(type="LoadImageFromNdarray"), dict(type="ResizeOCR", **resize), dict(type="ToTensorOCR"),
           dict(type="NormalizeOCR", mean=list(mean), std=list(std)), dict(type="Collect", keys=["img"], meta_keys=META_KEYS)]
    return cfg, dict(resize, mean=mean, std=std)


def _check(pipe, imgs, ref_kw):
    out, metas = pipe(imgs)
    ref, ref_metas = pipeline_batch(imgs, **ref_kw)
    assert out.shape == ref.shape and out.dtype == torch.float32 and out.device.type == "cuda"
    bad = (out.cpu() != ref).nonzero()
    assert len(bad) == 0, f"{len(bad)} values differ, first at {bad[0].tolist()}: {out.cpu()[tuple(bad[0])]} vs {ref[tuple(bad[0])]}"
    assert torch.equal(out.cpu(), ref)
    assert metas == ref_metas
    return out


CONFIGS = {
    "default": dict(),
    "stretch": dict(keep_aspect_ratio=False, mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)),
    "pad127_h48_w160": dict(height=48, min_width=16, max_width=160, img_pad_value=127, width_downsample_ratio=0.25,
                            mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)),
    "odd_widths_pad255": dict(max_width=100, min_width=8, width_downsample_ratio=1.0, img_pad_value=255, mean=(0.1, 0.9, 0.3),
                              std=(2.0, 0.07, 1.0)),
}


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_pipeline_matches_the_restatement(native_lib, name):
    cfg, ref_kw = config(**CONFIGS[name])
    pipe = T.TestPipeline(cfg, DEV)
    imgs = crops(96, seed=len(name))
    out = _check(pipe, imgs, ref_kw)
    if name == "pad127_h48_w160":                  # a padded column really holds (127 / 255 - mean) / std
        i = next(k for k, im in enumerate(imgs) if pipe.resize.resize_width(*im.shape[:2])[0] < 160)
        pad = (torch.tensor(127.0) / 255 - torch.tensor(0.485)) / torch.tensor(0.229)
        assert float(out[i, 0, 0, -1]) == float(pad)
    # a non-contiguous view and the pinned staging buffer reused by a second, smaller call
    imgs[5] = imgs[5][:, ::-1]
    imgs[6] = np.asfortranarray(imgs[6])
    _check(pipe, imgs[:17], ref_kw)


def test_pipeline_batch_1024_and_batch_1(native_lib):
    cfg, ref_kw = config(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
    pipe = T.TestPipeline(cfg, DEV)
    imgs = crops(1024, seed=5)
    _check(pipe, imgs, ref_kw)
    _check(pipe, imgs[700:701], ref_kw)
    _check(pipe, crops(1, seed=6), ref_kw)


def test_invalid_config_returns_the_library_error(native_lib):
    packed = torch.zeros(4 * 5 * 3, dtype=torch.uint8, device=DEV)
    desc = np.array([[0, 4, 5, 16]], dtype=np.int64)
    with pytest.raises(RuntimeError, match="std"):
        TF.ocr_prep(packed, desc, 32, 128, [0.5] * 3, [0.5, 0.0, 0.5])
    out = torch.empty((1, 3, 32, 128), device=DEV)
    d = torch.from_numpy(desc).to(DEV)
    for bad in (dict(out_w=0), dict(out_h=0), dict(n=0), dict(pad_value=256), dict(flags=1)):
        fields = dict(n=1, out_h=32, out_w=128, pad_value=0, flags=0)
        fields.update(bad)
        cfg = N.OcrPrepCfg(fields["n"], fields["out_h"], fields["out_w"], (N.c_float * 3)(0.5, 0.5, 0.5),
                           (N.c_float * 3)(0.5, 0.5, 0.5), fields["pad_value"], fields["flags"], packed.numel())
        rc = N.lib().tpspp_ocr_prep(N.ctypes.byref(cfg), N.c_void_p(packed.data_ptr()), N.c_void_p(d.data_ptr()),
                                    N.c_void_p(out.data_ptr()), N.c_void_p(torch.cuda.current_stream().cuda_stream))
        with pytest.raises(RuntimeError, match=list(bad)[0].split("_")[0]):
            N.check(rc, "tpspp_ocr_prep")


def _recognizer_config(batch_pipeline):
    return dict(
        model=dict(type="NRTR",
                   backbone=dict(type="ResNetABI_v2_large", arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]),
                   tpsnet=dict(type="TPS_PP"),
                   encoder=dict(type="NRTREncoder"),
                   decoder=dict(type="NRTRDecoder"),
                   label_convertor=dict(type="AttnConvertor", dict_type="DICT90", with_unknown=True, max_seq_len=40)),
        test_pipeline=batch_pipeline)


def test_model_inference_matches_simple_test_on_the_restatement(native_lib, tmp_path):
    cfg, ref_kw = config(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
    cfg[0] = dict(type="LoadImageFromFile")
    cfg[4]["meta_keys"] = ["filename", "ori_shape", "img_shape", "valid_ratio"]
    torch.manual_seed(0)                            # the weights of tests/test_nrtr_encoder_gpu.py::_recognizer
    model = T.init_recognizer(_recognizer_config(cfg), device=DEV)
    with torch.no_grad():
        model.decoder.classifier.weight.mul_(8.0)
    assert not model.training and next(model.parameters()).device.type == "cuda"
    imgs = crops(300, seed=21)
    results = T.model_inference(model, imgs, batch_size=256)
    assert model.backbone._last_stage_native and model.encoder.last_forward_native and model.decoder.last_test_native
    want = []
    with torch.no_grad():
        for s in (0, 256):
            ref, ref_metas = pipeline_batch(imgs[s:s + 256], **ref_kw)
            want += model.simple_test(ref.to(DEV), ref_metas)
    assert len(results) == 300
    assert [r["text"] for r in results] == [r["text"] for r in want]
    assert [r["score"] for r in results] == [r["score"] for r in want]
    one = T.model_inference(model, imgs[7])
    with torch.no_grad():
        ref, ref_metas = pipeline_batch(imgs[7:8], **ref_kw)
        want_one = model.simple_test(ref.to(DEV), ref_metas)[0]
    assert isinstance(one, dict) and one == want_one
    paths = []
    for i, img in enumerate(imgs[:40]):
        p = tmp_path / f"crop_{i}.png"
        assert cv2.imwrite(str(p), img)
        paths.append(str(p) if i % 2 else p)
    from_files = T.model_inference(model, paths, batch_size=16)
    from_arrays = T.model_inference(model, imgs[:40], batch_size=16)           # the same chunks of 16, 16 and 8
    assert from_files == from_arrays
    print(f"model_inference: 300 crops, texts {[r['text'] for r in results[:3]]}")


def test_init_recognizer_loads_a_checkpoint_strictly(native_lib, tmp_path):
    cfg, _ = config()
    conf = _recognizer_config(cfg)
    torch.manual_seed(3)
    src = T.build_recognizer(conf["model"])
    path = tmp_path / "nrtr.pth"
    torch.save({"state_dict": src.state_dict()}, path)
    model = T.init_recognizer(conf, str(path), device=DEV)
    for k, v in src.state_dict().items():
        assert torch.equal(model.state_dict()[k].cpu(), v), k
    bad = dict(src.state_dict())
    bad.pop(next(iter(bad)))
    with pytest.raises(RuntimeError, match="Missing"):
        T.init_recognizer(conf, bad, device=DEV)
