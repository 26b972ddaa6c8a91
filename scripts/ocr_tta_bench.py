#!/usr/bin/env python
"""Rotation test-time augmentation (mmocr's MultiRotateAugOCR, rotate_degrees [0, 90, 270]) from host uint8 crops, at 256 and
1024 images, a quarter of them tall:

* ``tpspp_ocr_prep`` device time per call, flag-less ([n, 4] descriptors, one row per image) and rotated ([n', 5], the rows
  TestPipeline makes: three per tall image over the same packed bytes), CUDA events around CUDA-graph replays of 20 launches;
  the odd quarter turns read stored columns, so the time per output row of the two is the figure to compare;
* ``model_inference`` with the rotating pipeline against the same crops through the plain pipeline, img/s (median of windows);
* the reference's way on a subset: per image, host ``np.rot90`` + ``cv2.resize`` + pad + ``to_tensor`` / ``normalize`` of each
  rotation, a batch-1 ``simple_test`` per rotation (``EncodeDecodeRecognizer.aug_test``), ``merge_aug_results``; img/s.

Crops are those of scripts/ocr_pipeline_bench.py (height 16-96, aspect 1-8), every fourth transposed.  The card's name and
power limit are read in the same call.  python scripts/ocr_tta_bench.py [--batches 256,1024] [--out profiles/r06_ocr_tta.json]"""
import argparse
import json
import os
import statistics
import sys
import time

import cv2
import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import tps_pp_b200 as T  # noqa: E402
from tps_pp_b200 import functional as TF  # noqa: E402
from ocr_pipeline_bench import MEAN, PIPELINE, STD, crops, median_ms  # noqa: E402
from recognizer_bench import build, card  # noqa: E402

DEGREES = [0, 90, 270]
ROTATING = [dict(type="LoadImageFromNdarray"),
            dict(type="MultiRotateAugOCR", rotate_degrees=DEGREES, transforms=[dict(t) for t in PIPELINE[1:]])]


def tta_crops(n, seed):
    return [np.ascontiguousarray(c.transpose(1, 0, 2)) if i % 4 == 3 else c for i, c in enumerate(crops(n, seed))]


def graph_ms(call, windows, reps=20):
    """Device ms per call: CUDA events around replays of a graph of ``reps`` calls."""
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        call()
    torch.cuda.current_stream().wait_stream(stream)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            call()
    g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / (5 * reps))
    return statistics.median(ts), ts


def host_candidate(img, degree, resize):
    """The reference's per-rotation host work: np.rot90, ResizeOCR with the unrotated image's width, to_tensor, normalize."""
    rw, ratio = resize.resize_width(*img.shape[:2])
    r = cv2.resize(np.ascontiguousarray(np.rot90(img, degree // 90)), (rw, resize.height), interpolation=cv2.INTER_LINEAR)
    if rw < resize.max_width:
        r = np.pad(r, ((0, 0), (0, resize.max_width - rw), (0, 0)), constant_values=resize.img_pad_value)
    t = torch.from_numpy(np.ascontiguousarray(r.transpose(2, 0, 1))).float().div(255)
    return t.sub_(torch.tensor(MEAN).view(3, 1, 1)).div_(torch.tensor(STD).view(3, 1, 1)), ratio


def reference_way(rec, pipe, imgs, dev):
    out = []
    for img in imgs:
        aug = []
        for d in pipe.rotate.degrees(*img.shape[:2]):
            t, ratio = host_candidate(img, d, pipe.resize)
            aug.append(rec.simple_test(t[None].to(dev), [dict(valid_ratio=ratio)]))
        out += rec.merge_aug_results(aug)
    return out


def bench_batch(rec, plain, rot, batch, dev, windows, subset):
    imgs = tta_crops(batch, seed=batch)
    res = {"batch": batch, "tall": sum(i.shape[0] > i.shape[1] for i in imgs)}
    offsets = np.cumsum([0] + [i.size for i in imgs])[:-1]
    packed = torch.from_numpy(np.concatenate([i.reshape(-1) for i in imgs])).to(dev)
    rows4, rows5 = [], []
    for o, img in zip(offsets.tolist(), imgs):
        h, w = img.shape[:2]
        rw = rot.resize.resize_width(h, w)[0]
        rows4.append((o, h, w, rw))
        rows5 += [(o, h, w, rw, d // 90) for d in rot.rotate.degrees(h, w)]
    res["rows_rotated"] = len(rows5)
    for name, rows in (("ocr_prep_plain", rows4), ("ocr_prep_rotated", rows5)):
        desc = np.array(rows, dtype=np.int64)
        desc_dev = torch.from_numpy(desc).to(dev)
        out = torch.empty((len(rows), 3, 32, 128), device=dev)
        call = lambda: TF.ocr_prep(packed, desc, 32, 128, MEAN, STD, 0, out=out, desc_dev=desc_dev)   # noqa: E731
        k_ms, ts = graph_ms(call, windows)
        res[name] = {"device_ms": k_ms, "rows": len(rows), "us_per_row": k_ms * 1e3 / len(rows), "windows_ms": ts}
    # the rotated call's rows against the pipeline's, and the k = 0 rows against the plain call
    with torch.no_grad():
        img_r, metas_r = rot(imgs)
        img_p, _ = plain(imgs)
        first = np.cumsum([0] + [len(g) for g in metas_r])[:-1]
        res["rotated_k0_rows_equal_plain"] = bool(torch.equal(img_r[torch.from_numpy(first).to(dev)], img_p))
        # model_inference, rotating pipeline against the plain one, same crops, alternating windows
        ts = {"rotating": [], "plain": []}
        for p in (rot, plain, rot, plain):
            rec.test_pipeline = p
            T.model_inference(rec, imgs, batch_size=batch)
        for _ in range(windows):
            for name, p in (("rotating", rot), ("plain", plain)):
                rec.test_pipeline = p
                t0 = time.perf_counter()
                T.model_inference(rec, imgs, batch_size=batch)
                torch.cuda.synchronize()
                ts[name].append((time.perf_counter() - t0) * 1e3)
        for name in ts:
            ms = statistics.median(ts[name])
            res[f"model_inference_{name}"] = {"ms": ms, "img_per_s": batch / (ms * 1e-3), "windows_ms": ts[name]}
        res["model_inference_rotating"]["rows_per_call"] = len(rows5)
        res["model_inference_rotating"]["native_stage_encoder_decoder"] = [
            bool(rec.backbone._last_stage_native), bool(rec.encoder.last_forward_native), bool(rec.decoder.last_test_native)]
        # the reference's way on a subset: batch-1 simple_test per rotation
        sub = imgs[:subset]
        rec.test_pipeline = rot
        reference_way(rec, rot, sub[:4], dev)
        r_ms, r_ts = median_ms(lambda: reference_way(rec, rot, sub, dev), max(3, windows // 2))
        res["reference_way"] = {"images": len(sub), "rows": sum(len(rot.rotate.degrees(*i.shape[:2])) for i in sub),
                                "ms": r_ms, "img_per_s": len(sub) / (r_ms * 1e-3), "windows_ms": r_ts,
                                "how": "per image: host np.rot90 + cv2.resize + pad + to_tensor/normalize per rotation, "
                                       "batch-1 simple_test per rotation, merge_aug_results"}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,1024")
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--subset", type=int, default=32, help="images the reference's way runs on")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():      # (initialises no device)
        raise SystemExit("ocr_tta_bench.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    info = card()
    rec = build(dev)
    plain, rot = T.TestPipeline(PIPELINE, dev), T.TestPipeline(ROTATING, dev)
    results = [bench_batch(rec, plain, rot, int(b), dev, args.windows, args.subset) for b in args.batches.split(",")]
    result = {"metric": "ocr_rotation_tta", "card": info, "torch": torch.__version__, "opencv": cv2.__version__,
              "what": "seeded uint8 crops (height 16-96, aspect 1-8, every fourth transposed) -> MultiRotateAugOCR([0, 90, 270]) "
                      "around ResizeOCR(32, min 32, max 128, keep aspect) + ToTensorOCR + NormalizeOCR; recogniser as "
                      "scripts/recognizer_bench.py (seeded NRTR, DICT90)",
              "results": results}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
