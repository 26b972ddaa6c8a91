#!/usr/bin/env python
"""The text-recognition test pipeline from host uint8 crops (tps_pp_b200.TestPipeline / tpspp_ocr_prep), and the NRTR recogniser
from host crops to strings (tps_pp_b200.model_inference), at batches of 256 and 1024:

* ``tpspp_ocr_prep`` device time per batch: CUDA events around CUDA-graph replays of 20 launches (so the host's launch rate does
  not bound it), with the algorithmic bytes (packed uint8 input + fp32 output) over that time;
* the host-to-device copy of one packed batch (pinned buffer, ``non_blocking``), CUDA events;
* ``TestPipeline.__call__`` whole (pack on the host + copy + kernel), host clock ending in a device synchronise;
* the reference's way on the host: per image ``cv2.resize`` + torch ``to_tensor`` / ``normalize``, ``torch.stack``, then the
  fp32 batch copied to the device -- once on one core and once split over a process pool of all host cores;
* ``model_inference`` from host arrays to strings in img/s (median of windows), beside ``simple_test`` on device-resident images
  of the same batch (the figure of scripts/recognizer_bench.py).

Crops are seeded: height uniform in 16-96, aspect ratio uniform in 1-8, 3 channels.  The card's name and power limit are read
in the same call.  python scripts/ocr_pipeline_bench.py [--batches 256,1024] [--out profiles/r04_ocr_pipeline.json]"""
import argparse
import json
import multiprocessing as mp
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
from recognizer_bench import build, card  # noqa: E402

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
PIPELINE = [dict(type="LoadImageFromNdarray"),
            dict(type="ResizeOCR", height=32, min_width=32, max_width=128, keep_aspect_ratio=True),
            dict(type="ToTensorOCR"),
            dict(type="NormalizeOCR", mean=list(MEAN), std=list(STD)),
            dict(type="Collect", keys=["img"], meta_keys=["filename", "ori_shape", "img_shape", "valid_ratio"])]


def crops(n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        h = int(rng.integers(16, 97))
        w = max(1, int(round(h * rng.uniform(1.0, 8.0))))
        out.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
    return out


def host_one(img, resize):
    """The reference's per-image work: ResizeOCR (cv2 + pad), ToTensorOCR, NormalizeOCR."""
    rw, ratio = resize.resize_width(*img.shape[:2])
    r = cv2.resize(img, (rw, resize.height), interpolation=cv2.INTER_LINEAR)
    if rw < resize.max_width:
        r = np.pad(r, ((0, 0), (0, resize.max_width - rw), (0, 0)), constant_values=resize.img_pad_value)
    t = torch.from_numpy(np.ascontiguousarray(r.transpose(2, 0, 1))).float().div(255)
    return t.sub_(torch.tensor(MEAN).view(3, 1, 1)).div_(torch.tensor(STD).view(3, 1, 1)), ratio


_POOL_RESIZE = None


def _pool_init(resize):
    global _POOL_RESIZE
    _POOL_RESIZE = resize
    torch.set_num_threads(1)
    cv2.setNumThreads(1)


def _pool_chunk(imgs):
    return torch.stack([host_one(i, _POOL_RESIZE)[0] for i in imgs]).numpy()


def median_ms(fn, windows, reps=1, sync=True):
    ts = []
    for _ in range(windows):
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        if sync:
            torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3 / reps)
    return statistics.median(ts), ts


def bench_batch(rec, pipe, pool, cores, batch, dev, windows):
    imgs = crops(batch, seed=batch)
    res = {"batch": batch}
    # ---- packed batch on the device, as TestPipeline uploads it
    desc = np.array([(0, *i.shape[:2], pipe.resize.resize_width(*i.shape[:2])[0]) for i in imgs], dtype=np.int64)
    desc[1:, 0] = np.cumsum([i.size for i in imgs])[:-1]
    packed_host = torch.from_numpy(np.concatenate([i.reshape(-1) for i in imgs])).pin_memory()
    packed = packed_host.to(dev)
    desc_dev = torch.from_numpy(desc).to(dev)
    out = torch.empty((batch, 3, 32, 128), device=dev)
    call = lambda: TF.ocr_prep(packed, desc, 32, 128, MEAN, STD, 0, out=out, desc_dev=desc_dev)   # noqa: E731
    call()
    ref = torch.stack([host_one(i, pipe.resize)[0] for i in imgs])
    res["ocr_prep_equals_host_reference"] = bool(torch.equal(out.cpu(), ref))
    reps = 20
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
    k_ms = statistics.median(ts)
    nbytes = packed.numel() + out.numel() * 4
    res["ocr_prep"] = {"device_ms": k_ms, "windows_ms": ts, "packed_bytes": packed.numel(), "out_bytes": out.numel() * 4,
                       "algorithmic_gb_per_s": nbytes / (k_ms * 1e-3) / 1e9,
                       "note": "input + output fit the 126 MB L2 after the first pass: the rate is not an HBM rate"}
    # ---- host-to-device copy of one packed batch (pinned), and of the fp32 batch the reference's way would copy
    for name, src in (("h2d_packed_uint8", packed_host), ("h2d_fp32_batch", ref.pin_memory())):
        dst = torch.empty(src.shape, dtype=src.dtype, device=dev)
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        tc = []
        for _ in range(windows):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dst.copy_(src, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            tc.append(e0.elapsed_time(e1))
        c_ms = statistics.median(tc)
        res[name] = {"ms": c_ms, "bytes": src.numel() * src.element_size(), "gb_per_s": src.numel() * src.element_size() / (c_ms * 1e-3) / 1e9,
                     "windows_ms": tc}
    # ---- TestPipeline whole: pack on the host, one copy, one launch
    pipe(imgs)
    p_ms, p_ts = median_ms(lambda: pipe(imgs), windows, reps=3)
    res["test_pipeline_call"] = {"ms": p_ms, "img_per_s": batch / (p_ms * 1e-3), "windows_ms": p_ts}
    # ---- the reference's way on the host: one core, then all cores
    def host_serial():
        torch.stack([host_one(i, pipe.resize)[0] for i in imgs]).pin_memory().to(dev, non_blocking=True)
    nt = torch.get_num_threads()
    torch.set_num_threads(1)
    cv2.setNumThreads(1)
    try:
        s_ms, s_ts = median_ms(host_serial, windows)
    finally:
        torch.set_num_threads(nt)
        cv2.setNumThreads(-1)
    chunks = [imgs[i::cores] for i in range(cores)]

    def host_pool():
        parts = pool.map(_pool_chunk, chunks)
        torch.from_numpy(np.concatenate(parts)).pin_memory().to(dev, non_blocking=True)
    host_pool()
    m_ms, m_ts = median_ms(host_pool, windows)
    res["host_reference_pipeline"] = {
        "one_core_ms": s_ms, "one_core_img_per_s": batch / (s_ms * 1e-3), "one_core_windows_ms": s_ts,
        "all_cores_ms": m_ms, "all_cores_img_per_s": batch / (m_ms * 1e-3), "all_cores_windows_ms": m_ts, "cores": cores,
        "how": "per image cv2.resize + np.pad + torch to_tensor/normalize, torch.stack, pinned copy to the device; all cores = a "
               "fork process pool of `cores` workers (1 torch / cv2 thread each), images dealt round-robin, arrays returned by pickle"}
    # ---- model_inference from host arrays to strings, and simple_test on device-resident images
    with torch.no_grad():
        T.model_inference(rec, imgs, batch_size=batch)
        mi_ms, mi_ts = median_ms(lambda: T.model_inference(rec, imgs, batch_size=batch), windows, reps=2)
        img_dev = torch.randn((batch, 3, 32, 128), device=dev, generator=torch.Generator(device=dev).manual_seed(batch))
        metas = [dict(valid_ratio=1.0) for _ in range(batch)]
        rec.simple_test(img_dev, metas)
        st_ms, st_ts = median_ms(lambda: rec.simple_test(img_dev, metas), windows, reps=2)
    res["model_inference"] = {"ms": mi_ms, "img_per_s": batch / (mi_ms * 1e-3), "windows_ms": mi_ts,
                              "native_stage_encoder_decoder": [bool(rec.backbone._last_stage_native),
                                                               bool(rec.encoder.last_forward_native),
                                                               bool(rec.decoder.last_test_native)]}
    res["simple_test_device_resident"] = {"ms": st_ms, "img_per_s": batch / (st_ms * 1e-3), "windows_ms": st_ts}
    res["example_texts"] = [r["text"] for r in T.model_inference(rec, imgs[:2])]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,1024")
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():      # (initialises no device)
        raise SystemExit("ocr_pipeline_bench.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    pipe = T.TestPipeline(PIPELINE, dev)
    cores = len(os.sched_getaffinity(0))
    # the host workers are forked before this process touches the device
    with mp.get_context("fork").Pool(cores, initializer=_pool_init, initargs=(pipe.resize,)) as pool:
        info = card()
        rec = build(dev)
        rec.test_pipeline = pipe
        results = [bench_batch(rec, pipe, pool, cores, int(b), dev, args.windows) for b in args.batches.split(",")]
    result = {"metric": "ocr_test_pipeline", "card": info, "torch": torch.__version__, "opencv": cv2.__version__,
              "host_cores": cores,
              "what": "seeded uint8 crops (height 16-96, aspect 1-8, 3 channels) -> ResizeOCR(32, min 32, max 128, keep aspect) + "
                      "ToTensorOCR + NormalizeOCR; recogniser as scripts/recognizer_bench.py (seeded NRTR, DICT90)",
              "results": results}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
