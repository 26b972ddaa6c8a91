#!/usr/bin/env python
"""NRTR recogniser from device-resident images [B, 3, 32, 128] to strings (tps_pp_b200.NRTR.simple_test; reference
recognizer/encode_decode_recognizer.py:184-225), with the NRTR encoder measured on its own:

* encoder, native (tcgen05 3xTF32 dense layers + tpspp_attn_encode) vs ``forward_library`` (the reference algorithm on torch /
  cuBLAS fp32 ops, TF32 off), same module and weights, timed alternately in the same process; median over windows, and the
  achieved TFLOP/s from the FLOPs the shapes need;
* ``tpspp_attn_encode`` alone (the encoder's q|k|v layout, all keys valid);
* ``simple_test`` end to end in img/s, and its parts: backbone stage, TPS_PP, layer3-5 (library ops), encoder, decode, convertor.

CUDA events around device work, warm-up before every timed window; the card's name and power limit go into the same JSON.
python scripts/recognizer_bench.py [--batches 256,1024] [--out profiles/r03_recognizer.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tps_pp_b200 as T  # noqa: E402
from tps_pp_b200 import functional as TF  # noqa: E402


def encoder_flops(batch, t=64, d=512, d_inner=256, layers=6, heads=8, head_dim=64):
    """(dense, attention) FLOPs of one encoder call: q|k|v, fc, w_1, w_2 per layer; q.K^T and P.V per head."""
    dense = 2 * batch * t * (3 * d * d + d * d + d * d_inner + d_inner * d) * layers
    attn = 2 * 2 * batch * heads * t * t * head_dim * layers
    return dense, attn


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in out.split(",")]
    except Exception as e:  # the measurement stands without it, but says so
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def window_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def build(dev):
    torch.manual_seed(0)
    rec = T.build_recognizer(dict(
        type="NRTR",
        backbone=dict(type="ResNetABI_v2_large", arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]),
        tpsnet=dict(type="TPS_PP"),
        encoder=dict(type="NRTREncoder"),
        decoder=dict(type="NRTRDecoder"),
        label_convertor=dict(type="AttnConvertor", dict_type="DICT90", with_unknown=True, max_seq_len=40)))
    with torch.no_grad():
        rec.decoder.classifier.weight.mul_(8.0)
    return rec.to(dev).eval()


def bench_batch(rec, batch, dev, windows):
    img = torch.randn((batch, 3, 32, 128), device=dev, generator=torch.Generator(device=dev).manual_seed(batch))
    metas = [dict(valid_ratio=1.0) for _ in range(batch)]
    enc = rec.encoder
    res = {"batch": batch}
    with torch.no_grad():
        feat = rec.extract_feat(img)
        assert tuple(feat.shape) == (batch, 512, 4, 16)
        # ---- encoder: native vs library, alternating windows
        nat = enc(feat, metas)
        assert enc.last_forward_native
        lib = enc.forward_library(feat, metas)
        res["encoder_max_abs_diff_native_vs_library"] = float((nat - lib).abs().max())
        iters = max(2, 2048 // batch)
        for _ in range(2):
            enc(feat, metas)
            enc.forward_library(feat, metas)
        torch.cuda.synchronize()
        tn, tl = [], []
        for _ in range(windows):
            tn.append(window_ms(lambda: enc(feat, metas), iters))
            tl.append(window_ms(lambda: enc.forward_library(feat, metas), iters))
        dense, attn = encoder_flops(batch)
        n_ms, l_ms = statistics.median(tn), statistics.median(tl)
        res["encoder"] = {"native_ms": n_ms, "library_ms": l_ms, "speedup": l_ms / n_ms, "native_windows_ms": tn,
                          "library_windows_ms": tl, "iters_per_window": iters, "gflop_dense": dense / 1e9, "gflop_attention": attn / 1e9,
                          "native_tflops": (dense + attn) / (n_ms * 1e-3) / 1e12, "library_tflops": (dense + attn) / (l_ms * 1e-3) / 1e12}
        # ---- tpspp_attn_encode alone: one layer's call
        d = 512
        qkv = torch.randn((batch * 64, 3 * d), device=dev)
        out = torch.empty((batch * 64, d), device=dev)
        call = lambda: TF.attn_encode(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], 8, 64, 8.0, out=out)   # noqa: E731
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        ta = [window_ms(call, 20) for _ in range(windows)]
        a_ms = statistics.median(ta)
        res["attn_encode"] = {"per_call_ms": a_ms, "windows_ms": ta, "gflop": attn / 6 / 1e9,
                              "tflops": attn / 6 / (a_ms * 1e-3) / 1e12}
        # ---- simple_test end to end, and split into its parts
        for _ in range(2):
            rec.simple_test(img, metas)
        torch.cuda.synchronize()
        te = []
        for _ in range(windows):
            t0 = time.perf_counter()
            n_it = 2
            for _ in range(n_it):
                rec.simple_test(img, metas)          # ends in the convertor's device-to-host copy: synchronous
            te.append((time.perf_counter() - t0) * 1e3 / n_it)
        e_ms = statistics.median(te)
        res["simple_test"] = {"ms": e_ms, "img_per_s": batch / (e_ms * 1e-3), "windows_ms": te}
        parts = {k: [] for k in ("stage", "tps_pp", "layer3_5_library", "encoder", "decode", "convertor")}
        bb = rec.backbone
        for _ in range(windows):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
            ev[0].record()
            x, outs = bb.stage(img)
            ev[1].record()
            x = rec.tpsnet(x, outs)["output"]
            ev[2].record()
            for name in bb.res_layers[2:]:
                x = getattr(bb, name)(x)
            ev[3].record()
            out_enc = enc(x, metas)
            ev[4].record()
            probs = rec.decoder(x, out_enc, None, metas, train_mode=False)
            ev[5].record()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            idx, _ = rec.label_convertor.tensor2idx(probs, metas)
            rec.label_convertor.idx2str(idx)
            parts["convertor"].append((time.perf_counter() - t0) * 1e3)
            for k, i in zip(("stage", "tps_pp", "layer3_5_library", "encoder", "decode"), range(5)):
                parts[k].append(ev[i].elapsed_time(ev[i + 1]))
        res["simple_test_parts_ms"] = {k: statistics.median(v) for k, v in parts.items()}
        res["example_texts"] = [r["text"] for r in rec.simple_test(img[:2], metas[:2])]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,1024")
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recognizer_bench.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.backends.cuda.matmul.allow_tf32 = False        # the library encoder in plain fp32, as the reference runs it
    rec = build(dev)
    result = {"metric": "nrtr_recognizer", "card": card(), "torch": torch.__version__,
              "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32, "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32,
              "what": "seeded NRTR (ResNetABI_v2_large strides [1,2,2,1,2] + TPS_PP + NRTREncoder 6x512 + NRTRDecoder 40 steps, "
                      "DICT90), random N(0,1) images resident on the device, valid_ratio 1.0",
              "results": [bench_batch(rec, int(b), dev, args.windows) for b in args.batches.split(",")]}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
