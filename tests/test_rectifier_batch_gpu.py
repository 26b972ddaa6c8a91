"""GPU: the rectifier forward bench.py times -- TPS_PP.forward, native head + fused warp -- against fp64 torch on the device,
at the batches and in the head modes bench.py runs, on bench.py's own weights and inputs.

The head's persistent kernels wrap many times at these batches (tests/test_rectifier_batch_cpu.py restates the launch plan):
at B = 256 down_fused_kernel makes 55 passes, conv_tma_kernel 6.9 and the Mlp / score kernels 13.8, where the stage tests
(tests/test_head_gpu.py) stay within one or two.  With the trained-like weights C' barely depends on the head's deep stages
(localization_fc2.weight ~ 5e-5), so every stage is compared on its own, not just the module's output.

Cases: (head mode, B) of tests/test_rectifier_batch_cpu.py::CASES.  Each is checked for
  1. every head stage (the workspace slots, feat_grid, C', pc_score) against fp64, by the rules of test_head_gpu.py;
  2. the module's output / mp_img against the fp64 forward, by the rule of test_module_gpu.py;
  3. the fused warp alone: output / mp_img against the fp64 warp of the module's own feat_grid, C' and pc_score;
  4. run to run, bit for bit;
  5. batch invariance: 8-image windows at the plan's pass boundaries bit-equal to a B = 8 call;
  6. the kernels that ran, under the profiler, against the plan (and against bench.py's launch labels).
tc-2048 compares a fixed sample of images (batch_sample: the first and last 8, and the images of every persistent kernel's
first wrap-around and last pass) instead of all 2048.

The fp64 references restate the oracle's head (oracle.tpspp_oracle.head_intermediates / tpe), tpspp_grid and the sampler
with device tensors, run in slices of 128 images, and are pinned to the oracle functions on 2 images first.  The fp32
floor is the same restatement in fp32 with cuDNN / cuBLAS TF32 off."""
import os
import subprocess
import sys
from collections import Counter

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bench
import tps_pp_b200 as T
from oracle import tpspp_oracle as O
from tps_pp_b200 import _native as N
from tps_pp_b200 import functional as TF

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_inference_batch_gpu import _true_fp32, _worst, rel  # noqa: E402
from test_rectifier_batch_cpu import CASES, batch_sample, head_plan, window_starts  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PIN_TOL = 1e-10        # device reference against its oracle function, both fp64
FLOOR_K = 1.5          # module pixels against the fp32 floor (tests/test_module_gpu.py)
WARP_TOL = 1e-5        # the fused warp on its own inputs (tier 3, tests/test_warp_gpu.py)
SLICE = 128            # images per fp64 reference slice
FULL = 1024            # batches up to this are compared image for image; larger ones on batch_sample
MODE = {"tc": (N.HEAD_TC, 0), "tc3x": (N.HEAD_TC, N.HEAD_FLAG_TF32X3_CONV), "bf16": (N.HEAD_BF16, 0), "fp32": (N.HEAD_FP32, 0)}
# per-image shapes of the workspace slots (NCHW; the bf16 mode stores BF16_SLOTS as bf16 [H, W, C])
SLOTS = dict(f0=(64, 32, 128), f1=(64, 32, 128), f2=(64, 16, 64), a0=(64, 16, 64), a1=(64, 16, 64), e0=(64, 16, 64),
             e1=(64, 8, 32), e2=(64, 4, 16), e3=(64, 2, 16), cbam=(64, 2, 16), d0=(64, 4, 16), d1=(64, 8, 32), d2=(64, 16, 64),
             de=(64, 16, 64), x1=(64, 16, 64), v=(64, 16, 64), de2=(64, 16, 64), p1=(32, 128))
BF16_SLOTS = {"f0", "f1", "f2", "a0", "a1", "e0", "d2"}
STAGES = ["f0", "f1", "f2", "a0", "a1", "feat_grid", "e0", "e1", "e2", "e3", "cbam", "d0", "d1", "d2", "de", "x1", "v", "de2",
          "p1", "c_prime", "pc_score"]
PX = torch.tensor([127 / 2, 31 / 2], dtype=torch.float64)     # grid units -> source pixels of feat_grid (32 x 128)


# ---------------------------------------------------------------- device references
def _w(sd, k, dt):
    return sd[k].to(DEV, dt)


def _conv_relu(sd, p, x, stride=1, padding=0):
    return F.relu(F.conv2d(x, _w(sd, p + ".conv.weight", x.dtype), _w(sd, p + ".conv.bias", x.dtype), stride=stride,
                           padding=padding))


def _linear(sd, p, x, bias=True):
    return F.linear(x, _w(sd, p + ".weight", x.dtype), _w(sd, p + ".bias", x.dtype) if bias else None)


def _cbam(sd, p, x):
    """O.cbam."""
    w0, w2 = _w(sd, p + ".channel_attention.shared_MLP.0.weight", x.dtype), _w(sd, p + ".channel_attention.shared_MLP.2.weight", x.dtype)

    def mlp(v):
        return F.conv2d(F.relu(F.conv2d(v, w0)), w2)
    out = torch.sigmoid(mlp(x.mean(dim=(2, 3), keepdim=True)) + mlp(x.amax(dim=(2, 3), keepdim=True))) * x
    sp = torch.cat([out.mean(dim=1, keepdim=True), out.amax(dim=1, keepdim=True)], dim=1)
    return torch.sigmoid(F.conv2d(sp, _w(sd, p + ".spatial_attention.conv2d.weight", x.dtype),
                                  _w(sd, p + ".spatial_attention.conv2d.bias", x.dtype), padding=1)) * out


def _head_ref(sd, x, o0, o1, dtype):
    """O.head_intermediates on device tensors, with C' and pc_score as O.tpe computes them (its DGAB output is de2)."""
    x, o0, o1 = x.to(dtype), o0.to(dtype), o1.to(dtype)
    r = {"f0": _conv_relu(sd, "down0", o0), "f1": _conv_relu(sd, "down1", o1), "f2": _conv_relu(sd, "down2", x)}
    r["a0"] = _conv_relu(sd, "down0_1", r["f0"], 2, 1)
    r["a1"] = _conv_relu(sd, "down1_1", r["f1"], 2, 1)
    up = F.interpolate(r["f2"], scale_factor=2, mode="nearest")
    r["feat_grid"] = _conv_relu(sd, "down_feat", torch.cat((r["f0"], r["f1"], up), dim=1))
    k = torch.cat((r["a0"], r["a1"], r["f2"]), dim=1)
    for i, s in enumerate([1, 2, 2, (2, 1)]):
        k = _conv_relu(sd, f"MSFA.conv.k_encoder.{i}", k, s, 1)
        r[f"e{i}"] = k
    k = r["cbam"] = _cbam(sd, "MSFA.conv.atten", r["e3"])
    skips = [r["e2"], r["e1"], r["e0"]]
    for i, sc in enumerate([(2, 1), 2, 2, 1]):
        if sc != 1:
            k = F.interpolate(k, scale_factor=sc, mode="nearest")
        k = _conv_relu(sd, f"MSFA.conv.k_decoder.{i}.1", k, 1, 1)
        if i < 3:
            k = r[f"d{i}"] = k + skips[i]
    r["de"] = k
    pre = "TPE.atten.0"
    en = r["e3"].flatten(2).transpose(1, 2)
    h, w = k.shape[2], k.shape[3]
    u = F.layer_norm(k, (h, w), _w(sd, pre + ".norm1.weight", dtype), _w(sd, pre + ".norm1.bias", dtype))
    yt = en.transpose(1, 2)
    lw = F.linear(torch.cat([u.mean(2), yt], 2), _w(sd, pre + ".attn.mlp_w.0.weight", dtype))
    lh = F.linear(torch.cat([u.mean(3), yt], 2), _w(sd, pre + ".attn.mlp_h.0.weight", dtype))
    v_w = lw[:, :, :-1].softmax(dim=-1).unsqueeze(2)
    v_h = lh[:, :, :-1].softmax(dim=-1).unsqueeze(3)
    a = v_h * u * lh[:, :, -1].unsqueeze(-1).unsqueeze(-1) + v_w * u * lw[:, :, -1].unsqueeze(-1).unsqueeze(-1)
    r["x1"] = k + _linear(sd, pre + ".attn.proj", a)
    r["v"] = F.layer_norm(r["x1"], (h, w), _w(sd, pre + ".norm2.weight", dtype), _w(sd, pre + ".norm2.bias", dtype))
    r["de2"] = r["x1"] + _linear(sd, pre + ".mlp.fc2", F.gelu(_linear(sd, pre + ".mlp.fc1", r["v"])))
    r["p1"] = _linear(sd, "TPE.p_linear.1", _linear(sd, "TPE.p_linear.0", en))
    z = F.relu(_linear(sd, "TPE.localization_fc1.2", F.relu(_linear(sd, "TPE.localization_fc1.0", en))))
    r["c_prime"] = _linear(sd, "TPE.localization_fc2", z.reshape(z.shape[0], -1)).view(z.shape[0], -1, 2)
    f = _linear(sd, "TPE.feat_linear.1", _linear(sd, "TPE.feat_linear.0", r["de2"].flatten(2).transpose(1, 2)))
    r["pc_score"] = torch.tanh(torch.einsum("bmc,bnc->bmn", f, r["p1"]) * 64 ** -0.5)
    return r


def _grid(cp, sc, consts, dtype):
    """O.tpspp_grid on device tensors -> [B, 16, 64, 2]."""
    hat, P, P_hat = (t.to(DEV, dtype) for t in consts)
    b, f = cp.shape[:2]
    n = P.shape[0]
    tm = torch.einsum("ij,bjk->bik", hat[:, :f], cp.to(dtype))
    phi = torch.cat([torch.ones((b, n, 1), dtype=dtype, device=DEV), P[None].expand(b, n, 2),
                     P_hat[None] * (sc.to(dtype) * O.THETA + 1)], dim=2)
    return torch.einsum("bpk,bkc->bpc", phi, tm).view(b, 16, 64, 2)


def _sample(src, grid):
    return F.grid_sample(src.to(grid.dtype), grid, padding_mode="border", align_corners=True)


# ---------------------------------------------------------------- module, inputs, read-back
def _module(mode):
    m = T.TPS_PP().to(DEV).eval()
    bench._trained_like_(m)
    m.head_precision, flags = MODE[mode]
    m.head_flags |= flags
    return m


def _state(m):
    return {k: v.detach() for k, v in m.state_dict().items()}


def _consts(m):
    at = m.atten_tps
    return at.hat_C, at.P, at.P_hat


def _bench_inputs(B, from_image=False):
    """x, o0, o1 as bench.py draws them; from_image: the native backbone stage's outputs for bench.py's images instead."""
    g = torch.Generator(device=DEV).manual_seed(1234)
    x = torch.randn((B, 64, 16, 64), device=DEV, generator=g)
    o0 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
    o1 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
    if not from_image:
        return x, o0, o1
    img = torch.randn((B, 3, 32, 128), device=DEV, generator=g)
    bb = T.ResNetABI_v2_large(arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]).to(DEV).eval()
    bench._trained_like_backbone_(bb)
    with torch.no_grad():
        x, outs = bb.stage(img)
    assert bb._last_stage_native
    return x, outs[0], outs[1]


def _slots(m, B, bf16):
    """The module's workspace slots of its last call as [B, C, H, W] (or [B, 32, 128]) float views (bf16 slots upcast)."""
    ws = m._head_ws[(torch.device(DEV).index, torch.cuda.current_stream().cuda_stream)][0]
    off = TF.head_workspace_offsets(TF.head_cfg(B, 16, 64, (2, 16), 2))
    out = {}
    for name, shp in SLOTS.items():
        n = B * int(np.prod(shp))
        if bf16 and name in BF16_SLOTS:
            c, h, w = shp
            out[name] = ws[off[name]: off[name] + 2 * n].view(torch.bfloat16).view(B, h, w, c).permute(0, 3, 1, 2)
        else:
            out[name] = ws[off[name]: off[name] + 4 * n].view(torch.float32).view(B, *shp)
    return out


def _kernels(fn):
    """fn once under the profiler -> the library's kernels, as 'name<template args>'."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof, torch.no_grad():
        fn()
        torch.cuda.synchronize()
    return [e.name.replace("void ", "").replace("tpspp::", "").split("(")[0] for e in prof.events() if "tpspp::" in e.name]


def _power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip() or "not read"
    except (OSError, subprocess.SubprocessError):
        return "not read"


def _tol(mode, name, floor, scale):
    """The small-batch rules of test_head_stages_vs_oracle (fp32 / tc / tc3x) and test_bf16_conv_mode_stated_tolerance, with
    three bounds raised.  Every image's error is a property of the image alone: each worst image is bit-equal to a B = 8 call
    on it.  The small-batch bounds were set on one 19-image batch; a 19-image batch drawn at random from bench.py's images
    already exceeds them in more than 5 % of draws (stage-input pc_score, bf16 pc_score and de2), and the batch checks take
    the maximum over every image.  Per-image max
    error, median / 90 % / 99 % / max over the batch, and the worst of 19 random images (2000 draws: median, 95 %), measured
    on an NVIDIA B200 at 1000 W (DESIGN.md "Parity tiers"):
      * tc pc_score (bound 2e-4 -> 4e-4): tc-256 5.2e-5 / 6.2e-5 / 8.1e-5 / 1.8e-4, 19 random 7.3e-5, 1.8e-4;
        stage-256 8.8e-5 / 1.1e-4 / 1.3e-4 / 3.5e-4, 19 random 1.2e-4, 3.5e-4; tc-683 max 2.1e-4; tc-1024 max 2.0e-4;
      * bf16 pc_score (0.15 -> 0.25): 0.071 / 0.088 / 0.12 / 0.185, 19 random 0.10, 0.185;
      * bf16 v / de2 (3e-2 -> 8e-2 of scale; scale 14.4 for de2, 26.5 for v): de2 0.13 / 0.24 / 0.58 / 1.03, 19 random
        0.39, 1.03; v 0.27 / 0.37 / 0.52 / 0.79, 19 random 0.41, 0.79."""
    if mode == "bf16":
        return {"c_prime": 1e-4, "pc_score": 0.25}.get(name, (8e-2 if name in ("v", "de2") else 3e-2) * scale)
    if mode == "fp32":
        return 4 * floor + 1e-6 * max(scale, 1.0)
    if name == "pc_score":
        return 4e-4
    return 4 * floor + 5e-5 * max(scale, 1.0)


class _Acc:
    """Running (max error, image, position) / fp32 floor / scale of one compared tensor over the reference slices."""

    def __init__(self):
        self.err, self.b, self.pos, self.floor, self.scale = 0.0, -1, None, 0.0, 0.0

    def add(self, got, r64, ii, r32=None):
        err, b, pos = _worst((got.double() - r64).abs())
        if err >= self.err:
            self.err, self.b, self.pos = err, int(ii[b]), pos
        if r32 is not None:
            self.floor = max(self.floor, float((r32.double() - r64).abs().max()))
        self.scale = max(self.scale, float(r64.abs().max()))


# ---------------------------------------------------------------- the references against the oracle
def test_references_match_oracle(native_lib):
    m = _module("tc")
    sd = _state(m)
    x, o0, o1 = _bench_inputs(2)
    r = _head_ref(sd, x, o0, o1, torch.float64)
    ref = O.head_intermediates(sd, x.cpu(), [o0.cpu(), o1.cpu()], dtype=torch.float64)
    errs = {k: rel(r[k], ref[k]) for k in STAGES}
    hat, P, P_hat = (t.cpu().numpy() for t in _consts(m))
    g = _grid(r["c_prime"], r["pc_score"], _consts(m), torch.float64)
    g_o = O.tpspp_grid(ref["c_prime"].numpy(), ref["pc_score"].numpy(), hat, P, P_hat)
    errs["grid"] = rel(g.view(2, -1, 2), g_o)
    out = _sample(r["feat_grid"], g)
    errs["grid_sample"] = rel(out, O.grid_sample(r["feat_grid"].cpu().numpy(), g.cpu().numpy(), dtype=np.float64))
    worst = max(errs, key=errs.get)
    print(f"device: {torch.cuda.get_device_name(DEV)}, power limit {_power_limit()}")
    print(f"device references vs oracle (fp64, 2 images): worst rel {errs[worst]:.1e} ({worst}; tol {PIN_TOL:.0e})")
    assert errs[worst] <= PIN_TOL, errs


# ---------------------------------------------------------------- the cases
@pytest.mark.parametrize("case", list(CASES))
def test_rectifier_forward_at_bench_batch(native_lib, case):
    mode, B = CASES[case]
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    plan = head_plan(B, sms, mode)
    m = _module(mode)
    sd, consts = _state(m), _consts(m)
    x, o0, o1 = _bench_inputs(B, from_image=case.startswith("stage"))
    idx = torch.arange(B, device=DEV) if B <= FULL else torch.tensor(batch_sample(B, sms, mode), device=DEV)
    bf16 = mode == "bf16"
    with torch.no_grad():
        m(x, [o0, o1])                                   # weight images and the workspace stamp
        r = m(x, [o0, o1])
        fg, cp, sc = m.head(x, [o0, o1])
    torch.cuda.synchronize()
    assert all(m.native_stages.values())
    assert torch.equal(sc, r["pc_score"])
    assert fg.dtype == (torch.bfloat16 if bf16 else torch.float32)    # bf16 mode: bf16 feat_grid into the staged warp
    got = {k: v[idx].float().clone() for k, v in _slots(m, B, bf16).items()}
    got.update(feat_grid=fg[idx].float(), c_prime=cp[idx], pc_score=sc[idx])

    # 1-3: against fp64, slice by slice
    acc = {k: _Acc() for k in STAGES + ["output", "mp_img", "warp_output", "warp_mp_img", "grid_px"]}
    for s in range(0, len(idx), SLICE):
        ii = idx[s:s + SLICE]
        j = slice(s, s + SLICE)
        r64 = _head_ref(sd, x[ii], o0[ii], o1[ii], torch.float64)
        with _true_fp32():
            r32 = _head_ref(sd, x[ii], o0[ii], o1[ii], torch.float32)
            g32 = _grid(r32["c_prime"], r32["pc_score"], consts, torch.float32)
            out32, mp32 = _sample(r32["feat_grid"], g32), _sample(x[ii], g32)
        del g32
        for k in STAGES:
            acc[k].add(got[k][j], r64[k], ii, r32[k])
        del r32
        g64 = _grid(r64["c_prime"], r64["pc_score"], consts, torch.float64)
        acc["output"].add(r["output"][ii], _sample(r64["feat_grid"], g64), ii, out32)
        acc["mp_img"].add(r["mp_img"][ii], _sample(x[ii], g64), ii, mp32)
        own = _grid(got["c_prime"][j], got["pc_score"][j], consts, torch.float64)
        acc["grid_px"].add(own * PX.to(DEV), g64 * PX.to(DEV), ii)
        acc["warp_output"].add(r["output"][ii], _sample(fg[ii], own), ii)
        acc["warp_mp_img"].add(r["mp_img"][ii], _sample(x[ii], own), ii)
        del r64, g64, own, out32, mp32
    over, rep = [], []
    for k in STAGES:
        a = acc[k]
        tol = _tol(mode, k, a.floor, a.scale)
        if k == "c_prime":
            tol = min(tol, 1e-4)
        rep.append(f"{k:10s} {a.err:.2e} (tol {tol:.2e}, fp32 floor {a.floor:.2e}, scale {a.scale:.2f}) image {a.b} at {a.pos}")
        if a.err > tol:
            over.append((k, a.err, tol, a.b, a.pos))
    for k in ("output", "mp_img"):
        a = acc[k]
        tol = 6e-2 * a.scale if bf16 else max(1e-5, FLOOR_K * a.floor)
        rep.append(f"{k:10s} {a.err:.2e} (tol {tol:.2e}, fp32 floor {a.floor:.2e}) image {a.b} at {a.pos}")
        if a.err > tol:
            over.append((k, a.err, tol, a.b, a.pos))
    for k in ("warp_output", "warp_mp_img"):
        a = acc[k]
        rep.append(f"{k:10s} {a.err:.2e} (tol {WARP_TOL:.0e}, fp64 warp of the module's own feat_grid / C' / pc_score) "
                   f"image {a.b} at {a.pos}")
        if a.err > WARP_TOL:
            over.append((k, a.err, WARP_TOL, a.b, a.pos))
    if bf16:
        a = acc["grid_px"]
        rep.append(f"grid       {a.err:.3f} source px (tol 0.5) image {a.b}")
        if a.err > 0.5:
            over.append(("grid_px", a.err, 0.5, a.b, a.pos))
    print(f"\n[{case}: {mode}, B={B}, {len(idx)} images against fp64]\n" + "\n".join(rep))
    assert not over, over
    del acc

    # 4. run to run, bit for bit
    with torch.no_grad():
        r2 = m(x, [o0, o1])
    for k in ("output", "mp_img", "pc_score"):
        assert torch.equal(r2[k], r[k]), k
    del r2
    for k, v in _slots(m, B, bf16).items():
        assert torch.equal(v[idx].float(), got[k]), f"workspace slot {k} differs run to run"
    del got

    # 6. the kernels that ran (cached weight images: no wprep launch)
    # Launch count from the library's own counters: the head's launches plus the warp's, one per planned launch
    with torch.no_grad():
        m(x, [o0, o1])
    assert m._last_head_launches + N.last_launch_count() == len(plan), (case, m._last_head_launches, N.last_launch_count())
    # Per-kernel launch counts under the profiler (a multiset: with programmatic dependent launch the kernels overlap, so the
    # trace's start times do not keep the launch order, which tests/test_rectifier_batch_cpu.py pins against bench.py's
    # labels).  Two calls are profiled: after many profiler sessions in one process the trace has been seen to drop the
    # first launches of the window, so the count may miss a prefix of the first call's launches -- and nothing else.
    kernels = [e["kernel"] for e in plan]
    seen = Counter(_kernels(lambda: [m(x, [o0, o1]) for _ in range(2)]))
    missing = Counter(kernels * 2) - seen
    assert not seen - Counter(kernels * 2), (case, seen - Counter(kernels * 2))
    assert any(missing == Counter(kernels[:d]) for d in range(len(kernels))), (case, missing)

    # 5. batch invariance
    starts = window_starts(B, sms, mode)
    with torch.no_grad():
        for lo in starts:
            part = m(x[lo:lo + 8], [o0[lo:lo + 8], o1[lo:lo + 8]])
            pfg, pcp, psc = m.head(x[lo:lo + 8], [o0[lo:lo + 8], o1[lo:lo + 8]])
            for k in ("output", "mp_img", "pc_score"):
                assert torch.equal(part[k], r[k][lo:lo + 8]), (lo, k)
            assert torch.equal(pfg, fg[lo:lo + 8]) and torch.equal(pcp, cp[lo:lo + 8]) and torch.equal(psc, sc[lo:lo + 8]), lo
    print(f"[{case}] run to run bit-equal; 8-image windows at {starts} bit-equal to B = 8 calls; kernels as planned")


def test_back_to_back_forwards_match_serial(native_lib):
    """bench.py's timed loop: TPS_PP.forward calls on different inputs issued with no synchronisation between them (the warp
    chained to the next call's head by programmatic dependent launch) -- each bit-equal to its serial result."""
    B, reps = 256, 8
    m = _module("tc")
    g = torch.Generator(device=DEV).manual_seed(99)
    ins = [(torch.randn((B, 64, 16, 64), device=DEV, generator=g), torch.randn((B, 32, 32, 128), device=DEV, generator=g),
            torch.randn((B, 32, 32, 128), device=DEV, generator=g)) for _ in range(reps)]
    keys = ("output", "mp_img", "pc_score")
    with torch.no_grad():
        serial = []
        for x, o0, o1 in ins:
            r = m(x, [o0, o1])
            torch.cuda.synchronize()
            serial.append([r[k].clone() for k in keys])
        outs = [m(x, [o0, o1]) for x, o0, o1 in ins]
        torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(outs, serial)):
        for k, v in zip(keys, b):
            assert torch.equal(a[k], v), (i, k)


def test_one_image_change_stays_in_its_image(native_lib):
    """Noise on a 2-row band of o0 in a late image moves that image's outputs and leaves every other image's bits alone."""
    B, hit = 256, 250
    m = _module("tc")
    x, o0, o1 = _bench_inputs(B)
    noisy = o0.clone()
    g = torch.Generator(device=DEV).manual_seed(7)
    noisy[hit, :, 20:22, :] += 4.0 * torch.randn((32, 2, 128), device=DEV, generator=g)
    with torch.no_grad():
        base = {k: v.clone() for k, v in m(x, [o0, o1]).items() if v is not None}
        moved = m(x, [noisy, o1])
    keep = torch.ones(B, dtype=torch.bool, device=DEV)
    keep[hit] = False
    shifts = {k: float((moved[k][hit] - base[k][hit]).abs().max()) for k in base}
    print(f"o0 rows 20-21 of image {hit} + noise: its outputs move by {shifts}")
    for k in base:
        assert shifts[k] > 0, k
        assert torch.equal(moved[k][keep], base[k][keep]), k

