"""GPU: the rectifier's training kernels at the batch the training step runs (B = 128, scripts/train_step_bench.py) against fp64
torch autograd on the device.

The work split of these kernels changes with the batch, and the other tests run them at B <= 8: there every persistent
convolution CTA takes one 128-pixel tile, a weight-gradient pixel split covers 8 to 13 chunks and half of the bias-gradient
batch splits are empty.  At B = 128 a CTA takes up to ~14 tiles, a split up to ~216 chunks, and the warp backward runs ~55
(image, channel) planes per CTA.  Here:

  * every training convolution (GEOMS and FUSED of test_conv_train_gpu.py) at B = 4 (the smallest batch that keeps every layer
    native; single-split weight gradients of the deepest layers), 128 and 132 (tiles, chunks and bias splits that do not
    divide evenly);
  * batch invariance: y and every gx of images [0:8] and [B-8:B] bit-equal to a B = 8 call on the same images (a pixel's
    output and data gradient take the same arithmetic whichever tile and CTA it lands in);
  * determinism of gx, gw and gb at B = 128 (fixed two-stage reductions, no atomics);
  * one real training step at B = 128 replayed layer by layer: every native convolution and dense layer re-run alone on the
    inputs and output gradient the step gave it, against fp64, and the step's parameter gradients bit-equal to the replay;
  * the staged warp backward at B = 128, C = 64, both sources."""
import os
import sys
import zlib
from collections import Counter

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import tps_pp_b200 as T
from oracle import tpspp_oracle as O
from tps_pp_b200 import _native as N
from tps_pp_b200 import functional as TF

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the per-layer tables beside these tests
from test_conv_train_gpu import FUSED, GEOMS, rel  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
Y_TOL, G_TOL = 2e-5, 1e-4          # convolution output / gradients (test_conv_train_gpu.py)
MAX_B = 132


def _norm_ups(ups, n):
    return [(1, 1)] * n if ups is None else [(u, u) if isinstance(u, int) else tuple(u) for u in ups]


def _stride_id(s):
    return str(s) if isinstance(s, int) else f"{s[0]}x{s[1]}"


# (id, channels per source, nearest-upsample factor per source, conv input h, w, kernel, stride)
CONVS = ([(f"cin{cin}-{h}x{w}-k{k}-s{_stride_id(s)}", [cin], [(1, 1)], h, w, k, s) for cin, h, w, k, s in GEOMS] +
         [(what, chans, _norm_ups(ups, len(chans)), h, w, k, 1) for chans, ups, h, w, k, what in FUSED])
CONV_IDS = [c[0] for c in CONVS]


def _draw(conv):
    """Sources, weight, bias and output gradient of MAX_B images; a smaller batch takes a slice."""
    cid, chans, ups, h, w, k, stride = conv
    g = torch.Generator(device=DEV).manual_seed(zlib.crc32(cid.encode()))
    srcs = [torch.randn((MAX_B, c, h // u[0], w // u[1]), device=DEV, generator=g) for c, u in zip(chans, ups)]
    cin = sum(chans)
    wt = torch.randn((64, cin, k, k), device=DEV, generator=g) * (2.0 / (cin * k * k)) ** 0.5
    bias = torch.randn(64, device=DEV, generator=g) * 0.1
    sh, sw = (stride, stride) if isinstance(stride, int) else stride
    gy = torch.randn((MAX_B, 64, h // sh, w // sw), device=DEV, generator=g)
    return srcs, wt, bias, gy


def _conv_native(srcs, wt, bias, stride, ups, gy, fn=None):
    """y, [gx per source], gw, gb of ``functional.conv_relu`` (or ``fn``, the same op) with output gradient gy."""
    xs = [t.clone().requires_grad_() for t in srcs]
    ws, bs = wt.clone().requires_grad_(), bias.clone().requires_grad_()
    assert TF.conv_relu_supported(xs, ws, stride, ups)
    y = (fn or TF.conv_relu)(xs, ws, bs, stride, True, ups)
    y.backward(gy)
    return y.detach(), [t.grad for t in xs], ws.grad, bs.grad


def _conv_errors(srcs, wt, bias, stride, ups, y, gy, gxs, gw, gb):
    """Errors relative to the reference's max of y, the worst gx, gw and gb against fp64 autograd of
    relu(conv2d(cat(interpolate(x_s)))); the ReLU mask is taken from our forward (pixels within rounding of zero)."""
    k = wt.shape[-1]
    xd = [t.double().requires_grad_() for t in srcs]
    wd, bd = wt.double().requires_grad_(), bias.double().requires_grad_()
    full = torch.cat([t if u == (1, 1) else F.interpolate(t, scale_factor=(float(u[0]), float(u[1])), mode="nearest")
                      for t, u in zip(xd, ups)], dim=1)
    yd = F.conv2d(full, wd, bd, stride=stride, padding=k // 2) * (y > 0).double()
    yd.backward(gy.double())
    for a, r in zip(gxs, xd):
        assert a.shape == r.grad.shape
    return rel(y, yd.detach()), max(rel(a, r.grad) for a, r in zip(gxs, xd)), rel(gw, wd.grad), rel(gb, bd.grad)


@pytest.mark.parametrize("batch", [4, 128, 132])
@pytest.mark.parametrize("conv", CONVS, ids=CONV_IDS)
def test_conv_matches_fp64_at_training_batches(native_lib, conv, batch):
    srcs, wt, bias, gy = _draw(conv)
    srcs, gy = [t[:batch] for t in srcs], gy[:batch]
    stride, ups = conv[6], conv[2]
    y, gxs, gw, gb = _conv_native(srcs, wt, bias, stride, ups, gy)
    e = _conv_errors(srcs, wt, bias, stride, ups, y, gy, gxs, gw, gb)
    print(f"conv [{conv[0]}, B={batch}]: y {e[0]:.2e} (tol {Y_TOL:.0e}); gx {e[1]:.2e}, gw {e[2]:.2e}, gb {e[3]:.2e} "
          f"(tol {G_TOL:.0e})")
    assert e[0] < Y_TOL and max(e[1:]) < G_TOL, e


@pytest.mark.parametrize("conv", CONVS, ids=CONV_IDS)
def test_conv_output_and_data_gradient_are_batch_invariant(native_lib, conv):
    """conv_tma_plan picks the tile from Ho x Wo alone and every pixel takes the same arithmetic in any tile or CTA, so the
    images of a B = 128 / 132 call must give the bits of a B = 8 call (gw and gb sum over the batch: excluded)."""
    srcs, wt, bias, gy = _draw(conv)
    stride, ups = conv[6], conv[2]
    for batch in (128, 132):
        y, gxs, _, _ = _conv_native([t[:batch] for t in srcs], wt, bias, stride, ups, gy[:batch])
        for lo in (0, batch - 8):
            y8, gx8, _, _ = _conv_native([t[lo:lo + 8] for t in srcs], wt, bias, stride, ups, gy[lo:lo + 8])
            assert torch.equal(y[lo:lo + 8], y8), (batch, lo)
            for s, (a, b) in enumerate(zip(gxs, gx8)):
                assert torch.equal(a[lo:lo + 8], b), (batch, lo, s)


@pytest.mark.parametrize("conv", CONVS, ids=CONV_IDS)
def test_conv_backward_is_deterministic_at_training_batch(native_lib, conv):
    srcs, wt, bias, gy = _draw(conv)
    srcs, gy = [t[:128] for t in srcs], gy[:128]
    stride, ups = conv[6], conv[2]
    y0, gx0, gw0, gb0 = _conv_native(srcs, wt, bias, stride, ups, gy)
    y1, gx1, gw1, gb1 = _conv_native(srcs, wt, bias, stride, ups, gy)
    assert torch.equal(y0, y1)
    assert all(torch.equal(a, b) for a, b in zip(gx0, gx1))
    assert torch.equal(gw0, gw1) and torch.equal(gb0, gb1)


# ---------------------------------------------------------------- one training step, replayed layer by layer
def _copy(a):
    if torch.is_tensor(a):
        return a.detach().clone()
    if isinstance(a, (list, tuple)) and any(torch.is_tensor(t) for t in a):
        return [t.detach().clone() for t in a]
    return a


def _recorder(kind, fn, calls):
    """``fn`` as is, plus a record of its inputs, its output and (by a hook, during backward) its output's gradient."""
    def record(*args):
        y = fn(*args)
        entry = {"kind": kind, "args": [_copy(a) for a in args], "ptrs": [a.data_ptr() if torch.is_tensor(a) else None for a in args],
                 "y": y.detach().clone(), "gy": None}
        calls.append(entry)
        y.register_hook(lambda g: entry.__setitem__("gy", g.detach().clone()))
        return y
    return record


def _dense_tols(kind, k, n, bias):
    """(y, gx, gw, gb) tolerances of tests/test_linear_train_gpu.py (3xTF32 with fp32 accumulation)."""
    if kind == "bmm_nt":
        return 2e-6, 2e-6, 5e-6, None
    return 3e-6 * max(1.0, (k / 256) ** 0.5), 3e-6 * max(1.0, (n / 256) ** 0.5), 8e-6, 5e-6 if bias else None


def test_training_step_layers_replayed_at_batch_128(native_lib, monkeypatch):
    """Every native convolution and dense layer of one training step at B = 128, on the inputs and output gradient the
    step gave it (real shapes: the DGAB MLP at 131072 rows, the score bmm with 128 weight batches; real activations and ReLU
    sparsity), against fp64; the step's parameter gradients must be the bits of the replayed weight / bias gradients."""
    m = T.TPS_PP().to(DEV).train()
    m.load_state_dict(O.trained_like_state(3), strict=True)
    orig = {name: getattr(TF, name) for name in ("conv_relu", "linear", "bmm_nt")}
    calls = []
    for name, fn in orig.items():
        monkeypatch.setattr(TF, name, _recorder(name, fn, calls))
    x, o0, o1 = (torch.from_numpy(a).to(DEV).requires_grad_() for a in O.synthetic_tpspp_inputs(128, 12))
    m(x, [o0, o1])["output"].square().mean().backward()
    monkeypatch.undo()
    assert m.training_stages == {"convs_native": 14, "convs_library": 0, "linears_native": 16, "linears_library": 0}
    assert Counter(c["kind"] for c in calls) == {"conv_relu": 14, "linear": 15, "bmm_nt": 1}
    assert all(c["gy"] is not None for c in calls)

    params = dict(m.named_parameters())
    name_of = {p.data_ptr(): name for name, p in params.items()}
    uses, replayed = Counter(), {}
    worst, over = {}, []
    for c in calls:
        kind, gy = c["kind"], c["gy"]
        if kind == "conv_relu":
            srcs, wt, bias, stride, relu, ups = c["args"]
            srcs = [srcs] if torch.is_tensor(srcs) else srcs
            ups = _norm_ups(ups, len(srcs))
            assert relu
            y, gxs, gw, gb = _conv_native(srcs, wt, bias, stride, ups, gy, orig[kind])
            errs = _conv_errors(srcs, wt, bias, stride, ups, y, gy, gxs, gw, gb)
            tols = (Y_TOL, G_TOL, G_TOL, G_TOL)
            shape = f"{len(srcs)}x{tuple(srcs[0].shape)} k{wt.shape[-1]} s{_stride_id(stride)}"
        else:
            xin, w = c["args"][0], c["args"][1]
            bias = c["args"][2] if kind == "linear" else None
            xs, ws = xin.clone().requires_grad_(), w.clone().requires_grad_()
            bs = bias.clone().requires_grad_() if bias is not None else None
            y = orig[kind](xs, ws, bs) if kind == "linear" else orig[kind](xs, ws)
            y.backward(gy)
            y, gw, gb = y.detach(), ws.grad, (bs.grad if bs is not None else None)
            xd, wd = xin.double().requires_grad_(), w.double().requires_grad_()
            bd = bias.double().requires_grad_() if bias is not None else None
            yd = F.linear(xd, wd, bd) if kind == "linear" else torch.bmm(xd, wd.transpose(1, 2))
            yd.backward(gy.double())
            errs = (rel(y, yd.detach()), rel(xs.grad, xd.grad), rel(gw, wd.grad), rel(gb, bd.grad) if bd is not None else 0.0)
            tols = _dense_tols(kind, w.shape[-1], w.shape[-2], bias is not None)
            shape = f"{tuple(xin.shape)} x {tuple(w.shape)}"
        assert torch.equal(y, c["y"]), "the replayed forward differs from the step's"
        label = "score bmm" if kind == "bmm_nt" else name_of[c["ptrs"][1]]
        for ptr, grad in ((c["ptrs"][1], gw), (c["ptrs"][2] if len(c["ptrs"]) > 2 else None, gb)):
            if ptr in name_of:
                uses[ptr] += 1
                replayed[ptr] = grad
        print(f"replay {label} [{kind} {shape}]: y {errs[0]:.2e}/{tols[0]:.0e}, gx {errs[1]:.2e}/{tols[1]:.0e}, "
              f"gw {errs[2]:.2e}/{tols[2]:.0e}" + (f", gb {errs[3]:.2e}/{tols[3]:.0e}" if tols[3] else ""))
        for i, what in enumerate(("y", "gx", "gw", "gb")):
            if tols[i] is not None:
                if errs[i] / tols[i] >= worst.get((kind, what), (-1.0, ""))[0]:
                    worst[(kind, what)] = (errs[i] / tols[i], label)
                if errs[i] > tols[i]:
                    over.append((label, what, errs[i], tols[i]))
    for (kind, what), (ratio, label) in sorted(worst.items()):
        print(f"replay worst {kind} {what}: {ratio:.2f} of its tolerance ({label})")
    assert not over, over
    # every parameter but the LayerNorms' (torch ops) feeds exactly one native call; its gradient from the step is that call's
    assert sorted(name_of[p] for p in uses) == sorted(n for n in params if ".norm" not in n)
    for ptr, count in uses.items():
        name = name_of[ptr]
        assert count == 1, name
        assert torch.equal(params[name].grad.reshape(-1), replayed[ptr].reshape(-1)), name


# ---------------------------------------------------------------- staged warp backward
def test_staged_warp_backward_at_training_batch(native_lib):
    """AUTO (staged) backward of the module's warp geometry (64 channels, 32x128 and 16x64 sources, both outputs' gradients)
    at B = 128 -- 8192 planes, ~55 per persistent CTA -- against fp64 autograd of bmm + grid_sample, and run to run."""
    c = O.tpspp_constants()
    hat, ph, P = (torch.from_numpy(np.ascontiguousarray(c[k])).float().to(DEV) for k in ("hat_C", "P_hat", "P"))
    B, C = 128, 64
    g = torch.Generator(device=DEV).manual_seed(128)
    fg = torch.randn((B, C, 32, 128), device=DEV, generator=g)
    x = torch.randn((B, C, 16, 64), device=DEV, generator=g)
    s = torch.tanh(0.5 * torch.randn((B, 1024, 32), device=DEV, generator=g))
    go0 = torch.randn((B, C, 16, 64), device=DEV, generator=g)
    go1 = torch.randn((B, C, 16, 64), device=DEV, generator=g)
    cp = torch.from_numpy(O.smooth_c_prime(O.tpspp_init_bias(), B, seed=9)).to(DEV)
    assert TF.BWD_VARIANT == N.VARIANT_AUTO
    runs = []
    for _ in range(2):
        leaves = [t.clone().requires_grad_() for t in (fg, x, cp, s)]
        out, mp = TF.tps_warp(*leaves, ph, P, hat, (16, 64))
        ((out * go0).sum() + (mp * go1).sum()).backward()
        runs.append((out.detach(), mp.detach(), [t.grad for t in leaves]))
    for a, b in zip(runs[0][2], runs[1][2]):
        assert torch.equal(a, b)
    d = torch.float64
    rfg, rx, rcp, rs = (t.double().requires_grad_() for t in (fg, x, cp, s))
    phi = torch.cat([torch.ones(B, 1024, 1, dtype=d, device=DEV), P.double()[None].repeat(B, 1, 1),
                     ph.double()[None] * (rs * 0.5 + 1)], 2)
    Tm = torch.bmm(hat.double()[None].repeat(B, 1, 1), torch.cat([rcp, torch.zeros(B, 3, 2, dtype=d, device=DEV)], 1))
    grid = torch.bmm(phi, Tm).reshape(B, 16, 64, 2)
    r0 = F.grid_sample(rfg, grid, padding_mode="border", align_corners=True)
    r1 = F.grid_sample(rx, grid, padding_mode="border", align_corners=True)
    ((r0 * go0.double()).sum() + (r1 * go1.double()).sum()).backward()
    out, mp, (gfg, gx, gcp, gs) = runs[0]
    e_out = max(float((out - r0).abs().max()), float((mp - r1).abs().max()))
    e_src = max(float((gfg - rfg.grad).abs().max()), float((gx - rx.grad).abs().max()))
    e_cp, e_s = rel(gcp, rcp.grad), rel(gs, rs.grad)
    print(f"staged warp backward [B={B}, C={C}]: outputs {e_out:.2e} (tol 1e-5); d src {e_src:.2e} (tol 1e-5 abs); "
          f"d C' {e_cp:.2e}, d score {e_s:.2e} (tol 2e-4 of the max)")
    assert e_out <= 1e-5 and e_src <= 1e-5
    assert e_cp <= 2e-4 and e_s <= 2e-4
