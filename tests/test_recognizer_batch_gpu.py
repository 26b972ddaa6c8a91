"""GPU: the NRTR recogniser's inference kernels at the batches model_inference runs -- chunks of 256 images by default, 1024
in the benchmark scripts, and a ragged last chunk of any size -- against fp64 on the device.

The full nrtr_tps++.py configuration (6 layers, width 512, 8 heads, d_inner 256, DICT90: 92 classifier outputs padded to 96,
64 source tokens).  How the dense layers split their work changes with the row count (the rule is restated and pinned in
tests/test_recognizer_batch_cpu.py); every case below is checked to take the branch its id names, under the profiler too:

  * each dense layer of NRTREncoder._encode (n x 64 rows) and NRTRDecoder._decode (one row per image, padded to 128) called
    the way those methods call it -- in-place residual, GELU, the next LayerNorm -- against fp64, bit-equal on a repeated call
    and, on the unsplit persistent path, bit-equal on its first and last rows to a call with fewer rows;
  * tpspp_attn_encode and both instantiations of tpspp_attn_decode at n = 1024 against fp64, bit-equal to n = 8 calls;
  * the whole encoder and the teacher-forced decoder at batch against fp64, within 4x the error of the fp32 library path;
  * repeatability of NRTR.simple_test stage by stage, with a call of another batch size in between."""
import contextlib
import math
import os
import re
import sys
import zlib

import pytest
import torch
import torch.nn.functional as F

from oracle import tpspp_oracle as O
from tps_pp_b200 import functional as TF
from tps_pp_b200.nrtr import NRTRDecoder, NRTREncoder

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the restatements and helpers beside these tests
from nrtr_encoder_restatement import nrtr_encoder_forward  # noqa: E402
from test_ocr_tta_gpu import _recognizer, crops, ref_kw, rotating_config  # noqa: E402
from test_recognizer_batch_cpu import attn_decode_plan, decoder_rows, encoder_rows, lin_plan  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
D, HEADS, T_SRC = 512, 8, 64
START, PAD = 91, 92                      # DICT90 with <UKN>: the recogniser's start / padding indexes


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-30))


@contextlib.contextmanager
def _true_fp32():
    """The fp32 library path without TF32 (cuBLAS and cuDNN)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            yield
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def _kernels(fn):
    """Runs fn once under the profiler -> the demangled names of the CUDA kernels it launched."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events()]


# ---------------------------------------------------------------- dense layers at the recogniser's shapes
ENC_LAYERS = [("qkv", 512, 1536, "plain"), ("fc", 512, 512, "res+ln"), ("w_1", 512, 256, "gelu"), ("w_2", 256, 512, "res+ln")]
# efc has fc's shape and call; q|k|v, q and the classifier are plain
DEC_LAYERS = [("qkv", 512, 1536, "plain"), ("fc", 512, 512, "res+ln"), ("q", 512, 512, "plain"), ("w_1", 512, 256, "gelu"),
              ("w_2", 256, 512, "res+ln"), ("classifier", 512, 96, "plain")]
DENSE = ([(f"enc-n{n}-{nm}", encoder_rows(n), k, c, kind) for n in (4, 44, 96, 256, 1024) for nm, k, c, kind in ENC_LAYERS]
         + [(f"dec-n{n}-{nm}", decoder_rows(n), k, c, kind) for n in (44, 512, 1024) for nm, k, c, kind in DEC_LAYERS]
         + [(f"dec-n{n}-memory_kv", encoder_rows(n), 512, 1024, "memory") for n in (44, 512, 1024)]
         + [("synthetic-split-ln", 9472, 512, 128, "res+ln")])
ATTN_DECODE = [("memory", 1024, 64), ("memory", 8, 64), ("append", 1024, 40), ("append", 8, 40)]


def _dense_inputs(name, rows, k, n, kind):
    g = torch.Generator(device=DEV).manual_seed(zlib.crc32(name.encode()) % 100000)
    x = torch.randn((rows, k), device=DEV, generator=g)
    w = torch.randn((n, k), device=DEV, generator=g) / k ** 0.5
    b = None if kind == "memory" else torch.randn((n,), device=DEV, generator=g)      # qkv_bias=False: no bias on k|v
    res = torch.randn((rows, n), device=DEV, generator=g)
    ln = torch.nn.LayerNorm(n).to(DEV)
    with torch.no_grad():
        ln.weight.copy_(1.0 + 0.1 * torch.randn((n,), device=DEV, generator=g))
        ln.bias.copy_(0.1 * torch.randn((n,), device=DEV, generator=g))
    return x, w, b, res, ln


def _dense_call(kind, op, x, w, res, ln):
    """One call as _encode / _decode make it -> (y, LN(y) or None)."""
    if kind == "memory":
        return TF.linear(x, w, None), None
    if kind == "res+ln":
        y = res.clone()
        hn = torch.full_like(y, float("nan"))
        op(x, out=y, residual=y, ln=ln, ln_out=hn)
        return y, hn
    return op(x, gelu=kind == "gelu"), None


def _dense_op(kind, w, b, rows):
    return None if kind == "memory" else TF.PreparedLinear(w, b, rows)


def test_cases_cover_every_branch(sms):
    plans = [lin_plan(rows, k, n, sms, ln=kind == "res+ln") for _, rows, k, n, kind in DENSE]
    assert {p["splitk"] for p in plans} >= {1, 2, 4}
    assert any(p["splitk"] == 1 and p["col_split"] and p["tiles_per_cta"] > 1 for p in plans)
    assert any(p["reduce_splits"] == 0 and p["reduce_passes"] > 1 for p in plans if p["reduce"] and "ln" in p["reduce"])
    assert any(p["reduce_splits"] > 0 and p["reduce_passes"] > 1 for p in plans if p["reduce"] and "ln" in p["reduce"])
    assert any(p["reduce"] == "lin_splitk_reduce_kernel" and p["reduce_passes"] > 1 for p in plans)
    assert {attn_decode_plan(b, HEADS, kv) for _, b, kv in ATTN_DECODE} == {"attn_decode_kernel<true>", "attn_decode_kernel<false>"}


def test_kernels_match_the_rule(native_lib, sms):
    """Each case once under the profiler: the reduction kernel behind the tensor-core kernel, its SPLITS, and the decode
    attention's instantiation are the ones the rule names."""
    for name, rows, k, n, kind in DENSE:
        plan = lin_plan(rows, k, n, sms, ln=kind == "res+ln")
        x, w, b, res, ln = _dense_inputs(name, rows, k, n, kind)
        op = _dense_op(kind, w, b, rows)
        names = _kernels(lambda: _dense_call(kind, op, x, w, res, ln))
        seen = sorted({m.group(0) for s in names for m in [re.search(r"lin_reduce_ln_kernel<\d+, \d+>|lin_splitk_reduce_kernel", s)] if m})
        print(f"{name:24s} rows {rows:6d} {k:4d}->{n:4d}: split-K {plan['splitk']}, grid {plan['grid']}, {plan['tiles_per_cta']} "
              f"tiles/CTA, reduce {plan['reduce']} x{plan['reduce_passes']} passes; profiler saw {seen}")
        assert any("lin_tma_kernel" in s for s in names), (name, names)
        assert seen == ([plan["reduce"]] if plan["reduce"] else []), (name, plan, seen)
        del x, res
    g = torch.Generator(device=DEV).manual_seed(5)
    instantiations = set()
    for form, b, kv in ATTN_DECODE:
        q = torch.randn((b, D), device=DEV, generator=g)
        k = torch.randn((b, HEADS, kv, 64), device=DEV, generator=g)
        v = torch.randn_like(k)
        if form == "memory":
            names = _kernels(lambda: TF.attn_decode(q, k, v, HEADS, kv, 8.0, kv_lens=torch.full((b,), kv, dtype=torch.int32, device=DEV),
                                                    head_major=True))
        else:
            names = _kernels(lambda: TF.attn_decode(q, k, v, HEADS, kv, 8.0, k_new=q, v_new=q, head_major=True))
        seen = sorted({m.group(0) for s in names for m in [re.search(r"attn_decode_kernel<\w+>", s)] if m})
        print(f"attn_decode {form} n={b} kv_len {kv}: rule {attn_decode_plan(b, HEADS, kv)}; profiler saw {seen}")
        # after many profiler sessions in one process the trace has been seen to lose this launch (the call's result is
        # checked in test_attn_decode_at_1024); a kernel the trace does hold must be the one the rule names
        assert seen in ([], [attn_decode_plan(b, HEADS, kv)]), (form, b, kv, seen)
        instantiations.update(seen)
    assert instantiations == {"attn_decode_kernel<true>", "attn_decode_kernel<false>"}


def _first_unsplit_rows(k, n, kind, sms, at_least=2048):
    return next(r for r in range(at_least, 1 << 20, 128) if lin_plan(r, k, n, sms, ln=kind == "res+ln")["splitk"] == 1)


@pytest.mark.parametrize("name,rows,k,n,kind", DENSE, ids=[c[0] for c in DENSE])
def test_dense_layer_vs_fp64(native_lib, sms, name, rows, k, n, kind):
    plan = lin_plan(rows, k, n, sms, ln=kind == "res+ln")
    x, w, b, res, ln = _dense_inputs(name, rows, k, n, kind)
    op = _dense_op(kind, w, b, rows)
    y, hn = _dense_call(kind, op, x, w, res, ln)
    y2, hn2 = _dense_call(kind, op, x, w, res, ln)           # PreparedLinear: the cached operand image
    assert torch.equal(y, y2) and (hn is None or torch.equal(hn, hn2)), "two calls differ"
    del y2, hn2
    ref = F.linear(x.double(), w.double(), None if b is None else b.double())
    with _true_fp32():
        f32 = F.linear(x, w, b)
    if kind == "gelu":
        ref, f32 = F.gelu(ref), F.gelu(f32)
    if kind == "res+ln":
        ref, f32 = ref + res.double(), f32 + res
    bound = 3e-6 * max(1.0, math.sqrt(k / 256))
    err, floor = _rel(y, ref), _rel(f32, ref)
    msg = f"{name}: rows {rows} split-K {plan['splitk']} {plan['tiles_per_cta']} tiles/CTA; |y - fp64| {err:.2e} (bound {bound:.1e}, fp32 {floor:.2e})"
    assert err <= bound, msg
    if hn is not None:
        ref_ln = F.layer_norm(ref, (n,), ln.weight.double(), ln.bias.double(), ln.eps)
        err_ln, floor_ln = _rel(hn, ref_ln), _rel(F.layer_norm(f32, (n,), ln.weight, ln.bias, ln.eps), ref_ln)
        msg += f"; |LN(y) - fp64| {err_ln:.2e} (bound {4 / 3 * bound:.1e}, fp32 {floor_ln:.2e}); LN pass SPLITS {plan['reduce_splits']} x{plan['reduce_passes']}"
        assert err_ln <= 4 / 3 * bound, msg
    del ref, f32
    if rows >= 16384 and plan["splitk"] == 1:
        # tile independence: a tile's arithmetic does not depend on the CTA or the loop iteration that computed it
        m = _first_unsplit_rows(k, n, kind, sms)
        assert lin_plan(m, k, n, sms, ln=kind == "res+ln")["splitk"] == 1
        small = _dense_op(kind, w, b, m)
        for sl in (slice(0, m), slice(rows - m, rows)):
            ys, hs = _dense_call(kind, small, x[sl].contiguous(), w, res[sl].contiguous(), ln)
            assert torch.equal(ys, y[sl]), f"{name}: rows {sl} differ from a {m}-row call"
            assert hs is None or torch.equal(hs, hn[sl]), f"{name}: LN rows {sl} differ from a {m}-row call"
        msg += f"; first / last {m} rows bit-equal to a {m}-row call"
    print(msg)


# ---------------------------------------------------------------- attention at the batches
def _encode_ref(q, k, v, b, t, lens, temp):
    qq = q.double().view(b, t, HEADS, 64).transpose(1, 2) / temp
    kk = k.double().view(b, t, HEADS, 64).transpose(1, 2)
    vv = v.double().view(b, t, HEADS, 64).transpose(1, 2)
    a = torch.matmul(qq, kk.transpose(2, 3))
    a = a.masked_fill(torch.arange(t, device=DEV)[None, None, None, :] >= lens.view(b, 1, 1, 1).long(), float("-inf"))
    return torch.matmul(torch.softmax(a, -1), vv).transpose(1, 2).reshape(b * t, HEADS * 64)


def _decode_ref(q, k, v, limit, temp):
    """q [b, heads*64], head-major k / v [b, heads, cap, 64]; keys t < limit (int or [b] tensor)."""
    b, h, cap, _ = k.shape
    a = torch.matmul(q.double().view(b, h, 1, 64) / temp, k.double().transpose(2, 3))
    lim = limit.view(b, 1, 1, 1) if torch.is_tensor(limit) else limit
    a = a.masked_fill(torch.arange(cap, device=DEV)[None, None, None, :] >= lim, float("-inf"))
    return torch.matmul(torch.softmax(a, -1), v.double()).reshape(b, h * 64)


def _lens(n, g, cap):
    lens = torch.randint(1, cap + 1, (n,), device=DEV, generator=g).int()
    lens[0], lens[1], lens[-2], lens[-1] = 1, cap, cap, 1
    return lens


def test_attn_encode_at_1024(native_lib):
    n, t = 1024, T_SRC
    g = torch.Generator(device=DEV).manual_seed(1024)
    fused = torch.randn((n * t, 3 * D), device=DEV, generator=g)
    q, k, v = fused[:, :D], fused[:, D:2 * D], fused[:, 2 * D:]
    lens = _lens(n, g, t)
    out = TF.attn_encode(q, k, v, HEADS, t, 8.0, kv_lens=lens)
    ref = _encode_ref(q, k, v, n, t, lens, 8.0)
    err = float((out.double() - ref).abs().max())
    bound = 2e-6 * max(1.0, float(ref.abs().max()))
    print(f"attn_encode n=1024 T=64: |out - fp64| {err:.2e} (bound {bound:.1e})")
    assert err <= bound
    for lo in (0, n - 8):
        rows = slice(lo * t, (lo + 8) * t)
        small = TF.attn_encode(q[rows], k[rows], v[rows], HEADS, t, 8.0, kv_lens=lens[lo:lo + 8].contiguous())
        assert torch.equal(small, out[rows]), lo


def test_attn_decode_at_1024(native_lib):
    n = 1024
    g = torch.Generator(device=DEV).manual_seed(2048)
    # the head-major encoder memory: capacity 64, per-image lengths
    q = torch.randn((n, D), device=DEV, generator=g)
    k = torch.randn((n, HEADS, T_SRC, 64), device=DEV, generator=g)
    v = torch.randn_like(k)
    lens = _lens(n, g, T_SRC)
    assert attn_decode_plan(n, HEADS, T_SRC) == "attn_decode_kernel<true>" and attn_decode_plan(8, HEADS, T_SRC).endswith("<false>")
    out = TF.attn_decode(q, k, v, HEADS, T_SRC, 8.0, kv_lens=lens, head_major=True)
    ref = _decode_ref(q, k, v, lens, 8.0)
    err, bound = float((out.double() - ref).abs().max()), 2e-6 * max(1.0, float(ref.abs().max()))
    print(f"attn_decode memory n=1024: |out - fp64| {err:.2e} (bound {bound:.1e})")
    assert err <= bound
    for lo in (0, n - 8):
        small = TF.attn_decode(q[lo:lo + 8], k[lo:lo + 8], v[lo:lo + 8], HEADS, T_SRC, 8.0, kv_lens=lens[lo:lo + 8].contiguous(), head_major=True)
        assert torch.equal(small, out[lo:lo + 8]), lo
    # the append form of the self-attention cache at its last step: capacity 40, kv_len 40, q | k_new | v_new one projection
    cap = 40
    fused = torch.randn((n, 3 * D), device=DEV, generator=g)
    kc0 = torch.randn((n, HEADS, cap, 64), device=DEV, generator=g)
    vc0 = torch.randn_like(kc0)
    assert attn_decode_plan(n, HEADS, cap) == "attn_decode_kernel<true>" and attn_decode_plan(8, HEADS, cap).endswith("<false>")
    kc, vc = kc0.clone(), vc0.clone()
    out = TF.attn_decode(fused[:, :D], kc, vc, HEADS, cap, 8.0, k_new=fused[:, D:2 * D], v_new=fused[:, 2 * D:], head_major=True)
    k2, v2 = kc0.clone(), vc0.clone()
    k2[:, :, cap - 1] = fused[:, D:2 * D].reshape(n, HEADS, 64)
    v2[:, :, cap - 1] = fused[:, 2 * D:].reshape(n, HEADS, 64)
    assert torch.equal(kc, k2) and torch.equal(vc, v2)                  # the appended rows are exact, nothing else written
    ref = _decode_ref(fused[:, :D], k2, v2, cap, 8.0)
    err, bound = float((out.double() - ref).abs().max()), 2e-6 * max(1.0, float(ref.abs().max()))
    print(f"attn_decode append n=1024 kv_len 40: |out - fp64| {err:.2e} (bound {bound:.1e})")
    assert err <= bound
    for lo in (0, n - 8):
        ks, vs = kc0[lo:lo + 8].clone(), vc0[lo:lo + 8].clone()
        f = fused[lo:lo + 8]
        small = TF.attn_decode(f[:, :D], ks, vs, HEADS, cap, 8.0, k_new=f[:, D:2 * D], v_new=f[:, 2 * D:], head_major=True)
        assert torch.equal(small, out[lo:lo + 8]), lo                   # the cache hint changes no bit
        assert torch.equal(ks, k2[lo:lo + 8]) and torch.equal(vs, v2[lo:lo + 8])


# ---------------------------------------------------------------- whole encoder and decoder at batch
def _ratios(n, seed):
    g = torch.Generator().manual_seed(seed)
    r = (0.02 + 0.98 * torch.rand(n, generator=g)).tolist()
    r[0], r[-1] = 1.0, 1.0 / 64
    return r


# From n = 75 images on 148 SMs every dense layer of the encoder is unsplit: one tcgen05 accumulation chain over all of K = 512
# instead of four chains of 128 summed in fp32.  Per layer that is 1.5-2.5x the error of an fp32 GEMM (test_dense_layer_vs_fp64
# above, within the dense-layer bound of 3e-6 x sqrt(K / 256), which allows 6x at K = 512), where the split calls of the small
# batches stay at or below 1x; the 4x-the-floor rule of test_nrtr_encoder_full_config_vs_twin (n = 3, all split) lands at 4.0x
# here.  The bound carries the dense-layer allowance over to the six layers.
ENCODER_AT_BATCH_FACTOR = 6


@pytest.mark.parametrize("n", [96, 256, 1024])
def test_encoder_at_batch_vs_fp64(native_lib, n):
    torch.manual_seed(0)
    enc = NRTREncoder().eval()
    sd = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    enc = enc.to(DEV)
    feat = torch.randn((n, D, 4, 16), device=DEV, generator=torch.Generator(device=DEV).manual_seed(n))
    ratios = _ratios(n, n)
    metas = [dict(valid_ratio=r) for r in ratios]
    with torch.no_grad():
        out = enc(feat, metas)
        assert enc.last_forward_native
        with _true_fp32():
            lib = enc.forward_library(feat, metas)
    ref = nrtr_encoder_forward(sd, feat, ratios, n_head=HEADS, dtype=torch.float64, device=DEV)
    assert out.shape == ref.shape == (n, T_SRC, D)
    err, floor = float((out.double() - ref).abs().max()), float((lib.double() - ref).abs().max())
    print(f"NRTREncoder n={n} ({encoder_rows(n)} rows): |native - fp64| {err:.3e} = {err / floor:.2f} x the fp32 floor {floor:.3e} "
          f"(bound {ENCODER_AT_BATCH_FACTOR} x)")
    assert err <= ENCODER_AT_BATCH_FACTOR * floor, (err, floor)


def _decoder():
    torch.manual_seed(0)
    dec = NRTRDecoder(start_idx=START, padding_idx=PAD).eval()
    with torch.no_grad():
        dec.classifier.weight.mul_(8.0)
    return dec.to(DEV)


@pytest.mark.parametrize("n", [44, 256, 1024])
def test_decoder_at_batch_vs_fp64_teacher_forced(native_lib, n):
    dec = _decoder()
    out_enc = torch.randn((n, T_SRC, D), device=DEV, generator=torch.Generator(device=DEV).manual_seed(n + 1))
    metas = [dict(valid_ratio=r) for r in _ratios(n, n + 1)]
    with torch.no_grad():
        probs = dec(None, out_enc, None, metas, train_mode=False)
        assert dec.last_test_native and probs.shape == (n, 40, 92)
        if n in (44, 1024):
            dec.decode_graph = False
            assert torch.equal(dec(None, out_enc, None, metas, train_mode=False), probs), "graph replay differs from the launches"
            dec.decode_graph = True
        # the native decode's own tokens, teacher-forced: step t sees tokens 0..t, so the greedy decode cannot flip a near-tie
        seq = torch.cat([torch.full((n, 1), START, dtype=torch.long, device=DEV), probs[:, :-1].argmax(-1)], 1)
        mask = dec._get_mask(out_enc, metas)
        dec64 = _decoder().double()                       # the same seeded weights (a decoder holding graphs does not deep-copy)
        p64 = F.softmax(dec64.classifier(dec64._attention(seq, out_enc.double(), mask.double())), -1)
        del dec64
        with _true_fp32():
            p32 = F.softmax(dec.classifier(dec._attention(seq, out_enc, mask)), -1)
    err, floor = float((probs.double() - p64).abs().max()), float((p32.double() - p64).abs().max())
    top2 = p64.topk(2, dim=-1).values
    sure = (top2[..., 0] - top2[..., 1]) >= 1e-3
    agree = bool((probs.argmax(-1) == p64.argmax(-1))[sure].all())
    print(f"NRTRDecoder n={n}: |probs - fp64| {err:.3e}, bound 4 x fp32 floor {floor:.3e}; arg-max equal on all "
          f"{int(sure.sum())} of {sure.numel()} steps with an fp64 margin >= 1e-3: {agree}")
    assert err <= 4 * floor, (err, floor)
    assert agree


# ---------------------------------------------------------------- repeatability of simple_test, stage by stage
NATIVE_STAGES = ["stage.o0", "stage.o1", "stage.x", "TPS_PP.output", "encoder", "decoder"]
LIBRARY_STAGES = ["layer3", "layer4", "layer5"]
ORDER = ["stage.o0", "stage.o1", "stage.x", "TPS_PP.output", "layer3", "layer4", "layer5", "encoder", "decoder"]


def _traced(model, img, metas):
    """simple_test with every stage's output recorded -> (outputs by stage, results)."""
    rec = {}
    bb = model.backbone
    stage = bb.stage

    def traced_stage(x):
        x2, outs = stage(x)
        rec["stage.o0"], rec["stage.o1"], rec["stage.x"] = outs[0].clone(), outs[1].clone(), x2.clone()
        return x2, outs

    def hook(name, pick=lambda o: o):
        return lambda mod, inp, out: rec.__setitem__(name, pick(out).clone())
    handles = [model.tpsnet.register_forward_hook(hook("TPS_PP.output", lambda o: o["output"])),
               model.encoder.register_forward_hook(hook("encoder")), model.decoder.register_forward_hook(hook("decoder"))]
    handles += [getattr(bb, nm).register_forward_hook(hook(nm)) for nm in LIBRARY_STAGES]
    bb.stage = traced_stage
    try:
        with torch.no_grad():
            res = model.simple_test(img, metas)
    finally:
        del bb.stage
        for h in handles:
            h.remove()
    return rec, res


def _compare(a, b, what):
    differ = [k for k in ORDER if not torch.equal(a[k], b[k])]
    print(f"simple_test {what}: stages that differ {differ or 'none'}")
    return differ


def test_simple_test_is_repeatable_stage_by_stage(native_lib):
    kw = ref_kw(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
    model = _recognizer(rotating_config(kw, [0, 90, 180, 270]))
    imgs = crops(12, seed=5)
    tall = next(im for im in imgs[6:] if im.shape[0] > im.shape[1])
    out, metas = model.test_pipeline([tall])             # the four rotations of one tall crop: the reported 4-row case
    four, four_metas = out.clone(), list(metas[0])
    assert four.shape[0] == 4
    big = torch.from_numpy(O.synthetic_images(256, seed=12)).to(DEV)
    big_metas = [dict(valid_ratio=r) for r in _ratios(256, 3)]
    mid = big[:96].clone()
    first, res1 = _traced(model, four, four_metas)
    second, res2 = _traced(model, four, four_metas)
    b1, bres1 = _traced(model, big, big_metas)
    b2, bres2 = _traced(model, big, big_metas)
    _traced(model, mid, big_metas[:96])
    third, res3 = _traced(model, four, four_metas)
    found = {"n=4, twice": (_compare(first, second, "n=4, twice"), res1 == res2),
             "n=256, twice": (_compare(b1, b2, "n=256, twice"), bres1 == bres2),
             "n=4 -> 96 -> 4": (_compare(first, third, "n=4 -> 96 -> 4"), res1 == res3)}
    assert all(not differ and same for differ, same in found.values()), found
