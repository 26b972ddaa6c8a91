"""GPU: tpspp_attn_encode against fp64 torch, the native NRTREncoder against the restatement's fp64 twin, its dispatch, and
the NRTR recogniser's fully native chain (image -> stage -> TPS_PP -> layer3-5 -> encoder -> decode -> strings) against the
fully library chain."""
import os
import sys

import numpy as np
import pytest
import torch

import tps_pp_b200 as T
from oracle import tpspp_oracle as O
from tps_pp_b200 import functional as TF

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the restatement beside these tests
from nrtr_encoder_restatement import nrtr_encoder_forward  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _attn_ref(q, k, v, b, heads, t, lens, temp):
    qq = q.double().view(b, t, heads, 64).transpose(1, 2) / temp
    kk = k.double().view(b, t, heads, 64).transpose(1, 2)
    vv = v.double().view(b, t, heads, 64).transpose(1, 2)
    a = torch.matmul(qq, kk.transpose(2, 3))
    if lens is not None:
        a = a.masked_fill(torch.arange(t, device=q.device)[None, None, None, :] >= lens.view(b, 1, 1, 1).long(), float("-inf"))
    return torch.matmul(torch.softmax(a, -1), vv).transpose(1, 2).reshape(b * t, heads * 64)


@pytest.mark.parametrize("b,heads,t", [(3, 2, 20), (7, 8, 64), (260, 8, 64), (2, 8, 256), (5, 8, 1), (4, 8, 33)])
def test_attn_encode_vs_torch(native_lib, b, heads, t):
    g = torch.Generator(device=DEV).manual_seed(b * 1000 + t)
    d = heads * 64
    fused = torch.randn((b * t, 3 * d), device=DEV, generator=g)
    q, k, v = fused[:, :d], fused[:, d:2 * d], fused[:, 2 * d:]
    lens = torch.randint(1, t + 1, (b,), device=DEV, generator=g).int()
    lens[0] = 1
    for use_lens in (False, True):
        kl = lens if use_lens else None
        out = TF.attn_encode(q, k, v, heads, t, 8.0, kv_lens=kl)
        ref = _attn_ref(q, k, v, b, heads, t, kl, 8.0)
        err = float((out.double() - ref).abs().max())
        assert err <= 2e-6 * max(1.0, float(ref.abs().max())), err
        # contiguous inputs: the same arithmetic, bit for bit
        out_c = torch.empty_like(out)
        TF.attn_encode(q.contiguous(), k.contiguous(), v.contiguous(), heads, t, 8.0, kv_lens=kl, out=out_c)
        assert torch.equal(out_c, out)
    # a temperature that is not a power of two (q is divided by it, as in the reference)
    out = TF.attn_encode(q, k, v, heads, t, 3.0, kv_lens=lens)
    ref = _attn_ref(q, k, v, b, heads, t, lens, 3.0)
    assert float((out.double() - ref).abs().max()) <= 2e-6 * max(1.0, float(ref.abs().max()))


def test_attn_encode_checks_its_arguments(native_lib):
    d = 128
    x = torch.randn((2 * 8, 3 * d), device=DEV)
    q, k, v = x[:, :d], x[:, d:2 * d], x[:, 2 * d:]
    with pytest.raises(RuntimeError, match="out"):
        TF.attn_encode(q, k, v, 2, 8, 8.0, out=torch.empty((16, d), device=DEV).t().contiguous().t())
    with pytest.raises(RuntimeError, match="out"):
        TF.attn_encode(q, k, v, 2, 8, 8.0, out=torch.empty((16, d), device=DEV, dtype=torch.float64))
    with pytest.raises(RuntimeError, match="out"):
        TF.attn_encode(q, k, v, 2, 8, 8.0, out=torch.empty((15, d), device=DEV))
    with pytest.raises(RuntimeError, match="out"):
        TF.attn_encode(q, k, v, 2, 8, 8.0, out=torch.empty((16, d)))
    with pytest.raises(RuntimeError, match="row stride"):
        TF.attn_encode(q, k.contiguous(), v, 2, 8, 8.0)
    with pytest.raises(RuntimeError, match="kv_lens"):
        TF.attn_encode(q, k, v, 2, 8, 8.0, kv_lens=torch.ones(2, dtype=torch.int64, device=DEV))
    with pytest.raises(RuntimeError):
        TF.attn_encode(q, k, v, 2, 5, 8.0)                           # 16 rows are not whole images of 5 tokens
    with pytest.raises(RuntimeError):
        TF.attn_encode(q.cpu(), k.cpu(), v.cpu(), 2, 8, 8.0)


def _encoder_vs_twin(cfg, shape, ratios, seed=0):
    torch.manual_seed(seed)
    enc = T.NRTREncoder(**cfg).eval()
    sd = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    feat = torch.randn(shape, generator=torch.Generator().manual_seed(seed + 1))
    metas = [dict(valid_ratio=r) for r in ratios]
    ref = nrtr_encoder_forward(sd, feat, ratios, n_head=enc.n_head, dtype=torch.float64)
    enc = enc.to(DEV)
    with torch.no_grad():
        out = enc(feat.to(DEV), metas)
        assert enc.last_forward_native
        lib = enc.forward_library(feat.to(DEV), metas)
    err = float((out.cpu().double() - ref).abs().max())
    floor = float((lib.cpu().double() - ref).abs().max())
    print(f"NRTREncoder {cfg or 'full'} {tuple(shape)}: |native - fp64| = {err:.3e}, |library fp32 - fp64| = {floor:.3e}")
    assert out.shape == ref.shape
    assert err <= 4 * floor, (err, floor)


def test_nrtr_encoder_full_config_vs_twin(native_lib):
    """nrtr_tps++.py's encoder (6 layers, 512 wide, 8 heads) on a 32x128 image's 4x16 feature map; every position compared,
    the padded ones (i >= valid length) included.  B*T = 192 is not a multiple of 128."""
    _encoder_vs_twin({}, (3, 512, 4, 16), [1.0, 0.5, 0.75])


def test_nrtr_encoder_reduced_config_vs_twin(native_lib):
    _encoder_vs_twin(dict(n_layers=2, d_model=128, n_head=2, d_inner=64), (3, 128, 4, 16), [1.0, 0.5, 0.75], seed=4)
    _encoder_vs_twin(dict(n_layers=2, d_model=128, n_head=2, d_inner=64), (5, 128, 2, 9), [1.0, 0.3, 0.75, 0.05, 1.0], seed=6)


def test_nrtr_encoder_dispatch(native_lib):
    torch.manual_seed(0)
    enc = T.NRTREncoder(n_layers=2, d_model=128, n_head=2, d_inner=64).to(DEV).eval()
    feat = torch.randn((2, 128, 4, 16), device=DEV)
    metas = [dict(valid_ratio=1.0), dict(valid_ratio=0.5)]
    with torch.no_grad():
        enc(feat, metas)
    assert enc.last_forward_native is True
    # autograd recording: the library path, differentiable into every parameter
    out = enc(feat, metas)
    assert enc.last_forward_native is False and out.requires_grad
    (out * torch.randn_like(out)).sum().backward()
    for name, p in enc.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all() and p.grad.abs().max() > 0, name
    # an image with no valid key: the reference's NaN rows (library path), the other image unaffected
    with torch.no_grad():
        out = enc(feat, [dict(valid_ratio=1.0), dict(valid_ratio=0.0)])
        ok = enc(feat[:1], [dict(valid_ratio=1.0)])
    assert enc.last_forward_native is True
    assert torch.isnan(out[1]).all() and torch.isfinite(out[0]).all()
    assert float((out[0] - ok[0]).abs().max()) <= 1e-4
    enc.train()
    with torch.no_grad():
        enc(feat, metas)
    assert enc.last_forward_native is False


def _recognizer():
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
    return rec.to(DEV).eval()


def test_nrtr_recognizer_native_chain_vs_library_chain(native_lib):
    rec = _recognizer()
    img = torch.from_numpy(O.synthetic_images(8, seed=11)).to(DEV)
    metas = [dict(valid_ratio=r) for r in (1.0, 0.5, 0.75, 1.0, 0.25, 1.0, 0.9, 0.6)]
    tf32 = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False   # library chain in plain fp32
    try:
        with torch.no_grad():
            feat = rec.extract_feat(img)
            assert rec.backbone._last_stage_native and all(rec.tpsnet.native_stages.values())
            out_enc = rec.encoder(feat, metas)
            assert rec.encoder.last_forward_native
            probs = rec.decoder(feat, out_enc, None, metas, train_mode=False)
            assert rec.decoder.last_test_native
            results = rec.simple_test(img, metas)
            rec.backbone.stage_impl = "library"
            rec.tpsnet.head_impl = "library"
            feat_l = rec.extract_feat(img)
            assert not rec.backbone._last_stage_native
            probs_l = rec.decoder.forward_test_library(None, rec.encoder.forward_library(feat_l, metas), metas)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
        rec.backbone.stage_impl = rec.tpsnet.head_impl = "auto"
    conv = rec.label_convertor
    assert [r["text"] for r in results] == conv.idx2str(conv.tensor2idx(probs)[0])
    top2 = probs_l.topk(2, dim=-1).values
    margin = top2[..., 0] - top2[..., 1]
    compared = 0
    for i in range(probs.shape[0]):
        weak = (margin[i] < 1e-3).nonzero()
        upto = int(weak[0]) if len(weak) else probs.shape[1]
        compared += upto
        assert torch.equal(probs[i, :upto].argmax(-1), probs_l[i, :upto].argmax(-1)), i
    print(f"recogniser: native vs library chain, identical token ids on {compared} of {probs.shape[0] * probs.shape[1]} steps "
          f"(each image up to its first step with a top-1 margin < 1e-3); texts {[r['text'] for r in results[:2]]}")
    assert compared > 0


def test_nrtr_recognizer_batch_256(native_lib):
    rec = _recognizer()
    img = torch.from_numpy(O.synthetic_images(256, seed=12)).to(DEV)
    with torch.no_grad():
        results = rec(img, None, return_loss=False)
    assert len(results) == 256
    assert all(isinstance(r["text"], str) and len(r["score"]) <= 40 for r in results)
    assert rec.encoder.last_forward_native and rec.decoder.last_test_native
