"""GPU: the NRTR training path -- encoder_train / decoder_train against the modules' torch-ops paths on fp64 copies (outputs and every
parameter gradient), NRTR.forward_train end to end (loss, native flag, gradients into every backbone / tpsnet / encoder / decoder
parameter), reproducible dropout under torch.manual_seed, and a fixed batch that 30 Adam steps fit."""
import copy
import random

import pytest
import torch

import tps_pp_b200 as T
from oracle import tpspp_oracle as O
from tps_pp_b200 import nrtr_train
from tps_pp_b200.nrtr import valid_lengths
from tps_pp_b200.recognizer import DICT90

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RATIOS = [1.0, 0.5, 0.75, 0.25, 1.0, 0.9]


def _words(n, seed):
    rng = random.Random(seed)
    return ["".join(rng.choice(DICT90) for _ in range(rng.randint(5, 12))) for _ in range(n)]


@pytest.fixture
def no_tf32():
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


def _check_grads(mod, mod64, tol=1e-3):
    named64 = dict(mod64.named_parameters())
    for name, p in mod.named_parameters():
        g64 = named64[name].grad
        assert p.grad is not None and g64 is not None, name
        err = float((p.grad.double() - g64).abs().max())
        assert err <= tol * float(g64.abs().max()), (name, err, float(g64.abs().max()))


def test_encoder_train_matches_the_library_path(native_lib, no_tf32):
    torch.manual_seed(0)
    enc = T.NRTREncoder(dropout=0.0).to(DEV).train()
    enc64 = copy.deepcopy(enc).double()
    feat = torch.randn((6, 512, 4, 16), device=DEV, requires_grad=True)
    metas = [dict(valid_ratio=r) for r in RATIOS]
    out = nrtr_train.encoder_train(enc, feat, valid_lengths(64, metas))
    feat64 = feat.detach().double().requires_grad_()
    ref = enc64.forward_library(feat64, metas)
    assert out.shape == ref.shape == (6, 64, 512)
    assert float((out.double() - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
    gout = torch.randn(out.shape, device=DEV)
    out.backward(gout)
    ref.backward(gout.double())
    _check_grads(enc, enc64)
    assert float((feat.grad.double() - feat64.grad).abs().max()) <= 1e-3 * float(feat64.grad.abs().max())


def test_decoder_train_matches_the_library_path(native_lib, no_tf32):
    torch.manual_seed(1)
    conv = T.AttnConvertor("DICT90", with_unknown=True, max_seq_len=40)
    dec = T.NRTRDecoder(dropout=0.0, num_classes=conv.num_classes(), start_idx=conv.start_idx,
                        padding_idx=conv.padding_idx, max_seq_len=40).to(DEV).train()
    dec64 = copy.deepcopy(dec).double()
    words = _words(5, 2) + ["x" * 45]                  # the last one is truncated: no pad token at all
    targets = conv.str2tensor(words)
    out_enc = torch.randn((6, 64, 512), device=DEV, requires_grad=True)
    metas = [dict(valid_ratio=r) for r in RATIOS]
    out = nrtr_train.decoder_train(dec, targets["padded_targets"], out_enc, valid_lengths(64, metas))
    enc64 = out_enc.detach().double().requires_grad_()
    ref = dec64.forward_train(None, enc64, targets, metas)
    assert out.shape == ref.shape == (6, 40, 92)
    assert float((out.double() - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
    gout = torch.randn(out.shape, device=DEV)
    out.backward(gout)
    ref.backward(gout.double())
    _check_grads(dec, dec64)
    assert float((out_enc.grad.double() - enc64.grad).abs().max()) <= 1e-3 * float(enc64.grad.abs().max())


def _recognizer(seed=0):
    torch.manual_seed(seed)
    rec = T.build_recognizer(dict(
        type="NRTR",
        backbone=dict(type="ResNetABI_v2_large", arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]),
        tpsnet=dict(type="TPS_PP"),
        encoder=dict(type="NRTREncoder"),
        decoder=dict(type="NRTRDecoder"),
        loss=dict(type="TFLoss"),
        label_convertor=dict(type="AttnConvertor", dict_type="DICT90", with_unknown=True, max_seq_len=40)))
    rec.tpsnet.load_state_dict(O.trained_like_state(3), strict=True)      # no zero-initialised layer in the rectifier
    return rec.to(DEV).train()


def test_forward_train_reaches_every_parameter(native_lib):
    rec = _recognizer()
    img = torch.from_numpy(O.synthetic_images(8, seed=21)).to(DEV)
    metas = [dict(text=w, valid_ratio=r) for w, r in zip(_words(8, 3), RATIOS + [0.6, 1.0])]
    metas[1] = dict(text=metas[1]["text"], resize_shape=(32, 64, 3))       # valid ratio 64 / 128
    losses = rec(img, metas, return_loss=True)
    assert set(losses) == {"loss_ce"} and losses["loss_ce"].shape == (8 * 39,)
    loss = losses["loss_ce"].mean()
    assert torch.isfinite(loss) and rec.last_train_native is True
    loss.backward()
    bad = []
    for name, p in rec.named_parameters():
        g = p.grad
        if name == "decoder.trg_word_emb.weight":
            assert torch.equal(g[rec.decoder.padding_idx], torch.zeros_like(g[0]))
            g = torch.cat([g[:rec.decoder.padding_idx], g[rec.decoder.padding_idx + 1:]])
        if g is None or not torch.isfinite(g).all() or float(g.abs().max()) == 0.0:
            bad.append(name)
    assert not bad, bad
    assert {n.split(".")[0] for n, _ in rec.named_parameters()} == {"backbone", "tpsnet", "encoder", "decoder"}


def _enc_dec_step(enc, dec, conv, feat, words, lens):
    f = feat.detach().clone().requires_grad_()
    targets = conv.str2tensor(words)
    logits = nrtr_train.decoder_train(dec, targets["padded_targets"], nrtr_train.encoder_train(enc, f, lens), lens)
    loss = T.TFLoss(ignore_index=conv.padding_idx)(logits, targets)["loss_ce"].mean()
    enc.zero_grad(set_to_none=True)
    dec.zero_grad(set_to_none=True)
    loss.backward()
    return loss.detach(), [f.grad] + [p.grad for p in list(enc.parameters()) + list(dec.parameters())]


def test_dropout_step_is_reproducible_under_manual_seed(native_lib):
    torch.manual_seed(4)
    conv = T.AttnConvertor("DICT90", with_unknown=True, max_seq_len=40)
    enc = T.NRTREncoder(dropout=0.1).to(DEV).train()
    dec = T.NRTRDecoder(dropout=0.1, num_classes=conv.num_classes(), start_idx=conv.start_idx, padding_idx=conv.padding_idx,
                        max_seq_len=40).to(DEV).train()
    feat = torch.randn((6, 512, 4, 16), device=DEV)
    words = _words(6, 5)
    lens = valid_lengths(64, [dict(valid_ratio=r) for r in RATIOS])
    runs = []
    for seed in (11, 11, 12):
        torch.manual_seed(seed)
        runs.append(_enc_dec_step(enc, dec, conv, feat, words, lens))
    (l1, g1), (l2, g2), (l3, _) = runs
    assert torch.equal(l1, l2) and all(torch.equal(a, b) for a, b in zip(g1, g2))
    assert not torch.equal(l1, l3)                     # another seed drops other units


def test_adam_steps_fit_a_fixed_batch(native_lib):
    rec = _recognizer(seed=7)
    img = torch.from_numpy(O.synthetic_images(8, seed=22)).to(DEV)
    metas = [dict(text=w, valid_ratio=1.0) for w in _words(8, 9)]
    opt = torch.optim.Adam(rec.parameters(), lr=1e-4)
    losses = []
    for _ in range(30):
        opt.zero_grad(set_to_none=True)
        loss = rec(img, metas, return_loss=True)["loss_ce"].mean()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    print(f"30 Adam steps on a fixed batch of 8: loss {losses[0]:.3f} -> {losses[-1]:.3f}")
    assert all(x == x for x in losses) and losses[-1] < losses[0]
