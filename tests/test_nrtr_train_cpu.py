"""CPU: the C layout of tpspp_attn_train_cfg, AttnConvertor.str2tensor and TFLoss on hand-written cases, and the argument checks
of the NRTR training path that run before any device work."""
import ctypes
import os
import shutil
import subprocess

import pytest
import torch
import torch.nn.functional as F

import tps_pp_b200 as T
from tps_pp_b200 import _native, nrtr_train

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_attn_train_cfg_has_the_header_layout(tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    mirror = _native.AttnTrainCfg
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "tpspp.h"', "int main(void) {",
             '  printf("%zu", sizeof(tpspp_attn_train_cfg));']
    lines += [f'  printf(" %zu", offsetof(tpspp_attn_train_cfg, {f}));' for f, _ in mirror._fields_]
    lines += ['  printf("\\n");', "  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    vals = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == ctypes.sizeof(mirror)
    assert vals[1:] == [getattr(mirror, f).offset for f, _ in mirror._fields_]
    assert [f for f, _ in mirror._fields_] == ["batch", "heads", "head_dim", "len_q", "len_k", "temperature", "causal", "dropout_p",
                                               "q_stride", "kv_stride"]


def test_str2tensor_hand_cases():
    conv = T.AttnConvertor("DICT90", with_unknown=True, max_seq_len=40)
    s, e, pad, ukn = conv.start_idx, conv.end_idx, conv.padding_idx, conv.unknown_idx
    assert (s, e, pad, ukn) == (91, 91, 92, 90)
    out = conv.str2tensor(["aB1", "aé"])
    assert [t.tolist() for t in out["targets"]] == [[10, 37, 1], [10, ukn]]
    pt = out["padded_targets"]
    assert pt.dtype == torch.long and pt.shape == (2, 40)
    assert pt[0].tolist() == [s, 10, 37, 1, e] + [pad] * 35
    assert pt[1].tolist() == [s, 10, ukn, e] + [pad] * 36
    # exactly 38 characters fill the 40 slots with start and end; more are cut at 40 (the end token is lost)
    full = conv.str2tensor(["0123456789" * 3 + "abcdefgh"])["padded_targets"][0].tolist()
    assert full == [s] + [conv.char2idx[c] for c in "0123456789" * 3 + "abcdefgh"] + [e]
    long = conv.str2tensor(["z" * 45])["padded_targets"][0].tolist()
    assert long == [s] + [35] * 39
    # lower-casing, and a dictionary without <UKN>
    low = T.AttnConvertor("DICT36", with_unknown=False, lower=True, max_seq_len=8)
    assert low.str2idx(["AbZ"]) == [[10, 11, 35]]
    assert low.str2tensor(["AB"])["padded_targets"].tolist() == [[36, 10, 11, 36, 37, 37, 37, 37]]
    with pytest.raises(ValueError):
        low.str2idx(["a-b"])
    assert T.AttnConvertor("DICT36", with_unknown=True).str2idx(["a-b"]) == [[10, 36, 11]]
    with pytest.raises(TypeError):
        conv.str2tensor("abc")


def test_tfloss_matches_a_hand_computation():
    pad = 4
    loss = T.build_loss(dict(type="TFLoss", ignore_index=pad))
    assert isinstance(loss, T.TFLoss) and "TFLoss" in T.LOSSES.module_dict
    logits = torch.tensor([[[2.0, 0.0, 0.0, 1.0], [0.0, 3.0, 0.0, 0.0], [1.0, 1.0, 1.0, 1.0]],
                           [[0.5, 0.0, 0.0, 0.0], [0.0, 0.0, 0.0, 0.0], [9.0, 9.0, 9.0, 9.0]]])
    targets = torch.tensor([[3, 0, 1], [3, 2, pad]])
    out = loss(logits, dict(padded_targets=targets))["loss_ce"]
    # step t predicts target t + 1; the last step has no target; the padding target contributes 0
    want = [-F.log_softmax(logits[0, 0], 0)[0], -F.log_softmax(logits[0, 1], 0)[1], -F.log_softmax(logits[1, 0], 0)[2], 0.0]
    assert out.shape == (4,)
    assert torch.allclose(out, torch.tensor([float(w) for w in want]), atol=1e-6)


def _rec(**kw):
    return T.build_recognizer(dict(
        type="NRTR",
        backbone=dict(type="ResNetABI_v2_large", arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]),
        tpsnet=dict(type="TPS_PP"),
        encoder=dict(type="NRTREncoder"),
        decoder=dict(type="NRTRDecoder"),
        label_convertor=dict(type="AttnConvertor", dict_type="DICT90", with_unknown=True, max_seq_len=40), **kw))


def test_forward_train_argument_errors():
    rec = _rec()
    # a missing loss config is TFLoss over the padding index
    assert isinstance(rec.loss, T.TFLoss) and rec.loss.loss_ce.ignore_index == rec.label_convertor.padding_idx
    img = torch.zeros((2, 3, 32, 128))
    with pytest.raises(RuntimeError, match="mmocr"):
        rec.forward_train(img, None)
    with pytest.raises(RuntimeError, match="text"):
        rec(img, [dict(text="ab"), dict(valid_ratio=1.0)], return_loss=True)
    with pytest.raises(ValueError):
        rec.forward_train(img, [dict(text="ab")])
    rec = _rec(loss=dict(type="TFLoss", ignore_index=0))
    assert rec.loss.loss_ce.ignore_index == rec.label_convertor.padding_idx


def test_decoder_train_rejects_pads_that_are_not_a_suffix():
    dec = T.NRTRDecoder(n_layers=1, d_embedding=128, n_head=2, d_model=128, d_inner=64, num_classes=8, padding_idx=7, max_seq_len=5)
    assert nrtr_train.target_lengths(torch.tensor([[6, 1, 2, 7, 7], [6, 1, 2, 3, 4], [6, 7, 7, 7, 7]]), 7) == [3, 5, 1]
    bad = torch.tensor([[6, 1, 2, 7, 7], [6, 7, 2, 6, 7]])
    with pytest.raises(ValueError, match="suffix"):
        nrtr_train.decoder_train(dec, bad, torch.zeros((2, 4, 128)))


def test_fused_source_keeps_a_grad_leaf_slice_apart():
    from tps_pp_b200.functional import _fused_source
    base = torch.randn((6, 384), requires_grad=True)
    q = base[:, 128:256]
    assert _fused_source(q)[0] is base and _fused_source(q)[1] == 128
    plain = torch.randn((6, 384))
    leaf = plain[:, 128:256].requires_grad_()          # a slice made a leaf: its gradient must not go to the base
    src, off = _fused_source(leaf)
    assert src is leaf and off == 0
