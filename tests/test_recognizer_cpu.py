"""CPU: the label convertor against the reference recogniser's own strings, registry construction of the encoder / convertor /
recogniser, the encoder's library path against the restatement, and the C layout of tpspp_attn_encode_cfg."""
import ctypes
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

import tps_pp_b200 as T
from tps_pp_b200 import _native

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the restatement beside these tests
from nrtr_encoder_restatement import nrtr_encoder_forward  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_attn_convertor_reproduces_the_reference_strings(golden):
    """nrtr_argmax.npz stores the reference recogniser's per-step arg-maxes and the strings its AttnConvertor made of them."""
    g = golden("nrtr_argmax.npz")
    conv = T.AttnConvertor("DICT90", with_unknown=True)
    assert (conv.num_classes(), conv.start_idx, conv.end_idx, conv.padding_idx, conv.unknown_idx) == (93, 91, 91, 92, 90)
    for tag in ("stock", "trained"):
        ids = torch.from_numpy(g[f"{tag}_ref_argmax"].astype(np.int64))
        probs = torch.nn.functional.one_hot(ids, 92).float()          # the decoder never predicts the padding class
        idx, scores = conv.tensor2idx(probs)
        assert conv.idx2str(idx) == list(g[f"{tag}_strings"])
        assert all(s == [1.0] * len(i) for i, s in zip(idx, scores))


def test_attn_convertor_skips_padding_and_stops_at_end():
    conv = T.AttnConvertor("DICT36", with_unknown=False)
    assert conv.num_classes() == 38 and conv.start_idx == conv.end_idx == 36 and conv.padding_idx == 37
    ids = torch.tensor([[10, 37, 11, 36, 12], [37, 0, 1, 2, 3]])
    probs = torch.nn.functional.one_hot(ids, 38).float() * 0.5
    idx, scores = conv.tensor2idx(probs)
    assert conv.idx2str(idx) == ["ab", "0123"] and scores == [[0.5, 0.5], [0.5] * 4]
    with pytest.raises(ValueError):
        T.AttnConvertor("DICT91")


def test_registry_builds_encoder_convertor_and_recognizer():
    torch.manual_seed(0)
    enc = T.build_encoder(dict(type="NRTREncoder"))
    assert isinstance(enc, T.NRTREncoder)
    assert sum(p.numel() for p in enc.parameters()) == 7_882_240
    per_layer = ["attn.linear_q.weight", "attn.linear_k.weight", "attn.linear_v.weight", "attn.fc.weight", "norm1.weight",
                 "norm1.bias", "mlp.w_1.weight", "mlp.w_1.bias", "mlp.w_2.weight", "mlp.w_2.bias", "norm2.weight", "norm2.bias"]
    keys = [f"layer_stack.{i}.{k}" for i in range(6) for k in per_layer] + ["layer_norm.weight", "layer_norm.bias"]
    assert list(enc.state_dict()) == keys
    assert isinstance(T.build_convertor(dict(type="AttnConvertor", dict_type="DICT90")), T.AttnConvertor)
    with pytest.raises(TypeError):
        T.NRTREncoder(no_such_kwarg=1)
    with pytest.raises(ValueError):
        T.NRTREncoder(operation_order=("self_attn", "norm", "ffn", "norm"))
    with pytest.raises(ValueError):
        T.NRTREncoder(act_cfg=dict(type="ReLU"))
    T.NRTREncoder(n_layers=1, operation_order=("norm", "self_attn", "norm", "ffn"), act_cfg=dict(type="mmcv.GELU"))
    rec = T.build_recognizer(dict(
        type="NRTR",
        backbone=dict(type="ResNetABI_v2_large", arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]),
        tpsnet=dict(type="TPS_PP"),
        encoder=dict(type="NRTREncoder"),
        decoder=dict(type="NRTRDecoder"),
        label_convertor=dict(type="AttnConvertor", dict_type="DICT90", with_unknown=True, max_seq_len=40)))
    assert isinstance(rec, T.NRTR) and isinstance(rec.tpsnet, T.TPS_PP) and isinstance(rec.encoder, T.NRTREncoder)
    # the decoder config is completed from the convertor, as EncodeDecodeRecognizer does
    assert rec.decoder.classifier.out_features == 92 and rec.decoder.padding_idx == 92 and rec.decoder.start_idx == 91
    prefixes = {k.split(".")[0] for k in rec.state_dict()}
    assert prefixes == {"backbone", "tpsnet", "encoder", "decoder"}
    rec.load_state_dict(rec.state_dict(), strict=True)
    with pytest.raises(RuntimeError, match="mmocr"):
        rec(torch.zeros((1, 3, 32, 128)), None, return_loss=True)


@pytest.mark.parametrize("cfg", [dict(), dict(n_layers=2, d_model=128, n_head=2, d_inner=64)])
def test_encoder_library_path_matches_the_restatement(cfg):
    torch.manual_seed(1)
    enc = T.NRTREncoder(**cfg).double().eval()
    sd = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    d = enc.d_model
    feat = torch.randn((3, d, 4, 16), generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    ratios = [1.0, 0.5, 0.75]
    metas = [dict(valid_ratio=r) for r in ratios]
    with torch.no_grad():
        out = enc.forward_library(feat, metas)
    ref = nrtr_encoder_forward(sd, feat, ratios, n_head=enc.n_head, dtype=torch.float64)
    assert out.shape == (3, 64, d)
    assert float((out - ref).abs().max()) <= 1e-5
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        enc(feat, metas)


def test_encoder_library_path_gives_nan_rows_for_an_empty_image():
    torch.manual_seed(1)
    enc = T.NRTREncoder(n_layers=1, d_model=128, n_head=2, d_inner=64).eval()
    feat = torch.randn((2, 128, 2, 8))
    with torch.no_grad():
        out = enc.forward_library(feat, [dict(valid_ratio=1.0), dict(valid_ratio=0.0)])
    assert torch.isfinite(out[0]).all() and torch.isnan(out[1]).all()


def test_valid_lengths_is_the_decoder_mask():
    from tps_pp_b200.nrtr import valid_lengths
    assert valid_lengths(64, None) is None
    assert valid_lengths(64, [dict(valid_ratio=1.0), dict(valid_ratio=0.5), dict(valid_ratio=0.01), dict(), dict(valid_ratio=2.0)]) == \
        [64, 32, 1, 64, 64]
    mask = T.NRTRDecoder._get_mask(torch.zeros((2, 24, 8)), [dict(valid_ratio=0.75), dict(valid_ratio=0.3)])
    assert mask.sum(1).tolist() == [18.0, 8.0]


def test_attn_encode_cfg_has_the_header_layout(tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    mirror = _native.AttnEncodeCfg
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "tpspp.h"', "int main(void) {",
             '  printf("%zu", sizeof(tpspp_attn_encode_cfg));']
    lines += [f'  printf(" %zu", offsetof(tpspp_attn_encode_cfg, {f}));' for f, _ in mirror._fields_]
    lines += ['  printf("\\n");', "  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    vals = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert vals[0] == ctypes.sizeof(mirror)
    assert vals[1:] == [getattr(mirror, f).offset for f, _ in mirror._fields_]
    assert [f for f, _ in mirror._fields_] == ["batch", "heads", "head_dim", "seq_len", "temperature", "row_stride"]
