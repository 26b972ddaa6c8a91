"""Training forward of the NRTR encoder and decoder on native kernels: teacher forcing over whole sequences, differentiable.

``encoder_train`` / ``decoder_train`` compute what ``NRTREncoder.forward_library`` and ``NRTRDecoder.forward_train`` compute, over
the same modules' parameters, with the reference's dropout (mmocr 0.4 common/modules/transformer_module.py: inside the attention on
the probabilities, ``proj_drop`` after each attention block's ``fc``, after ``w_2``; nrtr_decoder.py: after the embedding + position
sum), applied only when the module is in training mode, with ``p`` = the constructor's ``dropout``:

* dense layers: ``TF.linear`` (``tpspp_linear_fwd`` / ``_bwd``); q|k|v of a self-attention is one fused projection, k|v of the
  encoder memory one fused projection per decoder layer;
* attention: ``TF.attention`` (``tpspp_attn_train_fwd`` / ``_bwd``) with the key-length mask, the decoder's causal mask and the
  attention dropout; the gradients of the fused projections are written by its backward kernels;
* LayerNorm, GELU, the embedding, residual adds and the dropout outside the attention: torch ops.

These functions are the recogniser's training path (``NRTR.forward_train``); ``NRTREncoder.forward`` and
``NRTRDecoder.forward_train`` keep their torch-ops paths for training hosted by mmocr.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch
import torch.nn.functional as F

from . import functional as TF


def _check_heads(mod, name: str) -> None:
    if mod.d_k != 64 or mod.d_model != mod.n_head * 64:
        raise RuntimeError(f"tps_pp_b200: the native {name} training path needs d_k = d_v = 64 and d_model = n_head * 64")


def _drop(x: torch.Tensor, p: float) -> torch.Tensor:
    return F.dropout(x, p, training=True) if p > 0 else x


def _cat_linear(*lins):
    w = torch.cat([m.weight for m in lins], 0)
    return w, (None if lins[0].bias is None else torch.cat([m.bias for m in lins], 0))


def _self_attention(att, h: torch.Tensor, n_head: int, length: int, lens, causal: bool, p: float) -> torch.Tensor:
    """``proj_drop(fc(attention(h, h, h)))`` over [B*length, d] rows; q|k|v is one fused projection."""
    d = n_head * 64
    qkv = TF.linear(h, *_cat_linear(att.linear_q, att.linear_k, att.linear_v))
    o = TF.attention(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], n_head, length, length, 64 ** 0.5, kv_lens=lens, causal=causal,
                     dropout_p=p)
    return _drop(TF.linear(o, att.fc.weight, att.fc.bias), p)


def encoder_train(enc, feat: torch.Tensor, lens: Optional[Sequence[int]] = None) -> torch.Tensor:
    """``NRTREncoder`` (nrtr_encoder.py:66-87, pre-norm ``TFEncoderLayer``) on the native training kernels: feat [N, C, H, W] ->
    [N, H*W, C].  ``lens``: each image's valid source length (``nrtr.valid_lengths``), or None for all H*W."""
    _check_heads(enc, "NRTREncoder")
    n, c, h, w = feat.shape
    t = h * w
    p = float(enc.dropout) if enc.training else 0.0
    lens = TF.AttnLengths(lens, t, feat.device) if lens is not None else None      # checked and uploaded once for all layers
    x = feat.reshape(n, c, t).permute(0, 2, 1).reshape(n * t, c)
    for lyr in enc.layer_stack:
        x = x + _self_attention(lyr.attn, lyr.norm1(x), enc.n_head, t, lens, False, p)
        x = x + _drop(TF.linear(F.gelu(TF.linear(lyr.norm2(x), lyr.mlp.w_1.weight, lyr.mlp.w_1.bias)), lyr.mlp.w_2.weight,
                                lyr.mlp.w_2.bias), p)
    return enc.layer_norm(x).view(n, t, c)


def target_lengths(padded_targets: torch.Tensor, padding_idx: int) -> list:
    """Per row of ``padded_targets`` [N, L] its number of leading non-pad tokens.  The reference masks keys per token
    (``trg_seq != padding_idx``); that mask is a length only when the pad tokens of a row are a suffix, so other rows raise
    ``ValueError``."""
    tg = padded_targets.detach().cpu()
    if tg.dim() != 2:
        raise ValueError(f"tps_pp_b200: padded_targets must be [N, L], got {tuple(tg.shape)}")
    pad = tg == padding_idx
    lens = (~pad).long().cumprod(1).sum(1)
    tail = torch.arange(tg.shape[1])[None, :] >= lens[:, None]
    bad = (pad != tail).any(1).nonzero().flatten()
    if len(bad):
        raise ValueError(f"tps_pp_b200: row {int(bad[0])} of padded_targets has pad tokens ({padding_idx}) before other tokens: "
                         "the pad tokens of each row must be a suffix")
    return lens.tolist()


def decoder_train(dec, padded_targets: torch.Tensor, out_enc: torch.Tensor, src_lens: Optional[Sequence[int]] = None) -> torch.Tensor:
    """Teacher-forced ``NRTRDecoder.forward_train`` (nrtr_decoder.py:93-140) on the native training kernels: padded_targets
    [N, L] (``AttnConvertor.str2tensor``), out_enc [N, T, d] -> logits [N, L, num_classes - 1].  Per layer: causal self-attention
    over each row's target length, cross-attention over ``src_lens`` (or all T) source positions, the feed-forward block."""
    _check_heads(dec, "NRTRDecoder")
    tgt_lens = target_lengths(padded_targets, dec.padding_idx)
    n, L = padded_targets.shape
    _, t, d = out_enc.shape
    p = float(dec.dropout.p) if dec.training else 0.0
    tg = padded_targets.to(out_enc.device)
    tgt_lens = TF.AttnLengths(tgt_lens, L, out_enc.device)
    src_lens = TF.AttnLengths(src_lens, t, out_enc.device) if src_lens is not None else None
    x = dec.dropout(dec.trg_word_emb(tg) + dec.position_enc.position_table[:, :L]).reshape(n * L, d)
    mem = out_enc.reshape(n * t, d)
    for lyr in dec.layer_stack:
        x = x + _self_attention(lyr.self_attn, lyr.norm1(x), dec.n_head, L, tgt_lens, True, p)
        ea = lyr.enc_attn
        q = TF.linear(lyr.norm2(x), ea.linear_q.weight, ea.linear_q.bias)
        kv = TF.linear(mem, *_cat_linear(ea.linear_k, ea.linear_v))
        o = TF.attention(q, kv[:, :d], kv[:, d:], dec.n_head, L, t, 64 ** 0.5, kv_lens=src_lens, dropout_p=p)
        x = x + _drop(TF.linear(o, ea.fc.weight, ea.fc.bias), p)
        x = x + _drop(TF.linear(F.gelu(TF.linear(lyr.norm3(x), lyr.mlp.w_1.weight, lyr.mlp.w_1.bias)), lyr.mlp.w_2.weight,
                                lyr.mlp.w_2.bias), p)
    logits = TF.linear(dec.layer_norm(x), dec.classifier.weight, dec.classifier.bias)
    return logits.view(n, L, -1)
