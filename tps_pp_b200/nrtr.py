"""Drop-in ``NRTRDecoder`` (registry ``DECODERS``) and ``NRTREncoder`` (registry ``ENCODERS``, at the end of this file;
the encoder's attention is ``tpspp_attn_encode``).

``NRTRDecoder``: reference mmocr/models/textrecog/decoders/nrtr_decoder.py:13-177 over
``TFDecoderLayer`` / ``MultiHeadAttention`` / ``PositionwiseFeedForward`` / ``PositionalEncoding``,
common/layers/transformer_layers.py:76-167, common/modules/transformer_module.py:36-175 -- SURVEY.md section 8f rank 2.

Same constructor kwargs, sub-module names and ``state_dict`` keys (``trg_word_emb``, ``position_enc.position_table``,
``layer_stack.{i}.{norm1,norm2,norm3,self_attn.{linear_q,linear_k,linear_v,fc},enc_attn.{...},mlp.{w_1,w_2}}``,
``layer_norm``, ``classifier``), same creation order (so a seeded construction yields the reference's initial weights).

``forward_test`` is the greedy decode of the reference (``nrtr_decoder.py:153-177``) as an **incremental** decode: the
reference re-runs all six layers over the whole 41-token padded sequence at each of its 40 steps (54 of the recogniser's
60 GFLOP per image); here the keys / values of earlier positions and the projected encoder memory are kept, each step
processes ONE token per image -- dense layers on the tcgen05 3xTF32 kernels (``tpspp_linear_fwd``), attention over the
caches in ``tpspp_attn_decode``; residual adds, GELU and the LayerNorm in front of the next sub-layer run in the dense layers'
epilogues (``tpspp_linear_ln_fwd``); the embedding gather, the first LayerNorm of a step and the soft-max are torch ops.
Position ``t`` of the causal, pad-masked reference attends exactly to tokens ``0..t``, so the results are the reference's
up to fp32 summation order.  ``forward_train`` and ``forward_test_library`` (the reference's algorithm, for A/B) run torch ops; the recogniser's training
path is ``nrtr_train.decoder_train`` (native attention and dense layers, forward and backward, with the reference's dropout).
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as TF
from .rectifier import _BaseModule
from .registry import DECODERS, ENCODERS


def valid_lengths(t: int, img_metas) -> Optional[list]:
    """Valid length of each image's ``t``-token source sequence, ``min(t, ceil(t * valid_ratio))`` -- the source mask of both
    ``NRTRDecoder._get_mask`` (nrtr_decoder.py:114-127) and ``NRTREncoder._get_mask`` (nrtr_encoder.py); None without metas."""
    if img_metas is None:
        return None
    return [min(t, math.ceil(t * meta.get("valid_ratio", 1.0))) for meta in img_metas]


def _attn_lib(att, n_head, d_k, q, k, v, mask):
    """``MultiHeadAttention.forward`` (transformer_module.py:24-34,74-98) on torch ops, eval mode; ``mask`` [N, Lk] or
    [N, Lq, Lk], 0 = masked key."""
    b, lq, _ = q.shape
    lk = k.shape[1]
    qq = att.linear_q(q).view(b, lq, n_head, d_k).transpose(1, 2)
    kk = att.linear_k(k).view(b, lk, n_head, d_k).transpose(1, 2)
    vv = att.linear_v(v).view(b, lk, n_head, -1).transpose(1, 2)
    a = torch.matmul(qq / d_k ** 0.5, kk.transpose(2, 3))
    if mask is not None:
        a = a.masked_fill((mask.unsqueeze(1) if mask.dim() == 3 else mask[:, None, None, :]) == 0, float("-inf"))
    out = torch.matmul(F.softmax(a, dim=-1), vv).transpose(1, 2).contiguous().view(b, lq, -1)
    return att.fc(out)


def _sinusoid_table(n_position: int, d_hid: int) -> torch.Tensor:
    """transformer_module.py:141-154."""
    denominator = torch.Tensor([1.0 / np.power(10000, 2 * (j // 2) / d_hid) for j in range(d_hid)]).view(1, -1)
    table = torch.arange(n_position).unsqueeze(-1).float() * denominator
    table[:, 0::2] = torch.sin(table[:, 0::2])
    table[:, 1::2] = torch.cos(table[:, 1::2])
    return table.unsqueeze(0)


def _mha(n_head, d_model, d_k, d_v, qkv_bias):
    m = nn.Module()
    m.linear_q = nn.Linear(n_head * d_k, n_head * d_k, bias=qkv_bias)
    m.linear_k = nn.Linear(n_head * d_k, n_head * d_k, bias=qkv_bias)
    m.linear_v = nn.Linear(n_head * d_v, n_head * d_v, bias=qkv_bias)
    m.fc = nn.Linear(n_head * d_v, d_model, bias=qkv_bias)
    return m


@DECODERS.register_module()
class NRTRDecoder(_BaseModule):
    def __init__(self, n_layers=6, d_embedding=512, n_head=8, d_k=64, d_v=64, d_model=512, d_inner=256, n_position=200,
                 dropout=0.1, num_classes=93, max_seq_len=40, start_idx=1, padding_idx=92, init_cfg=None, qkv_bias=False, **kwargs):
        super().__init__(init_cfg=init_cfg)
        if d_k != 64 or d_v != 64 or d_embedding != d_model or d_model != n_head * d_k:
            raise ValueError("tps_pp_b200.NRTRDecoder: d_k = d_v = 64 and d_embedding = d_model = n_head * 64 (the NRTR configs)")
        self.padding_idx, self.start_idx, self.max_seq_len = padding_idx, start_idx, max_seq_len
        self.n_head, self.d_k, self.d_model, self.n_layers = n_head, d_k, d_model, n_layers
        self.trg_word_emb = nn.Embedding(num_classes, d_embedding, padding_idx=padding_idx)
        pe = nn.Module()
        pe.register_buffer("position_table", _sinusoid_table(n_position, d_embedding))
        self.position_enc = pe
        self.dropout = nn.Dropout(p=dropout)
        layers = []
        for _ in range(n_layers):
            lyr = nn.Module()
            lyr.norm1, lyr.norm2, lyr.norm3 = nn.LayerNorm(d_model), nn.LayerNorm(d_model), nn.LayerNorm(d_model)
            lyr.self_attn = _mha(n_head, d_model, d_k, d_v, qkv_bias)
            lyr.enc_attn = _mha(n_head, d_model, d_k, d_v, qkv_bias)
            mlp = nn.Module()
            mlp.w_1 = nn.Linear(d_model, d_inner)
            mlp.w_2 = nn.Linear(d_inner, d_model)
            lyr.mlp = mlp
            layers.append(lyr)
        self.layer_stack = nn.ModuleList(layers)
        self.layer_norm = nn.LayerNorm(d_model, eps=1e-6)
        self.classifier = nn.Linear(d_model, num_classes - 1)      # the padding class is never predicted (nrtr_decoder.py:77-78)
        self.last_test_native = None
        self.decode_graph = True          # replay forward_test's launches from a CUDA graph (one per batch / source length)

    # ------------------------------------------------------------------ reference algorithm on torch ops
    def _attn_lib(self, att, q, k, v, mask):
        return _attn_lib(att, self.n_head, self.d_k, q, k, v, mask)

    def _attention(self, trg_seq, src, src_mask=None):
        """nrtr_decoder.py:93-112 (pre-norm layers, transformer_layers.py:152-165); dropout is the identity in eval mode."""
        x = self.trg_word_emb(trg_seq)
        x = self.dropout(x + self.position_enc.position_table[:, :x.size(1)])
        ls = trg_seq.size(1)
        causal = (1 - torch.triu(torch.ones((ls, ls), device=trg_seq.device), diagonal=1)).unsqueeze(0).bool()
        trg_mask = (trg_seq != self.padding_idx).unsqueeze(-2) & causal
        for lyr in self.layer_stack:
            h = lyr.norm1(x)
            x = x + self._attn_lib(lyr.self_attn, h, h, h, trg_mask)
            x = x + self._attn_lib(lyr.enc_attn, lyr.norm2(x), src, src, src_mask)
            x = x + lyr.mlp.w_2(F.gelu(lyr.mlp.w_1(lyr.norm3(x))))
        return self.layer_norm(x)

    @staticmethod
    def _get_mask(logit, img_metas):
        """nrtr_decoder.py:114-127."""
        if img_metas is None:
            return None
        n, t, _ = logit.size()
        mask = logit.new_zeros((n, t))
        for i, width in enumerate(valid_lengths(t, img_metas)):
            mask[i, :width] = 1
        return mask

    def forward_train(self, feat, out_enc, targets_dict, img_metas):
        src_mask = self._get_mask(out_enc, img_metas)
        targets = targets_dict["padded_targets"].to(out_enc.device)
        return self.classifier(self._attention(targets, out_enc, src_mask=src_mask))

    def forward_test_library(self, feat, out_enc, img_metas):
        """The reference's greedy decode as written (full recompute of the padded prefix at every step), on torch ops."""
        src_mask = self._get_mask(out_enc, img_metas)
        n = out_enc.size(0)
        seq = torch.full((n, self.max_seq_len + 1), self.padding_idx, device=out_enc.device, dtype=torch.long)
        seq[:, 0] = self.start_idx
        outputs = []
        for step in range(self.max_seq_len):
            dec = self._attention(seq, out_enc, src_mask=src_mask)
            probs = F.softmax(self.classifier(dec[:, step, :]), dim=-1)
            outputs.append(probs)
            seq[:, step + 1] = probs.argmax(dim=-1)
        return torch.stack(outputs, dim=1)

    # ------------------------------------------------------------------ native incremental decode
    @torch.no_grad()
    def forward_test(self, feat, out_enc, img_metas):
        """Greedy decode -> probabilities [N, max_seq_len, num_classes - 1] (nrtr_decoder.py:153-177).  The ~4000 small launches
        of the 40 steps are replayed from one CUDA graph per (batch, source length) when ``self.decode_graph`` (default)."""
        if not out_enc.is_cuda:
            raise RuntimeError("tps_pp_b200.NRTRDecoder runs on CUDA (sm_100a) tensors only; there is no CPU fallback")
        self.last_test_native = True
        n, t_src, d = out_enc.shape
        lens = None
        if img_metas is not None:
            lens = torch.tensor(valid_lengths(t_src, img_metas), dtype=torch.int32, device=out_enc.device)
        if not getattr(self, "decode_graph", True) or torch.cuda.is_current_stream_capturing():
            return self._decode(out_enc, lens)
        key = (n, t_src, out_enc.device.index, lens is not None, tuple((p.data_ptr(), p._version) for p in self.parameters()))
        cache = self.__dict__.setdefault("_decode_graphs", {})
        ent = cache.get(key)
        if ent is None:
            if len(cache) >= 4:
                cache.clear()
            s_in = out_enc.detach().float().clone()
            s_lens = lens.clone() if lens is not None else None
            side = torch.cuda.Stream(device=out_enc.device)
            side.wait_stream(torch.cuda.current_stream(out_enc.device))
            with torch.cuda.stream(side):                      # lazy initialisations + allocator warm-up outside the capture
                self._decode(s_in, s_lens)
            torch.cuda.current_stream(out_enc.device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                s_out = self._decode(s_in, s_lens)
            ent = cache[key] = (graph, s_in, s_lens, s_out)
        graph, s_in, s_lens, s_out = ent
        s_in.copy_(out_enc)
        if lens is not None:
            s_lens.copy_(lens)
        graph.replay()
        return s_out.clone()

    def _decode(self, out_enc, lens):
        n, t_src, d = out_enc.shape
        dev = out_enc.device
        temp = self.d_k ** 0.5
        rows = (n + 127) // 128 * 128                 # the tensor-core dense kernels take multiples of 128 rows
        # encoder memory -> keys / values of every layer's enc_attn, once
        mrows = (n * t_src + 127) // 128 * 128
        mem = torch.zeros((mrows, d), dtype=torch.float32, device=dev)
        mem[: n * t_src] = out_enc.reshape(n * t_src, d).float()
        mem_k, mem_v, lin = [], [], []
        for lyr in self.layer_stack:
            ea, sa = lyr.enc_attn, lyr.self_attn
            kv = TF.linear(mem, torch.cat([ea.linear_k.weight, ea.linear_v.weight], 0),
                           None if ea.linear_k.bias is None else torch.cat([ea.linear_k.bias, ea.linear_v.bias], 0))
            # head-major [n, heads, t_src, 64]: every (image, head) attention CTA then reads one contiguous block
            mem_k.append(kv[: n * t_src, :d].reshape(n, t_src, self.n_head, 64).permute(0, 2, 1, 3).contiguous())
            mem_v.append(kv[: n * t_src, d:].reshape(n, t_src, self.n_head, 64).permute(0, 2, 1, 3).contiguous())
            # the layer's six dense operators with their operand images laid out once per decode (not once per step)
            lin.append(dict(
                qkv=TF.PreparedLinear(torch.cat([sa.linear_q.weight, sa.linear_k.weight, sa.linear_v.weight], 0),
                                      None if sa.linear_q.bias is None else torch.cat([sa.linear_q.bias, sa.linear_k.bias, sa.linear_v.bias], 0), rows),
                fc=TF.PreparedLinear(sa.fc.weight, sa.fc.bias, rows),
                q=TF.PreparedLinear(ea.linear_q.weight, ea.linear_q.bias, rows),
                efc=TF.PreparedLinear(ea.fc.weight, ea.fc.bias, rows),
                w1=TF.PreparedLinear(lyr.mlp.w_1.weight, lyr.mlp.w_1.bias, rows),
                w2=TF.PreparedLinear(lyr.mlp.w_2.weight, lyr.mlp.w_2.bias, rows)))
        ncls = self.classifier.weight.shape[0]
        npad = (ncls + 31) // 32 * 32                      # the tensor-core kernel takes output widths that are multiples of 32
        wc = torch.zeros((npad, d), dtype=torch.float32, device=dev)
        wc[:ncls] = self.classifier.weight
        bc = torch.zeros((npad,), dtype=torch.float32, device=dev)
        bc[:ncls] = self.classifier.bias
        cls = TF.PreparedLinear(wc, bc, rows)
        cap = self.max_seq_len
        k_cache = [torch.zeros((n, self.n_head, cap, 64), dtype=torch.float32, device=dev) for _ in self.layer_stack]
        v_cache = [torch.zeros((n, self.n_head, cap, 64), dtype=torch.float32, device=dev) for _ in self.layer_stack]
        tok = torch.full((n,), self.start_idx, dtype=torch.long, device=dev)
        x = torch.zeros((rows, d), dtype=torch.float32, device=dev)
        att = torch.zeros((rows, d), dtype=torch.float32, device=dev)
        pos = self.position_enc.position_table[0]
        outputs = []
        hn = torch.zeros((rows, d), dtype=torch.float32, device=dev)     # LN(x) for the next sub-layer, written by the dense layer before it
        layers = list(self.layer_stack)
        for step in range(self.max_seq_len):
            x[:n] = self.trg_word_emb(tok) + pos[step]
            hn[:n] = layers[0].norm1(x[:n])
            for li, lyr in enumerate(layers):
                ops = lin[li]
                qkv = ops["qkv"](hn)
                # q, and this step's k / v rows, are column slices of the fused projection; the kernel appends k / v to the cache
                TF.attn_decode(qkv[:n, :d], k_cache[li], v_cache[li], self.n_head, step + 1, temp, out=att[:n],
                               k_new=qkv[:n, d:2 * d], v_new=qkv[:n, 2 * d:], head_major=True)
                # x += fc(att) and hn = norm2(x): residual and the next LayerNorm in the kernel that finishes the dense layer
                ops["fc"](att, out=x, residual=x, ln=lyr.norm2, ln_out=hn)
                q = ops["q"](hn)
                TF.attn_decode(q[:n], mem_k[li], mem_v[li], self.n_head, t_src, temp, kv_lens=lens, out=att[:n], head_major=True)
                ops["efc"](att, out=x, residual=x, ln=lyr.norm3, ln_out=hn)
                nxt = layers[li + 1].norm1 if li + 1 < len(layers) else self.layer_norm
                ops["w2"](ops["w1"](hn, gelu=True), out=x, residual=x, ln=nxt, ln_out=hn)   # x += w_2(GELU(w_1(LN(x))))
            probs = F.softmax(cls(hn)[:n, :ncls], dim=-1)
            outputs.append(probs)
            tok = probs.argmax(dim=-1)
        return torch.stack(outputs, dim=1)

    def forward(self, feat, out_enc, targets_dict=None, img_metas=None, train_mode=True):
        """decoders/base_decoder.py: dispatch on ``train_mode``."""
        self.train_mode = train_mode
        if train_mode:
            return self.forward_train(feat, out_enc, targets_dict, img_metas)
        return self.forward_test(feat, out_enc, img_metas)


_PRE_NORM = ("norm", "self_attn", "norm", "ffn")


@ENCODERS.register_module()
class NRTREncoder(_BaseModule):
    """Drop-in ``NRTREncoder`` (registry ``ENCODERS``; reference mmocr/models/textrecog/encoders/nrtr_encoder.py over pre-norm
    ``TFEncoderLayer`` / ``MultiHeadAttention`` / ``PositionwiseFeedForward``, common/layers/transformer_layers.py,
    common/modules/transformer_module.py).  Same constructor kwargs, ``state_dict`` keys (``layer_stack.{i}.{attn.{linear_q,
    linear_k,linear_v,fc},norm1,mlp.{w_1,w_2},norm2}``, ``layer_norm``) and creation order as the reference.

    ``forward(feat [N, C, H, W], img_metas) -> [N, H*W, C]``.  In eval mode under ``torch.no_grad()`` on fp32 CUDA tensors it
    runs natively: per layer one fused q|k|v dense layer, ``tpspp_attn_encode`` over the whole sequence with the valid-ratio
    key mask, ``fc`` with the residual add and ``norm2`` in its epilogue, ``w_1`` with GELU, ``w_2`` with the residual add and
    the next layer's ``norm1`` (after the last layer: the final ``layer_norm``) -- the tcgen05 3xTF32 dense kernels of
    ``NRTRDecoder``.  ``forward_library`` is the reference algorithm on torch ops; ``forward`` uses it while autograd records,
    in training mode, for head sizes other than 64 or model widths that are not a multiple of 128, and for an image whose
    valid length is 0 (the reference's soft-max over no key: NaN rows).  Neither path applies dropout (the identity in eval
    mode); ``nrtr_train.encoder_train`` is the training forward with the reference's dropout (``p = dropout``) on native
    forward and backward kernels, which ``NRTR.forward_train`` uses."""

    def __init__(self, n_layers=6, n_head=8, d_k=64, d_v=64, d_model=512, d_inner=256, dropout=0.1, init_cfg=None, **kwargs):
        super().__init__(init_cfg=init_cfg)
        qkv_bias = kwargs.pop("qkv_bias", False)
        order = kwargs.pop("operation_order", None)
        act_cfg = kwargs.pop("act_cfg", None)
        if kwargs:
            raise TypeError(f"tps_pp_b200.NRTREncoder got unexpected keyword arguments {sorted(kwargs)}")
        if order is not None and tuple(order) != _PRE_NORM:
            raise ValueError(f"tps_pp_b200.NRTREncoder implements the pre-norm layer {_PRE_NORM} only, got operation_order={order!r}")
        if act_cfg is not None and dict(act_cfg) not in (dict(type="mmcv.GELU"), dict(type="GELU")):
            raise ValueError(f"tps_pp_b200.NRTREncoder implements the GELU feed-forward only, got act_cfg={act_cfg!r}")
        self.n_layers, self.n_head, self.d_k, self.d_v, self.d_model = n_layers, n_head, d_k, d_v, d_model
        self.dropout = dropout            # applied by nrtr_train.encoder_train in training mode
        layers = []
        for _ in range(n_layers):
            lyr = nn.Module()
            lyr.attn = _mha(n_head, d_model, d_k, d_v, qkv_bias)
            lyr.norm1 = nn.LayerNorm(d_model)
            mlp = nn.Module()
            mlp.w_1 = nn.Linear(d_model, d_inner)
            mlp.w_2 = nn.Linear(d_inner, d_model)
            lyr.mlp = mlp
            lyr.norm2 = nn.LayerNorm(d_model)
            layers.append(lyr)
        self.layer_stack = nn.ModuleList(layers)
        self.layer_norm = nn.LayerNorm(d_model)
        self.last_forward_native = None

    def _native_ok(self, feat, lens) -> bool:
        return (not self.training and not torch.is_grad_enabled() and feat.dtype == torch.float32 and feat.dim() == 4
                and self.d_k == 64 and self.d_v == 64 and self.d_model == self.n_head * 64 and self.d_model % 128 == 0
                and self.d_model <= 1024 and feat.shape[1] == self.d_model and (lens is None or min(lens, default=1) > 0))

    def forward(self, feat, img_metas=None):
        """nrtr_encoder.py:66-87: [N, C, H, W] -> [N, H*W, C]."""
        if not feat.is_cuda:
            raise RuntimeError("tps_pp_b200.NRTREncoder runs on CUDA (sm_100a) tensors only; there is no CPU fallback "
                               "(forward_library is the torch-ops A/B path)")
        lens = valid_lengths(feat.shape[2] * feat.shape[3], img_metas)
        self.last_forward_native = self._native_ok(feat, lens)
        if self.last_forward_native:
            return self._encode(feat, lens)
        return self.forward_library(feat, img_metas)

    def forward_library(self, feat, img_metas=None):
        """The reference's algorithm on torch ops (any device): pre-norm layers x += attn(norm1(x)); x += w_2(GELU(w_1(norm2(x))))."""
        n, c, h, w = feat.size()
        x = feat.view(n, c, h * w).permute(0, 2, 1).contiguous()
        lens = valid_lengths(h * w, img_metas)
        mask = None
        if lens is not None:
            mask = x.new_zeros((n, h * w))
            for i, width in enumerate(lens):
                mask[i, :width] = 1
        for lyr in self.layer_stack:
            hn = lyr.norm1(x)
            x = x + _attn_lib(lyr.attn, self.n_head, self.d_k, hn, hn, hn, mask)
            x = x + lyr.mlp.w_2(F.gelu(lyr.mlp.w_1(lyr.norm2(x))))
        return self.layer_norm(x)

    @torch.no_grad()
    def _encode(self, feat, lens):
        n, c, h, w = feat.shape
        t = h * w
        dev = feat.device
        rows = (n * t + 127) // 128 * 128              # the tensor-core dense kernels take multiples of 128 rows
        x = torch.zeros((rows, c), dtype=torch.float32, device=dev)
        x[: n * t].view(n, t, c).copy_(feat.reshape(n, c, t).permute(0, 2, 1))
        att = torch.zeros((rows, c), dtype=torch.float32, device=dev)
        kv_lens = torch.tensor(lens, dtype=torch.int32, device=dev) if lens is not None else None
        layers = list(self.layer_stack)
        hn = (layers[0].norm1 if layers else self.layer_norm)(x).contiguous()    # LN(x) for the next sub-layer
        temp = self.d_k ** 0.5
        for li, lyr in enumerate(layers):
            a, mlp = lyr.attn, lyr.mlp
            # the operand images of the layer's dense weights are laid out once per call (each is used once)
            qkv = TF.PreparedLinear(torch.cat([a.linear_q.weight, a.linear_k.weight, a.linear_v.weight], 0),
                                    None if a.linear_q.bias is None else torch.cat([a.linear_q.bias, a.linear_k.bias, a.linear_v.bias], 0),
                                    rows)(hn)
            # q, k, v are column slices of the fused projection
            TF.attn_encode(qkv[: n * t, :c], qkv[: n * t, c:2 * c], qkv[: n * t, 2 * c:], self.n_head, t, temp, kv_lens=kv_lens,
                           out=att[: n * t])
            # x += fc(att) and hn = norm2(x): residual and the next LayerNorm in the kernel that finishes the dense layer
            TF.PreparedLinear(a.fc.weight, a.fc.bias, rows)(att, out=x, residual=x, ln=lyr.norm2, ln_out=hn)
            mid = TF.PreparedLinear(mlp.w_1.weight, mlp.w_1.bias, rows)(hn, gelu=True)
            nxt = layers[li + 1].norm1 if li + 1 < len(layers) else self.layer_norm
            TF.PreparedLinear(mlp.w_2.weight, mlp.w_2.bias, rows)(mid, out=x, residual=x, ln=nxt, ln_out=hn)   # x += w_2(GELU(w_1(LN(x))))
        return hn[: n * t].view(n, t, c)
