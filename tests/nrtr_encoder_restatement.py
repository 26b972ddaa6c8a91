"""CPU restatement of the reference NRTR encoder for the encoder tests (torch functional, dtype-parametric), written from the
reference independently of tps_pp_b200: NRTREncoder.forward (encoders/nrtr_encoder.py:66-87) over pre-norm TFEncoderLayers
(common/layers/transformer_layers.py, operation_order ('norm', 'self_attn', 'norm', 'ffn')) and MultiHeadAttention /
ScaledDotProductAttention (common/modules/transformer_module.py:24-34,74-98), eval mode (dropout = identity).

It sits beside the tests rather than in oracle/ so that the pinned oracle stays as it is; it is not pinned against the
reference class by oracle/make_golden.py."""
import math

import numpy as np
import torch
import torch.nn.functional as F


def _t(state, key, dtype, device="cpu"):
    v = state[key]
    if isinstance(v, np.ndarray):
        v = torch.from_numpy(v)
    return v.detach().to(dtype=dtype, device=device)


def _linear(state, prefix, x, dtype):
    b = _t(state, prefix + ".bias", dtype, x.device) if (prefix + ".bias") in state else None
    return F.linear(x, _t(state, prefix + ".weight", dtype, x.device), b)


def _mha(state, prefix, q, k, v, mask, n_head, dk, dtype):
    """MultiHeadAttention.forward; ``mask`` [N, Lk], 0 = masked key (an all-masked row gives NaN, as in the reference)."""
    b, lq, lk = q.shape[0], q.shape[1], k.shape[1]
    qq = _linear(state, prefix + ".linear_q", q, dtype).view(b, lq, n_head, dk).transpose(1, 2)
    kk = _linear(state, prefix + ".linear_k", k, dtype).view(b, lk, n_head, dk).transpose(1, 2)
    vv = _linear(state, prefix + ".linear_v", v, dtype).view(b, lk, n_head, -1).transpose(1, 2)
    a = torch.matmul(qq / dk ** 0.5, kk.transpose(2, 3))
    if mask is not None:
        a = a.masked_fill(mask.unsqueeze(1).unsqueeze(1) == 0, float("-inf"))
    out = torch.matmul(F.softmax(a, dim=-1), vv).transpose(1, 2).contiguous().view(b, lq, -1)
    return _linear(state, prefix + ".fc", out, dtype)


def nrtr_encoder_forward(state, feat, valid_ratios=None, n_head=8, dtype=torch.float32, device="cpu"):
    """feat [N, C, H, W] -> [N, H*W, C] on ``device``; ``valid_ratios`` -> the key mask of ``_get_mask`` (keys
    t < min(T, ceil(T * r)))."""
    feat = torch.as_tensor(feat).to(dtype=dtype, device=device)
    n, c, h, w = feat.shape
    t = h * w
    dk = c // n_head
    x = feat.reshape(n, c, t).permute(0, 2, 1).contiguous()
    mask = None
    if valid_ratios is not None:
        mask = torch.zeros((n, t), dtype=dtype, device=device)
        for i, vr in enumerate(valid_ratios):
            mask[i, :min(t, math.ceil(t * vr))] = 1
    i = 0
    while f"layer_stack.{i}.norm1.weight" in state:
        p = f"layer_stack.{i}."

        def ln(nm, v):
            return F.layer_norm(v, (c,), _t(state, p + nm + ".weight", dtype, device), _t(state, p + nm + ".bias", dtype, device), 1e-5)

        hn = ln("norm1", x)
        x = x + _mha(state, p + "attn", hn, hn, hn, mask, n_head, dk, dtype)
        x = x + _linear(state, p + "mlp.w_2", F.gelu(_linear(state, p + "mlp.w_1", ln("norm2", x), dtype)), dtype)
        i += 1
    return F.layer_norm(x, (c,), _t(state, "layer_norm.weight", dtype, device), _t(state, "layer_norm.bias", dtype, device), 1e-5)
