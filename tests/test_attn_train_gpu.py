"""GPU: the training attention kernels (tpspp_attn_train_fwd / _bwd through TF.attention) against fp64 torch autograd on the device:
forward and dq / dk / dv at dropout 0 for the three calls of an NRTR training step and the edges of the supported range, the
dropout mask read back from the kernel and checked against the fp64 twin, the kept fraction, determinism, argument checks."""
import ctypes
import math

import pytest
import torch

from tps_pp_b200 import _native as N
from tps_pp_b200 import functional as TF

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _twin(q, k, v, b, heads, lq, lk, lens, causal, temp, keep=None, p=0.0):
    """The reference's ScaledDotProductAttention (transformer_module.py:24-34) over [b*l, heads*64] rows, in q's dtype."""
    qq = q.reshape(b, lq, heads, 64).transpose(1, 2) / temp
    kk = k.reshape(b, lk, heads, 64).transpose(1, 2)
    vv = v.reshape(b, lk, heads, 64).transpose(1, 2)
    a = torch.matmul(qq, kk.transpose(2, 3))
    valid = torch.ones((b, 1, lq, lk), dtype=torch.bool, device=q.device)
    if lens is not None:
        valid = valid & (torch.arange(lk, device=q.device)[None, None, None, :] < torch.as_tensor(lens, device=q.device).view(b, 1, 1, 1))
    if causal:
        valid = valid & (torch.arange(lk, device=q.device)[None, :] <= torch.arange(lq, device=q.device)[:, None])
    pr = torch.softmax(a.masked_fill(~valid, float("-inf")), -1)
    if keep is not None:
        pr = pr * keep.to(pr.dtype) / (1 - p)
    return torch.matmul(pr, vv).transpose(1, 2).reshape(b * lq, heads * 64)


def _lengths(kind, b, lq, lk, g):
    if kind is None:
        return None
    if kind == "target":            # decoder self-attention: each row's number of leading non-pad tokens
        lens = torch.randint(1, lk + 1, (b,), generator=g).tolist()
    elif kind == "ratio":           # the encoder's / the cross-attention's valid-ratio source lengths
        lens = [min(lk, math.ceil(lk * r)) for r in torch.tensor([1.0, 0.5, 0.75, 0.25, 0.9, 0.6])[torch.randint(0, 6, (b,), generator=g)].tolist()]
    else:
        lens = torch.randint(1, lk + 1, (b,), generator=g).tolist()
    lens[0] = lk if b > 1 else lens[0]
    lens[-1] = 1 if b > 2 else lens[-1]
    return lens


def _inputs(b, heads, lq, lk, g, fused):
    """q / k / v as column slices of the projections a training step makes: one fused q|k|v (self-attention) or q plus a fused
    k|v (cross-attention); returns the leaves and the three slices."""
    d = heads * 64
    if fused:
        qkv = torch.randn((b * lq, 3 * d), generator=g).to(DEV).requires_grad_()
        return [qkv], (qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:])
    q = torch.randn((b * lq, d), generator=g).to(DEV).requires_grad_()
    kv = torch.randn((b * lk, 2 * d), generator=g).to(DEV).requires_grad_()
    return [q, kv], (q, kv[:, :d], kv[:, d:])


SHAPES = [(40, 40, True, "target"), (40, 64, False, "ratio"), (64, 64, False, "ratio"), (1, 1, False, None), (33, 200, False, "random"),
          (256, 256, True, "random"), (256, 256, False, None)]


@pytest.mark.parametrize("heads,b", [(1, 1), (1, 130), (8, 3), (8, 130)])
@pytest.mark.parametrize("lq,lk,causal,lens_kind", SHAPES)
def test_attention_vs_fp64_autograd(native_lib, lq, lk, causal, lens_kind, heads, b):
    g = torch.Generator().manual_seed(lq * 1000 + lk + 7 * heads + b)
    lens = _lengths(lens_kind, b, lq, lk, g)
    leaves, (q, k, v) = _inputs(b, heads, lq, lk, g, fused=(lq == lk))
    temp = 8.0
    out = TF.attention(q, k, v, heads, lq, lk, temp, kv_lens=lens, causal=causal)
    gout = torch.randn(out.shape, generator=g).to(DEV)
    out.backward(gout)
    leaves64 = [t.detach().double().requires_grad_() for t in leaves]
    d = heads * 64
    q64, k64, v64 = ((leaves64[0][:, :d], leaves64[0][:, d:2 * d], leaves64[0][:, 2 * d:]) if len(leaves64) == 1
                     else (leaves64[0], leaves64[1][:, :d], leaves64[1][:, d:]))
    ref = _twin(q64, k64, v64, b, heads, lq, lk, lens, causal, temp)
    ref.backward(gout.double())
    err = float((out.double() - ref).abs().max())
    assert err <= 2e-6 * max(1.0, float(ref.abs().max())), err
    parts = ((leaves[0].grad[:, :d], leaves[0].grad[:, d:2 * d], leaves[0].grad[:, 2 * d:]) if len(leaves) == 1
             else (leaves[0].grad, leaves[1].grad[:, :d], leaves[1].grad[:, d:]))
    parts64 = ((leaves64[0].grad[:, :d], leaves64[0].grad[:, d:2 * d], leaves64[0].grad[:, 2 * d:]) if len(leaves64) == 1
               else (leaves64[0].grad, leaves64[1].grad[:, :d], leaves64[1].grad[:, d:]))
    for name, gn, gr in zip(("dq", "dk", "dv"), parts, parts64):
        # with one valid key per query the exact dq and dk are 0 (dS = P (dP - D) = dP - dP): then the scale is |gout|'s, 1
        e, scale = float((gn.double() - gr).abs().max()), float(gr.abs().max())
        assert e <= 1e-5 * (scale if scale > 0 else 1.0), (name, e, scale)


def _probe(b, heads, lq, lk, lens, causal, p, seed):
    """q = 0 and v[j] = e_j: out[i, h*64 + j] = keep(b, h, i, j) / (n_i (1 - p)) over the n_i valid keys of query i -> keep."""
    d = heads * 64
    q = torch.zeros((b * lq, d), device=DEV)
    k = torch.randn((b * lk, d), device=DEV)
    v = torch.zeros((b, lk, heads, 64), device=DEV)
    for j in range(lk):
        v[:, j, :, j] = 1.0
    torch.cuda.manual_seed(seed)
    out = TF.attention(q, k, v.reshape(b * lk, d), heads, lq, lk, 8.0, kv_lens=lens, causal=causal, dropout_p=p)
    return out.view(b, lq, heads, 64)[..., :lk].permute(0, 2, 1, 3)        # [b, heads, lq, lk]


@pytest.mark.parametrize("lq,lk,causal", [(40, 40, True), (40, 64, False), (64, 64, False)])
def test_dropout_mask_matches_the_fp64_twin(native_lib, lq, lk, causal):
    b, heads, p, seed = 5, 8, 0.1, 1234
    g = torch.Generator().manual_seed(lq + lk)
    lens = _lengths("ratio", b, lq, lk, g)
    probe = _probe(b, heads, lq, lk, lens, causal, p, seed)
    keep = probe > 0
    # every non-zero entry is exactly 1 / (n_i (1 - p))
    valid = (torch.arange(lk, device=DEV)[None, None, None, :] < torch.tensor(lens, device=DEV).view(b, 1, 1, 1))
    if causal:
        valid = valid & (torch.arange(lk, device=DEV)[None, :] <= torch.arange(lq, device=DEV)[:, None])
    n_valid = valid.sum(-1, keepdim=True).double()
    expect = torch.where(keep, 1.0 / (n_valid * (1 - p)), torch.zeros((), dtype=torch.float64, device=DEV))
    assert float((probe.double() - expect).abs().max()) <= 1e-6
    assert not (keep & ~valid).any()
    # the same seed on random inputs: the kernels use that mask, forward and backward
    leaves, (q, k, v) = _inputs(b, heads, lq, lk, g, fused=(lq == lk))
    torch.cuda.manual_seed(seed)
    out = TF.attention(q, k, v, heads, lq, lk, 8.0, kv_lens=lens, causal=causal, dropout_p=p)
    gout = torch.randn(out.shape, generator=g).to(DEV)
    out.backward(gout)
    leaves64 = [t.detach().double().requires_grad_() for t in leaves]
    d = heads * 64
    q64, k64, v64 = ((leaves64[0][:, :d], leaves64[0][:, d:2 * d], leaves64[0][:, 2 * d:]) if len(leaves64) == 1
                     else (leaves64[0], leaves64[1][:, :d], leaves64[1][:, d:]))
    # keep is only observable on valid keys; elsewhere the probability is 0 whatever the mask says
    ref = _twin(q64, k64, v64, b, heads, lq, lk, lens, causal, 8.0, keep=keep, p=p)
    ref.backward(gout.double())
    assert float((out.double() - ref).abs().max()) <= 2e-6 * max(1.0, float(ref.abs().max()))
    for t, t64 in zip(leaves, leaves64):
        for c0 in range(0, t.shape[1], d):
            gn, gr = t.grad[:, c0:c0 + d].double(), t64.grad[:, c0:c0 + d]
            assert float((gn - gr).abs().max()) <= 1e-5 * float(gr.abs().max())


def test_dropout_keeps_one_minus_p(native_lib):
    b, heads, L = 64, 8, 64                      # 2.1e6 draws
    for p in (0.1, 0.5):
        keep = _probe(b, heads, L, L, None, False, p, seed=99) > 0
        n = keep.numel()
        frac = float(keep.double().mean())
        sigma = math.sqrt(p * (1 - p) / n)
        assert n >= 10 ** 6 and abs(frac - (1 - p)) <= 5 * sigma, (p, frac, sigma)


def test_same_seed_same_bits_other_seed_other_mask(native_lib):
    b, heads, L, p = 6, 8, 40, 0.1
    g = torch.Generator().manual_seed(3)
    lens = _lengths("target", b, L, L, g)
    leaves, _ = _inputs(b, heads, L, L, g, fused=True)
    gout = torch.randn((b * L, heads * 64), generator=g).to(DEV)

    def run(seed):
        qkv = leaves[0].detach().clone().requires_grad_()
        d = heads * 64
        torch.cuda.manual_seed(seed)
        out = TF.attention(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], heads, L, L, 8.0, kv_lens=lens, causal=True, dropout_p=p)
        out.backward(gout)
        return out.detach(), qkv.grad

    o1, g1 = run(5)
    o2, g2 = run(5)
    assert torch.equal(o1, o2) and torch.equal(g1, g2)
    o3, g3 = run(6)
    assert not torch.equal(o1, o3)
    m1 = _probe(b, heads, L, L, lens, True, p, seed=5) > 0
    m2 = _probe(b, heads, L, L, lens, True, p, seed=6) > 0
    assert not torch.equal(m1, m2)


def test_attention_checks_its_arguments(native_lib):
    d = 128
    x = torch.randn((2 * 8, 3 * d), device=DEV)
    q, k, v = x[:, :d], x[:, d:2 * d], x[:, 2 * d:]
    with pytest.raises(ValueError):
        TF.attention(q, k, v, 2, 8, 8, 8.0, kv_lens=[8, 0])                 # an image with no valid key
    with pytest.raises(ValueError):
        TF.attention(q, k, v, 2, 8, 8, 8.0, kv_lens=[9, 1])
    with pytest.raises(ValueError):
        TF.attention(q, k, v, 2, 8, 8, 8.0, dropout_p=1.0)
    with pytest.raises(ValueError):
        TF.attention(torch.randn((257, d), device=DEV), torch.randn((257, d), device=DEV), torch.randn((257, d), device=DEV),
                     2, 257, 257, 8.0)
    with pytest.raises(RuntimeError, match="kv_lens"):
        TF.attention(q, k, v, 2, 8, 8, 8.0, kv_lens=[8])
    with pytest.raises(RuntimeError, match="row stride"):
        TF.attention(q, k.contiguous(), v, 2, 8, 8, 8.0)
    with pytest.raises(RuntimeError):
        TF.attention(q, k, v, 4, 8, 8, 8.0)                                 # 128 features are 2 heads, not 4
    with pytest.raises(RuntimeError):
        TF.attention(q, k, v, 2, 5, 5, 8.0)                                 # 16 rows are not whole images of 5 tokens
    with pytest.raises(RuntimeError):
        TF.attention(q.cpu(), k.cpu(), v.cpu(), 2, 8, 8, 8.0)
    # the ABI rejects malformed cfgs before it reads any pointer
    good = dict(batch=2, heads=2, head_dim=64, len_q=8, len_k=8, temperature=8.0, causal=0, dropout_p=0.0, q_stride=0, kv_stride=0)
    # (each rejection names its field, so a cfg check cannot be mistaken for the null-pointer check that follows it)
    cases = [(dict(head_dim=32), "head_dim"), (dict(len_q=0), "len_q, len_k"), (dict(len_k=257), "len_q, len_k"),
             (dict(causal=2), "causal"), (dict(dropout_p=1.0), "dropout_p"), (dict(dropout_p=-0.1), "dropout_p"),
             (dict(temperature=0.0), "temperature"), (dict(q_stride=130), "q_stride / kv_stride"),
             (dict(kv_stride=64), "q_stride / kv_stride"), (dict(heads=0), "heads"), (dict(dropout_p=0.1), "null pointer")]
    for bad, field in cases:
        cfg = N.AttnTrainCfg(**dict(good, **bad))
        null = [None] * 6
        assert N.lib().tpspp_attn_train_fwd(ctypes.byref(cfg), *null, None, None) != N.OK, bad
        assert field in N.last_error(), (bad, N.last_error())
        assert N.lib().tpspp_attn_train_bwd(ctypes.byref(cfg), *null, None, None, None, None, None, None) != N.OK, bad
        assert field in N.last_error(), (bad, N.last_error())
