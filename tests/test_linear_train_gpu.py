"""Native forward / backward of the head's dense layers (tpspp_linear_fwd / tpspp_linear_bwd, include/tpspp.h) against fp64
torch autograd on the device.  Shapes = every nn.Linear / bmm of the rectifier's training path at a small batch
(DGAB.py:11-23,28-36,52; tps_pp.py:250-273,293-299) plus ragged ones that must take the CUDA-core kernels."""
import pytest
import torch

pytestmark = pytest.mark.gpu

# (leading shape, in, out, bias, what)
CASES = [
    ((4, 64, 16), 64, 64, True, "DGAB attn.proj"),
    ((4, 64, 16), 64, 256, True, "Mlp fc1"),
    ((4, 64, 16), 256, 64, True, "Mlp fc2"),
    ((4, 1024), 64, 32, True, "feat_linear.0"),
    ((4, 1024), 32, 128, True, "feat_linear.1"),
    ((4, 32), 64, 256, True, "localization_fc1.0 (rows = 128)"),
    ((4, 32), 256, 2, True, "localization_fc1.2 (odd width)"),
    ((4,), 64, 64, True, "localization_fc2 (4 rows)"),
    ((4, 64), 96, 65, False, "DGAB mlp_w (odd width, no bias)"),
    ((4, 64), 48, 17, False, "DGAB mlp_h"),
    ((8, 4, 64, 16), 64, 256, True, "Mlp fc1, 32768 rows"),
    ((3, 37), 50, 7, True, "ragged"),
    ((256,), 512, 512, True, "transformer-sized 512 -> 512 (shared-memory-operand tcgen05 kernel)"),
    ((3, 128), 256, 1536, False, "fused QKV 256 -> 1536"),
    ((128,), 512, 96, True, "512 -> 96 (32-column tiles)"),
]


def _rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("lead,k,n,bias,what", CASES, ids=[c[4] for c in CASES])
def test_linear_fwd_bwd_vs_fp64(lead, k, n, bias, what):
    from tps_pp_b200 import functional as TF
    dev = torch.device("cuda", 0)
    import zlib
    g = torch.Generator(device=dev).manual_seed(zlib.crc32(what.encode()) % 1000)        # str hashes are randomised per process
    x = torch.randn(lead + (k,), device=dev, generator=g, requires_grad=True)
    w = (torch.randn((n, k), device=dev, generator=g) / k ** 0.5).requires_grad_()
    b = torch.randn((n,), device=dev, generator=g).requires_grad_() if bias else None
    gy = torch.randn(lead + (n,), device=dev, generator=g)
    y = TF.linear(x, w, b)
    y.backward(gy)
    xd, wd = x.detach().double().requires_grad_(), w.detach().double().requires_grad_()
    bd = b.detach().double().requires_grad_() if bias else None
    yd = torch.nn.functional.linear(xd, wd, bd)
    yd.backward(gy.double())
    # fp32-level: 3xTF32 with fp32 accumulation -- the bound grows with the square root of the contraction length
    assert _rel(y.detach(), yd.detach()) <= 3e-6 * max(1.0, (k / 256) ** 0.5), what
    assert _rel(x.grad, xd.grad) <= 3e-6 * max(1.0, (n / 256) ** 0.5), what
    assert _rel(w.grad, wd.grad) <= 8e-6, what
    if bias:
        assert _rel(b.grad, bd.grad) <= 5e-6, what


@pytest.mark.parametrize("bsz,rows,k,n", [(4, 1024, 128, 32), (3, 100, 20, 5)], ids=["score QK^T", "ragged"])
def test_bmm_nt_fwd_bwd_vs_fp64(bsz, rows, k, n):
    from tps_pp_b200 import functional as TF
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(rows)
    x = torch.randn((bsz, rows, k), device=dev, generator=g, requires_grad=True)
    w = (torch.randn((bsz, n, k), device=dev, generator=g) / k ** 0.5).requires_grad_()
    gy = torch.randn((bsz, rows, n), device=dev, generator=g)
    y = TF.bmm_nt(x, w)
    y.backward(gy)
    xd, wd = x.detach().double().requires_grad_(), w.detach().double().requires_grad_()
    yd = torch.bmm(xd, wd.transpose(1, 2))
    yd.backward(gy.double())
    assert _rel(y.detach(), yd.detach()) <= 2e-6
    assert _rel(x.grad, xd.grad) <= 2e-6
    assert _rel(w.grad, wd.grad) <= 5e-6


def test_linear_rejects_cpu_tensors():
    from tps_pp_b200 import functional as TF
    with pytest.raises(RuntimeError):
        TF.linear(torch.zeros(4, 8), torch.zeros(3, 8), None)


# on 148 SMs the "unsplit" ids take split-K too; tests/test_recognizer_batch_gpu.py covers the unsplit paths at the NRTR shapes
@pytest.mark.parametrize("rows,k,n", [(256, 512, 512), (1024, 512, 256), (256, 256, 512), (128, 64, 64)], ids=["split-K", "unsplit", "K=256", "small"])
def test_prepared_linear_residual_gelu(rows, k, n):
    """The inference form a transformer layer needs: act(x w^T + b) + residual in the dense kernel's epilogue (or in the split-K
    reduction), cached operand images, in-place residual."""
    from tps_pp_b200 import functional as TF
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(rows + k + n)
    x = torch.randn((rows, k), device=dev, generator=g)
    w = torch.randn((n, k), device=dev, generator=g) / k ** 0.5
    b = torch.randn((n,), device=dev, generator=g)
    r = torch.randn((rows, n), device=dev, generator=g)
    op = TF.PreparedLinear(w, b, rows)
    for gelu in (False, True):
        lin = torch.nn.functional.linear(x.double(), w.double(), b.double())
        ref = (torch.nn.functional.gelu(lin) if gelu else lin) + r.double()
        for _ in range(2):                                   # second call: cached operand image
            y = op(x, residual=r, gelu=gelu)
            assert _rel(y, ref) <= 3e-6 * max(1.0, (k / 256) ** 0.5)
        inplace = r.clone()
        op(x, out=inplace, residual=inplace, gelu=gelu)
        assert torch.equal(inplace, y)


# on 148 SMs the "unsplit" ids take split-K too; tests/test_recognizer_batch_gpu.py covers the unsplit paths at the NRTR shapes
@pytest.mark.parametrize("rows,k,n", [(256, 512, 512), (1024, 512, 256), (256, 256, 128), (64, 48, 128), (256, 512, 1024), (128, 1024, 768)],
                         ids=["split-K", "unsplit", "K=256", "cuda-core", "N=1024", "N=768"])
def test_prepared_linear_with_layernorm_output(rows, k, n):
    """``tpspp_linear_ln_fwd``: y = x w^T + b + residual and LN(y) for the next sub-layer from the kernel that finishes y
    (split-K reduction, or a warp-per-row pass behind the unsplit kernel); in-place residual; y itself unchanged by the LN."""
    from tps_pp_b200 import functional as TF
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(7 * rows + k + n)
    x = torch.randn((rows, k), device=dev, generator=g)
    w = torch.randn((n, k), device=dev, generator=g) / k ** 0.5
    b = torch.randn((n,), device=dev, generator=g)
    r = torch.randn((rows, n), device=dev, generator=g)
    ln = torch.nn.LayerNorm(n, eps=1e-6).to(dev)
    with torch.no_grad():
        ln.weight.copy_(1.0 + 0.1 * torch.randn((n,), device=dev, generator=g))
        ln.bias.copy_(0.1 * torch.randn((n,), device=dev, generator=g))
    op = TF.PreparedLinear(w, b, rows)
    plain = op(x, residual=r)
    ref = torch.nn.functional.linear(x.double(), w.double(), b.double()) + r.double()
    ref_ln = torch.nn.functional.layer_norm(ref, (n,), ln.weight.double(), ln.bias.double(), 1e-6)
    for _ in range(2):
        hn = torch.full((rows, n), float("nan"), device=dev)
        y = op(x, residual=r, ln=ln, ln_out=hn)
        assert torch.equal(y, plain)                       # same reduction order with or without the LayerNorm output
        assert _rel(hn, ref_ln) <= 4e-6 * max(1.0, (k / 256) ** 0.5)
        assert (hn - torch.nn.functional.layer_norm(y, (n,), ln.weight, ln.bias, 1e-6)).abs().max().item() <= 2e-6
    inplace = r.clone()
    hn2 = torch.empty_like(hn)
    op(x, out=inplace, residual=inplace, ln=ln, ln_out=hn2)
    assert torch.equal(inplace, plain) and torch.equal(hn2, hn)
    with pytest.raises(RuntimeError):
        op(x, residual=r, ln=ln, ln_out=None)
    with pytest.raises(RuntimeError):
        op(x, residual=r, gelu=True, ln=ln, ln_out=hn)      # LayerNorm output with an activation: rejected by the library
