"""GPU: the drop-in modules (TPS_PP, TPSPreprocessor) against reference vectors and the oracle."""
import numpy as np
import pytest
import torch

import tps_pp_b200 as T
from tps_pp_b200 import _native as N
from oracle import tpspp_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# whole-module pixels: |ours - ref64| against the reference's own fp32 error |ref32 - ref64| (SURVEY F6).  Two independent
# fp32 evaluations of the same function: the max over 131 K pixels of ours lands at 0.001-1.13x the reference's
# (measured, scripts/dev/floors.py), so 1.5x is the regression trip-wire (round 1 used 4x)
FLOOR_K = 1.5


def mx(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    return float(np.max(np.abs(a.astype(np.float64) - b.astype(np.float64))))


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield


def test_tps_pp_forward_vs_reference_golden(golden, native_lib):
    """Three-tier parity of the whole module (SURVEY F6): control points 1e-4 (north_star), pc_score,
    and pixels against the reference's fp64 twin with the reference's own fp32 error as the floor."""
    g = golden("tpspp_forward.npz")
    sd = O.trained_like_state(int(g["state_seed"]))
    m = T.TPS_PP().to(DEV).eval()
    m.load_state_dict(sd, strict=True)
    x, o0, o1 = O.synthetic_tpspp_inputs(int(g["batch"]), int(g["input_seed"]))
    with torch.no_grad():
        r = m(torch.from_numpy(x).to(DEV), [torch.from_numpy(o0).to(DEV), torch.from_numpy(o1).to(DEV)])
    assert set(r.keys()) == {"output", "logits", "mp_img", "pc_score"} and r["logits"] is None
    assert r["output"].shape == (2, 64, 16, 64) and r["mp_img"].shape == (2, 64, 16, 64)
    assert r["pc_score"].shape == (2, 1024, 32)
    assert mx(r["pc_score"], g["ref64_pc_score"]) <= 2e-4     # default head: tcgen05 3xTF32 (fp32 mode: 2e-5)
    floor_o = mx(g["ref32_output"], g["ref64_output"])
    floor_m = mx(g["ref32_mp_img"], g["ref64_mp_img"])
    e_o, e_m = mx(r["output"], g["ref64_output"]), mx(r["mp_img"], g["ref64_mp_img"])
    print(f"output |ours-ref64|={e_o:.3e} (ref32-ref64 floor {floor_o:.3e}); mp_img {e_m:.3e} (floor {floor_m:.3e})")
    assert e_o <= max(1e-5, FLOOR_K * floor_o)
    assert e_m <= max(1e-5, FLOOR_K * floor_m)


def test_tps_pp_bf16_mode_module_tolerance(golden, native_lib):
    """The module in its bf16 mode (bf16 operands + bf16 storage in the 3x3 convolutions, bf16 feat_grid into the warp): stated
    tolerance of the returned tensors against the reference's fp64 twin -- control points 1e-4, pc_score 0.15, the rectified
    feature maps 6e-2 of their range (mp_img samples the fp32 x with a grid that is within 0.5 source px: SURVEY F7)."""
    g = golden("tpspp_forward.npz")
    sd = O.trained_like_state(int(g["state_seed"]))
    m = T.TPS_PP().to(DEV).eval()
    m.load_state_dict(sd, strict=True)
    m.head_precision = N.HEAD_BF16
    x, o0, o1 = O.synthetic_tpspp_inputs(int(g["batch"]), int(g["input_seed"]))
    with torch.no_grad():
        r = m(torch.from_numpy(x).to(DEV), [torch.from_numpy(o0).to(DEV), torch.from_numpy(o1).to(DEV)])
    assert r["output"].dtype == torch.float32 and r["mp_img"].dtype == torch.float32
    assert mx(r["pc_score"], g["ref64_pc_score"]) <= 0.15
    for key in ("output", "mp_img"):
        ref = np.asarray(g["ref64_" + key])
        err = mx(r[key], ref)
        print(f"bf16 mode {key}: |ours - ref64| = {err:.3e} of range {float(np.abs(ref).max()):.2f}")
        assert err <= 6e-2 * float(np.abs(ref).max())


@pytest.mark.parametrize("weights", ["stock", "trained"])
@pytest.mark.parametrize("precision", ["tc", "fp32"])
def test_nrtr_argmax_proxy(golden, native_lib, weights, precision):
    """north_star "identical NRTR argmax decodes" / BASELINE config 1, on the GPU.  The fixture
    (oracle/make_golden.py::nrtr_fixture) holds what the reference backbone hands to ``tpsnet(x, outs)`` for a
    seeded 32x128 batch, the reference rectifier's fp32 ``output``, its fp64 twin, and ``safe_delta``: the largest
    perturbation of that output (uniform noise, several draws) under which the reference layer3-5 + NRTR greedy
    decode keeps every argmax.  The recogniser cannot travel to the GPU box, so the test asserts the sufficient
    condition ``|ours - ref32| <= safe_delta / 2`` -- and that we are at least as close to the exact (fp64) result
    as the reference's own fp32 path is.  (``|ours - ref32| <= 1e-4`` is not attainable by ANY independent
    implementation: on the stock weights the reference is 5.8e-4 away from its own fp64 twin, we are 4e-6 away.)"""
    from tps_pp_b200 import _native as N
    g = golden("nrtr_argmax.npz")
    if weights == "stock":
        torch.manual_seed(0)
        m = T.TPS_PP().to(DEV).eval()
    else:
        m = T.TPS_PP().to(DEV).eval()
        m.load_state_dict(O.trained_like_state(3), strict=True)
    keys = list(O.trained_like_state(3).keys()) if weights == "trained" else list(m.state_dict().keys())   # fixture order
    digest = np.array([float(m.state_dict()[k].double().abs().sum()) for k in keys])
    assert np.allclose(digest, g[f"{weights}_state_digest"], rtol=1e-6, atol=0), "fixture weights differ"   # (LAPACK inverse in the buffers)
    m.head_precision = N.HEAD_TC if precision == "tc" else N.HEAD_FP32
    x, o0, o1 = (torch.from_numpy(g[k]).to(DEV) for k in ("x", "o0", "o1"))
    with torch.no_grad():
        r = m(x, [o0, o1])
    assert all(m.native_stages.values())
    err32 = mx(r["output"], g[f"{weights}_ref_output"])
    err64 = mx(r["output"], g[f"{weights}_ref64_output"])
    floor = mx(g[f"{weights}_ref_output"], g[f"{weights}_ref64_output"])
    safe = float(g[f"{weights}_safe_delta"])
    print(f"nrtr proxy [{weights}/{precision}]: |ours - ref32| = {err32:.3e}, |ours - ref64| = {err64:.3e}, reference's own "
          f"|ref32 - ref64| = {floor:.3e}; decode-safe perturbation {safe:.0e}")
    assert safe >= 1e-3
    assert err32 <= 0.5 * safe
    assert err64 <= floor


def test_tps_pp_head_control_points(golden, native_lib):
    g = golden("tpspp_forward.npz")
    sd = O.trained_like_state(int(g["state_seed"]))
    m = T.TPS_PP().to(DEV).eval()
    m.load_state_dict(sd, strict=True)
    x, o0, o1 = O.synthetic_tpspp_inputs(int(g["batch"]), int(g["input_seed"]))
    with torch.no_grad():
        fg, cp, sc = m.head(torch.from_numpy(x).to(DEV), [torch.from_numpy(o0).to(DEV), torch.from_numpy(o1).to(DEV)])
    assert mx(cp, g["ref64_control_point"]) <= 1e-4          # north_star tolerance
    assert mx(cp, g["ref32_control_point"]) <= 1e-6
    assert mx(fg[:, ::16], g["ref32_feat_grid_ch"]) <= 5e-5


def test_tps_pp_random_init_matches_oracle(native_lib):
    """Stock initialisation (fc2.weight == 0): C' is the bias lattice, F5 coordinate quirk included."""
    torch.manual_seed(0)
    m = T.TPS_PP().to(DEV).eval()
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    x, o0, o1 = O.synthetic_tpspp_inputs(2, 5)
    with torch.no_grad():
        r = m(torch.from_numpy(x).to(DEV), [torch.from_numpy(o0).to(DEV), torch.from_numpy(o1).to(DEV)])
    r64 = O.tps_pp_forward(sd, x, [o0, o1], dtype=torch.float64, sampler="numpy")
    r32 = O.tps_pp_forward(sd, x, [o0, o1], dtype=torch.float32)
    floor = mx(r32["output"], r64["output"])
    assert mx(r["output"], r64["output"]) <= max(1e-5, FLOOR_K * floor)
    assert mx(r["mp_img"], r64["mp_img"]) <= max(1e-5, FLOOR_K * mx(r32["mp_img"], r64["mp_img"]))


@pytest.mark.parametrize("train_convs,batch", [("native", 4), ("native", 2), ("library", 2)])
def test_tps_pp_autograd_reaches_every_parameter(native_lib, train_convs, batch):
    """Training contract (SURVEY 8b): grads flow to batch_img, outs[*] and every parameter -- with the 14 ConvModules on the
    native forward/backward kernels (batch 4: all of them; batch 2: the deepest layers fall back to cuDNN) and on cuDNN."""
    sd = O.trained_like_state(3)
    m = T.TPS_PP().to(DEV)
    m.load_state_dict(sd, strict=True)
    m.train_convs = train_convs
    m.train_linears = train_convs            # the dense layers (CBAM, DGAB, localisation, score) follow the same switch
    x, o0, o1 = O.synthetic_tpspp_inputs(batch, 1)
    tx = torch.from_numpy(x).to(DEV).requires_grad_()
    t0 = torch.from_numpy(o0).to(DEV).requires_grad_()
    t1 = torch.from_numpy(o1).to(DEV).requires_grad_()
    r = m(tx, [t0, t1])
    ts = m.training_stages
    assert ts["convs_native"] + ts["convs_library"] == 14
    assert ts["linears_native" if train_convs == "native" else "linears_library"] == (16 if train_convs == "native" else 13), ts
    assert ts["linears_library" if train_convs == "native" else "linears_native"] == 0, ts
    if train_convs == "library":
        assert ts["convs_native"] == 0
    elif batch == 4:
        assert ts["convs_library"] == 0, ts
    else:
        assert ts["convs_native"] >= 10, ts
    r["output"].square().mean().backward()
    for name, p in m.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
    assert tx.grad is not None and t0.grad is not None and t1.grad is not None
    # against the oracle's torch-CPU autograd in fp64
    m64 = {k: v.double() for k, v in sd.items()}
    px = torch.from_numpy(x).double().requires_grad_()
    import torch.nn.functional as F
    st = {k: v.clone().requires_grad_(v.is_floating_point() and not k.startswith("atten_tps")) for k, v in m64.items()}

    def run():
        feat_cat, feat_grid = O.down_stage(st, px, torch.from_numpy(o0).double(), torch.from_numpy(o1).double())
        en, de = O.msfa(st, feat_cat)
        cp, score, _ = O.tpe(st, en, de)
        c = O.tpspp_constants()
        hat = torch.from_numpy(c["hat_C"]).double(); ph = torch.from_numpy(c["P_hat"]).double(); P = torch.from_numpy(c["P"]).double()
        B = cp.shape[0]
        phi = torch.cat([torch.ones(B, 1024, 1, dtype=torch.float64), P[None].repeat(B, 1, 1), ph[None] * (score * 0.5 + 1)], 2)
        Tm = torch.bmm(hat[None].repeat(B, 1, 1), torch.cat([cp, torch.zeros(B, 3, 2, dtype=torch.float64)], 1))
        grid = torch.bmm(phi, Tm).reshape(B, 16, 64, 2)
        return F.grid_sample(feat_grid, grid, padding_mode="border", align_corners=True)

    # _t() in the oracle detaches; patch it for this differentiable run
    orig = O._t
    O._t = lambda state, key, dtype: state[key]
    try:
        run().square().mean().backward()
    finally:
        O._t = orig
    worst = ("", 0.0)
    for name, p in m.named_parameters():
        ref = st[name].grad
        scale = max(float(ref.abs().max()), 1e-12)
        ratio = mx(p.grad, ref) / scale
        if ratio > worst[1]:
            worst = (name, ratio)
    print(f"autograd [{train_convs}, batch {batch}]: worst parameter-gradient error {worst[1]:.3e} of its scale ({worst[0]}); "
          f"d batch_img {mx(tx.grad, px.grad) / float(px.grad.abs().max()):.3e}")
    # fp32 head + the TPS solve's 1e2-1e3x rounding amplification (SURVEY F6) + ReLU masks that differ between an fp32 and an
    # fp64 forward at pixels within rounding of zero: percent-level agreement (each convolution alone is checked to 1e-4 in
    # tests/test_conv_train_gpu.py, and at the training batch in tests/test_train_batch_gpu.py)
    assert worst[1] <= 5e-2, worst
    assert mx(tx.grad, px.grad) <= 5e-2 * float(px.grad.abs().max())


def test_tps_preprocessor_like_reference_test(native_lib):
    """reference tests/test_models/test_ocr_preprocessor.py:19-29 (shape contract), on the GPU."""
    pre = T.TPSPreprocessor(num_fiducial=20, img_size=(32, 100), rectified_img_size=(32, 100), num_img_channel=1)
    pre.init_weights()
    pre.train()
    pre = pre.to(DEV)
    out = pre(torch.randn(1, 1, 32, 100, device=DEV))
    assert out.shape == torch.Size([1, 1, 32, 100])


def test_tps_preprocessor_vs_oracle(native_lib):
    torch.manual_seed(0)
    pre = T.TPSPreprocessor(20, (32, 100), (32, 100), 3).to(DEV).eval()
    with torch.no_grad():
        pre.LocalizationNetwork.localization_fc2.weight.normal_(0, 1e-2)
    sd = {k: v.detach().cpu() for k, v in pre.state_dict().items()}
    img = np.random.RandomState(0).standard_normal((3, 3, 32, 100)).astype(np.float32)
    with torch.no_grad():
        out = pre(torch.from_numpy(img).to(DEV))
        cp = pre.localize(torch.from_numpy(img).to(DEV))
    cpo = O.classical_localization(sd, torch.from_numpy(img))
    assert mx(cp, cpo) <= 1e-4
    cc = O.classical_constants(20, (32, 100))
    o64, _ = O.classical_warp(img, cp.cpu().numpy(), cc, (32, 100), dtype=np.float64)
    assert mx(out, o64) <= 1e-5


def test_large_shard_is_batch_independent(native_lib):
    """BASELINE config 5 (global batch 8192 = 1024 images per GPU on 8 GPUs): one shard-sized call must equal
    the same images pushed through in chunks -- images are independent, nothing may leak across the batch."""
    sd = O.trained_like_state(3)
    m = T.TPS_PP().to(DEV).eval()
    m.load_state_dict(sd, strict=True)
    B = 1024
    g = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn((B, 64, 16, 64), device=DEV, generator=g)
    o0 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
    o1 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
    with torch.no_grad():
        full = m(x, [o0, o1])
        out_full = full["output"].clone(); sc_full = full["pc_score"].clone()
        for lo in (0, 300, 1000):
            hi = min(B, lo + 24)
            part = m(x[lo:hi], [o0[lo:hi], o1[lo:hi]])
            assert torch.equal(part["output"], out_full[lo:hi])
            assert torch.equal(part["pc_score"], sc_full[lo:hi])
    assert torch.isfinite(out_full).all()


def test_training_step_launches_no_cudnn_or_cublas_kernel(native_lib):
    """VERDICT r01 item 4's criterion, driver-visible: with the 14 ConvModules on tpspp_convcat_fwd/bwd and the 16 dense
    layers on tpspp_linear_fwd/bwd, forward + backward of the rectifier launches no cuDNN / cuBLAS / CUTLASS kernel (CUPTI
    kernel names of one step; what remains next to the tpspp:: kernels are ATen element-wise / reduction kernels)."""
    from torch.profiler import profile, ProfilerActivity
    sd = O.trained_like_state(3)
    m = T.TPS_PP().to(DEV).train()
    m.load_state_dict(sd, strict=True)
    x, o0, o1 = O.synthetic_tpspp_inputs(4, 1)
    tx = torch.from_numpy(x).to(DEV).requires_grad_()
    t0, t1 = torch.from_numpy(o0).to(DEV).requires_grad_(), torch.from_numpy(o1).to(DEV).requires_grad_()
    for _ in range(2):                                   # warm-up (lazy initialisations), then the profiled step
        m(tx, [t0, t1])["output"].square().mean().backward()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m(tx, [t0, t1])["output"].square().mean().backward()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if e.self_device_time_total > 0]
    assert m.training_stages == {"convs_native": 14, "convs_library": 0, "linears_native": 16, "linears_library": 0}
    ours = [n for n in names if "tpspp::" in n]
    assert len(ours) >= 10, names
    bad = [n for n in names if any(t in n.lower() for t in ("cudnn", "cublas", "cutlass", "gemm", "implicit_convolve", "wgrad2d", "dgrad"))
           and "tpspp::" not in n]
    assert not bad, bad
