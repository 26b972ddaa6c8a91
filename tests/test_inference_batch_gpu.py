"""GPU: the inference paths bench.py times at large batches, against fp64 torch on the device at those batches.

How these kernels split work changes with the batch, and the other tests run them at small ones:

  * classical warp (BASELINE config 4: 64x256x3, F = 20 / 40, B = 1024).  AUTO takes the P_hat-stationary kernel from
    B x pixels >= 4 Mi.  Its batch slices (one resident wave: ~172 images each at B = 1024 on 148 SMs, 3 CTAs per SM) stream
    T in groups of 16 images through a two-buffer bulk-copy ring; at B = 64 a slice holds one group and the ring never turns
    over.  B = 1021 adds a short last slice, a short last group and a last pass of aliased images.
  * classical localisation network (tpspp_locnet_fwd) at B = 1024 / 1027: the stem and max-pool grid-stride loops make ~14
    and ~55 passes, every persistent convolution CTA walks ~110 tiles, and locnet_fc_kernel runs full 8-image CTAs before a
    partial tail (B = 1027: 3 images).
  * backbone stage (tpspp_stage_fwd) at B = 256 / 259: stem_kernel makes four grid-stride passes, the 32-channel
    convolutions ~28 tiles per CTA.

The fp64 references are the oracle's functions restated with device tensors (the oracle runs on host cores, too slow in fp64
for 1024 localisation networks); each is pinned to its oracle function on a few images first."""
import contextlib
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bench
import tps_pp_b200 as T
from oracle import tpspp_oracle as O
from tps_pp_b200 import _native as N
from tps_pp_b200 import functional as TF

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))        # the weight builders beside these tests
from test_locnet_gpu import _trained_like  # noqa: E402
from test_stage_gpu import _backbone  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PIX_TOL = 1e-5             # rectified pixels (test_warp_gpu.py)
TILED_VS_GENERIC = 2e-6    # the two classical kernels (test_warp_gpu.py)
PIN_TOL = 1e-10            # device reference against its oracle function, both fp64
RS = (64, 256)             # rectified size of BASELINE config 4
SLICE = 172                # images per batch slice of the tiled warp at B = 1024 (148 SMs x 3 CTAs / 64 pixel tiles)


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def mx(a, b):
    return float((a.double() - b.double()).abs().max())


def _worst(diff):
    """(max |diff|, image, (c, y, x)) of a [B, C, H, W] absolute difference."""
    per = diff.flatten(1).amax(1)
    b = int(per.argmax())
    pos = tuple(int(i) for i in np.unravel_index(int(diff[b].argmax()), tuple(diff.shape[1:])))
    return float(per[b]), b, pos


@contextlib.contextmanager
def _true_fp32():
    """The fp32 twin: cuDNN and cuBLAS without TF32 (the reference's numerics)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            yield
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


# ---------------------------------------------------------------- device references
def _classical_ref(img, cp, inv, ph, dtype):
    """O.classical_warp: grid = P_hat . (inv_delta_C[:, :F] . C'), then grid_sample (border, align_corners=True)."""
    b, f = cp.shape[:2]
    tm = torch.matmul(inv.to(dtype)[:, :f], cp.to(dtype))
    grid = torch.matmul(ph.to(dtype), tm).view(b, RS[0], RS[1], 2)
    return F.grid_sample(img.to(dtype), grid, padding_mode="border", align_corners=True)


def _locnet_one(sd, img, dtype):
    """O.classical_localization (eval-mode BatchNorm) on device tensors."""
    def w(k):
        return sd["LocalizationNetwork." + k].to(dtype)
    x = img.to(dtype)
    for ci, bi, pool in ((0, 1, True), (4, 5, True), (8, 9, True), (12, 13, False)):
        x = F.conv2d(x, w(f"conv.{ci}.weight"), None, 1, 1)
        x = F.batch_norm(x, w(f"conv.{bi}.running_mean"), w(f"conv.{bi}.running_var"), w(f"conv.{bi}.weight"),
                         w(f"conv.{bi}.bias"), False, 0.0, 1e-5)
        x = F.relu(x)
        if pool:
            x = F.max_pool2d(x, 2, 2)
    x = x.mean(dim=(2, 3))
    x = F.relu(F.linear(x, w("localization_fc1.0.weight"), w("localization_fc1.0.bias")))
    x = F.linear(x, w("localization_fc2.weight"), w("localization_fc2.bias"))
    return x.view(x.shape[0], -1, 2)


def _locnet_ref(sd, img, dtype, step=128):
    """In slices: the first fp64 activation of 1024 images at 64x256 is 8.6 GB."""
    return torch.cat([_locnet_one(sd, img[i:i + step], dtype) for i in range(0, img.shape[0], step)])


def _stage_ref(sd, img, dtype):
    """O.backbone_stage_forward on device tensors -> (x, [o0, o1])."""
    def t(k):
        return sd[k].to(DEV, dtype)

    def bn(p, x):
        return F.batch_norm(x, t(p + ".running_mean"), t(p + ".running_var"), t(p + ".weight"), t(p + ".bias"), False, 0.0,
                            O.BN_EPS)
    x = F.relu(bn("bn1", F.conv2d(img.to(dtype), t("conv1.weight"), t("conv1.bias"), padding=1)))
    outs = []
    for layer, blocks, _, _, stride in O.BACKBONE_STAGE_LAYERS:
        outs.append(x)
        for i in range(blocks):
            p = f"{layer}.{i}."
            s = stride if i == 0 else 1
            out = F.relu(bn(p + "bn1", F.conv2d(x, t(p + "conv1.weight"))))
            out = bn(p + "bn2", F.conv2d(out, t(p + "conv2.weight"), stride=s, padding=1))
            idn = x
            if (p + "downsample.0.weight") in sd:
                idn = bn(p + "downsample.1", F.conv2d(x, t(p + "downsample.0.weight"), stride=s))
            x = F.relu(out + idn)
    return x, outs


# ---------------------------------------------------------------- inputs
def _classical_inputs(f, batch):
    """The exact tensors `bench.py --workload classical64x256` times."""
    img, cp, inv, ph = bench._classical_inputs(f, batch, DEV, 1234)
    return img, cp.to(DEV), inv.to(DEV), ph.to(DEV)


def _warp(img, cp, inv, ph, variant=N.VARIANT_AUTO):
    return TF.tps_warp(img, None, cp, None, ph, None, inv, RS, mode=N.MODE_CLASSICAL, theta=0.0, variant=variant)[0]


def _preprocessor(chans, h, w, f):
    m = _trained_like(T.TPSPreprocessor(num_fiducial=f, img_size=(h, w), rectified_img_size=(h, w), num_img_channel=chans), 11 + f)
    m = m.to(DEV).eval()
    assert float(m.LocalizationNetwork.localization_fc2.weight.detach().abs().max()) > 0    # else C' is the fc2 bias whatever the convs do
    return m


def _state(m):
    return {k: v.detach() for k, v in m.state_dict().items()}


def _images(n, chans, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn((n, chans, h, w), device=DEV, generator=g)


# ---------------------------------------------------------------- the references against the oracle
def test_classical_reference_matches_oracle(native_lib):
    img, cp, inv, ph = bench._classical_inputs(40, 3, DEV, 5)
    o64, _ = O.classical_warp(img.cpu().numpy(), cp.numpy(), dict(inv_delta_C=inv.numpy(), P_hat=ph.numpy()), RS,
                              dtype=np.float64)
    got = _classical_ref(img, cp.to(DEV), inv.to(DEV), ph.to(DEV), torch.float64)
    e = rel(got, o64)
    print(f"classical reference vs oracle (fp64, 3 images): rel {e:.1e} (tol {PIN_TOL:.0e})")
    assert e <= PIN_TOL


def test_locnet_reference_matches_oracle(native_lib):
    m = _preprocessor(3, 64, 256, 20)
    img = _images(2, 3, 64, 256, 3)
    sd = _state(m)
    ref = O.classical_localization({k: (v.cpu().double() if v.is_floating_point() else v.cpu()) for k, v in sd.items()},
                                   img.cpu().double())
    e = rel(_locnet_ref(sd, img, torch.float64), ref)
    print(f"localisation reference vs oracle (fp64, 2 images): rel {e:.1e} (tol {PIN_TOL:.0e})")
    assert e <= PIN_TOL


def test_stage_reference_matches_oracle(native_lib):
    _, sd = _backbone()
    img = O.synthetic_images(2, 8)
    x64, outs64 = O.backbone_stage_forward(sd, img, torch.float64)
    x, outs = _stage_ref(sd, torch.from_numpy(img).to(DEV), torch.float64)
    e = max(rel(x, x64), rel(outs[0], outs64[0]), rel(outs[1], outs64[1]))
    print(f"stage reference vs oracle (fp64, 2 images): rel {e:.1e} (tol {PIN_TOL:.0e})")
    assert e <= PIN_TOL


# ---------------------------------------------------------------- 1. classical warp at BASELINE config 4
@pytest.mark.parametrize("batch", [1024, 1021])
@pytest.mark.parametrize("f", [20, 40])
def test_classical_warp_matches_fp64_at_bench_batch(native_lib, f, batch):
    """Every image of the bench's batch within PIX_TOL of fp64, the tiled kernel against the per-pixel one, run to run."""
    img, cp, inv, ph = _classical_inputs(f, batch)
    out = _warp(img, cp, inv, ph)
    assert N.last_launch_count() == 2          # classical_T_kernel + the P_hat-stationary kernel
    again = _warp(img, cp, inv, ph)
    gen = _warp(img, cp, inv, ph, N.VARIANT_GENERIC)
    assert N.last_launch_count() == 1
    ref64 = _classical_ref(img, cp, inv, ph, torch.float64)
    with _true_fp32():
        floor = mx(_classical_ref(img, cp, inv, ph, torch.float32), ref64)
    err, b, pos = _worst((out.double() - ref64).abs())
    d_gen = mx(out, gen)
    print(f"classical warp [F={f}, B={batch}]: {err:.2e} (tol {PIX_TOL:.0e}, fp32 floor {floor:.2e}) worst image {b} at "
          f"{pos}; tiled - generic {d_gen:.2e} (tol {TILED_VS_GENERIC:.0e})")
    assert err <= PIX_TOL, (b, pos)
    assert d_gen <= TILED_VS_GENERIC
    assert torch.equal(out, again)


@pytest.mark.parametrize("f", [20, 40])
def test_classical_warp_is_batch_invariant(native_lib, f):
    """A pixel's grid (T from classical_T_kernel, one fp64 chain over P_hat) and taps do not depend on the slice, group or
    pass its image lands in: 8-image windows of the B = 1024 call -- at the start and end, across slice boundaries and
    across the last (short) group of a slice -- give the bits of a tiled call on those 8 images alone."""
    B = 1024
    img, cp, inv, ph = _classical_inputs(f, B)
    out = _warp(img, cp, inv, ph)
    assert N.last_launch_count() == 2
    starts = [0, 12, SLICE - 4, 2 * SLICE - 4, 3 * SLICE + 156, 5 * SLICE - 4, B - 8]
    for lo in starts:
        part = _warp(img[lo:lo + 8], cp[lo:lo + 8], inv, ph, N.VARIANT_TILED)      # AUTO would take the per-pixel kernel
        assert N.last_launch_count() == 2
        assert torch.equal(out[lo:lo + 8], part), lo


# ---------------------------------------------------------------- 2. classical localisation network
LOC_CASES = [(3, 64, 256, 20, (1024, 1027)), (3, 64, 256, 40, (1024, 1027)), (1, 64, 128, 40, (1024,))]


@pytest.mark.parametrize("chans,h,w,f,batches", LOC_CASES, ids=[f"{c}x{h}x{w}-F{f}" for c, h, w, f, _ in LOC_CASES])
def test_locnet_matches_fp64_at_bench_batch(native_lib, chans, h, w, f, batches):
    """C' of every image within max(1e-5, 4 |ref32 - ref64|) of fp64 (the rule of test_locnet_vs_oracle_fp64)."""
    m = _preprocessor(chans, h, w, f)
    img = _images(max(batches), chans, h, w, 7 * f + w)
    sd = _state(m)
    ref64 = _locnet_ref(sd, img, torch.float64)
    with _true_fp32():
        ref32 = _locnet_ref(sd, img, torch.float32)
    for batch in batches:
        with torch.no_grad():
            cp = m.localize(img[:batch])
        assert m._last_locnet_native
        per = (cp.double() - ref64[:batch]).abs().flatten(1).amax(1)
        worst = int(per.argmax())
        floor = mx(ref32[:batch], ref64[:batch])
        tol = max(1e-5, 4 * floor)
        print(f"locnet [{chans}x{h}x{w}, F={f}, B={batch}]: |C' - ref64| {float(per[worst]):.2e} (tol {tol:.2e}, fp32 floor "
              f"{floor:.2e}) worst image {worst}")
        assert float(per[worst]) <= tol, worst


def test_locnet_sees_one_tile_and_keeps_images_apart(native_lib):
    """C' comes after an average pool and two dense layers: show the comparison above can see one tile of one late image,
    that nothing leaks into the other images, and that images come out of a B = 1024 call with the bits of a B = 8 call."""
    B, hit = 1024, 1000
    m = _preprocessor(3, 64, 256, 20)
    img = _images(B, 3, 64, 256, 21)
    sd = _state(m)
    ref64 = _locnet_ref(sd, img[896:], torch.float64)
    with _true_fp32():
        tol = max(1e-5, 4 * mx(_locnet_ref(sd, img[896:], torch.float32), ref64))
    # input rows 8..11 x columns 128..255: one 2 x 64 tile of the block-2 convolution at 32 x 128.  The fp64 reference moves
    # C' by ~1e-3 for noise of amplitude 4 there and ~3.5e-3 for 10 (most of it is averaged away by the pool)
    noisy = img.clone()
    g = torch.Generator(device=DEV).manual_seed(77)
    noisy[hit, :, 8:12, 128:256] += 10.0 * torch.randn((3, 4, 128), device=DEV, generator=g)
    with torch.no_grad():
        base = m.localize(img)
        again = m.localize(img)
        moved = m.localize(noisy)
        small = {lo: m.localize(img[lo:lo + 8]) for lo in (0, B - 8)}
        back = m.localize(img)              # 1024 -> 8 -> 1024: the batch is part of the workspace stamp, weights re-prepared
    shift = float((moved[hit] - base[hit]).abs().max())
    print(f"locnet one-tile change of image {hit}: C' moves {shift:.2e} = {shift / tol:.0f} x the tolerance {tol:.2e} "
          f"(needs > 100 x)")
    assert shift > 100 * tol
    keep = torch.ones(B, dtype=torch.bool, device=DEV)
    keep[hit] = False
    assert torch.equal(moved[keep], base[keep])
    assert torch.equal(again, base)
    for lo, part in small.items():
        assert torch.equal(part, base[lo:lo + 8]), lo
    assert torch.equal(back, base)


def test_preprocessor_forward_at_bench_batch(native_lib):
    """The whole module at B = 1024: its rectified images against the fp64 warp of its own C' (decouples the two kernels)."""
    m = _preprocessor(3, 64, 256, 20)
    img = _images(1024, 3, 64, 256, 5)
    with torch.no_grad():
        out = m(img)
        assert N.last_launch_count() == 2 and m._last_locnet_native
        cp = m.localize(img)
    gen = m.GridGenerator
    err, b, pos = _worst((out.double() - _classical_ref(img, cp, gen.inv_delta_C, gen.P_hat, torch.float64)).abs())
    print(f"TPSPreprocessor.forward [B=1024]: {err:.2e} (tol {PIX_TOL:.0e}) worst image {b} at {pos}")
    assert err <= PIX_TOL, (b, pos)


# ---------------------------------------------------------------- 3. backbone stage
@pytest.mark.parametrize("batch", [256, 259])
def test_stage_matches_fp64_at_bench_batch(native_lib, batch):
    """o0, o1 and x within 4 |ref32 - ref64| + 5e-5 max(scale, 1) of fp64 (the rule of test_stage_vs_oracle), bit-equal
    run to run, and images [0:8] / [B-8:B] bit-equal to a B = 8 call."""
    m, sd = _backbone()
    img = torch.from_numpy(O.synthetic_images(batch, 1234)).to(DEV)
    params = m.stage_tensors()
    with torch.no_grad():
        got = TF.stage_forward(img, params)[:3]
        again = TF.stage_forward(img, params)[:3]
        small = {lo: TF.stage_forward(img[lo:lo + 8], params)[:3] for lo in (0, batch - 8)}
    x64, outs64 = _stage_ref(sd, img, torch.float64)
    with _true_fp32():
        x32, outs32 = _stage_ref(sd, img, torch.float32)
    over = []
    for name, a, r32, r64 in zip(("o0", "o1", "x"), got, outs32 + [x32], outs64 + [x64]):
        scale = float(r64.abs().max())
        floor = mx(r32, r64)
        tol = 4 * floor + 5e-5 * max(scale, 1.0)
        err, b, pos = _worst((a.double() - r64).abs())
        print(f"stage {name} [B={batch}]: {err:.2e} (tol {tol:.2e}, fp32 floor {floor:.2e}, scale {scale:.2f}) "
              f"worst image {b} at {pos}")
        if err > tol:
            over.append((name, err, tol, b, pos))
    assert not over, over
    for a, b in zip(got, again):
        assert torch.equal(a, b)
    for lo, part in small.items():
        for a, b in zip(got, part):
            assert torch.equal(a[lo:lo + 8], b), lo


def test_backbone_stage_module_across_batch_changes(native_lib):
    """ResNetABI_v2_large.stage at 256 -> 8 -> 256 (the workspace and its prepared weights re-used and re-stamped)."""
    m, _ = _backbone()
    img = torch.from_numpy(O.synthetic_images(256, 77)).to(DEV)
    with torch.no_grad():
        x0, outs0 = m.stage(img)
        assert m._last_stage_native
        x8, outs8 = m.stage(img[:8])
        x1, outs1 = m.stage(img)
    for a, b, c in zip([x0] + outs0, [x1] + outs1, [x8] + outs8):
        assert torch.equal(a, b)
        assert torch.equal(a[:8], c)
