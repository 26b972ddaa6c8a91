"""The launch plan of the rectifier's native head (tpspp_head_fwd) and its fused warp, restated from the launchers, and pinned
to hand-worked values on 148 SMs (a B200).  tests/test_rectifier_batch_gpu.py calls the plan with the device's SM count: it
checks under the profiler that every case runs the kernels the plan names, and picks its batch-invariance windows and the
fp64 sample of its largest batch from the plan's pass boundaries.

``head_plan(B, sms, mode)`` lists the launches of one forward with cached weight images (no ``wprep_kernel``), in the order of
bench.py's ``_launch_names`` labels:
  * ``run_down_fused`` (csrc/head_tc.cu): B x 2h = 32 B row tiles over min(tiles, SMs) persistent CTAs;
  * ``run_conv_tc`` / ``conv_tma_plan``: the 3x3 layers whose output is a whole number of 128-pixel rectangles of one image
    (16 x 64: 8 tiles per image, 8 x 32: 2) run ``conv_tma_kernel<3, MODE, 64>`` persistently over min(tiles, 2 x SMs) CTAs;
    enc2 and dec0 (4 x 16 outputs) and enc3 (stride (2, 1), 2 x 16) do not fit a rectangle and run ``conv_ts_kernel<3, MODE>``
    with one CTA per 128 pixels, the last tile partial when B x pixels is not a multiple of 128;
  * ``cbam_kernel`` and ``loc_p1_kernel``: one CTA per image;
  * ``dgab_warp_kernel<16>``: one warp per (image, channel) plane, 16 warps per CTA, min(SMs, planes / 16) CTAs;
  * ``run_mlp_fused`` / ``run_score_fused``: B x 64 x 16 / 128 = 8 B row tiles (score: B x h / 2 = 8 B) over min(tiles, SMs);
  * the fused warp, ``warp_fwd_staged_kernel<true, S0BF>``: B x 64 planes; its grid comes from an occupancy query, so the plan
    gives its plane count only.
MODE is the operand mode of the 3x3 layers (csrc/head.cuh): CM_TF32X3 = 0 (``tc3x``), CM_BF16 = 1 (``bf16``), CM_MIX = 2
(``tc``, the default).  The ``fp32`` mode runs the CUDA-core kernels, one CTA per 128 output pixels (score_kernel: grid
(n / 128, B)), none of them persistent."""
import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402

H, W = 16, 64                 # x [B, 64, 16, 64]; o0 / o1 [B, 32, 32, 128]
MODES = {"tc": 2, "tc3x": 0, "bf16": 1}
DW_WARPS = 16                 # warps per dgab_warp_kernel CTA (csrc/head.cu)


def _cdiv(a, b):
    return -(-a // b)


def _launch(label, kernel, work, per_image, grid, per_pass=None):
    """work: tiles (or planes) of the launch; per_image: how many of them one image owns (None: a tile spans images)."""
    per_pass = per_pass or grid
    return dict(label=label, kernel=kernel, work=work, per_image=per_image, grid=grid, per_pass=per_pass,
                passes=work // per_pass, last=work % per_pass, persistent=work > per_pass, last_tile_px=None)


def _ts(label, kernel, B, px):
    """A non-persistent launch of one CTA per 128 output pixels; last_tile_px is the size of a partial last tile."""
    e = _launch(label, kernel, _cdiv(B * px, 128), None, _cdiv(B * px, 128))
    e["last_tile_px"] = (B * px) % 128 or None
    return e


def head_plan(B, sms, mode="tc"):
    """-> list of launches (dicts: label, kernel, work, per_image, grid, per_pass, passes, last, persistent, last_tile_px)."""
    if mode == "fp32":
        f3 = "conv_ffma_kernel<3>"
        plan = [_ts("down0", "conv_ffma_kernel<1>", B, 4 * H * W), _ts("down1", "conv_ffma_kernel<1>", B, 4 * H * W),
                _ts("down2", "conv_ffma_kernel<1>", B, H * W), _ts("down0_1", f3, B, H * W), _ts("down1_1", f3, B, H * W),
                _ts("down_feat", "conv_ffma_kernel<1>", B, 4 * H * W)]
    else:
        m = MODES[mode]
        tma, ts = f"conv_tma_kernel<3, {m}, 64>", f"conv_ts_kernel<3, {m}>"
        plan = [_launch(bench._DOWN[0][0], "down_fused_kernel", B * 2 * H, 2 * H, min(B * 2 * H, sms)),
                _launch("down0_1", tma, 8 * B, 8, min(8 * B, 2 * sms)), _launch("down1_1", tma, 8 * B, 8, min(8 * B, 2 * sms))]
    if mode == "fp32":
        f3 = "conv_ffma_kernel<3>"
        enc = [_ts("enc0", f3, B, H * W), _ts("enc1", f3, B, 256), _ts("enc2", f3, B, 64), _ts("enc3", f3, B, 32)]
        dec = [_ts("dec0", f3, B, 64), _ts("dec1", f3, B, 256), _ts("dec2", f3, B, H * W), _ts("dec3", f3, B, H * W)]
    else:
        enc = [_launch("enc0", tma, 8 * B, 8, min(8 * B, 2 * sms)), _launch("enc1", tma, 2 * B, 2, min(2 * B, 2 * sms)),
               _ts("enc2", ts, B, 64), _ts("enc3", ts, B, 32)]
        dec = [_ts("dec0", ts, B, 64), _launch("dec1", tma, 2 * B, 2, min(2 * B, 2 * sms)),
               _launch("dec2", tma, 8 * B, 8, min(8 * B, 2 * sms)), _launch("dec3", tma, 8 * B, 8, min(8 * B, 2 * sms))]
    dg = min(sms, _cdiv(64 * B, DW_WARPS))
    plan += enc + [_launch("cbam", "cbam_kernel", B, 1, B)] + dec + [
        _launch("localization+p_linear", "loc_p1_kernel", B, 1, B),
        _launch("dgab_gate", "dgab_warp_kernel<16>", 64 * B, 64, dg, dg * DW_WARPS)]
    if mode == "fp32":
        plan += [_ts("mlp_fused", "dgab_mlp_kernel", B, 64 * H), _launch("score", "score_kernel", 8 * B, 8, 8 * B)]
    else:
        plan += [_launch("mlp_fused", "mlp_fused_kernel", 8 * B, 8, min(8 * B, sms)),
                 _launch(bench._SCORE[0][0], "score_fused_kernel", 8 * B, 8, min(8 * B, sms))]
    warp = f"warp_fwd_staged_kernel<true, {'true' if mode == 'bf16' else 'false'}>"
    plan.append(dict(label="fused_warp", kernel=warp, work=64 * B, per_image=64, grid=None, per_pass=None, passes=None,
                     last=None, persistent=None, last_tile_px=None))
    return plan


def pass_images(e, k):
    """The images whose tiles (planes) launch e hands out in its pass k (0-based)."""
    lo, hi = k * e["per_pass"], min((k + 1) * e["per_pass"], e["work"])
    return range(lo // e["per_image"], (hi - 1) // e["per_image"] + 1)


def last_pass(e):
    return e["passes"] if e["last"] else e["passes"] - 1


# The batches of tests/test_rectifier_batch_gpu.py: (mode, B)
CASES = {"tc-256": ("tc", 256), "tc3x-256": ("tc3x", 256), "bf16-256": ("bf16", 256), "fp32-256": ("fp32", 256),
         "tc-683": ("tc", 683), "tc-1024": ("tc", 1024), "tc-2048": ("tc", 2048), "stage-256": ("tc", 256)}


def batch_sample(B, sms, mode="tc"):
    """The images of a large batch compared with fp64: the first and last 8, and for every persistent launch the images its
    first wrap-around (pass 1) and its last pass reach."""
    keep = set(range(8)) | set(range(B - 8, B))
    for e in head_plan(B, sms, mode):
        if e["persistent"]:
            keep |= set(pass_images(e, 1)) | set(pass_images(e, last_pass(e)))
    return sorted(keep)


def window_starts(B, sms, mode="tc"):
    """Starts of the 8-image batch-invariance windows: the first and last images, and 4 images before the image where
    down_fused_kernel, conv_tma_kernel (8 tiles per image) and score_fused_kernel begin their second and last passes."""
    starts = {0, B - 8}
    plan = {e["label"]: e for e in head_plan(B, sms, mode)}
    for lab in (bench._DOWN[0][0], "enc0", bench._SCORE[0][0]):
        e = plan.get(lab)             # (the fp32 mode has no fused down / score kernel)
        if e and e["persistent"]:
            for k in (1, last_pass(e)):
                starts.add(min(max(0, pass_images(e, k)[0] - 4), B - 8))
    return sorted(starts)


# (B) -> (work, grid, full passes, last partial pass) on 148 SMs, worked by hand, per label of the default (tc) mode
HAND = {
    8: {"down_fused": (256, 148, 1, 108), "down0_1": (64, 64, 1, 0), "enc1": (16, 16, 1, 0), "enc2": (4, 4, 1, 0),
        "enc3": (2, 2, 1, 0), "dgab_gate": (512, 32, 1, 0), "mlp_fused": (64, 64, 1, 0)},
    256: {"down_fused": (8192, 148, 55, 52), "down0_1": (2048, 296, 6, 272), "enc1": (512, 296, 1, 216),
          "enc2": (128, 128, 1, 0), "enc3": (64, 64, 1, 0), "dgab_gate": (16384, 148, 6, 2176), "mlp_fused": (2048, 148, 13, 124)},
    683: {"down_fused": (21856, 148, 147, 100), "down0_1": (5464, 296, 18, 136), "enc1": (1366, 296, 4, 182),
          "enc2": (342, 342, 1, 0), "enc3": (171, 171, 1, 0), "dgab_gate": (43712, 148, 18, 1088), "mlp_fused": (5464, 148, 36, 136)},
    1024: {"down_fused": (32768, 148, 221, 60), "down0_1": (8192, 296, 27, 200), "enc1": (2048, 296, 6, 272),
           "enc2": (512, 512, 1, 0), "enc3": (256, 256, 1, 0), "dgab_gate": (65536, 148, 27, 1600), "mlp_fused": (8192, 148, 55, 52)},
    2048: {"down_fused": (65536, 148, 442, 120), "down0_1": (16384, 296, 55, 104), "enc1": (4096, 296, 13, 248),
           "enc2": (1024, 1024, 1, 0), "enc3": (512, 512, 1, 0), "dgab_gate": (131072, 148, 55, 832), "mlp_fused": (16384, 148, 110, 104)},
}


@pytest.mark.parametrize("B", sorted(HAND))
def test_head_plan_on_148_sms(B):
    plan = {e["label"].split("(")[0]: e for e in head_plan(B, 148)}
    for lab, want in HAND[B].items():
        e = plan[lab]
        assert (e["work"], e["grid"], e["passes"], e["last"]) == want, (B, lab)
    # the launches that share a rule with a pinned one
    for a, b in (("down1_1", "down0_1"), ("enc0", "down0_1"), ("dec2", "down0_1"), ("dec3", "down0_1"), ("dec1", "enc1"),
                 ("dec0", "enc2"), ("score_fused", "mlp_fused")):
        assert [plan[a][k] for k in ("work", "grid", "passes", "last")] == [plan[b][k] for k in ("work", "grid", "passes", "last")]
    assert plan["cbam"]["grid"] == plan["localization+p_linear"]["grid"] == B
    assert plan["fused_warp"]["work"] == 64 * B
    # dgab: 16 warps per CTA, so a pass is 148 x 16 = 2368 planes (37 images) once 64 B / 16 > 148
    assert plan["dgab_gate"]["per_pass"] == (2368 if B >= 37 else 64 * B)


def test_conv_ts_partial_tiles():
    """enc2 / dec0 (64 pixels per image) end on a half tile when B is odd, enc3 (32 pixels) when B % 4 != 0."""
    for B, enc2, enc3 in ((256, None, None), (683, 64, 96), (1024, None, None), (2048, None, None), (7, 64, 96), (6, None, 64)):
        plan = {e["label"]: e for e in head_plan(B, 148)}
        assert plan["enc2"]["last_tile_px"] == plan["dec0"]["last_tile_px"] == enc2, B
        assert plan["enc3"]["last_tile_px"] == enc3, B
        assert plan["enc2"]["kernel"] == plan["enc3"]["kernel"] == plan["dec0"]["kernel"] == "conv_ts_kernel<3, 2>"


@pytest.mark.parametrize("mode", ["tc", "tc3x", "bf16"])
def test_plan_lines_up_with_bench_labels(mode):
    """bench.py's roofline_dominant picks a launch by its label: the plan (+ the warp) must have as many launches as the label
    list bench derives from the launch count, and the same labels in the same order."""
    plan = head_plan(256, 148, mode)
    assert [e["label"] for e in plan] == bench._launch_names(len(plan))
    assert bench._launch_names(len(plan) + 1) == ["wprep"] + [e["label"] for e in plan]
    assert [e["kernel"] for e in plan if e["label"] == "enc0"] == [f"conv_tma_kernel<3, {MODES[mode]}, 64>"]


def test_fp32_plan_has_no_persistent_kernel_but_dgab():
    plan = head_plan(256, 148, "fp32")
    assert len(plan) == 20 and [e["label"] for e in plan if e["persistent"]] == ["dgab_gate"]
    score = plan[-2]
    assert score["kernel"] == "score_kernel" and score["grid"] == 8 * 256     # grid (1024 / 128, B)


def test_batch_sample_and_windows():
    s = batch_sample(2048, 148)
    assert len(s) >= 256 and s[:8] == list(range(8)) and s[-8:] == list(range(2040, 2048))
    plan = {e["label"]: e for e in head_plan(2048, 148)}
    # conv_tma_kernel for the 16 x 64 layers wraps at tile 296 = image 37 and starts its last pass at tile 16280 = image 2035
    assert pass_images(plan["enc0"], 1)[0] == 37 and pass_images(plan["enc0"], last_pass(plan["enc0"]))[0] == 2035
    assert {37, 2035, 148, 1924} <= set(s)                 # enc1 / dec1 (2 tiles per image): images 148 and 1924
    # down_fused: pass 1 at image 4 (window 0), last pass at image 254; conv_tma: 37 and 222; score_fused: 18 and 240
    assert window_starts(256, 148) == [0, 14, 33, 218, 236, 248]


def test_cases_cover_every_branch():
    """The GPU cases together: more than one pass of every persistent head kernel, a partial last pass of each, a partial
    last conv_ts_kernel tile, all four head modes at B = 256 and the bf16-feat_grid warp."""
    multi, partial, ts_partial, modes = set(), set(), False, set()
    for mode, B in CASES.values():
        for e in head_plan(B, 148, mode):
            if e["persistent"]:
                multi.add(e["kernel"])
            if e["last"]:
                partial.add(e["kernel"])
            ts_partial |= e["kernel"].startswith("conv_ts") and e["last_tile_px"] is not None
        if B == 256:
            modes.add(mode)
    persistent_kernels = {"down_fused_kernel", "conv_tma_kernel<3, 2, 64>", "conv_tma_kernel<3, 0, 64>", "conv_tma_kernel<3, 1, 64>",
                          "dgab_warp_kernel<16>", "mlp_fused_kernel", "score_fused_kernel"}
    assert persistent_kernels <= multi and persistent_kernels <= partial
    assert ts_partial and modes == {"tc", "tc3x", "bf16", "fp32"}
    assert "warp_fwd_staged_kernel<true, true>" in {head_plan(B, 148, m)[-1]["kernel"] for m, B in CASES.values()}
