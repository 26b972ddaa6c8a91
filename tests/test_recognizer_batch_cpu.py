"""The dispatch rule of the dense layers and the decode attention, restated from the launchers, and pinned to hand-worked
values on 148 SMs (a B200).  tests/test_recognizer_batch_gpu.py calls the rule with the device's SM count, asserts that its
cases cover every branch, and checks under the profiler that each case runs the kernels the rule names.

``lin_plan`` restates, for a tensor-core call of ``tpspp_linear_fwd`` / ``tpspp_linear_ln_fwd`` (rows % 128 == 0, one weight):
  * ``lin_dims`` (csrc/linear_train.cu): split-K doubles up to 4 while (row tiles x column blocks) x 2 x split fits 2 CTAs per
    SM, the 32-column K chunks divide evenly and each split keeps at least two of them -- only for K >= 256;
  * ``lin_tma_plan`` + ``run_conv_tc`` (csrc/head_tc.cu): with more than two K chunks and several column blocks each CTA owns
    one column block (grid.y) and walks row tiles persistently over grid.x = min(tiles, 2 x SMs / blocks) CTAs;
  * behind the tensor-core kernel: ``lin_reduce_ln_kernel<PER, SPLITS>`` when a LayerNorm output is asked for (SPLITS = 0
    on an unsplit call), else ``lin_splitk_reduce_kernel`` on a split call; each with its grid-stride loop.
``attn_decode_plan`` restates ``tpspp_attn_decode``'s choice of ``attn_decode_kernel<true>`` (evict-first loads) when one
call's keys and values exceed the 126 MB L2."""
import pytest

LRL_WARPS = 4


def lin_plan(rows, k, n, sms, ln=False):
    """-> dict(splitk, col_split, grid (x, y, z), tiles_per_cta, reduce (kernel name or None), reduce_splits, reduce_passes)."""
    assert rows % 128 == 0 and rows > 0 and k % 32 == 0 and n % 32 == 0, "tensor-core shapes only"
    nt = 64 if n % 64 == 0 else 32
    tiles, blocks, chunks = rows // 128, n // nt, k // 32
    sk = 1
    if k >= 256:
        while sk < 4 and tiles * blocks * sk * 2 <= 2 * sms and chunks % (sk * 2) == 0 and chunks // (sk * 2) >= 2:
            sk *= 2
    col_split = chunks > 2 and blocks != 1
    gx = min(tiles, max(1, 2 * sms // blocks)) if col_split else min(tiles, 2 * sms)
    plan = dict(splitk=sk, col_split=col_split, grid=(gx, blocks if col_split else 1, sk), tiles_per_cta=-(-tiles // gx),
                reduce=None, reduce_splits=None, reduce_passes=0)
    if ln:
        grid = min(-(-rows // LRL_WARPS), 8 * sms)
        per = n // 128
        per = 2 if per <= 2 else 4 if per <= 4 else 8
        plan.update(reduce=f"lin_reduce_ln_kernel<{per}, {0 if sk == 1 else sk}>", reduce_splits=0 if sk == 1 else sk,
                    reduce_passes=-(-rows // (LRL_WARPS * grid)))
    elif sk > 1:
        total4 = rows * n // 4
        grid = min(-(-total4 // 256), 4 * sms)
        plan.update(reduce="lin_splitk_reduce_kernel", reduce_splits=sk, reduce_passes=-(-total4 // (256 * grid)))
    return plan


def attn_decode_plan(batch, heads, kv_len):
    """The instantiation ``tpspp_attn_decode`` launches: streaming loads when batch x heads x kv_len keys and values (256 bytes
    each) exceed the L2."""
    return "attn_decode_kernel<true>" if batch * heads * kv_len * 2 * 64 * 4 > (126 << 20) else "attn_decode_kernel<false>"


def encoder_rows(n):
    return (n * 64 + 127) // 128 * 128


def decoder_rows(n):
    return (n + 127) // 128 * 128


# (rows, K, N, ln) -> (splitk, grid, tiles per CTA, reduce kernel, reduce passes), worked by hand on 148 SMs
HAND = [
    # encoder q|k|v 512 -> 1536 (24 blocks, grid.x <= 12)
    ((256, 512, 1536, False), (4, (2, 24, 4), 1, "lin_splitk_reduce_kernel", 1)),
    ((384, 512, 1536, False), (4, (3, 24, 4), 1, "lin_splitk_reduce_kernel", 1)),
    ((768, 512, 1536, False), (2, (6, 24, 2), 1, "lin_splitk_reduce_kernel", 2)),
    ((896, 512, 1536, False), (1, (7, 24, 1), 1, None, 0)),
    ((16384, 512, 1536, False), (1, (12, 24, 1), 11, None, 0)),
    ((65536, 512, 1536, False), (1, (12, 24, 1), 43, None, 0)),
    # encoder fc / w_2 with the residual and the next LayerNorm (8 blocks, grid.x <= 37)
    ((256, 512, 512, True), (4, (2, 8, 4), 1, "lin_reduce_ln_kernel<4, 4>", 1)),
    ((2304, 512, 512, True), (2, (18, 8, 2), 1, "lin_reduce_ln_kernel<4, 2>", 1)),
    ((2432, 512, 512, True), (1, (19, 8, 1), 1, "lin_reduce_ln_kernel<4, 0>", 1)),
    ((2816, 256, 512, True), (1, (22, 8, 1), 1, "lin_reduce_ln_kernel<4, 0>", 1)),
    ((16384, 512, 512, True), (1, (37, 8, 1), 4, "lin_reduce_ln_kernel<4, 0>", 4)),
    ((65536, 256, 512, True), (1, (37, 8, 1), 14, "lin_reduce_ln_kernel<4, 0>", 14)),
    # encoder w_1 with GELU (4 blocks, grid.x <= 74)
    ((2816, 512, 256, False), (2, (22, 4, 2), 1, "lin_splitk_reduce_kernel", 2)),
    ((4736, 512, 256, False), (2, (37, 4, 2), 1, "lin_splitk_reduce_kernel", 2)),
    ((4864, 512, 256, False), (1, (38, 4, 1), 1, None, 0)),
    ((65536, 512, 256, False), (1, (74, 4, 1), 7, None, 0)),
    # decoder steps: q|k|v, fc + LN, the classifier (96 = 3 blocks of 32 columns)
    ((512, 512, 1536, False), (2, (4, 24, 2), 1, "lin_splitk_reduce_kernel", 2)),
    ((1024, 512, 1536, False), (1, (8, 24, 1), 1, None, 0)),
    ((1024, 512, 512, True), (4, (8, 8, 4), 1, "lin_reduce_ln_kernel<4, 4>", 1)),
    ((1024, 512, 96, False), (4, (8, 3, 4), 1, "lin_splitk_reduce_kernel", 1)),
    # decoder memory projection k|v 512 -> 1024 (16 blocks, grid.x <= 18)
    ((65536, 512, 1024, False), (1, (18, 16, 1), 29, None, 0)),
    # the synthetic split LayerNorm case with two grid-stride passes
    ((9472, 512, 128, True), (2, (74, 2, 2), 1, "lin_reduce_ln_kernel<2, 2>", 2)),
]


@pytest.mark.parametrize("shape,want", HAND, ids=[f"{r}x{k}x{n}{'+ln' if ln else ''}" for (r, k, n, ln), _ in HAND])
def test_lin_plan_on_148_sms(shape, want):
    rows, k, n, ln = shape
    p = lin_plan(rows, k, n, 148, ln=ln)
    assert (p["splitk"], p["grid"], p["tiles_per_cta"], p["reduce"], p["reduce_passes"]) == want


def test_first_unsplit_row_counts_on_148_sms():
    """The smallest calls that take the unsplit path: the row counts the tile-independence checks compare against."""
    def first(k, n, ln):
        return next(r for r in range(128, 1 << 20, 128) if lin_plan(r, k, n, 148, ln)["splitk"] == 1)
    assert first(512, 1536, False) == 896            # 7 tiles
    assert first(512, 1024, False) == 1280           # 10 tiles
    assert first(512, 512, True) == first(256, 512, True) == 2432
    assert first(512, 256, False) == 4864
    assert (encoder_rows(37), encoder_rows(75)) == (2432, 4864)


def test_attn_decode_plan():
    assert attn_decode_plan(1024, 8, 64) == attn_decode_plan(1024, 8, 40) == "attn_decode_kernel<true>"
    assert attn_decode_plan(504, 8, 64) == attn_decode_plan(806, 8, 40) == "attn_decode_kernel<false>"
    assert attn_decode_plan(505, 8, 64) == attn_decode_plan(807, 8, 40) == "attn_decode_kernel<true>"
    assert attn_decode_plan(8, 8, 64) == attn_decode_plan(1024, 8, 31) == "attn_decode_kernel<false>"
