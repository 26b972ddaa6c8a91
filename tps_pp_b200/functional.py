"""Autograd-aware Python entry points over the C ABI (include/tpspp.h).

``tps_warp``      fused grid generator + bilinear sampling (reference tps_pp.py:481-496,601-615;
                  tps_preprocessor.py:72-83,270-282)
``grid_sample_border`` the sampler alone for an explicit grid (ATen-compatible fp32 coordinates)
``ocr_prep``      the text-recognition test pipeline (ResizeOCR + ToTensorOCR + NormalizeOCR) for a ragged uint8 batch

Tensors must live on a CUDA device; there is no CPU path.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import numpy as np
import torch

from . import _native as N

_DT = {torch.float32: N.F32, torch.bfloat16: N.BF16}
# kernel variant of tpspp_warp_bwd: AUTO = shared-memory staged kernel where it applies (TPS++ geometry, fp32);
# GENERIC forces the per-pixel global-atomics kernel (tests / A-B measurements)
BWD_VARIANT = N.VARIANT_AUTO


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(t: torch.Tensor):
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _require_cuda(name: str, t: Optional[torch.Tensor], dtype=None):
    if t is None:
        return
    if not t.is_cuda:
        raise RuntimeError(f"tps_pp_b200: `{name}` must be a CUDA tensor (the TPS++ hot path has no CPU fallback)")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"tps_pp_b200: `{name}` must be {dtype}, got {t.dtype}")


def _cfg(src0, src1, out_size, num_fiducial, mode, theta, variant) -> N.WarpCfg:
    if src0.dtype not in _DT:
        raise RuntimeError(f"tps_pp_b200: unsupported feature dtype {src0.dtype} (fp32 or bf16)")
    dt = _DT[src0.dtype]
    if src1 is not None and src1.dtype != src0.dtype:
        # bf16 feat_grid + fp32 x: the hand-over of the head's bf16 mode (TPSPP_SRC0_BF16: fp32 outputs, staged kernel, inference)
        if src0.dtype == torch.bfloat16 and src1.dtype == torch.float32:
            dt = N.SRC0_BF16
        else:
            raise RuntimeError("tps_pp_b200: src0/src1 dtype mismatch")
    b, c0, h0, w0 = src0.shape
    c1, h1, w1 = (src1.shape[1:] if src1 is not None else (0, 0, 0))
    return N.WarpCfg(b, c0, h0, w0, c1, h1, w1, int(out_size[0]), int(out_size[1]), int(num_fiducial),
                     int(mode), float(theta), dt, int(variant))


class _TpsWarp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src0, src1, c_prime, pc_score, P_hat, P, inv_delta_C, out_size, mode, theta, variant):
        _require_cuda("src0", src0)
        _require_cuda("src1", src1)
        _require_cuda("c_prime", c_prime, torch.float32)
        _require_cuda("pc_score", pc_score, torch.float32)
        for nm, t in (("P_hat", P_hat), ("P", P), ("inv_delta_C", inv_delta_C)):
            _require_cuda(nm, t, torch.float32)
        src0 = src0.contiguous()
        src1 = src1.contiguous() if src1 is not None else None
        c_prime = c_prime.contiguous()
        pc_score = pc_score.contiguous() if pc_score is not None else None
        P_hat = P_hat.contiguous(); inv_delta_C = inv_delta_C.contiguous()
        P = P.contiguous() if P is not None else None
        b, f = c_prime.shape[0], c_prime.shape[1]
        n = out_size[0] * out_size[1]
        if c_prime.shape != (src0.shape[0], f, 2):
            raise RuntimeError(f"tps_pp_b200: c_prime must be [B,F,2], got {tuple(c_prime.shape)}")
        k_cols = f if mode == N.MODE_ATTENTION else f + 3
        if P_hat.shape != (n, k_cols):
            raise RuntimeError(f"tps_pp_b200: P_hat must be [{n},{k_cols}], got {tuple(P_hat.shape)}")
        if inv_delta_C.shape != (f + 3, f + 3):
            raise RuntimeError(f"tps_pp_b200: inv_delta_C must be [{f + 3},{f + 3}]")
        if mode == N.MODE_ATTENTION:
            if pc_score is None or pc_score.shape != (b, n, f):
                raise RuntimeError(f"tps_pp_b200: pc_score must be [{b},{n},{f}]")
            if P is None or P.shape != (n, 2):
                raise RuntimeError(f"tps_pp_b200: P must be [{n},2]")
        cfg = _cfg(src0, src1, out_size, f, mode, theta, variant)
        if cfg.feat_dtype == N.SRC0_BF16 and (src0.requires_grad or src1.requires_grad or c_prime.requires_grad):
            raise RuntimeError("tps_pp_b200: the bf16-feat_grid / fp32-x warp is an inference layout (no backward)")
        out0 = torch.empty((b, src0.shape[1], out_size[0], out_size[1]),
                           dtype=torch.float32 if cfg.feat_dtype == N.SRC0_BF16 else src0.dtype, device=src0.device)
        out1 = (torch.empty((b, src1.shape[1], out_size[0], out_size[1]), dtype=src1.dtype, device=src1.device)
                if src1 is not None else None)
        with torch.cuda.device(src0.device):
            nbytes = int(N.lib().tpspp_warp_fwd_workspace_bytes(ctypes.byref(cfg)))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=src0.device) if nbytes else None
            N.check(N.lib().tpspp_warp_fwd(ctypes.byref(cfg), _ptr(src0), _ptr(src1), _ptr(c_prime), _ptr(pc_score),
                                           _ptr(P_hat), _ptr(P), _ptr(inv_delta_C), _ptr(out0), _ptr(out1),
                                           None, _ptr(ws), _stream(src0)), "tpspp_warp_fwd")
        ctx.save_for_backward(src0, src1, c_prime, pc_score, P_hat, P, inv_delta_C)
        ctx.cfg_args = (out_size, mode, theta)
        return out0, out1

    @staticmethod
    def backward(ctx, g0, g1):
        src0, src1, c_prime, pc_score, P_hat, P, inv_delta_C = ctx.saved_tensors
        out_size, mode, theta = ctx.cfg_args
        f = c_prime.shape[1]
        cfg = _cfg(src0, src1, out_size, f, mode, theta, BWD_VARIANT)
        need = ctx.needs_input_grad
        if g0 is None:
            g0 = torch.zeros((src0.shape[0], src0.shape[1]) + tuple(out_size), dtype=src0.dtype, device=src0.device)
        g0 = g0.contiguous()
        g1 = g1.contiguous() if (g1 is not None and src1 is not None) else None
        gsrc0 = torch.empty_like(src0) if need[0] else None
        gsrc1 = torch.empty_like(src1) if (src1 is not None and need[1] and g1 is not None) else None
        gcp = torch.empty_like(c_prime) if need[2] else None
        gsc = torch.empty_like(pc_score) if (pc_score is not None and need[3]) else None
        with torch.cuda.device(src0.device):
            nbytes = int(N.lib().tpspp_warp_workspace_bytes(ctypes.byref(cfg)))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=src0.device)
            N.check(N.lib().tpspp_warp_bwd(ctypes.byref(cfg), _ptr(src0), _ptr(src1), _ptr(c_prime), _ptr(pc_score),
                                           _ptr(P_hat), _ptr(P), _ptr(inv_delta_C), _ptr(g0), _ptr(g1),
                                           _ptr(gsrc0), _ptr(gsrc1), _ptr(gcp), _ptr(gsc), _ptr(ws), _stream(src0)),
                    "tpspp_warp_bwd")
        if src1 is not None and need[1] and gsrc1 is None:
            gsrc1 = torch.zeros_like(src1)
        return gsrc0, gsrc1, gcp, gsc, None, None, None, None, None, None, None


def tps_warp(src0: torch.Tensor, src1: Optional[torch.Tensor], c_prime: torch.Tensor,
             pc_score: Optional[torch.Tensor], P_hat: torch.Tensor, P: Optional[torch.Tensor],
             inv_delta_C: torch.Tensor, out_size: Tuple[int, int], mode: int = N.MODE_ATTENTION,
             theta: float = 0.5, variant: int = N.VARIANT_AUTO):
    """Fused ``build_P_prime`` + ``grid_sample`` (x2).  Returns ``(out0, out1_or_None)``."""
    return _TpsWarp.apply(src0, src1, c_prime, pc_score, P_hat, P, inv_delta_C, tuple(out_size), mode, theta, variant)


def tps_grid(c_prime, pc_score, P_hat, P, inv_delta_C, out_size, mode=N.MODE_ATTENTION, theta=0.5):
    """Debug/test helper: the sampling grid [B,n,2] as the fused kernel computes it (generic variant)."""
    b, f = c_prime.shape[:2]
    dummy = torch.zeros((b, 1, 1, 1), dtype=torch.float32, device=c_prime.device)
    cfg = _cfg(dummy, None, out_size, f, mode, theta, N.VARIANT_GENERIC)
    n = out_size[0] * out_size[1]
    grid = torch.empty((b, n, 2), dtype=torch.float32, device=c_prime.device)
    out = torch.empty((b, 1) + tuple(out_size), dtype=torch.float32, device=c_prime.device)
    with torch.cuda.device(c_prime.device):
        N.check(N.lib().tpspp_warp_fwd(ctypes.byref(cfg), _ptr(dummy), None, _ptr(c_prime.contiguous()),
                                       _ptr(pc_score.contiguous() if pc_score is not None else None),
                                       _ptr(P_hat.contiguous()), _ptr(P.contiguous() if P is not None else None),
                                       _ptr(inv_delta_C.contiguous()), _ptr(out), None, _ptr(grid), None,
                                       _stream(dummy)), "tpspp_warp_fwd")
    return grid


def grid_sample_border(src0: torch.Tensor, grid: torch.Tensor, src1: Optional[torch.Tensor] = None):
    """``F.grid_sample(src, grid, padding_mode='border', align_corners=True)`` for one or two sources
    (forward only; the differentiable path is :func:`tps_warp`)."""
    _require_cuda("src0", src0); _require_cuda("src1", src1); _require_cuda("grid", grid, torch.float32)
    src0 = src0.contiguous(); grid = grid.contiguous()
    src1 = src1.contiguous() if src1 is not None else None
    b, hr, wr, two = grid.shape
    if two != 2 or b != src0.shape[0]:
        raise RuntimeError("tps_pp_b200: grid must be [B,Hr,Wr,2]")
    cfg = _cfg(src0, src1, (hr, wr), 1, N.MODE_CLASSICAL, 0.0, N.VARIANT_GENERIC)
    out0 = torch.empty((b, src0.shape[1], hr, wr), dtype=src0.dtype, device=src0.device)
    out1 = torch.empty((b, src1.shape[1], hr, wr), dtype=src1.dtype, device=src1.device) if src1 is not None else None
    with torch.cuda.device(src0.device):
        N.check(N.lib().tpspp_sample_fwd(ctypes.byref(cfg), _ptr(src0), _ptr(src1), _ptr(grid), _ptr(out0),
                                         _ptr(out1), _stream(src0)), "tpspp_sample_fwd")
    return (out0, out1) if src1 is not None else out0


# ----------------------------------------------------------------------------- head
def head_cfg(batch, height, width, point_size, p_stride, precision=N.HEAD_FP32, flags=0) -> N.HeadCfg:
    return N.HeadCfg(int(batch), int(height), int(width), int(point_size[0]), int(point_size[1]), int(p_stride),
                     int(precision), int(flags))


def head_param_shapes(h: int, w: int, f: int, c: int = 64):
    """Shapes of the 58 parameter tensors in state_dict order (SURVEY App. A-5) for an ``h x w`` feature map with
    ``f`` control points -- what the native kernels size their reads from."""
    conv3 = lambda ci, co: [(co, ci, 3, 3), (co,)]
    lin = lambda ci, co: [(co, ci), (co,)]
    shapes = conv3(3 * c, 64) + conv3(64, 64) * 3                                   # MSFA encoder
    shapes += [(64 // 16, 64, 1, 1), (64, 64 // 16, 1, 1), (1, 2, 3, 3), (1,)]      # CBAM
    shapes += conv3(64, 64) * 3 + conv3(64, c)                                      # MSFA decoder
    shapes += lin(c, 32) + lin(32, 128) + lin(c, 32) + lin(32, 128)                 # p_linear, feat_linear
    shapes += [(h, w), (h, w), (h + 1, h + f), (w + 1, w + f)] + lin(c, c) + [(h, w), (h, w)]   # DGAB gate
    shapes += lin(c, 4 * c) + lin(4 * c, c)                                         # Mlp
    shapes += lin(c, 256) + lin(256, 2) + lin(2 * f, 2 * f)                         # localisation
    shapes += [(c, 32, 1, 1), (c,)] * 2 + [(c, 64, 1, 1), (c,)] + conv3(c, c) * 2 + [(c, 3 * c, 1, 1), (c,)]   # down*
    return shapes


def head_workspace_offsets(cfg: N.HeadCfg):
    """{name: byte offset} of the intermediates inside the head workspace (tests / backward)."""
    arr = (ctypes.c_size_t * len(N.WS_NAMES))()
    N.check(N.lib().tpspp_head_workspace_offsets(ctypes.byref(cfg), arr), "tpspp_head_workspace_offsets")
    return dict(zip(N.WS_NAMES, [int(v) for v in arr]))


def head_forward(x: torch.Tensor, o0: torch.Tensor, o1: torch.Tensor, params, point_size, p_stride,
                 precision=N.HEAD_FP32, workspace: Optional[torch.Tensor] = None, weights_cached: bool = False,
                 flags: int = 0):
    """Native control-point attention head (reference tps_pp.py:581-594), inference only (no autograd).

    ``params``: the module's parameters in state_dict order (58 fp32 CUDA tensors).
    ``weights_cached``: ``workspace`` was last used by a call with the same parameter values (the tensor-core
    weight images inside it are reused; see ``TPSPP_HEAD_FLAG_WEIGHTS_CACHED`` in include/tpspp.h).
    Returns ``(feat_grid, c_prime, pc_score, workspace)``."""
    for nm, t in (("batch_img", x), ("outs[0]", o0), ("outs[1]", o1)):
        _require_cuda(nm, t, torch.float32)
    x = x.contiguous(); o0 = o0.contiguous(); o1 = o1.contiguous()
    b, c, h, w = x.shape
    if c != 64 or o0.shape != (b, 32, 2 * h, 2 * w) or o1.shape != (b, 32, 2 * h, 2 * w):
        raise RuntimeError(f"tps_pp_b200: TPS_PP expects batch_img [B,64,h,w] and outs 2x[B,32,2h,2w]; got "
                           f"{tuple(x.shape)}, {tuple(o0.shape)}, {tuple(o1.shape)}")
    params = list(params)
    if len(params) != N.P_COUNT:
        raise RuntimeError(f"tps_pp_b200: expected {N.P_COUNT} parameter tensors, got {len(params)}")
    f = point_size[0] * point_size[1]
    table = (ctypes.c_void_p * N.P_COUNT)()
    # the kernels size every weight read from (h, w, F): a module built for another geometry must fail here, like
    # the reference's layer_norm / linear calls do, instead of reading out of bounds
    for i, (p, shp) in enumerate(zip(params, head_param_shapes(h, w, f))):
        _require_cuda(f"param[{i}]", p, torch.float32)
        if not p.is_contiguous():
            raise RuntimeError(f"tps_pp_b200: param[{i}] must be contiguous")
        if tuple(p.shape) != shp:
            raise RuntimeError(f"tps_pp_b200: param[{i}] has shape {tuple(p.shape)} but a [{b},{c},{h},{w}] input with "
                               f"{f} control points needs {shp} (module built for another img_size / point_size?)")
        table[i] = p.data_ptr()
    cfg = head_cfg(b, h, w, point_size, p_stride, precision, flags)
    with torch.cuda.device(x.device):
        nbytes = int(N.lib().tpspp_head_workspace_bytes(ctypes.byref(cfg)))
        if nbytes == 0 and b > 0:
            raise RuntimeError("tpspp_head_workspace_bytes failed: " + N.last_error())
        if workspace is None or workspace.numel() < nbytes or workspace.device != x.device:
            workspace = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=x.device)
            weights_cached = False
        if weights_cached:
            cfg.flags |= N.HEAD_FLAG_WEIGHTS_CACHED
        fg_bf16 = precision == N.HEAD_BF16 and (flags & N.HEAD_FLAG_FEATGRID_BF16) != 0
        feat_grid = torch.empty((b, 64, 2 * h, 2 * w), dtype=torch.bfloat16 if fg_bf16 else torch.float32, device=x.device)
        c_prime = torch.empty((b, f, 2), dtype=torch.float32, device=x.device)
        score = torch.empty((b, h * w, f), dtype=torch.float32, device=x.device)
        N.check(N.lib().tpspp_head_fwd(ctypes.byref(cfg), _ptr(x), _ptr(o0), _ptr(o1), table, _ptr(feat_grid),
                                       _ptr(c_prime), _ptr(score), _ptr(workspace), _stream(x)), "tpspp_head_fwd")
    return feat_grid, c_prime, score, workspace


def stage_param_shapes():
    """Shapes of the 81 tensors ``tpspp_stage_fwd`` takes (include/tpspp.h TPSPP_SP_*): the stage's slice of the reference
    ``ResNetABI_v2_large`` state_dict without the int64 ``num_batches_tracked`` buffers."""
    def bn(c):
        return [(c,)] * 4
    shapes = [(32, 3, 3, 3), (32,)] + bn(32)
    for cin, planes, blocks, down in ((32, 32, 3, False), (32, 64, 4, True)):
        for i in range(blocks):
            ci = cin if i == 0 else planes
            shapes += [(planes, ci, 1, 1)] + bn(planes) + [(planes, planes, 3, 3)] + bn(planes)
            if i == 0 and down:
                shapes += [(planes, ci, 1, 1)] + bn(planes)
    return shapes


def stage_forward(img: torch.Tensor, params, workspace: Optional[torch.Tensor] = None, weights_cached: bool = False):
    """Native backbone stage in front of the rectifier (reference backbones/resnet_v2_large.py:176-191 up to the
    ``tpsnet(x, outs)`` call; eval-mode BatchNorm folded into the convolutions), inference only.

    ``img`` [B,3,H,128] fp32 CUDA; ``params``: the 81 stage tensors in state_dict order (``stage_param_shapes``).
    Returns ``(o0 [B,32,H,W], o1 [B,32,H,W], x [B,64,H/2,W/2], workspace)``."""
    _require_cuda("img", img, torch.float32)
    img = img.contiguous()
    b, c, h, w = img.shape
    if c != 3:
        raise RuntimeError(f"tps_pp_b200: the backbone stage takes 3-channel images, got {tuple(img.shape)}")
    params = list(params)
    shapes = stage_param_shapes()
    if len(params) != N.SP_COUNT:
        raise RuntimeError(f"tps_pp_b200: expected {N.SP_COUNT} stage tensors, got {len(params)}")
    table = (ctypes.c_void_p * N.SP_COUNT)()
    for i, (p, shp) in enumerate(zip(params, shapes)):
        _require_cuda(f"stage param[{i}]", p, torch.float32)
        if not p.is_contiguous() or tuple(p.shape) != shp:
            raise RuntimeError(f"tps_pp_b200: stage param[{i}] must be a contiguous {shp} tensor, got {tuple(p.shape)}")
        table[i] = p.data_ptr()
    cfg = N.StageCfg(b, h, w, N.HEAD_TC, 0)
    with torch.cuda.device(img.device):
        nbytes = int(N.lib().tpspp_stage_workspace_bytes(ctypes.byref(cfg)))
        if nbytes == 0 and b > 0:
            raise RuntimeError("tpspp_stage_workspace_bytes failed: " + N.last_error())
        if workspace is None or workspace.numel() < nbytes or workspace.device != img.device:
            workspace = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=img.device)
            weights_cached = False
        if weights_cached:
            cfg.flags |= N.HEAD_FLAG_WEIGHTS_CACHED
        o0 = torch.empty((b, 32, h, w), dtype=torch.float32, device=img.device)
        o1 = torch.empty((b, 32, h, w), dtype=torch.float32, device=img.device)
        x = torch.empty((b, 64, h // 2, w // 2), dtype=torch.float32, device=img.device)
        N.check(N.lib().tpspp_stage_fwd(ctypes.byref(cfg), _ptr(img), table, _ptr(o0), _ptr(o1), _ptr(x), _ptr(workspace),
                                        _stream(img)), "tpspp_stage_fwd")
    return o0, o1, x, workspace


def locnet_param_keys():
    """state_dict keys (relative to ``LocalizationNetwork.``) in the order ``tpspp_locnet_fwd`` takes them (TPSPP_LP_*)."""
    keys = []
    for ci in (0, 4, 8, 12):
        keys.append(f"conv.{ci}.weight")
        keys += [f"conv.{ci + 1}.{n}" for n in ("weight", "bias", "running_mean", "running_var")]
    return keys + ["localization_fc1.0.weight", "localization_fc1.0.bias", "localization_fc2.weight", "localization_fc2.bias"]


def locnet_param_shapes(channels: int, num_fiducial: int):
    """Shapes of the 24 tensors of :func:`locnet_param_keys` (tps_preprocessor.py:101-131)."""
    shapes = []
    chans = (channels, 64, 128, 256, 512)
    for i in range(4):
        shapes.append((chans[i + 1], chans[i], 3, 3))
        shapes += [(chans[i + 1],)] * 4
    return shapes + [(256, 512), (256,), (2 * num_fiducial, 256), (2 * num_fiducial,)]


def locnet_supported(channels: int, height: int, width: int, num_fiducial: int) -> bool:
    """Whether the native localisation network takes this geometry (include/tpspp.h ``tpspp_locnet_cfg``)."""
    cfg = N.LocnetCfg(1, channels, height, width, num_fiducial, 0)
    return int(N.lib().tpspp_locnet_workspace_bytes(ctypes.byref(cfg))) > 0


def locnet_forward(img: torch.Tensor, params, num_fiducial: int, workspace: Optional[torch.Tensor] = None,
                   weights_cached: bool = False):
    """``LocalizationNetwork.forward`` of the classical preprocessor (tps_preprocessor.py:143-156), eval mode, on the native
    kernels: img [B,C,H,W] fp32 -> (C' [B,F,2], workspace).  ``params``: the 24 tensors of :func:`locnet_param_keys`."""
    _require_cuda("img", img, torch.float32)
    if len(params) != N.LP_COUNT:
        raise RuntimeError(f"tps_pp_b200: the localisation network takes {N.LP_COUNT} parameter tensors, got {len(params)}")
    img = img.contiguous()
    b, c, h, w = img.shape
    # the kernels size every weight read from (channels, F): a module built for another configuration must fail here
    for i, (t, shp) in enumerate(zip(params, locnet_param_shapes(c, num_fiducial))):
        _require_cuda(f"params[{i}]", t, torch.float32)
        if not t.is_contiguous():
            raise RuntimeError(f"tps_pp_b200: params[{i}] must be contiguous")
        if tuple(t.shape) != shp:
            raise RuntimeError(f"tps_pp_b200: localisation-network params[{i}] has shape {tuple(t.shape)}, expected {shp} for "
                               f"{c} image channels and {num_fiducial} control points")
    cfg = N.LocnetCfg(b, c, h, w, num_fiducial, 0)
    table = (ctypes.c_void_p * N.LP_COUNT)(*[t.data_ptr() for t in params])
    with torch.cuda.device(img.device):
        nbytes = int(N.lib().tpspp_locnet_workspace_bytes(ctypes.byref(cfg)))
        if nbytes == 0 and b > 0:
            raise RuntimeError("tpspp_locnet_workspace_bytes failed: " + N.last_error())
        if workspace is None or workspace.numel() < nbytes or workspace.device != img.device:
            workspace = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=img.device)
            weights_cached = False
        if weights_cached:
            cfg.flags |= N.HEAD_FLAG_WEIGHTS_CACHED
        cp = torch.empty((b, num_fiducial, 2), dtype=torch.float32, device=img.device)
        N.check(N.lib().tpspp_locnet_fwd(ctypes.byref(cfg), _ptr(img), table, _ptr(cp), _ptr(workspace), _stream(img)),
                "tpspp_locnet_fwd")
    return cp, workspace


def _conv_cfg(b, cin, h, w, k, sh, sw, relu, ups):
    cfg = N.ConvCfg(b, cin, h, w, k, sh, sw, 1 if relu else 0, len(ups))
    for i, (uh, uw) in enumerate(ups):
        cfg.up_h[i] = uh
        cfg.up_w[i] = uw
    return cfg


def _ptr_array(ts):
    arr = (ctypes.c_void_p * 3)()
    for i, t in enumerate(ts):
        arr[i] = t.data_ptr() if t is not None else None
    return arr


class _ConvRelu(torch.autograd.Function):
    """One ``ConvModule`` (conv + bias + ReLU, reference tps_pp.py:126-131,149-154,538-548) with native forward AND backward
    (``tpspp_convcat_fwd`` / ``tpspp_convcat_bwd``): the training-path counterpart of the fused inference head.  The input is
    ``torch.cat([F.interpolate(x_s, scale_factor=ups[s]) for s], dim=1)`` without either being materialised
    (tps_pp.py:159-168,583-585)."""

    @staticmethod
    def forward(ctx, weight, bias, stride, relu, ups, *xs):
        _require_cuda("weight", weight, torch.float32)
        _require_cuda("bias", bias, torch.float32)
        xs = [x.contiguous() for x in xs]
        for x in xs:
            _require_cuda("x", x, torch.float32)
        weight = weight.contiguous(); bias = bias.contiguous()
        b = xs[0].shape[0]
        h, w = xs[0].shape[2] * ups[0][0], xs[0].shape[3] * ups[0][1]
        cin = sum(x.shape[1] for x in xs)
        for x, (uh, uw) in zip(xs, ups):
            if x.shape[0] != b or (x.shape[2] * uh, x.shape[3] * uw) != (h, w) or (len(xs) > 1 and x.shape[1] != 64):
                raise RuntimeError("tps_pp_b200: concatenated conv sources must share batch and (upsampled) size, 64 channels each")
        k = weight.shape[-1]
        if weight.shape[0] != 64 or weight.shape[1] != cin or weight.shape[2] != k:
            raise RuntimeError(f"tps_pp_b200: conv weight must be [64,{cin},k,k], got {tuple(weight.shape)}")
        sh, sw = (stride, stride) if isinstance(stride, int) else stride
        cfg = _conv_cfg(b, cin, h, w, k, sh, sw, relu, ups)
        dev = xs[0].device
        with torch.cuda.device(dev):
            nbytes = int(N.lib().tpspp_conv_workspace_bytes(ctypes.byref(cfg)))
            if nbytes == 0 and b > 0:
                raise RuntimeError("tpspp_conv_workspace_bytes failed: " + N.last_error())
            ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=dev)
            y = torch.empty((b, 64, h // sh, w // sw), dtype=torch.float32, device=dev)
            N.check(N.lib().tpspp_convcat_fwd(ctypes.byref(cfg), _ptr_array(xs), _ptr(weight), _ptr(bias), _ptr(y), _ptr(ws),
                                              _stream(y)), "tpspp_convcat_fwd")
        ctx.save_for_backward(weight, y, *xs)
        ctx.cfg = (b, cin, h, w, k, sh, sw, relu, tuple(ups))
        return y

    @staticmethod
    def backward(ctx, gy):
        weight, y, *xs = ctx.saved_tensors
        cfg = _conv_cfg(*ctx.cfg)
        gy = gy.contiguous()
        need = ctx.needs_input_grad
        gxs = [torch.empty_like(x) if need[5 + i] else None for i, x in enumerate(xs)]
        gw = torch.empty_like(weight) if need[0] else None
        gb = torch.empty(64, dtype=torch.float32, device=y.device) if need[1] else None
        with torch.cuda.device(y.device):
            nbytes = int(N.lib().tpspp_conv_workspace_bytes(ctypes.byref(cfg)))
            ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=y.device)
            N.check(N.lib().tpspp_convcat_bwd(ctypes.byref(cfg), _ptr_array(xs), _ptr(weight), _ptr(y), _ptr(gy), _ptr_array(gxs),
                                              _ptr(gw), _ptr(gb), _ptr(ws), _stream(y)), "tpspp_convcat_bwd")
        return (gw, gb, None, None, None, *gxs)


def conv_relu_supported(x, weight: torch.Tensor, stride=1, ups=None) -> bool:
    """Geometry the native training convolution covers (include/tpspp.h ``tpspp_conv_cfg``).  ``x``: one tensor or a sequence
    of up to three 64-channel tensors (fused ``torch.cat``); ``ups``: per-source nearest-upsample factors (fused ``F.interpolate``)."""
    xs = [x] if isinstance(x, torch.Tensor) else list(x)
    ups = _norm_ups(ups, len(xs))
    if not 1 <= len(xs) <= 3 or weight.dim() != 4 or weight.dtype != torch.float32:
        return False
    for t, (uh, uw) in zip(xs, ups):
        if not (t.is_cuda and t.dtype == torch.float32 and t.dim() == 4) or uh not in (1, 2) or uw not in (1, 2):
            return False
        if len(xs) > 1 and t.shape[1] != 64:
            return False
        if (t.shape[2] * t.shape[3]) % 4:
            return False
    b = xs[0].shape[0]
    h, w = xs[0].shape[2] * ups[0][0], xs[0].shape[3] * ups[0][1]
    if any(t.shape[0] != b or (t.shape[2] * u[0], t.shape[3] * u[1]) != (h, w) for t, u in zip(xs, ups)):
        return False
    cin = sum(t.shape[1] for t in xs)
    k = weight.shape[-1]
    sh, sw = (stride, stride) if isinstance(stride, int) else stride
    if weight.shape[0] != 64 or weight.shape[1] != cin or weight.shape[2] != k or k not in (1, 3):
        return False
    if cin % 32 or (cin > 64 and cin % 64) or cin > 512:
        return False
    if (sh, sw) != (1, 1) and not (k == 3 and sh == 2 and sw in (1, 2)):
        return False
    if (sh, sw) != (1, 1) and any(u != (1, 1) for u in ups):
        return False
    if h % sh or w % sw:
        return False
    ho, wo = h // sh, w // sw
    return b > 0 and (b * ho * wo) % 128 == 0 and (b * h * w) % 128 == 0 and (ho * wo) % 32 == 0 and (h * w) % 4 == 0


def _norm_ups(ups, n):
    if ups is None:
        return [(1, 1)] * n
    out = []
    for u in ups:
        out.append((int(u), int(u)) if isinstance(u, int) else (int(u[0]), int(u[1])))
    if len(out) != n:
        raise RuntimeError("tps_pp_b200: one upsample factor per conv source")
    return out


def conv_relu(x, weight: torch.Tensor, bias: torch.Tensor, stride=1, relu: bool = True, ups=None) -> torch.Tensor:
    """``relu(conv2d(cat([interpolate(x_s, ups[s]) ...], 1), weight, bias, stride, padding=k//2))`` with 64 output channels on the
    native kernels, differentiable.  ``x``: one tensor or a sequence of up to three 64-channel tensors."""
    xs = [x] if isinstance(x, torch.Tensor) else list(x)
    return _ConvRelu.apply(weight, bias, stride, relu, _norm_ups(ups, len(xs)), *xs)


class _Linear(torch.autograd.Function):
    """``nn.Linear`` / ``torch.bmm(x, w^T)`` of the head's dense stages with native forward AND backward
    (``tpspp_linear_fwd`` / ``tpspp_linear_bwd``; reference DGAB.py:11-23,28-36,52, tps_pp.py:250-273,293-299)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        _require_cuda("x", x, torch.float32)
        _require_cuda("weight", weight, torch.float32)
        _require_cuda("bias", bias, torch.float32)
        batches = weight.shape[0] if weight.dim() == 3 else 1
        n, k = weight.shape[-2], weight.shape[-1]
        if x.shape[-1] != k:
            raise RuntimeError(f"tps_pp_b200: linear input features {x.shape[-1]} != weight in_features {k}")
        if batches > 1 and (bias is not None or x.shape[0] != batches):
            raise RuntimeError("tps_pp_b200: batched linear (bmm) needs x [batches, rows, in] and no bias")
        x2 = x.contiguous()
        weight = weight.contiguous()
        bias = bias.contiguous() if bias is not None else None
        rows = x2.numel() // k
        cfg = N.LinearCfg(rows, k, n, batches, 0)
        y = torch.empty(x.shape[:-1] + (n,), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            nbytes = int(N.lib().tpspp_linear_workspace_bytes(ctypes.byref(cfg)))
            if nbytes == 0:
                raise RuntimeError("tpspp_linear_workspace_bytes failed: " + N.last_error())
            ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            N.check(N.lib().tpspp_linear_fwd(ctypes.byref(cfg), _ptr(x2), _ptr(weight), _ptr(bias), _ptr(y), _ptr(ws), _stream(x)),
                    "tpspp_linear_fwd")
        ctx.save_for_backward(x2, weight)
        ctx.cfg = (rows, k, n, batches)
        ctx.has_bias = bias is not None
        ctx.x_shape = x.shape
        return y

    @staticmethod
    def backward(ctx, gy):
        x2, weight = ctx.saved_tensors
        cfg = N.LinearCfg(*ctx.cfg, 0)
        gy = gy.contiguous()
        need = ctx.needs_input_grad
        want_w = need[1] or (ctx.has_bias and need[2])
        gx = torch.empty_like(x2) if need[0] else None
        gw = torch.empty_like(weight) if want_w else None
        gb = torch.empty(ctx.cfg[2], dtype=torch.float32, device=gy.device) if (ctx.has_bias and need[2]) else None
        with torch.cuda.device(gy.device):
            nbytes = int(N.lib().tpspp_linear_workspace_bytes(ctypes.byref(cfg)))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=gy.device)
            N.check(N.lib().tpspp_linear_bwd(ctypes.byref(cfg), _ptr(x2), _ptr(weight), _ptr(gy), _ptr(gx), _ptr(gw), _ptr(gb),
                                             _ptr(ws), _stream(gy)), "tpspp_linear_bwd")
        return (gx.view(ctx.x_shape) if gx is not None else None), (gw if need[1] else None), gb


def linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``F.linear(x, weight, bias)`` on the native kernels, differentiable (any leading shape, fp32)."""
    return _Linear.apply(x, weight, bias)


def bmm_nt(x: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """``torch.bmm(x, w.transpose(1, 2))`` -- x [B, rows, K], w [B, N, K] -> [B, rows, N] -- on the native kernels, differentiable
    (the einsum of ``atten_score``, tps_pp.py:293-299)."""
    return _Linear.apply(x, w, None)


class PreparedLinear:
    """Inference-side ``F.linear`` with a fixed weight: ``tpspp_linear_fwd`` on a persistent workspace, so the tensor-core
    operand image of the weight is laid out once (``TPSPP_LINEAR_FLAG_WEIGHTS_CACHED`` afterwards) instead of at every call --
    the NRTR decode calls each of its 43 dense layers 40 times per batch.  Forward only; rows fixed at construction."""

    def __init__(self, weight: torch.Tensor, bias: Optional[torch.Tensor], rows: int):
        _require_cuda("weight", weight, torch.float32)
        _require_cuda("bias", bias, torch.float32)
        self.weight = weight.detach().contiguous()
        self.bias = bias.detach().contiguous() if bias is not None else None
        self.rows = int(rows)
        self.n, self.k = self.weight.shape
        self.cfg = N.LinearCfg(self.rows, self.k, self.n, 1, 0)
        with torch.cuda.device(weight.device):
            nbytes = int(N.lib().tpspp_linear_workspace_bytes(ctypes.byref(self.cfg)))
        if nbytes == 0:
            raise RuntimeError("tpspp_linear_workspace_bytes failed: " + N.last_error())
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=weight.device)
        self.prepared = False

    def __call__(self, x: torch.Tensor, out: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
                 gelu: bool = False, ln: Optional[torch.nn.LayerNorm] = None, ln_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``act(x w^T + b) + residual`` (``tpspp_linear_ln_fwd``); ``out`` may be ``residual`` itself (x = x + f(.) in place).
        With ``ln`` (an ``nn.LayerNorm`` over the output features) and ``ln_out`` [rows, out]: ``ln_out = ln(result)`` is written by
        the kernel that finishes the result -- the LayerNorm a pre-norm transformer layer applies next, without its own launch."""
        if x.shape != (self.rows, self.k) or not x.is_contiguous() or x.dtype != torch.float32:
            raise RuntimeError(f"tps_pp_b200: PreparedLinear expects a contiguous fp32 [{self.rows}, {self.k}] input, got {tuple(x.shape)}")
        y = out if out is not None else torch.empty((self.rows, self.n), dtype=torch.float32, device=x.device)
        for nm, t in (("out", y), ("residual", residual)):
            if t is not None and (t.shape != (self.rows, self.n) or not t.is_contiguous() or t.dtype != torch.float32 or not t.is_cuda):
                raise RuntimeError(f"tps_pp_b200: PreparedLinear `{nm}` must be a contiguous fp32 CUDA [{self.rows}, {self.n}] tensor")
        lw = lb = None
        eps = 0.0
        if ln is not None:
            if ln_out is None or ln_out.shape != (self.rows, self.n) or not ln_out.is_contiguous() or ln_out.dtype != torch.float32 or not ln_out.is_cuda:
                raise RuntimeError(f"tps_pp_b200: PreparedLinear `ln_out` must be a contiguous fp32 CUDA [{self.rows}, {self.n}] tensor")
            if tuple(ln.normalized_shape) != (self.n,) or ln.weight is None:
                raise RuntimeError(f"tps_pp_b200: PreparedLinear `ln` must be an affine LayerNorm over the {self.n} output features")
            lw, lb, eps = ln.weight.detach(), (ln.bias.detach() if ln.bias is not None else None), float(ln.eps)
        self.cfg.flags = N.LINEAR_FLAG_WEIGHTS_CACHED if self.prepared else 0
        with torch.cuda.device(x.device):
            N.check(N.lib().tpspp_linear_ln_fwd(ctypes.byref(self.cfg), _ptr(x), _ptr(self.weight), _ptr(self.bias), _ptr(residual),
                                                N.ACT_GELU if gelu else N.ACT_NONE, _ptr(y), _ptr(lw), _ptr(lb), eps,
                                                _ptr(ln_out) if ln is not None else None, _ptr(self.ws), _stream(x)),
                    "tpspp_linear_ln_fwd")
        self.prepared = True
        return y


def attn_decode(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, kv_len: int, temperature: float,
                kv_lens: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                k_new: Optional[torch.Tensor] = None, v_new: Optional[torch.Tensor] = None, head_major: bool = False) -> torch.Tensor:
    """Single-query multi-head attention over a key/value cache (``tpspp_attn_decode``): q [B, heads*64], k / v
    [B, capacity, heads*64] (or, with ``head_major``, [B, heads, capacity, 64]) -> [B, heads*64]; keys ``t < kv_len`` (or ``kv_lens[b]``, int32 on the device).  ``k_new`` / ``v_new``
    [B, heads*64]: this step's rows, stored at cache position ``kv_len - 1`` by the kernel before it attends.  ``q`` / ``k_new`` /
    ``v_new`` may be column slices of one fused projection (unit stride along the features).  Forward only."""
    for nm, t in (("k", k), ("v", v)):
        _require_cuda(nm, t, torch.float32)
        if not t.is_contiguous():
            raise RuntimeError(f"tps_pp_b200: attn_decode `{nm}` must be contiguous")
    b, d = q.shape
    for nm, t in (("q", q), ("k_new", k_new), ("v_new", v_new)):
        _require_cuda(nm, t, torch.float32)
        if t is not None and (t.dim() != 2 or t.shape != (b, d) or t.stride(1) != 1):
            raise RuntimeError(f"tps_pp_b200: attn_decode `{nm}` must be [B, heads*64] with unit stride along the features")
    if (k_new is None) != (v_new is None) or (k_new is not None and k_new.stride(0) != v_new.stride(0)):
        raise RuntimeError("tps_pp_b200: attn_decode k_new / v_new come together, with the same row stride")
    want = (b, heads, k.shape[2] if k.dim() == 4 else 0, 64) if head_major else (b, k.shape[1], d)
    if d != heads * 64 or tuple(k.shape) != want or v.shape != k.shape:
        raise RuntimeError(f"tps_pp_b200: attn_decode shapes q {tuple(q.shape)} k {tuple(k.shape)} v {tuple(v.shape)} heads {heads} "
                           f"(head_major={head_major})")
    if kv_lens is not None and (kv_lens.dtype != torch.int32 or not kv_lens.is_cuda or kv_lens.numel() != b):
        raise RuntimeError("tps_pp_b200: kv_lens must be an int32 CUDA tensor with one entry per image")
    if out is None:
        out = torch.empty((b, d), dtype=torch.float32, device=q.device)
    cfg = N.AttnCfg(b, heads, 64, int(kv_len), k.shape[2] if head_major else k.shape[1], float(temperature),
                    int(q.stride(0)) if b > 1 else d, (int(k_new.stride(0)) if b > 1 else d) if k_new is not None else 0,
                    1 if head_major else 0)
    with torch.cuda.device(q.device):
        N.check(N.lib().tpspp_attn_decode(ctypes.byref(cfg), _ptr(q), _ptr(k), _ptr(v), _ptr(kv_lens), _ptr(k_new), _ptr(v_new),
                                          _ptr(out), _stream(q)), "tpspp_attn_decode")
    return out


def attn_encode(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, seq_len: int, temperature: float,
                kv_lens: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Multi-head self-attention over whole sequences (``tpspp_attn_encode``): q / k / v token-major [B*T, heads*64] -> out
    [B*T, heads*64]; image b's queries (all T of them) attend to its keys ``j < kv_lens[b]`` (int32 on the device) or to all T.
    ``q`` / ``k`` / ``v`` may be column slices of one fused projection: unit stride along the features, one common row stride.
    ``out`` (optional) must be a contiguous fp32 tensor of that shape on the same device.  Forward only."""
    for nm, t in (("q", q), ("k", k), ("v", v)):
        _require_cuda(nm, t, torch.float32)
    rows, d = q.shape if q.dim() == 2 else (-1, -1)
    seq_len = int(seq_len)
    if seq_len < 1 or d != heads * 64 or rows % seq_len:
        raise RuntimeError(f"tps_pp_b200: attn_encode q must be [B*T, heads*64] with T = {seq_len} >= 1, got {tuple(q.shape)} "
                           f"for {heads} heads")
    b = rows // seq_len
    for nm, t in (("q", q), ("k", k), ("v", v)):
        if t.shape != (rows, d) or t.stride(1) != 1 or t.device != q.device:
            raise RuntimeError(f"tps_pp_b200: attn_encode `{nm}` must be [{rows}, {d}] on {q.device} with unit stride along the features")
    stride = int(q.stride(0)) if rows > 1 else d
    if rows > 1 and (k.stride(0) != stride or v.stride(0) != stride):
        raise RuntimeError("tps_pp_b200: attn_encode q / k / v must share one row stride")
    if kv_lens is not None and (kv_lens.dtype != torch.int32 or not kv_lens.is_cuda or kv_lens.numel() != b
                                or kv_lens.device != q.device or not kv_lens.is_contiguous()):
        raise RuntimeError("tps_pp_b200: kv_lens must be a contiguous int32 tensor on the device of q with one entry per image")
    if out is None:
        out = torch.empty((rows, d), dtype=torch.float32, device=q.device)
    elif (out.dtype != torch.float32 or out.device != q.device or tuple(out.shape) != (rows, d) or not out.is_contiguous()):
        raise RuntimeError(f"tps_pp_b200: attn_encode `out` must be a contiguous fp32 [{rows}, {d}] tensor on {q.device}")
    cfg = N.AttnEncodeCfg(b, heads, 64, seq_len, float(temperature), stride)
    with torch.cuda.device(q.device):
        N.check(N.lib().tpspp_attn_encode(ctypes.byref(cfg), _ptr(q), _ptr(k), _ptr(v), _ptr(kv_lens), _ptr(out), _stream(q)),
                "tpspp_attn_encode")
    return out


def check_ocr_desc(desc, packed_bytes: int, out_w: int) -> np.ndarray:
    """Host-side check of the ``tpspp_ocr_prep`` descriptors (the kernel reads them on the device and cannot check them without
    a host sync): ``desc`` [n, 4] int64 rows (byte offset, h, w, resize_w) of images in a packed uint8 buffer of
    ``packed_bytes`` bytes, or [n, 5] rows with a fifth field ``k`` in [0, 3], the quarter turns of ``np.rot90(img, k)``
    (``h``, ``w`` are the stored image's).  Raises ``ValueError``; returns the rows as an int64 numpy array."""
    d = desc.numpy() if isinstance(desc, torch.Tensor) else np.asarray(desc)
    if isinstance(desc, torch.Tensor) and desc.device.type != "cpu":
        raise ValueError("tps_pp_b200: ocr_prep descriptors are checked on the host: pass them as a CPU tensor or numpy array")
    if d.dtype != np.int64 or d.ndim != 2 or d.shape[1] not in (4, 5) or d.shape[0] < 1:
        raise ValueError(f"tps_pp_b200: ocr_prep descriptors must be a non-empty int64 [n, 4] or [n, 5] array, got {d.dtype} {d.shape}")
    off, h, w, rw = d[:, 0], d[:, 1], d[:, 2], d[:, 3]
    checks = [("h >= 1", h < 1), ("w >= 1", w < 1), ("offset >= 0", off < 0),
              (f"1 <= resize_w <= out_w = {out_w}", (rw < 1) | (rw > out_w))]
    if d.shape[1] == 5:
        checks.append(("0 <= k <= 3 (quarter turns)", (d[:, 4] < 0) | (d[:, 4] > 3)))
    for what, bad in checks:
        if bad.any():
            i = int(np.flatnonzero(bad)[0])
            raise ValueError(f"tps_pp_b200: ocr_prep descriptor {i} {d[i].tolist()} breaks {what}")
    end = off + h * w * 3
    past = (end > int(packed_bytes)) | (end < off)
    if past.any():
        i = int(np.flatnonzero(past)[0])
        raise ValueError(f"tps_pp_b200: ocr_prep image {i} {d[i].tolist()} reaches past the end of the {packed_bytes}-byte buffer")
    return d


def ocr_prep(packed: torch.Tensor, desc, out_h: int, out_w: int, mean, std, pad_value: int = 0,
             out: Optional[torch.Tensor] = None, desc_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """mmocr's ResizeOCR + ToTensorOCR + NormalizeOCR for a ragged batch in one launch (``tpspp_ocr_prep``): ``packed`` uint8
    HWC 3-channel images one after the other (1-D CUDA tensor), ``desc`` their [n, 4] int64 descriptors (byte offset, h, w,
    resize_w) ON THE HOST, checked by :func:`check_ocr_desc` before anything is launched -> [n, 3, out_h, out_w] fp32.
    [n, 5] descriptors add ``k``: row i is then the image ``np.rot90(img, k)`` resized to (resize_w, out_h) (mmocr's
    ``MultiRotateAugOCR``; rows may share an offset), and the call sets ``TPSPP_OCR_FLAG_ROTATED``.
    ``desc_dev``: the same descriptors already on the device (a caller that uploads them with its images in one copy);
    otherwise they are copied here.  ``out`` (optional) must be a contiguous fp32 tensor of that shape on the same device."""
    d = check_ocr_desc(desc, packed.numel(), out_w)
    if len(mean) != 3 or len(std) != 3:
        raise ValueError(f"tps_pp_b200: ocr_prep takes 3 means and 3 stds, got {len(mean)} and {len(std)}")
    _require_cuda("packed", packed, torch.uint8)
    if packed.dim() != 1 or not packed.is_contiguous():
        raise RuntimeError("tps_pp_b200: ocr_prep `packed` must be a contiguous 1-D uint8 tensor")
    n, fields = d.shape
    if desc_dev is None:
        desc_dev = torch.from_numpy(d).to(packed.device)
    elif (desc_dev.dtype != torch.int64 or desc_dev.device != packed.device or tuple(desc_dev.shape) != (n, fields)
          or not desc_dev.is_contiguous()):
        raise RuntimeError(f"tps_pp_b200: ocr_prep `desc_dev` must be a contiguous int64 [{n}, {fields}] tensor on {packed.device}")
    shape = (n, 3, int(out_h), int(out_w))
    if out is None:
        out = torch.empty(tuple(max(s, 0) for s in shape), dtype=torch.float32, device=packed.device)
    elif out.dtype != torch.float32 or out.device != packed.device or tuple(out.shape) != shape or not out.is_contiguous():
        raise RuntimeError(f"tps_pp_b200: ocr_prep `out` must be a contiguous fp32 {list(shape)} tensor on {packed.device}")
    flags = N.OCR_FLAG_ROTATED if fields == 5 else 0
    cfg = N.OcrPrepCfg(n, int(out_h), int(out_w), (ctypes.c_float * 3)(*[float(m) for m in mean]),
                       (ctypes.c_float * 3)(*[float(s) for s in std]), int(pad_value), flags, packed.numel())
    with torch.cuda.device(packed.device):
        N.check(N.lib().tpspp_ocr_prep(ctypes.byref(cfg), _ptr(packed), _ptr(desc_dev), _ptr(out), _stream(packed)), "tpspp_ocr_prep")
    return out


def _fused_source(t: torch.Tensor):
    """``(base, column offset)`` when ``t`` is a column block of a contiguous 2-D tensor (a slice of a fused projection), else
    ``(t, 0)`` -- so that the attention's gradient lands in the fused projection's gradient without a ``torch.cat``."""
    b = t._base
    # the base stands in for t only when autograd treats them alike (a slice made a leaf by requires_grad_() has a base
    # that does not require grad: its gradient must stay with the slice)
    if (b is not None and b.requires_grad == t.requires_grad and b.dim() == 2 and b.is_contiguous() and t.dim() == 2 and t.stride(1) == 1
            and t.shape[0] == b.shape[0] and (t.shape[0] <= 1 or t.stride(0) == b.stride(0))):
        off = t.storage_offset() - b.storage_offset()
        if 0 <= off and off + t.shape[1] <= b.shape[1]:
            return b, off
    return t, 0


class AttnLengths:
    """Key lengths of an attention call checked on the host (each in [1, len_k], ``ValueError`` otherwise: the reference's soft-max
    over no key gives NaN rows) and uploaded once, so several ``attention`` calls share them without a read-back or a copy."""

    def __init__(self, lens, len_k: int, device):
        if isinstance(lens, torch.Tensor):
            if lens.dtype not in (torch.int32, torch.int64) or lens.dim() != 1:
                raise RuntimeError("tps_pp_b200: kv_lens must be a 1-D integer tensor or a sequence of ints")
            host = lens.tolist()                     # a device tensor is read back once: the lengths are checked before any launch
        else:
            host = [int(x) for x in lens]
        bad = [x for x in host if not 1 <= x <= int(len_k)]
        if bad:
            raise ValueError(f"tps_pp_b200: attention key lengths must lie in [1, {len_k}], got {bad[0]} (an image without a valid "
                             "key has no soft-max: the reference gives NaN rows)")
        self.host, self.len_k = tuple(host), int(len_k)
        self.dev = torch.tensor(host, dtype=torch.int32).to(device, non_blocking=True)


class _Attention(torch.autograd.Function):
    """Multi-head attention with native forward AND backward (``tpspp_attn_train_fwd`` / ``tpspp_attn_train_bwd``).  The inputs
    are the tensors q / k / v are column blocks of (``srcs``; ``where[n] = (source index, column offset)``); the gradient of
    each source is written by the kernels in place of its column blocks.  ``calls`` counts the forward launches."""

    calls = 0

    @staticmethod
    def forward(ctx, meta, *srcs):
        where, cfg_args, kv_lens = meta
        q, k, v = [srcs[s][:, off:off + cfg_args[1] * 64] for s, off in where]
        cfg = N.AttnTrainCfg(*cfg_args[:8], int(srcs[where[0][0]].stride(0)), int(srcs[where[1][0]].stride(0)))
        rows_q, d = cfg.batch * cfg.len_q, cfg.heads * 64
        out = torch.empty((rows_q, d), dtype=torch.float32, device=q.device)
        lse = torch.empty((cfg.batch, cfg.heads, cfg.len_q), dtype=torch.float32, device=q.device)
        _Attention.calls += 1
        seed = None
        if cfg.dropout_p > 0:
            # drawn on the device from torch's CUDA generator: torch.manual_seed reproduces it, no host sync
            seed = torch.randint(0, 2 ** 62, (1,), dtype=torch.int64, device=q.device)
        with torch.cuda.device(q.device):
            N.check(N.lib().tpspp_attn_train_fwd(ctypes.byref(cfg), _ptr(q), _ptr(k), _ptr(v), _ptr(kv_lens), _ptr(seed), _ptr(out),
                                                 _ptr(lse), _stream(q)), "tpspp_attn_train_fwd")
        ctx.save_for_backward(out, lse, *srcs)
        ctx.meta = (where, cfg_args, kv_lens, seed)
        ctx.mark_non_differentiable(lse)
        return out, lse

    @staticmethod
    def backward(ctx, gout, _glse):
        out, lse, *srcs = ctx.saved_tensors
        where, cfg_args, kv_lens, seed = ctx.meta
        d = cfg_args[1] * 64
        covered = [0] * len(srcs)
        for s, _ in where:
            covered[s] += d
        grads = [torch.empty_like(t) if covered[i] == t.shape[1] else torch.zeros_like(t) for i, t in enumerate(srcs)]
        q, k, v = [srcs[s][:, off:off + d] for s, off in where]
        gq, gk, gv = [grads[s][:, off:off + d] for s, off in where]
        cfg = N.AttnTrainCfg(*cfg_args[:8], int(srcs[where[0][0]].stride(0)), int(srcs[where[1][0]].stride(0)))
        gout = gout.contiguous()
        with torch.cuda.device(out.device):
            N.check(N.lib().tpspp_attn_train_bwd(ctypes.byref(cfg), _ptr(q), _ptr(k), _ptr(v), _ptr(out), _ptr(gout), _ptr(lse),
                                                 _ptr(kv_lens), _ptr(seed), _ptr(gq), _ptr(gk), _ptr(gv), _stream(out)),
                    "tpspp_attn_train_bwd")
        return (None, *grads)


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, len_q: int, len_k: int, temperature: float,
              kv_lens=None, causal: bool = False, dropout_p: float = 0.0) -> torch.Tensor:
    """Multi-head attention over whole sequences with native forward and backward (``tpspp_attn_train_fwd`` / ``_bwd``),
    differentiable in q, k and v: the reference's ``MultiHeadAttention`` core (transformer_module.py:24-34,74-98) between the
    projections, with its attention dropout.

    q [B*len_q, heads*64], k / v [B*len_k, heads*64] token-major fp32 -> out [B*len_q, heads*64].  Image b's query i attends to its
    keys j < kv_lens[b] (all len_k without ``kv_lens``) and, with ``causal``, j <= i; ``dropout_p`` > 0 drops probabilities with a
    seed drawn from torch's CUDA generator.  ``kv_lens``: an :class:`AttnLengths` (checked and uploaded once, for calls that
    share lengths), or host ints (a list or CPU tensor; a CUDA tensor is read back once) each in [1, len_k] -- ``ValueError``
    otherwise.  q / k / v may be column slices of one fused projection (k / v must share a row stride):
    their gradients are then written straight into the fused projection's gradient.  1 <= len_q, len_k <= 256."""
    for nm, t in (("q", q), ("k", k), ("v", v)):
        _require_cuda(nm, t, torch.float32)
    len_q, len_k, heads = int(len_q), int(len_k), int(heads)
    d = heads * 64
    if not (1 <= len_q <= 256 and 1 <= len_k <= 256):
        raise ValueError(f"tps_pp_b200: attention takes 1 <= len_q, len_k <= 256, got {len_q}, {len_k}")
    if not 0.0 <= float(dropout_p) < 1.0:
        raise ValueError(f"tps_pp_b200: attention dropout_p must lie in [0, 1), got {dropout_p}")
    if q.dim() != 2 or q.shape[1] != d or q.shape[0] % len_q:
        raise RuntimeError(f"tps_pp_b200: attention q must be [B*{len_q}, {d}] for {heads} heads, got {tuple(q.shape)}")
    b = q.shape[0] // len_q
    for nm, t, L in (("q", q, len_q), ("k", k, len_k), ("v", v, len_k)):
        if t.dim() != 2 or t.shape != (b * L, d) or t.stride(1) != 1 or t.device != q.device:
            raise RuntimeError(f"tps_pp_b200: attention `{nm}` must be [{b * L}, {d}] on {q.device} with unit stride along the features")
    srcs, where = [], []
    for t in (q, k, v):
        base, off = _fused_source(t)
        s = next((i for i, x in enumerate(srcs) if x is base), None)
        # the same columns used twice (attention(h, h, h)): a separate gradient buffer, summed by autograd
        if s is not None and any(ws == s and wo == off for ws, wo in where):
            s = None
        if s is None:
            if base is t and t.stride(0) != d and t.shape[0] > 1:
                base = t.contiguous()
            srcs.append(base)
            s = len(srcs) - 1
        where.append((s, off))
    if srcs[where[1][0]].stride(0) != srcs[where[2][0]].stride(0):
        raise RuntimeError("tps_pp_b200: attention k / v must share one row stride")
    lens = None
    if kv_lens is not None:
        if not isinstance(kv_lens, AttnLengths):
            kv_lens = AttnLengths(kv_lens, len_k, q.device)
        if len(kv_lens.host) != b or kv_lens.len_k > len_k or kv_lens.dev.device != q.device:
            raise RuntimeError(f"tps_pp_b200: kv_lens must have one entry per image ({b}), each <= len_k = {len_k}, on {q.device}")
        lens = kv_lens.dev
    cfg_args = (b, heads, 64, len_q, len_k, float(temperature), 1 if causal else 0, float(dropout_p))
    out, _ = _Attention.apply((tuple(where), cfg_args, lens), *srcs)
    return out
