/*
 * tpspp.h -- C ABI of libtpspp.so: the B200-native (sm_100a) TPS++ rectifier hot path.
 *
 * This is the drop-in boundary for the path  TPS_PP.forward / TPSPreprocessor.forward
 * of simplify23/TPS_PP (an MMOCR 0.4.0 fork).  The reference is pure Python/PyTorch and has
 * no FFI of its own; every entry point below names the reference code it replaces
 * (paths relative to mmocr/models/textrecog/ in the reference tree).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless stated otherwise
 *   - the caller owns every buffer, including the workspace; the library never allocates
 *     device memory and never synchronises the host with the device
 *   - all work is enqueued on the given stream; calls are re-entrant per stream
 *   - return value: 0 = ok, negative = error (TPSPP_E_*); tpspp_last_error() gives a
 *     thread-local human readable message.  No C++ exception crosses this boundary.
 *   - tensors are dense row-major ("contiguous" NCHW); feature dtype is fp32 unless
 *     cfg.feat_dtype says bf16; coordinates, scores and control points are always fp32
 */
#ifndef TPSPP_H_
#define TPSPP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TPSPP_ABI_VERSION 2

#if defined(__GNUC__)
#define TPSPP_API __attribute__((visibility("default")))
#else
#define TPSPP_API
#endif

typedef struct CUstream_st* tpspp_stream_t; /* == cudaStream_t */

enum {
  TPSPP_OK = 0,
  TPSPP_E_INVALID = -1,     /* bad argument / unsupported shape */
  TPSPP_E_CUDA = -2,        /* a CUDA runtime call failed (message has the cudaError) */
  TPSPP_E_UNSUPPORTED = -3, /* requested variant cannot run this configuration */
  TPSPP_E_NO_DEVICE = -4    /* no sm_100 device */
};

/* TPSPP_SRC0_BF16: src0 is bf16, src1 and both outputs are fp32 -- the bf16 mode of the head hands its `feat_grid` to the
 * warp this way (staged TPS++ kernel only, forward only). */
enum { TPSPP_F32 = 0, TPSPP_BF16 = 1, TPSPP_SRC0_BF16 = 2 };

/* Which Phi the grid generator uses. */
enum {
  /* TPS++ : Phi[b,p,:] = [1, P_p, P_hat[p,:] * (1 + theta * pc_score[b,p,:])]
   *         backbones/tps_pp/tps_pp.py:467-479 (P_hat_score_process), P_hat is [n, F]        */
  TPSPP_MODE_ATTENTION = 0,
  /* RARE  : Phi[p,:] = P_hat[p,:] with P_hat already [n, F+3] = [1, P, rbf]
   *         preprocessor/tps_preprocessor.py:255-268,270-282                                  */
  TPSPP_MODE_CLASSICAL = 1
};

/* Kernel variant selection (0 lets the library choose; the others are for tests/bench). */
enum {
  TPSPP_VARIANT_AUTO = 0,
  TPSPP_VARIANT_GENERIC = 1, /* one thread per output pixel, direct global gathers            */
  TPSPP_VARIANT_STAGED = 2,  /* persistent CTAs, TMA bulk-copied source planes in shared mem  */
  TPSPP_VARIANT_TILED = 3    /* classical mode: P_hat tile resident in shared mem, batch-sliced */
};

/* Geometry of one fused warp call.  src1/out1 are the optional second sampled tensor
 * (TPS_PP samples feat_grid and batch_img with the same grid: tps_pp.py:606-615).          */
typedef struct tpspp_warp_cfg {
  int32_t batch;          /* B                                                              */
  int32_t channels0;      /* C of src0 / out0                                               */
  int32_t src0_h, src0_w; /* source plane of src0                                           */
  int32_t channels1;      /* C of src1 / out1, 0 when there is no second tensor             */
  int32_t src1_h, src1_w;
  int32_t out_h, out_w;   /* rectified size (Hr, Wr); n = Hr*Wr                             */
  int32_t num_fiducial;   /* F                                                              */
  int32_t mode;           /* TPSPP_MODE_*                                                   */
  float theta;            /* 0.5 in the reference ("thela", tps_pp.py:341)                  */
  int32_t feat_dtype;     /* TPSPP_F32 | TPSPP_BF16 (dtype of src0/src1/out0/out1) | TPSPP_SRC0_BF16 */
  int32_t variant;        /* TPSPP_VARIANT_*                                                */
} tpspp_warp_cfg;

TPSPP_API int tpspp_version(void);
TPSPP_API const char* tpspp_last_error(void);

/* Number of SMs of the current device and the cubin architecture that was loaded (e.g. 100). */
TPSPP_API int tpspp_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Measurement aid (bench.py): after tpspp_launch_profile(1) on the calling thread, tpspp_head_fwd records one CUDA
 * event on its stream before its first and after each of its kernel launches (the library creates up to 65 events
 * once and keeps them); tpspp_launch_profile_read synchronises on the last one and returns the milliseconds of the
 * launches of the most recent call in launch order (wprep, the 14 convolutions with cbam after the 10th, localisation,
 * DGAB gate, Mlp, feat_linear.0, feat_linear.1, score) followed by the launches of later calls on the same thread
 * (the module's tpspp_warp_fwd) until the next tpspp_head_fwd.  tpspp_launch_profile(0) turns it off. */
TPSPP_API int tpspp_launch_profile(int enable);
TPSPP_API int tpspp_launch_profile_read(float* ms, int capacity, int* count);

/* Bytes of scratch tpspp_warp_bwd needs for this cfg. */
TPSPP_API size_t tpspp_warp_workspace_bytes(const tpspp_warp_cfg* cfg);

/* Bytes of OPTIONAL scratch for tpspp_warp_fwd (0 in attention mode).  In classical mode with a large
 * rectified grid (>= 1024 pixels, batch x pixels >= 4 Mi, F <= 64) a 256-byte-aligned workspace of this size lets the
 * forward compute T = inv_delta_C[:, :F] . C' once per batch (tps_preprocessor.py:276-277) and run the
 * P_hat-stationary kernel (~2x faster at 64x256); with workspace == NULL the per-pixel kernel is used.
 * Results are the same either way. */
TPSPP_API size_t tpspp_warp_fwd_workspace_bytes(const tpspp_warp_cfg* cfg);

/*
 * Fused TPS grid generator + bilinear grid_sample (border padding, align_corners=True).
 *
 * Replaces, in one launch and without materialising Phi, T or the grid in HBM:
 *   Attention_Enhanced_TPS.build_P_prime + P_hat_score_process  (tps_pp.py:467-496)
 *   the reshape and both F.grid_sample calls of TPS_PP.forward   (tps_pp.py:601-615)
 * and for TPSPP_MODE_CLASSICAL
 *   GridGenerator.build_P_prime + F.grid_sample of TPSPreprocessor.forward
 *                                                     (tps_preprocessor.py:72-83,270-282)
 *
 *   src0        [B, C0, H0, W0]           feature map that is rectified ("feat_grid")
 *   src1        [B, C1, H1, W1] or NULL   second tensor sampled with the same grid ("batch_img")
 *   c_prime     [B, F, 2]      fp32       predicted control points C'
 *   pc_score    [B, n, F]      fp32       attention scores (ATTENTION mode) or NULL
 *   P_hat       ATTENTION: [n, F] rbf columns;  CLASSICAL: [n, F+3]           (module buffer)
 *   P           [n, 2] fp32 target pixel centres (ATTENTION mode; tps_pp.py:472) or NULL
 *   inv_delta_C [F+3, F+3] fp32 (module buffer "hat_C" / "inv_delta_C")
 *   out0        [B, C0, Hr, Wr]
 *   out1        [B, C1, Hr, Wr] or NULL
 *   grid_out    [B, n, 2] fp32 or NULL -- optional copy of the sampling grid (tests only;
 *               the generic variant writes it, the staged variant rejects a non-NULL value)
 *   workspace   NULL, or >= tpspp_warp_fwd_workspace_bytes(cfg) bytes, 256-byte aligned (see there)
 *
 * Arithmetic: T and Phi.T are evaluated in fp64 from the fp32 inputs and the source
 * coordinates / bilinear weights are derived in fp64; the four taps are blended in fp32 in
 * ATen's order (nw, ne, sw, se).
 */
TPSPP_API int tpspp_warp_fwd(const tpspp_warp_cfg* cfg, const void* src0, const void* src1,
                   const float* c_prime, const float* pc_score, const float* P_hat,
                   const float* P, const float* inv_delta_C, void* out0, void* out1,
                   float* grid_out, void* workspace, tpspp_stream_t stream);

/*
 * Bilinear sampler alone, for a caller-provided grid [B, Hr, Wr, 2] (x, y in [-1, 1]).
 * Bit-compatible restatement of torch's grid_sampler_2d CUDA kernel for
 * (bilinear, border, align_corners=True) -- the call at tps_pp.py:606-615 and
 * tps_preprocessor.py:79-83 -- in fp32 coordinate arithmetic.  Uses cfg geometry fields only.
 */
TPSPP_API int tpspp_sample_fwd(const tpspp_warp_cfg* cfg, const void* src0, const void* src1,
                     const float* grid, void* out0, void* out1, tpspp_stream_t stream);

/*
 * Backward of tpspp_warp_fwd (autograd of tps_pp.py:481-496,606-615 /
 * tps_preprocessor.py:72-83).  Recomputes the grid instead of saving it.
 *
 *   gout0/gout1  upstream gradients of out0/out1 (gout1 may be NULL)
 *   gsrc0/gsrc1  [like src0/src1] written (not accumulated); NULL skips that gradient
 *   g_c_prime    [B, F, 2] written; NULL skips
 *   g_pc_score   [B, n, F] written (ATTENTION mode); NULL skips
 *   workspace    >= tpspp_warp_workspace_bytes(cfg)
 */
TPSPP_API int tpspp_warp_bwd(const tpspp_warp_cfg* cfg, const void* src0, const void* src1,
                   const float* c_prime, const float* pc_score, const float* P_hat,
                   const float* P, const float* inv_delta_C, const void* gout0,
                   const void* gout1, void* gsrc0, void* gsrc1, float* g_c_prime,
                   float* g_pc_score, void* workspace, tpspp_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Control-point attention head: everything in TPS_PP.forward before the warp
 * (tps_pp.py:581-594): down0/1/2, down0_1/1_1, grid()/down_feat, MSFA encoder/CBAM/decoder,
 * TPE (DGAB, localization_fc1/2 -> C', p_linear/feat_linear + tanh(QK^T/8) -> pc_score).
 * ------------------------------------------------------------------------------------------ */
enum {
  TPSPP_HEAD_FP32 = 0,  /* CUDA-core fp32 FMAs everywhere (parity mode)                          */
  TPSPP_HEAD_TC = 1,    /* tcgen05 tensor cores, 3xTF32 error compensation: fp32-level accuracy          */
  TPSPP_HEAD_BF16 = 2   /* as TC, but the 14 convolutions use single-pass bf16 operands (fp32 accumulate) */
};

typedef struct tpspp_head_cfg {
  int32_t batch;            /* B                                                                 */
  int32_t height, width;    /* of batch_img (16, 64); outs are 2x that; width must be 64         */
  int32_t point_h, point_w; /* control-point lattice (2, 16)                                     */
  int32_t p_stride;         /* stride of the third MSFA encoder conv (2)                         */
  int32_t precision;        /* TPSPP_HEAD_*                                                      */
  int32_t flags;            /* TPSPP_HEAD_FLAG_* (0 = none)                                      */
} tpspp_head_cfg;

/* flags.  WEIGHTS_CACHED: the caller guarantees that `workspace` was last written by a tpspp_head_fwd call with the
 * same cfg and the same parameter VALUES (pointers and contents unchanged since), so the tensor-core weight images in
 * TPSPP_WS_WPREP are still valid and their re-layout launch is skipped.  The caller owns that invariant -- the
 * library cannot see weight updates (tps_pp_b200/rectifier.py keys it on torch's per-tensor version counters). */
/* UNFUSED_DOWN / UNFUSED_SCORE: run down0/down1/down2/down_feat (feat_linear.0/.1/QK^T) as separate launches instead of
 * the fused kernels (A/B measurements, tests).
 * TF32X3_CONV: run the 3x3 convolutions as all-tf32 3xTF32 (12 MMAs per 32-channel chunk) instead of the default tf32 main
 * term + bf16 correction terms (8 MMAs, same fp32-level accuracy; DESIGN.md section 4) -- A/B measurements, tests. */
/* FEATGRID_BF16 (precision TPSPP_HEAD_BF16 only): `feat_grid` is written as bf16 planes [B,64,2h,2w] (half the bytes of the
 * buffer are used) -- pass it to tpspp_warp_fwd as src0 with feat_dtype = TPSPP_SRC0_BF16. */
enum { TPSPP_HEAD_FLAG_WEIGHTS_CACHED = 1, TPSPP_HEAD_FLAG_UNFUSED_DOWN = 2, TPSPP_HEAD_FLAG_UNFUSED_SCORE = 4,
       TPSPP_HEAD_FLAG_TF32X3_CONV = 8, TPSPP_HEAD_FLAG_FEATGRID_BF16 = 16 };

/* Index of each learnable tensor in the `params` pointer table = state_dict order of the
 * reference module (SURVEY App. A-5; tps_pp.py:94-119,253-285,538-548).                      */
enum {
  TPSPP_P_ENC0_W = 0, TPSPP_P_ENC0_B, TPSPP_P_ENC1_W, TPSPP_P_ENC1_B, TPSPP_P_ENC2_W, TPSPP_P_ENC2_B,
  TPSPP_P_ENC3_W, TPSPP_P_ENC3_B, TPSPP_P_CBAM_MLP0_W, TPSPP_P_CBAM_MLP2_W, TPSPP_P_CBAM_SP_W,
  TPSPP_P_CBAM_SP_B, TPSPP_P_DEC0_W, TPSPP_P_DEC0_B, TPSPP_P_DEC1_W, TPSPP_P_DEC1_B, TPSPP_P_DEC2_W,
  TPSPP_P_DEC2_B, TPSPP_P_DEC3_W, TPSPP_P_DEC3_B, TPSPP_P_PLIN0_W, TPSPP_P_PLIN0_B, TPSPP_P_PLIN1_W,
  TPSPP_P_PLIN1_B, TPSPP_P_FLIN0_W, TPSPP_P_FLIN0_B, TPSPP_P_FLIN1_W, TPSPP_P_FLIN1_B,
  TPSPP_P_NORM1_W, TPSPP_P_NORM1_B, TPSPP_P_MLP_H_W, TPSPP_P_MLP_W_W, TPSPP_P_PROJ_W, TPSPP_P_PROJ_B,
  TPSPP_P_NORM2_W, TPSPP_P_NORM2_B, TPSPP_P_FC1_W, TPSPP_P_FC1_B, TPSPP_P_FC2_W, TPSPP_P_FC2_B,
  TPSPP_P_LOC1A_W, TPSPP_P_LOC1A_B, TPSPP_P_LOC1B_W, TPSPP_P_LOC1B_B, TPSPP_P_LOC2_W, TPSPP_P_LOC2_B,
  TPSPP_P_DOWN0_W, TPSPP_P_DOWN0_B, TPSPP_P_DOWN1_W, TPSPP_P_DOWN1_B, TPSPP_P_DOWN2_W, TPSPP_P_DOWN2_B,
  TPSPP_P_DOWN0_1_W, TPSPP_P_DOWN0_1_B, TPSPP_P_DOWN1_1_W, TPSPP_P_DOWN1_1_B, TPSPP_P_DOWNFEAT_W,
  TPSPP_P_DOWNFEAT_B, TPSPP_P_COUNT
};

/* Intermediates kept in the workspace (float offsets via tpspp_head_workspace_offsets; tests and
 * the backward pass read them). */
enum {
  TPSPP_WS_F0 = 0, TPSPP_WS_F1, TPSPP_WS_F2, TPSPP_WS_A0, TPSPP_WS_A1, TPSPP_WS_E0, TPSPP_WS_E1,
  TPSPP_WS_E2, TPSPP_WS_E3 /* en_feat, pre-CBAM */, TPSPP_WS_CBAM, TPSPP_WS_D0, TPSPP_WS_D1, TPSPP_WS_D2,
  TPSPP_WS_DE /* de_feat */, TPSPP_WS_X1, TPSPP_WS_V, TPSPP_WS_DE2 /* de_feat after DGAB */,
  TPSPP_WS_P1 /* p_linear(en) [B,F,128] */,
  TPSPP_WS_WPREP /* tensor-core weight images */, TPSPP_WS_T1, TPSPP_WS_FS /* feat_linear outputs */,
  TPSPP_WS_HID /* Mlp hidden */, TPSPP_WS_P1IMG /* per-image score weights */, TPSPP_WS_COUNT
};

TPSPP_API size_t tpspp_head_workspace_bytes(const tpspp_head_cfg* cfg);
/* offsets[TPSPP_WS_COUNT] in BYTES from the workspace base (host call) */
TPSPP_API int tpspp_head_workspace_offsets(const tpspp_head_cfg* cfg, size_t* offsets);

/*
 * x [B,64,h,w], o0/o1 [B,32,2h,2w] fp32 NCHW; params: HOST array of TPSPP_P_COUNT DEVICE pointers
 * (each contiguous and 16-byte aligned, as torch allocates them).
 * Outputs: feat_grid [B,64,2h,2w] (tps_pp.py:585), c_prime [B,F,2] (tps_pp.py:321-323),
 *          pc_score [B,h*w,F] (tps_pp.py:324).  workspace: 256-byte aligned,
 *          >= tpspp_head_workspace_bytes(cfg).
 */
TPSPP_API int tpspp_head_fwd(const tpspp_head_cfg* cfg, const float* x, const float* o0, const float* o1,
                             const float* const* params, float* feat_grid, float* c_prime,
                             float* pc_score, void* workspace, tpspp_stream_t stream);

/* ---- Backbone stage in front of the rectifier (SURVEY.md section 8f rank 3) -------------------------------------
 * Replaces what `ResNetABI_v2_large.forward` computes before it calls `tpsnet(x, outs)`
 * (backbones/resnet_v2_large.py:131-135 stem, :109-129 layers, :176-191 forward; block = layers/conv_layer.py:12-33 over
 * mmcv's BasicBlock), eval mode: stem conv+BN+ReLU, layer1 (3 blocks, 32 ch), layer2 (4 blocks, 64 ch, stride 2).
 * The reference-side binding is `tps_pp_b200/backbone.py` (drop-in `ResNetABI_v2_large`). */
typedef struct {
  int32_t batch;
  int32_t height, width;    /* image size (32 x 128); o0/o1 are [B,32,H,W], x is [B,64,H/2,W/2]      */
  int32_t precision;        /* TPSPP_HEAD_TC                                                     */
  int32_t flags;            /* TPSPP_HEAD_FLAG_WEIGHTS_CACHED: folded BN + weight images in `workspace` still valid */
} tpspp_stage_cfg;

/* params table = the stage's slice of the reference state_dict, in its order, without the int64 num_batches_tracked
 * buffers: conv1.{weight,bias}, bn1.{weight,bias,running_mean,running_var}, then per block conv1.weight, bn1 x4,
 * conv2.weight, bn2 x4 and, for layer2.0, downsample.0.weight, downsample.1 x4. */
enum {
  TPSPP_SP_CONV1_W = 0, TPSPP_SP_CONV1_B, TPSPP_SP_BN1_W, TPSPP_SP_BN1_B, TPSPP_SP_BN1_MEAN, TPSPP_SP_BN1_VAR,
  TPSPP_SP_LAYER1 = 6,      /* 3 blocks x 10 tensors  */
  TPSPP_SP_LAYER2 = 36,     /* 15 tensors (with downsample) + 3 blocks x 10 */
  TPSPP_SP_COUNT = 81
};

TPSPP_API size_t tpspp_stage_workspace_bytes(const tpspp_stage_cfg* cfg);
/* img [B,3,H,W] fp32 NCHW -> o0 (stem output) and o1 (layer1 output) [B,32,H,W], x (layer2 output) [B,64,H/2,W/2]:
 * exactly the tensors tpspp_head_fwd / tpspp_warp_fwd take.  params: HOST array of TPSPP_SP_COUNT DEVICE pointers.
 * workspace: 256-byte aligned, >= tpspp_stage_workspace_bytes(cfg). */
TPSPP_API int tpspp_stage_fwd(const tpspp_stage_cfg* cfg, const float* img, const float* const* params, float* o0, float* o1,
                              float* x, void* workspace, tpspp_stream_t stream);

/* ---- Classical (RARE) localisation network (SURVEY.md section 8f rank 4) -------------------------------------------
 * Replaces `TPSPreprocessor.LocalizationNetwork.forward` (preprocessor/tps_preprocessor.py:96-156), eval mode: four
 * conv3x3 + BatchNorm + ReLU blocks (C -> 64 -> 128 -> 256 -> 512, MaxPool2d(2) after the first three, AdaptiveAvgPool2d(1)
 * after the last), localization_fc1 (512 -> 256, ReLU), localization_fc2 (256 -> 2F) -> C' [B, F, 2], which
 * tpspp_warp_fwd (classical mode) takes.  The reference-side binding is `tps_pp_b200/classical.py::TPSPreprocessor.localize`. */
typedef struct {
  int32_t batch, channels;  /* channels: 1 or 3                                                              */
  int32_t height, width;    /* multiples of 8 whose /2, /4, /8 maps tile into 128-pixel rectangles: 64x256, 64x128, 32x256, ... */
  int32_t num_fiducial;
  int32_t flags;            /* TPSPP_HEAD_FLAG_WEIGHTS_CACHED: folded BN + weight images in `workspace` still valid */
} tpspp_locnet_cfg;
/* params table = the LocalizationNetwork slice of the reference state_dict, in its order, without num_batches_tracked:
 * conv.{0,4,8,12}.weight each followed by its BatchNorm's weight, bias, running_mean, running_var; then
 * localization_fc1.0.{weight,bias}, localization_fc2.{weight,bias}. */
enum { TPSPP_LP_FC1_W = 20, TPSPP_LP_FC1_B, TPSPP_LP_FC2_W, TPSPP_LP_FC2_B, TPSPP_LP_COUNT = 24 };
TPSPP_API size_t tpspp_locnet_workspace_bytes(const tpspp_locnet_cfg* cfg);   /* 0: unsupported geometry (tpspp_last_error) */
/* img [B,C,H,W] fp32 -> c_prime [B, F, 2].  params: HOST array of TPSPP_LP_COUNT DEVICE pointers. */
TPSPP_API int tpspp_locnet_fwd(const tpspp_locnet_cfg* cfg, const float* img, const float* const* params, float* c_prime,
                               void* workspace, tpspp_stream_t stream);

/* ---- Training-path convolution: forward and backward of one ConvModule (conv + bias + ReLU; reference
 * tps_pp.py:126-131,149-154,538-548), so that autograd of the rectifier's convolutions runs on native kernels
 * (north_star (4); the reference side is torch autograd of nn.Conv2d + ReLU).  NCHW fp32, 64 output channels. */
typedef struct {
  int32_t batch, cin;       /* cin: 32 or a multiple of 64                                        */
  int32_t height, width;    /* input size; output = input / stride                                */
  int32_t ksize;            /* 1 (stride 1) or 3 (pad 1)                                          */
  int32_t stride_h, stride_w; /* (1,1), (2,2) or (2,1)                                            */
  int32_t relu;             /* 1: y = relu(conv + b), 0: y = conv + b                             */
  /* torch.cat / F.interpolate fused into the convolution (tps_pp.py:159-168,583-585); all zero = one plain source */
  int32_t nsrc;             /* 0/1: one source; 2/3: the input is the channel concatenation of nsrc 64-channel sources (cin = 64 nsrc) */
  int32_t up_h[3], up_w[3]; /* nearest-upsample factor of each source (0/1 or 2): source s is stored [B, C, height/up_h, width/up_w] */
} tpspp_conv_cfg;
TPSPP_API size_t tpspp_conv_workspace_bytes(const tpspp_conv_cfg* cfg);   /* covers both calls */
/* y [B,64,H/sh,W/sw] = act(conv(x [B,cin,H,W], w [64,cin,k,k]) + bias [64]) */
TPSPP_API int tpspp_conv_fwd(const tpspp_conv_cfg* cfg, const float* x, const float* w, const float* bias, float* y,
                             void* workspace, tpspp_stream_t stream);
/* gradients of the above given y (the saved output) and gy: gx [B,cin,H,W], gw [64,cin,k,k], gb [64]; each may be NULL */
TPSPP_API int tpspp_conv_bwd(const tpspp_conv_cfg* cfg, const float* x, const float* w, const float* y, const float* gy,
                             float* gx, float* gw, float* gb, void* workspace, tpspp_stream_t stream);

/* ---- Training-path linear layers: forward and backward of the reference's nn.Linear / torch.bmm calls (DGAB.py:11-23,
 * 28-36,52; tps_pp.py:250-273 localization_fc1/fc2, p_linear, feat_linear; :293-299 the einsum of atten_score), so that
 * autograd of the rectifier's dense layers runs on native kernels instead of cuBLAS.  Row-major fp32:
 *   y [rows, out] = x [rows, in] . w[out, in]^T + bias          (weight_batches == 1: nn.Linear)
 *   y_b = x_b . w_b^T for weight_batches equal groups of rows     (weight_batches  > 1: torch.bmm(x, w.transpose(1, 2)))
 * tcgen05 3xTF32 kernels when rows (per batch) % 128 == 0 and in/out features % 32 == 0 (the TMA-fed kernel for in <= 64 or
 * out <= 64, the shared-memory-operand kernel for larger layers such as 512 -> 1536); fp32 CUDA-core kernels for every other shape.  No activation: the caller applies it (and its derivative). */
typedef struct {
  int64_t rows;             /* product of the leading dimensions                                  */
  int32_t in_features, out_features;
  int32_t weight_batches;   /* 1, or the number of [out, in] weights (rows % weight_batches == 0)  */
  int32_t flags;            /* TPSPP_LINEAR_FLAG_WEIGHTS_CACHED: `workspace` still holds the operand images of these weight VALUES
                             * from an earlier tpspp_linear_fwd call with the same cfg (their re-layout launch is skipped; the
                             * caller owns that invariant, as for TPSPP_HEAD_FLAG_WEIGHTS_CACHED) */
} tpspp_linear_cfg;
enum { TPSPP_LINEAR_FLAG_WEIGHTS_CACHED = 1 };
TPSPP_API size_t tpspp_linear_workspace_bytes(const tpspp_linear_cfg* cfg);   /* covers both calls */
TPSPP_API int tpspp_linear_fwd(const tpspp_linear_cfg* cfg, const float* x, const float* w, const float* bias /* or NULL */,
                               float* y, void* workspace, tpspp_stream_t stream);
/* y = act(x w^T + bias) + residual: the inference form with the epilogue a transformer layer needs (residual [rows, out] or
 * NULL; act = TPSPP_ACT_NONE | TPSPP_ACT_GELU (erf form)); weight_batches must be 1. */
enum { TPSPP_ACT_NONE = 0, TPSPP_ACT_GELU = 1 };
TPSPP_API int tpspp_linear_fwd_ex(const tpspp_linear_cfg* cfg, const float* x, const float* w, const float* bias, const float* residual,
                                  int32_t act, float* y, void* workspace, tpspp_stream_t stream);
/* ... and with the NEXT sub-layer's LayerNorm attached (a pre-norm transformer layer, nrtr_decoder.py / tf_layers: x = x + f(.)
 * is followed at once by LN(x)): y as above, y_ln = LayerNorm(y; ln_weight, ln_bias or NULL, ln_eps) [rows, out] -- computed by the
 * kernel that finishes y (the split-K reduction), one warp per row.  y_ln == NULL: exactly tpspp_linear_fwd_ex.  With y_ln:
 * act must be TPSPP_ACT_NONE, out_features % 128 == 0 and <= 1024, y_ln must not alias x / y / residual, 16-byte aligned pointers. */
TPSPP_API int tpspp_linear_ln_fwd(const tpspp_linear_cfg* cfg, const float* x, const float* w, const float* bias, const float* residual,
                                  int32_t act, float* y, const float* ln_weight, const float* ln_bias, float ln_eps, float* y_ln,
                                  void* workspace, tpspp_stream_t stream);
/* gx [rows, in] (or NULL), gw [batches, out, in] (or NULL), gb [out] (or NULL; needs gw) from gy [rows, out] */
TPSPP_API int tpspp_linear_bwd(const tpspp_linear_cfg* cfg, const float* x, const float* w, const float* gy, float* gx,
                               float* gw, float* gb, void* workspace, tpspp_stream_t stream);

/* The same pair for a ConvModule whose input is torch.cat(sources, dim=1) and/or F.interpolate(source, mode="nearest"):
 * xs / gxs are arrays of cfg->nsrc pointers (gxs entries may be NULL); gxs[s] has the STORED (low-resolution) shape of source s. */
TPSPP_API int tpspp_convcat_fwd(const tpspp_conv_cfg* cfg, const float* const* xs, const float* w, const float* bias, float* y,
                                void* workspace, tpspp_stream_t stream);
TPSPP_API int tpspp_convcat_bwd(const tpspp_conv_cfg* cfg, const float* const* xs, const float* w, const float* y, const float* gy,
                                float* const* gxs, float* gw, float* gb, void* workspace, tpspp_stream_t stream);

/* ---- Single-query attention over a key/value cache: the per-step attention of NRTRDecoder.forward_test (reference
 * decoders/nrtr_decoder.py:153-177; MultiHeadAttention / ScaledDotProductAttention, common/modules/transformer_module.py:
 * 24-34,74-98) for a greedy decode that keeps the keys / values of earlier positions (SURVEY.md section 8f rank 2; the
 * reference-side binding is tps_pp_b200/nrtr.py::NRTRDecoder.forward_test).
 *   out[b,h,:] = sum_t softmax_t((q[b,h,:] / temperature) . K[b,t,h,:]) V[b,t,h,:],  t < kv_len (or kv_lens[b] when given)
 * q / out [batch, heads*64] row-major fp32; k / v [batch, kv_capacity, heads*64]. */
typedef struct {
  int32_t batch, heads, head_dim;   /* head_dim = 64                                                        */
  int32_t kv_len, kv_capacity;      /* keys used (all images) / rows allocated per image                    */
  float temperature;                /* d_k ** 0.5 in the reference                                          */
  int32_t q_stride, new_stride;     /* floats between consecutive images' rows of q and of k_new / v_new (0 = heads*64): lets q, k_new,
                                       v_new be column slices of one fused q|k|v projection                                     */
  int32_t kv_head_major;            /* 0: k / v are [batch, kv_capacity, heads*64]; 1: [batch, heads, kv_capacity, 64] (contiguous per head) */
} tpspp_attn_cfg;
/* k_new / v_new (or NULL): this step's key / value rows; the kernel stores them at cache position kv_len - 1 (kv_lens[b] - 1)
 * before it attends, so the caller needs no separate cache-append copy. */
TPSPP_API int tpspp_attn_decode(const tpspp_attn_cfg* cfg, const float* q, float* k, float* v,
                                const int32_t* kv_lens /* [batch] device pointer or NULL */, const float* k_new, const float* v_new,
                                float* out, tpspp_stream_t stream);

/* ---- Multi-head self-attention over whole sequences: the attention of NRTREncoder (reference encoders/nrtr_encoder.py:66-87;
 * TFEncoderLayer -> MultiHeadAttention / ScaledDotProductAttention, common/modules/transformer_module.py:24-34,74-98) with the
 * encoder's source mask (_get_mask); the reference-side binding is tps_pp_b200/nrtr.py::NRTREncoder.
 *   out[b,i,h,:] = sum_{j < len(b)} softmax_j((q[b,i,h,:] / temperature) . K[b,j,h,:]) V[b,j,h,:]   for every i < seq_len
 * q / k / v: token-major [batch*seq_len, heads*64] fp32 rows `row_stride` floats apart (column slices of one fused q|k|v
 * projection allowed); out: [batch*seq_len, heads*64] row-major.  len(b) = kv_lens[b] (clamped to [0, seq_len]) or seq_len.
 * Every query row is computed, also i >= len(b); len(b) = 0 gives NaN rows (the reference's soft-max over no key).
 * fp32 on CUDA cores, online soft-max; any seq_len >= 1.  Pointers 16-byte aligned. */
typedef struct tpspp_attn_encode_cfg {
  int32_t batch, heads, head_dim;   /* batch <= 65535; head_dim = 64                                        */
  int32_t seq_len;                  /* T: tokens per image (queries and keys)                               */
  float temperature;                /* d_k ** 0.5 in the reference                                          */
  int32_t row_stride;               /* floats between consecutive token rows of q / k / v (0 = heads*64; a multiple of 4) */
} tpspp_attn_encode_cfg;
TPSPP_API int tpspp_attn_encode(const tpspp_attn_encode_cfg* cfg, const float* q, const float* k, const float* v,
                                const int32_t* kv_lens /* [batch] device pointer or NULL */, float* out, tpspp_stream_t stream);

/* ---- Training attention: forward and backward of the NRTR encoder's self-attention, the decoder's causal self-attention and
 * its cross-attention over the encoder memory, with the reference's attention dropout (ScaledDotProductAttention,
 * common/modules/transformer_module.py:24-34: P_drop = P * keep / (1 - dropout_p)).
 *   S[b,h,i,j] = (q[b,i,h,:] / temperature) . k[b,j,h,:]   over keys j < len(b) and, with `causal`, j <= i
 *   out[b,i,h,:] = sum_j softmax_j(S)[b,h,i,j] keep(b,h,i,j) / (1 - dropout_p) v[b,j,h,:]      for every i < len_q
 * q [batch*len_q, heads*64] rows q_stride floats apart; k / v [batch*len_k, heads*64] rows kv_stride floats apart (q, k, v may be
 * column slices of one fused q|k|v projection, k / v of one fused k|v projection); out [batch*len_q, heads*64] row-major;
 * lse [batch, heads, len_q]: the log-sum-exp of each row of S over its valid keys, which the backward pass recomputes P from.
 * len(b) = kv_lens[b] (device int32, >= 1; the caller checks it) or len_k.  Every query row is computed, also i >= len(b).
 * keep(b,h,i,j) is bit r = i mod 4 of Philox4x32-10 (counter (j, i / 4, h, b), key = the 64-bit seed at seed_ptr) compared with
 * dropout_p * 2^32: no mask is stored and the backward pass regenerates it.  seed_ptr is a device pointer (read by the kernels,
 * so a seed drawn on the device needs no host sync, and with device-resident kv_lens the calls can be captured in a graph); with dropout_p = 0 nothing is
 * drawn and seed_ptr may be NULL.  1 <= len_q, len_k <= 256; fp32 on CUDA cores; pointers 16-byte aligned. */
typedef struct tpspp_attn_train_cfg {
  int32_t batch, heads, head_dim;   /* batch <= 65535; head_dim = 64                                        */
  int32_t len_q, len_k;             /* queries / keys per image, 1..256                                     */
  float temperature;                /* d_k ** 0.5 in the reference                                          */
  int32_t causal;                   /* 1: key j is also masked for query i < j (decoder self-attention)     */
  float dropout_p;                  /* attention dropout, 0 <= p < 1                                        */
  int32_t q_stride, kv_stride;      /* floats between consecutive rows of q (and gq) / of k, v (and gk, gv); 0 = heads*64; multiples of 4 */
} tpspp_attn_train_cfg;
TPSPP_API int tpspp_attn_train_fwd(const tpspp_attn_train_cfg* cfg, const float* q, const float* k, const float* v,
                                   const int32_t* kv_lens /* [batch] device pointer or NULL */, const uint64_t* seed_ptr,
                                   float* out, float* lse, tpspp_stream_t stream);
/* dq / dk / dv from gout (= dL/dout) by recomputation: P = exp(S - lse), D = rowsum(gout * out), dS = P * (dP - D) with
 * dP = (gout . v^T) * keep / (1 - p).  gq has q's row stride, gk / gv kv_stride (they may be column slices of one fused gradient
 * buffer); every row is written (zeros for keys j >= len(b)).  No floating-point atomics: query-block CTAs write dq, key-block
 * CTAs dk and dv, so two calls on the same inputs give the same bits. */
TPSPP_API int tpspp_attn_train_bwd(const tpspp_attn_train_cfg* cfg, const float* q, const float* k, const float* v, const float* out,
                                   const float* gout, const float* lse, const int32_t* kv_lens, const uint64_t* seed_ptr,
                                   float* gq, float* gk, float* gv, tpspp_stream_t stream);

/* ---- Text-recognition test pipeline: mmocr 0.4 ResizeOCR -> ToTensorOCR -> NormalizeOCR (reference
 * datasets/pipelines/ocr_transforms.py:67-130) for a whole ragged batch of uint8 images in one launch.
 *   packed  uint8 HWC images, 3 channels in the caller's channel order (no BGR/RGB swap), one after the other
 *   desc    [n][4] int64 device array: byte offset of the image in `packed`, h, w, resize_w (the width ResizeOCR chose);
 *           with TPSPP_OCR_FLAG_ROTATED [n][5]: the same four (h, w of the STORED image), then k, the number of quarter turns
 *           counter-clockwise (np.rot90(img, k)); the kernel uses k & 3.  Several descriptors may share one offset.
 *   out     [n, 3, out_h, out_w] fp32 NCHW
 * Pixel (c, y, x) of image i: x < resize_w: cv2.resize(img, (resize_w, out_h), INTER_LINEAR) on uint8 (OpenCV's fixed-point
 * arithmetic, bit for bit), where img is np.rot90(stored, k) with TPSPP_OCR_FLAG_ROTATED (w x h for odd k) and the stored
 * image otherwise; x >= resize_w: pad_value (mmcv.impad).  Then ((float)u8 / 255 - mean[c]) / std[c] in fp32 with
 * IEEE divisions (torchvision to_tensor + normalize).  The library cannot read the descriptors without a host sync, so it does
 * not validate them; every read of `packed` is bounded by packed_bytes, so a corrupt descriptor gives wrong pixels but never an
 * out-of-range access.  The Python wrapper (tps_pp_b200/functional.py::ocr_prep) checks descriptors on the host. */
typedef struct tpspp_ocr_prep_cfg {
  int32_t n;                /* images (descriptors)                                                 */
  int32_t out_h, out_w;     /* ResizeOCR height, max_width                                          */
  float mean[3], std[3];    /* NormalizeOCR, per channel of the caller's order; std != 0            */
  int32_t pad_value;        /* ResizeOCR img_pad_value, uint8 domain [0, 255]                       */
  int32_t flags;            /* 0 or TPSPP_OCR_FLAG_ROTATED; any other bit is rejected               */
  int64_t packed_bytes;     /* size of `packed`: every read stays below it                          */
} tpspp_ocr_prep_cfg;
enum { TPSPP_OCR_FLAG_ROTATED = 2 };  /* desc is [n][5]: rotation test-time augmentation (mmocr MultiRotateAugOCR) */
TPSPP_API int tpspp_ocr_prep(const tpspp_ocr_prep_cfg* cfg, const uint8_t* packed, const int64_t* desc, float* out,
                             tpspp_stream_t stream);

/* Number of kernel launches the most recent call on this host thread enqueued
 * (bench.py uses it to report gpu_launches). */
TPSPP_API int tpspp_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* TPSPP_H_ */
