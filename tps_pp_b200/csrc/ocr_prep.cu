// The text-recognition test pipeline of mmocr 0.4 -- ResizeOCR, ToTensorOCR, NormalizeOCR (reference
// datasets/pipelines/ocr_transforms.py:67-130) -- for a ragged batch of packed uint8 HWC images in one launch.
// One CTA per (image, output row), one thread per output column (looping when out_w > 128).  Each thread derives its column's
// source index and 11-bit weights itself, in the arithmetic of OpenCV's cv2.resize(INTER_LINEAR) on uint8:
//   per axis (src s, dst d): scale = 1 / (double(d) / s); f = float32((i + 0.5) * scale - 0.5); i0 = floor(f); f -= i0
//   x only: i0 < 0 -> (0, 0); i0 >= s - 1 -> (s - 1, 0).  y: rows i0, i0 + 1 clamped to [0, h - 1], weights unchanged
//   a0 = rint((1 - f) * 2048), a1 = rint(f * 2048)
//   H = S[i0x] a0 + S[min(i0x + 1, w - 1)] a1 (int32); v = ((H0 >> 4) b0 >> 16) + ((H1 >> 4) b1 >> 16); u = clamp((v + 2) >> 2)
// then columns x >= resize_w take the pad value (mmcv.impad in the uint8 domain), and every value becomes
// (u / 255.f - mean[c]) / std[c] with IEEE divisions (torchvision to_tensor + normalize).  The coefficient arithmetic uses
// explicit _rn intrinsics so that no multiply-add is contracted into an FMA: OpenCV's x86 build rounds each step.
// The rows of the fp32 output are written coalesced; the source bytes are gathered through L1 and every read is bounded by
// cfg.packed_bytes (the descriptors are not validated on the device).
// With TPSPP_OCR_FLAG_ROTATED (mmocr's MultiRotateAugOCR) a descriptor has a fifth field k, and the image resampled is
// np.rot90(S, k & 3) of the stored H x W image S (W x H for odd k).  The arithmetic above runs on the rotated frame's sizes, and
// each tap (i, j) of the rotated frame is read at its stored address off + 3 * (base + i * si + j * sj):
//   k = 0: S[i, j]          si =  W, sj =  1, base = 0
//   k = 1: S[j, W-1-i]      si = -1, sj =  W, base = W - 1
//   k = 2: S[H-1-i, W-1-j]  si = -W, sj = -1, base = H W - 1
//   k = 3: S[H-1-j, i]      si =  1, sj = -W, base = (H - 1) W
// so several descriptors can point at the same packed bytes.  The flag-less kernel is the ROTATED = false instantiation.
#include "common.cuh"

namespace tpspp {

constexpr int OP_THREADS = 128;

struct OcrPrepArgs {
  int out_h, out_w;
  float mean[3], std_[3];
  int pad;
  long long packed_bytes;
};

// source index and fractional part of destination index i along an axis of s source / d destination pixels
__device__ __forceinline__ float op_src_coord(int i, int s, int d, float* fl) {
  const double scale = __ddiv_rn(1.0, __ddiv_rn((double)d, (double)s));
  const float f = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)i, 0.5), scale), 0.5));
  *fl = floorf(f);
  return __fsub_rn(f, *fl);
}

__device__ __forceinline__ int op_coef(float w) { return __float2int_rn(__fmul_rn(w, 2048.f)); }

__device__ __forceinline__ float op_norm(int u, float mean, float std_) {
  return __fdiv_rn(__fsub_rn(__fdiv_rn((float)u, 255.f), mean), std_);
}

template <bool ROTATED>
__global__ void __launch_bounds__(OP_THREADS) ocr_prep_kernel(const uint8_t* __restrict__ packed, const long long* __restrict__ desc,
                                                              float* __restrict__ out, const OcrPrepArgs a) {
  constexpr int NF = ROTATED ? 5 : 4;       // descriptor fields
  const int img = blockIdx.x, y = blockIdx.y;
  const long long off = desc[NF * img];
  // clamped so that a corrupt descriptor cannot divide by zero or overflow the index arithmetic; reads are bounded below
  const int h = (int)min(max(desc[NF * img + 1], 1LL), 1LL << 30);
  const int w = (int)min(max(desc[NF * img + 2], 1LL), 1LL << 30);
  const int rw = (int)min(max(desc[NF * img + 3], 0LL), (long long)a.out_w);
  // the frame that is resampled (sh x sw) and its tap addresses relative to the image: base + i * si + j * sj pixels
  int sh = h, sw = w;
  long long si = w, sj = 1, base = 0;
  if constexpr (ROTATED) {
    const int k = (int)(desc[NF * img + 4] & 3);
    if (k & 1) { sh = w; sw = h; }
    si = k == 0 ? (long long)w : k == 1 ? -1LL : k == 2 ? -(long long)w : 1LL;
    sj = k == 0 ? 1LL : k == 1 ? (long long)w : k == 2 ? -1LL : -(long long)w;
    base = k == 0 ? 0LL : k == 1 ? (long long)w - 1 : k == 2 ? (long long)h * w - 1 : (long long)(h - 1) * w;
  }
  // vertical: rows and weights of this output row
  float fly = 0.f;
  const float fy = rw > 0 ? op_src_coord(y, sh, a.out_h, &fly) : 0.f;
  const int y0 = (int)fly;
  long long row0, row1;
  if constexpr (ROTATED) {
    row0 = off + 3LL * (base + si * min(max(y0, 0), sh - 1));
    row1 = off + 3LL * (base + si * min(max(y0 + 1, 0), sh - 1));
  } else {
    row0 = off + 3LL * w * min(max(y0, 0), h - 1);
    row1 = off + 3LL * w * min(max(y0 + 1, 0), h - 1);
  }
  const int b0 = op_coef(__fsub_rn(1.f, fy)), b1 = op_coef(fy);
  const size_t plane = (size_t)a.out_h * a.out_w;
  float* o = out + (size_t)img * 3 * plane + (size_t)y * a.out_w;
  for (int x = threadIdx.x; x < a.out_w; x += OP_THREADS) {
    int u[3] = {a.pad, a.pad, a.pad};
    if (x < rw) {
      float flx;
      float fx = op_src_coord(x, sw, rw, &flx);
      int x0;
      if (flx < 0.f) { x0 = 0; fx = 0.f; }
      else if (flx >= (float)(sw - 1)) { x0 = sw - 1; fx = 0.f; }
      else x0 = (int)flx;
      const int a0 = op_coef(__fsub_rn(1.f, fx)), a1 = op_coef(fx);
      const long long c0 = 3LL * sj * x0, c1 = 3LL * sj * min(x0 + 1, sw - 1);
      const long long at[4] = {row0 + c0, row0 + c1, row1 + c0, row1 + c1};
      int s[4][3];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const bool in = at[k] >= 0 && at[k] <= a.packed_bytes - 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) s[k][c] = in ? (int)__ldg(packed + at[k] + c) : 0;
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int h0 = s[0][c] * a0 + s[1][c] * a1, h1 = s[2][c] * a0 + s[3][c] * a1;
        const int v = (((h0 >> 4) * b0) >> 16) + (((h1 >> 4) * b1) >> 16);
        u[c] = min(max((v + 2) >> 2, 0), 255);
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) o[c * plane + x] = op_norm(u[c], a.mean[c], a.std_[c]);
  }
}

}  // namespace tpspp

using namespace tpspp;

extern "C" int tpspp_ocr_prep(const tpspp_ocr_prep_cfg* cfg, const uint8_t* packed, const int64_t* desc, float* out,
                              tpspp_stream_t stream) {
  reset_launch_count();
  TPSPP_REQUIRE(cfg != nullptr, "ocr_prep cfg is NULL");
  TPSPP_REQUIRE(cfg->n >= 1, "ocr_prep: n must be >= 1, got %d", cfg->n);
  TPSPP_REQUIRE(cfg->out_h >= 1 && cfg->out_w >= 1, "ocr_prep: out_h and out_w must be >= 1, got %d x %d", cfg->out_h, cfg->out_w);
  TPSPP_REQUIRE(cfg->out_h <= 65535, "ocr_prep: out_h must be <= 65535, got %d", cfg->out_h);
  for (int c = 0; c < 3; ++c)
    TPSPP_REQUIRE(cfg->std[c] != 0.f, "ocr_prep: std[%d] is 0 (NormalizeOCR divides by it)", c);
  TPSPP_REQUIRE(cfg->pad_value >= 0 && cfg->pad_value <= 255, "ocr_prep: pad_value must be in [0, 255], got %d", cfg->pad_value);
  TPSPP_REQUIRE((cfg->flags & ~TPSPP_OCR_FLAG_ROTATED) == 0, "ocr_prep: flags must be 0 or TPSPP_OCR_FLAG_ROTATED (%d), got %d",
                TPSPP_OCR_FLAG_ROTATED, cfg->flags);
  TPSPP_REQUIRE(cfg->packed_bytes >= 0, "ocr_prep: packed_bytes must be >= 0");
  TPSPP_REQUIRE(packed && desc && out, "tpspp_ocr_prep: null pointer");
  OcrPrepArgs a;
  a.out_h = cfg->out_h;
  a.out_w = cfg->out_w;
  for (int c = 0; c < 3; ++c) { a.mean[c] = cfg->mean[c]; a.std_[c] = cfg->std[c]; }
  a.pad = cfg->pad_value;
  a.packed_bytes = cfg->packed_bytes;
  const long long* d = reinterpret_cast<const long long*>(desc);
  if (cfg->flags & TPSPP_OCR_FLAG_ROTATED)
    ocr_prep_kernel<true><<<dim3(cfg->n, cfg->out_h), OP_THREADS, 0, (cudaStream_t)stream>>>(packed, d, out, a);
  else
    ocr_prep_kernel<false><<<dim3(cfg->n, cfg->out_h), OP_THREADS, 0, (cudaStream_t)stream>>>(packed, d, out, a);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  return TPSPP_OK;
}
