// Backward of the fused warp (autograd of reference tps_pp.py:481-496,606-615 and
// tps_preprocessor.py:72-83,270-282; sampler rules from ATen grid_sampler_2d_backward).
//
//   K-B1 warp_bwd_sample_kernel : recompute grid -> d src (scatter-add) and d grid
//   K-B2 grid_bwd_reduce_kernel : d pc_score (elementwise) and partial dT = Phi^T . dgrid
//   K-B3 cprime_bwd_kernel      : dC' = inv_delta_C[:, :F]^T . dT
//
// Maths (SURVEY App. A-3): with taps v_nw..v_se (0 outside the plane) and upstream G[c]
//   d/d ix = sum_c G[c] * (uy*(v_ne - v_nw) + ty*(v_se - v_sw))
//   d/d iy = sum_c G[c] * (ux*(v_sw - v_nw) + tx*(v_se - v_ne))
//   d/d gx = d/d ix * (W-1)/2 * [0 < ix_unclipped < W-1]          (same for y)
//   dT = Phi^T dgrid,  dC' = inv_delta_C[:, :F]^T dT,  dpc_score = theta * P_hat o (dgrid . T[3:]^T)
#include "common.cuh"

namespace tpspp {

template <typename FT>
__device__ __forceinline__ void atomic_addf(FT* p, float v);
template <>
__device__ __forceinline__ void atomic_addf<float>(float* p, float v) { atomicAdd(p, v); }
template <>
__device__ __forceinline__ void atomic_addf<__nv_bfloat16>(__nv_bfloat16* p, float v) {
  atomicAdd(p, __float2bfloat16_rn(v));
}

template <typename FT>
__device__ __forceinline__ void bwd_one_source(const FT* __restrict__ src, const FT* __restrict__ gout,
                                               FT* __restrict__ gsrc, const TapsGrad& g, int c_lo, int c_hi,
                                               size_t plane, int n, float& gix, float& giy) {
  const int dx = g.t.dx, dy = g.t.dy;
  for (int c = c_lo; c < c_hi; ++c) {
    const float G = ldf(gout + (size_t)c * n);
    const FT* s = src + (size_t)c * plane + g.t.off;
    const float vnw = ldf(s);
    const float vne = dx ? ldf(s + dx) : 0.f;
    const float vsw = dy ? ldf(s + dy) : 0.f;
    const float vse = (dx && dy) ? ldf(s + dy + dx) : 0.f;
    gix = __fmaf_rn(G, g.uy * (vne - vnw) + g.ty * (vse - vsw), gix);
    giy = __fmaf_rn(G, g.ux * (vsw - vnw) + g.tx * (vse - vne), giy);
    if (gsrc != nullptr) {
      FT* d = gsrc + (size_t)c * plane + g.t.off;
      atomic_addf<FT>(d, G * g.t.w[0]);
      if (dx) atomic_addf<FT>(d + dx, G * g.t.w[1]);
      if (dy) atomic_addf<FT>(d + dy, G * g.t.w[2]);
      if (dx && dy) atomic_addf<FT>(d + dy + dx, G * g.t.w[3]);
    }
  }
}

template <typename FT, int MODE>
__global__ void __launch_bounds__(256) warp_bwd_sample_kernel(WarpParams p, int cchunk, int use_atomic_grid) {
  extern __shared__ double Tsm[];
  const int b = blockIdx.y;
  compute_T(p, b, Tsm, threadIdx.x, blockDim.x);
  __syncthreads();
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= p.n) return;
  double gx, gy;
  pixel_grid<MODE>(p, Tsm, b, pix, gx, gy);
  const int cb = blockIdx.z * cchunk;
  float ggx = 0.f, ggy = 0.f;
  {
    const TapsGrad g = make_taps_grad<double>(gx, gy, p.W0, p.H0);
    const size_t plane = (size_t)p.H0 * p.W0;
    float gix = 0.f, giy = 0.f;
    const int ce = min(p.C0, cb + cchunk);
    if (cb < ce)
      bwd_one_source<FT>((const FT*)p.src0 + (size_t)b * p.C0 * plane,
                         (const FT*)p.gout0 + (size_t)b * p.C0 * p.n + pix,
                         p.gsrc0 ? (FT*)p.gsrc0 + (size_t)b * p.C0 * plane : nullptr, g, cb, ce, plane, p.n,
                         gix, giy);
    ggx = gix * g.mx; ggy = giy * g.my;
  }
  if (p.C1 > 0 && p.gout1 != nullptr) {
    const TapsGrad g = make_taps_grad<double>(gx, gy, p.W1, p.H1);
    const size_t plane = (size_t)p.H1 * p.W1;
    float gix = 0.f, giy = 0.f;
    const int ce = min(p.C1, cb + cchunk);
    if (cb < ce)
      bwd_one_source<FT>((const FT*)p.src1 + (size_t)b * p.C1 * plane,
                         (const FT*)p.gout1 + (size_t)b * p.C1 * p.n + pix,
                         p.gsrc1 ? (FT*)p.gsrc1 + (size_t)b * p.C1 * plane : nullptr, g, cb, ce, plane, p.n,
                         gix, giy);
    ggx = __fmaf_rn(gix, g.mx, ggx); ggy = __fmaf_rn(giy, g.my, ggy);
  }
  float* gg = p.g_grid + ((size_t)b * p.n + pix) * 2;
  if (use_atomic_grid) {
    atomicAdd(gg, ggx);
    atomicAdd(gg + 1, ggy);
  } else {
    gg[0] = ggx;
    gg[1] = ggy;
  }
}

// One warp per pixel step: lane <-> rbf column (coalesced rows of P_hat / pc_score / g_pc_score),
// 8 pixel rows per CTA, fp64 accumulation of the column sums, deterministic partials.
//   partial layout: [B][nsplit][K][2] doubles
constexpr int GB_ROWS = 8;
constexpr int GB_MAXI = 4;   // ceil(128/32) column groups per lane

template <int MODE>
__global__ void __launch_bounds__(32 * GB_ROWS) grid_bwd_reduce_kernel(WarpParams p, int nsplit, double* partial) {
  extern __shared__ double sm[];          // T[2K] then reduction scratch [GB_ROWS][2K]
  double* Tsm = sm;
  double* red = sm + 2 * p.K;
  const int b = blockIdx.y, split = blockIdx.x;
  const int lane = threadIdx.x & 31, row = threadIdx.x >> 5;
  compute_T(p, b, Tsm, threadIdx.x, blockDim.x);
  __syncthreads();
  const int per = (p.n + nsplit - 1) / nsplit;
  const int p_lo = split * per, p_hi = min(p.n, p_lo + per);
  const int ncol = (MODE == 0) ? p.F : p.K;          // streamed columns of P_hat
  double ax[GB_MAXI], ay[GB_MAXI];
#pragma unroll
  for (int i = 0; i < GB_MAXI; ++i) { ax[i] = 0.0; ay[i] = 0.0; }
  double a0x = 0, a0y = 0, a1x = 0, a1y = 0, a2x = 0, a2y = 0;   // affine columns (attention, lane 0)
  const float th = p.theta;
  if (MODE == 0 && p.F == 32 &&
      (((uintptr_t)p.P_hat | (uintptr_t)p.score | (uintptr_t)p.g_score | (uintptr_t)p.P) & 15) == 0) {
    // TPS++ geometry (F = 32), 16-byte aligned tensors.  A warp takes FOUR consecutive pixel rows per step: lane = (row, column quad), so a row's 32
    // scores / P_hat entries / score gradients are one 16-byte access per lane (the rows are contiguous: 512 bytes per warp
    // access), and each lane keeps fp64 column sums for its four columns.  Two steps are loaded before anything is stored (the
    // pointers may alias).  ~13 instead of ~70 instructions per pixel row (the one-column-per-lane loop below paid address
    // arithmetic, conversions and a divergent lane-0 branch for the affine columns per row: 85 us at B = 256 for 70 MB).
    const int rg = lane >> 3, cq = lane & 7;
    double t3x[4], t3y[4], sx[4], sy[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      t3x[i] = Tsm[2 * (3 + 4 * cq + i)]; t3y[i] = Tsm[2 * (3 + 4 * cq + i) + 1];
      sx[i] = 0.0; sy[i] = 0.0;
    }
    const double thd = (double)th;
    for (int pix0 = p_lo + 4 * row; pix0 < p_hi; pix0 += 8 * GB_ROWS) {
      float4 s4[2], h4[2];
      float2 gg[2], pp[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int pix = pix0 + j * 4 * GB_ROWS + rg;
        const bool ok = pix < p_hi;
        const size_t r = (size_t)b * p.n + (ok ? pix : p_lo);
        s4[j] = ok ? __ldg(reinterpret_cast<const float4*>(p.score + r * 32) + cq) : make_float4(0.f, 0.f, 0.f, 0.f);
        h4[j] = ok ? __ldg(reinterpret_cast<const float4*>(p.P_hat + (size_t)pix * 32) + cq) : make_float4(0.f, 0.f, 0.f, 0.f);
        gg[j] = ok ? __ldg(reinterpret_cast<const float2*>(p.g_grid + r * 2)) : make_float2(0.f, 0.f);
        pp[j] = (ok && cq == 0) ? __ldg(reinterpret_cast<const float2*>(p.P + 2 * pix)) : make_float2(0.f, 0.f);
      }
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int pix = pix0 + j * 4 * GB_ROWS + rg;
        const bool ok = pix < p_hi;
        const double dgx = (double)gg[j].x, dgy = (double)gg[j].y;       // zero for rows past the end: they add nothing
        const float sv[4] = {s4[j].x, s4[j].y, s4[j].z, s4[j].w}, hv[4] = {h4[j].x, h4[j].y, h4[j].z, h4[j].w};
        float o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const double h = (double)hv[i];
          const double phi = h * (1.0 + thd * (double)sv[i]);
          sx[i] = fma(phi, dgx, sx[i]);
          sy[i] = fma(phi, dgy, sy[i]);
          o[i] = (float)(thd * h * (dgx * t3x[i] + dgy * t3y[i]));
        }
        if (ok && p.g_score != nullptr)
          __stcs(reinterpret_cast<float4*>(p.g_score + ((size_t)b * p.n + pix) * 32) + cq, make_float4(o[0], o[1], o[2], o[3]));
        // affine columns: the quad-0 lane of each row (predicated: pp and dg are zero elsewhere / past the end)
        const double px = (double)pp[j].x, py = (double)pp[j].y, m = cq == 0 ? 1.0 : 0.0;
        a0x = fma(m, dgx, a0x); a0y = fma(m, dgy, a0y);
        a1x = fma(px, dgx, a1x); a1y = fma(px, dgy, a1y);
        a2x = fma(py, dgx, a2x); a2y = fma(py, dgy, a2y);
      }
    }
    // fold the four row groups (lanes l, l ^ 8, l ^ 16, l ^ 24): fixed butterfly = deterministic
#pragma unroll
    for (int off = 8; off <= 16; off <<= 1) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        sx[i] += __shfl_xor_sync(0xffffffffu, sx[i], off);
        sy[i] += __shfl_xor_sync(0xffffffffu, sy[i], off);
      }
      a0x += __shfl_xor_sync(0xffffffffu, a0x, off); a0y += __shfl_xor_sync(0xffffffffu, a0y, off);
      a1x += __shfl_xor_sync(0xffffffffu, a1x, off); a1y += __shfl_xor_sync(0xffffffffu, a1y, off);
      a2x += __shfl_xor_sync(0xffffffffu, a2x, off); a2y += __shfl_xor_sync(0xffffffffu, a2y, off);
    }
    double* mine = red + (size_t)row * 2 * p.K;
    if (rg == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) { mine[2 * (3 + 4 * cq + i)] = sx[i]; mine[2 * (3 + 4 * cq + i) + 1] = sy[i]; }
      if (cq == 0) { mine[0] = a0x; mine[1] = a0y; mine[2] = a1x; mine[3] = a1y; mine[4] = a2x; mine[5] = a2y; }
    }
    __syncthreads();
    double* outp = partial + ((size_t)b * nsplit + split) * 2 * p.K;
    for (int o = threadIdx.x; o < 2 * p.K; o += blockDim.x) {
      double acc = 0.0;
#pragma unroll
      for (int r = 0; r < GB_ROWS; ++r) acc += red[(size_t)r * 2 * p.K + o];
      outp[o] = acc;
    }
    return;
  } else
  // independent pixel rows: unrolled so that the loads of four rows are in flight together (the loop is latency-bound)
#pragma unroll 4
  for (int pix = p_lo + row; pix < p_hi; pix += GB_ROWS) {
    const float2 gg = __ldg(reinterpret_cast<const float2*>(p.g_grid + ((size_t)b * p.n + pix) * 2));
    const double dgx = (double)gg.x, dgy = (double)gg.y;
    const float* ph = p.P_hat + (size_t)pix * ncol;
    if (MODE == 0) {
      const float* s = p.score + ((size_t)b * p.n + pix) * p.F;
      float* gs = p.g_score ? p.g_score + ((size_t)b * p.n + pix) * p.F : nullptr;
#pragma unroll
      for (int i = 0; i < GB_MAXI; ++i) {
        const int k = lane + 32 * i;
        if (k < p.F) {
          const double h = (double)__ldg(ph + k);
          const double phi = h * (1.0 + (double)th * (double)__ldg(s + k));
          ax[i] = fma(phi, dgx, ax[i]);
          ay[i] = fma(phi, dgy, ay[i]);
          if (gs) {
            const double dphi = dgx * Tsm[2 * (3 + k)] + dgy * Tsm[2 * (3 + k) + 1];
            __stcs(gs + k, (float)((double)th * h * dphi));
          }
        }
      }
      if (lane == 0) {
        const double px = (double)__ldg(p.P + 2 * pix), py = (double)__ldg(p.P + 2 * pix + 1);
        a0x += dgx; a0y += dgy;
        a1x = fma(px, dgx, a1x); a1y = fma(px, dgy, a1y);
        a2x = fma(py, dgx, a2x); a2y = fma(py, dgy, a2y);
      }
    } else {
#pragma unroll
      for (int i = 0; i < GB_MAXI; ++i) {
        const int k = lane + 32 * i;
        if (k < p.K) {
          const double phi = (double)__ldg(ph + k);
          ax[i] = fma(phi, dgx, ax[i]);
          ay[i] = fma(phi, dgy, ay[i]);
        }
      }
    }
  }
  // per-row partial sums -> shared, then fixed-order sum over rows
  double* mine = red + (size_t)row * 2 * p.K;
  const int base = (MODE == 0) ? 3 : 0;
#pragma unroll
  for (int i = 0; i < GB_MAXI; ++i) {
    const int k = lane + 32 * i;
    if (k < ncol) { mine[2 * (base + k)] = ax[i]; mine[2 * (base + k) + 1] = ay[i]; }
  }
  if (MODE == 0 && lane == 0) {
    mine[0] = a0x; mine[1] = a0y; mine[2] = a1x; mine[3] = a1y; mine[4] = a2x; mine[5] = a2y;
  }
  __syncthreads();
  double* out = partial + ((size_t)b * nsplit + split) * 2 * p.K;
  for (int o = threadIdx.x; o < 2 * p.K; o += blockDim.x) {
    double acc = 0.0;
#pragma unroll
    for (int r = 0; r < GB_ROWS; ++r) acc += red[(size_t)r * 2 * p.K + o];
    out[o] = acc;
  }
}

__global__ void __launch_bounds__(256) cprime_bwd_kernel(WarpParams p, int nsplit, const double* partial) {
  extern __shared__ double dT[];   // [K][2]
  const int b = blockIdx.x;
  for (int o = threadIdx.x; o < 2 * p.K; o += blockDim.x) {
    double acc = 0.0;
    for (int s = 0; s < nsplit; ++s) acc += partial[((size_t)b * nsplit + s) * 2 * p.K + o];
    dT[o] = acc;
  }
  __syncthreads();
  for (int o = threadIdx.x; o < 2 * p.F; o += blockDim.x) {
    const int f = o >> 1, c = o & 1;
    double acc = 0.0;
    for (int k = 0; k < p.K; ++k) acc = fma((double)__ldg(p.hatC + (size_t)k * p.K + f), dT[2 * k + c], acc);
    p.g_c_prime[(size_t)b * p.F * 2 + o] = (float)acc;
  }
}

// ------------------------------------------------------------------------------------------
// Staged backward for the TPS++ geometry (attention mode, F = 32, n <= 1024, fp32, source planes <= 4096 pixels): three
// kernels, no global atomics on d src, no memset of it.
//
//   K-B1c warp_bwd_csr_kernel   one CTA per image: T, the sampling grid (fp64), the taps -- and the scatter
//                               "output pixel -> its four taps", which is the same for all channels of an image, INVERTED
//                               into a CSR table per source (counting sort by source pixel: for every source pixel the
//                               list of (output pixel, bilinear weight) that touch it, ordered by pixel), written to the
//                               workspace (68 KB per image).
//   K-B1g warp_bwd_grid_kernel  the forward kernel's structure (persistent CTAs over contiguous ranges of (image, channel)
//                               planes; [src0 | src1 | gout0 | gout1] of a plane arrive by bulk copies through a 4-stage
//                               ring; taps / fractions / clip masks of a thread's two pixels in registers): d grid
//                               accumulates in registers over the channel loop, one slot per image segment, which
//                               grid_seg_sum_kernel adds up in a fixed order into g_grid.
//   K-B1s warp_bwd_src_kernel   d src as a GATHER: persistent CTAs over (image, 8-channel block) units; the image's CSR
//                               table and the block's gout planes are bulk-copied to shared memory; a thread owns four (two)
//                               consecutive source pixels and sums  gsrc[s, ch] = sum_e w_e * gout[ch][pix_e]  for the 8
//                               channels at once (the entry fetch and the loop are amortised over 8 FMAs), then writes
//                               coalesced 16-byte (8-byte) rows.  Deterministic: fixed summation order.
// Why not shared-memory float atomics into a staged d-src plane: sm_100 has no native one (ATOMS.CAST.SPIN loops), measured
// 508 us for the scatter alone at B = 256 against 650 us for the global-atomics kernel; a one-plane-at-a-time gather with a
// thread per source pixel is issue-bound (two dependent shared loads per FMA, divergent trip counts): 730 us.
// ------------------------------------------------------------------------------------------
constexpr int BS_WARPS = 16;
constexpr int BS_CONSUMERS = BS_WARPS * 32;     // 512
constexpr int BS_THREADS = BS_CONSUMERS + 32;   // + producer warp
constexpr int BS_PPT = 2;
constexpr int BS_MAX_N = BS_CONSUMERS * BS_PPT; // 1024
constexpr int BS_F = 32, BS_K = BS_F + 3;
constexpr int BS_IN_STAGES = 4;
constexpr int BS_MAX_S0 = 4096, BS_MAX_S1 = 1024;   // source pixels per plane the CSR tables are sized for
constexpr int BS_CB = 8;                            // channels per unit of the gather kernel
constexpr int BS_SORT_MAX = 64;                     // lists longer than this stay in arrival order (pathological warps)
// CSR blob of one image (same layout in the workspace and in shared memory):
//   end0 u32[S0max] | end1 u32[S1max] | w0 f32[4n] | w1 f32[4n] | pix0 u16[4n] | pix1 u16[4n]
constexpr size_t BS_CSR_BYTES = (size_t)(BS_MAX_S0 + BS_MAX_S1) * 4 + (size_t)2 * 4 * BS_MAX_N * 6;   // 69632

struct BwdCsr {                             // one source: end[s] = one past the last entry of source pixel s
  uint32_t* end;
  uint16_t* pix;
  float* w;
};
__device__ __forceinline__ void csr_views(unsigned char* blob, BwdCsr& c0, BwdCsr& c1) {
  c0.end = reinterpret_cast<uint32_t*>(blob);
  c1.end = c0.end + BS_MAX_S0;
  c0.w = reinterpret_cast<float*>(c1.end + BS_MAX_S1);
  c1.w = c0.w + 4 * BS_MAX_N;
  c0.pix = reinterpret_cast<uint16_t*>(c1.w + 4 * BS_MAX_N);
  c1.pix = c0.pix + 4 * BS_MAX_N;
}

struct BwdStagedArgs {
  WarpParams p;
  int planes_total;
  int dual;
  uint32_t s0_bytes, s1_bytes, g_bytes;     // one src0 / src1 / gout plane
  uint32_t in_stage;                        // 128-byte aligned stage size of the d-grid kernel
  unsigned char* csr;                       // [B] blobs of BS_CSR_BYTES
  float2* seg;                              // [B][seg_max][n] d grid of each image segment (see bwd_cta_of)
  int seg_max;
};

// The d-grid kernel's persistent CTA k of `ctas` owns planes [k P / ctas, (k + 1) P / ctas) of the P = B * C (image, channel)
// planes, so an image is split over consecutive CTAs; the CTA that holds plane x:
__host__ __device__ __forceinline__ int bwd_cta_of(long long x, int ctas, long long planes) {
  return (int)(((x + 1) * ctas - 1) / planes);
}
static int bwd_grid_ctas(long long planes) { return (int)(planes < sm_count() ? planes : sm_count()); }
// most CTAs one image is split over: a partial first segment, whole CTA ranges of at least floor(P / ctas) planes, a partial last one
static int bwd_seg_max(int C, long long planes, int ctas) {
  const long long whole = C > 2 ? (C - 2) / (planes / ctas) : 0;
  return (int)(whole + 2 < C ? whole + 2 : C);
}

// fp64 sampling grid of image b into gridsm (8 lanes per pixel, coalesced float4 rows of pc_score / P_hat); NW warps
template <int NW>
__device__ __forceinline__ void staged_grid_phase(const WarpParams& p, const double* T, int b, double2* gridsm, int warp, int lane) {
  const int kq = (lane & 7) * 4;
  double tx[4], ty[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { tx[i] = T[2 * (3 + kq + i)]; ty[i] = T[2 * (3 + kq + i) + 1]; }
  const double th = (double)p.theta;
  const float* sbase = p.score + (size_t)b * p.n * BS_F;
  const int pix0 = warp * (BS_MAX_N / NW) + (lane >> 3);
#pragma unroll 4
  for (int step = 0; step < BS_MAX_N / NW / 4; ++step) {
    const int pix = pix0 + step * 4;
    const bool ok = pix < p.n;
    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), h4 = s4;
    if (ok) {
      s4 = __ldg(reinterpret_cast<const float4*>(sbase + (size_t)pix * BS_F + kq));
      h4 = __ldg(reinterpret_cast<const float4*>(p.P_hat + (size_t)pix * BS_F + kq));
    }
    const double f0 = (double)h4.x * (1.0 + th * (double)s4.x);
    const double f1 = (double)h4.y * (1.0 + th * (double)s4.y);
    const double f2 = (double)h4.z * (1.0 + th * (double)s4.z);
    const double f3 = (double)h4.w * (1.0 + th * (double)s4.w);
    double ax = fma(f3, tx[3], fma(f2, tx[2], fma(f1, tx[1], f0 * tx[0])));
    double ay = fma(f3, ty[3], fma(f2, ty[2], fma(f1, ty[1], f0 * ty[0])));
#pragma unroll
    for (int m = 1; m < 8; m <<= 1) { ax += shfl_xor_f64(ax, m); ay += shfl_xor_f64(ay, m); }
    if (ok && (lane & 7) == 0) {
      const double px = (double)__ldg(p.P + 2 * pix), py = (double)__ldg(p.P + 2 * pix + 1);
      gridsm[pix] = make_double2(T[0] + px * T[2] + py * T[4] + ax, T[1] + px * T[3] + py * T[5] + ay);
    }
  }
}

// ---- K-B1c ----
__global__ void __launch_bounds__(BS_CONSUMERS, 2) warp_bwd_csr_kernel(BwdStagedArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const WarpParams& p = a.p;
  BwdCsr csr0, csr1;
  csr_views(smem, csr0, csr1);
  double2* gridsm = reinterpret_cast<double2*>(smem + BS_CSR_BYTES);
  double* T = reinterpret_cast<double*>(gridsm + BS_MAX_N);
  uint32_t* wsum = reinterpret_cast<uint32_t*>(T + 2 * BS_K);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x, n = p.n;
  const int S0 = p.H0 * p.W0, S1 = a.dual ? p.H1 * p.W1 : 0;
  const bool sc0 = p.gsrc0 != nullptr, sc1 = a.dual && p.gsrc1 != nullptr;
  compute_T(p, b, T, tid, BS_CONSUMERS);
  for (int i = tid; i < BS_MAX_S0 + BS_MAX_S1; i += BS_CONSUMERS) csr0.end[i] = 0u;
  __syncthreads();
  staged_grid_phase<BS_WARPS>(p, T, b, gridsm, warp, lane);
  __syncthreads();
  // pass 1: taps of this thread's pixels; count the entries of every source pixel
  Taps t0[BS_PPT], t1[BS_PPT];
#pragma unroll
  for (int j = 0; j < BS_PPT; ++j) {
    const int pix = tid + BS_CONSUMERS * j;
    double2 g = make_double2(0.0, 0.0);
    if (pix < n) g = gridsm[pix];
    t0[j] = make_taps<double>(g.x, g.y, p.W0, p.H0);
    if (pix < n && sc0) {
      atomicAdd(&csr0.end[t0[j].off], 1u);
      if (t0[j].dx) atomicAdd(&csr0.end[t0[j].off + t0[j].dx], 1u);
      if (t0[j].dy) atomicAdd(&csr0.end[t0[j].off + t0[j].dy], 1u);
      if (t0[j].dx && t0[j].dy) atomicAdd(&csr0.end[t0[j].off + t0[j].dy + t0[j].dx], 1u);
    }
    if (a.dual) {
      t1[j] = make_taps<double>(g.x, g.y, p.W1, p.H1);
      if (pix < n && sc1) {
        atomicAdd(&csr1.end[t1[j].off], 1u);
        if (t1[j].dx) atomicAdd(&csr1.end[t1[j].off + t1[j].dx], 1u);
        if (t1[j].dy) atomicAdd(&csr1.end[t1[j].off + t1[j].dy], 1u);
        if (t1[j].dx && t1[j].dy) atomicAdd(&csr1.end[t1[j].off + t1[j].dy + t1[j].dx], 1u);
      }
    }
  }
  __syncthreads();
  // pass 2: exclusive prefix sums (counts -> start positions, kept in `end` as running cursors)
  {
    const int per0 = (S0 + BS_CONSUMERS - 1) / BS_CONSUMERS, per1 = (S1 + BS_CONSUMERS - 1) / BS_CONSUMERS;
    uint32_t sum0 = 0, sum1 = 0;
    for (int i = 0; i < per0; ++i) { const int s = tid * per0 + i; if (s < S0) sum0 += csr0.end[s]; }
    for (int i = 0; i < per1; ++i) { const int s = tid * per1 + i; if (s < S1) sum1 += csr1.end[s]; }
    uint32_t inc0 = sum0, inc1 = sum1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t u0 = __shfl_up_sync(0xffffffffu, inc0, d), u1 = __shfl_up_sync(0xffffffffu, inc1, d);
      if (lane >= d) { inc0 += u0; inc1 += u1; }
    }
    if (lane == 31) { wsum[warp] = inc0; wsum[BS_WARPS + warp] = inc1; }
    __syncthreads();
    uint32_t base0 = inc0 - sum0, base1 = inc1 - sum1;
    for (int w = 0; w < warp; ++w) { base0 += wsum[w]; base1 += wsum[BS_WARPS + w]; }
    for (int i = 0; i < per0; ++i) {
      const int s = tid * per0 + i;
      if (s < S0) { const uint32_t c = csr0.end[s]; csr0.end[s] = base0; base0 += c; }
    }
    for (int i = 0; i < per1; ++i) {
      const int s = tid * per1 + i;
      if (s < S1) { const uint32_t c = csr1.end[s]; csr1.end[s] = base1; base1 += c; }
    }
  }
  __syncthreads();
  // pass 3: fill (the cursor of a source pixel ends one past its last entry)
#pragma unroll
  for (int j = 0; j < BS_PPT; ++j) {
    const int pix = tid + BS_CONSUMERS * j;
    if (pix < n && sc0) {
      const int offs[4] = {t0[j].off, t0[j].off + t0[j].dx, t0[j].off + t0[j].dy, t0[j].off + t0[j].dy + t0[j].dx};
      const bool ok[4] = {true, t0[j].dx != 0, t0[j].dy != 0, t0[j].dx != 0 && t0[j].dy != 0};
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (ok[k]) {
          const uint32_t pos = atomicAdd(&csr0.end[offs[k]], 1u);
          csr0.pix[pos] = (uint16_t)pix; csr0.w[pos] = t0[j].w[k];
        }
    }
    if (a.dual && pix < n && sc1) {
      const int offs[4] = {t1[j].off, t1[j].off + t1[j].dx, t1[j].off + t1[j].dy, t1[j].off + t1[j].dy + t1[j].dx};
      const bool ok[4] = {true, t1[j].dx != 0, t1[j].dy != 0, t1[j].dx != 0 && t1[j].dy != 0};
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (ok[k]) {
          const uint32_t pos = atomicAdd(&csr1.end[offs[k]], 1u);
          csr1.pix[pos] = (uint16_t)pix; csr1.w[pos] = t1[j].w[k];
        }
    }
  }
  __syncthreads();
  // pass 4: order every list by output pixel so that the gather sums in a fixed order whatever the atomics' arrival order
  // was.  Lists of up to 8 entries: insertion sort by the thread that owns the source pixel; 9 .. 64 entries (border
  // pixels that collect the clamped samples): queued and rank-sorted by a whole warp (one thread sorting a 30-entry list
  // kept the other 511 waiting at the barrier: half of this kernel's time); longer ones stay in arrival order.
  uint32_t* queue = reinterpret_cast<uint32_t*>(gridsm);     // the grid is no longer needed: [0] = count, then items
  if (tid == 0) queue[0] = 0u;
  __syncthreads();
  for (int src = 0; src < (a.dual ? 2 : 1); ++src) {
    const BwdCsr& t = src == 0 ? csr0 : csr1;
    const int S = src == 0 ? S0 : S1;
    for (int s = tid; s < S; s += BS_CONSUMERS) {
      const uint32_t beg = s == 0 ? 0u : t.end[s - 1], en = t.end[s];
      const uint32_t L = en - beg;
      if (L > (uint32_t)BS_SORT_MAX || L < 2) continue;
      if (L > 8) {
        const uint32_t slot = atomicAdd(&queue[0], 1u);
        if (slot < 2047u) queue[1 + slot] = beg | (L << 16) | ((uint32_t)src << 31);
        continue;
      }
      for (uint32_t i = beg + 1; i < en; ++i) {
        const uint16_t kp = t.pix[i];
        const float kw = t.w[i];
        uint32_t j = i;
        while (j > beg && t.pix[j - 1] > kp) { t.pix[j] = t.pix[j - 1]; t.w[j] = t.w[j - 1]; --j; }
        t.pix[j] = kp; t.w[j] = kw;
      }
    }
  }
  __syncthreads();
  {
    const uint32_t nq = min(queue[0], 2047u);
    for (uint32_t qi = warp; qi < nq; qi += BS_WARPS) {
      const uint32_t item = queue[1 + qi];
      const BwdCsr& t = (item >> 31) ? csr1 : csr0;
      const uint32_t beg = item & 0xffffu, L = (item >> 16) & 0x7fffu;
      // two entries per lane (L <= 64); keys are distinct within a list (a pixel's four taps hit four different source
      // pixels), so rank = number of smaller keys
      uint32_t k0 = 0xffffffffu, k1 = 0xffffffffu;
      float v0 = 0.f, v1 = 0.f;
      if ((uint32_t)lane < L) { k0 = t.pix[beg + lane]; v0 = t.w[beg + lane]; }
      if ((uint32_t)lane + 32 < L) { k1 = t.pix[beg + lane + 32]; v1 = t.w[beg + lane + 32]; }
      uint32_t r0 = 0, r1 = 0;
      for (uint32_t i = 0; i < L; ++i) {
        const uint32_t ki = t.pix[beg + i];
        r0 += ki < k0; r1 += ki < k1;
      }
      __syncwarp();
      if ((uint32_t)lane < L) { t.pix[beg + r0] = (uint16_t)k0; t.w[beg + r0] = v0; }
      if ((uint32_t)lane + 32 < L) { t.pix[beg + r1] = (uint16_t)k1; t.w[beg + r1] = v1; }
    }
  }
  __syncthreads();
  uint4* dst = reinterpret_cast<uint4*>(a.csr + (size_t)b * BS_CSR_BYTES);
  const uint4* srcv = reinterpret_cast<const uint4*>(smem);
  for (int i = tid; i < (int)(BS_CSR_BYTES / 16); i += BS_CONSUMERS) dst[i] = srcv[i];
}

// ---- K-B1g ----
struct BwdStagedTail {
  double T[2 * BS_K];
  uint64_t full[BS_IN_STAGES];
  uint64_t empty[BS_IN_STAGES];
};
struct TapG {            // what the channel loop needs of one (pixel, source)
  int off, dx, dy;
  float tx, ty, ux, uy, mx, my;
};
__device__ __forceinline__ TapG make_tapg(double gx, double gy, int W, int H) {
  const TapsGrad g = make_taps_grad<double>(gx, gy, W, H);
  TapG t;
  t.off = g.t.off; t.dx = g.t.dx; t.dy = g.t.dy;
  t.tx = g.tx; t.ty = g.ty; t.ux = g.ux; t.uy = g.uy; t.mx = g.mx; t.my = g.my;
  return t;
}
// d grid contribution of one (pixel, source, channel)
__device__ __forceinline__ void bwd_tap(const float* __restrict__ s, float G, const TapG& t, float& gix, float& giy) {
  const float* q = s + t.off;
  const float vnw = q[0];
  const float vne = t.dx ? q[t.dx] : 0.f;
  const float vsw = t.dy ? q[t.dy] : 0.f;
  const float vse = (t.dx && t.dy) ? q[t.dy + t.dx] : 0.f;
  gix = __fmaf_rn(G, t.uy * (vne - vnw) + t.ty * (vse - vsw), gix);
  giy = __fmaf_rn(G, t.ux * (vsw - vnw) + t.tx * (vse - vne), giy);
}

template <bool DUAL>
__global__ void __launch_bounds__(BS_THREADS, 1) warp_bwd_grid_kernel(BwdStagedArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const WarpParams& p = a.p;
  unsigned char* in_ring = smem;
  double2* gridsm = reinterpret_cast<double2*>(smem + (size_t)BS_IN_STAGES * a.in_stage);
  BwdStagedTail* tail = reinterpret_cast<BwdStagedTail*>(gridsm + BS_MAX_N);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = p.C0;
  const int p_begin = (int)(((long long)blockIdx.x * a.planes_total) / gridDim.x);
  const int p_end = (int)(((long long)(blockIdx.x + 1) * a.planes_total) / gridDim.x);
  if (tid == 0) {
    for (int s = 0; s < BS_IN_STAGES; ++s) { mbar_init(&tail->full[s], 1); mbar_init(&tail->empty[s], BS_WARPS); }
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == BS_WARPS) {
    // ===== producer: one lane streams [src0 | src1 | gout0 | gout1] of each plane through the ring =====
    if (lane == 0) {
      const uint64_t pol = policy_evict_first();
      const unsigned char* g0 = (const unsigned char*)p.src0;
      const unsigned char* g1 = (const unsigned char*)p.src1;
      const unsigned char* go0 = (const unsigned char*)p.gout0;
      const unsigned char* go1 = (const unsigned char*)p.gout1;
      int it = 0;
      for (int plane = p_begin; plane < p_end; ++plane, ++it) {
        const int s = it % BS_IN_STAGES;
        const uint32_t ph = (uint32_t)((it / BS_IN_STAGES) & 1);
        mbar_wait(&tail->empty[s], ph ^ 1u);
        unsigned char* dst = in_ring + (size_t)s * a.in_stage;
        mbar_arrive_expect_tx(&tail->full[s], a.s0_bytes + a.g_bytes + (DUAL ? a.s1_bytes + a.g_bytes : 0u));
        bulk_g2s(dst, g0 + (size_t)plane * a.s0_bytes, a.s0_bytes, &tail->full[s], pol);
        bulk_g2s(dst + a.s0_bytes + a.s1_bytes, go0 + (size_t)plane * a.g_bytes, a.g_bytes, &tail->full[s], pol);
        if (DUAL) {
          bulk_g2s(dst + a.s0_bytes, g1 + (size_t)plane * a.s1_bytes, a.s1_bytes, &tail->full[s], pol);
          bulk_g2s(dst + a.s0_bytes + a.s1_bytes + a.g_bytes, go1 + (size_t)plane * a.g_bytes, a.g_bytes, &tail->full[s], pol);
        }
      }
    }
    return;
  }

  // ===== consumers =====
  const int n = p.n;
  int it = 0;
  int plane = p_begin;
  while (plane < p_end) {
    const int b = plane / C;
    const int c_begin = plane - b * C;
    const int c_end = min(C, c_begin + (p_end - plane));

    named_bar_sync(1, BS_CONSUMERS);                 // everyone is done with the previous image's T / grid
    compute_T(p, b, tail->T, tid, BS_CONSUMERS);
    named_bar_sync(1, BS_CONSUMERS);
    staged_grid_phase<BS_WARPS>(p, tail->T, b, gridsm, warp, lane);
    named_bar_sync(1, BS_CONSUMERS);

    TapG t0[BS_PPT], t1[BS_PPT];
    float gix0[BS_PPT], giy0[BS_PPT], gix1[BS_PPT], giy1[BS_PPT];
#pragma unroll
    for (int j = 0; j < BS_PPT; ++j) {
      const int pix = tid + BS_CONSUMERS * j;
      double2 g = make_double2(0.0, 0.0);
      if (pix < n) g = gridsm[pix];
      t0[j] = make_tapg(g.x, g.y, p.W0, p.H0);
      if (DUAL) t1[j] = make_tapg(g.x, g.y, p.W1, p.H1);
      gix0[j] = giy0[j] = gix1[j] = giy1[j] = 0.f;
    }
    for (int c = c_begin; c < c_end; ++c, ++it) {
      const int s = it % BS_IN_STAGES;
      const uint32_t ph = (uint32_t)((it / BS_IN_STAGES) & 1);
      mbar_wait(&tail->full[s], ph);
      const unsigned char* st = in_ring + (size_t)s * a.in_stage;
      const float* s0 = reinterpret_cast<const float*>(st);
      const float* s1 = reinterpret_cast<const float*>(st + a.s0_bytes);
      const float* G0 = reinterpret_cast<const float*>(st + a.s0_bytes + a.s1_bytes);
      const float* G1 = reinterpret_cast<const float*>(st + a.s0_bytes + a.s1_bytes + a.g_bytes);
#pragma unroll
      for (int j = 0; j < BS_PPT; ++j) {
        const int pix = tid + BS_CONSUMERS * j;
        if (pix < n) {
          bwd_tap(s0, G0[pix], t0[j], gix0[j], giy0[j]);
          if (DUAL) bwd_tap(s1, G1[pix], t1[j], gix1[j], giy1[j]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->empty[s]);
    }
    // d grid of this image segment: chain rule through the un-normalisation (and its clip masks), summed over sources, into
    // the segment's own slot (rank of this CTA among the image's CTAs).  grid_seg_sum_kernel adds the slots in rank order:
    // float atomics into g_grid summed in arrival order, which is not deterministic once three CTAs share an image (B = 128).
    const int rank = (int)blockIdx.x - bwd_cta_of((long long)b * C, gridDim.x, a.planes_total);
    float2* seg = a.seg + ((size_t)b * a.seg_max + rank) * n;
#pragma unroll
    for (int j = 0; j < BS_PPT; ++j) {
      const int pix = tid + BS_CONSUMERS * j;
      if (pix < n) {
        float ggx = gix0[j] * t0[j].mx, ggy = giy0[j] * t0[j].my;
        if (DUAL) { ggx = __fmaf_rn(gix1[j], t1[j].mx, ggx); ggy = __fmaf_rn(giy1[j], t1[j].my, ggy); }
        seg[pix] = make_float2(ggx, ggy);
      }
    }
    plane += (c_end - c_begin);
  }
}

// g_grid[b][pix] = the image's segment slots summed in rank order (fixed order: deterministic)
__global__ void __launch_bounds__(256) grid_seg_sum_kernel(BwdStagedArgs a, int ctas) {
  const WarpParams& p = a.p;
  const long long total = (long long)p.B * p.n;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int b = (int)(i / p.n), pix = (int)(i - (long long)b * p.n);
    const long long first = (long long)b * p.C0;
    const int nseg = bwd_cta_of(first + p.C0 - 1, ctas, a.planes_total) - bwd_cta_of(first, ctas, a.planes_total) + 1;
    const float2* s = a.seg + (size_t)b * a.seg_max * p.n + pix;
    float2 acc = s[0];
    for (int r = 1; r < nseg; ++r) {
      const float2 v = s[(size_t)r * p.n];
      acc.x += v.x; acc.y += v.y;
    }
    reinterpret_cast<float2*>(p.g_grid)[i] = acc;
  }
}

// ---- K-B1s ----
constexpr int BSRC_THREADS = BS_CONSUMERS + 32;
constexpr int BSRC_STAGES = 4;                      // ring items: gout0 set of unit u, gout1 set of unit u, gout0 of u+1, ...
struct BwdSrcTail {
  uint64_t full[BSRC_STAGES];
  uint64_t empty[BSRC_STAGES];
  uint64_t csr_full;
};
// sum_e w_e * G[ch][pix_e] over the list [beg, end) for BS_CB channels (planes n floats apart)
__device__ __forceinline__ void csr_accum(const BwdCsr& t, const float* __restrict__ G, int n, uint32_t beg, uint32_t end, float (&acc)[BS_CB]) {
#pragma unroll
  for (int ch = 0; ch < BS_CB; ++ch) acc[ch] = 0.f;
  for (uint32_t e = beg; e < end; ++e) {
    const float w = t.w[e];
    const float* g = G + t.pix[e];
#pragma unroll
    for (int ch = 0; ch < BS_CB; ++ch) acc[ch] = __fmaf_rn(g[ch * n], w, acc[ch]);
  }
}

__global__ void __launch_bounds__(BSRC_THREADS, 1) warp_bwd_src_kernel(BwdStagedArgs a, int units_total, int blocks_per_img) {
  extern __shared__ __align__(128) unsigned char smem[];
  const WarpParams& p = a.p;
  unsigned char* csr_blob = smem;
  unsigned char* ring = smem + BS_CSR_BYTES;
  const int n = p.n;
  const uint32_t gset = (uint32_t)(BS_CB * n * 4);            // gout planes of one source for a unit = one ring stage
  const int nsrc = a.dual ? 2 : 1;
  BwdSrcTail* tail = reinterpret_cast<BwdSrcTail*>(ring + (size_t)BSRC_STAGES * gset);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int u_begin = (int)(((long long)blockIdx.x * units_total) / gridDim.x);
  const int u_end = (int)(((long long)(blockIdx.x + 1) * units_total) / gridDim.x);
  if (tid == 0) {
    for (int s = 0; s < BSRC_STAGES; ++s) { mbar_init(&tail->full[s], 1); mbar_init(&tail->empty[s], BS_WARPS); }
    mbar_init(&tail->csr_full, 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (warp == BS_WARPS) {
    // ===== producer: the 8 gout planes of (unit, source) per ring item, up to three items ahead of the consumers =====
    if (lane == 0) {
      const uint64_t pol = policy_evict_first();
      int it = 0;
      for (int u = u_begin; u < u_end; ++u) {
        const int b = u / blocks_per_img, cb = (u - b * blocks_per_img) * BS_CB;
        const int nch = min(BS_CB, p.C0 - cb);
        const uint32_t bytes = (uint32_t)(nch * n * 4);
        for (int src = 0; src < nsrc; ++src, ++it) {
          const int s = it % BSRC_STAGES;
          const uint32_t ph = (uint32_t)((it / BSRC_STAGES) & 1);
          mbar_wait(&tail->empty[s], ph ^ 1u);
          mbar_arrive_expect_tx(&tail->full[s], bytes);
          bulk_g2s(ring + (size_t)s * gset, (const unsigned char*)(src == 0 ? p.gout0 : p.gout1) + ((size_t)b * p.C0 + cb) * n * 4, bytes,
                   &tail->full[s], pol);
        }
      }
    }
    return;
  }
  // ===== consumers =====
  BwdCsr csr0, csr1;
  csr_views(csr_blob, csr0, csr1);
  const int S0 = p.H0 * p.W0, S1 = a.dual ? p.H1 * p.W1 : 0;
  const bool sc0 = p.gsrc0 != nullptr, sc1 = a.dual && p.gsrc1 != nullptr;
  int cur_img = -1, csr_loads = 0;
  int it = 0;
  for (int u = u_begin; u < u_end; ++u) {
    const int b = u / blocks_per_img, cb = (u - b * blocks_per_img) * BS_CB;
    const int nch = min(BS_CB, p.C0 - cb);
    if (b != cur_img) {                 // the image's CSR table: one bulk copy, everybody waits for it
      named_bar_sync(1, BS_CONSUMERS);  // nobody still reads the previous table
      if (tid == 0) {
        mbar_arrive_expect_tx(&tail->csr_full, (uint32_t)BS_CSR_BYTES);
        bulk_g2s(csr_blob, a.csr + (size_t)b * BS_CSR_BYTES, (uint32_t)BS_CSR_BYTES, &tail->csr_full, policy_evict_last());
      }
      mbar_wait(&tail->csr_full, (uint32_t)(csr_loads & 1));
      ++csr_loads;
      cur_img = b;
    }
    {
      const int s = it % BSRC_STAGES;
      mbar_wait(&tail->full[s], (uint32_t)((it / BSRC_STAGES) & 1));
      const float* G0 = reinterpret_cast<const float*>(ring + (size_t)s * gset);
      if (sc0) {
        float* dst = (float*)p.gsrc0 + ((size_t)b * p.C0 + cb) * S0;
        for (int q = tid; q < S0 / 4; q += BS_CONSUMERS) {
          const uint4 e4 = *reinterpret_cast<const uint4*>(csr0.end + 4 * q);
          const uint32_t e0 = q == 0 ? 0u : csr0.end[4 * q - 1];
          float r0[BS_CB], r1[BS_CB], r2[BS_CB], r3[BS_CB];
          csr_accum(csr0, G0, n, e0, e4.x, r0);
          csr_accum(csr0, G0, n, e4.x, e4.y, r1);
          csr_accum(csr0, G0, n, e4.y, e4.z, r2);
          csr_accum(csr0, G0, n, e4.z, e4.w, r3);
#pragma unroll
          for (int ch = 0; ch < BS_CB; ++ch)
            if (ch < nch) *reinterpret_cast<float4*>(dst + (size_t)ch * S0 + 4 * q) = make_float4(r0[ch], r1[ch], r2[ch], r3[ch]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->empty[s]);
      ++it;
    }
    if (a.dual) {
      const int s = it % BSRC_STAGES;
      mbar_wait(&tail->full[s], (uint32_t)((it / BSRC_STAGES) & 1));
      const float* G1 = reinterpret_cast<const float*>(ring + (size_t)s * gset);
      if (sc1) {
        float* dst = (float*)p.gsrc1 + ((size_t)b * p.C0 + cb) * S1;
        for (int q = tid; q < S1 / 2; q += BS_CONSUMERS) {
          const uint2 e2 = *reinterpret_cast<const uint2*>(csr1.end + 2 * q);
          const uint32_t e0 = q == 0 ? 0u : csr1.end[2 * q - 1];
          float r0[BS_CB], r1[BS_CB];
          csr_accum(csr1, G1, n, e0, e2.x, r0);
          csr_accum(csr1, G1, n, e2.x, e2.y, r1);
#pragma unroll
          for (int ch = 0; ch < BS_CB; ++ch)
            if (ch < nch) *reinterpret_cast<float2*>(dst + (size_t)ch * S1 + 2 * q) = make_float2(r0[ch], r1[ch]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->empty[s]);
      ++it;
    }
  }
}

static bool bwd_staged_plan(const tpspp_warp_cfg* cfg, const WarpParams& p, BwdStagedArgs* a, size_t* smem_grid, size_t* smem_src) {
  if (cfg->mode != TPSPP_MODE_ATTENTION || cfg->num_fiducial != BS_F || cfg->feat_dtype != TPSPP_F32) return false;
  const int n = cfg->out_h * cfg->out_w;
  if (n > BS_MAX_N || (n & 3)) return false;
  const bool dual = cfg->channels1 > 0 && p.gout1 != nullptr;
  if (dual && cfg->channels1 != cfg->channels0) return false;
  const int S0 = cfg->src0_h * cfg->src0_w, S1 = dual ? cfg->src1_h * cfg->src1_w : 0;
  if (S0 > BS_MAX_S0 || S1 > BS_MAX_S1 || (S0 & 3) || (S1 & 3)) return false;
  const size_t b0 = (size_t)S0 * 4, b1 = (size_t)S1 * 4;
  for (const void* q : {p.src0, p.src1, p.gout0, p.gout1, (const void*)p.gsrc0, (const void*)p.gsrc1, (const void*)p.score,
                        (const void*)p.P_hat})
    if ((uintptr_t)q & 15) return false;
  a->p = p;
  a->dual = dual ? 1 : 0;
  a->planes_total = p.B * p.C0;
  a->s0_bytes = (uint32_t)b0; a->s1_bytes = (uint32_t)b1; a->g_bytes = (uint32_t)n * 4;
  a->in_stage = (uint32_t)((b0 + b1 + (dual ? 2 : 1) * (size_t)n * 4 + 127) / 128 * 128);
  *smem_grid = (size_t)BS_IN_STAGES * a->in_stage + (size_t)BS_MAX_N * sizeof(double2) + sizeof(BwdStagedTail) + 128;
  *smem_src = BS_CSR_BYTES + (size_t)BSRC_STAGES * BS_CB * n * 4 + sizeof(BwdSrcTail) + 128;
  return *smem_grid <= 227 * 1024 && *smem_src <= 227 * 1024;
}
static size_t bwd_csr_smem() { return BS_CSR_BYTES + (size_t)BS_MAX_N * sizeof(double2) + 2 * BS_K * sizeof(double) + 2 * BS_WARPS * 4 + 128; }

int bwd_nsplit(const tpspp_warp_cfg* cfg) {
  const int n = cfg->out_h * cfg->out_w;
  // pixel splits of grid_bwd_reduce_kernel: ~8 CTAs per SM
  int ns = (8 * 148 + cfg->batch - 1) / (cfg->batch > 0 ? cfg->batch : 1);
  const int maxs = (n + 63) / 64;
  if (ns > maxs) ns = maxs;
  if (ns < 1) ns = 1;
  return ns;
}

static size_t align256(size_t v) { return (v + 255) / 256 * 256; }

template <typename FT>
static int launch_bwd_t(const tpspp_warp_cfg* cfg, WarpParams p, void* workspace, cudaStream_t st) {
  const int n = p.n;
  const int nsplit = bwd_nsplit(cfg);
  p.g_grid = reinterpret_cast<float*>(workspace);
  double* partial = reinterpret_cast<double*>((char*)workspace + align256((size_t)p.B * n * 2 * sizeof(float)));

  // TPS++ geometry: staged kernels (CSR gather for d src: no global atomics, no memset of it)
  BwdStagedArgs sa;
  size_t smem_grid = 0, smem_src = 0;
  if (sizeof(FT) == 4 && cfg->variant != TPSPP_VARIANT_GENERIC && bwd_staged_plan(cfg, p, &sa, &smem_grid, &smem_src)) {
    sa.p.g_grid = p.g_grid;
    sa.csr = reinterpret_cast<unsigned char*>(partial) + align256((size_t)p.B * nsplit * 2 * p.K * sizeof(double));
    const int grid = bwd_grid_ctas(sa.planes_total);
    sa.seg = reinterpret_cast<float2*>(sa.csr + align256((size_t)p.B * BS_CSR_BYTES));
    sa.seg_max = bwd_seg_max(p.C0, sa.planes_total, grid);
    const bool dual = sa.dual != 0;
    auto kgrid = dual ? warp_bwd_grid_kernel<true> : warp_bwd_grid_kernel<false>;
    TPSPP_CHECK_CUDA(cudaFuncSetAttribute(kgrid, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_grid));
    TPSPP_CHECK_CUDA(cudaFuncSetAttribute(warp_bwd_src_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_src));
    TPSPP_CHECK_CUDA(cudaFuncSetAttribute(warp_bwd_csr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_csr_smem()));
    if (!dual && p.gsrc1) { TPSPP_CHECK_CUDA(cudaMemsetAsync(p.gsrc1, 0, (size_t)p.B * p.C1 * p.H1 * p.W1 * sizeof(FT), st)); count_launch(); }
    const bool want_src = p.gsrc0 != nullptr || (dual && p.gsrc1 != nullptr);
    if (want_src) {
      warp_bwd_csr_kernel<<<p.B, BS_CONSUMERS, bwd_csr_smem(), st>>>(sa);
      count_launch();
      TPSPP_CHECK_CUDA(cudaGetLastError());
    }
    kgrid<<<grid, BS_THREADS, smem_grid, st>>>(sa);
    count_launch();
    TPSPP_CHECK_CUDA(cudaGetLastError());
    grid_seg_sum_kernel<<<(unsigned)min(((long long)p.B * n + 255) / 256, 4LL * sm_count()), 256, 0, st>>>(sa, grid);
    count_launch();
    TPSPP_CHECK_CUDA(cudaGetLastError());
    if (want_src) {
      const int blocks_per_img = (p.C0 + BS_CB - 1) / BS_CB;
      const int units = p.B * blocks_per_img;
      int g2 = sm_count();
      if (g2 > units) g2 = units;
      warp_bwd_src_kernel<<<g2, BSRC_THREADS, smem_src, st>>>(sa, units, blocks_per_img);
      count_launch();
      TPSPP_CHECK_CUDA(cudaGetLastError());
    }
  } else {
  const size_t es = sizeof(FT);
  if (p.gsrc0) { TPSPP_CHECK_CUDA(cudaMemsetAsync(p.gsrc0, 0, (size_t)p.B * p.C0 * p.H0 * p.W0 * es, st)); count_launch(); }
  if (p.gsrc1) { TPSPP_CHECK_CUDA(cudaMemsetAsync(p.gsrc1, 0, (size_t)p.B * p.C1 * p.H1 * p.W1 * es, st)); count_launch(); }

  const int maxc = p.C0 > p.C1 ? p.C0 : p.C1;
  const int tiles = (n + 255) / 256;
  int zsplit = 1;
  const long long want = 4LL * sm_count();
  while ((long long)tiles * p.B * zsplit < want && zsplit < maxc && zsplit < 16) zsplit *= 2;
  const int cchunk = (maxc + zsplit - 1) / zsplit;
  zsplit = (maxc + cchunk - 1) / cchunk;
  const int use_atomic = zsplit > 1;
  if (use_atomic) { TPSPP_CHECK_CUDA(cudaMemsetAsync(p.g_grid, 0, (size_t)p.B * n * 2 * sizeof(float), st)); count_launch(); }
  dim3 grid(tiles, p.B, zsplit);
  const size_t smemT = (size_t)2 * p.K * sizeof(double);
  if (p.mode == TPSPP_MODE_ATTENTION)
    warp_bwd_sample_kernel<FT, 0><<<grid, 256, smemT, st>>>(p, cchunk, use_atomic);
  else
    warp_bwd_sample_kernel<FT, 1><<<grid, 256, smemT, st>>>(p, cchunk, use_atomic);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  }

  if (p.g_c_prime != nullptr || p.g_score != nullptr) {
    dim3 g2(nsplit, p.B);
    const size_t smem2 = (size_t)(1 + GB_ROWS) * 2 * p.K * sizeof(double);
    if (p.mode == TPSPP_MODE_ATTENTION)
      grid_bwd_reduce_kernel<0><<<g2, 32 * GB_ROWS, smem2, st>>>(p, nsplit, partial);
    else
      grid_bwd_reduce_kernel<1><<<g2, 32 * GB_ROWS, smem2, st>>>(p, nsplit, partial);
    count_launch();
    TPSPP_CHECK_CUDA(cudaGetLastError());
    if (p.g_c_prime != nullptr) {
      cprime_bwd_kernel<<<p.B, 256, (size_t)2 * p.K * sizeof(double), st>>>(p, nsplit, partial);
      count_launch();
      TPSPP_CHECK_CUDA(cudaGetLastError());
    }
  }
  return TPSPP_OK;
}

}  // namespace tpspp

using namespace tpspp;

extern "C" size_t tpspp_warp_workspace_bytes(const tpspp_warp_cfg* cfg) {
  if (validate_cfg(cfg) != TPSPP_OK) return 0;
  const size_t n = (size_t)cfg->out_h * cfg->out_w;
  const size_t K = (size_t)cfg->num_fiducial + 3;
  // the staged kernels' image-segment slots of d grid (only their geometry can use them)
  size_t seg = 0;
  if (cfg->mode == TPSPP_MODE_ATTENTION && cfg->num_fiducial == BS_F && cfg->feat_dtype == TPSPP_F32 && cfg->batch > 0) {
    const long long planes = (long long)cfg->batch * cfg->channels0;
    seg = (size_t)cfg->batch * bwd_seg_max(cfg->channels0, planes, bwd_grid_ctas(planes)) * n * sizeof(float2);
  }
  return align256((size_t)cfg->batch * n * 2 * sizeof(float)) +
         align256((size_t)cfg->batch * bwd_nsplit(cfg) * 2 * K * sizeof(double)) +
         align256((size_t)cfg->batch * BS_CSR_BYTES) /* per-image scatter tables of the staged kernels */ + align256(seg) + 256;
}

extern "C" int tpspp_warp_bwd(const tpspp_warp_cfg* cfg, const void* src0, const void* src1,
                              const float* c_prime, const float* pc_score, const float* P_hat,
                              const float* P, const float* inv_delta_C, const void* gout0,
                              const void* gout1, void* gsrc0, void* gsrc1, float* g_c_prime,
                              float* g_pc_score, void* workspace, tpspp_stream_t stream) {
  reset_launch_count();
  int rc = validate_cfg(cfg);
  if (rc != TPSPP_OK) return rc;
  if (cfg->batch == 0) return TPSPP_OK;
  TPSPP_REQUIRE(src0 && gout0 && c_prime && P_hat && inv_delta_C && workspace,
                "tpspp_warp_bwd: null required pointer");
  TPSPP_REQUIRE(((uintptr_t)workspace & 255) == 0, "tpspp_warp_bwd: workspace must be 256-byte aligned");
  TPSPP_REQUIRE((cfg->channels1 == 0) == (src1 == nullptr), "tpspp_warp_bwd: src1 must be given exactly when channels1 > 0");
  TPSPP_REQUIRE(cfg->channels1 > 0 || (gout1 == nullptr && gsrc1 == nullptr), "tpspp_warp_bwd: gout1/gsrc1 without src1");
  TPSPP_REQUIRE(gsrc1 == nullptr || gout1 != nullptr, "tpspp_warp_bwd: gsrc1 requested without gout1");
  if (cfg->mode == TPSPP_MODE_ATTENTION)
    TPSPP_REQUIRE(pc_score && P, "tpspp_warp_bwd: attention mode needs pc_score and P");
  else
    TPSPP_REQUIRE(g_pc_score == nullptr, "tpspp_warp_bwd: classical mode has no pc_score gradient");
  if (cfg->batch == 0) return TPSPP_OK;
  WarpParams p;
  fill_params(cfg, &p);
  p.src0 = src0; p.src1 = src1; p.c_prime = c_prime; p.score = pc_score; p.P_hat = P_hat; p.P = P;
  p.hatC = inv_delta_C; p.gout0 = gout0; p.gout1 = gout1; p.gsrc0 = gsrc0; p.gsrc1 = gsrc1;
  p.g_c_prime = g_c_prime; p.g_score = g_pc_score;
  TPSPP_REQUIRE(p.B <= 65535, "batch %d exceeds the backward kernels' grid.y limit (65535)", p.B);
  TPSPP_REQUIRE(cfg->feat_dtype != TPSPP_SRC0_BF16, "tpspp_warp_bwd: TPSPP_SRC0_BF16 is a forward-only (inference) layout");
  if (cfg->feat_dtype == TPSPP_BF16) return launch_bwd_t<__nv_bfloat16>(cfg, p, workspace, (cudaStream_t)stream);
  return launch_bwd_t<float>(cfg, p, workspace, (cudaStream_t)stream);
}
