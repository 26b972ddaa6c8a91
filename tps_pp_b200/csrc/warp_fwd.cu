// Fused TPS grid generator + bilinear grid_sample, forward.
//
// Replaces Attention_Enhanced_TPS.build_P_prime / P_hat_score_process and both
// F.grid_sample calls of TPS_PP.forward (reference backbones/tps_pp/tps_pp.py:467-496,
// 601-615) and GridGenerator.build_P_prime + F.grid_sample of TPSPreprocessor.forward
// (preprocessor/tps_preprocessor.py:72-83,270-282).
//
// Two kernels:
//   warp_fwd_generic_kernel  any geometry / mode / dtype: one thread per output pixel,
//                            fp64 grid in registers, direct global gathers.
//   warp_fwd_staged_kernel   the TPS++ geometry (F=32, n<=1024, fp32): persistent CTAs own a
//                            contiguous range of (image, channel) planes; a producer lane
//                            streams whole source planes into a shared-memory ring with
//                            cp.async.bulk (TMA engine) + mbarriers, 8 consumer warps gather
//                            the 4 bilinear taps from shared memory and write coalesced rows.
//                            The sampling grid lives in shared memory / registers only.
#include "common.cuh"

#include <string.h>

namespace tpspp {

// MODE: 0 attention, 1 classical, 2 explicit grid (sampler only, ATen fp32 coordinate math)
template <typename FT, int MODE>
__global__ void __launch_bounds__(256) warp_fwd_generic_kernel(WarpParams p, int cchunk) {
  extern __shared__ double Tsm[];
  const int b = blockIdx.y;
  if (MODE != 2) {
    compute_T(p, b, Tsm, threadIdx.x, blockDim.x);
    __syncthreads();
  }
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= p.n) return;

  Taps t0, t1;
  if (MODE == 2) {
    const float gx = __ldg(p.grid_in + ((size_t)b * p.n + pix) * 2);
    const float gy = __ldg(p.grid_in + ((size_t)b * p.n + pix) * 2 + 1);
    t0 = make_taps<float>(gx, gy, p.W0, p.H0);
    if (p.C1 > 0) t1 = make_taps<float>(gx, gy, p.W1, p.H1);
  } else {
    double gx, gy;
    pixel_grid<MODE>(p, Tsm, b, pix, gx, gy);
    if (p.grid_out != nullptr && blockIdx.z == 0) {
      p.grid_out[((size_t)b * p.n + pix) * 2] = (float)gx;
      p.grid_out[((size_t)b * p.n + pix) * 2 + 1] = (float)gy;
    }
    t0 = make_taps<double>(gx, gy, p.W0, p.H0);
    if (p.C1 > 0) t1 = make_taps<double>(gx, gy, p.W1, p.H1);
  }

  const int cb = blockIdx.z * cchunk;
  {
    const int ce = min(p.C0, cb + cchunk);
    const size_t plane = (size_t)p.H0 * p.W0;
    const FT* src = (const FT*)p.src0 + ((size_t)b * p.C0 + cb) * plane + t0.off;
    FT* out = (FT*)p.out0 + ((size_t)b * p.C0 + cb) * p.n + pix;
#pragma unroll 4
    for (int c = cb; c < ce; ++c, src += plane, out += p.n) {
      const float r = blend4(ldf(src), ldf(src + t0.dx), ldf(src + t0.dy), ldf(src + t0.dy + t0.dx), t0.w);
      stf(out, r);
    }
  }
  if (p.C1 > 0) {
    const int ce = min(p.C1, cb + cchunk);
    const size_t plane = (size_t)p.H1 * p.W1;
    const FT* src = (const FT*)p.src1 + ((size_t)b * p.C1 + cb) * plane + t1.off;
    FT* out = (FT*)p.out1 + ((size_t)b * p.C1 + cb) * p.n + pix;
#pragma unroll 4
    for (int c = cb; c < ce; ++c, src += plane, out += p.n) {
      const float r = blend4(ldf(src), ldf(src + t1.dx), ldf(src + t1.dy), ldf(src + t1.dy + t1.dx), t1.w);
      stf(out, r);
    }
  }
}

// ------------------------------------------------------------------------------------------
// staged persistent kernel
// ------------------------------------------------------------------------------------------
constexpr int ST_CONSUMER_WARPS = 8;
constexpr int ST_CONSUMERS = ST_CONSUMER_WARPS * 32;  // 256
constexpr int ST_THREADS = ST_CONSUMERS + 32;         // + producer warp
constexpr int ST_PPT = 4;                             // output pixels per consumer thread
constexpr int ST_MAX_N = ST_CONSUMERS * ST_PPT;       // 1024
constexpr int ST_F = 32;
constexpr int ST_K = ST_F + 3;
constexpr int ST_MAX_STAGES = 8;

struct StagedArgs {
  WarpParams p;
  int nstages;
  int planes_total;       // B * C
  uint32_t s0_bytes;      // bytes of one src0 plane
  uint32_t s1_bytes;      // bytes of one src1 plane (0 if !DUAL)
  uint32_t stage_bytes;   // 128B-aligned s0+s1
};

struct StagedSmemTail {   // lives after the stage ring and the grid
  double T[2 * ST_K];
  uint64_t full[ST_MAX_STAGES];
  uint64_t empty[ST_MAX_STAGES];
};

// S0BF: the src0 planes are bf16 (TPSPP_SRC0_BF16: feat_grid of the head's bf16 mode) -- half the bytes per stage for the
// larger source; src1 and both outputs stay fp32
template <bool DUAL, bool S0BF = false>
__global__ void __launch_bounds__(ST_THREADS, 2) warp_fwd_staged_kernel(StagedArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const WarpParams& p = a.p;
  unsigned char* ring = smem;
  double2* gridsm = reinterpret_cast<double2*>(smem + (size_t)a.nstages * a.stage_bytes);
  StagedSmemTail* tail = reinterpret_cast<StagedSmemTail*>(gridsm + ST_MAX_N);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int C = p.C0;
  const int p_begin = (int)(((long long)blockIdx.x * a.planes_total) / gridDim.x);
  const int p_end = (int)(((long long)(blockIdx.x + 1) * a.planes_total) / gridDim.x);

  if (tid == 0) {
    for (int s = 0; s < a.nstages; ++s) {
      mbar_init(&tail->full[s], 1);
      mbar_init(&tail->empty[s], ST_CONSUMER_WARPS);
    }
    fence_barrier_init();
  }
  __syncthreads();
  pdl_trigger();          // chained behind the head's last kernel (programmatic dependent launch, common.cuh): barriers are
  pdl_wait();             // set up while that grid drains; no-op in a plain launch

  if (warp == ST_CONSUMER_WARPS) {
    // ===== producer: one lane streams whole planes through the ring =====
    if (lane == 0) {
      const uint64_t pol = policy_evict_first();   // every source byte is read exactly once
      const unsigned char* g0 = (const unsigned char*)p.src0;
      const unsigned char* g1 = (const unsigned char*)p.src1;
      int it = 0;
      for (int plane = p_begin; plane < p_end; ++plane, ++it) {
        const int s = it % a.nstages;
        const uint32_t ph = (uint32_t)((it / a.nstages) & 1);
        mbar_wait(&tail->empty[s], ph ^ 1u);
        unsigned char* dst = ring + (size_t)s * a.stage_bytes;
        mbar_arrive_expect_tx(&tail->full[s], a.s0_bytes + a.s1_bytes);
        bulk_g2s(dst, g0 + (size_t)plane * a.s0_bytes, a.s0_bytes, &tail->full[s], pol);
        if (DUAL) bulk_g2s(dst + a.s0_bytes, g1 + (size_t)plane * a.s1_bytes, a.s1_bytes, &tail->full[s], pol);
      }
    }
    return;
  }

  // ===== consumers =====
  const int n = p.n;
  const int kq = (lane & 7) * 4;     // this lane's 4 rbf columns in the grid phase
  int it = 0;
  int plane = p_begin;
  while (plane < p_end) {
    const int b = plane / C;
    const int c_begin = plane - b * C;
    const int c_end = min(C, c_begin + (p_end - plane));

    named_bar_sync(1, ST_CONSUMERS);  // everyone is done with the previous image's T / grid
    compute_T(p, b, tail->T, tid, ST_CONSUMERS);
    named_bar_sync(1, ST_CONSUMERS);

    // ---- grid phase: 8 lanes per pixel, 4 pixels per warp step, coalesced float4 loads ----
    {
      double tx[4], ty[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        tx[i] = tail->T[2 * (3 + kq + i)];
        ty[i] = tail->T[2 * (3 + kq + i) + 1];
      }
      const double th = (double)p.theta;
      const float* sbase = p.score + (size_t)b * n * ST_F;
      const int pix0 = warp * (ST_MAX_N / ST_CONSUMER_WARPS) + (lane >> 3);
#pragma unroll 4
      for (int step = 0; step < ST_MAX_N / ST_CONSUMER_WARPS / 4; ++step) {
        const int pix = pix0 + step * 4;
        const bool ok = pix < n;
        float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), h4 = s4;
        if (ok) {
          s4 = __ldg(reinterpret_cast<const float4*>(sbase + (size_t)pix * ST_F + kq));
          h4 = __ldg(reinterpret_cast<const float4*>(p.P_hat + (size_t)pix * ST_F + kq));
        }
        const double f0 = (double)h4.x * (1.0 + th * (double)s4.x);
        const double f1 = (double)h4.y * (1.0 + th * (double)s4.y);
        const double f2 = (double)h4.z * (1.0 + th * (double)s4.z);
        const double f3 = (double)h4.w * (1.0 + th * (double)s4.w);
        double ax = fma(f3, tx[3], fma(f2, tx[2], fma(f1, tx[1], f0 * tx[0])));
        double ay = fma(f3, ty[3], fma(f2, ty[2], fma(f1, ty[1], f0 * ty[0])));
#pragma unroll
        for (int m = 1; m < 8; m <<= 1) {
          ax += shfl_xor_f64(ax, m);
          ay += shfl_xor_f64(ay, m);
        }
        if (ok && (lane & 7) == 0) {
          const double px = (double)__ldg(p.P + 2 * pix), py = (double)__ldg(p.P + 2 * pix + 1);
          const double gx = tail->T[0] + px * tail->T[2] + py * tail->T[4] + ax;
          const double gy = tail->T[1] + px * tail->T[3] + py * tail->T[5] + ay;
          gridsm[pix] = make_double2(gx, gy);
        }
      }
    }
    named_bar_sync(1, ST_CONSUMERS);

    // ---- per-thread taps for its 4 pixels (pixel = tid + 256*j: neighbouring lanes sample
    //      neighbouring source columns, which keeps shared-memory bank conflicts low) ----
    Taps t0[ST_PPT], t1[ST_PPT];
#pragma unroll
    for (int j = 0; j < ST_PPT; ++j) {
      const int pix = tid + ST_CONSUMERS * j;
      double2 g = make_double2(0.0, 0.0);
      if (pix < n) g = gridsm[pix];
      t0[j] = make_taps<double>(g.x, g.y, p.W0, p.H0);
      if (DUAL) t1[j] = make_taps<double>(g.x, g.y, p.W1, p.H1);
    }

    // ---- channel loop over the ring ----
    for (int c = c_begin; c < c_end; ++c, ++it) {
      const int s = it % a.nstages;
      const uint32_t ph = (uint32_t)((it / a.nstages) & 1);
      mbar_wait(&tail->full[s], ph);
      const float* s0 = reinterpret_cast<const float*>(ring + (size_t)s * a.stage_bytes);
      const float* s1 = reinterpret_cast<const float*>(ring + (size_t)s * a.stage_bytes + a.s0_bytes);
      float* o0 = (float*)p.out0 + ((size_t)b * C + c) * n;
      float* o1 = (float*)p.out1 + ((size_t)b * C + c) * n;
      float r0[ST_PPT], r1[ST_PPT];
#pragma unroll
      for (int j = 0; j < ST_PPT; ++j) {
        if (S0BF) {
          const __nv_bfloat16* q = reinterpret_cast<const __nv_bfloat16*>(s0) + t0[j].off;
          r0[j] = blend4(__bfloat162float(q[0]), __bfloat162float(q[t0[j].dx]), __bfloat162float(q[t0[j].dy]),
                         __bfloat162float(q[t0[j].dy + t0[j].dx]), t0[j].w);
        } else {
          const float* q = s0 + t0[j].off;
          r0[j] = blend4(q[0], q[t0[j].dx], q[t0[j].dy], q[t0[j].dy + t0[j].dx], t0[j].w);
        }
        if (DUAL) {
          const float* r = s1 + t1[j].off;
          r1[j] = blend4(r[0], r[t1[j].dx], r[t1[j].dy], r[t1[j].dy + t1[j].dx], t1[j].w);
        }
      }
      // The stage is read through the generic proxy and refilled by the producer's bulk copy, which writes through the async
      // proxy: without this fence the refill may land before these reads have been performed (seen as a few wrong src1 taps
      // per B = 256 call once the grid overlaps its neighbours under programmatic dependent launch)
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->empty[s]);   // the stage may be refilled
#pragma unroll
      for (int j = 0; j < ST_PPT; ++j) {
        const int pix = tid + ST_CONSUMERS * j;
        if (pix < n) {
          __stcs(o0 + pix, r0[j]);
          if (DUAL) __stcs(o1 + pix, r1[j]);
        }
      }
    }
    plane += (c_end - c_begin);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static size_t staged_fixed_smem() { return (size_t)ST_MAX_N * sizeof(double2) + sizeof(StagedSmemTail) + 128; }

// returns nstages (0 = not eligible)
static int staged_plan(const tpspp_warp_cfg* cfg, uint32_t* s0, uint32_t* s1, uint32_t* stage) {
  if (cfg->mode != TPSPP_MODE_ATTENTION || cfg->num_fiducial != ST_F) return 0;
  if (cfg->feat_dtype != TPSPP_F32 && cfg->feat_dtype != TPSPP_SRC0_BF16) return 0;
  const int n = cfg->out_h * cfg->out_w;
  if (n > ST_MAX_N) return 0;
  if (cfg->channels1 != 0 && cfg->channels1 != cfg->channels0) return 0;
  const size_t b0 = (size_t)cfg->src0_h * cfg->src0_w * (cfg->feat_dtype == TPSPP_SRC0_BF16 ? 2 : 4);
  const size_t b1 = cfg->channels1 ? (size_t)cfg->src1_h * cfg->src1_w * 4 : 0;
  if (b0 % 16 || b1 % 16) return 0;
  const size_t st = (b0 + b1 + 127) / 128 * 128;
  const size_t per_cta_two = (232448 / 2) - 1024;   // two CTAs per SM
  const size_t per_cta_one = 232448 - 1024;
  size_t avail = per_cta_two > staged_fixed_smem() ? per_cta_two - staged_fixed_smem() : 0;
  int ns = (int)(avail / st);
  if (ns < 3) {
    avail = per_cta_one > staged_fixed_smem() ? per_cta_one - staged_fixed_smem() : 0;
    ns = (int)(avail / st);
  }
  if (ns > ST_MAX_STAGES) ns = ST_MAX_STAGES;
  if (ns < 2) return 0;
  *s0 = (uint32_t)b0; *s1 = (uint32_t)b1; *stage = (uint32_t)st;
  return ns;
}

static int launch_staged(const tpspp_warp_cfg* cfg, const WarpParams& p, cudaStream_t stream) {
  StagedArgs a;
  a.p = p;
  a.nstages = staged_plan(cfg, &a.s0_bytes, &a.s1_bytes, &a.stage_bytes);
  if (a.nstages == 0) {
    set_error("staged warp variant does not support this configuration "
              "(needs attention mode, F=32, n<=1024, fp32, C1 in {0,C0}, planes that fit shared memory)");
    return TPSPP_E_UNSUPPORTED;
  }
  if (p.grid_out != nullptr) {
    set_error("staged warp variant keeps the grid on chip; grid_out must be NULL");
    return TPSPP_E_UNSUPPORTED;
  }
  if (((uintptr_t)p.src0 & 15) || ((uintptr_t)p.src1 & 15) || ((uintptr_t)p.score & 15) ||
      ((uintptr_t)p.P_hat & 15)) {
    set_error("staged warp variant needs 16-byte aligned src/pc_score/P_hat pointers");
    return TPSPP_E_UNSUPPORTED;
  }
  a.planes_total = p.B * p.C0;
  const size_t smem = (size_t)a.nstages * a.stage_bytes + staged_fixed_smem();
  const bool dual = p.C1 > 0;
  const bool s0bf = cfg->feat_dtype == TPSPP_SRC0_BF16;
  auto kern = s0bf ? (dual ? warp_fwd_staged_kernel<true, true> : warp_fwd_staged_kernel<false, true>)
                   : (dual ? warp_fwd_staged_kernel<true> : warp_fwd_staged_kernel<false>);
  TPSPP_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int ctas_per_sm = 0;
  TPSPP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kern, ST_THREADS, smem));
  if (ctas_per_sm < 1) {
    set_error("staged warp kernel does not fit on an SM (smem %zu)", smem);
    return TPSPP_E_UNSUPPORTED;
  }
  int grid = sm_count() * ctas_per_sm;
  if (grid > a.planes_total) grid = a.planes_total;
  pdl_scope(true);
  launch_k(kern, dim3(grid), dim3(ST_THREADS), smem, stream, a);
  pdl_scope(false);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  return TPSPP_OK;
}

template <typename FT>
static int launch_generic_t(const WarpParams& p, int mode, cudaStream_t stream) {
  const int maxc = p.C0 > p.C1 ? p.C0 : p.C1;
  // enough CTAs to fill the machine a few times over, without shredding the channel loop
  const int tiles = (p.n + 255) / 256;
  int zsplit = 1;
  const long long want = 4LL * sm_count();
  while ((long long)tiles * p.B * zsplit < want && zsplit < maxc && zsplit < 16) zsplit *= 2;
  const int cchunk = (maxc + zsplit - 1) / zsplit;
  zsplit = (maxc + cchunk - 1) / cchunk;
  dim3 grid(tiles, p.B, zsplit);
  const size_t smem = (size_t)2 * p.K * sizeof(double);
  if (mode == 0) warp_fwd_generic_kernel<FT, 0><<<grid, 256, smem, stream>>>(p, cchunk);
  else if (mode == 1) warp_fwd_generic_kernel<FT, 1><<<grid, 256, smem, stream>>>(p, cchunk);
  else warp_fwd_generic_kernel<FT, 2><<<grid, 256, smem, stream>>>(p, cchunk);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  return TPSPP_OK;
}

// ------------------------------------------------------------------------------------------
// classical TPS (RARE) with a large rectified grid: P_hat is [n, F+3] and *constant over the batch*
// (tps_preprocessor.py:255-282), so at 64x256 / F=40 it is 2.8 MB -- far bigger than an image.  The
// generic kernel re-reads a pixel's P_hat row for every image (TBs of L2 traffic per launch), and its
// fp64 grid arithmetic is one dependent chain per pixel.  Here a CTA keeps the rows of its 256-pixel tile
// in shared memory and walks a slice of the batch ("P_hat-stationary"), four images per pass: 8 independent
// fp64 chains per thread, then 16 independent gathers per channel.  ncu (profiles/r01_classical_tiled.md):
// the fp64 pipe is < 20 % busy; the kernel is bound by gather latency, so the grid is sized to exactly one
// resident wave and the gathers are batched.  (mma.sync.m8n8k4.f64 for the grid GEMM was tried: no gain.)
// ------------------------------------------------------------------------------------------
constexpr int CT_PIX = 256, CT_TB = 16, CT_IB = 4;

// T[b] = inv_delta_C[:, :F] . C'[b] in fp64, once per batch (tps_preprocessor.py:276-277), one thread per
// output; the tiled kernel then streams it with bulk copies instead of recomputing it in every pixel tile.
__global__ void __launch_bounds__(256) classical_T_kernel(WarpParams p) {
  const int o = blockIdx.x * 256 + threadIdx.x;
  if (o >= p.B * 2 * p.K) return;
  const int b = o / (2 * p.K), r = o - b * 2 * p.K, k = r >> 1, c = r & 1;
  const float* row = p.hatC + (size_t)k * p.K;
  const float* cp = p.c_prime + (size_t)b * p.F * 2 + c;
  double a0 = 0.0, a1 = 0.0;
  int f = 0;
  for (; f + 1 < p.F; f += 2) {
    a0 = fma((double)__ldg(row + f), (double)__ldg(cp + 2 * f), a0);
    a1 = fma((double)__ldg(row + f + 1), (double)__ldg(cp + 2 * f + 2), a1);
  }
  if (f < p.F) a0 = fma((double)__ldg(row + f), (double)__ldg(cp + 2 * f), a0);
  p.T_ws[o] = a0 + a1;
}

template <typename FT>
__global__ void __launch_bounds__(CT_PIX, 3) warp_fwd_classical_tiled_kernel(WarpParams p, int imgs_per_cta) {
  extern __shared__ __align__(16) unsigned char csm[];
  __shared__ __align__(8) uint64_t tbar[2];
  const int tid = threadIdx.x, K = p.K;
  const int TG = CT_TB * K * 2;                                         // doubles per T buffer
  double* Tbuf = reinterpret_cast<double*>(csm);                        // [2][CT_TB images][K][2]
  float* Ph = reinterpret_cast<float*>(Tbuf + 2 * (size_t)TG);          // [CT_PIX][PITCH] rows, odd pitch
  const int PITCH = K | 1;
  const int pix0 = blockIdx.x * CT_PIX;
  const int npix = min(CT_PIX, p.n - pix0);
  const int b_lo = blockIdx.y * imgs_per_cta, b_hi = min(p.B, b_lo + imgs_per_cta);
  for (int i = tid; i < 2 * TG; i += CT_PIX) Tbuf[i] = 0.0;             // rows past a short group stay finite
  if (tid == 0) { mbar_init(&tbar[0], 1); mbar_init(&tbar[1], 1); fence_barrier_init(); }
  __syncthreads();
  // producer side (thread 0): group g of the slice -> buffer g & 1, one bulk copy of nb * 2K doubles
  auto prefetch = [&](int g) {
    const int gb0 = b_lo + g * CT_TB;
    if (gb0 >= b_hi) return;
    const uint32_t bytes = (uint32_t)(min(CT_TB, b_hi - gb0) * 2 * K * sizeof(double));
    fence_proxy_async();
    mbar_arrive_expect_tx(&tbar[g & 1], bytes);
    bulk_g2s(Tbuf + (size_t)(g & 1) * TG, p.T_ws + (size_t)gb0 * 2 * K, bytes, &tbar[g & 1], policy_evict_last());
  };
  if (tid == 0) prefetch(0);
  for (int i = tid; i < npix * K; i += CT_PIX) {
    const int r = i / K, k = i - r * K;
    Ph[(size_t)r * PITCH + k] = __ldg(p.P_hat + (size_t)pix0 * K + i);
  }
  const int pix = pix0 + tid;
  const bool active = tid < npix;
  const float* ph = Ph + (size_t)tid * PITCH;
  for (int b0 = b_lo, g = 0; b0 < b_hi; b0 += CT_TB, ++g) {
    const int nb = min(CT_TB, b_hi - b0);
    __syncthreads();                            // everyone is done with group g-1's buffer (and Ph is visible)
    if (tid == 0) prefetch(g + 1);
    mbar_wait(&tbar[g & 1], (g >> 1) & 1);
    const double* Tsm = Tbuf + (size_t)(g & 1) * TG;
    if (!active) continue;
    // CT_IB images per pass: one P_hat load + conversion feeds 2*CT_IB independent fp64 FMA chains, and the
    // (Tx, Ty) pair of an image is one 16-byte broadcast load
    for (int bq = 0; bq < nb; bq += CT_IB) {
      double gx[CT_IB], gy[CT_IB];
#pragma unroll
      for (int i = 0; i < CT_IB; ++i) gx[i] = gy[i] = 0.0;
      const double2* T0 = reinterpret_cast<const double2*>(Tsm + (size_t)bq * 2 * K);
      for (int k = 0; k < K; ++k) {
        const double h = (double)ph[k];
#pragma unroll
        for (int i = 0; i < CT_IB; ++i) {
          const double2 tk = T0[(size_t)i * K + k];      // images past nb read stale-but-finite T rows; results unused
          gx[i] = fma(h, tk.x, gx[i]);
          gy[i] = fma(h, tk.y, gy[i]);
        }
      }
      // taps of all CT_IB images first, then channel by channel 4*CT_IB independent gathers in flight per
      // thread (the kernel is bound by gather latency, not by the fp64 pipe); images past nb alias the last
      // valid one and only their stores are predicated off
      float w[CT_IB][4];
      const FT* q[CT_IB];
      FT* op[CT_IB];
      const size_t plane = (size_t)p.H0 * p.W0;
      const int W = p.W0;
#pragma unroll
      for (int i = 0; i < CT_IB; ++i) {
        const int b = min(b0 + bq + i, b_hi - 1);
        if (p.grid_out != nullptr && bq + i < nb) {
          p.grid_out[((size_t)b * p.n + pix) * 2] = (float)gx[i];
          p.grid_out[((size_t)b * p.n + pix) * 2 + 1] = (float)gy[i];
        }
        const int off = make_taps_lean(gx[i], gy[i], W, p.H0, w[i]);
        q[i] = (const FT*)p.src0 + (size_t)b * p.C0 * plane + off;
        op[i] = (FT*)p.out0 + (size_t)b * p.C0 * p.n + pix;
      }
      for (int c = 0; c < p.C0; ++c) {
        float v[CT_IB][4];
#pragma unroll
        for (int i = 0; i < CT_IB; ++i) {
          v[i][0] = ldf(q[i]); v[i][1] = ldf(q[i] + 1); v[i][2] = ldf(q[i] + W); v[i][3] = ldf(q[i] + W + 1);
          q[i] += plane;
        }
#pragma unroll
        for (int i = 0; i < CT_IB; ++i) {
          if (bq + i < nb) stf(op[i], blend4(v[i][0], v[i][1], v[i][2], v[i][3], w[i]));
          op[i] += p.n;
        }
      }
    }
  }
}

// structural requirements of the P_hat-stationary kernel ...
static bool classical_tiled_supported(const tpspp_warp_cfg* cfg, const WarpParams& p) {
  return cfg->mode == TPSPP_MODE_CLASSICAL && p.C1 == 0 && p.K <= 67 && p.W0 >= 2 && p.H0 >= 2 && p.T_ws != nullptr;
}
// ... and when AUTO picks it: every CTA first loads its tile's P_hat rows, which only pays off with enough
// images per CTA (64x256 from B = 256; 32x100 from B ~ 1300 -- below that the per-pixel kernel is faster)
static bool classical_tiled_eligible(const tpspp_warp_cfg* cfg, const WarpParams& p) {
  return classical_tiled_supported(cfg, p) && p.n >= 4 * CT_PIX && (size_t)p.B * p.n >= ((size_t)1 << 22);
}

template <typename FT>
static int launch_classical_tiled_t(const WarpParams& p, cudaStream_t stream) {
  const int tiles = (p.n + CT_PIX - 1) / CT_PIX;
  const size_t smem = 2 * (size_t)CT_TB * p.K * 2 * sizeof(double) + (size_t)CT_PIX * (p.K | 1) * sizeof(float);
  TPSPP_CHECK_CUDA(cudaFuncSetAttribute(warp_fwd_classical_tiled_kernel<FT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // exactly one resident wave: batch slices sized so that tiles x chunks fits the CTAs the chip can hold
  int resident = 0;
  TPSPP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, warp_fwd_classical_tiled_kernel<FT>, CT_PIX, smem));
  int chunks = max(1, resident * sm_count() / tiles);
  int per = (p.B + chunks - 1) / chunks;
  per = (per + CT_IB - 1) / CT_IB * CT_IB;
  chunks = (p.B + per - 1) / per;
  classical_T_kernel<<<(p.B * 2 * p.K + 255) / 256, 256, 0, stream>>>(p);
  count_launch();
  dim3 grid(tiles, chunks);
  warp_fwd_classical_tiled_kernel<FT><<<grid, CT_PIX, smem, stream>>>(p, per);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  return TPSPP_OK;
}

static int launch_generic(const tpspp_warp_cfg* cfg, const WarpParams& p, int mode, cudaStream_t stream) {
  TPSPP_REQUIRE(cfg->feat_dtype != TPSPP_SRC0_BF16,
                "TPSPP_SRC0_BF16 (bf16 src0 with fp32 src1 / outputs) exists for the staged TPS++ kernel only (attention mode, F = 32, "
                "n <= 1024, 16-byte aligned tensors, grid_out NULL)");
  // an explicit TPSPP_VARIANT_GENERIC request keeps the plain kernel (tests compare the two)
  if (mode == 1 && cfg->variant == TPSPP_VARIANT_AUTO && classical_tiled_eligible(cfg, p)) {
    if (cfg->feat_dtype == TPSPP_BF16) return launch_classical_tiled_t<__nv_bfloat16>(p, stream);
    return launch_classical_tiled_t<float>(p, stream);
  }
  TPSPP_REQUIRE(p.B <= 65535, "batch %d exceeds the generic kernel's grid.y limit (65535)", p.B);
  if (cfg->feat_dtype == TPSPP_BF16) return launch_generic_t<__nv_bfloat16>(p, mode, stream);
  return launch_generic_t<float>(p, mode, stream);
}

void fill_params(const tpspp_warp_cfg* cfg, WarpParams* p) {
  memset(p, 0, sizeof(*p));
  p->B = cfg->batch; p->C0 = cfg->channels0; p->H0 = cfg->src0_h; p->W0 = cfg->src0_w;
  p->C1 = cfg->channels1; p->H1 = cfg->src1_h; p->W1 = cfg->src1_w;
  p->n = cfg->out_h * cfg->out_w; p->F = cfg->num_fiducial; p->K = cfg->num_fiducial + 3;
  p->mode = cfg->mode; p->theta = cfg->theta;
}

}  // namespace tpspp

using namespace tpspp;

extern "C" size_t tpspp_warp_fwd_workspace_bytes(const tpspp_warp_cfg* cfg) {
  if (validate_cfg(cfg) != TPSPP_OK || cfg->mode != TPSPP_MODE_CLASSICAL) return 0;
  return ((size_t)cfg->batch * (cfg->num_fiducial + 3) * 2 * sizeof(double) + 255) & ~(size_t)255;
}

extern "C" int tpspp_warp_fwd(const tpspp_warp_cfg* cfg, const void* src0, const void* src1,
                              const float* c_prime, const float* pc_score, const float* P_hat,
                              const float* P, const float* inv_delta_C, void* out0, void* out1,
                              float* grid_out, void* workspace, tpspp_stream_t stream) {
  reset_launch_count();
  int rc = validate_cfg(cfg);
  if (rc != TPSPP_OK) return rc;
  if (cfg->batch == 0) return TPSPP_OK;   // empty batch: nothing to do (pointers may be NULL)
  TPSPP_REQUIRE(src0 && out0 && c_prime && P_hat && inv_delta_C, "tpspp_warp_fwd: null required pointer");
  TPSPP_REQUIRE((cfg->channels1 == 0) == (src1 == nullptr) && (cfg->channels1 == 0) == (out1 == nullptr),
                "tpspp_warp_fwd: src1/out1 must be given exactly when channels1 > 0");
  if (cfg->mode == TPSPP_MODE_ATTENTION)
    TPSPP_REQUIRE(pc_score && P, "tpspp_warp_fwd: attention mode needs pc_score and P");
  if (cfg->batch == 0) return TPSPP_OK;
  WarpParams p;
  fill_params(cfg, &p);
  p.src0 = src0; p.src1 = src1; p.c_prime = c_prime; p.score = pc_score; p.P_hat = P_hat; p.P = P;
  p.hatC = inv_delta_C; p.out0 = out0; p.out1 = out1; p.grid_out = grid_out;
  TPSPP_REQUIRE(((uintptr_t)workspace & 255) == 0, "tpspp_warp_fwd: workspace must be 256-byte aligned");
  p.T_ws = reinterpret_cast<double*>(workspace);
  cudaStream_t st = (cudaStream_t)stream;
  int variant = cfg->variant;
  if (variant == TPSPP_VARIANT_AUTO) {
    uint32_t a, b, c;
    const bool aligned = !(((uintptr_t)src0 | (uintptr_t)src1 | (uintptr_t)pc_score | (uintptr_t)P_hat) & 15);
    variant = (grid_out == nullptr && aligned && staged_plan(cfg, &a, &b, &c) > 0) ? TPSPP_VARIANT_STAGED
                                                                                  : TPSPP_VARIANT_GENERIC;
  }
  if (variant == TPSPP_VARIANT_STAGED) return launch_staged(cfg, p, st);
  if (variant == TPSPP_VARIANT_GENERIC) return launch_generic(cfg, p, cfg->mode, st);
  if (variant == TPSPP_VARIANT_TILED) {
    TPSPP_REQUIRE(classical_tiled_supported(cfg, p),
                  "tpspp_warp_fwd: TPSPP_VARIANT_TILED needs classical mode, one source, F <= 64, a source of at "
                  "least 2x2 and a workspace of tpspp_warp_fwd_workspace_bytes()");
    if (cfg->feat_dtype == TPSPP_BF16) return launch_classical_tiled_t<__nv_bfloat16>(p, st);
    return launch_classical_tiled_t<float>(p, st);
  }
  set_error("tpspp_warp_fwd: unknown variant %d", cfg->variant);
  return TPSPP_E_INVALID;
}

extern "C" int tpspp_sample_fwd(const tpspp_warp_cfg* cfg, const void* src0, const void* src1,
                                const float* grid, void* out0, void* out1, tpspp_stream_t stream) {
  reset_launch_count();
  int rc = validate_cfg(cfg);
  if (rc != TPSPP_OK) return rc;
  if (cfg->batch == 0) return TPSPP_OK;
  TPSPP_REQUIRE(src0 && out0 && grid, "tpspp_sample_fwd: null required pointer");
  TPSPP_REQUIRE((cfg->channels1 == 0) == (src1 == nullptr) && (cfg->channels1 == 0) == (out1 == nullptr),
                "tpspp_sample_fwd: src1/out1 must be given exactly when channels1 > 0");
  if (cfg->batch == 0) return TPSPP_OK;
  WarpParams p;
  fill_params(cfg, &p);
  p.src0 = src0; p.src1 = src1; p.grid_in = grid; p.out0 = out0; p.out1 = out1;
  return launch_generic(cfg, p, 2, (cudaStream_t)stream);
}
