// Multi-head attention over whole sequences for training: forward and backward, with key-length and causal masks and the
// reference's attention dropout (common/modules/transformer_module.py:24-34 ScaledDotProductAttention; the three calls of an
// NRTR training step: encoder self-attention, decoder causal self-attention, decoder cross-attention).
//
// Forward (attn_train_fwd_kernel): the attn_encode scheme -- one CTA per (image, head, block of 64 queries), eight warps of
// eight queries, keys / values through shared memory in tiles of 64, online soft-max in fp32 -- with separate query / key
// lengths, the causal mask, the dropout mask applied to the probabilities that multiply V (the soft-max normaliser is the
// undropped one), and the row log-sum-exp written for the backward pass.
//
// Backward: the recompute scheme.  P = exp(S - lse), D = rowsum(dO * O), dP = (dO V^T) * M, dS = P * (dP - D), with
// M = keep / (1 - p).  Two kernels, neither with atomics: attn_train_dq_kernel (one CTA per query block) loops over key tiles
// and owns its dq rows; attn_train_dkv_kernel (one CTA per key block) loops over query tiles and owns its dk / dv rows.  Both
// compute the 64 x 64 (query, key) tile of P * M and dS with the same device function (bwd_tile), so they agree bit for bit.
//
// Dropout: keep(b, h, i, j) = Philox4x32-10(counter (j, i / 4, h, b), key = seed).word[i % 4] >= p * 2^32, regenerated where
// needed; the seed is read from device memory.
#include <curand_philox4x32_x.h>

#include "common.cuh"

namespace tpspp {

constexpr int AT_DIM = 64;                   // head dimension (d_k = d_v = 64)
constexpr int AT_MAXLEN = 256;               // len_q, len_k <= 256 (the sequences of one NRTR step are 40 and 64 long)
// forward: the attn_encode tiling
constexpr int AT_WARPS = 8;
constexpr int AT_QW = 8;                     // queries per warp
constexpr int AT_QB = AT_WARPS * AT_QW;      // queries per CTA
constexpr int AT_TK = 64;                    // keys per shared-memory tile
constexpr int AT_KP = AT_DIM + 4;            // K pitch: the float4 reads of 8 lanes (8 keys) hit 32 distinct banks
constexpr size_t AT_FWD_SMEM = (size_t)(AT_QB * AT_DIM + AT_TK * AT_KP + AT_TK * AT_DIM + AT_WARPS * AT_QW * 32) * sizeof(float)
                               + AT_TK * AT_WARPS;   // + the keep bits of the key tile: one byte per (key, warp), bit u = query u
// backward: 64 x 64 tiles with an odd pitch; thread (ty, tx) of 16 x 16 owns rows 4 ty .. 4 ty + 3 and columns tx + 16 c
constexpr int AT_BT = 64;
constexpr int AT_BP = AT_BT + 1;
constexpr int AT_TILE = AT_BT * AT_BP;
constexpr size_t AT_BWD_SMEM = (size_t)(6 * AT_TILE + 2 * AT_BT) * sizeof(float);

struct DropParams {
  uint2 key;                                 // Philox key (the 64-bit seed)
  uint32_t thr;                              // keep when the draw >= thr
  float scale;                               // 1 / (1 - p)
  bool on;
};

__device__ __forceinline__ DropParams drop_params(float p, const unsigned long long* seed_ptr) {
  DropParams d;
  d.on = p > 0.f;
  d.key = make_uint2(0u, 0u);
  d.thr = 0u;
  d.scale = 1.f;
  if (d.on) {
    const unsigned long long s = *seed_ptr;
    d.key = make_uint2((uint32_t)s, (uint32_t)(s >> 32));
    d.thr = (uint32_t)fminf(p * 4294967296.f, 4294967295.f);
    d.scale = 1.f / (1.f - p);
  }
  return d;
}

// the four draws of queries 4 i4 .. 4 i4 + 3 against key j
__device__ __forceinline__ uint4 keep_draws(const DropParams& d, int b, int h, int i4, int j) {
  return curand_Philox4x32_10(make_uint4((uint32_t)j, (uint32_t)i4, (uint32_t)h, (uint32_t)b), d.key);
}

__device__ __forceinline__ uint32_t word(const uint4& w, int r) {
  return r == 0 ? w.x : (r == 1 ? w.y : (r == 2 ? w.z : w.w));
}

__device__ __forceinline__ int clamp_len(const int* kv_lens, int b, int Lk) {
  int len = kv_lens != nullptr ? kv_lens[b] : Lk;
  return len < 0 ? 0 : (len > Lk ? Lk : len);
}

__global__ void __launch_bounds__(AT_WARPS * 32, 2)
attn_train_fwd_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                      const int* __restrict__ kv_lens, const unsigned long long* __restrict__ seed_ptr, float* __restrict__ out,
                      float* __restrict__ lse, int Lq, int Lk, int heads, float temperature, int causal, float dropout_p,
                      int q_stride, int kv_stride) {
  extern __shared__ __align__(16) float at_sm[];
  float* Qs = at_sm;                         // [QB][64]   q / temperature
  float* Ks = Qs + AT_QB * AT_DIM;           // [TK][KP]
  float* Vs = Ks + AT_TK * AT_KP;            // [TK][64]
  float* Ps = Vs + AT_TK * AT_DIM;           // [WARPS][QW][32] dropped probabilities of the current 32 keys
  uint8_t* Kb = reinterpret_cast<uint8_t*>(Ps + AT_WARPS * AT_QW * 32);   // [TK][WARPS] keep bits
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = blockIdx.x * AT_QB, h = blockIdx.y, b = blockIdx.z;
  const int D = heads * AT_DIM, col = h * AT_DIM;
  const size_t qimg = (size_t)b * Lq;
  const int len = clamp_len(kv_lens, b, Lk);
  const int kend = causal ? min(len, i0 + AT_QB) : len;     // the keys any query of this block sees
  const DropParams dp = drop_params(dropout_p, seed_ptr);
  k += (size_t)b * Lk * kv_stride + col;     // this (image, head)'s keys / values
  v += (size_t)b * Lk * kv_stride + col;
  for (int e = tid; e < AT_QB * AT_DIM / 4; e += AT_WARPS * 32) {
    const int r = e >> 4, c = (e & 15) * 4;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i0 + r < Lq) {
      x = *reinterpret_cast<const float4*>(q + (qimg + i0 + r) * q_stride + col + c);
      x.x /= temperature; x.y /= temperature; x.z /= temperature; x.w /= temperature;   // the reference scales q, then multiplies
    }
    *reinterpret_cast<float4*>(Qs + r * AT_DIM + c) = x;
  }
  const int iw = i0 + warp * AT_QW;          // the warp's first query (a multiple of 4)
  const bool active = iw < Lq;
  const float* Qw = Qs + warp * AT_QW * AT_DIM;
  float* Pw = Ps + warp * AT_QW * 32;
  float m[AT_QW], l[AT_QW], a0[AT_QW], a1[AT_QW];
#pragma unroll
  for (int u = 0; u < AT_QW; ++u) { m[u] = -INFINITY; l[u] = 0.f; a0[u] = 0.f; a1[u] = 0.f; }
  for (int t0 = 0; t0 < kend; t0 += AT_TK) {
    __syncthreads();                         // the previous tile is consumed
    for (int e = tid; e < AT_TK * AT_DIM / 4; e += AT_WARPS * 32) {
      const int r = e >> 4, c = (e & 15) * 4;
      float4 kx = make_float4(0.f, 0.f, 0.f, 0.f), vx = kx;
      if (t0 + r < kend) {                   // keys past the end are zero rows: their probability is 0, and 0 * 0 stays 0
        const int off = (t0 + r) * kv_stride + c;
        kx = *reinterpret_cast<const float4*>(k + off);
        vx = *reinterpret_cast<const float4*>(v + off);
      }
      *reinterpret_cast<float4*>(Ks + r * AT_KP + c) = kx;
      *reinterpret_cast<float4*>(Vs + r * AT_DIM + c) = vx;
    }
    if (dp.on) {                             // drawn here, where few registers are live: 2 x 2 Philox calls per thread
      const int jl = tid & (AT_TK - 1);
#pragma unroll
      for (int k2 = 0; k2 < 2; ++k2) {
        const int w8 = (tid >> 6) + 4 * k2;  // the warp whose eight queries this byte serves
        uint32_t bits = 0u;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          const uint4 w = keep_draws(dp, b, h, ((i0 + w8 * AT_QW) >> 2) + g, t0 + jl);
#pragma unroll
          for (int r = 0; r < 4; ++r) bits |= (word(w, r) >= dp.thr ? 1u : 0u) << (4 * g + r);
        }
        Kb[jl * AT_WARPS + w8] = (uint8_t)bits;
      }
    }
    __syncthreads();
    if (!active) continue;
    for (int s0 = 0; s0 < AT_TK && t0 + s0 < kend; s0 += 32) {
      const int j = t0 + s0 + lane;      // this lane's key
      const uint32_t keep = dp.on ? Kb[(s0 + lane) * AT_WARPS + warp] : 0xffu;
      const float* kr = Ks + (s0 + lane) * AT_KP;
      float s[AT_QW];
#pragma unroll
      for (int u = 0; u < AT_QW; ++u) s[u] = 0.f;
#pragma unroll 2
      for (int d = 0; d < AT_DIM; d += 4) {
        const float4 kk = *reinterpret_cast<const float4*>(kr + d);
#pragma unroll
        for (int u = 0; u < AT_QW; ++u) {
          const float4 qq = *reinterpret_cast<const float4*>(Qw + u * AT_DIM + d);
          s[u] = fmaf(qq.x, kk.x, s[u]);
          s[u] = fmaf(qq.y, kk.y, s[u]);
          s[u] = fmaf(qq.z, kk.z, s[u]);
          s[u] = fmaf(qq.w, kk.w, s[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < AT_QW; ++u) {
        const bool valid = j < kend && (!causal || j <= iw + u);
        const float x = valid ? s[u] : -INFINITY;
        float mx = x;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float mn = fmaxf(m[u], mx);    // finite: key 0 is valid for every query (len >= 1) and comes first
        const float c = __expf(m[u] - mn);   // m = -inf before the first key: c = 0
        const float p = __expf(x - mn);      // masked key: 0
        l[u] = l[u] * c + p;                 // per-lane partial sum of the undropped probabilities, reduced once at the end
        a0[u] *= c;
        a1[u] *= c;
        m[u] = mn;
        Pw[u * 32 + lane] = (keep >> u) & 1u ? p * dp.scale : 0.f;   // the dropout mask on what multiplies V
      }
      __syncwarp();
#pragma unroll 2
      for (int jj0 = 0; jj0 < 32; jj0 += 4) {
        float2 vv[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) vv[jj] = *reinterpret_cast<const float2*>(Vs + (s0 + jj0 + jj) * AT_DIM + 2 * lane);
#pragma unroll
        for (int u = 0; u < AT_QW; ++u) {
          const float4 pp = *reinterpret_cast<const float4*>(Pw + u * 32 + jj0);
          a0[u] = fmaf(pp.x, vv[0].x, a0[u]); a1[u] = fmaf(pp.x, vv[0].y, a1[u]);
          a0[u] = fmaf(pp.y, vv[1].x, a0[u]); a1[u] = fmaf(pp.y, vv[1].y, a1[u]);
          a0[u] = fmaf(pp.z, vv[2].x, a0[u]); a1[u] = fmaf(pp.z, vv[2].y, a1[u]);
          a0[u] = fmaf(pp.w, vv[3].x, a0[u]); a1[u] = fmaf(pp.w, vv[3].y, a1[u]);
        }
      }
      __syncwarp();                          // Pw is rewritten by the next 32 keys
    }
  }
  if (!active) return;
#pragma unroll
  for (int u = 0; u < AT_QW; ++u) {
    float L = l[u];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) L += __shfl_xor_sync(0xffffffffu, L, o);
    const int i = iw + u;
    if (i < Lq) {
      *reinterpret_cast<float2*>(out + (qimg + i) * D + col + 2 * lane) = make_float2(a0[u] / L, a1[u] / L);
      if (lane == 0) lse[((size_t)b * heads + h) * Lq + i] = m[u] + logf(L);
    }
  }
}

// rows [row0, row0 + 64) of a [*, heads*64] tensor (column block col) -> smem [64][AT_BP], zeros from row `end` on;
// optionally times `scale`
__device__ __forceinline__ void load_tile(float* dst, const float* __restrict__ src, size_t img, int row0, int end, int stride,
                                          int col, float scale) {
  for (int e = threadIdx.x; e < AT_BT * AT_DIM / 4; e += blockDim.x) {
    const int r = e >> 4, c = (e & 15) * 4;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row0 + r < end) x = *reinterpret_cast<const float4*>(src + (img + row0 + r) * stride + col + c);
    float* d = dst + r * AT_BP + c;
    d[0] = x.x * scale; d[1] = x.y * scale; d[2] = x.z * scale; d[3] = x.w * scale;
  }
}

// the per-query values of query rows [i0, i0 + 64): Qs = q / temperature, dOs = gout, lse, D = rowsum(gout * out)
__device__ __forceinline__ void load_queries(float* Qs, float* dOs, float* lse_s, float* D_s, const float* __restrict__ q,
                                             const float* __restrict__ out, const float* __restrict__ gout,
                                             const float* __restrict__ lse, int b, int h, int heads, int i0, int Lq, int q_stride,
                                             float temperature) {
  const int D = heads * AT_DIM, col = h * AT_DIM;
  const size_t qimg = (size_t)b * Lq;
  load_tile(Qs, q, qimg, i0, Lq, q_stride, col, 1.f / temperature);
  load_tile(dOs, gout, qimg, i0, Lq, D, col, 1.f);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = warp; r < AT_BT; r += blockDim.x >> 5) {
    const int i = i0 + r;
    float dsum = 0.f, ls = 0.f;
    if (i < Lq) {
      const float2 o = *reinterpret_cast<const float2*>(out + (qimg + i) * D + col + 2 * lane);
      const float2 g = *reinterpret_cast<const float2*>(gout + (qimg + i) * D + col + 2 * lane);
      dsum = o.x * g.x + o.y * g.y;
      ls = lse[((size_t)b * heads + h) * Lq + i];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
    if (lane == 0) { D_s[r] = dsum; lse_s[r] = ls; }
  }
}

// the (query, key) tile [i0, i0 + 64) x [j0, j0 + 64): Pd = P * M and dS = P * (dP * M - D), both stored [query][key]
__device__ __forceinline__ void bwd_tile(const float* Qs, const float* dOs, const float* Ks, const float* Vs, const float* lse_s,
                                         const float* D_s, float* Pd, float* dS, int i0, int j0, int Lq, int len, int causal,
                                         const DropParams& dp, int b, int h) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float s[4][4], g[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) { s[r][c] = 0.f; g[r][c] = 0.f; }
#pragma unroll 4
  for (int d = 0; d < AT_DIM; ++d) {
    float qa[4], oa[4], kb[4], vb[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) { qa[r] = Qs[(4 * ty + r) * AT_BP + d]; oa[r] = dOs[(4 * ty + r) * AT_BP + d]; }
#pragma unroll
    for (int c = 0; c < 4; ++c) { kb[c] = Ks[(tx + 16 * c) * AT_BP + d]; vb[c] = Vs[(tx + 16 * c) * AT_BP + d]; }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) { s[r][c] = fmaf(qa[r], kb[c], s[r][c]); g[r][c] = fmaf(oa[r], vb[c], g[r][c]); }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int jl = tx + 16 * c, j = j0 + jl;
    uint4 w = make_uint4(0u, 0u, 0u, 0u);
    if (dp.on) w = keep_draws(dp, b, h, (i0 >> 2) + ty, j);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int il = 4 * ty + r, i = i0 + il;
      const bool valid = i < Lq && j < len && (!causal || j <= i);
      const float p = valid ? __expf(s[r][c] - lse_s[il]) : 0.f;
      const float mk = dp.on ? (word(w, r) >= dp.thr ? dp.scale : 0.f) : 1.f;
      Pd[il * AT_BP + jl] = p * mk;
      dS[il * AT_BP + jl] = p * (g[r][c] * mk - D_s[il]);
    }
  }
}

__global__ void __launch_bounds__(256, 2)
attn_train_dq_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                     const float* __restrict__ out, const float* __restrict__ gout, const float* __restrict__ lse,
                     const int* __restrict__ kv_lens, const unsigned long long* __restrict__ seed_ptr, float* __restrict__ gq,
                     int Lq, int Lk, int heads, float temperature, int causal, float dropout_p, int q_stride, int kv_stride) {
  extern __shared__ __align__(16) float at_sm[];
  float *Qs = at_sm, *dOs = Qs + AT_TILE, *Ks = dOs + AT_TILE, *Vs = Ks + AT_TILE, *Pd = Vs + AT_TILE, *dS = Pd + AT_TILE;
  float *lse_s = dS + AT_TILE, *D_s = lse_s + AT_BT;
  const int i0 = blockIdx.x * AT_BT, h = blockIdx.y, b = blockIdx.z, col = h * AT_DIM;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int len = clamp_len(kv_lens, b, Lk);
  const int kend = causal ? min(len, i0 + AT_BT) : len;
  const DropParams dp = drop_params(dropout_p, seed_ptr);
  load_queries(Qs, dOs, lse_s, D_s, q, out, gout, lse, b, h, heads, i0, Lq, q_stride, temperature);
  float acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
  for (int j0 = 0; j0 < kend; j0 += AT_BT) {
    __syncthreads();                         // the previous key tile is consumed (and, the first time, the queries are loaded)
    load_tile(Ks, k, (size_t)b * Lk, j0, kend, kv_stride, col, 1.f);
    load_tile(Vs, v, (size_t)b * Lk, j0, kend, kv_stride, col, 1.f);
    __syncthreads();
    bwd_tile(Qs, dOs, Ks, Vs, lse_s, D_s, Pd, dS, i0, j0, Lq, kend, causal, dp, b, h);
    __syncthreads();
    // dq[i, d] += sum_j dS[i, j] k[j, d]
#pragma unroll 4
    for (int jl = 0; jl < AT_BT; ++jl) {
      float a[4], kb[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) a[r] = dS[(4 * ty + r) * AT_BP + jl];
#pragma unroll
      for (int c = 0; c < 4; ++c) kb[c] = Ks[jl * AT_BP + tx + 16 * c];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(a[r], kb[c], acc[r][c]);
    }
  }
  const float inv_t = 1.f / temperature;     // S = (q / temperature) k^T
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i = i0 + 4 * ty + r;
    if (i < Lq) {
#pragma unroll
      for (int c = 0; c < 4; ++c) gq[((size_t)b * Lq + i) * q_stride + col + tx + 16 * c] = acc[r][c] * inv_t;
    }
  }
}

__global__ void __launch_bounds__(256, 2)
attn_train_dkv_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                      const float* __restrict__ out, const float* __restrict__ gout, const float* __restrict__ lse,
                      const int* __restrict__ kv_lens, const unsigned long long* __restrict__ seed_ptr, float* __restrict__ gk,
                      float* __restrict__ gv, int Lq, int Lk, int heads, float temperature, int causal, float dropout_p,
                      int q_stride, int kv_stride) {
  extern __shared__ __align__(16) float at_sm[];
  float *Qs = at_sm, *dOs = Qs + AT_TILE, *Ks = dOs + AT_TILE, *Vs = Ks + AT_TILE, *Pd = Vs + AT_TILE, *dS = Pd + AT_TILE;
  float *lse_s = dS + AT_TILE, *D_s = lse_s + AT_BT;
  const int j0 = blockIdx.x * AT_BT, h = blockIdx.y, b = blockIdx.z, col = h * AT_DIM;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int len = clamp_len(kv_lens, b, Lk);
  const DropParams dp = drop_params(dropout_p, seed_ptr);
  float ak[4][4], av[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) { ak[r][c] = 0.f; av[r][c] = 0.f; }
  if (j0 < len) {
    load_tile(Ks, k, (size_t)b * Lk, j0, len, kv_stride, col, 1.f);
    load_tile(Vs, v, (size_t)b * Lk, j0, len, kv_stride, col, 1.f);
    // causal: queries i < j0 see none of these keys (j0 is a multiple of the query tile)
    for (int i0 = causal ? j0 : 0; i0 < Lq; i0 += AT_BT) {
      __syncthreads();                       // the previous query tile is consumed
      load_queries(Qs, dOs, lse_s, D_s, q, out, gout, lse, b, h, heads, i0, Lq, q_stride, temperature);
      __syncthreads();
      bwd_tile(Qs, dOs, Ks, Vs, lse_s, D_s, Pd, dS, i0, j0, Lq, len, causal, dp, b, h);
      __syncthreads();
      // dv[j, d] += sum_i Pd[i, j] gout[i, d];  dk[j, d] += sum_i dS[i, j] (q / temperature)[i, d]
#pragma unroll 2
      for (int il = 0; il < AT_BT; ++il) {
        float pa[4], sa[4], ob[4], qb[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) { pa[r] = Pd[il * AT_BP + 4 * ty + r]; sa[r] = dS[il * AT_BP + 4 * ty + r]; }
#pragma unroll
        for (int c = 0; c < 4; ++c) { ob[c] = dOs[il * AT_BP + tx + 16 * c]; qb[c] = Qs[il * AT_BP + tx + 16 * c]; }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c < 4; ++c) { av[r][c] = fmaf(pa[r], ob[c], av[r][c]); ak[r][c] = fmaf(sa[r], qb[c], ak[r][c]); }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int j = j0 + 4 * ty + r;
    if (j < Lk) {
      const size_t row = ((size_t)b * Lk + j) * kv_stride + col;
#pragma unroll
      for (int c = 0; c < 4; ++c) { gk[row + tx + 16 * c] = ak[r][c]; gv[row + tx + 16 * c] = av[r][c]; }
    }
  }
}

static int check_cfg(const tpspp_attn_train_cfg* cfg, int* qs, int* kvs) {
  TPSPP_REQUIRE(cfg != nullptr, "attn_train cfg is NULL");
  TPSPP_REQUIRE(cfg->batch >= 0 && cfg->batch <= 65535 && cfg->heads > 0 && cfg->heads <= 65535,
                "attn_train: 0 <= batch <= 65535, 1 <= heads <= 65535");
  TPSPP_REQUIRE(cfg->head_dim == AT_DIM, "attn_train: head_dim must be 64 (d_k = d_v = 64 in the NRTR configs), got %d", cfg->head_dim);
  TPSPP_REQUIRE(cfg->len_q >= 1 && cfg->len_q <= AT_MAXLEN && cfg->len_k >= 1 && cfg->len_k <= AT_MAXLEN,
                "attn_train: 1 <= len_q, len_k <= %d, got %d, %d", AT_MAXLEN, cfg->len_q, cfg->len_k);
  TPSPP_REQUIRE(cfg->temperature > 0.f && cfg->temperature < INFINITY, "attn_train: temperature must be positive and finite");
  TPSPP_REQUIRE(cfg->causal == 0 || cfg->causal == 1, "attn_train: causal must be 0 or 1, got %d", cfg->causal);
  TPSPP_REQUIRE(cfg->dropout_p >= 0.f && cfg->dropout_p < 1.f, "attn_train: dropout_p must be in [0, 1)");
  const int D = cfg->heads * AT_DIM;
  *qs = cfg->q_stride > 0 ? cfg->q_stride : D;
  *kvs = cfg->kv_stride > 0 ? cfg->kv_stride : D;
  TPSPP_REQUIRE(*qs >= D && *qs % 4 == 0 && *kvs >= D && *kvs % 4 == 0 && *kvs < (1 << 22),
                "attn_train: q_stride / kv_stride must be multiples of 4, >= heads * 64 and < 2^22, got %d / %d", *qs, *kvs);
  return TPSPP_OK;
}

}  // namespace tpspp

using namespace tpspp;

extern "C" int tpspp_attn_train_fwd(const tpspp_attn_train_cfg* cfg, const float* q, const float* k, const float* v,
                                    const int32_t* kv_lens, const uint64_t* seed_ptr, float* out, float* lse,
                                    tpspp_stream_t stream) {
  reset_launch_count();
  int qs = 0, kvs = 0;
  const int rc = check_cfg(cfg, &qs, &kvs);
  if (rc != TPSPP_OK) return rc;
  if (cfg->batch == 0) return TPSPP_OK;
  TPSPP_REQUIRE(q && k && v && out && lse, "tpspp_attn_train_fwd: null pointer");
  TPSPP_REQUIRE(cfg->dropout_p == 0.f || seed_ptr != nullptr, "tpspp_attn_train_fwd: dropout_p > 0 needs seed_ptr");
  TPSPP_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)out) & 15) == 0,
                "tpspp_attn_train_fwd: buffers must be 16-byte aligned");
  TPSPP_CHECK_CUDA(cudaFuncSetAttribute(attn_train_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AT_FWD_SMEM));
  const dim3 grid((cfg->len_q + AT_QB - 1) / AT_QB, cfg->heads, cfg->batch);
  attn_train_fwd_kernel<<<grid, AT_WARPS * 32, AT_FWD_SMEM, (cudaStream_t)stream>>>(
      q, k, v, kv_lens, reinterpret_cast<const unsigned long long*>(seed_ptr), out, lse, cfg->len_q, cfg->len_k, cfg->heads,
      cfg->temperature, cfg->causal, cfg->dropout_p, qs, kvs);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  return TPSPP_OK;
}

extern "C" int tpspp_attn_train_bwd(const tpspp_attn_train_cfg* cfg, const float* q, const float* k, const float* v,
                                    const float* out, const float* gout, const float* lse, const int32_t* kv_lens,
                                    const uint64_t* seed_ptr, float* gq, float* gk, float* gv, tpspp_stream_t stream) {
  reset_launch_count();
  int qs = 0, kvs = 0;
  const int rc = check_cfg(cfg, &qs, &kvs);
  if (rc != TPSPP_OK) return rc;
  if (cfg->batch == 0) return TPSPP_OK;
  TPSPP_REQUIRE(q && k && v && out && gout && lse && gq && gk && gv, "tpspp_attn_train_bwd: null pointer");
  TPSPP_REQUIRE(cfg->dropout_p == 0.f || seed_ptr != nullptr, "tpspp_attn_train_bwd: dropout_p > 0 needs seed_ptr");
  TPSPP_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)out | (uintptr_t)gout) & 15) == 0,
                "tpspp_attn_train_bwd: buffers must be 16-byte aligned");
  const unsigned long long* seed = reinterpret_cast<const unsigned long long*>(seed_ptr);
  TPSPP_CHECK_CUDA(cudaFuncSetAttribute(attn_train_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AT_BWD_SMEM));
  TPSPP_CHECK_CUDA(cudaFuncSetAttribute(attn_train_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AT_BWD_SMEM));
  const dim3 gq_grid((cfg->len_q + AT_BT - 1) / AT_BT, cfg->heads, cfg->batch);
  attn_train_dq_kernel<<<gq_grid, 256, AT_BWD_SMEM, (cudaStream_t)stream>>>(q, k, v, out, gout, lse, kv_lens, seed, gq, cfg->len_q,
                                                                           cfg->len_k, cfg->heads, cfg->temperature, cfg->causal,
                                                                           cfg->dropout_p, qs, kvs);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  const dim3 gkv_grid((cfg->len_k + AT_BT - 1) / AT_BT, cfg->heads, cfg->batch);
  attn_train_dkv_kernel<<<gkv_grid, 256, AT_BWD_SMEM, (cudaStream_t)stream>>>(q, k, v, out, gout, lse, kv_lens, seed, gk, gv,
                                                                             cfg->len_q, cfg->len_k, cfg->heads, cfg->temperature,
                                                                             cfg->causal, cfg->dropout_p, qs, kvs);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  return TPSPP_OK;
}
