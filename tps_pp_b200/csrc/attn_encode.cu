// Multi-head self-attention over whole sequences: the attention of the NRTR encoder (reference encoders/nrtr_encoder.py:66-87
// -> TFEncoderLayer -> MultiHeadAttention / ScaledDotProductAttention, common/modules/transformer_module.py:24-34,74-98) with the
// encoder's source mask (nrtr_encoder.py _get_mask: image b attends to its keys j < len(b) only).
//   out[b,i,h,:] = sum_{j < len(b)} softmax_j((q[b,i,h,:] / temperature) . K[b,j,h,:]) V[b,j,h,:]   for every i < T
// Every query row is computed, the padded ones (i >= len(b)) included, as the reference does.  q / k / v: token-major
// [batch*T, heads*64] with one row stride (column slices of a fused q|k|v projection); out: [batch*T, heads*64] row-major.
// One CTA per (image, head, block of 64 queries), eight warps of eight queries.  The keys / values of the (image, head) pass
// through shared memory in tiles of 64 (K with a padded pitch); for q.K^T each lane owns one key (its dot products against
// the warp's eight queries, q broadcast from shared memory), for P.V each lane owns two of the 64 head dimensions (the
// probabilities broadcast from shared memory).  fp32 FMAs on CUDA cores, online soft-max in fp32.
#include "common.cuh"

namespace tpspp {

constexpr int AE_DIM = 64;                   // head dimension (d_k = d_v = 64 in the NRTR configs)
constexpr int AE_WARPS = 8;
constexpr int AE_QW = 8;                     // queries per warp
constexpr int AE_QB = AE_WARPS * AE_QW;      // queries per CTA
constexpr int AE_TK = 64;                    // keys per shared-memory tile
constexpr int AE_KP = AE_DIM + 4;            // K pitch: the float4 reads of 8 lanes (8 keys) hit 32 distinct banks
constexpr size_t AE_SMEM = (size_t)(AE_QB * AE_DIM + AE_TK * AE_KP + AE_TK * AE_DIM + AE_WARPS * AE_QW * 32) * sizeof(float);

__global__ void __launch_bounds__(AE_WARPS * 32, 2) attn_encode_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                                   const float* __restrict__ v, const int* __restrict__ kv_lens,
                                                                   float* __restrict__ out, int T, int heads, float temperature,
                                                                   int row_stride) {
  extern __shared__ __align__(16) float ae_sm[];
  float* Qs = ae_sm;                         // [QB][64]   q / temperature
  float* Ks = Qs + AE_QB * AE_DIM;           // [TK][KP]
  float* Vs = Ks + AE_TK * AE_KP;            // [TK][64]
  float* Ps = Vs + AE_TK * AE_DIM;           // [WARPS][QW][32] probabilities of the current 32 keys
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i0 = blockIdx.x * AE_QB, h = blockIdx.y, b = blockIdx.z;
  const int D = heads * AE_DIM, col = h * AE_DIM;
  const size_t img = (size_t)b * T;
  int len = kv_lens != nullptr ? kv_lens[b] : T;
  len = len < 0 ? 0 : (len > T ? T : len);
  for (int e = tid; e < AE_QB * AE_DIM / 4; e += AE_WARPS * 32) {
    const int r = e >> 4, c = (e & 15) * 4;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i0 + r < T) {
      x = *reinterpret_cast<const float4*>(q + (img + i0 + r) * row_stride + col + c);
      x.x /= temperature; x.y /= temperature; x.z /= temperature; x.w /= temperature;   // the reference scales q, then multiplies
    }
    *reinterpret_cast<float4*>(Qs + r * AE_DIM + c) = x;
  }
  const bool active = i0 + warp * AE_QW < T;
  const float* Qw = Qs + warp * AE_QW * AE_DIM;
  float* Pw = Ps + warp * AE_QW * 32;
  float m[AE_QW], l[AE_QW], a0[AE_QW], a1[AE_QW];
#pragma unroll
  for (int u = 0; u < AE_QW; ++u) { m[u] = -INFINITY; l[u] = 0.f; a0[u] = 0.f; a1[u] = 0.f; }
  for (int t0 = 0; t0 < len; t0 += AE_TK) {
    __syncthreads();                         // the previous tile is consumed
    for (int e = tid; e < AE_TK * AE_DIM / 4; e += AE_WARPS * 32) {
      const int r = e >> 4, c = (e & 15) * 4;
      float4 kx = make_float4(0.f, 0.f, 0.f, 0.f), vx = kx;
      if (t0 + r < len) {                    // keys past len(b) are zero rows: their probability is 0, and 0 * 0 stays 0
        const size_t off = (img + t0 + r) * row_stride + col + c;
        kx = *reinterpret_cast<const float4*>(k + off);
        vx = *reinterpret_cast<const float4*>(v + off);
      }
      *reinterpret_cast<float4*>(Ks + r * AE_KP + c) = kx;
      *reinterpret_cast<float4*>(Vs + r * AE_DIM + c) = vx;
    }
    __syncthreads();
    if (!active) continue;
    for (int s0 = 0; s0 < AE_TK && t0 + s0 < len; s0 += 32) {
      // scores: lane = key s0 + lane of the tile, against the warp's eight queries
      const float* kr = Ks + (s0 + lane) * AE_KP;
      float s[AE_QW];
#pragma unroll
      for (int u = 0; u < AE_QW; ++u) s[u] = 0.f;
#pragma unroll 2
      for (int d = 0; d < AE_DIM; d += 4) {
        const float4 kk = *reinterpret_cast<const float4*>(kr + d);
#pragma unroll
        for (int u = 0; u < AE_QW; ++u) {
          const float4 qq = *reinterpret_cast<const float4*>(Qw + u * AE_DIM + d);
          s[u] = fmaf(qq.x, kk.x, s[u]);
          s[u] = fmaf(qq.y, kk.y, s[u]);
          s[u] = fmaf(qq.z, kk.z, s[u]);
          s[u] = fmaf(qq.w, kk.w, s[u]);
        }
      }
      const bool valid = t0 + s0 + lane < len;
#pragma unroll
      for (int u = 0; u < AE_QW; ++u) {
        const float x = valid ? s[u] : -INFINITY;
        float mx = x;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float mn = fmaxf(m[u], mx);    // finite: key s0 (lane 0) is valid
        const float c = __expf(m[u] - mn);   // m = -inf before the first key: c = 0
        const float p = __expf(x - mn);      // masked key: 0
        l[u] = l[u] * c + p;                 // per-lane partial sum, reduced once at the end
        a0[u] *= c;
        a1[u] *= c;
        m[u] = mn;
        Pw[u * 32 + lane] = p;
      }
      __syncwarp();
      // P.V: lane = head dimensions 2 lane, 2 lane + 1
#pragma unroll 2
      for (int j = 0; j < 32; j += 4) {
        float2 vv[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) vv[jj] = *reinterpret_cast<const float2*>(Vs + (s0 + j + jj) * AE_DIM + 2 * lane);
#pragma unroll
        for (int u = 0; u < AE_QW; ++u) {
          const float4 pp = *reinterpret_cast<const float4*>(Pw + u * 32 + j);
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
  for (int u = 0; u < AE_QW; ++u) {
    float L = l[u];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) L += __shfl_xor_sync(0xffffffffu, L, o);
    const int i = i0 + warp * AE_QW + u;
    // len = 0: 0 / 0 = NaN, the reference's soft-max over an all-masked row
    if (i < T) *reinterpret_cast<float2*>(out + (img + i) * D + col + 2 * lane) = make_float2(a0[u] / L, a1[u] / L);
  }
}

}  // namespace tpspp

using namespace tpspp;

extern "C" int tpspp_attn_encode(const tpspp_attn_encode_cfg* cfg, const float* q, const float* k, const float* v,
                                 const int32_t* kv_lens, float* out, tpspp_stream_t stream) {
  reset_launch_count();
  TPSPP_REQUIRE(cfg != nullptr, "attn_encode cfg is NULL");
  TPSPP_REQUIRE(cfg->batch >= 0 && cfg->batch <= 65535 && cfg->heads > 0 && cfg->heads <= 65535,
                "attn_encode: 0 <= batch <= 65535, 1 <= heads <= 65535");
  TPSPP_REQUIRE(cfg->head_dim == AE_DIM, "attn_encode: head_dim must be 64 (d_k = d_v = 64 in the NRTR configs), got %d", cfg->head_dim);
  TPSPP_REQUIRE(cfg->seq_len >= 1, "attn_encode: seq_len must be >= 1, got %d", cfg->seq_len);
  TPSPP_REQUIRE(cfg->temperature > 0.f && cfg->temperature < INFINITY, "attn_encode: temperature must be positive and finite");
  if (cfg->batch == 0) return TPSPP_OK;
  TPSPP_REQUIRE(q && k && v && out, "tpspp_attn_encode: null pointer");
  TPSPP_REQUIRE((((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)out) & 15) == 0,
                "tpspp_attn_encode: buffers must be 16-byte aligned");
  const int D = cfg->heads * AE_DIM;
  const int rs = cfg->row_stride > 0 ? cfg->row_stride : D;
  TPSPP_REQUIRE(rs >= D && rs % 4 == 0, "tpspp_attn_encode: row_stride must be a multiple of 4 and >= heads * 64, got %d", rs);
  TPSPP_CHECK_CUDA(cudaFuncSetAttribute(attn_encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AE_SMEM));
  const dim3 grid((cfg->seq_len + AE_QB - 1) / AE_QB, cfg->heads, cfg->batch);
  attn_encode_kernel<<<grid, AE_WARPS * 32, AE_SMEM, (cudaStream_t)stream>>>(q, k, v, kv_lens, out, cfg->seq_len, cfg->heads,
                                                                             cfg->temperature, rs);
  count_launch();
  TPSPP_CHECK_CUDA(cudaGetLastError());
  return TPSPP_OK;
}
