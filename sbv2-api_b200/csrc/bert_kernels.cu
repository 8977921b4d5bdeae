// DeBERTa-v2 glue kernels: embedding gather, wide LayerNorm with planar fp16 copy, disentangled
// attention (HF modeling_deberta_v2.py:137-345 restated), output scatter.
#include <cuda_fp16.h>
#include <math_constants.h>

#include <type_traits>

#include "kernels.h"

namespace sbv2 {
namespace {

// two-term fp16 split of 8 fp32 values stored as the plane blocks [h0 | h1 | h0] (umma_conv.h make_split_conv1d_layer)
__device__ __forceinline__ void store_split8_attn(__half* base, long long blk, const float* f, float scale) {
  uint4 o0, o1;
  __half2* q0 = reinterpret_cast<__half2*>(&o0);
  __half2* q1 = reinterpret_cast<__half2*>(&o1);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float x0 = f[2 * e] * scale, x1 = f[2 * e + 1] * scale;
    const __half2 h0 = __floats2half2_rn(x0, x1);
    const float2 g0 = __half22float2(h0);
    q0[e] = h0;
    q1[e] = __floats2half2_rn(x0 - g0.x, x1 - g0.y);
  }
  *reinterpret_cast<uint4*>(base) = o0;
  *reinterpret_cast<uint4*>(base + blk) = o1;
  *reinterpret_cast<uint4*>(base + 2 * blk) = o0;
}

__global__ void embed_rows_kernel(float* h, const float* table, const int* ids, int C, int n_vocab, int64_t rows) {
  int64_t row = blockIdx.x;
  if (row >= rows) return;
  int id = ids[row];
  id = id < 0 ? 0 : (id >= n_vocab ? n_vocab - 1 : id);
  const float4* src = reinterpret_cast<const float4*>(table + (size_t)id * C);
  float4* dst = reinterpret_cast<float4*>(h + (size_t)row * C);
  for (int i = threadIdx.x; i < C / 4; i += blockDim.x) dst[i] = src[i];
}

// one warp per row; lane handles planes lane, lane+32, ... (NPL of them)
template <int NPL>
__global__ void ln_planar_wide_kernel(float* h, __half* hp, __half* hp2, const float* y32, const float* gamma, const float* beta,
                                      float eps, int C, PlanarSegs s) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (t >= s.len[b]) return;
  const int planes = C / 8;
  const size_t row = (size_t)s.start[b] + t;
  const size_t prow = (size_t)(s.pstart[b] + t) * 8;
  float v[NPL][8];
  float sum = 0.f;
#pragma unroll
  for (int q = 0; q < NPL; ++q) {
    const int pl = lane + 32 * q;
#pragma unroll
    for (int e = 0; e < 8; ++e) v[q][e] = 0.f;
    if (pl < planes) {
      const float4 x0 = *reinterpret_cast<const float4*>(h + row * C + pl * 8);
      const float4 x1 = *reinterpret_cast<const float4*>(h + row * C + pl * 8 + 4);
      v[q][0] = x0.x; v[q][1] = x0.y; v[q][2] = x0.z; v[q][3] = x0.w;
      v[q][4] = x1.x; v[q][5] = x1.y; v[q][6] = x1.z; v[q][7] = x1.w;
      if (y32) {
        const float4 y0 = *reinterpret_cast<const float4*>(y32 + (size_t)pl * s.plane_stride + prow);
        const float4 y1 = *reinterpret_cast<const float4*>(y32 + (size_t)pl * s.plane_stride + prow + 4);
        v[q][0] += y0.x; v[q][1] += y0.y; v[q][2] += y0.z; v[q][3] += y0.w;
        v[q][4] += y1.x; v[q][5] += y1.y; v[q][6] += y1.z; v[q][7] += y1.w;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) sum += v[q][e];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int q = 0; q < NPL; ++q) {
    if (lane + 32 * q < planes) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float d = v[q][e] - mean;
        sq += d * d;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = 1.0f / sqrtf(sq / (float)C + eps);
#pragma unroll
  for (int q = 0; q < NPL; ++q) {
    const int pl = lane + 32 * q;
    if (pl >= planes) continue;
    float r[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) r[e] = (v[q][e] - mean) * rstd * gamma[pl * 8 + e] + beta[pl * 8 + e];
    *reinterpret_cast<float4*>(h + row * C + pl * 8) = make_float4(r[0], r[1], r[2], r[3]);
    *reinterpret_cast<float4*>(h + row * C + pl * 8 + 4) = make_float4(r[4], r[5], r[6], r[7]);
    uint4 o;
    __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
    for (int e = 0; e < 4; ++e) oh[e] = __floats2half2_rn(r[2 * e], r[2 * e + 1]);
    if (hp) *reinterpret_cast<uint4*>(hp + (size_t)pl * s.plane_stride + prow) = o;
    if (hp2) *reinterpret_cast<uint4*>(hp2 + (size_t)pl * s.plane_stride + prow) = o;
  }
}

// Exact mode: h = LN(a + addin) (fp32 row-major, one warp per row, 8 channels per lane and iteration) and, in the same pass,
// the split-planar operand [h0 | h1 | h0] of the GEMM that consumes h.  NV8 = C / 256.
constexpr int LN_ROWS = 8;  // rows (= warps) per block

template <int NV8>
__device__ __forceinline__ void ln_split_row(float* out, __half* split, float split_scale, const float* a, const float* addin,
                                             const float* gamma, const float* beta, float eps, int C, const PlanarSegs& s, int b, int t,
                                             uint8_t* stage_raw) {
  const int lane = threadIdx.x & 31;
  const size_t base = ((size_t)s.start[b] + t) * C;
  float v[NV8][8];
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    const int c = (i * 32 + lane) * 8;
    float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
    if (c < C) {
      x0 = *reinterpret_cast<const float4*>(a + base + c);
      x1 = *reinterpret_cast<const float4*>(a + base + c + 4);
    }
    v[i][0] = x0.x; v[i][1] = x0.y; v[i][2] = x0.z; v[i][3] = x0.w; v[i][4] = x1.x; v[i][5] = x1.y; v[i][6] = x1.z; v[i][7] = x1.w;
  }
  if (addin) {
    float w[NV8][8];
#pragma unroll
    for (int i = 0; i < NV8; ++i) {
      const int c = (i * 32 + lane) * 8;
      float4 y0 = make_float4(0.f, 0.f, 0.f, 0.f), y1 = y0;
      if (c < C) {
        y0 = *reinterpret_cast<const float4*>(addin + base + c);
        y1 = *reinterpret_cast<const float4*>(addin + base + c + 4);
      }
      w[i][0] = y0.x; w[i][1] = y0.y; w[i][2] = y0.z; w[i][3] = y0.w; w[i][4] = y1.x; w[i][5] = y1.y; w[i][6] = y1.z; w[i][7] = y1.w;
    }
#pragma unroll
    for (int i = 0; i < NV8; ++i)
#pragma unroll
      for (int e = 0; e < 8; ++e) v[i][e] += w[i][e];
  }
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV8; ++i)
#pragma unroll
    for (int e = 0; e < 8; ++e) sum += v[i][e];  // lanes past C hold zeros
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    if ((i * 32 + lane) * 8 < C) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float d = v[i][e] - mean;
        sq += d * d;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = 1.0f / sqrtf(sq / (float)C + eps);
  // The split planes are staged in shared memory, [row of this block][term][plane][16 B] (+ one 16-byte pad per row: the
  // transposed read below is then conflict-free), and written out by the whole
  // block afterwards: a plane then receives the block's 8 consecutive rows as one 128-byte run instead of eight 16-byte
  // stores from eight warps (384 half-filled sectors per row were what the kernel spent its time on).
  uint4* stage = reinterpret_cast<uint4*>(stage_raw);
  const int w = threadIdx.x >> 5, planes = C / 8;
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    const int c = (i * 32 + lane) * 8;
    if (c >= C) continue;
    float r[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) r[e] = (v[i][e] - mean) * rstd * gamma[c + e] + beta[c + e];
    if (out) {
      *reinterpret_cast<float4*>(out + base + c) = make_float4(r[0], r[1], r[2], r[3]);
      *reinterpret_cast<float4*>(out + base + c + 4) = make_float4(r[4], r[5], r[6], r[7]);
    }
    if (split) {
      uint4 o0, o1;
      __half2* q0 = reinterpret_cast<__half2*>(&o0);
      __half2* q1 = reinterpret_cast<__half2*>(&o1);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float x0 = r[2 * e] * split_scale, x1 = r[2 * e + 1] * split_scale;
        const __half2 h0 = __floats2half2_rn(x0, x1);
        const float2 g0 = __half22float2(h0);
        q0[e] = h0;
        q1[e] = __floats2half2_rn(x0 - g0.x, x1 - g0.y);
      }
      stage[(size_t)w * (2 * planes + 1) + (c >> 3)] = o0;
      stage[(size_t)w * (2 * planes + 1) + planes + (c >> 3)] = o1;
    }
  }
}

// second half of ln_split: the block's staged split planes -> [h0 | h1 | h0] plane blocks, 128-byte runs
__device__ __forceinline__ void ln_split_flush(__half* split, const uint4* stage, int C, int t0, int nrows, const PlanarSegs& s, int b) {
  const int planes = C / 8;
  const long long blk = (long long)planes * s.plane_stride;
  const size_t prow0 = (size_t)(s.pstart[b] + t0) * 8;
  const int r = threadIdx.x & (LN_ROWS - 1);
  if (r >= nrows) return;
  for (int seg = threadIdx.x / LN_ROWS; seg < 2 * planes; seg += blockDim.x / LN_ROWS) {
    const int term = seg >= planes ? 1 : 0, pl = seg - term * planes;
    const uint4 val = stage[(size_t)r * (2 * planes + 1) + seg];
    __half* dst = split + (size_t)pl * s.plane_stride + prow0 + (size_t)r * 8;
    if (term == 0) {
      *reinterpret_cast<uint4*>(dst) = val;
      *reinterpret_cast<uint4*>(dst + 2 * blk) = val;
    } else {
      *reinterpret_cast<uint4*>(dst + blk) = val;
    }
  }
}

template <int NV8>
__global__ void __launch_bounds__(32 * LN_ROWS) ln_split_kernel(float* out, __half* split, float split_scale, const float* a,
                                                                const float* addin, const float* gamma, const float* beta, float eps, int C,
                                                                PlanarSegs s) {
  extern __shared__ __align__(16) uint8_t ln_stage[];  // [LN_ROWS][2 terms x C / 8 planes + 1][16 B]
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * LN_ROWS, t = t0 + (threadIdx.x >> 5);
  const int len = s.len[b];
  if (t0 >= len) return;  // block-uniform
  if (t < len) ln_split_row<NV8>(out, split, split_scale, a, addin, gamma, beta, eps, C, s, b, t, ln_stage);
  if (split == nullptr) return;
  __syncthreads();
  ln_split_flush(split, reinterpret_cast<const uint4*>(ln_stage), C, t0, min(LN_ROWS, len - t0), s, b);
}

__global__ void scatter_rows_kernel(float* out, const float* h, int C, int S, PlanarSegs s) {
  const int b = blockIdx.y, t = blockIdx.x;
  float4* dst = reinterpret_cast<float4*>(out + ((size_t)b * S + t) * C);
  if (t < s.len[b]) {
    const float4* src = reinterpret_cast<const float4*>(h + (size_t)(s.start[b] + t) * C);
    for (int i = threadIdx.x; i < C / 4; i += blockDim.x) dst[i] = src[i];
  } else {
    for (int i = threadIdx.x; i < C / 4; i += blockDim.x) dst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// ---------------------------------------------------------------------------------------------
// disentangled attention: 64 queries x 64 keys per step, D = 64, fp32 math on fp16 q|k|v.
// score[i][j] = (Q_i.K_j + Q_i.posK[idx(i-j)] + K_j.posQ[idx(i-j)]) / sqrt(3 D)
// For one (query tile, key tile) pair the needed position rows form one contiguous range of at
// most 127 rows (idx is monotone in i-j), so both bias terms are small tile GEMMs followed by a gather.
// ---------------------------------------------------------------------------------------------
constexpr int BQ = 64, BK = 64, BD = 64, BP = 128;
// row pitches (floats) of the shared-memory tiles: multiples of 4 so that the GEMM inner loops read their operands with
// 16-byte loads (3 LDS.128 per 32 FMA instead of 12 LDS.32)
constexpr int PQ = BQ + 4, PK = BK + 4, PPS = BQ + 4, PPT = BP + 4, PCP = BP + 2;

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ void from_f32(float& d, float v) { d = v; }
__device__ __forceinline__ void from_f32(__half& d, float v) { d = __float2half_rn(v); }

// pos_k_t / pos_q_t: the position projections transposed to [hidden][n_pos] so that a tile's rows load coalesced.
// F32 = false: q|k|v planar fp16 in, planar fp16 context out, V and the bias tiles staged as fp16 (the fast path's
// fallback for sequences the tensor-core kernel does not cover).
// F32 = true ("exact" mode, SBV2_B200_BERT=exact): q|k|v fp32 row-major [rows, 3*heads*64] in, fp32 row-major context
// [rows, heads*64] out, everything staged in fp32 — the features feed ceil() in the synthesizer (tts_util.rs:120-154 ->
// model.rs:66-68), and fp16 storage between the GEMMs alone costs 5e-4 relative.
// F32 with split_scale > 0: the context is written as the split-planar operand [h0 | h1 | h0] of the output projection
// (out_v = __half*, blocks of heads * 8 planes) instead of fp32 row-major — no separate split pass.
template <bool F32>
__global__ void __launch_bounds__(256) deberta_attention_kernel(void* out_v, const void* qkv_v, const float* pos_k_t, const float* pos_q_t,
                                                                int n_pos, const int* bucket_idx, int max_rel, int heads, PlanarSegs s,
                                                                float split_scale) {
  using TS = typename std::conditional<F32, float, __half>::type;
  __half* out = static_cast<__half*>(out_v);
  const __half* qkv = static_cast<const __half*>(qkv_v);
  float* out32 = static_cast<float*>(out_v);
  const float* qkv32 = static_cast<const float*>(qkv_v);
  extern __shared__ __align__(16) float sm[];
  float* Qt = sm;                     // [BD][PQ]   (scaled)
  float* Kt = Qt + BD * PQ;           // [BD][PK]
  float* Pt = Kt + BD * PK;           // [BD][PPT]  position rows (transposed), posK then posQ
  float* Pst = Pt;                    // [BK][PPS]  probabilities, key-major (Pt is dead once both bias tiles exist)
  TS* Vs = reinterpret_cast<TS*>(Pt + BD * PPT);  // [BK][BD]
  TS* C2P = Vs + BK * BD;             // [BQ][PCP]  bias tiles (fp16: 110 KB per CTA, two CTAs per SM overlap each
  TS* P2C = C2P + BQ * PCP;           // [BK][PCP]   other's synchronous load phases; fp32: 152 KB, one CTA per SM)

  const int b = blockIdx.z, h = blockIdx.y;
  const int len = s.len[b];
  const int q0 = blockIdx.x * BQ;
  if (q0 >= len) return;
  const long long pbase = s.pstart[b];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  constexpr int DP = BD / 8;
  const int HD = heads * BD;
  const float scale = 1.0f / sqrtf(3.0f * BD);
  const int q_plane0 = h * DP, k_plane0 = heads * DP + h * DP, v_plane0 = 2 * heads * DP + h * DP;
  const size_t ld32 = (size_t)3 * HD;          // F32: row pitch of qkv32
  const size_t row32 = (size_t)s.start[b];     // F32: first packed row of this sequence

  for (int i = tid; i < BQ * DP; i += 256) {
    const int r = i % BQ, pl = i / BQ;
    float f[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] = 0.f;
    if (q0 + r < len) {
      if (F32) {
        const float4* src = reinterpret_cast<const float4*>(qkv32 + (row32 + q0 + r) * ld32 + h * BD + pl * 8);
        const float4 a = src[0], c = src[1];
        f[0] = a.x * scale; f[1] = a.y * scale; f[2] = a.z * scale; f[3] = a.w * scale;
        f[4] = c.x * scale; f[5] = c.y * scale; f[6] = c.z * scale; f[7] = c.w * scale;
      } else {
        const uint4 u = *reinterpret_cast<const uint4*>(qkv + (size_t)(q_plane0 + pl) * s.plane_stride + (pbase + q0 + r) * 8);
        const __half2* uh = reinterpret_cast<const __half2*>(&u);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 y = __half22float2(uh[e]);
          f[2 * e] = y.x * scale;
          f[2 * e + 1] = y.y * scale;
        }
      }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) Qt[(pl * 8 + e) * PQ + r] = f[e];
  }

  float m_run[4], l_run[4], o[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m_run[i] = -CUDART_INF_F;
    l_run[i] = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) o[i][c] = 0.f;
  }

  for (int k0 = 0; k0 < len; k0 += BK) {
    __syncthreads();
    // K, V tiles
    for (int i = tid; i < BK * DP; i += 256) {
      const int r = i % BK, pl = i / BK;
      float kf[8], vf[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) kf[e] = vf[e] = 0.f;
      if (k0 + r < len) {
        if (F32) {
          const float4* ks = reinterpret_cast<const float4*>(qkv32 + (row32 + k0 + r) * ld32 + HD + h * BD + pl * 8);
          const float4* vs = reinterpret_cast<const float4*>(qkv32 + (row32 + k0 + r) * ld32 + 2 * HD + h * BD + pl * 8);
          const float4 a0 = ks[0], a1 = ks[1], c0 = vs[0], c1 = vs[1];
          kf[0] = a0.x; kf[1] = a0.y; kf[2] = a0.z; kf[3] = a0.w; kf[4] = a1.x; kf[5] = a1.y; kf[6] = a1.z; kf[7] = a1.w;
          vf[0] = c0.x; vf[1] = c0.y; vf[2] = c0.z; vf[3] = c0.w; vf[4] = c1.x; vf[5] = c1.y; vf[6] = c1.z; vf[7] = c1.w;
        } else {
          const uint4 uk = *reinterpret_cast<const uint4*>(qkv + (size_t)(k_plane0 + pl) * s.plane_stride + (pbase + k0 + r) * 8);
          const uint4 uv = *reinterpret_cast<const uint4*>(qkv + (size_t)(v_plane0 + pl) * s.plane_stride + (pbase + k0 + r) * 8);
          const __half2* kh = reinterpret_cast<const __half2*>(&uk);
          const __half2* vh = reinterpret_cast<const __half2*>(&uv);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 a = __half22float2(kh[e]), c = __half22float2(vh[e]);
            kf[2 * e] = a.x; kf[2 * e + 1] = a.y;
            vf[2 * e] = c.x; vf[2 * e + 1] = c.y;
          }
        }
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        Kt[(pl * 8 + e) * PK + r] = kf[e];
        from_f32(Vs[r * BD + pl * 8 + e], vf[e]);
      }
    }
    // position range of this tile pair: delta = i - j in [q0-k0-63, q0-k0+63], both ends clamped to the table's +-max_rel
    // (beyond max_rel + 63 tokens apart a whole range lies outside it)
    const int dmin = min(max(q0 - k0 - (BK - 1), -max_rel), max_rel), dmax = min(max(q0 - k0 + (BQ - 1), -max_rel), max_rel);
    const int pmin = bucket_idx[dmin + max_rel], pmax = bucket_idx[dmax + max_rel];
    const int np = pmax - pmin + 1;  // <= 127
    for (int phase = 0; phase < 2; ++phase) {
      const float* pos = phase == 0 ? pos_k_t : pos_q_t;
      __syncthreads();  // Pt free (and K/V/Q tiles visible on the first pass)
      for (int d = tid >> 5; d < BD; d += 8) {
        const float* src = pos + (size_t)(h * BD + d) * n_pos + pmin;
        for (int pr = tid & 31; pr < BP; pr += 32) Pt[d * PPT + pr] = pr < np ? src[pr] : 0.f;
      }
      __syncthreads();
      // [64 x 128] = X[64 x 64] . Pt[64 x 128]; thread: rows ty*4.., cols tx*8..
      float acc[4][8];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[i][c] = 0.f;
      const float* X = phase == 0 ? Qt : Kt;
      const int px = phase == 0 ? PQ : PK;
#pragma unroll 4
      for (int d = 0; d < BD; ++d) {
        const float4 xa = *reinterpret_cast<const float4*>(X + d * px + ty * 4);
        const float4 p0 = *reinterpret_cast<const float4*>(Pt + d * PPT + tx * 8);
        const float4 p1 = *reinterpret_cast<const float4*>(Pt + d * PPT + tx * 8 + 4);
        const float xr[4] = {xa.x, xa.y, xa.z, xa.w};
        const float pb[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int c = 0; c < 8; ++c) acc[i][c] = fmaf(xr[i], pb[c], acc[i][c]);
      }
      TS* dst = phase == 0 ? C2P : P2C;
      const float mul = phase == 0 ? 1.0f : scale;  // Q is pre-scaled, K is not
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 8; ++c) from_f32(dst[(ty * 4 + i) * PCP + tx * 8 + c], acc[i][c] * mul);
    }
    __syncthreads();
    float sc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) sc[i][j] = 0.f;
#pragma unroll 4
    for (int d = 0; d < BD; ++d) {
      const float4 q4 = *reinterpret_cast<const float4*>(Qt + d * PQ + ty * 4);
      const float4 k4 = *reinterpret_cast<const float4*>(Kt + d * PK + tx * 4);
      const float qa[4] = {q4.x, q4.y, q4.z, q4.w};
      const float kb[4] = {k4.x, k4.y, k4.z, k4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) sc[i][j] = fmaf(qa[i], kb[j], sc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int qi = q0 + ty * 4 + i;
      float mx = -CUDART_INF_F;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int kj = k0 + tx * 4 + j;
        int delta = qi - kj;
        delta = delta < -max_rel ? -max_rel : (delta > max_rel ? max_rel : delta);
        int pi = bucket_idx[delta + max_rel] - pmin;
        pi = pi < 0 ? 0 : (pi >= np ? np - 1 : pi);
        sc[i][j] += to_f32(C2P[(ty * 4 + i) * PCP + pi]) + to_f32(P2C[(tx * 4 + j) * PCP + pi]);
        if (kj >= len) sc[i][j] = -CUDART_INF_F;
        mx = fmaxf(mx, sc[i][j]);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float m_new = fmaxf(m_run[i], mx);
      const float corr = (m_run[i] == -CUDART_INF_F) ? 0.f : expf(m_run[i] - m_new);
      float psum = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float pv = (sc[i][j] == -CUDART_INF_F) ? 0.f : expf(sc[i][j] - m_new);
        Pst[(tx * 4 + j) * PPS + ty * 4 + i] = pv;
        psum += pv;
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, off);
      l_run[i] = l_run[i] * corr + psum;
      m_run[i] = m_new;
#pragma unroll
      for (int c = 0; c < 4; ++c) o[i][c] *= corr;
    }
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < BK; ++j) {
      const float4 p4 = *reinterpret_cast<const float4*>(Pst + j * PPS + ty * 4);
      const float pv[4] = {p4.x, p4.y, p4.z, p4.w};
      float vv[4];
      if (F32) {
        const float4 v4 = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(Vs) + j * BD + tx * 4);
        vv[0] = v4.x; vv[1] = v4.y; vv[2] = v4.z; vv[3] = v4.w;
      } else {
        const uint2 v4 = *reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(Vs) + j * BD + tx * 4);
        const float2 va = __half22float2(*reinterpret_cast<const __half2*>(&v4.x)), vb = __half22float2(*reinterpret_cast<const __half2*>(&v4.y));
        vv[0] = va.x; vv[1] = va.y; vv[2] = vb.x; vv[3] = vb.y;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) o[i][c] = fmaf(pv[i], vv[c], o[i][c]);
    }
  }
  __syncthreads();
  float* Os = Kt;  // [BQ][BD] fits in BD*PK
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float inv = 1.0f / l_run[i];
#pragma unroll
    for (int c = 0; c < 4; ++c) Os[(ty * 4 + i) * BD + tx * 4 + c] = o[i][c] * inv;
  }
  __syncthreads();
  for (int i = tid; i < BQ * DP; i += 256) {
    const int r = i % BQ, pl = i / BQ;
    if (q0 + r >= len) continue;
    if (F32 && split_scale > 0.f) {
      store_split8_attn(out + (size_t)(h * DP + pl) * s.plane_stride + (pbase + q0 + r) * 8, (long long)heads * DP * s.plane_stride,
                        Os + r * BD + pl * 8, split_scale);
      continue;
    }
    if (F32) {
      float4* dst = reinterpret_cast<float4*>(out32 + (row32 + q0 + r) * (size_t)HD + h * BD + pl * 8);
      const float* o8 = Os + r * BD + pl * 8;
      dst[0] = make_float4(o8[0], o8[1], o8[2], o8[3]);
      dst[1] = make_float4(o8[4], o8[5], o8[6], o8[7]);
      continue;
    }
    uint4 u;
    __half2* uh = reinterpret_cast<__half2*>(&u);
#pragma unroll
    for (int e = 0; e < 4; ++e) uh[e] = __floats2half2_rn(Os[r * BD + pl * 8 + 2 * e], Os[r * BD + pl * 8 + 2 * e + 1]);
    *reinterpret_cast<uint4*>(out + (size_t)(h * DP + pl) * s.plane_stride + (pbase + q0 + r) * 8) = u;
  }
}

// mean[a, c] = (float)((sum_t (double)feat[row0 + a][t][c]) / len[row0 + a]), t = 0 .. len-1 in order.  One thread per
// column: the threads of a warp read 32 consecutive floats of one token row (coalesced), and every group of TM_UNROLL
// loads is issued before the dependent fp64 adds consume it.  The sequential fp64 sum is what the host restates bit for bit.
constexpr int TM_THREADS = 128, TM_UNROLL = 8;
__global__ void __launch_bounds__(TM_THREADS) token_mean_kernel(float* __restrict__ mean, const float* __restrict__ feat,
                                                                const int* __restrict__ len, int row0, int S, int H) {
  const int a = blockIdx.y, c = blockIdx.x * TM_THREADS + threadIdx.x;
  if (c >= H) return;
  const int n = len[row0 + a];
  const float* p = feat + (size_t)(row0 + a) * S * H + c;
  double acc = 0.0;
  int t = 0;
  for (; t + TM_UNROLL <= n; t += TM_UNROLL) {
    float v[TM_UNROLL];
#pragma unroll
    for (int k = 0; k < TM_UNROLL; ++k) v[k] = __ldg(p + (size_t)(t + k) * H);
#pragma unroll
    for (int k = 0; k < TM_UNROLL; ++k) acc += (double)v[k];
  }
  for (; t < n; ++t) acc += (double)__ldg(p + (size_t)t * H);
  mean[(size_t)a * H + c] = (float)(acc / (double)n);
}

}  // namespace

#define POST_LAUNCH(ctx)            \
  do {                              \
    CUDA_CHECK(cudaGetLastError()); \
    (ctx).count();                  \
  } while (0)

void launch_embed_rows(const LaunchCtx& ctx, float* h, const float* table, const int* ids, int C, int n_vocab, int64_t rows) {
  if (rows <= 0) return;
  embed_rows_kernel<<<(unsigned)rows, 128, 0, ctx.stream>>>(h, table, ids, C, n_vocab, rows);
  POST_LAUNCH(ctx);
}

void launch_ln_planar_wide(const LaunchCtx& ctx, float* h, __half* hp, __half* hp2, const float* y32, const float* gamma,
                           const float* beta, float eps, int C, const PlanarSegs& s) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (C % 8 != 0 || C > 1024) fail(SBV2_ERR_UNSUPPORTED, "ln_planar_wide: C must be a multiple of 8 and <= 1024");
  dim3 grid((s.max_len + 7) / 8, s.n);
  const int planes = C / 8;
  if (planes <= 32) ln_planar_wide_kernel<1><<<grid, 256, 0, ctx.stream>>>(h, hp, hp2, y32, gamma, beta, eps, C, s);
  else if (planes <= 64) ln_planar_wide_kernel<2><<<grid, 256, 0, ctx.stream>>>(h, hp, hp2, y32, gamma, beta, eps, C, s);
  else ln_planar_wide_kernel<4><<<grid, 256, 0, ctx.stream>>>(h, hp, hp2, y32, gamma, beta, eps, C, s);
  POST_LAUNCH(ctx);
}

bool ln_split_supported(int C) { return C % 8 == 0 && C >= 8 && C <= 1024; }

void launch_ln_split(const LaunchCtx& ctx, float* out, __half* split, float split_scale, const float* a, const float* addin,
                     const float* gamma, const float* beta, float eps, int C, const PlanarSegs& s) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (!ln_split_supported(C)) fail(SBV2_ERR_UNSUPPORTED, "ln_split: hidden size must be a multiple of 8 and <= 1024");
  dim3 grid((s.max_len + LN_ROWS - 1) / LN_ROWS, s.n);
  const size_t smem = size_t(2 * (C / 8) + 1) * LN_ROWS * 16;  // <= 33 KB
  if (C <= 256) ln_split_kernel<1><<<grid, 32 * LN_ROWS, smem, ctx.stream>>>(out, split, split_scale, a, addin, gamma, beta, eps, C, s);
  else if (C <= 512) ln_split_kernel<2><<<grid, 32 * LN_ROWS, smem, ctx.stream>>>(out, split, split_scale, a, addin, gamma, beta, eps, C, s);
  else if (C <= 768) ln_split_kernel<3><<<grid, 32 * LN_ROWS, smem, ctx.stream>>>(out, split, split_scale, a, addin, gamma, beta, eps, C, s);
  else ln_split_kernel<4><<<grid, 32 * LN_ROWS, smem, ctx.stream>>>(out, split, split_scale, a, addin, gamma, beta, eps, C, s);
  POST_LAUNCH(ctx);
}

void launch_scatter_rows(const LaunchCtx& ctx, float* out, const float* h, int C, int S, const PlanarSegs& s) {
  if (s.n <= 0 || S <= 0) return;
  dim3 grid(S, s.n);
  scatter_rows_kernel<<<grid, 128, 0, ctx.stream>>>(out, h, C, S, s);
  POST_LAUNCH(ctx);
}

void launch_token_mean(const LaunchCtx& ctx, float* mean, const float* feat, const int* len, int row0, int n, int S, int H) {
  if (n <= 0 || H <= 0) return;
  dim3 grid((H + TM_THREADS - 1) / TM_THREADS, n);
  token_mean_kernel<<<grid, TM_THREADS, 0, ctx.stream>>>(mean, feat, len, row0, S, H);
  POST_LAUNCH(ctx);
}

void launch_deberta_attention(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const float* pos_k_t, const float* pos_q_t,
                              int n_pos, const int* bucket_idx, int max_rel, int heads, int head_dim, const PlanarSegs& s) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (head_dim != BD) fail(SBV2_ERR_UNSUPPORTED, "deberta attention: head_dim must be 64");
  size_t smem = sizeof(float) * (size_t)(BD * PQ + BD * PK + BD * PPT) + sizeof(__half) * (size_t)(BK * BD + BQ * PCP + BK * PCP);
  static PerDeviceOnce attr_once;
  attr_once.run([&] { CUDA_CHECK(cudaFuncSetAttribute(deberta_attention_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); });
  dim3 grid((s.max_len + BQ - 1) / BQ, heads, s.n);
  deberta_attention_kernel<false><<<grid, 256, smem, ctx.stream>>>(ctx_out, qkv, pos_k_t, pos_q_t, n_pos, bucket_idx, max_rel, heads, s, 0.f);
  POST_LAUNCH(ctx);
}

void launch_deberta_attention_f32(const LaunchCtx& ctx, float* ctx_out, __half* ctx_split, float split_scale, const float* qkv,
                                  const float* pos_k_t, const float* pos_q_t, int n_pos, const int* bucket_idx, int max_rel, int heads,
                                  int head_dim, const PlanarSegs& s) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (head_dim != BD) fail(SBV2_ERR_UNSUPPORTED, "deberta attention: head_dim must be 64");
  size_t smem = sizeof(float) * (size_t)(BD * PQ + BD * PK + BD * PPT) + sizeof(float) * (size_t)(BK * BD + BQ * PCP + BK * PCP);
  static PerDeviceOnce attr_once;
  attr_once.run([&] { CUDA_CHECK(cudaFuncSetAttribute(deberta_attention_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); });
  dim3 grid((s.max_len + BQ - 1) / BQ, heads, s.n);
  if (ctx_split)
    deberta_attention_kernel<true><<<grid, 256, smem, ctx.stream>>>(ctx_split, qkv, pos_k_t, pos_q_t, n_pos, bucket_idx, max_rel, heads, s, split_scale);
  else
    deberta_attention_kernel<true><<<grid, 256, smem, ctx.stream>>>(ctx_out, qkv, pos_k_t, pos_q_t, n_pos, bucket_idx, max_rel, heads, s, 0.f);
  POST_LAUNCH(ctx);
}

}  // namespace sbv2
