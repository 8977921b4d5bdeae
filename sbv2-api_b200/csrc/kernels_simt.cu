// fp32 CUDA-core kernels: the exact path (text encoder, duration predictors, length regulator,
// alignment) and the glue around the tensor-core kernels.  See kernels.h for layouts.
#include <math_constants.h>

#include <climits>
#include <cstdlib>

#include "kernels.h"

namespace sbv2 {
namespace {

__device__ __forceinline__ float apply_act(float v, int act) {
  switch (act) {
    case ACT_RELU: return v > 0.f ? v : 0.f;
    case ACT_LRELU: return v > 0.f ? v : v * 0.1f;
    case ACT_LRELU01: return v > 0.f ? v : v * 0.01f;
    case ACT_GELU: return 0.5f * v * (1.f + erff(v * 0.70710678118654752440f));
    case ACT_TANH: return tanhf(v);
    default: return v;
  }
}

// ---------------------------------------------------------------------------------------------
// generic conv / linear: 64 rows x 64 couts per block, 256 threads, 4x4 outputs per thread
// ---------------------------------------------------------------------------------------------
constexpr int CT = 64, CN = 64, CK = 16;

template <bool VEC>
__global__ void __launch_bounds__(256) conv_kernel(ConvArgs a) {
  __shared__ float As[CK][CT + 4];
  __shared__ float Bs[CK][CN + 4];
  const int b = blockIdx.z;
  const int len = a.seg.len[b];
  const int t0 = blockIdx.x * CT;
  if (t0 >= len) return;
  const int in_base = a.seg.start[b];
  const int out_base = a.seg_out_start ? a.seg_out_start[b] : in_base;
  const int co0 = blockIdx.y * CN;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int a_r = tid >> 2;         // 0..63 row of the A tile this thread loads
  const int a_c = (tid & 3) * 4;    // ci offset 0,4,8,12
  const int b_r = tid >> 4;         // 0..15 ci row of the B tile
  const int b_c = (tid & 15) * 4;   // cout offset

  // fragment of step (m, c0) -> registers (global loads of the next step overlap the FMAs of this one)
  auto load_frag = [&](int m, int c0, float (&av)[4], float (&bv)[4]) {
    const int tin = t0 + a_r + a.off + m * a.dil;
    const bool row_ok = (t0 + a_r < len) && tin >= 0 && tin < len;
    const float* in_row = a.in + (size_t)(in_base + tin) * a.in_ld;
    const int ci = c0 + a_c;
    if (VEC) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row_ok && ci < a.cin) v = *reinterpret_cast<const float4*>(in_row + ci);
      av[0] = apply_act(v.x, a.act_in); av[1] = apply_act(v.y, a.act_in);
      av[2] = apply_act(v.z, a.act_in); av[3] = apply_act(v.w, a.act_in);
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) av[q] = (row_ok && ci + q < a.cin) ? apply_act(in_row[ci + q], a.act_in) : 0.f;
    }
    const float* wrow = a.w + ((size_t)m * a.cin + (c0 + b_r)) * a.cout;
    const int co = co0 + b_c;
    if (VEC) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c0 + b_r < a.cin && co < a.cout) v = *reinterpret_cast<const float4*>(wrow + co);
      bv[0] = v.x; bv[1] = v.y; bv[2] = v.z; bv[3] = v.w;
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) bv[q] = (c0 + b_r < a.cin && co + q < a.cout) ? wrow[co + q] : 0.f;
    }
  };

  const int kchunks = (a.cin + CK - 1) / CK;
  const int nsteps = a.taps * kchunks;
  float av[4], bv[4];
  load_frag(0, 0, av, bv);
  for (int step = 0; step < nsteps; ++step) {
#pragma unroll
    for (int q = 0; q < 4; ++q) As[a_c + q][a_r] = av[q];
    *reinterpret_cast<float4*>(&Bs[b_r][b_c]) = make_float4(bv[0], bv[1], bv[2], bv[3]);
    __syncthreads();
    if (step + 1 < nsteps) {
      const int ns = step + 1;
      const int m = ns / kchunks;
      load_frag(m, (ns - m * kchunks) * CK, av, bv);
    }
#pragma unroll
    for (int kk = 0; kk < CK; ++kk) {
      const float4 ar = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 br = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float arr[4] = {ar.x, ar.y, ar.z, ar.w}, brr[4] = {br.x, br.y, br.z, br.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(arr[i], brr[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int t = t0 + ty * 4 + i;
    if (t >= len) continue;
    size_t orow = (size_t)out_base + (size_t)t * a.out_row_mul + a.out_row_off;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int co = co0 + tx * 4 + j;
      if (co >= a.cout) continue;
      float v = acc[i][j];
      if (a.bias) v += a.bias[co];
      if (a.bias_utt) v += a.bias_utt[(size_t)b * a.cout + co];
      size_t o = orow * a.out_ld + co;
      if (a.residual) v += a.residual[o];
      v = apply_act(v, a.act_out);
      if (a.out) a.out[o] = v;
      if (a.accum_mode == ACC_SET) a.accum_out[o] = v;
      else if (a.accum_mode == ACC_ADD) a.accum_out[o] += v;
      else if (a.accum_mode == ACC_ADD_SCALE) a.accum_out[o] = (a.accum_out[o] + v) / a.accum_div;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// layout changes
// ---------------------------------------------------------------------------------------------
__global__ void cm_to_rm_kernel(const float* src, const int64_t* src_off, const int* src_ld, float* dst, int C, Segs seg) {
  __shared__ float tile[32][33];
  int b = blockIdx.z;
  int len = seg.len[b];
  int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  if (t0 >= len) return;
  const float* s = src + src_off[b];
  const int ld = src_ld ? src_ld[b] : len;
  int t = t0 + threadIdx.x;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int c = c0 + i;
    tile[i][threadIdx.x] = (c < C && t < len) ? s[(size_t)c * ld + t] : 0.f;
  }
  __syncthreads();
  int c = c0 + threadIdx.x;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int tt = t0 + i;
    if (tt < len && c < C) dst[(size_t)(seg.start[b] + tt) * C + c] = tile[threadIdx.x][i];
  }
}

__global__ void rm_to_cm_kernel(const float* src, float* dst, const int64_t* dst_off, int C, Segs seg) {
  __shared__ float tile[32][33];
  int b = blockIdx.z;
  int len = seg.len[b];
  int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  if (t0 >= len) return;
  float* d = dst + dst_off[b];
  int c = c0 + threadIdx.x;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int tt = t0 + i;
    tile[i][threadIdx.x] = (tt < len && c < C) ? src[(size_t)(seg.start[b] + tt) * C + c] : 0.f;
  }
  __syncthreads();
  int t = t0 + threadIdx.x;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int cc = c0 + i;
    if (cc < C && t < len) d[(size_t)cc * len + t] = tile[threadIdx.x][i];
  }
}

__global__ void embed_combine_kernel(float* h, const int* x, const int* tone, const int* lang, const float* emb,
                                     const float* tone_emb, const float* lang_emb, const float* style_emb, int C,
                                     int n_vocab, int n_tones, int n_lang, Segs seg, float scale) {
  int b = blockIdx.y;
  int t = blockIdx.x;
  if (t >= seg.len[b]) return;
  int row = seg.start[b] + t;
  int xi = min(max(x[row], 0), n_vocab - 1), ti = min(max(tone[row], 0), n_tones - 1), li = min(max(lang[row], 0), n_lang - 1);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    // same association order as the graph: (((emb + tone) + lang) + bert) + style
    float v = __fadd_rn(emb[(size_t)xi * C + c], tone_emb[(size_t)ti * C + c]);
    v = __fadd_rn(v, lang_emb[(size_t)li * C + c]);
    v = __fadd_rn(v, h[(size_t)row * C + c]);
    v = __fadd_rn(v, style_emb[(size_t)b * C + c]);
    h[(size_t)row * C + c] = __fmul_rn(v, scale);
  }
}

__global__ void gather_rows_kernel(float* out, const float* table, const int64_t* idx, int n, int C, int n_rows) {
  int b = blockIdx.x;
  int64_t i = idx[b];
  if (i < 0) i = 0;
  if (i >= n_rows) i = n_rows - 1;
  for (int c = threadIdx.x; c < C; c += blockDim.x) out[(size_t)b * C + c] = table[(size_t)i * C + c];
}

// out[b, :] = table[idx[b], :] * c_row + mean[slot[b], :] * c_mean with coef[s] = (c_row, c_mean), rounded after each
// product and after the sum (no FMA contraction: the host restatement reproduces it bit for bit); slot -1 copies the row.
template <bool VEC>
__global__ void gather_rows_blend_kernel(float* __restrict__ out, const float* __restrict__ table, const int64_t* __restrict__ idx,
                                         const int* __restrict__ slot, const float* __restrict__ mean, const float2* __restrict__ coef,
                                         int C, int n_rows, int n_slots) {
  const int b = blockIdx.x;
  int64_t i = idx[b];
  if (i < 0) i = 0;
  if (i >= n_rows) i = n_rows - 1;
  const int s = slot[b];
  const float* src = table + (size_t)i * C;
  float* dst = out + (size_t)b * C;
  if (s < 0 || s >= n_slots) {
    if (VEC)
      for (int c = threadIdx.x; c < C / 4; c += blockDim.x) reinterpret_cast<float4*>(dst)[c] = __ldg(reinterpret_cast<const float4*>(src) + c);
    else
      for (int c = threadIdx.x; c < C; c += blockDim.x) dst[c] = src[c];
    return;
  }
  const float2 k = coef[s];
  const float* m = mean + (size_t)s * C;
  if (VEC) {
    for (int c = threadIdx.x; c < C / 4; c += blockDim.x) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(src) + c), y = __ldg(reinterpret_cast<const float4*>(m) + c);
      reinterpret_cast<float4*>(dst)[c] =
          make_float4(__fadd_rn(__fmul_rn(x.x, k.x), __fmul_rn(y.x, k.y)), __fadd_rn(__fmul_rn(x.y, k.x), __fmul_rn(y.y, k.y)),
                      __fadd_rn(__fmul_rn(x.z, k.x), __fmul_rn(y.z, k.y)), __fadd_rn(__fmul_rn(x.w, k.x), __fmul_rn(y.w, k.y)));
    }
  } else {
    for (int c = threadIdx.x; c < C; c += blockDim.x) dst[c] = __fadd_rn(__fmul_rn(src[c], k.x), __fmul_rn(m[c], k.y));
  }
}

__global__ void add_utt_vec_kernel(float* out, const float* x, const float* v, int C, int v_ld, Segs seg) {
  int b = blockIdx.y;
  int t = blockIdx.x;
  if (t >= seg.len[b]) return;
  size_t row = (size_t)seg.start[b] + t;
  for (int c = threadIdx.x; c < C; c += blockDim.x) out[row * C + c] = x[row * C + c] + v[(size_t)b * v_ld + c];
}

// ---------------------------------------------------------------------------------------------
// layer norm over channels; one warp per row
// ---------------------------------------------------------------------------------------------
template <int MAXPER>
__global__ void layernorm_kernel(float* out, const float* a, const float* addin, const float* res, const float* gamma,
                                 const float* beta, float eps, int act, int C, int rows) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  size_t base = (size_t)warp * C;
  float v[MAXPER];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < MAXPER; ++i) {
    int c = lane + i * 32;
    float x = 0.f;
    if (c < C) {
      x = a[base + c];
      if (addin) x += addin[base + c];
    }
    v[i] = x;
    sum += x;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  float mean = sum / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < MAXPER; ++i) {
    int c = lane + i * 32;
    float d = (c < C) ? v[i] - mean : 0.f;
    sq += d * d;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  float rstd = 1.0f / sqrtf(sq / (float)C + eps);
#pragma unroll
  for (int i = 0; i < MAXPER; ++i) {
    int c = lane + i * 32;
    if (c < C) {
      float y = (v[i] - mean) * rstd * gamma[c] + beta[c];
      y = apply_act(y, act);
      if (res) y += res[base + c];
      out[base + c] = y;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// window-relative attention, flash style. 16 * RQ queries x 64 keys per step, 256 threads (thread = RQ rows x 4 keys).
// A row's arithmetic does not depend on RQ (its 16 threads hold the same 4 keys each in the same order), so the variants
// are bit-identical; few phoneme rows (one utterance) use RQ = 1 for four times the CTAs.
// ---------------------------------------------------------------------------------------------
constexpr int AK = 64;

// plain (not .nc) volatile loads: ptxas sinks read-only loads below the barrier that follows them, next to their first use,
// and the tile load becomes a chain of dependent round trips again
__device__ __forceinline__ float4 ldg_f4_issue_now(const float* p) {
  float4 v;
  asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

template <int D, int RQ>
__global__ void __launch_bounds__(256) rel_attention_kernel(float* out, const float* __restrict__ qkv, const float* __restrict__ rel_k,
                                                            const float* __restrict__ rel_v, int heads, int window, Segs seg) {
  extern __shared__ float sm[];
  constexpr int AQ = 16 * RQ;
  constexpr int DC = D / 16;  // output columns per thread
  constexpr int D4 = D / 4;
  const int R = 2 * window + 1;
  float* Qt = sm;                    // [D][AQ+1]
  float* Kt = Qt + D * (AQ + 1);     // [D][AK+1]
  float* Vs = Kt + D * (AK + 1);     // [AK][D]
  float* Ps = Vs + AK * D;           // [AQ][AK+1]
  float* Ek = Ps + AQ * (AK + 1);    // [R][D]
  float* Ev = Ek + R * D;            // [R][D]
  float* Qrel = Ev + R * D;          // [AQ][R]

  const int b = blockIdx.z, h = blockIdx.y;
  const int len = seg.len[b];
  const int q0 = blockIdx.x * AQ;
  if (q0 >= len) return;
  const int base = seg.start[b];
  const int ld = 3 * heads * D;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const float scale = 1.0f / sqrtf((float)D);

  for (int i = tid; i < R * D; i += 256) {
    Ek[i] = rel_k[i];
    Ev[i] = rel_v[i];
  }
  // 16-byte loads, all of a thread's loads issued before the first use: these phases are memory-latency bound
#pragma unroll
  for (int u = 0; u < (AQ * D4 + 255) / 256; ++u) {
    const int i = tid + u * 256;
    if (i < AQ * D4) {
      const int r = i / D4, d4 = i - r * D4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q0 + r < len) v = __ldg(reinterpret_cast<const float4*>(qkv + (size_t)(base + q0 + r) * ld + h * D) + d4);
      Qt[(d4 * 4 + 0) * (AQ + 1) + r] = v.x * scale;
      Qt[(d4 * 4 + 1) * (AQ + 1) + r] = v.y * scale;
      Qt[(d4 * 4 + 2) * (AQ + 1) + r] = v.z * scale;
      Qt[(d4 * 4 + 3) * (AQ + 1) + r] = v.w * scale;
    }
  }
  __syncthreads();
  for (int i = tid; i < AQ * R; i += 256) {
    int r = i / R, rr = i % R;
    float s = 0.f;
    for (int d = 0; d < D; ++d) s = fmaf(Qt[d * (AQ + 1) + r], Ek[rr * D + d], s);
    Qrel[r * R + rr] = s;
  }

  float m_run[RQ], l_run[RQ], o[RQ][DC];
#pragma unroll
  for (int i = 0; i < RQ; ++i) {
    m_run[i] = -CUDART_INF_F;
    l_run[i] = 0.f;
#pragma unroll
    for (int c = 0; c < DC; ++c) o[i][c] = 0.f;
  }

  constexpr int KV_PER = AK * D4 / 256;  // float4 loads per thread and operand
  static_assert(AK * D4 % 256 == 0, "K/V tile must divide over the block");
  float4 kq[KV_PER], vq[KV_PER];
  auto load_kv = [&](int k0) {
#pragma unroll
    for (int u = 0; u < KV_PER; ++u) {
      const int i = tid + u * 256;
      const int r = i / D4, d4 = i - r * D4;
      kq[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      vq[u] = kq[u];
      if (k0 + r < len) {
        const float* row = qkv + (size_t)(base + k0 + r) * ld;
        kq[u] = ldg_f4_issue_now(row + heads * D + h * D + d4 * 4);
        vq[u] = ldg_f4_issue_now(row + 2 * heads * D + h * D + d4 * 4);
      }
    }
  };
  load_kv(0);
  for (int k0 = 0; k0 < len; k0 += AK) {
    __syncthreads();  // previous step's consumers of Kt/Vs/Ps are done (also orders Qrel)
#pragma unroll
    for (int u = 0; u < KV_PER; ++u) {
      const int i = tid + u * 256;
      const int r = i / D4, d4 = i - r * D4;
      Kt[(d4 * 4 + 0) * (AK + 1) + r] = kq[u].x;
      Kt[(d4 * 4 + 1) * (AK + 1) + r] = kq[u].y;
      Kt[(d4 * 4 + 2) * (AK + 1) + r] = kq[u].z;
      Kt[(d4 * 4 + 3) * (AK + 1) + r] = kq[u].w;
      *reinterpret_cast<float4*>(Vs + r * D + d4 * 4) = vq[u];
    }
    __syncthreads();
    if (k0 + AK < len) load_kv(k0 + AK);  // in flight while this tile is computed
    float s[RQ][4];
#pragma unroll
    for (int i = 0; i < RQ; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
    for (int d = 0; d < D; ++d) {
      float qa[RQ], kb[4];
#pragma unroll
      for (int i = 0; i < RQ; ++i) qa[i] = Qt[d * (AQ + 1) + ty * RQ + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) kb[j] = Kt[d * (AK + 1) + tx * 4 + j];
#pragma unroll
      for (int i = 0; i < RQ; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) s[i][j] = fmaf(qa[i], kb[j], s[i][j]);
    }
    // relative-key bias, key validity, running softmax
#pragma unroll
    for (int i = 0; i < RQ; ++i) {
      int qi = q0 + ty * RQ + i;
      float mx = -CUDART_INF_F;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        int kj = k0 + tx * 4 + j;
        int rel = kj - qi;
        if (rel >= -window && rel <= window) s[i][j] += Qrel[(ty * RQ + i) * R + rel + window];
        if (kj >= len) s[i][j] = -CUDART_INF_F;
        mx = fmaxf(mx, s[i][j]);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      float m_new = fmaxf(m_run[i], mx);
      float corr = (m_run[i] == -CUDART_INF_F) ? 0.f : expf(m_run[i] - m_new);
      float psum = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float p = (s[i][j] == -CUDART_INF_F) ? 0.f : expf(s[i][j] - m_new);
        Ps[(ty * RQ + i) * (AK + 1) + tx * 4 + j] = p;
        psum += p;
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, off);
      l_run[i] = fmaf(l_run[i], corr, psum);  // explicit: ptxas may or may not fuse a*b+c, and differently per instantiation
      m_run[i] = m_new;
#pragma unroll
      for (int c = 0; c < DC; ++c) o[i][c] *= corr;
    }
    __syncthreads();
    // O += P V
    for (int j = 0; j < AK; ++j) {
      float pv[RQ], vv[DC];
#pragma unroll
      for (int i = 0; i < RQ; ++i) pv[i] = Ps[(ty * RQ + i) * (AK + 1) + j];
#pragma unroll
      for (int c = 0; c < DC; ++c) vv[c] = Vs[j * D + tx * DC + c];
#pragma unroll
      for (int i = 0; i < RQ; ++i)
#pragma unroll
        for (int c = 0; c < DC; ++c) o[i][c] = fmaf(pv[i], vv[c], o[i][c]);
    }
    // relative-value term for keys of this tile inside the window
#pragma unroll
    for (int i = 0; i < RQ; ++i) {
      int qi = q0 + ty * RQ + i;
      for (int rr = 0; rr < R; ++rr) {
        int kj = qi + rr - window;
        if (kj >= k0 && kj < k0 + AK && kj < len && kj >= 0) {
          float p = Ps[(ty * RQ + i) * (AK + 1) + (kj - k0)];
#pragma unroll
          for (int c = 0; c < DC; ++c) o[i][c] = fmaf(p, Ev[rr * D + tx * DC + c], o[i][c]);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < RQ; ++i) {
    int qi = q0 + ty * RQ + i;
    if (qi >= len) continue;
    float inv = 1.0f / l_run[i];
#pragma unroll
    for (int c = 0; c < DC; ++c) out[(size_t)(base + qi) * (heads * D) + h * D + tx * DC + c] = o[i][c] * inv;
  }
}

// ---------------------------------------------------------------------------------------------
// per-utterance vector through a Linear (k = 1 conv on one row per utterance: speaker / style conditioning).
// 32 outputs x 8 K slices per block; the generic conv kernel walks K in 16-channel steps at one memory latency each
// (37 us for 512 inputs), this one issues its 64 loads per thread in unrolled batches.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) utt_linear_kernel(ConvArgs a) {
  __shared__ float red[8][33];
  const int b = blockIdx.z, t = blockIdx.y;
  if (t >= a.seg.len[b]) return;
  const int in_base = a.seg.start[b] + t;
  const int out_base = (a.seg_out_start ? a.seg_out_start[b] : a.seg.start[b]) + t * a.out_row_mul;
  const int col = threadIdx.x & 31, ks = threadIdx.x >> 5;
  const int co = blockIdx.x * 32 + col;
  const int per = (a.cin + 7) / 8;
  const int c_lo = ks * per, c_hi = min(a.cin, c_lo + per);
  const float* __restrict__ in = a.in + (size_t)in_base * a.in_ld;
  const float* __restrict__ w = a.w;
  float acc = 0.f;
  if (co < a.cout) {
    if (a.act_in == ACT_NONE) {  // the branchy activation switch inside the loop keeps the loads from being batched
#pragma unroll 16
      for (int ci = c_lo; ci < c_hi; ++ci) acc = fmaf(__ldg(in + ci), __ldg(w + (size_t)ci * a.cout + co), acc);
    } else {
      for (int ci = c_lo; ci < c_hi; ++ci) acc = fmaf(apply_act(__ldg(in + ci), a.act_in), __ldg(w + (size_t)ci * a.cout + co), acc);
    }
  }
  red[ks][col] = acc;
  __syncthreads();
  if (ks != 0 || co >= a.cout) return;
  float v = red[0][col];
#pragma unroll
  for (int q = 1; q < 8; ++q) v += red[q][col];
  if (a.bias) v += a.bias[co];
  if (a.bias_utt) v += a.bias_utt[(size_t)b * a.cout + co];
  const size_t o = ((size_t)out_base + a.out_row_off) * a.out_ld + co;
  if (a.residual) v += a.residual[o];
  v = apply_act(v, a.act_out);
  if (a.out) a.out[o] = v;
}

// ---------------------------------------------------------------------------------------------
// DDSConv / SDP pieces
// ---------------------------------------------------------------------------------------------
__global__ void dwconv3_kernel(float* out, const float* in, const float* w, const float* bias, int C, int dil, Segs seg) {
  int b = blockIdx.y, t = blockIdx.x;
  int len = seg.len[b];
  if (t >= len) return;
  size_t base = seg.start[b];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc = bias[c];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      int tt = t + (j - 1) * dil;
      if (tt >= 0 && tt < len) acc = fmaf(w[c * 3 + j], in[(base + tt) * C + c], acc);
    }
    out[(base + t) * C + c] = acc;
  }
}

__global__ void sdp_init_kernel(float* z, const float* noise, const float* nsw, Segs seg) {
  int b = blockIdx.y;
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= seg.len[b]) return;
  size_t row = (size_t)seg.start[b] + t;
  z[row * 2 + 0] = noise[row * 2 + 0] * nsw[b];
  z[row * 2 + 1] = noise[row * 2 + 1] * nsw[b];
}

__global__ void sdp_flip_kernel(float* z, int rows) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows) return;
  float a = z[t * 2], b = z[t * 2 + 1];
  z[t * 2] = b;
  z[t * 2 + 1] = a;
}

__global__ void convflow_pre_kernel(float* h, const float* z, const float* w, const float* b, const float* g, int C,
                                    int rows) {
  int t = blockIdx.x;
  if (t >= rows) return;
  float x0 = z[t * 2];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float v = fmaf(w[c], x0, b[c]);
    h[(size_t)t * C + c] = v + g[(size_t)t * C + c];
  }
}

__device__ __forceinline__ float softplusf(float x) { return x > 20.f ? x : log1pf(expf(x)); }

// One thread per row; 10 bins.  Follows upstream transforms.rational_quadratic_spline (inverse).
template <int NB>
__global__ void convflow_spline_kernel(float* z, const float* proj, int ld, float tail_bound, float inv_sqrt_filter,
                                       int rows) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows) return;
  float x = z[t * 2 + 1];
  if (!(x >= -tail_bound && x <= tail_bound)) return;  // linear tails: identity
  const float* p = proj + (size_t)t * ld;
  const float min_w = 1e-3f, min_h = 1e-3f, min_d = 1e-3f;
  float uw[NB], uh[NB], ud[NB + 1];
  float mw = -CUDART_INF_F, mh = -CUDART_INF_F;
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    uw[i] = p[i] * inv_sqrt_filter;
    uh[i] = p[NB + i] * inv_sqrt_filter;
    mw = fmaxf(mw, uw[i]);
    mh = fmaxf(mh, uh[i]);
  }
  const float cst = logf(expf(1.f - min_d) - 1.f);
  ud[0] = cst;
  ud[NB] = cst;
#pragma unroll
  for (int i = 1; i < NB; ++i) ud[i] = p[2 * NB + i - 1];
  float sw = 0.f, sh = 0.f;
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    uw[i] = expf(uw[i] - mw);
    sw += uw[i];
    uh[i] = expf(uh[i] - mh);
    sh += uh[i];
  }
  float cumw[NB + 1], cumh[NB + 1];
  float aw = 0.f, ah = 0.f;
  cumw[0] = -tail_bound;
  cumh[0] = -tail_bound;
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    float wi = min_w + (1.f - min_w * NB) * (uw[i] / sw);
    float hi = min_h + (1.f - min_h * NB) * (uh[i] / sh);
    aw += wi;
    ah += hi;
    cumw[i + 1] = 2.f * tail_bound * aw + (-tail_bound);
    cumh[i + 1] = 2.f * tail_bound * ah + (-tail_bound);
  }
  cumw[NB] = tail_bound;
  cumh[NB] = tail_bound;
  // searchsorted on cumheights (last edge + eps)
  int bin = -1;
#pragma unroll
  for (int i = 0; i <= NB; ++i) {
    float edge = cumh[i] + (i == NB ? 1e-6f : 0.f);
    bin += (x >= edge) ? 1 : 0;
  }
  bin = min(max(bin, 0), NB - 1);
  float in_cw = 0.f, in_w = 1.f, in_ch = 0.f, in_h = 1.f, d0 = 1.f, d1 = 1.f;
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    if (i == bin) {
      in_cw = cumw[i];
      in_w = cumw[i + 1] - cumw[i];
      in_ch = cumh[i];
      in_h = cumh[i + 1] - cumh[i];
      d0 = min_d + softplusf(ud[i]);
      d1 = min_d + softplusf(ud[i + 1]);
    }
  }
  float delta = in_h / in_w;
  float dy = x - in_ch;
  float s2 = d0 + d1 - 2.f * delta;
  float a = dy * s2 + in_h * (delta - d0);
  float bq = in_h * d0 - dy * s2;
  float c = -delta * dy;
  float disc = bq * bq - 4.f * a * c;
  disc = fmaxf(disc, 0.f);
  float root = (2.f * c) / (-bq - sqrtf(disc));
  z[t * 2 + 1] = root * in_w + in_cw;
}

__global__ void sdp_affine_kernel(float* z, const float* m, const float* logs, int rows) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows) return;
  z[t * 2 + 0] = (z[t * 2 + 0] - m[0]) * expf(-logs[0]);
  z[t * 2 + 1] = (z[t * 2 + 1] - m[1]) * expf(-logs[1]);
}

// ---------------------------------------------------------------------------------------------
// length regulator
// ---------------------------------------------------------------------------------------------
// kGiven: utterance b takes the caller's integers given[] when given_flag[b] != 0 (the DP / SDP outputs are not read
// for it) and the predicted durations otherwise; both go through the same clamp, scan, cum and ylen rules.
template <bool kGiven>
__device__ __forceinline__ void durations_body(const float* logw_dp, const float* z_sdp, const float* sdp_ratio, const float* length_scale,
                                               const int* given, const int* given_flag, float* w_out, int* dur, int* cum, int* ylen,
                                               const Segs& seg) {
  // one warp per utterance: chunked inclusive scan
  int b = blockIdx.x;
  int lane = threadIdx.x;
  int len = seg.len[b];
  int base = seg.start[b];
  float ratio = sdp_ratio[b], ls = length_scale[b];
  const bool use_given = kGiven && given_flag[b] != 0;
  // 64-bit total: 2^20 phonemes of up to 1e6 frames each exceed int32.  ylen saturates at INT_MAX, which the host
  // rejects as too long; whenever it accepts the batch, every prefix in cum fits in int32.
  long long carry = 0;
  for (int t0 = 0; t0 < len; t0 += 32) {
    int t = t0 + lane;
    int d = 0;
    if (t < len && use_given) {
      d = min(max(given[base + t], 0), 1000000);
      if (w_out) w_out[base + t] = (float)d;
      dur[base + t] = d;
    } else if (t < len) {
      float dp = logw_dp[base + t];
      float logw;
      if (z_sdp) {
        // logw = sdp * ratio + dp * (1 - ratio), products rounded separately as the graph does
        logw = __fadd_rn(__fmul_rn(z_sdp[(size_t)(base + t) * 2], ratio), __fmul_rn(dp, __fsub_rn(1.f, ratio)));
      } else {
        logw = __fmul_rn(dp, __fsub_rn(1.f, ratio));
      }
      float w = __fmul_rn(expf(logw), ls);
      if (w_out) w_out[base + t] = w;
      float c = ceilf(w);
      // clamp so a pathological duration cannot overflow the scan (still reported as-is in w_out)
      c = fminf(fmaxf(c, 0.f), 1.0e6f);
      d = (int)c;
      dur[base + t] = d;
    }
    int s = d;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int n = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += n;
    }
    if (t < len) cum[base + t] = (int)(carry + s);
    carry += __shfl_sync(0xffffffffu, s, 31);  // one chunk: at most 32e6
  }
  if (lane == 0) ylen[b] = (int)min(max(carry, 1LL), (long long)INT_MAX);
}

__global__ void durations_kernel(const float* logw_dp, const float* z_sdp, const float* sdp_ratio, const float* length_scale,
                                 float* w_out, int* dur, int* cum, int* ylen, Segs seg) {
  durations_body<false>(logw_dp, z_sdp, sdp_ratio, length_scale, nullptr, nullptr, w_out, dur, cum, ylen, seg);
}

__global__ void durations_given_kernel(const float* logw_dp, const float* z_sdp, const float* sdp_ratio, const float* length_scale,
                                       const int* given, const int* given_flag, float* w_out, int* dur, int* cum, int* ylen, Segs seg) {
  durations_body<true>(logw_dp, z_sdp, sdp_ratio, length_scale, given, given_flag, w_out, dur, cum, ylen, seg);
}

__global__ void expand_kernel(float* z_p, int* frame2ph, const float* stats, const int* cum, const float* eps,
                              const float* noise_scale, int C, Segs xseg, Segs yseg) {
  int b = blockIdx.y, j = blockIdx.x;
  if (j >= yseg.len[b]) return;
  int xb = xseg.start[b], xl = xseg.len[b];
  const int* cb = cum + xb;
  // upper_bound: first i with cum[i] > j
  int lo = 0, hi = xl;
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (cb[mid] <= j) lo = mid + 1;
    else hi = mid;
  }
  int i = lo;  // == xl when j is beyond the total (only when total == 0)
  size_t yrow = (size_t)yseg.start[b] + j;
  if (threadIdx.x == 0) frame2ph[yrow] = (i < xl) ? i : -1;
  float ns = noise_scale[b];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float m = 0.f, logs = 0.f;
    if (i < xl) {
      m = stats[(size_t)(xb + i) * 2 * C + c];
      logs = stats[(size_t)(xb + i) * 2 * C + C + c];
    }
    float e = eps[yrow * C + c];
    z_p[yrow * C + c] = __fadd_rn(m, __fmul_rn(__fmul_rn(e, expf(logs)), ns));
  }
}

// Philox4x32-10 + Box-Muller
__device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
  uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
  uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
  c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

__global__ void randn_kernel(float* out, int64_t n, uint64_t seed, uint64_t offset) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
  int64_t e0 = i * 4;
  if (e0 >= n) return;
  uint64_t ctr = offset + (uint64_t)i;
  uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0x5bd1e995u, c3 = 0x2545F491u;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c0, c1, c2, c3, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  const float two_pi = 6.283185307179586f;
  float u0 = ((float)c0 + 1.0f) * 2.3283064365386963e-10f, u1 = (float)c1 * 2.3283064365386963e-10f;
  float u2 = ((float)c2 + 1.0f) * 2.3283064365386963e-10f, u3 = (float)c3 * 2.3283064365386963e-10f;
  float r0 = sqrtf(-2.f * logf(u0)), r1 = sqrtf(-2.f * logf(u2));
  float v[4] = {r0 * cosf(two_pi * u1), r0 * sinf(two_pi * u1), r1 * cosf(two_pi * u3), r1 * sinf(two_pi * u3)};
  for (int q = 0; q < 4; ++q)
    if (e0 + q < n) out[e0 + q] = v[q];
}

// ---------------------------------------------------------------------------------------------
// flow helpers
// ---------------------------------------------------------------------------------------------
__global__ void flip_channels_kernel(float* out, const float* in, int C, int64_t rows) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * C) return;
  int64_t r = i / C;
  int c = (int)(i % C);
  out[i] = in[r * C + (C - 1 - c)];
}

__global__ void coupling_sub_kernel(float* z, const float* m, int C, int64_t rows) {
  int H = C / 2;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * H) return;
  int64_t r = i / H;
  int c = (int)(i % H);
  z[r * C + H + c] -= m[i];
}

__global__ void wn_gate_kernel(float* acts, const float* a, const float* g, int g_ld, int goff, int H, Segs seg) {
  int b = blockIdx.y, t = blockIdx.x;
  if (t >= seg.len[b]) return;
  size_t row = (size_t)seg.start[b] + t;
  const float* gb = g + (size_t)b * g_ld + goff;
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    float ta = a[row * 2 * H + c] + gb[c];
    float sa = a[row * 2 * H + H + c] + gb[H + c];
    acts[row * H + c] = tanhf(ta) * (1.f / (1.f + expf(-sa)));
  }
}

__global__ void wn_res_skip_kernel(float* x, float* skip, const float* rs, int H, int last, int first, int64_t rows) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * H) return;
  int64_t r = i / H;
  int c = (int)(i % H);
  if (!last) {
    x[i] += rs[r * 2 * H + c];
    float s = rs[r * 2 * H + H + c];
    skip[i] = first ? s : skip[i] + s;
  } else {
    float s = rs[r * H + c];
    skip[i] = first ? s : skip[i] + s;
  }
}

__global__ void dec_post_kernel(float* out, const float* x, const float* w, int C, int k, Segs seg) {
  extern __shared__ float ws[];  // [k][C]
  for (int i = threadIdx.x; i < C * k; i += blockDim.x) {
    int c = i / k, j = i % k;
    ws[j * C + c] = w[i];  // weight [1][C][k]
  }
  __syncthreads();
  int b = blockIdx.y;
  int len = seg.len[b];
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= len) return;
  size_t base = seg.start[b];
  int pad = (k - 1) / 2;
  float acc = 0.f;
  for (int j = 0; j < k; ++j) {
    int tt = t + j - pad;
    if (tt < 0 || tt >= len) continue;
    const float* row = x + (base + tt) * C;
    for (int c = 0; c < C; ++c) {
      float v = row[c];
      v = v > 0.f ? v : v * 0.01f;
      acc = fmaf(ws[j * C + c], v, acc);
    }
  }
  out[base + t] = tanhf(acc);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// launch wrappers
// ---------------------------------------------------------------------------------------------
#define POST_LAUNCH(ctx)           \
  do {                             \
    CUDA_CHECK(cudaGetLastError()); \
    (ctx).count();                 \
  } while (0)

void launch_conv(const LaunchCtx& ctx, const ConvArgs& a) {
  if (a.seg.n <= 0 || a.seg.max_len <= 0) return;
  if (a.seg.vectors && a.taps == 1 && a.off == 0) {  // per-utterance conditioning vectors
    dim3 grid((a.cout + 31) / 32, a.seg.max_len, a.seg.n);
    utt_linear_kernel<<<grid, 256, 0, ctx.stream>>>(a);
    POST_LAUNCH(ctx);
    return;
  }
  dim3 grid((a.seg.max_len + CT - 1) / CT, (a.cout + CN - 1) / CN, a.seg.n);
  const bool vec = a.cin % 4 == 0 && a.cout % 4 == 0 && a.in_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(a.in) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(a.w) & 15) == 0;
  if (vec) conv_kernel<true><<<grid, 256, 0, ctx.stream>>>(a);
  else conv_kernel<false><<<grid, 256, 0, ctx.stream>>>(a);
  POST_LAUNCH(ctx);
}

void launch_cm_to_rm(const LaunchCtx& ctx, const float* src, const int64_t* src_off, const int* src_ld, float* dst, int C, const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  dim3 grid((seg.max_len + 31) / 32, (C + 31) / 32, seg.n);
  cm_to_rm_kernel<<<grid, dim3(32, 8), 0, ctx.stream>>>(src, src_off, src_ld, dst, C, seg);
  POST_LAUNCH(ctx);
}

void launch_rm_to_cm(const LaunchCtx& ctx, const float* src, float* dst, const int64_t* dst_off, int C, const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  dim3 grid((seg.max_len + 31) / 32, (C + 31) / 32, seg.n);
  rm_to_cm_kernel<<<grid, dim3(32, 8), 0, ctx.stream>>>(src, dst, dst_off, C, seg);
  POST_LAUNCH(ctx);
}

void launch_embed_combine(const LaunchCtx& ctx, float* h, const int* x, const int* tone, const int* lang, const float* emb,
                          const float* tone_emb, const float* lang_emb, const float* style_emb, int C, int n_vocab,
                          int n_tones, int n_lang, const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  dim3 grid(seg.max_len, seg.n);
  embed_combine_kernel<<<grid, 64, 0, ctx.stream>>>(h, x, tone, lang, emb, tone_emb, lang_emb, style_emb, C, n_vocab,
                                                    n_tones, n_lang, seg, sqrtf((float)C));
  POST_LAUNCH(ctx);
}

void launch_gather_rows(const LaunchCtx& ctx, float* out, const float* table, const int64_t* idx, int n, int C, int n_rows) {
  if (n <= 0) return;
  gather_rows_kernel<<<n, 128, 0, ctx.stream>>>(out, table, idx, n, C, n_rows);
  POST_LAUNCH(ctx);
}

void launch_gather_rows_blend(const LaunchCtx& ctx, float* out, const float* table, const int64_t* idx, const int* slot, const float* mean,
                              const float2* coef, int n, int C, int n_rows, int n_slots) {
  if (n <= 0) return;
  const bool vec = C % 4 == 0 && ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(table) | reinterpret_cast<uintptr_t>(mean)) & 15) == 0;
  if (vec) gather_rows_blend_kernel<true><<<n, 128, 0, ctx.stream>>>(out, table, idx, slot, mean, coef, C, n_rows, n_slots);
  else gather_rows_blend_kernel<false><<<n, 128, 0, ctx.stream>>>(out, table, idx, slot, mean, coef, C, n_rows, n_slots);
  POST_LAUNCH(ctx);
}

void launch_add_utt_vec(const LaunchCtx& ctx, float* out, const float* x, const float* v, int C, int v_ld, const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  dim3 grid(seg.max_len, seg.n);
  add_utt_vec_kernel<<<grid, 64, 0, ctx.stream>>>(out, x, v, C, v_ld, seg);
  POST_LAUNCH(ctx);
}

// Wide rows (C a multiple of 128, e.g. DeBERTa's 1024): one warp per row, NV float4 per lane, every load of the row issued
// before the first use.  The scalar kernel's conditional loads were consumed one by one, i.e. one memory round trip per
// 32 channels — 35-41 us for a 7-row LayerNorm of 1024 channels (profiles/r2_launches_bert_exact_s7.csv).
template <int NV>
__global__ void layernorm_vec_kernel(float* out, const float* a, const float* addin, const float* res, const float* gamma,
                                     const float* beta, float eps, int act, int rows) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  constexpr int C = NV * 128;
  const size_t base = (size_t)warp * C;
  float4 v[NV], w[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(a + base + (i * 32 + lane) * 4);
  if (addin) {
#pragma unroll
    for (int i = 0; i < NV; ++i) w[i] = *reinterpret_cast<const float4*>(addin + base + (i * 32 + lane) * 4);
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = make_float4(v[i].x + w[i].x, v[i].y + w[i].y, v[i].z + w[i].z, v[i].w + w[i].w);
  }
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
    sq += (dx * dx + dy * dy) + (dz * dz + dw * dw);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = 1.0f / sqrtf(sq / (float)C + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 4;
    const float4 g = *reinterpret_cast<const float4*>(gamma + c), bt = *reinterpret_cast<const float4*>(beta + c);
    float4 y = make_float4(apply_act((v[i].x - mean) * rstd * g.x + bt.x, act), apply_act((v[i].y - mean) * rstd * g.y + bt.y, act),
                           apply_act((v[i].z - mean) * rstd * g.z + bt.z, act), apply_act((v[i].w - mean) * rstd * g.w + bt.w, act));
    if (res) {
      const float4 r = *reinterpret_cast<const float4*>(res + base + c);
      y = make_float4(y.x + r.x, y.y + r.y, y.z + r.z, y.w + r.w);
    }
    *reinterpret_cast<float4*>(out + base + c) = y;
  }
}

void launch_layernorm(const LaunchCtx& ctx, float* out, const float* a, const float* addin, const float* res,
                      const float* gamma, const float* beta, float eps, int act, int C, int rows) {
  if (rows <= 0) return;
  int blocks = (rows + 7) / 8;  // 8 warps per block
  if (C == 1024) {
    layernorm_vec_kernel<8><<<blocks, 256, 0, ctx.stream>>>(out, a, addin, res, gamma, beta, eps, act, rows);
    POST_LAUNCH(ctx);
    return;
  }
  if (C == 512 || C == 768) {
    if (C == 512) layernorm_vec_kernel<4><<<blocks, 256, 0, ctx.stream>>>(out, a, addin, res, gamma, beta, eps, act, rows);
    else layernorm_vec_kernel<6><<<blocks, 256, 0, ctx.stream>>>(out, a, addin, res, gamma, beta, eps, act, rows);
    POST_LAUNCH(ctx);
    return;
  }
  if (C <= 256) layernorm_kernel<8><<<blocks, 256, 0, ctx.stream>>>(out, a, addin, res, gamma, beta, eps, act, C, rows);
  else if (C <= 1024) layernorm_kernel<32><<<blocks, 256, 0, ctx.stream>>>(out, a, addin, res, gamma, beta, eps, act, C, rows);
  else fail(SBV2_ERR_UNSUPPORTED, "layernorm: C > 1024");
  POST_LAUNCH(ctx);
}

void launch_rel_attention(const LaunchCtx& ctx, float* out, const float* qkv, const float* rel_k, const float* rel_v,
                          int heads, int head_dim, int window, const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  if (head_dim != 96) fail(SBV2_ERR_UNSUPPORTED, "rel_attention: head_dim must be 96");
  constexpr int D = 96;
  int R = 2 * window + 1;
  auto smem_for = [&](int aq) { return sizeof(float) * (size_t)(D * (aq + 1) + D * (AK + 1) + AK * D + aq * (AK + 1) + 2 * R * D + aq * R); };
  static PerDeviceOnce attr_once;
  attr_once.run([&] {
    CUDA_CHECK(cudaFuncSetAttribute(rel_attention_kernel<D, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    CUDA_CHECK(cudaFuncSetAttribute(rel_attention_kernel<D, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  });
  static const int force_rq = [] { const char* e = getenv("SBV2_B200_TEXT_ATTN_RQ"); return e ? atoi(e) : 0; }();  // test hook
  if (force_rq == 1 || (force_rq == 0 && (long long)seg.max_len * seg.n <= 1024)) {  // few phoneme rows: 16-query CTAs
    dim3 grid((seg.max_len + 15) / 16, heads, seg.n);
    rel_attention_kernel<D, 1><<<grid, 256, smem_for(16), ctx.stream>>>(out, qkv, rel_k, rel_v, heads, window, seg);
  } else {
    dim3 grid((seg.max_len + 63) / 64, heads, seg.n);
    rel_attention_kernel<D, 4><<<grid, 256, smem_for(64), ctx.stream>>>(out, qkv, rel_k, rel_v, heads, window, seg);
  }
  POST_LAUNCH(ctx);
}

void launch_dwconv3(const LaunchCtx& ctx, float* out, const float* in, const float* w, const float* bias, int C, int dil,
                    const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  dim3 grid(seg.max_len, seg.n);
  dwconv3_kernel<<<grid, 64, 0, ctx.stream>>>(out, in, w, bias, C, dil, seg);
  POST_LAUNCH(ctx);
}

void launch_sdp_init(const LaunchCtx& ctx, float* z, const float* noise_rm, const float* nsw, const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  dim3 grid((seg.max_len + 127) / 128, seg.n);
  sdp_init_kernel<<<grid, 128, 0, ctx.stream>>>(z, noise_rm, nsw, seg);
  POST_LAUNCH(ctx);
}

void launch_sdp_flip(const LaunchCtx& ctx, float* z, int rows) {
  if (rows <= 0) return;
  sdp_flip_kernel<<<(rows + 127) / 128, 128, 0, ctx.stream>>>(z, rows);
  POST_LAUNCH(ctx);
}

void launch_convflow_pre(const LaunchCtx& ctx, float* h, const float* z, const float* w, const float* b, const float* g,
                         int C, int rows) {
  if (rows <= 0) return;
  convflow_pre_kernel<<<rows, 64, 0, ctx.stream>>>(h, z, w, b, g, C, rows);
  POST_LAUNCH(ctx);
}

void launch_convflow_spline(const LaunchCtx& ctx, float* z, const float* proj, int ld, int num_bins, float tail_bound,
                            float inv_sqrt_filter, int rows) {
  if (rows <= 0) return;
  if (num_bins != 10) fail(SBV2_ERR_UNSUPPORTED, "ConvFlow: num_bins must be 10");
  convflow_spline_kernel<10><<<(rows + 63) / 64, 64, 0, ctx.stream>>>(z, proj, ld, tail_bound, inv_sqrt_filter, rows);
  POST_LAUNCH(ctx);
}

void launch_sdp_affine(const LaunchCtx& ctx, float* z, const float* m, const float* logs, int rows) {
  if (rows <= 0) return;
  sdp_affine_kernel<<<(rows + 127) / 128, 128, 0, ctx.stream>>>(z, m, logs, rows);
  POST_LAUNCH(ctx);
}

void launch_durations(const LaunchCtx& ctx, const float* logw_dp, const float* z_sdp, const float* sdp_ratio_utt,
                      const float* length_scale_utt, float* w_out, int* dur, int* cum, int* ylen, const Segs& seg) {
  if (seg.n <= 0) return;
  durations_kernel<<<seg.n, 32, 0, ctx.stream>>>(logw_dp, z_sdp, sdp_ratio_utt, length_scale_utt, w_out, dur, cum, ylen, seg);
  POST_LAUNCH(ctx);
}

void launch_durations_given(const LaunchCtx& ctx, const float* logw_dp, const float* z_sdp, const float* sdp_ratio_utt,
                            const float* length_scale_utt, const int* given, const int* given_flag, float* w_out, int* dur, int* cum,
                            int* ylen, const Segs& seg) {
  if (seg.n <= 0) return;
  durations_given_kernel<<<seg.n, 32, 0, ctx.stream>>>(logw_dp, z_sdp, sdp_ratio_utt, length_scale_utt, given, given_flag, w_out, dur,
                                                       cum, ylen, seg);
  POST_LAUNCH(ctx);
}

void launch_expand(const LaunchCtx& ctx, float* z_p, int* frame2ph, const float* stats, const int* cum, const float* eps_rm,
                   const float* noise_scale_utt, int C, const Segs& xseg, const Segs& yseg) {
  if (yseg.n <= 0 || yseg.max_len <= 0) return;
  dim3 grid(yseg.max_len, yseg.n);
  expand_kernel<<<grid, 64, 0, ctx.stream>>>(z_p, frame2ph, stats, cum, eps_rm, noise_scale_utt, C, xseg, yseg);
  POST_LAUNCH(ctx);
}

void launch_randn(const LaunchCtx& ctx, float* out, int64_t n, uint64_t seed, uint64_t offset) {
  if (n <= 0) return;
  int64_t threads = (n + 3) / 4;
  randn_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, ctx.stream>>>(out, n, seed, offset);
  POST_LAUNCH(ctx);
}

void launch_flip_channels(const LaunchCtx& ctx, float* out, const float* in, int C, int64_t rows) {
  if (rows <= 0) return;
  int64_t n = rows * C;
  flip_channels_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx.stream>>>(out, in, C, rows);
  POST_LAUNCH(ctx);
}

void launch_coupling_sub(const LaunchCtx& ctx, float* z, const float* m, int C, int64_t rows) {
  if (rows <= 0) return;
  int64_t n = rows * (C / 2);
  coupling_sub_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx.stream>>>(z, m, C, rows);
  POST_LAUNCH(ctx);
}

void launch_wn_gate(const LaunchCtx& ctx, float* acts, const float* a, const float* g_utt, int g_ld, int goff, int H,
                    const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  dim3 grid(seg.max_len, seg.n);
  wn_gate_kernel<<<grid, 64, 0, ctx.stream>>>(acts, a, g_utt, g_ld, goff, H, seg);
  POST_LAUNCH(ctx);
}

void launch_wn_res_skip(const LaunchCtx& ctx, float* x, float* skip, const float* rs, int H, int last, int first,
                        int64_t rows) {
  if (rows <= 0) return;
  int64_t n = rows * H;
  wn_res_skip_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx.stream>>>(x, skip, rs, H, last, first, rows);
  POST_LAUNCH(ctx);
}

void launch_dec_post(const LaunchCtx& ctx, float* out, const float* x, const float* w, int C, int k, const Segs& seg) {
  if (seg.n <= 0 || seg.max_len <= 0) return;
  dim3 grid((seg.max_len + 255) / 256, seg.n);
  dec_post_kernel<<<grid, 256, sizeof(float) * C * k, ctx.stream>>>(out, x, w, C, k, seg);
  POST_LAUNCH(ctx);
}

}  // namespace sbv2
