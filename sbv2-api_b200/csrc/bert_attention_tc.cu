// DeBERTa-v2 disentangled attention on tcgen05 tensor cores: one query tile and one key tile per (utterance, head) for
// sequences of at most 128 tokens, 128 x 128 tile pairs with an online softmax beyond (the multi-tile kernels below).
//
//   score[i][j] = (Q_i.K_j + Q_i.posK[b(i-j)] + K_j.posQ[b(i-j)]) / sqrt(3 D),   out = softmax(score) V
//
// For |i - j| <= 127 the log-bucket map b() of HF `make_log_bucket_position` is linear (b = i - j + span, checked on the
// host), so the two bias terms are windows of two dense products against 256 consecutive position rows:
//   C2P = Q posK_win^T  [128 x 256]     c2p(i, j) = C2P[i][i - j + 127]
//   P2C = K posQ_win^T  [128 x 256]     p2c(i, j) = P2C[j][i - j + 127]
// Both run as N = 256 MMAs into TMEM.  Their diagonal windows cannot be read from TMEM directly (a tcgen05.ld addresses
// the same columns for every lane), so each thread copies the 128 entries of its row that are needed into a skewed
// fp16 tile in shared memory — C2P as [i][127 - j], P2C transposed as [i][j] — and the softmax then reads plain rows.
// P (unnormalised, fp16) goes back to shared memory as the A operand of O = P V; the row sums divide O in the epilogue.
// oracle: oracle/deberta.py (HF DebertaV2Model, DisentangledSelfAttention).
#include <cuda_fp16.h>
#include <math_constants.h>

#include <cassert>

#include "kernels.h"

namespace sbv2 {
namespace {

constexpr int T = 128, D = 64, DPL = D / 8, W = 256;     // tile, head dim, planes per head, position window
constexpr uint32_t QKV_BYTES = DPL * T * 16;              // 16 KB per Q / K / V tile
constexpr uint32_t POS_BYTES = DPL * W * 16;              // 32 KB per position window
constexpr uint32_t P_BYTES = (T / 8) * T * 16;            // 32 KB
constexpr int PCS = T + 2;                                // skewed bias tiles: row pitch in halfs
constexpr uint32_t SKEW_BYTES = T * PCS * 2;              // 33 280 B each
constexpr int TM_S = 0, TM_B = 128, TM_O = 384, TM_COLS = 512;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity), "r"(0x989680u)  // suspend-time hint (ns): a waiting warp sleeps in hardware instead of re-polling
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_ld1(uint32_t taddr, uint32_t& v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 %%rx;\n"
      ".reg .pred %%px;\n"
      "elect.sync %%rx|%%px, %1;\n"
      "@%%px mov.s32 %0, 1;\n"
      "}\n"
      : "+r"(pred)
      : "r"(0xffffffffu));
  return pred;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// no-swizzle descriptor: start (16-B units), LBO, SBO in bytes
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) |
         ((uint64_t)1 << 46);
}
constexpr uint32_t idesc_f16(int n, int b_mn_major) {
  return (1u << 4) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// warps 0..3: one query row (and, while staging P2C, one key row) per thread; warp 4: loads + MMA issue
// pos_k_p / pos_q_p: fp16 [heads][D/8][n_pos][8]; win0: first position row of the window (span - 127)
__global__ void __launch_bounds__(160, 1) deberta_attention_tc_kernel(__half* out, const __half* qkv, const __half* pos_k_p,
                                                                      const __half* pos_q_p, int n_pos, int win0, int heads,
                                                                      PlanarSegs s) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int h = blockIdx.x, b = blockIdx.y;
  const int len = s.len[b];
  if (len <= 0) return;
  const long long pbase = s.pstart[b];

  const uint32_t sQ = smem_u32(smem);
  const uint32_t sK = sQ + QKV_BYTES, sV = sK + QKV_BYTES, sPK = sV + QKV_BYTES, sPQ = sPK + POS_BYTES, sP = sPQ + POS_BYTES;
  const uint32_t sC = sP + P_BYTES, sDd = sC + SKEW_BYTES, sBar = sDd + SKEW_BYTES;
  const uint32_t bar_load = sBar, bar_s1 = sBar + 8, bar_c = sBar + 16, bar_s2 = sBar + 24, bar_p = sBar + 32, bar_o = sBar + 40;
  const uint32_t tmem_slot = sBar + 48;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + (tmem_slot - sQ));
  __half* Cs = reinterpret_cast<__half*>(smem + (sC - sQ));   // c2p(i, j) at [i][127 - j]
  __half* Ds = reinterpret_cast<__half*>(smem + (sDd - sQ));  // p2c(i, j) at [i][j]

  if (threadIdx.x == 0) {
    mbar_init(bar_load, 1);
    mbar_init(bar_s1, 1);
    mbar_init(bar_c, 128);
    mbar_init(bar_s2, 1);
    mbar_init(bar_p, 128);
    mbar_init(bar_o, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;

  const int q_plane0 = h * DPL, k_plane0 = heads * DPL + h * DPL, v_plane0 = 2 * heads * DPL + h * DPL;

  if (warp == 4) {
    // ---------------- control warp: loads and MMA issue ----------------
    if (lane == 0) mbar_expect_tx(bar_load, 3 * QKV_BYTES + 2 * POS_BYTES);
    __syncwarp();
    if (lane < DPL) {
      const size_t row8 = (size_t)pbase * 8;
      bulk_g2s(sQ + lane * T * 16, qkv + (size_t)(q_plane0 + lane) * s.plane_stride + row8, T * 16, bar_load);
      bulk_g2s(sK + lane * T * 16, qkv + (size_t)(k_plane0 + lane) * s.plane_stride + row8, T * 16, bar_load);
      bulk_g2s(sV + lane * T * 16, qkv + (size_t)(v_plane0 + lane) * s.plane_stride + row8, T * 16, bar_load);
    } else if (lane < 2 * DPL) {
      const int pl = lane - DPL;
      bulk_g2s(sPK + pl * W * 16, pos_k_p + ((size_t)(h * DPL + pl) * n_pos + win0) * 8, W * 16, bar_load);
    } else if (lane < 3 * DPL) {
      const int pl = lane - 2 * DPL;
      bulk_g2s(sPQ + pl * W * 16, pos_q_p + ((size_t)(h * DPL + pl) * n_pos + win0) * 8, W * 16, bar_load);
    }
    __syncwarp();
    mbar_wait(bar_load, 0);
    tc_fence_after();
    const uint64_t dq = make_desc(sQ, T * 16, 128), dk = make_desc(sK, T * 16, 128);
    const uint64_t dpk = make_desc(sPK, W * 16, 128), dpq = make_desc(sPQ, W * 16, 128);
    const uint64_t dp = make_desc(sP, T * 16, 128);
    const uint64_t dv = make_desc(sV, 128, T * 16);  // MN-major B: SBO = next 8-column plane, LBO = next 8 K rows
    constexpr uint32_t ID_S = idesc_f16(T, 0), ID_B = idesc_f16(W, 0), ID_O = idesc_f16(D, 1);
    if (elect_one_sync()) {
#pragma unroll
      for (int k = 0; k < D / 16; ++k) tc_mma_f16(tmem + TM_S, dq + (uint64_t)(k * 2 * T), dk + (uint64_t)(k * 2 * T), ID_S, k > 0 ? 1u : 0u);
#pragma unroll
      for (int k = 0; k < D / 16; ++k) tc_mma_f16(tmem + TM_B, dq + (uint64_t)(k * 2 * T), dpk + (uint64_t)(k * 2 * W), ID_B, k > 0 ? 1u : 0u);
      tc_commit(bar_s1);
    }
    __syncwarp();
    mbar_wait(bar_c, 0);  // C2P has been copied out of TMEM
    tc_fence_after();
    if (elect_one_sync()) {
#pragma unroll
      for (int k = 0; k < D / 16; ++k) tc_mma_f16(tmem + TM_B, dk + (uint64_t)(k * 2 * T), dpq + (uint64_t)(k * 2 * W), ID_B, k > 0 ? 1u : 0u);
      tc_commit(bar_s2);
    }
    __syncwarp();
    mbar_wait(bar_p, 0);  // P tile (and the zeroed V rows) visible to the async proxy
    tc_fence_after();
    if (elect_one_sync()) {
#pragma unroll
      for (int k = 0; k < T / 16; ++k) tc_mma_f16(tmem + TM_O, dp + (uint64_t)(k * 2 * T), dv + (uint64_t)(k * 16), ID_O, k > 0 ? 1u : 0u);
      tc_commit(bar_o);
    }
    __syncwarp();
  } else {
    // ---------------- softmax threads ----------------
    const int row = warp * 32 + lane;  // query row i; also key row j while staging P2C
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    const float c_scale = 1.4426950408889634f / sqrtf(3.0f * (float)D);  // log2(e) / sqrt(3 d)
    // rows of V past the utterance must be finite (they meet P = 0): the buffer tail is not written by anyone
    mbar_wait(bar_load, 0);
    if (row >= len) {
      const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int pl = 0; pl < DPL; ++pl) *reinterpret_cast<uint4*>(smem + (sV - sQ) + (size_t)(pl * T + row) * 16) = z;
    }
    // C2P: keep columns c = i - j + 127, j in [0, 127], at Cs[i][c - i]
    mbar_wait(bar_s1, 0);
    tc_fence_after();
#pragma unroll 1
    for (int q = 0; q < W / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_B + q * 32, v);
      tc_wait_ld();
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int jj = q * 32 + e - row;  // 127 - j
        if (jj >= 0 && jj < T) Cs[row * PCS + jj] = __float2half_rn(__uint_as_float(v[e]));
      }
    }
    tc_fence_before();
    mbar_arrive(bar_c);
    // P2C: thread = key row j; entry for query i = c + j - 127 goes to Ds[i][j]
    mbar_wait(bar_s2, 0);
    tc_fence_after();
#pragma unroll 1
    for (int q = 0; q < W / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_B + q * 32, v);
      tc_wait_ld();
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int ii = q * 32 + e + row - (T - 1);
        if (ii >= 0 && ii < T) Ds[ii * PCS + row] = __float2half_rn(__uint_as_float(v[e]));
      }
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");  // all of Ds (and Cs) written
    // pass 1: row maximum
    const __half* crow = Cs + row * PCS;
    const __half* drow = Ds + row * PCS;
    float m = -CUDART_INF_F;
#pragma unroll 1
    for (int q = 0; q < T / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_S + q * 32, v);
      tc_wait_ld();
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int j = q * 32 + e;
        const float sc = __uint_as_float(v[e]) + __half2float(crow[T - 1 - j]) + __half2float(drow[j]);
        m = fmaxf(m, j < len ? sc : -CUDART_INF_F);
      }
    }
    // pass 2: p = 2^((s - m) * c), unnormalised, fp16 into the P tile; row sum in fp32
    float l = 0.f;
    uint8_t* prow = smem + (sP - sQ) + row * 16;
    const float mc = m * c_scale;
#pragma unroll 1
    for (int q = 0; q < T / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_S + q * 32, v);
      tc_wait_ld();
      float pv[32];
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int j = q * 32 + e;
        const float sc = __uint_as_float(v[e]) + __half2float(crow[T - 1 - j]) + __half2float(drow[j]);
        const float p = j < len ? ex2_approx(fmaf(sc, c_scale, -mc)) : 0.f;
        pv[e] = p;
        l += p;
      }
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 u;
        __half2* uh = reinterpret_cast<__half2*>(&u);
#pragma unroll
        for (int e = 0; e < 4; ++e) uh[e] = __floats2half2_rn(pv[g * 8 + 2 * e], pv[g * 8 + 2 * e + 1]);
        *reinterpret_cast<uint4*>(prow + (size_t)(q * 4 + g) * T * 16) = u;
      }
    }
    tc_fence_before();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // P and V-row writes -> visible to the MMA's async proxy
    mbar_arrive(bar_p);
    // epilogue: O / l -> fp16 planar ctx
    mbar_wait(bar_o, 0);
    tc_fence_after();
    const float inv_l = 1.0f / l;
#pragma unroll 1
    for (int q = 0; q < D / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_O + q * 32, v);
      tc_wait_ld();
      if (row < len) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 u;
          __half2* uh = reinterpret_cast<__half2*>(&u);
#pragma unroll
          for (int e = 0; e < 4; ++e)
            uh[e] = __floats2half2_rn(__uint_as_float(v[g * 8 + 2 * e]) * inv_l, __uint_as_float(v[g * 8 + 2 * e + 1]) * inv_l);
          *reinterpret_cast<uint4*>(out + (size_t)(h * DPL + q * 4 + g) * s.plane_stride + (pbase + row) * 8) = u;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)TM_COLS) : "memory");
  }
}


// Multi-tile kernels.  A (query tile, key tile) pair's 256-row window covers rel in [(qt-kt)*T - (T-1), (qt-kt)*T + T].  The
// bucket table saturates at +-max_rel (bert_bucket_table), so when that whole range lies at or beyond one of the bounds
// every window row is the same position row: C2P is one value per query row (Q_i.posK[pr]) and P2C one value per key
// (K_j.posQ[pr]).  Such a FAR pair gathers WF rows instead of W, issues both bias products with N = WF, reads column 0 of
// each, and skips the skewed copies; the scores are then formed with the roundings and order of the generic path, so the
// two paths agree bit for bit.  The class depends only on (qt, kt) and max_rel, the same for the control warp and the
// softmax threads, and every barrier is arrived on and waited for once per key tile on either path.
constexpr int WF = 16;
__device__ __forceinline__ bool far_pair(int qt, int kt, int max_rel) {
  const int d = (qt - kt) * T;
  return d - (T - 1) >= max_rel || d + T <= -max_rel;
}
// position row of window row w of pair (qt, kt)
__device__ __forceinline__ int window_row(const int* bucket_idx, int max_rel, int n_pos, int qt, int kt, int w, bool far) {
  int rel = (qt - kt) * T + w - (T - 1);
  rel = rel < -max_rel ? -max_rel : (rel > max_rel ? max_rel : rel);
  const int pr = bucket_idx[rel + max_rel];
#ifdef SBV2_DEBUG_HOOKS
  assert(pr >= 0 && pr < n_pos);
  if (far) assert(pr == bucket_idx[(qt > kt ? max_rel : -max_rel) + max_rel]);
#endif
  return pr;
}

// Sequences of more than 128 tokens: one CTA per (head, utterance, 128-query tile), key tiles visited in order with an online
// softmax (running maximum / sum per row, O kept in registers and rescaled per key tile).  A (query tile, key tile) pair
// sees 255 consecutive relative positions rel = i - j; beyond |rel| = span / 2 HF's log buckets map several of them to
// one position row, so the two 256-row position windows are GATHERED through bucket_idx (row w = position of
// rel = (qt - kt) * 128 + w - 127) instead of bulk-copied.  With the windows in rel order, the products, the skewed
// copies and the softmax are those of the single-tile kernel.  Far pairs: see far_pair; the P2C column goes to row 0 of Ds.
__global__ void __launch_bounds__(160, 1) deberta_attention_tc_multi_kernel(__half* out, const __half* qkv, const __half* pos_k_p,
                                                                            const __half* pos_q_p, int n_pos, const int* bucket_idx,
                                                                            int max_rel, int heads, bool far_pairs, PlanarSegs s) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int h = blockIdx.x, b = blockIdx.y, qt = blockIdx.z;
  const int len = s.len[b];
  if (qt * T >= len) return;
  const int nk = (len + T - 1) / T;
  const long long pbase = s.pstart[b];

  const uint32_t sQ = smem_u32(smem);
  const uint32_t sK = sQ + QKV_BYTES, sV = sK + QKV_BYTES, sPK = sV + QKV_BYTES, sPQ = sPK + POS_BYTES, sP = sPQ + POS_BYTES;
  const uint32_t sC = sP + P_BYTES, sDd = sC + SKEW_BYTES, sBar = sDd + SKEW_BYTES;
  const uint32_t bar_q = sBar, bar_s1 = sBar + 8, bar_c = sBar + 16, bar_s2 = sBar + 24, bar_p = sBar + 32, bar_o = sBar + 40,
                 bar_kv = sBar + 48, bar_g = sBar + 56;
  const uint32_t tmem_slot = sBar + 64;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + (tmem_slot - sQ));
  __half* Cs = reinterpret_cast<__half*>(smem + (sC - sQ));
  __half* Ds = reinterpret_cast<__half*>(smem + (sDd - sQ));

  if (threadIdx.x == 0) {
    mbar_init(bar_q, 1);
    mbar_init(bar_s1, 1);
    mbar_init(bar_c, 128);
    mbar_init(bar_s2, 1);
    mbar_init(bar_p, 128);
    mbar_init(bar_o, 1);
    mbar_init(bar_kv, 1);
    mbar_init(bar_g, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  const int q_plane0 = h * DPL, k_plane0 = heads * DPL + h * DPL, v_plane0 = 2 * heads * DPL + h * DPL;

  if (warp == 4) {
    // ---------------- control warp: Q / K / V loads and MMA issue ----------------
    if (lane == 0) mbar_expect_tx(bar_q, QKV_BYTES);
    __syncwarp();
    if (lane < DPL) bulk_g2s(sQ + lane * T * 16, qkv + (size_t)(q_plane0 + lane) * s.plane_stride + (size_t)(pbase + qt * T) * 8, T * 16, bar_q);
    const uint64_t dq = make_desc(sQ, T * 16, 128), dk = make_desc(sK, T * 16, 128);
    const uint64_t dpk = make_desc(sPK, W * 16, 128), dpq = make_desc(sPQ, W * 16, 128);
    const uint64_t dp = make_desc(sP, T * 16, 128);
    const uint64_t dv = make_desc(sV, 128, T * 16);
    constexpr uint32_t ID_S = idesc_f16(T, 0), ID_B = idesc_f16(W, 0), ID_BF = idesc_f16(WF, 0), ID_O = idesc_f16(D, 1);
    for (int kt = 0; kt < nk; ++kt) {
      const uint32_t par = kt & 1;
      const uint32_t id_b = far_pairs && far_pair(qt, kt, max_rel) ? ID_BF : ID_B;
      // every MMA of the previous key tile has completed (bar_o below): its K / V tiles can be overwritten
      if (lane == 0) mbar_expect_tx(bar_kv, 2 * QKV_BYTES);
      __syncwarp();
      if (lane < DPL) {
        const size_t row8 = (size_t)(pbase + kt * T) * 8;
        bulk_g2s(sK + lane * T * 16, qkv + (size_t)(k_plane0 + lane) * s.plane_stride + row8, T * 16, bar_kv);
        bulk_g2s(sV + lane * T * 16, qkv + (size_t)(v_plane0 + lane) * s.plane_stride + row8, T * 16, bar_kv);
      }
      __syncwarp();
      if (kt == 0) mbar_wait(bar_q, 0);
      mbar_wait(bar_kv, par);
      mbar_wait(bar_g, par);  // position windows gathered and visible to the async proxy
      tc_fence_after();
      if (elect_one_sync()) {
#pragma unroll
        for (int k = 0; k < D / 16; ++k) tc_mma_f16(tmem + TM_S, dq + (uint64_t)(k * 2 * T), dk + (uint64_t)(k * 2 * T), ID_S, k > 0 ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < D / 16; ++k) tc_mma_f16(tmem + TM_B, dq + (uint64_t)(k * 2 * T), dpk + (uint64_t)(k * 2 * W), id_b, k > 0 ? 1u : 0u);
        tc_commit(bar_s1);
      }
      __syncwarp();
      mbar_wait(bar_c, par);
      tc_fence_after();
      if (elect_one_sync()) {
#pragma unroll
        for (int k = 0; k < D / 16; ++k) tc_mma_f16(tmem + TM_B, dk + (uint64_t)(k * 2 * T), dpq + (uint64_t)(k * 2 * W), id_b, k > 0 ? 1u : 0u);
        tc_commit(bar_s2);
      }
      __syncwarp();
      mbar_wait(bar_p, par);
      tc_fence_after();
      if (elect_one_sync()) {
#pragma unroll
        for (int k = 0; k < T / 16; ++k) tc_mma_f16(tmem + TM_O, dp + (uint64_t)(k * 2 * T), dv + (uint64_t)(k * 16), ID_O, k > 0 ? 1u : 0u);
        tc_commit(bar_o);
      }
      __syncwarp();
      mbar_wait(bar_o, par);
    }
  } else {
    // ---------------- softmax threads ----------------
    const int row = warp * 32 + lane;  // query row within the tile; key row within the tile while staging P2C
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    const float c_scale = 1.4426950408889634f / sqrtf(3.0f * (float)D);
    float m = -CUDART_INF_F, l = 0.f;
    float o[D];
#pragma unroll
    for (int e = 0; e < D; ++e) o[e] = 0.f;
    const __half* crow = Cs + row * PCS;
    const __half* drow = Ds + row * PCS;
    uint8_t* prow = smem + (sP - sQ) + row * 16;
    for (int kt = 0; kt < nk; ++kt) {
      const uint32_t par = kt & 1;
      const int klen = len - kt * T;  // keys of this tile below klen are real
      const bool fr = far_pairs && far_pair(qt, kt, max_rel);
      // position windows of this tile pair (the previous pair's MMAs have completed: bar_o was waited for)
#pragma unroll 1
      for (int w = row; w < (fr ? WF : W); w += T) {
        const int pr = window_row(bucket_idx, max_rel, n_pos, qt, kt, w, fr);
#pragma unroll
        for (int pl = 0; pl < DPL; ++pl) {
          const size_t src = ((size_t)(h * DPL + pl) * n_pos + pr) * 8;
          *reinterpret_cast<uint4*>(smem + (sPK - sQ) + (size_t)(pl * W + w) * 16) = *reinterpret_cast<const uint4*>(pos_k_p + src);
          *reinterpret_cast<uint4*>(smem + (sPQ - sQ) + (size_t)(pl * W + w) * 16) = *reinterpret_cast<const uint4*>(pos_q_p + src);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(bar_g);
      mbar_wait(bar_kv, par);
      if (row >= klen) {
        const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int pl = 0; pl < DPL; ++pl) *reinterpret_cast<uint4*>(smem + (sV - sQ) + (size_t)(pl * T + row) * 16) = z;
      }
      mbar_wait(bar_s1, par);
      tc_fence_after();
      float c_far = 0.f;  // far pair: c2p of this query row, rounded to fp16 as Cs holds it
      if (fr) {
        uint32_t v;
        tc_ld1(lane_addr + TM_B, v);
        tc_wait_ld();
        c_far = __half2float(__float2half_rn(__uint_as_float(v)));
      } else {
#pragma unroll 1
        for (int q = 0; q < W / 32; ++q) {
          uint32_t v[32];
          tc_ld32(lane_addr + TM_B + q * 32, v);
          tc_wait_ld();
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int jj = q * 32 + e - row;
            if (jj >= 0 && jj < T) Cs[row * PCS + jj] = __float2half_rn(__uint_as_float(v[e]));
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar_c);
      mbar_wait(bar_s2, par);
      tc_fence_after();
      if (fr) {
        uint32_t v;
        tc_ld1(lane_addr + TM_B, v);
        tc_wait_ld();
        Ds[row] = __float2half_rn(__uint_as_float(v));  // p2c of key `row`, the same for every query
      } else {
#pragma unroll 1
        for (int q = 0; q < W / 32; ++q) {
          uint32_t v[32];
          tc_ld32(lane_addr + TM_B + q * 32, v);
          tc_wait_ld();
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int ii = q * 32 + e + row - (T - 1);
            if (ii >= 0 && ii < T) Ds[ii * PCS + row] = __float2half_rn(__uint_as_float(v[e]));
          }
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const __half* dr = fr ? Ds : drow;
      float mt = -CUDART_INF_F;
#pragma unroll 1
      for (int q = 0; q < T / 32; ++q) {
        uint32_t v[32];
        tc_ld32(lane_addr + TM_S + q * 32, v);
        tc_wait_ld();
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const int j = q * 32 + e;
          const float sc = __uint_as_float(v[e]) + (fr ? c_far : __half2float(crow[T - 1 - j])) + __half2float(dr[j]);
          mt = fmaxf(mt, j < klen ? sc : -CUDART_INF_F);
        }
      }
      const float m_new = fmaxf(m, mt);
      const float mc = m_new * c_scale;
      const float alpha = ex2_approx(fmaf(m, c_scale, -mc));  // 0 on the first tile (m = -inf)
      m = m_new;
      float lt = 0.f;
#pragma unroll 1
      for (int q = 0; q < T / 32; ++q) {
        uint32_t v[32];
        tc_ld32(lane_addr + TM_S + q * 32, v);
        tc_wait_ld();
        float pv[32];
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const int j = q * 32 + e;
          const float sc = __uint_as_float(v[e]) + (fr ? c_far : __half2float(crow[T - 1 - j])) + __half2float(dr[j]);
          const float p = j < klen ? ex2_approx(fmaf(sc, c_scale, -mc)) : 0.f;
          pv[e] = p;
          lt += p;
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 u;
          __half2* uh = reinterpret_cast<__half2*>(&u);
#pragma unroll
          for (int e = 0; e < 4; ++e) uh[e] = __floats2half2_rn(pv[g * 8 + 2 * e], pv[g * 8 + 2 * e + 1]);
          *reinterpret_cast<uint4*>(prow + (size_t)(q * 4 + g) * T * 16) = u;
        }
      }
      l = fmaf(l, alpha, lt);
      tc_fence_before();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(bar_p);
      mbar_wait(bar_o, par);
      tc_fence_after();
#pragma unroll
      for (int q = 0; q < D / 32; ++q) {
        uint32_t v[32];
        tc_ld32(lane_addr + TM_O + q * 32, v);
        tc_wait_ld();
#pragma unroll
        for (int e = 0; e < 32; ++e) o[q * 32 + e] = fmaf(o[q * 32 + e], alpha, __uint_as_float(v[e]));
      }
      tc_fence_before();
    }
    const float inv_l = 1.0f / l;
    const int grow = qt * T + row;
    if (grow < len) {
#pragma unroll
      for (int g = 0; g < DPL; ++g) {
        uint4 u;
        __half2* uh = reinterpret_cast<__half2*>(&u);
#pragma unroll
        for (int e = 0; e < 4; ++e) uh[e] = __floats2half2_rn(o[g * 8 + 2 * e] * inv_l, o[g * 8 + 2 * e + 1] * inv_l);
        *reinterpret_cast<uint4*>(out + (size_t)(h * DPL + g) * s.plane_stride + (pbase + grow) * 8) = u;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)TM_COLS) : "memory");
  }
}


// ---------------------------------------------------------------------------------------------------------------------
// Exact-numerics variant (SBV2_B200_BERT=exact, the default) for sequences of at most 128 tokens: every operand is a
// two-term fp16 split x = h0 + h1 (the plane blocks [h0 | h1 | h0] the split GEMMs exchange), every product is the three
// cross terms h0 g0 + h0 g1 + h1 g0 accumulated in fp32, the position-bias windows go through ONE fp32 shared-memory tile
// (c2p written, p2c added), and the probabilities are split as well before P V.  Replaces the fp32 CUDA-core kernel
// (deberta_attention_kernel<true>) there; measured error against it: see tests/test_gpu_bert.py.
//   qkv_s : split planar [h0 | h1 | h0] x [3 * heads * 8 planes][rows][8], values scaled by sc (power of two)
//   pos_*_s: fp16 [2 terms][heads][8][n_pos][8], scaled by sc
//   out_s : split planar ctx [h0 | h1 | h0] x [heads * 8 planes], scaled by sc (= V's scale: O needs no rescaling)
// Shared memory: six 16 KB operand tiles, one 64 KB buffer (posK terms, then posQ terms, then P terms), the fp32 bias tile.
constexpr int BCS = T + 4;                               // bias tile row pitch (floats): 16-byte row reads, odd * 4 skew
constexpr uint32_t BIAS_BYTES = T * BCS * 4;             // 67 584 B
constexpr uint32_t EX_SMEM = 6 * QKV_BYTES + 2 * POS_BYTES + BIAS_BYTES + 128;

__global__ void __launch_bounds__(160, 1) deberta_attention_tc_exact_kernel(__half* out_s, long long out_blk, const __half* qkv_s,
                                                                            long long qkv_blk, const __half* pos_k_s, const __half* pos_q_s,
                                                                            int n_pos, int win0, int heads, float inv_sc2, PlanarSegs s) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int h = blockIdx.x, b = blockIdx.y;
  const int len = s.len[b];
  if (len <= 0) return;
  const long long pbase = s.pstart[b];

  const uint32_t sQ0 = smem_u32(smem);
  const uint32_t sQ1 = sQ0 + QKV_BYTES, sK0 = sQ1 + QKV_BYTES, sK1 = sK0 + QKV_BYTES, sV0 = sK1 + QKV_BYTES, sV1 = sV0 + QKV_BYTES;
  const uint32_t sW0 = sV1 + QKV_BYTES, sW1 = sW0 + POS_BYTES;  // window terms 0 / 1; later P terms 0 / 1
  const uint32_t sBias = sW1 + POS_BYTES, sBar = sBias + BIAS_BYTES;
  const uint32_t bar_load = sBar, bar_s1 = sBar + 8, bar_c = sBar + 16, bar_s2 = sBar + 24, bar_p = sBar + 32, bar_o = sBar + 40,
                 bar_w2 = sBar + 48;
  const uint32_t tmem_slot = sBar + 56;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + (tmem_slot - sQ0));
  float* Bs = reinterpret_cast<float*>(smem + (sBias - sQ0));  // bias(i, j) = c2p + p2c at [i][j]

  if (threadIdx.x == 0) {
    mbar_init(bar_load, 1);
    mbar_init(bar_s1, 1);
    mbar_init(bar_c, 128);
    mbar_init(bar_s2, 1);
    mbar_init(bar_p, 128);
    mbar_init(bar_o, 1);
    mbar_init(bar_w2, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  const int q_plane0 = h * DPL, k_plane0 = heads * DPL + h * DPL, v_plane0 = 2 * heads * DPL + h * DPL;
  const size_t pos_term = (size_t)heads * DPL * n_pos * 8;  // halves between the two terms of a position table

  if (warp == 4) {
    // ---------------- control warp: loads and MMA issue ----------------
    if (lane == 0) mbar_expect_tx(bar_load, 6 * QKV_BYTES + 2 * POS_BYTES);
    __syncwarp();
    {
      const size_t row8 = (size_t)pbase * 8;
      // 48 operand planes (q / k / v x 2 terms x 8) and 16 window planes over the 32 lanes
      for (int i = lane; i < 48; i += 32) {
        const int which = i / 16, term = (i >> 3) & 1, pl = i & 7;  // which: 0 q, 1 k, 2 v
        const int plane0 = which == 0 ? q_plane0 : (which == 1 ? k_plane0 : v_plane0);
        const uint32_t dst = sQ0 + (uint32_t)(which * 2 + term) * QKV_BYTES + pl * T * 16;
        bulk_g2s(dst, qkv_s + (size_t)term * qkv_blk + (size_t)(plane0 + pl) * s.plane_stride + row8, T * 16, bar_load);
      }
      if (lane < 16) {
        const int term = lane >> 3, pl = lane & 7;
        bulk_g2s(sW0 + term * POS_BYTES + pl * W * 16, pos_k_s + term * pos_term + ((size_t)(h * DPL + pl) * n_pos + win0) * 8, W * 16, bar_load);
      }
    }
    __syncwarp();
    mbar_wait(bar_load, 0);
    tc_fence_after();
    const uint64_t dq0 = make_desc(sQ0, T * 16, 128), dq1 = make_desc(sQ1, T * 16, 128);
    const uint64_t dk0 = make_desc(sK0, T * 16, 128), dk1 = make_desc(sK1, T * 16, 128);
    const uint64_t dw0 = make_desc(sW0, W * 16, 128), dw1 = make_desc(sW1, W * 16, 128);
    const uint64_t dp0 = make_desc(sW0, T * 16, 128), dp1 = make_desc(sW1, T * 16, 128);  // P terms reuse the window buffer
    const uint64_t dv0 = make_desc(sV0, 128, T * 16), dv1 = make_desc(sV1, 128, T * 16);
    constexpr uint32_t ID_S = idesc_f16(T, 0), ID_B = idesc_f16(W, 0), ID_O = idesc_f16(D, 1);
    // three cross terms of a product, K-major x K-major: (a0, b0), (a0, b1), (a1, b0)
    auto cross = [&](uint32_t tm, uint64_t a0, uint64_t a1, uint64_t b0, uint64_t b1, uint32_t astep, uint32_t bstep, uint32_t id, int nk) {
      for (int k = 0; k < nk; ++k) tc_mma_f16(tm, a0 + (uint64_t)(k * astep), b0 + (uint64_t)(k * bstep), id, k > 0 ? 1u : 0u);
      for (int k = 0; k < nk; ++k) tc_mma_f16(tm, a0 + (uint64_t)(k * astep), b1 + (uint64_t)(k * bstep), id, 1u);
      for (int k = 0; k < nk; ++k) tc_mma_f16(tm, a1 + (uint64_t)(k * astep), b0 + (uint64_t)(k * bstep), id, 1u);
    };
    if (elect_one_sync()) {
      cross(tmem + TM_S, dq0, dq1, dk0, dk1, 2 * T, 2 * T, ID_S, D / 16);
      cross(tmem + TM_B, dq0, dq1, dw0, dw1, 2 * T, 2 * W, ID_B, D / 16);
      tc_commit(bar_s1);
    }
    __syncwarp();
    // the posK windows have been consumed once those MMAs complete: fetch the posQ windows into the same buffer
    mbar_wait(bar_s1, 0);
    if (lane == 0) mbar_expect_tx(bar_w2, 2 * POS_BYTES);
    __syncwarp();
    if (lane < 16) {
      const int term = lane >> 3, pl = lane & 7;
      bulk_g2s(sW0 + term * POS_BYTES + pl * W * 16, pos_q_s + term * pos_term + ((size_t)(h * DPL + pl) * n_pos + win0) * 8, W * 16, bar_w2);
    }
    __syncwarp();
    mbar_wait(bar_w2, 0);
    mbar_wait(bar_c, 0);  // C2P has been copied out of TMEM
    tc_fence_after();
    if (elect_one_sync()) {
      cross(tmem + TM_B, dk0, dk1, dw0, dw1, 2 * T, 2 * W, ID_B, D / 16);
      tc_commit(bar_s2);
    }
    __syncwarp();
    mbar_wait(bar_p, 0);  // P terms (and the zeroed V rows) visible to the async proxy
    tc_fence_after();
    if (elect_one_sync()) {
      // O = P0 V0 + P0 V1 + P1 V0: A K-major (P), B MN-major (V)
      for (int k = 0; k < T / 16; ++k) tc_mma_f16(tmem + TM_O, dp0 + (uint64_t)(k * 2 * T), dv0 + (uint64_t)(k * 16), ID_O, k > 0 ? 1u : 0u);
      for (int k = 0; k < T / 16; ++k) tc_mma_f16(tmem + TM_O, dp0 + (uint64_t)(k * 2 * T), dv1 + (uint64_t)(k * 16), ID_O, 1u);
      for (int k = 0; k < T / 16; ++k) tc_mma_f16(tmem + TM_O, dp1 + (uint64_t)(k * 2 * T), dv0 + (uint64_t)(k * 16), ID_O, 1u);
      tc_commit(bar_o);
    }
    __syncwarp();
  } else {
    // ---------------- softmax threads ----------------
    const int row = warp * 32 + lane;  // query row i; also key row j while staging P2C
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    const float c_scale = 1.4426950408889634f / sqrtf(3.0f * (float)D) * inv_sc2;  // log2(e) / sqrt(3 d), operands carry sc each
    mbar_wait(bar_load, 0);
    if (row >= len) {
      const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int pl = 0; pl < DPL; ++pl) {
        *reinterpret_cast<uint4*>(smem + (sV0 - sQ0) + (size_t)(pl * T + row) * 16) = z;
        *reinterpret_cast<uint4*>(smem + (sV1 - sQ0) + (size_t)(pl * T + row) * 16) = z;
      }
    }
    // C2P: column c = i - j + 127 of row i goes to Bs[i][j], j = i + 127 - c
    mbar_wait(bar_s1, 0);
    tc_fence_after();
#pragma unroll 1
    for (int q = 0; q < W / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_B + q * 32, v);
      tc_wait_ld();
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int j = row + (T - 1) - (q * 32 + e);
        if (j >= 0 && j < T) Bs[row * BCS + j] = __uint_as_float(v[e]);
      }
    }
    tc_fence_before();
    mbar_arrive(bar_c);
    asm volatile("bar.sync 1, 128;" ::: "memory");  // every c2p entry is written before any p2c entry is added
    // P2C: thread = key row j; column c belongs to query i = c + j - 127: Bs[i][j] += it
    mbar_wait(bar_s2, 0);
    tc_fence_after();
#pragma unroll 1
    for (int q = 0; q < W / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_B + q * 32, v);
      tc_wait_ld();
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int ii = q * 32 + e + row - (T - 1);
        if (ii >= 0 && ii < T) Bs[ii * BCS + row] += __uint_as_float(v[e]);
      }
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    // pass 1: row maximum of s = S + bias
    const float* brow = Bs + row * BCS;
    float m = -CUDART_INF_F;
#pragma unroll 1
    for (int q = 0; q < T / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_S + q * 32, v);
      tc_wait_ld();
#pragma unroll
      for (int e4 = 0; e4 < 8; ++e4) {
        const float4 bb = *reinterpret_cast<const float4*>(brow + q * 32 + 4 * e4);
        const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = q * 32 + 4 * e4 + u;
          const float sc = __uint_as_float(v[4 * e4 + u]) + bv[u];
          m = fmaxf(m, j < len ? sc : -CUDART_INF_F);
        }
      }
    }
    // pass 2: p = 2^((s - m) c), unnormalised; two fp16 terms into the P tiles (the window buffer: the posQ MMAs have completed)
    float l = 0.f;
    uint8_t* prow0 = smem + (sW0 - sQ0) + row * 16;
    uint8_t* prow1 = smem + (sW1 - sQ0) + row * 16;
    const float mc = m * c_scale;
#pragma unroll 1
    for (int q = 0; q < T / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_S + q * 32, v);
      tc_wait_ld();
      float pv[32];
#pragma unroll
      for (int e4 = 0; e4 < 8; ++e4) {
        const float4 bb = *reinterpret_cast<const float4*>(brow + q * 32 + 4 * e4);
        const float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = q * 32 + 4 * e4 + u;
          const float sc = __uint_as_float(v[4 * e4 + u]) + bv[u];
          const float p = j < len ? ex2_approx(fmaf(sc, c_scale, -mc)) : 0.f;
          pv[4 * e4 + u] = p;
          l += p;
        }
      }
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 u0, u1;
        __half2* h0 = reinterpret_cast<__half2*>(&u0);
        __half2* h1 = reinterpret_cast<__half2*>(&u1);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float x0 = pv[g * 8 + 2 * e], x1 = pv[g * 8 + 2 * e + 1];
          const __half2 a = __floats2half2_rn(x0, x1);
          const float2 af = __half22float2(a);
          h0[e] = a;
          h1[e] = __floats2half2_rn(x0 - af.x, x1 - af.y);
        }
        *reinterpret_cast<uint4*>(prow0 + (size_t)(q * 4 + g) * T * 16) = u0;
        *reinterpret_cast<uint4*>(prow1 + (size_t)(q * 4 + g) * T * 16) = u1;
      }
    }
    tc_fence_before();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_arrive(bar_p);
    // epilogue: O / l (carries V's scale sc, the scale of the consuming split GEMM) -> split planar ctx
    mbar_wait(bar_o, 0);
    tc_fence_after();
    const float inv_l = 1.0f / l;
#pragma unroll 1
    for (int q = 0; q < D / 32; ++q) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_O + q * 32, v);
      tc_wait_ld();
      if (row < len) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 u0, u1;
          __half2* h0 = reinterpret_cast<__half2*>(&u0);
          __half2* h1 = reinterpret_cast<__half2*>(&u1);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float x0 = __uint_as_float(v[g * 8 + 2 * e]) * inv_l, x1 = __uint_as_float(v[g * 8 + 2 * e + 1]) * inv_l;
            const __half2 a = __floats2half2_rn(x0, x1);
            const float2 af = __half22float2(a);
            h0[e] = a;
            h1[e] = __floats2half2_rn(x0 - af.x, x1 - af.y);
          }
          __half* dst = out_s + (size_t)(h * DPL + q * 4 + g) * s.plane_stride + (pbase + row) * 8;
          *reinterpret_cast<uint4*>(dst) = u0;
          *reinterpret_cast<uint4*>(dst + out_blk) = u1;
          *reinterpret_cast<uint4*>(dst + 2 * out_blk) = u0;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)TM_COLS) : "memory");
  }
}


// Exact numerics, more than 128 tokens: the tile-pair loop / online softmax / gathered log-bucket windows of
// deberta_attention_tc_multi_kernel with the split operands, fp32 bias tile and split probabilities of
// deberta_attention_tc_exact_kernel.  Per key tile the 64 KB window buffer holds the gathered posK terms, then the gathered
// posQ terms, then the two P terms.  Far pairs (far_pair): c2p stays in a register, the p2c column goes to row 0 of Bs, and
// the bias is fl(c2p + p2c) as the generic path's Bs holds it.
__global__ void __launch_bounds__(160, 1)
    deberta_attention_tc_exact_multi_kernel(__half* out_s, long long out_blk, const __half* qkv_s, long long qkv_blk, const __half* pos_k_s,
                                            const __half* pos_q_s, int n_pos, const int* bucket_idx, int max_rel, int heads, float inv_sc2,
                                            bool far_pairs, PlanarSegs s) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int h = blockIdx.x, b = blockIdx.y, qt = blockIdx.z;
  const int len = s.len[b];
  if (qt * T >= len) return;
  const int nk = (len + T - 1) / T;
  const long long pbase = s.pstart[b];

  const uint32_t sQ0 = smem_u32(smem);
  const uint32_t sQ1 = sQ0 + QKV_BYTES, sK0 = sQ1 + QKV_BYTES, sK1 = sK0 + QKV_BYTES, sV0 = sK1 + QKV_BYTES, sV1 = sV0 + QKV_BYTES;
  const uint32_t sW0 = sV1 + QKV_BYTES, sW1 = sW0 + POS_BYTES;
  const uint32_t sBias = sW1 + POS_BYTES, sBar = sBias + BIAS_BYTES;
  const uint32_t bar_q = sBar, bar_s1 = sBar + 8, bar_g2 = sBar + 16, bar_s2 = sBar + 24, bar_p = sBar + 32, bar_o = sBar + 40,
                 bar_kv = sBar + 48, bar_g1 = sBar + 56;
  const uint32_t tmem_slot = sBar + 64;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + (tmem_slot - sQ0));
  float* Bs = reinterpret_cast<float*>(smem + (sBias - sQ0));

  if (threadIdx.x == 0) {
    mbar_init(bar_q, 1);
    mbar_init(bar_s1, 1);
    mbar_init(bar_g2, 128);
    mbar_init(bar_s2, 1);
    mbar_init(bar_p, 128);
    mbar_init(bar_o, 1);
    mbar_init(bar_kv, 1);
    mbar_init(bar_g1, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  const int q_plane0 = h * DPL, k_plane0 = heads * DPL + h * DPL, v_plane0 = 2 * heads * DPL + h * DPL;
  const size_t pos_term = (size_t)heads * DPL * n_pos * 8;

  if (warp == 4) {
    // ---------------- control warp ----------------
    if (lane == 0) mbar_expect_tx(bar_q, 2 * QKV_BYTES);
    __syncwarp();
    if (lane < 16) {
      const int term = lane >> 3, pl = lane & 7;
      bulk_g2s(sQ0 + term * QKV_BYTES + pl * T * 16,
               qkv_s + (size_t)term * qkv_blk + (size_t)(q_plane0 + pl) * s.plane_stride + (size_t)(pbase + qt * T) * 8, T * 16, bar_q);
    }
    const uint64_t dq0 = make_desc(sQ0, T * 16, 128), dq1 = make_desc(sQ1, T * 16, 128);
    const uint64_t dk0 = make_desc(sK0, T * 16, 128), dk1 = make_desc(sK1, T * 16, 128);
    const uint64_t dw0 = make_desc(sW0, W * 16, 128), dw1 = make_desc(sW1, W * 16, 128);
    const uint64_t dp0 = make_desc(sW0, T * 16, 128), dp1 = make_desc(sW1, T * 16, 128);
    const uint64_t dv0 = make_desc(sV0, 128, T * 16), dv1 = make_desc(sV1, 128, T * 16);
    constexpr uint32_t ID_S = idesc_f16(T, 0), ID_B = idesc_f16(W, 0), ID_BF = idesc_f16(WF, 0), ID_O = idesc_f16(D, 1);
    auto cross = [&](uint32_t tm, uint64_t a0, uint64_t a1, uint64_t b0, uint64_t b1, uint32_t astep, uint32_t bstep, uint32_t id, int nk16) {
      for (int k = 0; k < nk16; ++k) tc_mma_f16(tm, a0 + (uint64_t)(k * astep), b0 + (uint64_t)(k * bstep), id, k > 0 ? 1u : 0u);
      for (int k = 0; k < nk16; ++k) tc_mma_f16(tm, a0 + (uint64_t)(k * astep), b1 + (uint64_t)(k * bstep), id, 1u);
      for (int k = 0; k < nk16; ++k) tc_mma_f16(tm, a1 + (uint64_t)(k * astep), b0 + (uint64_t)(k * bstep), id, 1u);
    };
    for (int kt = 0; kt < nk; ++kt) {
      const uint32_t par = kt & 1;
      const uint32_t id_b = far_pairs && far_pair(qt, kt, max_rel) ? ID_BF : ID_B;
      if (lane == 0) mbar_expect_tx(bar_kv, 4 * QKV_BYTES);
      __syncwarp();
      {
        const int which = lane >> 4, term = (lane >> 3) & 1, pl = lane & 7;  // which: 0 k, 1 v
        const int plane0 = which == 0 ? k_plane0 : v_plane0;
        bulk_g2s(sK0 + (uint32_t)(which * 2 + term) * QKV_BYTES + pl * T * 16,
                 qkv_s + (size_t)term * qkv_blk + (size_t)(plane0 + pl) * s.plane_stride + (size_t)(pbase + kt * T) * 8, T * 16, bar_kv);
      }
      __syncwarp();
      if (kt == 0) mbar_wait(bar_q, 0);
      mbar_wait(bar_kv, par);
      mbar_wait(bar_g1, par);  // posK terms gathered
      tc_fence_after();
      if (elect_one_sync()) {
        cross(tmem + TM_S, dq0, dq1, dk0, dk1, 2 * T, 2 * T, ID_S, D / 16);
        cross(tmem + TM_B, dq0, dq1, dw0, dw1, 2 * T, 2 * W, id_b, D / 16);
        tc_commit(bar_s1);
      }
      __syncwarp();
      mbar_wait(bar_g2, par);  // C2P copied out of TMEM, posQ terms gathered
      tc_fence_after();
      if (elect_one_sync()) {
        cross(tmem + TM_B, dk0, dk1, dw0, dw1, 2 * T, 2 * W, id_b, D / 16);
        tc_commit(bar_s2);
      }
      __syncwarp();
      mbar_wait(bar_p, par);
      tc_fence_after();
      if (elect_one_sync()) {
        for (int k = 0; k < T / 16; ++k) tc_mma_f16(tmem + TM_O, dp0 + (uint64_t)(k * 2 * T), dv0 + (uint64_t)(k * 16), ID_O, k > 0 ? 1u : 0u);
        for (int k = 0; k < T / 16; ++k) tc_mma_f16(tmem + TM_O, dp0 + (uint64_t)(k * 2 * T), dv1 + (uint64_t)(k * 16), ID_O, 1u);
        for (int k = 0; k < T / 16; ++k) tc_mma_f16(tmem + TM_O, dp1 + (uint64_t)(k * 2 * T), dv0 + (uint64_t)(k * 16), ID_O, 1u);
        tc_commit(bar_o);
      }
      __syncwarp();
      mbar_wait(bar_o, par);
    }
  } else {
    // ---------------- softmax threads ----------------
    const int row = warp * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    const float c_scale = 1.4426950408889634f / sqrtf(3.0f * (float)D) * inv_sc2;
    float m = -CUDART_INF_F, l = 0.f;
    float o[D];
#pragma unroll
    for (int e = 0; e < D; ++e) o[e] = 0.f;
    const float* brow = Bs + row * BCS;
    uint8_t* prow0 = smem + (sW0 - sQ0) + row * 16;
    uint8_t* prow1 = smem + (sW1 - sQ0) + row * 16;
    for (int kt = 0; kt < nk; ++kt) {
      const uint32_t par = kt & 1;
      const int klen = len - kt * T;
      const bool fr = far_pairs && far_pair(qt, kt, max_rel);
      auto gather = [&](const __half* tab) {
#pragma unroll 1
        for (int w = row; w < (fr ? WF : W); w += T) {
          const int pr = window_row(bucket_idx, max_rel, n_pos, qt, kt, w, fr);
#pragma unroll
          for (int i = 0; i < 2 * DPL; ++i) {
            const int term = i >> 3, pl = i & 7;
            *reinterpret_cast<uint4*>(smem + (sW0 - sQ0) + (size_t)term * POS_BYTES + (size_t)(pl * W + w) * 16) =
                *reinterpret_cast<const uint4*>(tab + term * pos_term + ((size_t)(h * DPL + pl) * n_pos + pr) * 8);
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      };
      gather(pos_k_s);  // the previous tile pair's MMAs have completed (bar_o below): the window buffer is free
      mbar_arrive(bar_g1);
      mbar_wait(bar_kv, par);
      if (row >= klen) {
        const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int pl = 0; pl < DPL; ++pl) {
          *reinterpret_cast<uint4*>(smem + (sV0 - sQ0) + (size_t)(pl * T + row) * 16) = z;
          *reinterpret_cast<uint4*>(smem + (sV1 - sQ0) + (size_t)(pl * T + row) * 16) = z;
        }
      }
      mbar_wait(bar_s1, par);
      tc_fence_after();
      float c_far = 0.f;  // far pair: c2p of this query row
      if (fr) {
        uint32_t v;
        tc_ld1(lane_addr + TM_B, v);
        tc_wait_ld();
        c_far = __uint_as_float(v);
      } else {
#pragma unroll 1
        for (int q = 0; q < W / 32; ++q) {
          uint32_t v[32];
          tc_ld32(lane_addr + TM_B + q * 32, v);
          tc_wait_ld();
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int j = row + (T - 1) - (q * 32 + e);
            if (j >= 0 && j < T) Bs[row * BCS + j] = __uint_as_float(v[e]);
          }
        }
      }
      tc_fence_before();
      gather(pos_q_s);  // the posK terms have been consumed (bar_s1)
      mbar_arrive(bar_g2);
      asm volatile("bar.sync 1, 128;" ::: "memory");  // every c2p entry is written before any p2c entry is added
      mbar_wait(bar_s2, par);
      tc_fence_after();
      if (fr) {
        uint32_t v;
        tc_ld1(lane_addr + TM_B, v);
        tc_wait_ld();
        Bs[row] = __uint_as_float(v);  // p2c of key `row`, the same for every query
      } else {
#pragma unroll 1
        for (int q = 0; q < W / 32; ++q) {
          uint32_t v[32];
          tc_ld32(lane_addr + TM_B + q * 32, v);
          tc_wait_ld();
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int ii = q * 32 + e + row - (T - 1);
            if (ii >= 0 && ii < T) Bs[ii * BCS + row] += __uint_as_float(v[e]);
          }
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const float* br = fr ? Bs : brow;
      float mt = -CUDART_INF_F;
#pragma unroll 1
      for (int q = 0; q < T / 32; ++q) {
        uint32_t v[32];
        tc_ld32(lane_addr + TM_S + q * 32, v);
        tc_wait_ld();
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) {
          const float4 bb = *reinterpret_cast<const float4*>(br + q * 32 + 4 * e4);
          const float bv[4] = {fr ? c_far + bb.x : bb.x, fr ? c_far + bb.y : bb.y, fr ? c_far + bb.z : bb.z, fr ? c_far + bb.w : bb.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int j = q * 32 + 4 * e4 + u;
            const float sc = __uint_as_float(v[4 * e4 + u]) + bv[u];
            mt = fmaxf(mt, j < klen ? sc : -CUDART_INF_F);
          }
        }
      }
      const float m_new = fmaxf(m, mt);
      const float mc = m_new * c_scale;
      const float alpha = ex2_approx(fmaf(m, c_scale, -mc));  // 0 on the first tile (m = -inf)
      m = m_new;
      float lt = 0.f;
#pragma unroll 1
      for (int q = 0; q < T / 32; ++q) {
        uint32_t v[32];
        tc_ld32(lane_addr + TM_S + q * 32, v);
        tc_wait_ld();
        float pv[32];
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) {
          const float4 bb = *reinterpret_cast<const float4*>(br + q * 32 + 4 * e4);
          const float bv[4] = {fr ? c_far + bb.x : bb.x, fr ? c_far + bb.y : bb.y, fr ? c_far + bb.z : bb.z, fr ? c_far + bb.w : bb.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int j = q * 32 + 4 * e4 + u;
            const float sc = __uint_as_float(v[4 * e4 + u]) + bv[u];
            const float p = j < klen ? ex2_approx(fmaf(sc, c_scale, -mc)) : 0.f;
            pv[4 * e4 + u] = p;
            lt += p;
          }
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 u0, u1;
          __half2* h0 = reinterpret_cast<__half2*>(&u0);
          __half2* h1 = reinterpret_cast<__half2*>(&u1);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float x0 = pv[g * 8 + 2 * e], x1 = pv[g * 8 + 2 * e + 1];
            const __half2 a = __floats2half2_rn(x0, x1);
            const float2 af = __half22float2(a);
            h0[e] = a;
            h1[e] = __floats2half2_rn(x0 - af.x, x1 - af.y);
          }
          *reinterpret_cast<uint4*>(prow0 + (size_t)(q * 4 + g) * T * 16) = u0;
          *reinterpret_cast<uint4*>(prow1 + (size_t)(q * 4 + g) * T * 16) = u1;
        }
      }
      l = fmaf(l, alpha, lt);
      tc_fence_before();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(bar_p);
      mbar_wait(bar_o, par);
      tc_fence_after();
#pragma unroll
      for (int q = 0; q < D / 32; ++q) {
        uint32_t v[32];
        tc_ld32(lane_addr + TM_O + q * 32, v);
        tc_wait_ld();
#pragma unroll
        for (int e = 0; e < 32; ++e) o[q * 32 + e] = fmaf(o[q * 32 + e], alpha, __uint_as_float(v[e]));
      }
      tc_fence_before();
    }
    const float inv_l = 1.0f / l;
    const int grow = qt * T + row;
    if (grow < len) {
#pragma unroll
      for (int g = 0; g < DPL; ++g) {
        uint4 u0, u1;
        __half2* h0 = reinterpret_cast<__half2*>(&u0);
        __half2* h1 = reinterpret_cast<__half2*>(&u1);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float x0 = o[g * 8 + 2 * e] * inv_l, x1 = o[g * 8 + 2 * e + 1] * inv_l;
          const __half2 a = __floats2half2_rn(x0, x1);
          const float2 af = __half22float2(a);
          h0[e] = a;
          h1[e] = __floats2half2_rn(x0 - af.x, x1 - af.y);
        }
        __half* dst = out_s + (size_t)(h * DPL + g) * s.plane_stride + (pbase + grow) * 8;
        *reinterpret_cast<uint4*>(dst) = u0;
        *reinterpret_cast<uint4*>(dst + out_blk) = u1;
        *reinterpret_cast<uint4*>(dst + 2 * out_blk) = u0;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)TM_COLS) : "memory");
  }
}

}  // namespace

bool deberta_attention_tc_supported(int head_dim, int span, int max_len) { return head_dim == D && span >= 254 && max_len <= T; }

bool deberta_attention_tc_multi_supported(int head_dim) { return head_dim == D; }

void launch_deberta_attention_tc(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const __half* pos_k_p, const __half* pos_q_p,
                                 int n_pos, int span, int heads, const PlanarSegs& s) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (!deberta_attention_tc_supported(D, span, s.max_len)) fail(SBV2_ERR_INTERNAL, "tensor-core DeBERTa attention: unsupported shape");
  const int win0 = span - (T - 1);
  if (win0 < 0 || win0 + W > n_pos) fail(SBV2_ERR_INTERNAL, "tensor-core DeBERTa attention: position window out of range");
  const size_t smem = 3 * QKV_BYTES + 2 * POS_BYTES + P_BYTES + 2 * SKEW_BYTES + 128;
  static PerDeviceOnce attr_once;
  attr_once.run([&] { CUDA_CHECK(cudaFuncSetAttribute(deberta_attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); });
  dim3 grid(heads, s.n);
  deberta_attention_tc_kernel<<<grid, 160, smem, ctx.stream>>>(ctx_out, qkv, pos_k_p, pos_q_p, n_pos, win0, heads, s);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

void launch_deberta_attention_tc_multi(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const __half* pos_k_p, const __half* pos_q_p,
                                       int n_pos, const int* bucket_idx, int max_rel, int heads, bool far_pairs, const PlanarSegs& s) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (!deberta_attention_tc_multi_supported(D) || s.max_len > kMaxBertTokens)
    fail(SBV2_ERR_INTERNAL, "tensor-core DeBERTa attention (multi-tile): unsupported shape");
  const size_t smem = 3 * QKV_BYTES + 2 * POS_BYTES + P_BYTES + 2 * SKEW_BYTES + 128;
  static PerDeviceOnce attr_once;
  attr_once.run([&] { CUDA_CHECK(cudaFuncSetAttribute(deberta_attention_tc_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); });
  dim3 grid(heads, s.n, (s.max_len + T - 1) / T);
  deberta_attention_tc_multi_kernel<<<grid, 160, smem, ctx.stream>>>(ctx_out, qkv, pos_k_p, pos_q_p, n_pos, bucket_idx, max_rel, heads, far_pairs, s);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

// Exact-numerics tensor-core attention (<= 128 tokens).  qkv_s / ctx_s are split-planar [h0 | h1 | h0] buffers scaled by `sc`
// (qkv_blk / ctx_blk: halves between plane blocks); pos_*_s: two-term fp16 position tables scaled by `sc` as well.
void launch_deberta_attention_tc_exact(const LaunchCtx& ctx, __half* ctx_s, long long ctx_blk, const __half* qkv_s, long long qkv_blk,
                                       const __half* pos_k_s, const __half* pos_q_s, int n_pos, int span, int heads, float sc,
                                       const PlanarSegs& s) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (!deberta_attention_tc_supported(D, span, s.max_len)) fail(SBV2_ERR_INTERNAL, "tensor-core DeBERTa attention: unsupported shape");
  const int win0 = span - (T - 1);
  if (win0 < 0 || win0 + W > n_pos) fail(SBV2_ERR_INTERNAL, "tensor-core DeBERTa attention: position window out of range");
  static PerDeviceOnce attr_once;
  attr_once.run(
      [&] { CUDA_CHECK(cudaFuncSetAttribute(deberta_attention_tc_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EX_SMEM)); });
  dim3 grid(heads, s.n);
  deberta_attention_tc_exact_kernel<<<grid, 160, EX_SMEM, ctx.stream>>>(ctx_s, ctx_blk, qkv_s, qkv_blk, pos_k_s, pos_q_s, n_pos, win0, heads,
                                                                         1.0f / (sc * sc), s);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

void launch_deberta_attention_tc_exact_multi(const LaunchCtx& ctx, __half* ctx_s, long long ctx_blk, const __half* qkv_s, long long qkv_blk,
                                             const __half* pos_k_s, const __half* pos_q_s, int n_pos, const int* bucket_idx, int max_rel,
                                             int heads, float sc, bool far_pairs, const PlanarSegs& s) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (!deberta_attention_tc_multi_supported(D) || s.max_len > kMaxBertTokens)
    fail(SBV2_ERR_INTERNAL, "tensor-core DeBERTa attention (exact, multi-tile): unsupported shape");
  static PerDeviceOnce attr_once;
  attr_once.run([&] {
    CUDA_CHECK(cudaFuncSetAttribute(deberta_attention_tc_exact_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EX_SMEM));
  });
  dim3 grid(heads, s.n, (s.max_len + T - 1) / T);
  deberta_attention_tc_exact_multi_kernel<<<grid, 160, EX_SMEM, ctx.stream>>>(ctx_s, ctx_blk, qkv_s, qkv_blk, pos_k_s, pos_q_s, n_pos, bucket_idx,
                                                                               max_rel, heads, 1.0f / (sc * sc), far_pairs, s);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

}  // namespace sbv2
