// Window-relative multi-head attention of the transformer flow on tcgen05 tensor cores.
//
// One CTA = (utterance, head, 128-query tile).  Scores S = Q K^T are produced 128 keys at a time
// into TMEM, the softmax runs on 128 threads (one query row each), probabilities go back to
// shared memory as the fp16 A operand of O += P V, with V read as an MN-major B operand straight
// from the planar activation layout.  The window terms are two extra tiny MMAs: Srel = Q Ek^T
// (9 relative keys, padded to 16) before the loop and O += Prel Ev after it.
// Softmax is exact two-pass (pass A: row max only; pass B: unnormalised probabilities 2^(x - max) and their row sum;
// the epilogue divides by the sum), so the O accumulator is never rescaled and each logit costs one exponential.
// Replaces rel_attention_planar_kernel (fp32 CUDA cores) in the flow; oracle: oracle/vits.py MultiHeadAttention.attention.
#include <cuda_fp16.h>
#include <math_constants.h>

#include "kernels.h"

namespace sbv2 {
namespace {

constexpr int QT = 128, KT = 128, D = 96, DP = D / 8, RP = 16;  // RP: relative positions padded to 16
constexpr uint32_t TILE_BYTES = DP * KT * 16;                   // one Q / K / V tile: 24 KB
constexpr uint32_t P_BYTES = (KT / 8) * QT * 16;                // 32 KB
constexpr uint32_t PREL_BYTES = (RP / 8) * QT * 16;             // 4 KB
constexpr uint32_t REL_BYTES = DP * RP * 16;                    // 3 KB
constexpr int TM_O = 0, TM_SREL = 96, TM_S = 128 /* two sets: +0, +128 */, TM_COLS = 512;
constexpr int NKV = 3;        // K/V tile buffers (prefetch depth)
constexpr int NSM_WARPS = 8;  // softmax warps: two per TMEM lane quarter, each takes half of the keys of a tile

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
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
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

// debug timeline (sbv2_debug_attn_trace): trace[(tile * 8 + event)] = clock64() of CTA (0, 0, 0)
#define ATRACE(ev, i)                                                                                   \
  do {                                                                                                   \
    if (trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (i) < 64) trace[(i) * 8 + (ev)] = clock64(); \
  } while (0)

// warps 0..7: softmax / epilogue (query row = 32*(w&3)+lane, key half = w>>2)
// warp 8: control (bulk loads + MMA issue)
__global__ void __launch_bounds__(288, 1) flow_attention_tc_kernel(__half* out, const __half* qkv, const __half* rel_k_p,
                                                                    const __half* rel_v_p, int heads, int window, PlanarSegs s,
                                                                    long long* trace) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  // grid slots are handed out in (x, y, z) order: with z walking the utterances longest-first the long CTAs start early
  // and the short ones fill the last wave
  const int b = s.order ? s.order[blockIdx.z] : (int)blockIdx.z, h = blockIdx.y;
  const int len = s.len[b];
  const int q0 = blockIdx.x * QT;
  if (q0 >= len) return;  // uniform per CTA
  const long long pbase = s.pstart[b];
  const int n_kt = (len + KT - 1) / KT;

  const uint32_t sQ = smem_u32(smem);
  const uint32_t sK0 = sQ + TILE_BYTES;             // K tiles [NKV]
  const uint32_t sV0 = sK0 + NKV * TILE_BYTES;      // V tiles [NKV]
  const uint32_t sP = sV0 + NKV * TILE_BYTES;       // P tile
  const uint32_t sPrel = sP + P_BYTES;
  const uint32_t sEk = sPrel + PREL_BYTES;
  const uint32_t sEv = sEk + REL_BYTES;
  const uint32_t sBar = sEv + REL_BYTES;
  // barriers
  const uint32_t bar_q = sBar, bar_kv = sBar + 8 /*[4]*/, bar_kvfree = sBar + 40 /*[4]*/, bar_s = sBar + 72 /*[2]*/,
                 bar_sfree = sBar + 88 /*[2]*/, bar_p = sBar + 104, bar_pfree = sBar + 112, bar_done = sBar + 120;
  const uint32_t tmem_slot = sBar + 128;
  float* ml_x = reinterpret_cast<float*>(smem + (sBar - sQ) + 256);  // [2 halves][128 rows][2] (m, l) exchange
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + (tmem_slot - sQ));

  if (threadIdx.x == 0) {
    mbar_init(bar_q, 1);
    for (int i = 0; i < NKV; ++i) {
      mbar_init(bar_kv + 8 * i, 1);
      mbar_init(bar_kvfree + 8 * i, 1);
    }
    mbar_init(bar_s, 1);
    mbar_init(bar_s + 8, 1);
    mbar_init(bar_sfree, 32 * NSM_WARPS);
    mbar_init(bar_sfree + 8, 32 * NSM_WARPS);
    mbar_init(bar_p, 32 * NSM_WARPS);
    mbar_init(bar_pfree, 1);
    mbar_init(bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == NSM_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)TM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // zero Prel (own row) before anything is accumulated into it
  if (threadIdx.x < 128) {
    const uint4 z = make_uint4(0, 0, 0, 0);
    *reinterpret_cast<uint4*>(smem + (sPrel - sQ) + threadIdx.x * 16) = z;
    *reinterpret_cast<uint4*>(smem + (sPrel - sQ) + QT * 16 + threadIdx.x * 16) = z;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot_ptr;
  pdl_launch_dependents();
  pdl_wait();  // PDL: the qkv projection's output is visible from here on

  const int q_plane0 = h * DP, k_plane0 = heads * DP + h * DP, v_plane0 = 2 * heads * DP + h * DP;
  const int n_tiles_total = 2 * n_kt;  // pass A tiles then pass B tiles

  if (warp == NSM_WARPS) {
    // ---------------- control warp ----------------
    auto load_tile = [&](int i) {  // i-th tile of the (pass A, pass B) sequence; lanes issue the plane copies in parallel
      const int buf = i % NKV;
      const uint32_t par = ((i / NKV) & 1) ^ 1;
      const int kt = i < n_kt ? i : i - n_kt;
      const bool with_v = i >= n_kt;
      const long long row0 = pbase + (long long)kt * KT;
      mbar_wait(bar_kvfree + 8 * buf, par);
      if (lane == 0) mbar_expect_tx(bar_kv + 8 * buf, with_v ? 2 * TILE_BYTES : TILE_BYTES);
      __syncwarp();
      if (lane < DP) {
        bulk_g2s(sK0 + buf * TILE_BYTES + lane * KT * 16, qkv + (size_t)(k_plane0 + lane) * s.plane_stride + row0 * 8, KT * 16,
                 bar_kv + 8 * buf);
      } else if (lane < 2 * DP && with_v) {
        const int pl = lane - DP;
        bulk_g2s(sV0 + buf * TILE_BYTES + pl * KT * 16, qkv + (size_t)(v_plane0 + pl) * s.plane_stride + row0 * 8, KT * 16,
                 bar_kv + 8 * buf);
      }
      __syncwarp();
    };
    if (elect_one_sync()) {
      mbar_expect_tx(bar_q, TILE_BYTES + 2 * REL_BYTES);
      for (int pl = 0; pl < DP; ++pl)
        bulk_g2s(sQ + pl * QT * 16, qkv + (size_t)(q_plane0 + pl) * s.plane_stride + (pbase + q0) * 8, QT * 16, bar_q);
      bulk_g2s(sEk, rel_k_p, REL_BYTES, bar_q);
      bulk_g2s(sEv, rel_v_p, REL_BYTES, bar_q);
    }
    __syncwarp();
    for (int i = 0; i < NKV && i < n_tiles_total; ++i) load_tile(i);
    mbar_wait(bar_q, 0);
    tc_fence_after();
    // K-major operands: LBO = rows*16 (next 8-channel plane), SBO = 128
    const uint64_t dq = make_desc(sQ, QT * 16, 128);
    const uint64_t dek = make_desc(sEk, RP * 16, 128);
    const uint64_t dp = make_desc(sP, QT * 16, 128);
    const uint64_t dprel = make_desc(sPrel, QT * 16, 128);
    // MN-major B operands (V, Ev): SBO = next 8-column plane, LBO = next 8 K rows (128 B)
    const uint64_t dev = make_desc(sEv, 128, RP * 16);
    constexpr uint32_t ID_S = idesc_f16(KT, 0), ID_REL = idesc_f16(RP, 0), ID_O = idesc_f16(D, 1);
    // Srel = Q Ek^T
    if (elect_one_sync()) {
      for (int k = 0; k < D / 16; ++k)
        tc_mma_f16(tmem + TM_SREL, dq + (uint64_t)(k * 2 * QT), dek + (uint64_t)(k * 2 * RP), ID_REL, k > 0 ? 1u : 0u);
    }
    __syncwarp();
    auto issue_s = [&](int i) {  // S(i) = Q K_i^T into accumulator set i & 1
      const int sb = i & 1, kb = i % NKV;
      mbar_wait(bar_kv + 8 * kb, (i / NKV) & 1);
      if (lane == 0) ATRACE(0, i);
      mbar_wait(bar_sfree + 8 * sb, ((i >> 1) & 1) ^ 1);  // softmax threads have read S(i-2)
      tc_fence_after();
      if (lane == 0) ATRACE(1, i);
      const uint64_t dk = make_desc(sK0 + kb * TILE_BYTES, KT * 16, 128);
      if (elect_one_sync()) {
        for (int k = 0; k < D / 16; ++k)
          tc_mma_f16(tmem + TM_S + sb * KT, dq + (uint64_t)(k * 2 * QT), dk + (uint64_t)(k * 2 * KT), ID_S, k > 0 ? 1u : 0u);
        tc_commit(bar_s + 8 * sb);
        if (i < n_kt) tc_commit(bar_kvfree + 8 * kb);  // pass A: the K tile is free once S is done
      }
      __syncwarp();
    };
    issue_s(0);
    for (int i = 0; i < n_tiles_total; ++i) {
      const int kb = i % NKV;
      if (i + 1 < n_tiles_total) issue_s(i + 1);  // overlaps the softmax of tile i
      if (i >= n_kt) {
        const int j = i - n_kt;
        mbar_wait(bar_p, j & 1);  // P tile written (and visible to the async proxy)
        tc_fence_after();
        if (lane == 0) ATRACE(2, i);
        const uint64_t dv = make_desc(sV0 + kb * TILE_BYTES, 128, KT * 16);
        if (elect_one_sync()) {
          for (int k = 0; k < KT / 16; ++k)
            tc_mma_f16(tmem + TM_O, dp + (uint64_t)(k * 2 * QT), dv + (uint64_t)(k * 16), ID_O, (j > 0 || k > 0) ? 1u : 0u);
          tc_commit(bar_pfree);
          tc_commit(bar_kvfree + 8 * kb);
        }
        __syncwarp();
      }
      if (i + NKV < n_tiles_total) load_tile(i + NKV);
      if (lane == 0) ATRACE(3, i);
    }
    // window value term: O += Prel Ev   (Prel complete: the last bar_p wait covered it)
    if (elect_one_sync()) {
      tc_mma_f16(tmem + TM_O, dprel, dev, ID_O, 1u);
      tc_commit(bar_done);
    }
    __syncwarp();
  } else {
    // ---------------- softmax / epilogue threads ----------------
    const int quarter = warp & 3, half = warp >> 2;
    const int row = quarter * 32 + lane;
    const int qi = q0 + row;
    const uint32_t lane_addr = tmem + ((uint32_t)(quarter * 32) << 16);
    const float c_scale = 1.4426950408889634f / sqrtf((float)D);  // log2(e) / sqrt(d)
    // relative-key logits of this row
    float srel[9];
    {
      // Srel is issued before S(0) on the same in-order MMA queue: S(0) complete implies Srel complete
      mbar_wait(bar_s, 0);
      tc_fence_after();
      uint32_t v[16];
      tc_ld16(lane_addr + TM_SREL, v);
      tc_wait_ld();
#pragma unroll
      for (int r = 0; r < 9; ++r) srel[r] = __uint_as_float(v[r]) * c_scale;
    }
    float m2 = -CUDART_INF_F, l = 0.f, mb = 0.f;  // running max (pass A); mb = row max, l = row sum of 2^(x - mb) (pass B)
    uint8_t* prow = smem + (sP - sQ) + row * 16;
    uint8_t* prel_row = smem + (sPrel - sQ) + row * 16;
    // pass A on 32 logits x[e] * c: running maximum only (no exponentials: the row sum is accumulated in pass B)
    auto pass_a = [&](const float* x, float c) {
      float mx = x[0];
#pragma unroll
      for (int e = 1; e < 32; ++e) mx = fmaxf(mx, x[e]);
      m2 = fmaxf(m2, mx * c);  // finite: the caller skips chunks without a valid key
    };
    // pass B: p[e] = 2^(x[e] * c - mb), unnormalised, fp16 into the P tile (columns 32 * c32 ...); the epilogue divides by l
    auto pass_b_store = [&](const float* x, float c, int c32, float* pv) {
      float sum = 0.f;
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        pv[e] = ex2_approx(fmaf(x[e], c, -mb));
        sum += pv[e];
      }
      l += sum;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 u;
        __half2* uh = reinterpret_cast<__half2*>(&u);
#pragma unroll
        for (int e = 0; e < 4; ++e) uh[e] = __floats2half2_rn(pv[q * 8 + 2 * e], pv[q * 8 + 2 * e + 1]);
        *reinterpret_cast<uint4*>(prow + (size_t)(c32 * 4 + q) * QT * 16) = u;
      }
    };
    for (int i = 0; i < n_tiles_total; ++i) {
      const bool pass_b = i >= n_kt;
      const int kt = pass_b ? i - n_kt : i;
      const int k0 = kt * KT;
      const int buf = i & 1;
      if (i > 0) {
        mbar_wait(bar_s + 8 * buf, (i >> 1) & 1);
        tc_fence_after();
      }
      if (threadIdx.x == 0) ATRACE(4, i);
      if (i == n_kt) {
        // combine the two key-halves of each row: the row maximum
        ml_x[(half * QT + row) * 2] = m2;
        asm volatile("bar.sync 1, %0;" ::"r"(32 * NSM_WARPS) : "memory");
        mb = fmaxf(m2, ml_x[((half ^ 1) * QT + row) * 2]);  // finite: key 0 is always valid
      }
      if (pass_b && kt > 0) mbar_wait(bar_pfree, (kt - 1) & 1);  // previous P tile consumed by the MMA
      if (threadIdx.x == 0) ATRACE(5, i);
#pragma unroll 1
      for (int cc = 0; cc < KT / 64; ++cc) {
        const int c = half * (KT / 64) + cc;
        const int kc0 = k0 + c * 32;
        if (kc0 >= len) {  // no valid key in this chunk (warp-uniform)
          if (pass_b) {
            const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(prow + (size_t)(c * 4 + q) * QT * 16) = z;
          }
          continue;
        }
        uint32_t v[32];
        tc_ld32(lane_addr + TM_S + buf * KT + c * 32, v);
        tc_wait_ld();
        float* x = reinterpret_cast<float*>(v);
        const int j0 = kc0 - qi + 4;  // index into srel of element 0: element e is relative position j0 + e - 4
        const bool band = j0 <= 8 && j0 + 31 >= 0;
        const bool tail = kc0 + 32 > len;
        if (!__any_sync(0xffffffffu, band) && !tail) {
          // fast path: plain scaled logits
          if (!pass_b) {
            pass_a(x, c_scale);
          } else {
            float pv[32];
            pass_b_store(x, c_scale, c, pv);
          }
          continue;
        }
        // slow path (a chunk that touches the diagonal band or the end of the utterance): build the logits first.
        // Selects only — data-dependent branches here diverge per lane and cost tens of thousands of cycles.
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const int r = j0 + e;
          float add = 0.f;
#pragma unroll
          for (int rr = 0; rr < 9; ++rr) add = (r == rr) ? srel[rr] : add;
          x[e] = (kc0 + e < len) ? fmaf(x[e], c_scale, add) : -CUDART_INF_F;
        }
        if (!pass_b) {
          pass_a(x, 1.0f);
        } else {
          float pv[32];
          pass_b_store(x, 1.0f, c, pv);
#pragma unroll
          for (int rr = 0; rr < 9; ++rr) {
            const int e = rr - j0;
            float val = 0.f;
#pragma unroll
            for (int ee = 0; ee < 32; ++ee) val = (e == ee) ? pv[ee] : val;
            if (e >= 0 && e < 32) *reinterpret_cast<__half*>(prel_row + (size_t)(rr >> 3) * QT * 16 + (rr & 7) * 2) = __float2half_rn(val);
          }
        }
      }
      // this thread's part of S is read
      if (threadIdx.x == 0) ATRACE(6, i);
      tc_fence_before();
      mbar_arrive(bar_sfree + 8 * buf);
      if (pass_b) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // P / Prel writes -> visible to the MMA's async proxy
        mbar_arrive(bar_p);
      }
    }
    // epilogue: O / l -> fp16 planar ctx (half 0: columns 0..63, half 1: 64..95); l = the two halves' sums
    ml_x[(half * QT + row) * 2 + 1] = l;
    asm volatile("bar.sync 1, %0;" ::"r"(32 * NSM_WARPS) : "memory");
    const float inv_l = 1.0f / (l + ml_x[((half ^ 1) * QT + row) * 2 + 1]);
    mbar_wait(bar_done, 0);
    tc_fence_after();
#pragma unroll 1
    for (int c = half * 2; c < (half == 0 ? 2 : D / 32); ++c) {
      uint32_t v[32];
      tc_ld32(lane_addr + TM_O + c * 32, v);
      tc_wait_ld();
      if (qi < len) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 u;
          __half2* uh = reinterpret_cast<__half2*>(&u);
#pragma unroll
          for (int e = 0; e < 4; ++e)
            uh[e] = __floats2half2_rn(__uint_as_float(v[q * 8 + 2 * e]) * inv_l, __uint_as_float(v[q * 8 + 2 * e + 1]) * inv_l);
          *reinterpret_cast<uint4*>(out + (size_t)(h * DP + c * 4 + q) * s.plane_stride + (pbase + qi) * 8) = u;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NSM_WARPS) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)TM_COLS) : "memory");
  }
}

}  // namespace

std::vector<__half> pack_flow_rel_table(const float* table, int window, int head_dim) {
  const int R = 2 * window + 1;
  if (head_dim != D || R > RP) fail(SBV2_ERR_UNSUPPORTED, "tensor-core attention: head_dim must be 96 and window at most 7");
  std::vector<__half> pk(size_t(DP) * RP * 8, __float2half(0.f));
  for (int r = 0; r < R; ++r)
    for (int d = 0; d < D; ++d) pk[(size_t(d / 8) * RP + r) * 8 + d % 8] = __float2half_rn(table[size_t(r) * D + d]);
  return pk;
}

// rel_k_p / rel_v_p: fp16 [D/8][16][8] packings of emb_rel_k / emb_rel_v ([2w+1, D], rows >= 2w+1 zero)
void launch_flow_attention_tc(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const __half* rel_k_p, const __half* rel_v_p,
                              int heads, int head_dim, int window, const PlanarSegs& s, long long* trace) {
  if (s.n <= 0 || s.max_len <= 0) return;
  if (head_dim != D || window != 4) fail(SBV2_ERR_UNSUPPORTED, "tensor-core attention: head_dim must be 96 and window 4");
  const size_t smem = (1 + 2 * NKV) * TILE_BYTES + P_BYTES + PREL_BYTES + 2 * REL_BYTES + 256 + 2 * QT * 2 * 4;
  static PerDeviceOnce attr_once;
  attr_once.run([&] { CUDA_CHECK(cudaFuncSetAttribute(flow_attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); });
  dim3 grid((s.max_len + QT - 1) / QT, heads, s.n);
  launch_pdl(ctx.pdl, flow_attention_tc_kernel, grid, dim3(32 * (NSM_WARPS + 1)), smem, ctx.stream, ctx_out, qkv, rel_k_p, rel_v_p, heads, window, s,
             trace);
  ctx.count();
}

}  // namespace sbv2

#ifdef SBV2_DEBUG_HOOKS  // only in libsbv2_b200_debug.so (build.py)
// ---- test hook: timeline + timing of the attention kernel on a synthetic batch ------------------------------------
#include "model.h"
#include "umma_conv.h"
extern "C" int sbv2_debug_attn_trace(int T, int n_utt, int heads, long long* out_trace /*[64*8]*/, float* out_ms) {
  using namespace sbv2;
  return guarded([&] {
    sbv2_model owner;
    owner.device = 0;
    CUDA_CHECK(cudaSetDevice(0));
    CUDA_CHECK(cudaStreamCreateWithFlags(&owner.stream, cudaStreamNonBlocking));
    LaunchCtx ctx = owner.ctx();
    DBuf meta, qkv, out, tr, rel;
    PinnedBuf pin;
    for (DBuf* b : {&meta, &qkv, &out, &tr, &rel}) b->stream = owner.stream;
    std::vector<int> ystart, ylen, muls{1};
    for (int i = 0; i < n_utt; ++i) {
      ystart.push_back(i * T);
      ylen.push_back(T);
    }
    BatchGeom bg = build_geoms(&owner, meta, pin, ystart, ylen, muls);
    const Geom& G = bg.g[0];
    const int C = heads * D;
    qkv.ensure(size_t(G.rows_tot) * 3 * C * 2);
    out.ensure(size_t(G.rows_tot) * C * 2);
    rel.ensure(2 * REL_BYTES);
    tr.ensure(64 * 8 * 8);
    CUDA_CHECK(cudaMemsetAsync(qkv.p, 0x11, size_t(G.rows_tot) * 3 * C * 2, owner.stream));  // small positive fp16 values
    CUDA_CHECK(cudaMemsetAsync(rel.p, 0, 2 * REL_BYTES, owner.stream));
    CUDA_CHECK(cudaMemsetAsync(tr.p, 0, 64 * 8 * 8, owner.stream));
    PlanarSegs ps;
    ps.start = bg.d_ystart;
    ps.pstart = G.d_pstart;
    ps.len = G.d_len;
    ps.n = n_utt;
    ps.max_len = T;
    ps.plane_stride = G.rows_tot * 8;
    const __half* rk = rel.as<__half>();
    const __half* rv = rk + REL_BYTES / 2;
    for (int i = 0; i < 2; ++i) launch_flow_attention_tc(ctx, out.as<__half>(), qkv.as<__half>(), rk, rv, heads, D, 4, ps, nullptr);
    cudaEvent_t e0, e1;
    CUDA_CHECK(cudaEventCreate(&e0));
    CUDA_CHECK(cudaEventCreate(&e1));
    CUDA_CHECK(cudaEventRecord(e0, owner.stream));
    for (int i = 0; i < 5; ++i) launch_flow_attention_tc(ctx, out.as<__half>(), qkv.as<__half>(), rk, rv, heads, D, 4, ps, nullptr);
    CUDA_CHECK(cudaEventRecord(e1, owner.stream));
    launch_flow_attention_tc(ctx, out.as<__half>(), qkv.as<__half>(), rk, rv, heads, D, 4, ps, tr.as<long long>());
    CUDA_CHECK(cudaStreamSynchronize(owner.stream));
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    if (out_ms) *out_ms = ms / 5.f;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (out_trace) CUDA_CHECK(cudaMemcpy(out_trace, tr.p, 64 * 8 * 8, cudaMemcpyDeviceToHost));
  });
}
#endif  // SBV2_DEBUG_HOOKS
