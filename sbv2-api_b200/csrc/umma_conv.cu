// tcgen05 / TMEM implicit-GEMM convolution (sm_100a only).
//
// Data layout ("planar fp16"): a [rows, C] activation is stored as C/8 planes, plane p holding
// channels [8p, 8p+8) of every row as one 16-byte item: half buf[C/8][rows][8].  Utterances of a
// batch are packed along rows with GAP zero rows around each one, so "same" zero padding is
// obtained by reading neighbouring rows, and rows that are never written stay zero.
//
// Why this layout: tcgen05.mma reads K-major operands as 8-row x 16-byte core matrices.  With
// SWIZZLE_NONE the descriptor (start, LBO = byte distance between the two 16-byte K chunks,
// SBO = byte distance between 8-row groups) addresses exactly plane-major shared memory
// [plane][row][16 B]: LBO = rows*16, SBO = 128.  A filter tap shifted by s rows is the same tile
// with start += 16*s — any s, no swizzle phase to respect — so one halo'd activation chunk, loaded
// once with plain 1-D bulk copies (cp.async.bulk, no tensor map), feeds every tap of the filter.
//
// Per CTA: rows [t0, t0 + 128*MT) of one utterance x NB output channels, K loop over
// (64-channel chunk, tap).
//   warp 0   : activation producer — bulk copies of activation chunks (ring of A slots), completion on mbarriers
//   warp 18  : weight producer — bulk copies of the packed weights (ring of B stages).  Its own thread since round 2:
//              issued from the activation producer's loop, a weight stage was only requested once the NEXT activation
//              slot had been obtained, i.e. one round trip late whenever the activation ring was the one that blocked
//              (few-rows GEMMs ran at one K chunk per L2 round trip: profiles/r2_launches_bert_exact_s7.csv)
//   warp 1   : TMEM alloc + single-thread tcgen05.mma issue, MT accumulators of 128 x NB fp32
//   warps 2-17: epilogue — tcgen05.ld, bias, residual, MRF accumulation, activation, fp16 store
// Two CTAs fit on an SM for every decoder shape (<= 113 KB smem, <= 256 TMEM columns), so one CTA's
// epilogue overlaps the other's MMA phase.
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <unordered_map>

#include "kernels.h"
#include "model.h"
#include "umma_conv.h"
#include "umma_device.cuh"

namespace sbv2 {
namespace {

constexpr int GAP = UMMA_GAP;
constexpr int TAIL_ROWS = UMMA_TAIL_ROWS;
constexpr int MAX_TAPS = UMMA_MAX_TAPS;
constexpr int MAX_ASLOTS = 8;
constexpr int MAX_STAGES = 8;
constexpr int SMEM_LIMIT = 227 * 1024;
constexpr int NUM_EPI_WARPS = 16;
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS + 32;  // + the weight producer (last warp)
constexpr int B_PRODUCER_WARP = 2 + NUM_EPI_WARPS;

struct UmmaConvArgs {
  CUtensorMap tmap;            // `in` as a 3-D tensor {8, rows, planes}, box {8, RA, kc / 8} (use_tmap), 64-byte aligned
  int use_tmap;                // activation chunks by one tensor-map TMA request instead of kc / 8 bulk copies
  const __half* in;
  long long in_plane_stride;   // elements between planes of `in`
  __half* out;
  long long out_plane_stride;
  const __half* residual;      // geometry of `out`; stored post-lrelu(0.1)
  const __half* residual2;     // further post-lrelu terms added the same way (MRF: other resblocks' outputs)
  const __half* residual3;
  float out_div;               // result divided by this before the activation (MRF mean), 1 = off
  float* accum;                // fp32 planar, geometry of `out`
  const __half* w;             // packed [nblk][kc][tap][KC/8][NB][8]
  const float* bias;           // [n_nblk*NB]
  const float* bias_utt;       // [n_utt][bias_utt_ld] or null
  int bias_utt_ld;
  int gate_half;               // > 0: WaveNet gate epilogue (N block = [tanh half | sigmoid half])
  // Thread-block cluster of `cluster` CTAs (1 = none): the CTAs of a cluster work on `cluster` consecutive row tiles of
  // the SAME (N block, group), so they consume the same weight stages; every CTA fetches 1/cluster of each stage and
  // multicasts it to all of them (L2 -> SM weight traffic and L2 request pressure divided by `cluster`)
  int cluster;
  int n_tiles;                 // row tiles of this launch (tile_prefix[n_utt])
  const int* tile_prefix;      // [n_utt+1]
  const int* pstart_in;        // [n_utt] first planar row of each utterance in `in`
  const int* pstart_out;
  const int* len;              // [n_utt] rows (input resolution)
  int n_utt;
  int cin, nb, n_nblk, n_items, taps, kc, nkc, mt, sps, nstages, nloads, total_steps, a_slots, b_resident;
  int n_groups;
  int tap_shift[UMMA_MAX_GROUPS * MAX_TAPS];
  int group_out_off[UMMA_MAX_GROUPS];
  int halo_lo, halo_hi;
  int out_mul, out_off;
  int act_out;
  float act_slope;             // max(v, slope*v): 1 none, 0 relu, 0.1 / 0.01 leaky relu
  int has_res, accum_mode, act_on_accum;
  float accum_div;
  int tmem_cols;
  unsigned idesc;
  float* rm_out;        // fp32 row-major output (or null)
  float rm_scale;       // accumulator scale of the row-major epilogue
  int rm_ld;
  const int* rm_start;
  __half* split_out;    // the row-major epilogue's values as a split-planar operand (geometry of `out`), or null
  int split_npl;        // planes per split block (= output channels / 8)
  float split_scale;    // the consuming split layer's in_scale
  long long* trace;  // debug: [grid][64 items][8 events] clock64 stamps, or null
};

// ---- the kernel ----------------------------------------------------------------------------------
// Persistent: one CTA per SM walks work items (tile, N block) round-robin.  The producer streams
// activation chunks and weight stages through their rings without regard to item boundaries, the
// MMA thread alternates between two TMEM accumulator sets, and the epilogue warps drain set i while
// the MMA thread fills set i^1 — loads, tensor work and stores of neighbouring tiles overlap.
struct TileInfo {
  int b, t0, len, nblk, grp;
};
#define TRACE(ev, itv)                                                                         \
  do {                                                                                         \
    if (p.trace && (itv) < 64) p.trace[((size_t)blockIdx.x * 64 + (itv)) * 8 + (ev)] = clock64(); \
  } while (0)

// Work item `item` of this CTA.  Without clusters: item = tile * per_tile + (grp, nblk).  With clusters the unit is a
// cluster item = (group of `cluster` consecutive tiles, (grp, nblk)) and CTA `rank` takes tile group * cluster + rank; a
// tile past the end is a dummy (no valid rows) that still runs the K loop, so the cluster's weight pipeline stays in step.
template <bool CLUSTER>
__device__ __forceinline__ TileInfo locate_item(const UmmaConvArgs& p, int item, int rank) {
  TileInfo ti;
  const int per_tile = p.n_nblk * p.n_groups;
  const int tgroup = item / per_tile;
  const int rem = item - tgroup * per_tile;
  const int tile = CLUSTER ? tgroup * p.cluster + rank : tgroup;
  ti.grp = rem / p.n_nblk;
  ti.nblk = rem - ti.grp * p.n_nblk;
  if (CLUSTER && tile >= p.n_tiles) {
    ti.b = p.n_utt - 1;
    ti.len = p.len[ti.b];
    ti.t0 = ti.len;  // every row invalid; the A tile is read from the (zero, allocated) rows after the last utterance
    return ti;
  }
  int lo = 0, hi = p.n_utt;  // largest b with tile_prefix[b] <= tile
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (p.tile_prefix[mid] <= tile) lo = mid;
    else hi = mid;
  }
  ti.b = lo;
  ti.t0 = (tile - p.tile_prefix[lo]) * 128 * p.mt;
  ti.len = p.len[lo];
  return ti;
}

// VARIANT bit 0: WaveNet gate epilogue; bit 1: thread-block clusters with multicast weight stages; bit 2: fp32 row-major
// epilogue (text encoder, exact-mode DeBERTa: bias + ReLU / GELU).  The plain kernel (VARIANT 0: every decoder and
// transformer-flow launch) is compiled with the planar epilogue only, so the other paths cost it no registers (96
// registers per thread at 576 threads: the epilogue is the part that spills first).
template <int VARIANT>
__global__ void __launch_bounds__(NUM_THREADS, 1) umma_conv_kernel(const __grid_constant__ UmmaConvArgs p) {
  constexpr bool GATE = (VARIANT & 1) != 0, ROWMAJOR = (VARIANT & 4) != 0;
  // bit 3: CTA pair (cta_group::2): clusters of two CTAs, ONE M = 256 MMA per K step issued by rank 0, each CTA holding
  // its own 128-row activation tile and half (by N) of every weight stage.  Uses the cluster item mapping; no multicast.
  constexpr bool PAIR2 = (VARIANT & 8) != 0;
  constexpr bool CLUSTER = (VARIANT & 2) != 0 || PAIR2;
  constexpr bool MCAST = (VARIANT & 2) != 0 && !PAIR2;
  // bit 4: split-K over a cluster (few-rows GEMMs with a deep K: one sentence through DeBERTa).  The `cluster` CTAs of a
  // cluster share ONE item; CTA `rank` accumulates K chunks [rank * nkc / cluster, (rank + 1) * nkc / cluster) — the serial
  // MMA chain and the weight bytes one SM has to pull both shrink by `cluster`.  The partial accumulators are exchanged
  // through distributed shared memory and summed in rank order (deterministic), each CTA finishing 128 / cluster rows.
  constexpr bool SPLITK = (VARIANT & 16) != 0;
  extern __shared__ __align__(128) uint8_t smem[];
  // warp index made provably warp-uniform so that role branches are uniform and the MMA
  // descriptors stay in uniform registers (UTCHMMA takes UR operands; R2UR per MMA is slow)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int TM = 128 * p.mt;
  const int RA = TM + p.halo_lo + p.halo_hi;
  const int planes_per_chunk = p.kc / 8;
  const uint32_t slot_bytes = (uint32_t)planes_per_chunk * RA * 16;
  const uint32_t step_bytes = (uint32_t)(PAIR2 ? p.nb / 2 : p.nb) * p.kc * 2;  // per CTA: a pair CTA holds half of N
  const uint32_t stage_bytes = step_bytes * p.sps;
  const uint32_t sA = smem_u32(smem);
  const uint32_t sB = sA + ((slot_bytes * p.a_slots + 127u) & ~127u);
  const uint32_t sBar = sB + stage_bytes * p.nstages;
  // barriers: a_full[8], a_empty[8], b_full[4], b_empty[4], acc_full[2], acc_empty[2]; tmem slot; bias[2][NB]
  const uint32_t bar_af = sBar, bar_ae = bar_af + 8 * MAX_ASLOTS, bar_bf = bar_ae + 8 * MAX_ASLOTS, bar_be = bar_bf + 8 * MAX_STAGES,
                 bar_accf = bar_be + 8 * MAX_STAGES, bar_acce = bar_accf + 16;
  const uint32_t tmem_slot = bar_acce + 16;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + (tmem_slot - sA));
  float* bias_s = reinterpret_cast<float*>(smem + (sBar - sA) + 320);  // [2][NB] (after 36 barriers + the TMEM slot)
  const int acc_cols = p.mt * p.nb;  // TMEM columns of one accumulator set
  // pair mode, leader side: "the peer's slot / stage / accumulator set is ready" (arrivals come from the peer CTA)
  const uint32_t bar_paf = sBar + 3072, bar_pbf = bar_paf + 8 * MAX_ASLOTS, bar_pacce = bar_pbf + 8 * MAX_STAGES;
  const int nc = (CLUSTER || SPLITK) ? p.cluster : 1;
  const int rank = (CLUSTER || SPLITK) ? (int)cluster_ctarank() : 0;
  const int kc_lo = SPLITK ? rank * p.nkc / nc : 0, kc_hi = SPLITK ? (rank + 1) * p.nkc / nc : p.nkc;  // this CTA's K chunks
  const int step_lo = kc_lo * p.taps, step_hi = kc_hi * p.taps;
  const int unit0 = (int)blockIdx.x / nc, unit_step = (int)gridDim.x / nc;  // this CTA's (cluster's) first item and stride
  const uint16_t cta_mask = (uint16_t)((1u << nc) - 1u);

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.a_slots; ++i) {
      mbar_init(bar_af + 8 * i, 1);
      mbar_init(bar_ae + 8 * i, 1);
    }
    for (int i = 0; i < p.nstages; ++i) {
      mbar_init(bar_bf + 8 * i, 1);
      mbar_init(bar_be + 8 * i, MCAST ? nc : 1);  // multicast: free again when every CTA of the cluster has consumed it
    }
    if (PAIR2) {
      for (int i = 0; i < p.a_slots; ++i) mbar_init(bar_paf + 8 * i, 1);
      for (int i = 0; i < p.nstages; ++i) mbar_init(bar_pbf + 8 * i, 1);
      for (int i = 0; i < 2; ++i) mbar_init(bar_pacce + 8 * i, NUM_EPI_WARPS);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_accf + 8 * i, 1);
      mbar_init(bar_acce + 8 * i, NUM_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (PAIR2) {  // both CTAs of the pair, same warp, same shared-memory offset for the result
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)p.tmem_cols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)p.tmem_cols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CLUSTER) cluster_sync_all();  // every CTA's barriers are initialised before a peer multicasts into them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // PDL: everything above overlapped the previous kernel's tail; its results are visible after the wait
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- activation producer ----------------
      uint32_t a_it = 0;  // running ring counter
      uint32_t pit = 0;
      for (int item = unit0; item < p.n_items; item += unit_step, ++pit) {
        const TileInfo ti = locate_item<CLUSTER>(p, item, rank);
        TRACE(0, pit);
        const long long in_row0 = (long long)p.pstart_in[ti.b] + ti.t0 - p.halo_lo;
        // Rows of the tile that can matter: the utterance's remaining rows plus the halo (rows past the utterance's end
        // are the zero padding the last valid outputs read).  A ragged last tile — or a one-sentence DeBERTa call, 7 rows
        // of a 128-row tile — copies only those; the rest of the slot keeps stale bytes, which only reach output rows
        // that the epilogue discards (every output row depends on its own input rows only).
        const uint32_t rows_ld = (uint32_t)min(RA, max(ti.len - ti.t0, 0) + p.halo_lo + p.halo_hi);
        auto load_a_chunk = [&](int kc) {
          const uint32_t slot = a_it % p.a_slots;
          mbar_wait_poll(bar_ae + 8 * slot, ((a_it / p.a_slots) & 1) ^ 1);
          if (p.use_tmap) {
            mbar_expect_tx(bar_af + 8 * slot, slot_bytes);  // the whole box, rows past the buffer's end are zero-filled
            tma_load_3d(sA + slot_bytes * slot, &p.tmap, 0, (int)in_row0, kc * planes_per_chunk, bar_af + 8 * slot);
            ++a_it;
            return;
          }
          mbar_expect_tx(bar_af + 8 * slot, (uint32_t)planes_per_chunk * rows_ld * 16);
          if (rows_ld > 0)
            for (int q = 0; q < planes_per_chunk; ++q) {
              const int plane = kc * planes_per_chunk + q;
              bulk_g2s(sA + slot_bytes * slot + (uint32_t)q * RA * 16, p.in + (size_t)plane * p.in_plane_stride + in_row0 * 8, rows_ld * 16,
                       bar_af + 8 * slot);
            }
          ++a_it;
        };
        for (int kc = kc_lo; kc < kc_hi; ++kc) load_a_chunk(kc);
        TRACE(1, pit);
      }
    }
    if (SPLITK) {
      __syncwarp();
      cluster_sync_all();  // split-K exchange point: every CTA's partial tile is in its shared memory
    }
  } else if (warp == B_PRODUCER_WARP) {
    if (lane == 0) {
      // ---------------- weight producer ----------------
      uint32_t b_it = 0;  // running ring counter
      bool first = true;
      for (int item = unit0; item < p.n_items; item += unit_step, first = false) {
        if (p.b_resident && !first) continue;  // resident weights are fetched once per CTA
        const TileInfo ti = locate_item<CLUSTER>(p, item, rank);
        // pair mode: the layer is packed in N blocks of nb / 2; this CTA streams block 2 * nblk + rank
        const __half* wbase = PAIR2 ? p.w + (size_t)((ti.grp * p.n_nblk + ti.nblk) * 2 + rank) * p.total_steps * (step_bytes / 2)
                                    : p.w + (size_t)(ti.grp * p.n_nblk + ti.nblk) * p.total_steps * (step_bytes / 2);
        auto load_b = [&](int i) {  // i-th stage load of this item
          const uint32_t st = b_it % p.nstages;
          mbar_wait_poll(bar_be + 8 * st, ((b_it / p.nstages) & 1) ^ 1);
          const int first_step = step_lo + i * p.sps;
          const int nsteps = min(p.sps, step_hi - first_step);
          const uint32_t bytes = step_bytes * nsteps;
          mbar_expect_tx(bar_bf + 8 * st, bytes);
          if (MCAST) {
            // this CTA's 1/nc of the stage goes to every CTA of the cluster (all of them expect the whole stage)
            const uint32_t slice = bytes / (uint32_t)nc;
            bulk_g2s_multicast(sB + stage_bytes * st + (uint32_t)rank * slice,
                               reinterpret_cast<const uint8_t*>(wbase + (size_t)first_step * (step_bytes / 2)) + (size_t)rank * slice, slice,
                               bar_bf + 8 * st, cta_mask);
          } else {
            bulk_g2s(sB + stage_bytes * st, wbase + (size_t)first_step * (step_bytes / 2), bytes, bar_bf + 8 * st);
          }
          ++b_it;
        };
        const int nloads = SPLITK ? (step_hi - step_lo + p.sps - 1) / p.sps : p.nloads;
        for (int i = 0; i < nloads; ++i) load_b(i);
      }
    }
    if (SPLITK) {
      __syncwarp();
      cluster_sync_all();
    }
  } else if (warp == 1) {
    {
      // ---------------- MMA issuer (whole warp runs the control flow, one elected lane issues) ----------------
      // Descriptors are built once; per MMA only the 14-bit start-address field advances (the issuing
      // thread's instruction latency, not the tensor pipe, was the bottleneck with per-MMA rebuilds).
      const int k16_per_chunk = p.kc / 16;
      const uint64_t desc_hi = (uint64_t)(0x4000u | (128u >> 4)) << 32;  // version 1, SBO = 128 B
      const uint64_t a_desc0 = desc_hi | ((uint64_t)((uint32_t)RA & 0x3FFF) << 16);    // LBO = RA*16 B
      const uint32_t nb_cta = PAIR2 ? (uint32_t)p.nb / 2 : (uint32_t)p.nb;              // weight rows (N) in this CTA's shared memory
      const uint64_t b_desc0 = desc_hi | ((uint64_t)(nb_cta & 0x3FFF) << 16);           // LBO = nb_cta*16 B
      const uint32_t a_kstep = 2u * (uint32_t)RA, b_kstep = 2u * nb_cta;                // two planes per K=16 step (16-B units)
      const uint32_t nb_u = (uint32_t)p.nb, idesc = p.idesc;
      // In a cluster launch the shared-window address of CTA rank r carries r in bits 24+ (0x0r000400 on sm_100); the
      // matrix descriptor's 14-bit start-address field is CTA-local, so strip the window base before it is added in.
      const uint32_t cta_win = sA & 0xFF000000u;
      const bool leader = elect_one_sync() != 0;  // the same lane issues every MMA / commit of this CTA
      // MT / K16 are compile-time (dispatched once, below): a per-tap switch or elect costs ~140 cycles per tap, which
      // the tensor pipe does not hide — it starts each MMA as it is issued (umma_microbench.cu, "issue shape")
      auto run = [&](auto mtk) {
        constexpr int MT = decltype(mtk)::mt, K16 = decltype(mtk)::k16;
        uint32_t a_slot_i = 0, a_par = 0, b_st = 0, b_par = 0, it = 0;
        if (PAIR2 && rank != 0) {
          // ---- peer CTA of a pair: no MMAs here.  This warp relays "my slot / stage has landed" to the leader, in the
          // order the leader consumes them; slots, stages and accumulators are released by the leader's multicast commits.
          for (int item = unit0; item < p.n_items; item += unit_step, ++it) {
            int step = 0, si = 0;
            for (int kc = 0; kc < p.nkc; ++kc) {
              mbar_wait_poll(bar_af + 8 * a_slot_i, a_par);
              if (lane == 0) mbar_arrive_remote(bar_paf + 8 * a_slot_i, 0);
              for (int tap = 0; tap < p.taps; ++tap, ++step) {
                if (p.b_resident) {
                  if (it == 0 && step == 0) {
                    mbar_wait_poll(bar_bf, 0);
                    if (lane == 0) mbar_arrive_remote(bar_pbf, 0);
                  }
                } else {
                  if (si == 0) {
                    mbar_wait_poll(bar_bf + 8 * b_st, b_par);
                    if (lane == 0) mbar_arrive_remote(bar_pbf + 8 * b_st, 0);
                  }
                  ++si;
                  if (si == p.sps || step == p.total_steps - 1) {
                    si = 0;
                    if (++b_st == (uint32_t)p.nstages) {
                      b_st = 0;
                      b_par ^= 1;
                    }
                  }
                }
              }
              if (++a_slot_i == (uint32_t)p.a_slots) {
                a_slot_i = 0;
                a_par ^= 1;
              }
            }
          }
          return;
        }
        for (int item = unit0; item < p.n_items; item += unit_step, ++it) {
          const uint32_t buf = it & 1;
          mbar_wait_poll(bar_acce + 8 * buf, ((it >> 1) & 1) ^ 1);  // epilogue has drained this accumulator set
          if (PAIR2) mbar_wait_poll_cluster(bar_pacce + 8 * buf, ((it >> 1) & 1) ^ 1);  // ... and so has the peer's
          tc_fence_after();
          if (lane == 0) TRACE(2, it);
          const uint32_t tmem_acc = tmem_base + buf * acc_cols;
          const int grp = (item % (p.n_nblk * p.n_groups)) / p.n_nblk;
          int step = step_lo, si = 0;
          for (int kc = kc_lo; kc < kc_hi; ++kc) {
            mbar_wait_poll(bar_af + 8 * a_slot_i, a_par);
            if (PAIR2) mbar_wait_poll_cluster(bar_paf + 8 * a_slot_i, a_par);
            if (kc == kc_lo && lane == 0) TRACE(3, it);
            const uint64_t a_chunk = a_desc0 + ((sA - cta_win + slot_bytes * a_slot_i) >> 4) + (uint32_t)p.halo_lo;
            for (int tap = 0; tap < p.taps; ++tap, ++step) {
              uint32_t b_addr;
              if (p.b_resident) {
                if (it == 0 && step == 0) {
                  mbar_wait_poll(bar_bf, 0);
                  if (PAIR2) mbar_wait_poll_cluster(bar_pbf, 0);
                }
                b_addr = sB + step_bytes * step;
              } else {
                if (si == 0) {
                  mbar_wait_poll(bar_bf + 8 * b_st, b_par);
                  if (PAIR2) mbar_wait_poll_cluster(bar_pbf + 8 * b_st, b_par);
                }
                b_addr = sB + stage_bytes * b_st + step_bytes * si;
              }
              const uint64_t a_tap = a_chunk + (int64_t)p.tap_shift[grp * MAX_TAPS + tap];
              const uint64_t b_d = b_desc0 + ((b_addr - cta_win) >> 4);
              const uint32_t accf = step > step_lo ? 1u : 0u;
              if (leader) {
                if (PAIR2) issue_mmas_pair<MT, K16>(tmem_acc, a_tap, b_d, a_kstep, b_kstep, nb_u, idesc, accf);
                else issue_mmas<MT, K16>(tmem_acc, a_tap, b_d, a_kstep, b_kstep, nb_u, idesc, accf);
              }
              if (!p.b_resident) {
                ++si;
                if (si == p.sps || step == step_hi - 1) {
                  if (leader) {
                    if (PAIR2) tc_commit_pair(bar_be + 8 * b_st);
                    else if (MCAST) tc_commit_multicast(bar_be + 8 * b_st, cta_mask);
                    else tc_commit(bar_be + 8 * b_st);
                  }
                  si = 0;
                  if (++b_st == (uint32_t)p.nstages) {
                    b_st = 0;
                    b_par ^= 1;
                  }
                }
              }
            }
            if (leader) {
              if (PAIR2) tc_commit_pair(bar_ae + 8 * a_slot_i);
              else tc_commit(bar_ae + 8 * a_slot_i);
            }
            if (++a_slot_i == (uint32_t)p.a_slots) {
              a_slot_i = 0;
              a_par ^= 1;
            }
          }
          if (leader) {
            if (PAIR2) tc_commit_pair(bar_accf + 8 * buf);
            else tc_commit(bar_accf + 8 * buf);
          }
          __syncwarp();
          if (lane == 0) TRACE(4, it);
        }
      };
#define SBV2_ROLE_CASE(M, K) \
  case (M) * 8 + (K):        \
    run(MtK<M, K>{});        \
    break;
      switch (p.mt * 8 + k16_per_chunk) {
        SBV2_ROLE_CASE(1, 1) SBV2_ROLE_CASE(1, 2) SBV2_ROLE_CASE(1, 3) SBV2_ROLE_CASE(1, 4)
        SBV2_ROLE_CASE(2, 1) SBV2_ROLE_CASE(2, 2) SBV2_ROLE_CASE(2, 3) SBV2_ROLE_CASE(2, 4)
        SBV2_ROLE_CASE(4, 1) SBV2_ROLE_CASE(4, 2) SBV2_ROLE_CASE(4, 3) SBV2_ROLE_CASE(4, 4)
        SBV2_ROLE_CASE(8, 1) SBV2_ROLE_CASE(8, 2) SBV2_ROLE_CASE(8, 3) SBV2_ROLE_CASE(8, 4)
        SBV2_ROLE_CASE(16, 1) SBV2_ROLE_CASE(16, 2) SBV2_ROLE_CASE(16, 3) SBV2_ROLE_CASE(16, 4)
        default: __trap();  // make_layer only produces the combinations above (kc in {16, 32, 48, 64})
      }
#undef SBV2_ROLE_CASE
    }
    if (SPLITK) {
      __syncwarp();
      cluster_sync_all();
    }
  } else {
    // ---------------- epilogue warps ----------------
    const int wq = warp & 3;           // TMEM lane quarter this warp may access
    const int part = (warp - 2) >> 2;  // NUM_EPI_WARPS/4 warps per quarter split the work items
    const int etid = threadIdx.x - 64;
    const bool wide = !ROWMAJOR && (p.nb % 32 == 0) && p.accum_mode == UACC_NONE && p.has_res != 3;
    const int nch = wide ? 32 : 16;
    const int items_per_acc = p.nb / nch;
    const int n_sub = p.mt * items_per_acc;
    const bool bias_per_item = p.n_nblk > 1 || p.bias_utt != nullptr;
    // drain one accumulator set: rows [row_lo, row_hi) of the tile (the whole tile unless split-K)
    auto drain = [&](const TileInfo& ti, uint32_t tmem_acc, const float* bias, int row_lo, int row_hi) {
      if (GATE) {
        const int per_acc = p.gate_half / 16;
        for (int sub = part; sub < p.mt * per_acc; sub += NUM_EPI_WARPS / 4) {
          const int a = sub / per_acc;
          const int c0 = (sub - a * per_acc) * 16;
          const int t = ti.t0 + a * 128 + wq * 32 + lane;
          const long long orow = (long long)p.pstart_out[ti.b] + t;
          const uint32_t taddr = tmem_acc + ((uint32_t)(wq * 32) << 16) + (uint32_t)(a * p.nb + c0);
          epilogue_gate(p, taddr, taddr + (uint32_t)p.gate_half, t < ti.len, orow, ti.nblk * p.gate_half + c0, bias + c0,
                        bias + p.gate_half + c0);
        }
      } else
      for (int sub = part; sub < n_sub; sub += NUM_EPI_WARPS / 4) {
        const int a = sub / items_per_acc;
        const int c0 = (sub - a * items_per_acc) * nch;
        const int r = a * 128 + wq * 32 + lane;
        const int t = ti.t0 + r;
        const bool valid = t < ti.len && (!SPLITK || (r >= row_lo && r < row_hi));
        const long long orow = (long long)p.pstart_out[ti.b] + (long long)t * p.out_mul + p.out_off + p.group_out_off[ti.grp];
        const uint32_t taddr = tmem_acc + ((uint32_t)(wq * 32) << 16) + (uint32_t)(a * p.nb + c0);
        const int cg = ti.nblk * p.nb + c0;
        if (ROWMAJOR) {
          epilogue_item_rm(p, taddr, valid, p.rm_out != nullptr ? (long long)p.rm_start[ti.b] + t : 0, orow, cg, bias + c0);
        } else if (p.accum_mode != UACC_NONE) {
          if (p.has_res) epilogue_item<16, true, 1>(p, taddr, valid, orow, cg, bias + c0);
          else epilogue_item<16, true, 0>(p, taddr, valid, orow, cg, bias + c0);
        } else if (p.has_res == 3) {
          epilogue_item<16, false, 3>(p, taddr, valid, orow, cg, bias + c0);
        } else if (wide) {
          if (p.has_res) epilogue_item<32, false, 1>(p, taddr, valid, orow, cg, bias + c0);
          else epilogue_item<32, false, 0>(p, taddr, valid, orow, cg, bias + c0);
        } else {
          if (p.has_res) epilogue_item<16, false, 1>(p, taddr, valid, orow, cg, bias + c0);
          else epilogue_item<16, false, 0>(p, taddr, valid, orow, cg, bias + c0);
        }
      }
    };
    auto load_bias = [&](const TileInfo& ti, float* bias) {
      for (int i = etid; i < p.nb; i += NUM_EPI_WARPS * 32) {
        float v = p.bias[(size_t)ti.nblk * p.nb + i];
        if (p.bias_utt) v += p.bias_utt[(size_t)ti.b * p.bias_utt_ld + (size_t)ti.nblk * p.nb + i];
        bias[i] = v;
      }
      asm volatile("bar.sync 1, %0;" ::"r"(NUM_EPI_WARPS * 32) : "memory");
    };
    if (SPLITK) {
      // One item per cluster (launch_umma).  (1) every CTA copies its partial accumulators (valid rows) into its own shared
      // memory — the activation ring: all of this CTA's MMAs, the ring's only readers, have completed; (2) cluster barrier;
      // (3) CTA `rank` sums rows [rank * 128 / nc, ...) over the peers in rank order through DSMEM, puts the sums back into
      // its TMEM accumulators and drains those rows through the ordinary epilogue.
      const bool have = unit0 < p.n_items;
      TileInfo ti{};
      const int dpitch = p.nb + 4;  // floats per dumped row
      const int n16 = p.nb / 16;
      const int r = wq * 32 + lane;
      if (have) {
        ti = locate_item<false>(p, unit0, 0);
        load_bias(ti, bias_s);
        mbar_wait(bar_accf, 0);
        tc_fence_after();
        if (threadIdx.x == 64) TRACE(5, 0);
        float* dump = reinterpret_cast<float*>(smem) + (size_t)r * dpitch;
        for (int g = part; g < n16; g += NUM_EPI_WARPS / 4) {
          uint32_t v[16];
          tc_ld16(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(g * 16), v);
          tc_wait_ld();
          if (ti.t0 + r < ti.len) {
#pragma unroll
            for (int q = 0; q < 4; ++q)
              *reinterpret_cast<uint4*>(dump + g * 16 + 4 * q) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          }
        }
      }
      __syncwarp();
      cluster_sync_all();
      if (have) {
        const int row_lo = rank * 128 / nc, row_hi = (rank + 1) * 128 / nc;
        const bool mine = r >= row_lo && r < row_hi && ti.t0 + r < ti.len;
        if (wq * 32 < row_hi && wq * 32 + 32 > row_lo) {  // warp-uniform: this warp's lane quarter overlaps the slice
          for (int g = part; g < n16; g += NUM_EPI_WARPS / 4) {
            float acc[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) acc[e] = 0.f;
            if (mine) {
              const uint32_t local = sA + (uint32_t)((r * dpitch + g * 16) * 4);
              for (int q = 0; q < nc; ++q) {
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                  const float4 f = ld_dsmem_f4(local + 16 * v4, (uint32_t)q);
                  acc[4 * v4] += f.x;
                  acc[4 * v4 + 1] += f.y;
                  acc[4 * v4 + 2] += f.z;
                  acc[4 * v4 + 3] += f.w;
                }
              }
            }
            __syncwarp();
            tc_st16(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(g * 16), reinterpret_cast<const uint32_t*>(acc));
          }
          tc_wait_st();
        }
        tc_fence_before();
        asm volatile("bar.sync 1, %0;" ::"r"(NUM_EPI_WARPS * 32) : "memory");  // the drain's column split differs from the sum's
        tc_fence_after();
        drain(ti, tmem_base, bias_s, row_lo, row_hi);
        tc_fence_before();
        if (threadIdx.x == 64) TRACE(6, 0);
      }
    } else {
    uint32_t it = 0;
    for (int item = unit0; item < p.n_items; item += unit_step, ++it) {
      const uint32_t buf = it & 1;
      const TileInfo ti = locate_item<CLUSTER>(p, item, rank);
      float* bias = bias_s + (bias_per_item ? buf * p.nb : 0);
      // (per item: the set used two items ago has been fully consumed — its acc_empty arrivals happen after the last read)
      if (bias_per_item || it == 0) load_bias(ti, bias);
      mbar_wait(bar_accf + 8 * buf, (it >> 1) & 1);
      tc_fence_after();
      if (threadIdx.x == 64) TRACE(5, it);
      drain(ti, tmem_base + buf * acc_cols, bias, 0, TM);
      // release the accumulator set
      tc_fence_before();
      __syncwarp();
      if (threadIdx.x == 64) TRACE(6, it);
      if (lane == 0) {
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_acce + 8 * buf) : "memory");
        if (PAIR2 && rank != 0) mbar_arrive_remote(bar_pacce + 8 * buf, 0);  // the leader issues the MMAs into both TMEMs
      }
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CLUSTER || SPLITK) cluster_sync_all();  // no CTA leaves while a peer may still multicast into / read from its shared memory
  if (warp == 1) {
    if (PAIR2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}

// ---- glue kernels ----------------------------------------------------------------------------------
// packed fp32 -> planar fp16 split.  TERMS = 2: x ~ h0 + h1, planes [h0 | h1 | h0]; TERMS = 3: x ~ h0 + h1 + h2,
// planes [h0 | h1 | h2 | h0 | h1 | h0] (h0 = fp16(x), h1 = fp16(x - h0), h2 = fp16(x - h0 - h1))
template <int TERMS>
__global__ void split_planar_kernel(__half* out, long long plane_stride, const float* in, int in_ld, int C, const int* start,
                                    const int* pstart, const int* len, float in_scale) {
  int b = blockIdx.y;
  int t = blockIdx.x * blockDim.y + threadIdx.y;
  if (t >= len[b]) return;
  const float* row = in + (size_t)(start[b] + t) * in_ld;
  const int npl = C / 8;
  for (int pl = threadIdx.x; pl < npl; pl += blockDim.x) {
    uint4 o0, o1, o2;
    __half2* q0 = reinterpret_cast<__half2*>(&o0);
    __half2* q1 = reinterpret_cast<__half2*>(&o1);
    __half2* q2 = reinterpret_cast<__half2*>(&o2);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float x0 = row[pl * 8 + 2 * e] * in_scale, x1 = row[pl * 8 + 2 * e + 1] * in_scale;  // power of two: exact
      const __half2 h0 = __floats2half2_rn(x0, x1);
      const float2 f0 = __half22float2(h0);
      const float r0 = x0 - f0.x, r1 = x1 - f0.y;  // exact
      const __half2 h1 = __floats2half2_rn(r0, r1);
      const float2 f1 = __half22float2(h1);
      q0[e] = h0;
      q1[e] = h1;
      q2[e] = __floats2half2_rn(r0 - f1.x, r1 - f1.y);
    }
    const size_t r8 = (size_t)(pstart[b] + t) * 8;
    __half* base = out + (size_t)pl * plane_stride + r8;
    const size_t blk = (size_t)npl * plane_stride;
    if (TERMS == 2) {
      *reinterpret_cast<uint4*>(base) = o0;
      *reinterpret_cast<uint4*>(base + blk) = o1;
      *reinterpret_cast<uint4*>(base + 2 * blk) = o0;
    } else {
      *reinterpret_cast<uint4*>(base) = o0;
      *reinterpret_cast<uint4*>(base + blk) = o1;
      *reinterpret_cast<uint4*>(base + 2 * blk) = o2;
      *reinterpret_cast<uint4*>(base + 3 * blk) = o0;
      *reinterpret_cast<uint4*>(base + 4 * blk) = o1;
      *reinterpret_cast<uint4*>(base + 5 * blk) = o0;
    }
  }
}
// planar fp32 -> planar fp16, utterance rows only: one 16-byte item (8 channels of one row) per thread; consecutive
// threads take consecutive rows of a plane, so a warp reads 1 KB and writes 512 B contiguous
__global__ void planar_cast_kernel(__half* out, const float* in, long long plane_stride, const int* pstart, const int* len) {
  const int b = blockIdx.z, pl = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= len[b]) return;
  const size_t o = (size_t)pl * plane_stride + (size_t)(pstart[b] + t) * 8;
  const float4 x0 = *reinterpret_cast<const float4*>(in + o), x1 = *reinterpret_cast<const float4*>(in + o + 4);
  uint4 v;
  __half2* vh = reinterpret_cast<__half2*>(&v);
  vh[0] = __floats2half2_rn(x0.x, x0.y);
  vh[1] = __floats2half2_rn(x0.z, x0.w);
  vh[2] = __floats2half2_rn(x1.x, x1.y);
  vh[3] = __floats2half2_rn(x1.z, x1.w);
  *reinterpret_cast<uint4*>(out + o) = v;
}

// packed fp32 [rows, in_ld] (utterance b at rows start[b]..) -> planar fp16 with gaps
__global__ void to_planar_kernel(__half* out, long long plane_stride, const float* in, int in_ld, int C, const int* start,
                                 const int* pstart, const int* len, int act) {
  int b = blockIdx.y;
  int t = blockIdx.x * blockDim.y + threadIdx.y;
  if (t >= len[b]) return;
  const float* row = in + (size_t)(start[b] + t) * in_ld;
  for (int pl = threadIdx.x; pl < C / 8; pl += blockDim.x) {
    uint4 o;
    __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
    for (int e = 0; e < 4; ++e) oh[e] = __floats2half2_rn(act_apply(row[pl * 8 + 2 * e], act), act_apply(row[pl * 8 + 2 * e + 1], act));
    *reinterpret_cast<uint4*>(out + (size_t)pl * plane_stride + (size_t)(pstart[b] + t) * 8) = o;
  }
}

// planar fp16 -> packed fp32 [rows, C] (debug / tests)
__global__ void from_planar_kernel(float* out, const __half* in, long long plane_stride, int C, const int* start, const int* pstart,
                                   const int* len) {
  int b = blockIdx.y;
  int t = blockIdx.x * blockDim.y + threadIdx.y;
  if (t >= len[b]) return;
  float* row = out + (size_t)(start[b] + t) * C;
  for (int pl = threadIdx.x; pl < C / 8; pl += blockDim.x) {
    uint4 r = *reinterpret_cast<const uint4*>(in + (size_t)pl * plane_stride + (size_t)(pstart[b] + t) * 8);
    const __half2* rh = reinterpret_cast<const __half2*>(&r);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 y = __half22float2(rh[e]);
      row[pl * 8 + 2 * e] = y.x;
      row[pl * 8 + 2 * e + 1] = y.y;
    }
  }
}

// zero the GAP rows before each utterance, after the last one, plus the tail
__global__ void zero_gaps_kernel(__half* buf, long long plane_stride, const int* pstart, const int* len, int n_utt, int tail) {
  int gi = blockIdx.x, pl = blockIdx.y;
  long long r0, r1;
  if (gi == 0) {
    r0 = 0;
    r1 = pstart[0];
  } else {
    r0 = (long long)pstart[gi - 1] + len[gi - 1];
    r1 = (gi < n_utt) ? pstart[gi] : r0 + tail;
  }
  uint4 z = make_uint4(0, 0, 0, 0);
  for (long long r = r0 + threadIdx.x; r < r1; r += blockDim.x)
    *reinterpret_cast<uint4*>(buf + (size_t)pl * plane_stride + r * 8) = z;
}

int pow2_at_least(int v) {
  int p = 32;
  while (p < v) p <<= 1;
  return p;
}

uint16_t f2h(float f) { return __half_as_ushort(__float2half_rn(f)); }

// wsel(g, co, ci, tap) returns the weight of group g, output channel co, input channel ci, tap index `tap`;
// shifts[g][tap] the input-row shift of that tap.
template <class WSel>
ConvLayer make_layer(sbv2_model* owner, int cin, int cout, int taps, int n_groups, const int (*shifts)[MAX_TAPS], const int* group_out_off,
                     const float* bias, WSel wsel, int mt_pref, int nb_max = 256) {
  ConvLayer L;
  L.cin = cin;
  L.cout = cout;
  L.taps = taps;
  L.n_groups = n_groups;
  if (taps > MAX_TAPS) fail(SBV2_ERR_UNSUPPORTED, "conv has too many taps for the tensor-core plan");
  if (n_groups > UMMA_MAX_GROUPS) fail(SBV2_ERR_UNSUPPORTED, "too many polyphase groups");
  if (cin % 16 != 0 || cout % 16 != 0) fail(SBV2_ERR_UNSUPPORTED, "tensor-core conv needs channel counts divisible by 16");
  // N block: largest multiple of 16 that divides cout and is <= 256
  L.nb = 0;
  for (int nb = std::min(cout, std::max(16, std::min(nb_max, 256))); nb >= 16; nb -= 16)
    if (cout % nb == 0) {
      L.nb = nb;
      break;
    }
  L.n_nblk = cout / L.nb;
  L.kc = cin % 64 == 0 ? 64 : (cin % 48 == 0 ? 48 : (cin % 32 == 0 ? 32 : 16));
  L.nkc = cin / L.kc;
  int lo = 0, hi = 0;
  for (int g = 0; g < n_groups; ++g) {
    L.group_out_off[g] = group_out_off ? group_out_off[g] : 0;
    for (int i = 0; i < taps; ++i) {
      L.tap_shift[g][i] = shifts[g][i];
      lo = std::min(lo, shifts[g][i]);
      hi = std::max(hi, shifts[g][i]);
    }
  }
  L.halo_lo = -lo;
  L.halo_hi = hi;
  if (L.halo_lo > GAP || L.halo_hi > GAP) fail(SBV2_ERR_UNSUPPORTED, "conv halo exceeds the packing gap");
  L.total_steps = taps * L.nkc;
  const size_t step_bytes = size_t(L.nb) * L.kc * 2;
  const size_t w_bytes = step_bytes * L.total_steps;
  // accumulators per CTA: two sets of MT*NB <= 256 TMEM columns (double-buffered across work items)
  int mt = 1;
  while (mt * 2 <= std::min(mt_pref, 256 / L.nb)) mt *= 2;
  const int ppc = L.kc / 8;
  const size_t kMisc = 4096;  // barriers (256 B) + two bias sets
  const size_t budget = size_t(SMEM_LIMIT) - kMisc;
  bool placed = false;
  for (; mt >= 1 && !placed; mt >>= 1) {
    const int ra = 128 * mt + L.halo_lo + L.halo_hi;
    const size_t slot = size_t(ppc) * ra * 16;
    // weights resident for the whole kernel when they fit next to a double-buffered activation tile
    const int min_slots = std::max(2, std::min(L.nkc + 1, MAX_ASLOTS));
    if (L.n_nblk == 1 && L.n_groups == 1 && w_bytes + slot * std::min(2 * L.nkc, MAX_ASLOTS) <= budget && w_bytes <= 100 * 1024) {
      L.b_resident = 1;
      L.sps = L.total_steps;
      L.nloads = 1;
      L.nstages = 1;
      L.mt = mt;
      L.a_slots = std::min(2 * L.nkc, MAX_ASLOTS);
      while (L.a_slots < MAX_ASLOTS && w_bytes + slot * (L.a_slots + 1) <= budget && L.a_slots < 3 * L.nkc) ++L.a_slots;
      L.smem = ((slot * L.a_slots + 127) & ~size_t(127)) + w_bytes + kMisc;
      placed = true;
      break;
    }
    L.b_resident = 0;
    L.sps = int(std::max<size_t>(1, (16 * 1024) / step_bytes));
    L.sps = std::min(L.sps, L.total_steps);
    L.nloads = (L.total_steps + L.sps - 1) / L.sps;
    const size_t stage_bytes = step_bytes * L.sps;
    // Weight stages first: a stage is 16-25 KB and arrives after ~2 us of L2 latency, so the bytes in flight set the
    // streaming rate (4 stages = 64 KB gave ~17 B/clk where the big decoder layers consume 32 B/clk); the activation
    // ring needs far fewer bytes in flight, three chunk slots keep one chunk of lookahead.
    const int ring_min_slots = std::max(2, std::min(L.nkc + 1, 3));
    // Few-rows packing (N blocks <= 64, 128-row items: one sentence through DeBERTa, a batch-1 utterance): per 64-channel
    // K chunk the activation slot (16 KB) is larger than the weight step (8 KB) and every chunk costs one L2 / HBM round
    // trip, so the chunks in flight set the rate — K = 12288 with three slots is 64 round trips in a row
    // (profiles/r2_launches_bert_exact_s7.csv).  There the activation ring gets the depth first.
    const bool latency_mode = nb_max <= 64 && mt == 1 && L.nkc > 4;
    if (latency_mode) {
      for (int slots = std::min(MAX_ASLOTS, L.nkc + 1); slots >= ring_min_slots && !placed; --slots)
        for (int ns = std::min(MAX_STAGES, std::max(2, L.nloads)); ns >= 2 && !placed; --ns) {
          size_t sm = ((slot * slots + 127) & ~size_t(127)) + stage_bytes * ns + kMisc;
          if (sm <= size_t(SMEM_LIMIT) && (ns >= 4 || ns >= L.nloads)) {
            L.mt = mt;
            L.a_slots = slots;
            L.nstages = ns;
            L.smem = sm;
            placed = true;
          }
        }
    }
    // Deep-K GEMMs (one tap, 128-row items: DeBERTa): a K chunk consumes one activation slot AND one weight step, and with
    // 0.27 us of MMA work per chunk against ~1.5 us of L2 latency the chunks in flight set the rate — give both rings the
    // same depth in chunks instead of the weight ring first (slots 3 / stages 5 -> 4 / 4 for N = 256; 6 / 6 for N = 128)
    if (!latency_mode && taps == 1 && mt == 1 && L.nkc >= 8 && !placed) {
      int best = 0, bs = 0, bn = 0;
      for (int slots = ring_min_slots; slots <= MAX_ASLOTS; ++slots)
        for (int ns = 2; ns <= MAX_STAGES; ++ns) {
          const size_t sm = ((slot * slots + 127) & ~size_t(127)) + stage_bytes * ns + kMisc;
          if (sm > size_t(SMEM_LIMIT)) continue;
          const int depth = std::min(slots, ns * L.sps);
          if (depth > best || (depth == best && slots + ns > bs + bn)) {
            best = depth;
            bs = slots;
            bn = ns;
          }
        }
      if (best > 0) {
        L.mt = mt;
        L.a_slots = bs;
        L.nstages = bn;
        L.smem = ((slot * bs + 127) & ~size_t(127)) + stage_bytes * bn + kMisc;
        placed = true;
      }
    }
    for (int ns = std::min(MAX_STAGES, std::max(2, L.nloads)); ns >= 2 && !placed; --ns) {
      for (int slots = std::min(MAX_ASLOTS, std::max(ring_min_slots, L.nkc + 1)); slots >= ring_min_slots && !placed; --slots) {
        size_t sm = ((slot * slots + 127) & ~size_t(127)) + stage_bytes * ns + kMisc;
        if (sm <= size_t(SMEM_LIMIT)) {
          L.mt = mt;
          L.a_slots = slots;
          L.nstages = ns;
          L.smem = sm;
          placed = true;
        }
      }
    }
    if (mt == 1) break;
  }
  if (!placed) fail(SBV2_ERR_UNSUPPORTED, "conv tile does not fit in shared memory");
  L.tmem_cols = pow2_at_least(2 * L.mt * L.nb);
  L.idesc = (1u << 4) | (0u << 7) | (0u << 10) | ((unsigned)(L.nb >> 3) << 17) | ((unsigned)(128 >> 4) << 24);
  // pack weights: [group][nblk][kc][tap][KC/8][NB][8]
  std::vector<uint16_t> pk(size_t(n_groups) * L.n_nblk * L.total_steps * L.nb * L.kc);
  size_t o = 0;
  for (int g = 0; g < n_groups; ++g)
    for (int nbk = 0; nbk < L.n_nblk; ++nbk)
      for (int kc = 0; kc < L.nkc; ++kc)
        for (int tap = 0; tap < taps; ++tap)
          for (int pl = 0; pl < L.kc / 8; ++pl)
            for (int n = 0; n < L.nb; ++n)
              for (int e = 0; e < 8; ++e) pk[o++] = f2h(wsel(g, nbk * L.nb + n, kc * L.kc + pl * 8 + e, tap));
  L.w = static_cast<__half*>(owner->upload_bytes(pk.data(), pk.size() * 2));
  std::vector<float> bz(size_t(cout), 0.f);
  if (bias) std::copy(bias, bias + cout, bz.begin());
  L.bias = static_cast<float*>(owner->upload_bytes(bz.data(), bz.size() * 4));
  return L;
}

int mt_slot(int mt) { return mt == 1 ? 0 : (mt == 2 ? 1 : (mt == 4 ? 2 : (mt == 8 ? 3 : 4))); }

// ---- tensor maps for the activation operand ----------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      p = nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}
struct TmapKey {
  const void* ptr;
  long long rows_tot;
  int planes, box_rows, box_planes;
  bool operator==(const TmapKey& o) const {
    return ptr == o.ptr && rows_tot == o.rows_tot && planes == o.planes && box_rows == o.box_rows && box_planes == o.box_planes;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    size_t h = std::hash<const void*>()(k.ptr);
    for (long long v : {k.rows_tot, (long long)k.planes, (long long)k.box_rows, (long long)k.box_planes}) h = h * 1000003u ^ std::hash<long long>()(v);
    return h;
  }
};
// planar fp16 buffer [planes][rows_tot][8] as {8 halves, rows_tot, planes}; box {8, box_rows, box_planes}.  Encoding costs
// a few microseconds of host time, so the maps are cached by (buffer, geometry, box); a map holds no device state.
bool activation_tmap(const __half* base, long long rows_tot, int planes, int box_rows, int box_planes, CUtensorMap* out) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || box_rows > 256 || box_planes > 256 || (reinterpret_cast<uintptr_t>(base) & 15) != 0) return false;
  static std::mutex mu;
  static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  const TmapKey key{base, rows_tot, planes, box_rows, box_planes};
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(key);
  if (it != cache.end()) {
    *out = it->second;
    return true;
  }
  const cuuint64_t dims[3] = {8, (cuuint64_t)rows_tot, (cuuint64_t)planes};
  const cuuint64_t strides[2] = {16, (cuuint64_t)rows_tot * 16};
  const cuuint32_t box[3] = {8, (cuuint32_t)box_rows, (cuuint32_t)box_planes};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap m;
  const CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<__half*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return false;
  if (cache.size() > 4096) cache.clear();
  cache.emplace(key, m);
  *out = m;
  return true;
}

void set_smem_attr() {
  static PerDeviceOnce attr_once;
  attr_once.run([&] {
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    CUDA_CHECK(cudaFuncSetAttribute(umma_conv_kernel<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
  });
}

}  // namespace

ConvLayer make_conv1d_layer(sbv2_model* owner, const HostConv& c, int dil, int mt_pref, int nb_max) {
  int shifts[1][MAX_TAPS] = {{0}};
  if (c.k > MAX_TAPS) fail(SBV2_ERR_UNSUPPORTED, "kernel size too large");
  // "same" padding as the graph builds it: left (k-1)/2 * dil (FFN even kernels pad ((k-1)/2, k/2))
  for (int j = 0; j < c.k; ++j) shifts[0][j] = (j - (c.k - 1) / 2) * dil;
  const int cin = c.d1, k = c.k;
  const float* w = c.w.data();
  return make_layer(owner, c.d1, c.d0, c.k, 1, shifts, nullptr, c.b.empty() ? nullptr : c.b.data(),
                    [=](int, int co, int ci, int tap) { return w[(size_t(co) * cin + ci) * k + tap]; }, mt_pref, nb_max);
}

ConvLayer make_gated_conv1d_layer(sbv2_model* owner, const HostConv& c, int dil, int mt_pref, int* gate_half, std::vector<int>* perm) {
  const int H = c.d0 / 2;
  if (c.d0 % 2 != 0 || H % 16 != 0) fail(SBV2_ERR_UNSUPPORTED, "gated conv: output channels must be 2 * (multiple of 16)");
  int hb = 0;
  for (int v = std::min(H, 128) / 16 * 16; v >= 16; v -= 16)
    if (H % v == 0) {
      hb = v;
      break;
    }
  if (hb == 0) fail(SBV2_ERR_UNSUPPORTED, "gated conv: no N block divides the hidden size");
  perm->resize(size_t(2) * H);
  for (int j = 0; j < H / hb; ++j)
    for (int i = 0; i < hb; ++i) {
      (*perm)[size_t(j) * 2 * hb + i] = j * hb + i;           // tanh half
      (*perm)[size_t(j) * 2 * hb + hb + i] = H + j * hb + i;  // sigmoid half
    }
  HostConv p = c;
  const size_t per_out = size_t(c.d1) * c.k;
  for (int i = 0; i < 2 * H; ++i) {
    std::copy(c.w.begin() + size_t((*perm)[size_t(i)]) * per_out, c.w.begin() + size_t((*perm)[size_t(i)] + 1) * per_out, p.w.begin() + size_t(i) * per_out);
    if (!c.b.empty()) p.b[size_t(i)] = c.b[size_t((*perm)[size_t(i)])];
  }
  ConvLayer L = make_conv1d_layer(owner, p, dil, mt_pref, 2 * hb);
  if (L.nb != 2 * hb) fail(SBV2_ERR_INTERNAL, "gated conv: unexpected N block");
  *gate_half = hb;
  return L;
}

ConvLayer make_split_conv1d_layer(sbv2_model* owner, const HostConv& c, int dil, int mt_pref, int terms, int nb_max) {
  // [Cout][n*Cin][k]: terms = 2: input planes [h0 | h1 | h0] meet weights [w0 | w0 | w1];
  // terms = 3: [h0 | h1 | h2 | h0 | h1 | h0] meet [w0 | w0 | w0 | w1 | w1 | w2]
  const int nblk = terms == 3 ? 6 : 3;
  static const int wsel2[3] = {0, 0, 1}, wsel3[6] = {0, 0, 0, 1, 1, 2};
  const int* wsel = terms == 3 ? wsel3 : wsel2;
  HostConv s3;
  s3.d0 = c.d0;
  s3.d1 = nblk * c.d1;
  s3.k = c.k;
  s3.b = c.b;
  s3.w.resize(size_t(s3.d0) * s3.d1 * s3.k);
  // weight scale: the largest power of two with max|w| * scale <= 2^13 (fp16 overflows at 65504)
  float wmax = 0.f;
  for (float v : c.w) wmax = std::max(wmax, std::fabs(v));
  int wexp = 0;
  if (wmax > 0.f) {
    std::frexp(wmax, &wexp);  // wmax = m * 2^wexp, m in [0.5, 1)
    wexp = 13 - wexp;
  }
  const float wscale = std::ldexp(1.0f, wexp);
  // activations with |x| < 4095 stay finite in fp16: 16 * 4094.97 rounds to 65504, 16 * 4095 = 65520 rounds to infinity
  const float in_scale = 16.f;
  for (int co = 0; co < c.d0; ++co)
    for (int ci = 0; ci < c.d1; ++ci)
      for (int j = 0; j < c.k; ++j) {
        const float w = c.w[(size_t(co) * c.d1 + ci) * c.k + j] * wscale;
        float wt[3];
        wt[0] = __half2float(__float2half_rn(w));
        wt[1] = __half2float(__float2half_rn(w - wt[0]));
        wt[2] = __half2float(__float2half_rn(w - wt[0] - wt[1]));
        for (int q = 0; q < nblk; ++q) s3.w[(size_t(co) * s3.d1 + size_t(q) * c.d1 + ci) * c.k + j] = wt[wsel[q]];
      }
  s3.b.clear();  // the bias is added after the accumulator has been scaled back: keep it out of the packed layer ...
  ConvLayer L = make_conv1d_layer(owner, s3, dil, mt_pref, nb_max);
  if (!c.b.empty()) L.bias = owner->upload_f32(c.b);  // ... and attach the unscaled one
  L.in_scale = in_scale;
  L.out_scale = 1.0f / (in_scale * wscale);
  return L;
}

ConvLayer make_upsample_layer(sbv2_model* owner, const HostConv& c, int u, int mt_pref) {
  // out[u*q + r] = bias + sum_m sum_ci w[ci][co][rr + u*m] * in[q + cc - m],  s = r + pad, rr = s % u, cc = s / u
  const int k = c.k, pad = (k - u) / 2, taps = k / u;
  if (u > UMMA_MAX_GROUPS || taps > MAX_TAPS) fail(SBV2_ERR_UNSUPPORTED, "upsample rate / kernel not supported by the tensor-core plan");
  int shifts[UMMA_MAX_GROUPS][MAX_TAPS] = {{0}};
  int offs[UMMA_MAX_GROUPS] = {0};
  int rrs[UMMA_MAX_GROUPS] = {0};
  for (int r = 0; r < u; ++r) {
    const int s = r + pad;
    rrs[r] = s % u;
    for (int m = 0; m < taps; ++m) shifts[r][m] = s / u - m;
    offs[r] = r;
  }
  const int cout = c.d1;
  const float* w = c.w.data();
  std::vector<int> rr(rrs, rrs + UMMA_MAX_GROUPS);
  return make_layer(owner, c.d0, c.d1, taps, u, shifts, offs, c.b.empty() ? nullptr : c.b.data(),
                    [=](int g, int co, int ci, int tap) { return w[(size_t(ci) * cout + co) * k + rr[g] + u * tap]; }, mt_pref);
}

long long* g_trace = nullptr;  // debug hook, see sbv2_debug_conv_trace

void launch_umma(const LaunchCtx& ctx, const ConvLayer& L, const Geom& gi, const Geom& go, const ConvCall& c, int n_utt) {
  set_smem_attr();
  UmmaConvArgs a;
  a.in = c.in;
  a.in_plane_stride = gi.rows_tot * 8;
  {
    // one tensor-map request per activation chunk when the tile (rows incl. halo) fits a TMA box; SBV2_B200_TMAP=0 keeps
    // the per-plane bulk copies
    static int tmap_on = -1;
    if (tmap_on < 0) {
      const char* e = getenv("SBV2_B200_TMAP");
      tmap_on = !(e && e[0] == '0');
    }
    const int ra = 128 * L.mt + L.halo_lo + L.halo_hi;
    a.use_tmap = c.tmap && tmap_on && ra <= 256 && activation_tmap(c.in, gi.rows_tot, L.cin / 8, ra, L.kc / 8, &a.tmap) ? 1 : 0;
  }
  a.out = c.out;
  a.out_plane_stride = go.rows_tot * 8;
  a.residual = c.residual;
  a.accum = c.accum;
  a.w = L.w;
  a.bias = L.bias;
  a.bias_utt = c.bias_utt;
  a.bias_utt_ld = c.bias_utt_ld > 0 ? c.bias_utt_ld : L.n_nblk * L.nb;
  a.gate_half = c.gate_half;
  if (c.gate_half > 0 && (2 * c.gate_half != L.nb || c.residual || c.accum || c.rm_out || !c.out || c.out_mul != 1 || L.n_groups != 1))
    fail(SBV2_ERR_INTERNAL, "gated conv: unsupported epilogue combination");
  const int slot = mt_slot(L.mt);
  a.tile_prefix = gi.d_prefix[slot];
  a.pstart_in = gi.d_pstart;
  a.pstart_out = go.d_pstart;
  a.len = gi.d_len;
  a.n_utt = n_utt;
  a.cin = L.cin;
  a.nb = L.nb;
  a.n_nblk = L.n_nblk;
  a.b_resident = L.b_resident;
  a.taps = L.taps;
  a.kc = L.kc;
  a.nkc = L.nkc;
  a.mt = L.mt;
  a.sps = L.sps;
  a.nstages = L.nstages;
  a.nloads = L.nloads;
  a.total_steps = L.total_steps;
  a.a_slots = L.a_slots;
  a.n_groups = L.n_groups;
  for (int g = 0; g < UMMA_MAX_GROUPS; ++g) {
    a.group_out_off[g] = L.group_out_off[g];
    for (int i = 0; i < MAX_TAPS; ++i) a.tap_shift[g * MAX_TAPS + i] = L.tap_shift[g][i];
  }
  a.halo_lo = L.halo_lo;
  a.halo_hi = L.halo_hi;
  a.out_mul = c.out_mul;
  a.out_off = c.out_off;
  a.act_out = c.act_out;
  a.act_slope = c.act_out == ACT_LRELU ? 0.1f : (c.act_out == ACT_LRELU01 ? 0.01f : (c.act_out == ACT_RELU ? 0.f : 1.f));
  a.has_res = c.residual ? (c.residual2 ? 3 : 1) : 0;
  a.residual2 = c.residual2;
  a.residual3 = c.residual3;
  a.out_div = c.out_div;
  a.accum_mode = c.accum_mode;
  a.act_on_accum = c.act_on_accum ? 1 : 0;
  a.accum_div = c.accum_div;
  a.tmem_cols = L.tmem_cols;
  a.idesc = L.idesc;
  a.rm_out = c.rm_out;
  a.rm_scale = L.out_scale;
  a.rm_ld = c.rm_ld;
  a.rm_start = c.rm_start;
  a.split_out = c.split_out;
  a.split_npl = L.cout / 8;
  a.split_scale = c.split_scale;
  a.trace = g_trace;
  if (c.report) *c.report = UmmaLaunchReport{};
  if (gi.n_tiles[slot] <= 0) return;
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    CUDA_CHECK(cudaGetDevice(&dev));
    CUDA_CHECK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  // Thread-block clusters with multicast weight stages (SBV2_B200_CLUSTER = 1 / 2 / 4).  OFF by default: measured on the
  // bench workload the lock-step of the cluster (every CTA waits for all peers' slices and all peers' MMAs per stage) costs
  // more than the divided L2 -> SM weight traffic saves — decoder 20.05 / 20.73 / 27.94 ms, flow 7.44 / 7.84 / 8.84 ms
  // for 1 / 2 / 4 CTAs per cluster (profiles/r2_cluster_multicast.log); results are identical in all three modes
  // (tools/umma_conv_check.py).  Streaming layers only: resident weights are fetched once per CTA anyway.
  // ON (2 CTAs) where it was measured to pay — the DeBERTa GEMMs ask for it through ConvCall::cluster: 32 x 128 tokens
  // 12.9 -> 12.0 ms exact, 6.2 -> 6.0 ms fp16 (4 CTAs: 14.0 / 7.0 ms); the environment variable overrides either way.
  static int cluster_pref = -1;  // 0: SBV2_B200_CLUSTER not set
  if (cluster_pref < 0) {
    const char* e = getenv("SBV2_B200_CLUSTER");
    cluster_pref = e ? atoi(e) : 0;
    if (cluster_pref != 0 && cluster_pref != 1 && cluster_pref != 2 && cluster_pref != 4) cluster_pref = 1;
  }
  int nc = L.b_resident ? 1 : (cluster_pref > 0 ? cluster_pref : (c.cluster == 2 || c.cluster == 4 ? c.cluster : 1));
  while (nc > 1 && (gi.n_tiles[slot] < nc || (size_t(L.nb) * L.kc * 2) % (size_t(16) * nc) != 0)) nc >>= 1;
  if (cluster_pref == 0 && nc > 1) {
    // a caller's preference must not turn one wave into two (dummy tiles of a ragged last cluster count as CTAs):
    // three short sentences, 144 items -> 192 clustered CTAs, measured 5.5 -> 6.1 ms
    const long long plain = (long long)gi.n_tiles[slot] * L.n_nblk * L.n_groups;
    const long long clustered = (long long)((gi.n_tiles[slot] + nc - 1) / nc) * nc * L.n_nblk * L.n_groups;
    if (clustered > num_sms && plain < 2LL * num_sms) nc = 1;
  }
  // CTA pairs (cta_group::2, SBV2_B200_PAIR2=1 or ConvCall::pair): two adjacent N blocks of the layer's packing form the N
  // of one M = 256 MMA, each CTA of the pair streams one of them.  Needs an even number of N blocks, N = 2 * nb <= 256 and
  // both accumulator sets (2 * mt * N columns) in TMEM.
  static int pair_env = -1;
  if (pair_env < 0) {
    const char* e = getenv("SBV2_B200_PAIR2");
    pair_env = e ? atoi(e) : 0;
  }
  const bool pair = (c.pair || pair_env == 1) && pair_env != 2 && !L.b_resident && L.n_groups == 1 && c.gate_half == 0 && L.n_nblk % 2 == 0 &&
                    2 * L.nb <= 256 && 4 * L.mt * L.nb <= 512 && gi.n_tiles[slot] >= 2;
  if (pair) {
    nc = 2;
    a.nb = 2 * L.nb;
    a.n_nblk = L.n_nblk / 2;
    a.tmem_cols = pow2_at_least(4 * L.mt * L.nb);
    a.idesc = (1u << 4) | ((unsigned)(a.nb >> 3) << 17) | ((unsigned)(256 >> 4) << 24);  // M = 256 across the pair
  }
  // split-K (below) takes precedence over multicast clusters: it is decided on the single-CTA item count
  int splitk = 1;
  {
    static int splitk_env = -1;
    if (splitk_env < 0) {
      const char* e = getenv("SBV2_B200_SPLITK");
      splitk_env = e ? atoi(e) : 1;
    }
    const int n_items1 = gi.n_tiles[slot] * L.n_nblk * L.n_groups;
    if (c.splitk && splitk_env != 0 && !pair && L.mt == 1 && !L.b_resident && L.n_groups == 1 && c.gate_half == 0 && L.nkc >= 8 &&
        size_t(128) * (L.nb + 4) * 4 <= size_t(L.a_slots) * (L.kc / 8) * (128 + L.halo_lo + L.halo_hi) * 16) {
      for (int sk = 8; sk >= 2 && splitk == 1; sk >>= 1)
        if (n_items1 * sk <= num_sms && L.nkc % sk == 0 && L.nkc / sk >= 2) splitk = sk;
    }
    if (splitk > 1) nc = 1;
  }
  a.cluster = nc;
  a.n_tiles = gi.n_tiles[slot];
  a.n_items = ((gi.n_tiles[slot] + nc - 1) / nc) * a.n_nblk * L.n_groups;  // cluster items
  // Split-K over a cluster (ConvCall::splitk: DeBERTa's GEMMs when a call has few tokens).  With 16-64 items each CTA
  // walks the whole K alone: K / 16 MMAs in a row and K * nb * 2 bytes of weights through one SM's few stages in flight
  // (one 7-token sentence: 40 us per GEMM for 1-2 us of work).  S CTAs per item divide both.  SBV2_B200_SPLITK=0: off.
  dim3 grid(std::min(a.n_items, num_sms / nc) * nc);
  if (splitk > 1) {
    nc = splitk;
    a.cluster = splitk;
    grid = dim3(a.n_items * splitk);  // one item per cluster
  }
  void (*kernel)(UmmaConvArgs) = nullptr;
  const int variant =
      (c.gate_half > 0 ? 1 : 0) | (pair ? 8 : (splitk > 1 ? 16 : (nc > 1 ? 2 : 0))) | ((c.rm_out != nullptr || c.split_out != nullptr) ? 4 : 0);
  if (c.report) *c.report = UmmaLaunchReport{variant, nc, splitk, a.use_tmap};
  switch (variant) {
    case 0: kernel = umma_conv_kernel<0>; break;
    case 1: kernel = umma_conv_kernel<1>; break;
    case 2: kernel = umma_conv_kernel<2>; break;
    case 3: kernel = umma_conv_kernel<3>; break;
    case 4: kernel = umma_conv_kernel<4>; break;
    case 6: kernel = umma_conv_kernel<6>; break;
    case 8: kernel = umma_conv_kernel<8>; break;
    case 12: kernel = umma_conv_kernel<12>; break;
    case 16: kernel = umma_conv_kernel<16>; break;
    case 20: kernel = umma_conv_kernel<20>; break;
    default: fail(SBV2_ERR_INTERNAL, "conv kernel: unsupported epilogue combination");
  }
  launch_pdl_cluster(ctx.pdl && !pair, nc, kernel, grid, dim3(NUM_THREADS), L.smem, ctx.stream, a);
  ctx.count();
}

void launch_zero_gaps(const LaunchCtx& ctx, __half* buf, int C, const Geom& g, int n_utt) {
  dim3 grid(n_utt + 1, C / 8);
  zero_gaps_kernel<<<grid, 64, 0, ctx.stream>>>(buf, g.rows_tot * 8, g.d_pstart, g.d_len, n_utt, GAP);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

BatchGeom build_geoms(sbv2_model* owner, DBuf& dev, PinnedBuf& pin, const std::vector<int>& ystart, const std::vector<int>& ylen,
                      const std::vector<int>& muls, const std::vector<std::vector<int>>* extra_heights, bool pin_idle,
                      const std::vector<long long>* wstart) {
  const int B = int(ylen.size());
  BatchGeom bg;
  bg.g.resize(muls.size());
  // ints: per geom: pstart[B], len[B], prefix x5 [(B+1)*5], extra prefixes [(B+1) each]; then ystart[B], wstart[B]
  std::vector<size_t> goff(muls.size() + 1, 0);
  for (size_t s = 0; s < muls.size(); ++s) {
    const size_t n_extra = extra_heights && s < extra_heights->size() ? (*extra_heights)[s].size() : 0;
    goff[s + 1] = goff[s] + size_t(2) * B + size_t(5 + n_extra) * (B + 1);
  }
  const size_t total = goff.back() + size_t(3) * B;  // + ystart, wstart, order
  // the pinned blob of the previous run may still be in flight on the stream
  if (!pin_idle) CUDA_CHECK(cudaStreamSynchronize(owner->stream));
  pin.ensure(total * 4);
  int* h = pin.as<int>();
  for (size_t s = 0; s < muls.size(); ++s) {
    Geom& G = bg.g[s];
    G.mul = muls[s];
    G.pstart.resize(B);
    G.len.resize(B);
    long long r = GAP;
    int* hp = h + goff[s];
    for (int b = 0; b < B; ++b) {
      long long l = (long long)ylen[b] * muls[s];
      if (r + l + GAP + TAIL_ROWS > 2000000000LL) fail(SBV2_ERR_INVALID_ARGUMENT, "batch too long for the decoder's 32-bit row index");
      G.pstart[b] = int(r);
      G.len[b] = int(l);
      G.max_len = std::max(G.max_len, int(l));
      hp[b] = int(r);
      hp[B + b] = int(l);
      r += l + GAP;
    }
    G.rows_tot = r + TAIL_ROWS;
    auto fill = [&](int* pf, int tm) {
      int acc = 0;
      for (int b = 0; b < B; ++b) {
        pf[b] = acc;
        acc += (G.len[b] + tm - 1) / tm;
      }
      pf[B] = acc;
      return acc;
    };
    for (int slot = 0; slot < 5; ++slot) G.n_tiles[slot] = fill(hp + 2 * B + slot * (B + 1), 128 << slot);
    if (extra_heights && s < extra_heights->size()) {
      for (size_t e = 0; e < (*extra_heights)[s].size(); ++e) {
        const int hgt = (*extra_heights)[s][e];
        int n = fill(hp + 2 * B + (5 + int(e)) * (B + 1), hgt);
        G.extra[hgt] = std::make_pair(static_cast<const int*>(nullptr), n);
      }
    }
  }
  int* tail = h + goff.back();
  long long hop = muls.back();
  for (int b = 0; b < B; ++b) {
    tail[b] = ystart[b];
    const long long ws = wstart ? (*wstart)[size_t(b)] : (long long)ystart[b] * hop;
    if (ws < 0 || ws > 2000000000LL) fail(SBV2_ERR_INVALID_ARGUMENT, "waveform offset exceeds the 32-bit sample index");
    tail[B + b] = int(ws);
  }
  {
    // utterances by decreasing length: kernels with one CTA per (utterance, tile) start the long ones first
    std::vector<int> order(B);
    for (int b = 0; b < B; ++b) order[b] = b;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return ylen[x] > ylen[y]; });
    for (int b = 0; b < B; ++b) tail[2 * B + b] = order[b];
  }
  dev.stream = owner->stream;
  dev.ensure(total * 4);
  CUDA_CHECK(cudaMemcpyAsync(dev.p, h, total * 4, cudaMemcpyHostToDevice, owner->stream));
  const int* d = dev.as<int>();
  for (size_t s = 0; s < muls.size(); ++s) {
    Geom& G = bg.g[s];
    const int* dp = d + goff[s];
    G.d_pstart = dp;
    G.d_len = dp + B;
    for (int slot = 0; slot < 5; ++slot) G.d_prefix[slot] = dp + 2 * B + slot * (B + 1);
    if (extra_heights && s < extra_heights->size())
      for (size_t e = 0; e < (*extra_heights)[s].size(); ++e) G.extra[(*extra_heights)[s][e]].first = dp + 2 * B + (5 + int(e)) * (B + 1);
  }
  bg.d_ystart = d + goff.back();
  bg.d_wstart = bg.d_ystart + B;
  bg.d_order = bg.d_ystart + 2 * B;
  return bg;
}

void launch_to_planar(const LaunchCtx& ctx, __half* out, const float* in, int in_ld, int C, const int* d_start, const Geom& g,
                      int n_utt, int act) {
  dim3 block(std::min(32, C / 8), 8);
  dim3 grid((g.max_len + 7) / 8, n_utt);
  to_planar_kernel<<<grid, block, 0, ctx.stream>>>(out, g.rows_tot * 8, in, in_ld, C, d_start, g.d_pstart, g.d_len, act);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

void launch_planar_cast(const LaunchCtx& ctx, __half* out, const float* in, int C, const Geom& g, int n_utt) {
  if (g.max_len <= 0 || n_utt <= 0) return;
  dim3 grid((g.max_len + 255) / 256, C / 8, n_utt);
  planar_cast_kernel<<<grid, 256, 0, ctx.stream>>>(out, in, g.rows_tot * 8, g.d_pstart, g.d_len);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

void launch_split_planar(const LaunchCtx& ctx, __half* out, const float* in, int in_ld, int C, const int* d_start, const Geom& g,
                         int n_utt, int terms, float in_scale) {
  dim3 block(std::min(32, C / 8), 8);
  dim3 grid((g.max_len + 7) / 8, n_utt);
  if (terms == 3)
    split_planar_kernel<3><<<grid, block, 0, ctx.stream>>>(out, g.rows_tot * 8, in, in_ld, C, d_start, g.d_pstart, g.d_len, in_scale);
  else
    split_planar_kernel<2><<<grid, block, 0, ctx.stream>>>(out, g.rows_tot * 8, in, in_ld, C, d_start, g.d_pstart, g.d_len, in_scale);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

void launch_from_planar(const LaunchCtx& ctx, float* out, const __half* in, int C, const int* d_start, const Geom& g, int n_utt) {
  dim3 block(std::min(32, C / 8), 8);
  dim3 grid((g.max_len + 7) / 8, n_utt);
  from_planar_kernel<<<grid, block, 0, ctx.stream>>>(out, in, g.rows_tot * 8, C, d_start, g.d_pstart, g.d_len);
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

}  // namespace sbv2
