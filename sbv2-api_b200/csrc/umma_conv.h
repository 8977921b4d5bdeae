// Tensor-core (tcgen05 / TMEM) implicit-GEMM convolution used by the HiFi-GAN decoder and the
// transformer flow.  See umma_conv.cu for the kernel and the data layout ("planar fp16").
#pragma once
#include <cuda_fp16.h>

#include <map>
#include <vector>

#include "common.h"
#include "kernels.h"

struct sbv2_model;

namespace sbv2 {

constexpr int UMMA_GAP = 32;         // zero rows around each utterance (>= largest halo: 5*(11-1)/2 = 25)
constexpr int UMMA_TAIL_ROWS = 2304;  // slack rows after the last utterance (a tile may over-read)
constexpr int UMMA_MAX_TAPS = 16;
constexpr int UMMA_MAX_GROUPS = 8;    // polyphase groups of one launch (ConvTranspose phases)

struct HostConv {
  std::vector<float> w, b;  // PyTorch layout: Conv1d [d0=Cout, d1=Cin, k]; ConvTranspose1d [d0=Cin, d1=Cout, k]
  int d0 = 0, d1 = 0, k = 1;
};

struct DecoderHostWeights {
  HostConv pre, cond, post;
  std::vector<HostConv> ups;
  std::vector<int> up_u;
  std::vector<std::vector<HostConv>> res_c1, res_c2;  // [resblock][layer]
  std::vector<std::vector<int>> res_dil;
  int per = 3;  // resblocks per stage
  int gin = 512;
};

// One convolution prepared for the tensor-core kernel (weights repacked to fp16 on the device).
struct ConvLayer {
  __half* w = nullptr;   // [nblk][kc][tap][KC/8][NB][8]
  float* bias = nullptr; // [cout]
  int cin = 0, cout = 0, nb = 0, n_nblk = 1, taps = 1, kc = 64, nkc = 1, mt = 1, sps = 1, nstages = 2, nloads = 1, total_steps = 1;
  int a_slots = 1;
  int b_resident = 0;  // all weight steps stay in shared memory for the whole (persistent) kernel
  // groups: independent weight sets sharing the input tile (the u phases of a ConvTranspose1d); group g uses
  // row shifts tap_shift[g][*] and writes output rows t*out_mul + group_out_off[g]
  int n_groups = 1;
  int tap_shift[UMMA_MAX_GROUPS][UMMA_MAX_TAPS] = {{0}};
  int group_out_off[UMMA_MAX_GROUPS] = {0};
  int halo_lo = 0, halo_hi = 0;
  size_t smem = 0;
  int tmem_cols = 32;
  unsigned idesc = 0;
  float in_scale = 1.f, out_scale = 1.f;  // split layers: power-of-two operand scaling (see make_split_conv1d_layer)
};

// Conv1d weight [Cout][Cin][k], "same" padding, dilation dil.
// mt_pref: preferred number of 128-row tiles per work item; nb_max: largest N block (output channels per item).  A work
// item streams its N block's weights once, so few-row problems (flow, text encoder) want nb_max = 128 and mt_pref = 2:
// twice the rows per weight byte read from L2.
ConvLayer make_conv1d_layer(sbv2_model* owner, const HostConv& c, int dil, int mt_pref, int nb_max = 256);
// Conv1d(C -> 2H) of a WaveNet layer whose output feeds tanh(first H) * sigmoid(last H): output channels are permuted so
// that every N block of 2 * hb channels holds [tanh j*hb .. | sigmoid j*hb ..] and the gate is fused into the epilogue
// (ConvCall::gate_half = *gate_half).  perm (size 2H) receives the permutation: packed channel i = original perm[i]
// (apply it to the conditioning vector that goes in as ConvCall::bias_utt).
ConvLayer make_gated_conv1d_layer(sbv2_model* owner, const HostConv& c, int dil, int mt_pref, int* gate_half, std::vector<int>* perm);
// ConvTranspose1d weight [Cin][Cout][k], stride u, pad (k-u)/2 as u polyphase groups of k/u taps (one launch;
// launch with ConvCall::out_mul = u)
ConvLayer make_upsample_layer(sbv2_model* owner, const HostConv& c, int u, int mt_pref);

// One time resolution of one packed batch.
struct Geom {
  int mul = 1;
  long long rows_tot = 0;
  std::vector<int> pstart, len;
  const int* d_pstart = nullptr;
  const int* d_len = nullptr;
  const int* d_prefix[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // tiles of 128 * {1, 2, 4, 8, 16} rows
  int n_tiles[5] = {0, 0, 0, 0, 0};
  // tile tables for other tile heights (fused ResBlock pairs use 128*MT - 2*halo rows per tile)
  std::map<int, std::pair<const int*, int>> extra;  // height -> (device prefix [n+1], number of tiles)
  int max_len = 0;
};
struct BatchGeom {
  std::vector<Geom> g;
  const int* d_ystart = nullptr;  // first row of each utterance in the packed fp32 [rows, C] matrices
  const int* d_wstart = nullptr;  // sample offset of each utterance in the waveform buffer
  const int* d_order = nullptr;   // utterance indices by decreasing length
};
struct DBuf;
struct PinnedBuf;
// The tables are staged in `pin` and copied to `dev` asynchronously.  `pin_idle`: the caller guarantees that the previous
// copy out of `pin` has completed (it synchronised the stream since); otherwise build_geoms synchronises the stream itself.
BatchGeom build_geoms(sbv2_model* owner, DBuf& dev, PinnedBuf& pin, const std::vector<int>& ystart, const std::vector<int>& ylen,
                      const std::vector<int>& muls, const std::vector<std::vector<int>>* extra_heights = nullptr, bool pin_idle = false,
                      const std::vector<long long>* wstart = nullptr /* sample offset of each utterance in the waveform buffer */);

// Conv1d evaluated to ~fp32 accuracy on the fp16 tensor cores by splitting both operands into fp16 terms
// (x = h0 + h1 [+ h2], w = w0 + w1 [+ w2]) and stacking the cross products along K:
//   terms = 2: h0 w0 + h1 w0 + h0 w1                               (3*Cin input channels, ~2^-21 relative error)
//   terms = 3: h0 w0 + h1 w0 + h2 w0 + h0 w1 + h1 w1 + h0 w2        (6*Cin input channels, fp32-level error)
// Both operands are scaled by powers of two first (weights so that max|w| ~ 2^13, activations by ConvLayer::in_scale)
// so that the low-order terms stay out of fp16's subnormal range; the fp32 row-major epilogue multiplies the
// accumulator by ConvLayer::out_scale = 1 / (in_scale * weight scale) — exact.
// The layer's input is the planar tensor written by launch_split_planar with the same `terms` and in_scale.
ConvLayer make_split_conv1d_layer(sbv2_model* owner, const HostConv& c, int dil, int mt_pref, int terms, int nb_max = 256);
// packed fp32 [rows, in_ld] (first C columns) * in_scale -> planar fp16 split terms in plane blocks [h0 | h1 | h0]
// (terms = 2) or [h0 | h1 | h2 | h0 | h1 | h0] (terms = 3), each block C / 8 planes; gap rows are not written
void launch_split_planar(const LaunchCtx& ctx, __half* out, const float* in, int in_ld, int C, const int* d_start, const Geom& g,
                         int n_utt, int terms, float in_scale);
enum UAccum { UACC_NONE = 0, UACC_SET = 1, UACC_ADD = 2, UACC_FINAL = 3 };
// What launch_umma chose for one call (ConvCall::report): the umma_conv_kernel VARIANT, CTAs per thread-block cluster
// (multicast, CTA pair or split-K; 1: none), the split-K factor S (1: none) and whether activation chunks came by tensor
// map.  All zero when the launch had no rows.
struct UmmaLaunchReport {
  int variant = 0, cluster = 0, splitk = 0, tmap = 0;
};
struct ConvCall {
  const __half* in = nullptr;
  __half* out = nullptr;          // planar fp16 (optional)
  const __half* residual = nullptr;  // planar fp16 stored post-lrelu(0.1): x = y >= 0 ? y : 10 y is added
  const __half* residual2 = nullptr;  // MRF: two more post-lrelu terms (both or neither), summed first, then
  const __half* residual3 = nullptr;  //      (r2 + r3 + v) / out_div before the activation
  float out_div = 1.f;
  float* accum = nullptr;         // planar fp32 (geometry of out)
  int accum_mode = UACC_NONE;
  float accum_div = 1.f;
  int act_out = ACT_NONE;         // ACT_NONE / ACT_RELU / ACT_LRELU / ACT_LRELU01 / ACT_GELU
  bool act_on_accum = false;      // apply act_out before the fp32 accumulate/store instead of on the fp16 output
  const float* bias_utt = nullptr;
  int bias_utt_ld = 0;            // floats between consecutive utterances of bias_utt (0: the layer's cout)
  // WaveNet gate (make_gated_conv1d_layer): every N block holds [tanh half | sigmoid half] of gate_half channels each;
  // out (planar fp16, cout / 2 channels) = tanh(.) * sigmoid(.); no residual / accumulate / row-major output
  int gate_half = 0;
  int out_mul = 1, out_off = 0;
  // fp32 row-major output [packed rows, rm_ld] instead of the planar ones (text encoder): packed row = rm_start[b] + t;
  // act_out ACT_NONE / ACT_RELU / ACT_GELU only
  float* rm_out = nullptr;
  int rm_ld = 0;
  const int* rm_start = nullptr;
  // and / or the same values (bias and activation applied) written as the split-planar operand [h0 | h1 | h0] of the next
  // split layer (geometry `go`, cout / 8 planes per block): fuses launch_split_planar into the producing GEMM
  __half* split_out = nullptr;
  float split_scale = 16.f;
  // activation chunks by one tensor-map TMA request (cp.async.bulk.tensor.3d) instead of one bulk copy per plane, when the
  // tile incl. halo fits a 256-row box.  Measured: DeBERTa one sentence 6.8 -> 6.4 ms (exact), 2.8 -> 2.7 ms (fp16); the
  // synthesizer's few-rows layers lose 4 % (the box always carries all rows of the tile, the bulk copies only the valid
  // ones), batches are unchanged — so DeBERTa asks for it and the synthesizer does not.
  bool tmap = false;
  // thread-block clusters of 2 / 4 CTAs with multicast weight stages (0: none unless SBV2_B200_CLUSTER says otherwise)
  int cluster = 0;
  // run as CTA pairs (tcgen05 cta_group::2, M = 256) when the layer's packing allows it (see launch_umma)
  bool pair = false;
  // split K over a thread-block cluster when the launch has few items (see launch_umma): the fp32 sums are formed in a
  // different order than without the split, so callers that promise batch == single results bit for bit must not ask
  bool splitk = false;
  // tests: receives what launch_umma chose (null in production calls)
  UmmaLaunchReport* report = nullptr;
};
void launch_umma(const LaunchCtx& ctx, const ConvLayer& L, const Geom& gi, const Geom& go, const ConvCall& c, int n_utt);
void launch_zero_gaps(const LaunchCtx& ctx, __half* buf, int C, const Geom& g, int n_utt);
// planar fp32 -> planar fp16 over the first C channels (utterance rows only; 32-byte loads, 16-byte stores)
void launch_planar_cast(const LaunchCtx& ctx, __half* out, const float* in, int C, const Geom& g, int n_utt);
// packed fp32 [rows, in_ld] (first C columns) -> planar fp16
void launch_to_planar(const LaunchCtx& ctx, __half* out, const float* in, int in_ld, int C, const int* d_start, const Geom& g,
                      int n_utt, int act);
void launch_from_planar(const LaunchCtx& ctx, float* out, const __half* in, int C, const int* d_start, const Geom& g, int n_utt);

// A fused ResBlock1 pair (umma_pair.cu): out = conv2(lrelu(conv1(in) + b1)) + b2 + x, the intermediate stays on chip.
struct PairLayer {
  __half* w1 = nullptr;  // [kc][tap][KC/8][C][8]
  __half* w2 = nullptr;
  float* bias1 = nullptr;
  float* bias2 = nullptr;
  int c = 0, taps = 1, kc = 16, nkc = 1, mt = 1, t1rows = 128, t1pitch = 144, out_rows = 128, h1 = 0, h2 = 0;
  int shift1[UMMA_MAX_TAPS] = {0};
  int sps = 1, nstages = 1, nloads = 1, total_steps = 1, a_slots = 2, b_resident = 0;
  size_t smem = 0;
  int tmem_cols = 512;
  unsigned idesc = 0;
};
struct PairCall {
  const __half* in = nullptr;  // post-lrelu planar fp16; also the residual.  Must not alias out.
  __half* out = nullptr;
  const __half* residual2 = nullptr;  // as ConvCall
  const __half* residual3 = nullptr;
  float out_div = 1.f;
  int act_out = ACT_LRELU;
};
// false when the pair does not fit the fused plan (channel count, taps, shared memory); c1 has dilation dil, c2 dilation 1
bool make_pair_layer(sbv2_model* owner, const HostConv& c1, int dil, const HostConv& c2, PairLayer* out);
// g.extra must hold the tile table for L.out_rows (build_geoms extra_heights)
void launch_umma_pair(const LaunchCtx& ctx, const PairLayer& L, const Geom& g, const PairCall& c, int n_utt);

struct UmmaDecoder;
UmmaDecoder* umma_decoder_create(const DecoderHostWeights& w, sbv2_model* owner);
void umma_decoder_free(UmmaDecoder* d);
// z: packed [Ny, Cin] fp32 (time-major), g: [B, gin] fp32, wave: fp32 (all device).  Utterance b's samples start at
// wave[wstart[b]] (null: back to back, ystart[b] * hop).  The caller must have synchronised the owner's stream since the
// previous umma_decoder_run of this decoder (its pinned geometry blob is rewritten without a further synchronisation).
void umma_decoder_run(UmmaDecoder* d, sbv2_model* owner, const float* z, const float* g, int B,
                      const std::vector<int>& ystart, const std::vector<int>& ylen, float* wave,
                      const std::vector<long long>* wstart = nullptr);
// The decoder's conv_post: wave[wstart[b] + t] = tanh(sum_j sum_c w[c][j] * x[t + j - (k-1)/2][c]) for t < len[b] of
// geometry g.  x: planar fp16, already lrelu(0.01)-activated, zero gap rows (the kernels read the halo without a bounds
// test).  d_w: device fp32 [C][k]; w_host: the same values, which the 16 x 7 kernel takes as constant-bank operands.
// force_generic: run the generic kernel at 16 x 7 too (it sums in the same order: bit-identical results).
void launch_dec_post_planar(const LaunchCtx& ctx, float* wave, const __half* x, const Geom& g, const int* d_wstart, int n_utt,
                            const float* d_w, const std::vector<float>& w_host, int C, int k, bool force_generic);

}  // namespace sbv2
