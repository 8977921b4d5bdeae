// Unit-test hooks of the synthesizer kernels between the text encoder and the decoder: the flow's window attention
// (tensor-core and planar CUDA-core), the text encoder's fp32 attention, the inverse spline of the stochastic duration
// predictor, the length regulator, the HiFi-GAN decoder's tensor-core layers and conv_post, the split-fp16 layers, the
// WaveNet gate and DeBERTa's kernels.  Linked into libsbv2_b200_debug.so only (build.py DEBUG_ONLY).  Every hook runs on
// its own stream, takes host arrays and returns host arrays before it returns; tests/test_gpu_synth_kernels.py,
// tests/test_gpu_decoder_kernels.py and tests/test_gpu_split_gemm.py compare the results with float64 references.
#include <cuda_fp16.h>

#include <algorithm>
#include <climits>
#include <cstring>
#include <functional>

#include "model.h"
#include "umma_conv.h"

namespace {
using namespace sbv2;

constexpr int kHeadDim = 96, kWindow = 4, kRel = 2 * kWindow + 1;

void open_owner(sbv2_model& owner) {
  owner.device = 0;
  CUDA_CHECK(cudaSetDevice(0));
  CUDA_CHECK(cudaStreamCreateWithFlags(&owner.stream, cudaStreamNonBlocking));
}

template <class T>
T* upload(sbv2_model& owner, const T* host, size_t n) {
  return static_cast<T*>(owner.upload_bytes(host, n * sizeof(T)));
}

template <class T>
void download(sbv2_model& owner, T* host, const T* dev, size_t n) {
  CUDA_CHECK(cudaMemcpyAsync(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost, owner.stream));
  CUDA_CHECK(cudaStreamSynchronize(owner.stream));
}

// packed segments of `lens` back to back; returns the host row offsets
std::vector<int> make_segs(sbv2_model& owner, const int* lens, int n, Segs* seg) {
  SBV2_REQUIRE(n > 0, "need at least one utterance");
  std::vector<int> start(size_t(n), 0);
  long long rows = 0;
  int max_len = 0;
  for (int b = 0; b < n; ++b) {
    SBV2_REQUIRE(lens[b] >= 1, "utterance lengths must be positive");
    start[size_t(b)] = int(rows);
    rows += lens[b];
    max_len = std::max(max_len, lens[b]);
    SBV2_REQUIRE(rows < INT_MAX, "too many rows");
  }
  seg->start = upload(owner, start.data(), size_t(n));
  seg->len = upload(owner, lens, size_t(n));
  seg->n = n;
  seg->max_len = max_len;
  return start;
}

}  // namespace

// Window-relative attention of the transformer flow on planar fp16 operands.  qkv: fp16 row-major [sum(lens), 3*heads*96]
// (channel h*96+d of q, k, v in turn); rel_k / rel_v: fp32 [9][96].  mode 0: launch_flow_attention_tc, mode 1:
// launch_rel_attention_planar.  The planar rows of no utterance (gaps and tail, which the kernels read and must mask)
// hold gap_fill.  out: fp16 row-major [sum(lens), heads*96]; *out_pad_rows: planar output rows outside every utterance
// that the kernel wrote (the output buffer is pre-filled with a sentinel).
extern "C" int sbv2_debug_flow_attention(const uint16_t* qkv_f16, const int* lens, int n, int heads, const float* rel_k,
                                         const float* rel_v, int mode, uint16_t gap_fill, uint16_t* out_f16,
                                         long long* out_pad_rows) {
  return guarded([&] {
    SBV2_REQUIRE(n > 0 && heads > 0 && (mode == 0 || mode == 1), "bad arguments");
    sbv2_model owner;
    open_owner(owner);
    const LaunchCtx ctx = owner.ctx();
    std::vector<int> ystart(lens, lens + n), ylen(lens, lens + n), muls{1};
    long long rows = 0;
    for (int b = 0; b < n; ++b) {
      SBV2_REQUIRE(lens[b] >= 1, "utterance lengths must be positive");
      ystart[size_t(b)] = int(rows);
      rows += lens[b];
    }
    DBuf meta;
    PinnedBuf pin;
    meta.stream = owner.stream;
    BatchGeom bg = build_geoms(&owner, meta, pin, ystart, ylen, muls);
    const Geom& G = bg.g[0];
    const int C = heads * kHeadDim, C3 = 3 * C;
    const size_t plane = size_t(G.rows_tot) * 8;
    std::vector<uint16_t> hq(size_t(C3 / 8) * plane, gap_fill);
    std::vector<char> in_utt(size_t(G.rows_tot), 0);
    for (int b = 0; b < n; ++b)
      for (int t = 0; t < lens[b]; ++t) {
        const size_t pr = size_t(G.pstart[size_t(b)]) + t;
        in_utt[pr] = 1;
        const uint16_t* src = qkv_f16 + (size_t(ystart[size_t(b)]) + t) * C3;
        for (int c = 0; c < C3; ++c) hq[size_t(c / 8) * plane + pr * 8 + c % 8] = src[c];
      }
    const uint16_t kSentinel = 0x7D5A;  // an fp16 NaN payload: no kernel writes it
    std::vector<uint16_t> ho(size_t(C / 8) * plane, kSentinel);
    const __half* d_qkv = reinterpret_cast<const __half*>(upload(owner, hq.data(), hq.size()));
    __half* d_out = reinterpret_cast<__half*>(upload(owner, ho.data(), ho.size()));
    PlanarSegs ps;
    ps.start = bg.d_ystart;
    ps.pstart = G.d_pstart;
    ps.len = G.d_len;
    ps.order = bg.d_order;
    ps.n = n;
    ps.max_len = G.max_len;
    ps.plane_stride = G.rows_tot * 8;
    if (mode == 0) {
      const std::vector<__half> pk = pack_flow_rel_table(rel_k, kWindow, kHeadDim), pv = pack_flow_rel_table(rel_v, kWindow, kHeadDim);
      launch_flow_attention_tc(ctx, d_out, d_qkv, upload(owner, pk.data(), pk.size()), upload(owner, pv.data(), pv.size()), heads, kHeadDim,
                               kWindow, ps);
    } else {
      launch_rel_attention_planar(ctx, d_out, d_qkv, upload(owner, rel_k, size_t(kRel) * kHeadDim), upload(owner, rel_v, size_t(kRel) * kHeadDim),
                                  heads, kHeadDim, kWindow, ps);
    }
    download(owner, ho.data(), reinterpret_cast<const uint16_t*>(d_out), ho.size());
    for (int b = 0; b < n; ++b)
      for (int t = 0; t < lens[b]; ++t) {
        const size_t pr = size_t(G.pstart[size_t(b)]) + t;
        uint16_t* dst = out_f16 + (size_t(ystart[size_t(b)]) + t) * C;
        for (int c = 0; c < C; ++c) dst[c] = ho[size_t(c / 8) * plane + pr * 8 + c % 8];
      }
    long long written = 0;
    for (size_t pr = 0; pr < size_t(G.rows_tot); ++pr) {
      if (in_utt[pr]) continue;
      bool w = false;
      for (int pl = 0; pl < C / 8 && !w; ++pl)
        for (int e = 0; e < 8; ++e) w |= ho[size_t(pl) * plane + pr * 8 + e] != kSentinel;
      written += w ? 1 : 0;
    }
    if (out_pad_rows) *out_pad_rows = written;
  });
}

// The text encoder's fp32 attention (launch_rel_attention) on a ragged batch: qkv fp32 row-major [sum(lens), 3*heads*96],
// rel_k / rel_v fp32 [9][96], out fp32 row-major [sum(lens), heads*96].
extern "C" int sbv2_debug_rel_attention(const float* qkv_f32, const int* lens, int n, int heads, const float* rel_k, const float* rel_v,
                                        float* out_f32) {
  return guarded([&] {
    SBV2_REQUIRE(heads > 0, "bad arguments");
    sbv2_model owner;
    open_owner(owner);
    Segs seg;
    const std::vector<int> start = make_segs(owner, lens, n, &seg);
    const size_t rows = size_t(start.back()) + size_t(lens[n - 1]), C = size_t(heads) * kHeadDim;
    const float* d_qkv = upload(owner, qkv_f32, rows * 3 * C);
    float* d_out = upload(owner, out_f32, rows * C);
    launch_rel_attention(owner.ctx(), d_out, d_qkv, upload(owner, rel_k, size_t(kRel) * kHeadDim), upload(owner, rel_v, size_t(kRel) * kHeadDim),
                         heads, kHeadDim, kWindow, seg);
    download(owner, out_f32, d_out, rows * C);
  });
}

// Inverse rational-quadratic spline of a ConvFlow (launch_convflow_spline, 10 bins): z fp32 [rows, 2] in / out (column 1
// is transformed), proj fp32 [rows, ld] (10 width, 10 height, 9 derivative logits).
extern "C" int sbv2_debug_convflow_spline(float* z, const float* proj, int ld, int rows, float tail_bound, float inv_sqrt_filter) {
  return guarded([&] {
    SBV2_REQUIRE(rows > 0 && ld >= 29, "bad arguments");
    sbv2_model owner;
    open_owner(owner);
    float* d_z = upload(owner, z, size_t(rows) * 2);
    launch_convflow_spline(owner.ctx(), d_z, upload(owner, proj, size_t(rows) * ld), ld, 10, tail_bound, inv_sqrt_filter, rows);
    download(owner, z, d_z, size_t(rows) * 2);
  });
}

// Length regulator: launch_durations on logw_dp [rows] and z_sdp [rows, 2] (null: no SDP term) with per-utterance ratio
// and length_scale; returns w [rows], dur [rows], cum [rows], ylen [n].  With frame2ph (int [sum ylen]) and a total that
// fits in int32, launch_expand then maps frames to phonemes (zero statistics and noise).
extern "C" int sbv2_debug_durations(const float* logw_dp, const float* z_sdp, const float* ratio, const float* length_scale, const int* lens,
                                    int n, float* w_out, int* dur, int* cum, int* ylen, int* frame2ph) {
  return guarded([&] {
    sbv2_model owner;
    open_owner(owner);
    const LaunchCtx ctx = owner.ctx();
    Segs xseg;
    const std::vector<int> start = make_segs(owner, lens, n, &xseg);
    const size_t rows = size_t(start.back()) + size_t(lens[n - 1]);
    std::vector<float> zero_f(rows * 2, 0.f);
    std::vector<int> zero_i(rows, 0);
    float* d_w = upload(owner, zero_f.data(), rows);
    int* d_dur = upload(owner, zero_i.data(), rows);
    int* d_cum = upload(owner, zero_i.data(), rows);
    int* d_ylen = upload(owner, zero_i.data(), size_t(n));
    launch_durations(ctx, upload(owner, logw_dp, rows), z_sdp ? upload(owner, z_sdp, rows * 2) : nullptr, upload(owner, ratio, size_t(n)),
                     upload(owner, length_scale, size_t(n)), d_w, d_dur, d_cum, d_ylen, xseg);
    download(owner, w_out, d_w, rows);
    download(owner, dur, d_dur, rows);
    download(owner, cum, d_cum, rows);
    download(owner, ylen, d_ylen, size_t(n));
    if (!frame2ph) return;
    std::vector<int> ystart(lens, lens + n);
    long long ny = 0;
    int ymax = 0;
    for (int b = 0; b < n; ++b) {
      ystart[size_t(b)] = int(std::min<long long>(ny, INT_MAX));
      ny += ylen[b];
      ymax = std::max(ymax, ylen[b]);
    }
    if (ny > INT_MAX) return;
    Segs yseg;
    yseg.start = upload(owner, ystart.data(), size_t(n));
    yseg.len = d_ylen;
    yseg.n = n;
    yseg.max_len = ymax;
    std::vector<float> zy(size_t(ny), 0.f);
    const float* d_zero_y = upload(owner, zy.data(), zy.size());
    float* d_zp = upload(owner, zy.data(), zy.size());
    int* d_f2p = reinterpret_cast<int*>(upload(owner, zy.data(), zy.size()));
    launch_expand(ctx, d_zp, d_f2p, upload(owner, zero_f.data(), rows * 2), d_cum, d_zero_y, upload(owner, zero_f.data(), size_t(n)), 1, xseg,
                  yseg);
    download(owner, frame2ph, d_f2p, size_t(ny));
  });
}

// ---- the decoder's tensor-core layers ---------------------------------------------------------------------------
namespace {
using namespace sbv2;

constexpr uint16_t kHalfSentinel = 0x7D5A;       // an fp16 NaN payload: no kernel writes it
constexpr uint32_t kFloatSentinel = 0x7FC0A5A5u;  // an fp32 NaN payload

// packed fp32 [sum(lens), C] -> planar fp16 [C/8][rows_tot][8] with zero gaps (launch_zero_gaps, launch_to_planar)
__half* planar_input(sbv2_model& owner, const float* packed, int C, const int* d_start, const Geom& g, int n) {
  const LaunchCtx ctx = owner.ctx();
  long long rows = 0;
  for (int b = 0; b < n; ++b) rows += g.len[size_t(b)];
  std::vector<uint16_t> zero(size_t(C / 8) * g.rows_tot * 8, 0);
  __half* d = reinterpret_cast<__half*>(upload(owner, zero.data(), zero.size()));
  launch_zero_gaps(ctx, d, C, g, n);
  launch_to_planar(ctx, d, upload(owner, packed, size_t(rows) * C), C, C, d_start, g, n, ACT_NONE);
  return d;
}

}  // namespace

// One tensor-core layer (launch_umma) on a ragged batch, as the HiFi-GAN decoder runs it.
//   up == 0: Conv1d, w [cout][cin][k], dilation dil: make_conv1d_layer(mt_pref, nb_max); utterance b has lens[b] rows.
//   up == u: ConvTranspose1d, w [cin][cout][k], stride u, padding (k - u) / 2: make_upsample_layer(mt_pref), launched
//            with out_mul = u; utterance b has lens[b] input rows and u * lens[b] output rows.
// bias [cout] or null.  x: packed fp32 [sum(lens), cin], stored as planar fp16 with zero gaps and no activation (pass the
// values the layer reads).  Epilogue inputs, all optional: bias_utt [n][cout]; residual = the input (cin == cout);
// res2 / res3 (both or neither): packed fp32 [output rows, cout] stored the same way, with out_div; accum_mode (UAccum)
// with accum: packed fp32 [output rows, cout] that pre-fills the planar fp32 accumulate buffer and receives it back, and
// accum_div; act_out (Act).
// out: packed fp32 [output rows, cout] <- the fp16 output (left untouched for UACC_SET / UACC_ADD, which store none).
// The output buffer holds a sentinel in every row before the launch, the accumulate buffer outside the utterance rows:
// pad_rows[0] / [1] count the planar rows outside every utterance that the layer wrote in either.  cfg[3]: the layer's
// mt (128-row tiles per work item, in input rows), nb and n_nblk.
extern "C" int sbv2_debug_umma_layer(const float* w, const float* bias, int cin, int cout, int k, int dil, int up, int mt_pref,
                                     int nb_max, const float* x, const int* lens, int n, const float* bias_utt, int residual,
                                     const float* res2, const float* res3, float out_div, int accum_mode, float* accum,
                                     float accum_div, int act_out, float* out, long long* pad_rows, int* cfg) {
  return guarded([&] {
    SBV2_REQUIRE(w && x && lens && out && n > 0 && cin > 0 && cout > 0 && k > 0 && up >= 0, "bad arguments");
    SBV2_REQUIRE(!residual || cin == cout, "the residual is the layer's input: needs cin == cout");
    SBV2_REQUIRE(!res2 == !res3, "res2 and res3 go together");
    SBV2_REQUIRE(accum_mode >= UACC_NONE && accum_mode <= UACC_FINAL && (accum_mode == UACC_NONE || accum),
                 "an accumulate mode needs the accumulate buffer");
    sbv2_model owner;
    open_owner(owner);
    const LaunchCtx ctx = owner.ctx();
    HostConv hc;
    hc.d0 = up ? cin : cout;
    hc.d1 = up ? cout : cin;
    hc.k = k;
    hc.w.assign(w, w + size_t(cin) * cout * k);
    if (bias) hc.b.assign(bias, bias + cout);
    const ConvLayer L = up ? make_upsample_layer(&owner, hc, up, mt_pref) : make_conv1d_layer(&owner, hc, dil, mt_pref, nb_max);
    if (cfg) {
      cfg[0] = L.mt;
      cfg[1] = L.nb;
      cfg[2] = L.n_nblk;
    }
    const int mul = up ? up : 1;
    std::vector<int> ystart(lens, lens + n), ostart(lens, lens + n), ylen(lens, lens + n), muls{1};
    if (up) muls.push_back(up);
    long long rows = 0;
    for (int b = 0; b < n; ++b) {
      SBV2_REQUIRE(lens[b] >= 1, "utterance lengths must be positive");
      ystart[size_t(b)] = int(rows);
      ostart[size_t(b)] = int(rows * mul);
      rows += lens[b];
      SBV2_REQUIRE(rows * mul < INT_MAX, "too many rows");
    }
    DBuf meta;
    PinnedBuf pin;
    meta.stream = owner.stream;
    BatchGeom bg = build_geoms(&owner, meta, pin, ystart, ylen, muls);
    const Geom& Gi = bg.g[0];
    const Geom& Go = bg.g.back();
    const int* d_ostart = upload(owner, ostart.data(), size_t(n));
    const size_t oplane = size_t(Go.rows_tot) * 8;
    std::vector<char> in_utt(size_t(Go.rows_tot), 0);
    for (int b = 0; b < n; ++b)
      for (int t = 0; t < Go.len[size_t(b)]; ++t) in_utt[size_t(Go.pstart[size_t(b)]) + t] = 1;

    ConvCall c;
    c.in = planar_input(owner, x, cin, bg.d_ystart, Gi, n);
    if (residual) c.residual = c.in;
    if (res2) {
      c.residual2 = planar_input(owner, res2, cout, d_ostart, Go, n);
      c.residual3 = planar_input(owner, res3, cout, d_ostart, Go, n);
      c.out_div = out_div;
    }
    if (bias_utt) c.bias_utt = upload(owner, bias_utt, size_t(n) * cout);
    std::vector<uint16_t> ho(size_t(cout / 8) * oplane, kHalfSentinel);
    __half* d_out = reinterpret_cast<__half*>(upload(owner, ho.data(), ho.size()));
    const bool stores = accum_mode != UACC_SET && accum_mode != UACC_ADD;
    c.out = stores ? d_out : nullptr;
    std::vector<uint32_t> ha;
    float* d_acc = nullptr;
    if (accum_mode != UACC_NONE) {
      ha.assign(size_t(cout / 8) * oplane, kFloatSentinel);
      for (int b = 0; b < n; ++b)
        for (int t = 0; t < Go.len[size_t(b)]; ++t)
          for (int co = 0; co < cout; ++co)
            memcpy(&ha[size_t(co / 8) * oplane + (size_t(Go.pstart[size_t(b)]) + t) * 8 + co % 8],
                   accum + (size_t(ostart[size_t(b)]) + t) * cout + co, 4);
      d_acc = reinterpret_cast<float*>(upload(owner, ha.data(), ha.size()));
      c.accum = d_acc;
      c.accum_mode = accum_mode;
      c.accum_div = accum_div;
    }
    c.act_out = act_out;
    c.out_mul = mul;
    launch_umma(ctx, L, Gi, Go, c, n);
    download(owner, ho.data(), reinterpret_cast<const uint16_t*>(d_out), ho.size());
    if (d_acc) download(owner, ha.data(), reinterpret_cast<const uint32_t*>(d_acc), ha.size());
    for (int b = 0; b < n; ++b)
      for (int t = 0; t < Go.len[size_t(b)]; ++t) {
        const size_t pr = size_t(Go.pstart[size_t(b)]) + t, orow = size_t(ostart[size_t(b)]) + t;
        for (int co = 0; co < cout; ++co) {
          const size_t e = size_t(co / 8) * oplane + pr * 8 + co % 8;
          if (stores) out[orow * cout + co] = __half2float(__ushort_as_half(ho[e]));
          if (d_acc) memcpy(accum + orow * cout + co, &ha[e], 4);
        }
      }
    long long written[2] = {0, 0};
    for (size_t pr = 0; pr < size_t(Go.rows_tot); ++pr) {
      if (in_utt[pr]) continue;
      bool wo = false, wa = false;
      for (int e = 0; e < cout; ++e) {
        const size_t i = size_t(e / 8) * oplane + pr * 8 + e % 8;
        wo |= ho[i] != kHalfSentinel;
        wa |= d_acc && ha[i] != kFloatSentinel;
      }
      written[0] += wo ? 1 : 0;
      written[1] += wa ? 1 : 0;
    }
    if (pad_rows) {
      pad_rows[0] = written[0];
      pad_rows[1] = written[1];
    }
  });
}

// The decoder's conv_post (launch_dec_post_planar) on a ragged batch.  x: packed fp32 [sum(lens), C] (the lrelu(0.01)
// values it reads), stored as planar fp16 with zero gaps; w fp32 [C][k]; utterance b's samples go to
// wave[wstart[b] .. wstart[b] + lens[b]).  wave [wave_len] in / out: the whole buffer goes up and comes back, so every
// sample outside the utterances keeps what the caller put there unless the kernel wrote it.  force_generic: the generic
// kernel also at C = 16, k = 7.
extern "C" int sbv2_debug_dec_post(const float* x, const int* lens, const long long* wstart, int n, const float* w, int C, int k,
                                   int force_generic, float* wave, long long wave_len) {
  return guarded([&] {
    SBV2_REQUIRE(x && lens && wstart && w && wave && n > 0 && C > 0 && C % 8 == 0 && k > 0 && k % 2 == 1, "bad arguments");
    sbv2_model owner;
    open_owner(owner);
    std::vector<int> ystart(lens, lens + n), ylen(lens, lens + n), muls{1};
    std::vector<long long> ws(wstart, wstart + n);
    long long rows = 0;
    for (int b = 0; b < n; ++b) {
      SBV2_REQUIRE(lens[b] >= 1, "utterance lengths must be positive");
      SBV2_REQUIRE(wstart[b] >= 0 && wstart[b] + lens[b] <= wave_len, "utterance outside the waveform buffer");
      ystart[size_t(b)] = int(rows);
      rows += lens[b];
      SBV2_REQUIRE(rows < INT_MAX, "too many rows");
    }
    DBuf meta;
    PinnedBuf pin;
    meta.stream = owner.stream;
    BatchGeom bg = build_geoms(&owner, meta, pin, ystart, ylen, muls, nullptr, false, &ws);
    const Geom& G = bg.g[0];
    const __half* d_x = planar_input(owner, x, C, bg.d_ystart, G, n);
    const std::vector<float> wh(w, w + size_t(C) * k);
    float* d_wave = upload(owner, wave, size_t(wave_len));
    launch_dec_post_planar(owner.ctx(), d_wave, d_x, G, bg.d_wstart, n, upload(owner, wh.data(), wh.size()), wh, C, k, force_generic != 0);
    download(owner, wave, d_wave, size_t(wave_len));
  });
}

// ---- split-fp16 layers, the WaveNet gate, DeBERTa's LayerNorms -----------------------------------------------------
namespace {

// A ragged batch packed back to back (ystart) and its planar geometry (one time resolution).
struct Ragged {
  DBuf meta;
  PinnedBuf pin;
  BatchGeom bg;
  std::vector<int> ystart;
  long long rows = 0;
  std::vector<char> in_utt;  // planar rows that belong to an utterance
  const Geom& g() const { return bg.g[0]; }
};

void ragged(sbv2_model& owner, const int* lens, int n, Ragged* r) {
  SBV2_REQUIRE(lens && n > 0, "need at least one utterance");
  r->ystart.assign(lens, lens + n);
  const std::vector<int> ylen(lens, lens + n), muls{1};
  for (int b = 0; b < n; ++b) {
    SBV2_REQUIRE(lens[b] >= 1, "utterance lengths must be positive");
    r->ystart[size_t(b)] = int(r->rows);
    r->rows += lens[b];
    SBV2_REQUIRE(r->rows < INT_MAX, "too many rows");
  }
  r->meta.stream = owner.stream;
  r->bg = build_geoms(&owner, r->meta, r->pin, r->ystart, ylen, muls);
  r->in_utt.assign(size_t(r->g().rows_tot), 0);
  for (int b = 0; b < n; ++b)
    for (int t = 0; t < lens[b]; ++t) r->in_utt[size_t(r->g().pstart[size_t(b)]) + t] = 1;
}

PlanarSegs planar_segs(const Ragged& r, int n) {
  PlanarSegs ps;
  ps.start = r.bg.d_ystart;
  ps.pstart = r.g().d_pstart;
  ps.len = r.g().d_len;
  ps.order = r.bg.d_order;
  ps.n = n;
  ps.max_len = r.g().max_len;
  ps.plane_stride = r.g().rows_tot * 8;
  return ps;
}

// planar 16-bit [planes][rows_tot][8] -> packed [rows][planes * 8] (utterance rows only)
void unplanar(uint16_t* dst, const std::vector<uint16_t>& buf, int planes, const Ragged& r, int n) {
  const Geom& G = r.g();
  const size_t plane = size_t(G.rows_tot) * 8;
  for (int b = 0; b < n; ++b)
    for (int t = 0; t < G.len[size_t(b)]; ++t) {
      const size_t pr = size_t(G.pstart[size_t(b)]) + t;
      uint16_t* row = dst + (size_t(r.ystart[size_t(b)]) + t) * planes * 8;
      for (int c = 0; c < planes * 8; ++c) row[c] = buf[size_t(c / 8) * plane + pr * 8 + c % 8];
    }
}

// planar rows outside every utterance in which some element of the fp16 buffer no longer holds kHalfSentinel
long long stray_rows(const std::vector<uint16_t>& buf, int planes, const Ragged& r) {
  const size_t plane = size_t(r.g().rows_tot) * 8;
  long long n = 0;
  for (size_t pr = 0; pr < size_t(r.g().rows_tot); ++pr) {
    if (r.in_utt[pr]) continue;
    bool w = false;
    for (int pl = 0; pl < planes && !w; ++pl)
      for (int e = 0; e < 8; ++e) w |= buf[size_t(pl) * plane + pr * 8 + e] != kHalfSentinel;
    n += w ? 1 : 0;
  }
  return n;
}

}  // namespace

// One split-fp16 layer (make_split_conv1d_layer(terms, mt_pref, nb_max), dilation dil) on a ragged batch, as the text
// encoder and exact-mode DeBERTa run it.  w [cout][cin][k], bias [cout] or null, x packed fp32 [sum(lens), cin] (the
// values the layer receives): the input split planes come from launch_split_planar, with zero gaps (launch_zero_gaps),
// in a buffer that holds kHalfSentinel everywhere before.  bias_utt [n][cout] or null; act_out ACT_NONE / ACT_RELU /
// ACT_GELU; tmap, splitk, cluster as the ConvCall fields.
//   rm:    out fp32 [sum(lens), cout] <- the row-major output (each element holds an fp32 NaN payload before the launch)
//   split: out_split [sum(lens)][3 * cout] <- the ConvCall::split_out plane blocks [h0 | h1 | h0], scaled by split_scale
// in_split [sum(lens)][3 or 6 * cin] <- the input plane blocks.  pad_rows[0] / [1]: planar rows outside every utterance
// written by launch_split_planar / into split_out (both buffers start as kHalfSentinel).  cfg[4]: the layer's mt, nb,
// n_nblk, nkc; scales[2]: in_scale, out_scale; report[4]: what launch_umma chose (UmmaLaunchReport: variant, cluster,
// splitk, tmap).
extern "C" int sbv2_debug_split_layer(const float* w, const float* bias, int cin, int cout, int k, int dil, int terms, int mt_pref, int nb_max,
                                      const float* x, const int* lens, int n, const float* bias_utt, int act_out, int rm, int split,
                                      float split_scale, int tmap, int splitk, int cluster, float* out, uint16_t* out_split,
                                      uint16_t* in_split, long long* pad_rows, int* cfg, float* scales, int* report) {
  return guarded([&] {
    SBV2_REQUIRE(w && x && in_split && cin > 0 && cout > 0 && k > 0 && (terms == 2 || terms == 3), "bad arguments");
    SBV2_REQUIRE((rm || split) && (!rm || out) && (!split || out_split), "the layer needs an output");
    SBV2_REQUIRE(act_out == ACT_NONE || act_out == ACT_RELU || act_out == ACT_GELU, "the row-major epilogue applies none, relu or gelu");
    sbv2_model owner;
    open_owner(owner);
    const LaunchCtx ctx = owner.ctx();
    HostConv hc;
    hc.d0 = cout;
    hc.d1 = cin;
    hc.k = k;
    hc.w.assign(w, w + size_t(cin) * cout * k);
    if (bias) hc.b.assign(bias, bias + cout);
    const ConvLayer L = make_split_conv1d_layer(&owner, hc, dil, mt_pref, terms, nb_max);
    if (cfg) {
      cfg[0] = L.mt;
      cfg[1] = L.nb;
      cfg[2] = L.n_nblk;
      cfg[3] = L.nkc;
    }
    if (scales) {
      scales[0] = L.in_scale;
      scales[1] = L.out_scale;
    }
    Ragged R;
    ragged(owner, lens, n, &R);
    const Geom& G = R.g();
    const int nblk = terms == 3 ? 6 : 3;
    const size_t plane = size_t(G.rows_tot) * 8;
    std::vector<uint16_t> hi(size_t(nblk) * (cin / 8) * plane, kHalfSentinel);
    __half* d_in = reinterpret_cast<__half*>(upload(owner, hi.data(), hi.size()));
    launch_split_planar(ctx, d_in, upload(owner, x, size_t(R.rows) * cin), cin, cin, R.bg.d_ystart, G, n, terms, L.in_scale);
    download(owner, hi.data(), reinterpret_cast<const uint16_t*>(d_in), hi.size());
    unplanar(in_split, hi, nblk * cin / 8, R, n);
    const long long stray_in = stray_rows(hi, nblk * cin / 8, R);
    launch_zero_gaps(ctx, d_in, nblk * cin, G, n);

    ConvCall c;
    c.in = d_in;
    c.act_out = act_out;
    if (bias_utt) c.bias_utt = upload(owner, bias_utt, size_t(n) * cout);
    std::vector<uint32_t> ho;
    if (rm) {
      ho.assign(size_t(R.rows) * cout, kFloatSentinel);
      c.rm_out = reinterpret_cast<float*>(upload(owner, ho.data(), ho.size()));
      c.rm_ld = cout;
      c.rm_start = R.bg.d_ystart;
    }
    std::vector<uint16_t> hs;
    if (split) {
      hs.assign(size_t(3) * (cout / 8) * plane, kHalfSentinel);
      c.split_out = reinterpret_cast<__half*>(upload(owner, hs.data(), hs.size()));
      c.split_scale = split_scale;
    }
    c.tmap = tmap != 0;
    c.splitk = splitk != 0;
    c.cluster = cluster;
    UmmaLaunchReport rep;
    c.report = &rep;
    launch_umma(ctx, L, G, G, c, n);
    if (rm) {
      download(owner, ho.data(), reinterpret_cast<const uint32_t*>(c.rm_out), ho.size());
      memcpy(out, ho.data(), ho.size() * 4);
    }
    long long stray_out = 0;
    if (split) {
      download(owner, hs.data(), reinterpret_cast<const uint16_t*>(c.split_out), hs.size());
      unplanar(out_split, hs, 3 * cout / 8, R, n);
      stray_out = stray_rows(hs, 3 * cout / 8, R);
    }
    if (pad_rows) {
      pad_rows[0] = stray_in;
      pad_rows[1] = stray_out;
    }
    if (report) {
      report[0] = rep.variant;
      report[1] = rep.cluster;
      report[2] = rep.splitk;
      report[3] = rep.tmap;
    }
  });
}

// One WaveNet in_layer (make_gated_conv1d_layer, Conv1d cin -> 2 * hidden, k taps, dilation dil) on a ragged batch,
// launched as the WN flow launches it: gate_half, and the conditioning as bias_utt with a row stride (bias_utt_ld) wider
// than 2 * hidden.  w [2 * hidden][cin][k] and bias [2 * hidden] (or null) in the original channel order: channels
// [0, hidden) feed tanh, [hidden, 2 * hidden) the sigmoid.  cond [n][2 * hidden]: each utterance's conditioning, also in
// the original order; the hook permutes it with the layer's perm as the model permutes cond_layer.  x packed fp32
// [sum(lens), cin], stored as planar fp16 with zero gaps.  out [sum(lens)][hidden] <- tanh(.) * sigmoid(.) as fp16
// values; pad_rows[0]: planar output rows outside every utterance written.  cfg[4]: gate_half, nb, n_nblk, mt.
extern "C" int sbv2_debug_gated_layer(const float* w, const float* bias, int cin, int hidden, int k, int dil, int mt_pref, const float* x,
                                      const int* lens, int n, const float* cond, float* out, long long* pad_rows, int* cfg) {
  return guarded([&] {
    SBV2_REQUIRE(w && x && cond && out && cin > 0 && hidden > 0 && k > 0, "bad arguments");
    sbv2_model owner;
    open_owner(owner);
    const LaunchCtx ctx = owner.ctx();
    HostConv hc;
    hc.d0 = 2 * hidden;
    hc.d1 = cin;
    hc.k = k;
    hc.w.assign(w, w + size_t(cin) * 2 * hidden * k);
    if (bias) hc.b.assign(bias, bias + 2 * hidden);
    int gate_half = 0;
    std::vector<int> perm;
    const ConvLayer L = make_gated_conv1d_layer(&owner, hc, dil, mt_pref, &gate_half, &perm);
    if (cfg) {
      cfg[0] = gate_half;
      cfg[1] = L.nb;
      cfg[2] = L.n_nblk;
      cfg[3] = L.mt;
    }
    Ragged R;
    ragged(owner, lens, n, &R);
    const Geom& G = R.g();
    const int ld = 2 * hidden + 32;
    std::vector<float> cp(size_t(n) * ld, 0.f);
    for (int b = 0; b < n; ++b)
      for (int i = 0; i < 2 * hidden; ++i) cp[size_t(b) * ld + i] = cond[size_t(b) * 2 * hidden + perm[size_t(i)]];
    const size_t plane = size_t(G.rows_tot) * 8;
    std::vector<uint16_t> ho(size_t(hidden / 8) * plane, kHalfSentinel);
    ConvCall c;
    c.in = planar_input(owner, x, cin, R.bg.d_ystart, G, n);
    c.out = reinterpret_cast<__half*>(upload(owner, ho.data(), ho.size()));
    c.gate_half = gate_half;
    c.bias_utt = upload(owner, cp.data(), cp.size());
    c.bias_utt_ld = ld;
    launch_umma(ctx, L, G, G, c, n);
    download(owner, ho.data(), reinterpret_cast<const uint16_t*>(c.out), ho.size());
    std::vector<uint16_t> packed(size_t(R.rows) * hidden);
    unplanar(packed.data(), ho, hidden / 8, R, n);
    for (size_t i = 0; i < packed.size(); ++i) out[i] = __half2float(__ushort_as_half(packed[i]));
    if (pad_rows) pad_rows[0] = stray_rows(ho, hidden / 8, R);
  });
}

// One of DeBERTa's LayerNorms on a ragged batch: a, addin packed fp32 [sum(lens), C] (addin may be null), gamma / beta [C].
//   mode 0: launch_ln_split(out, split, split_scale, a, addin): out [sum(lens)][C] <- LN(a + addin) (each element holds an
//           fp32 NaN payload before), planes [sum(lens)][3 * C] <- the split blocks [h0 | h1 | h0]
//   mode 1: launch_ln_planar_wide(h = a, hp, hp2, y32 = addin as planar fp32): out <- h, planes [sum(lens)][2 * C] <- hp | hp2
// pad_rows[0]: planar rows outside every utterance written into the planes (which hold kHalfSentinel before).
extern "C" int sbv2_debug_bert_layernorm(int mode, const float* a, const float* addin, const float* gamma, const float* beta, float eps, int C,
                                         const int* lens, int n, float split_scale, float* out, uint16_t* planes, long long* pad_rows) {
  return guarded([&] {
    SBV2_REQUIRE(a && gamma && beta && out && planes && (mode == 0 || mode == 1) && C > 0, "bad arguments");
    sbv2_model owner;
    open_owner(owner);
    const LaunchCtx ctx = owner.ctx();
    Ragged R;
    ragged(owner, lens, n, &R);
    const Geom& G = R.g();
    const PlanarSegs ps = planar_segs(R, n);
    const size_t plane = size_t(G.rows_tot) * 8, elems = size_t(R.rows) * C;
    const int nbuf = mode == 0 ? 3 : 2;
    std::vector<uint16_t> hp(size_t(nbuf) * (C / 8) * plane, kHalfSentinel);
    __half* d_hp = reinterpret_cast<__half*>(upload(owner, hp.data(), hp.size()));
    const float* d_g = upload(owner, gamma, size_t(C));
    const float* d_b = upload(owner, beta, size_t(C));
    float* d_out;
    if (mode == 0) {
      const std::vector<uint32_t> sentinel(elems, kFloatSentinel);
      d_out = reinterpret_cast<float*>(upload(owner, sentinel.data(), elems));
      launch_ln_split(ctx, d_out, d_hp, split_scale, upload(owner, a, elems), addin ? upload(owner, addin, elems) : nullptr, d_g, d_b, eps, C, ps);
    } else {
      d_out = upload(owner, a, elems);
      const float* d_y = nullptr;
      if (addin) {
        std::vector<float> y((C / 8) * plane, 0.f);
        for (int b = 0; b < n; ++b)
          for (int t = 0; t < lens[b]; ++t)
            for (int c = 0; c < C; ++c)
              y[size_t(c / 8) * plane + (size_t(G.pstart[size_t(b)]) + t) * 8 + c % 8] = addin[(size_t(R.ystart[size_t(b)]) + t) * C + c];
        d_y = upload(owner, y.data(), y.size());
      }
      launch_ln_planar_wide(ctx, d_out, d_hp, d_hp + size_t(C / 8) * plane, d_y, d_g, d_b, eps, C, ps);
    }
    download(owner, out, d_out, elems);
    download(owner, hp.data(), reinterpret_cast<const uint16_t*>(d_hp), hp.size());
    unplanar(planes, hp, nbuf * C / 8, R, n);
    if (pad_rows) pad_rows[0] = stray_rows(hp, nbuf * C / 8, R);
  });
}

// ---- DeBERTa ----------------------------------------------------------------------------------------------------
// The relative-position bucket table the model builds at load (bert_bucket_table), on the host: *max_rel = its saturation
// bound R; out (null: R only) receives the 2R + 1 entries for delta = -R..R.  Needs no device.
extern "C" int sbv2_debug_bert_bucket_table(int span, int* max_rel, int* out) {
  return guarded([&] {
    SBV2_REQUIRE(max_rel != nullptr, "bad arguments");
    const std::vector<int> tab = bert_bucket_table(span, max_rel);
    if (out) memcpy(out, tab.data(), tab.size() * sizeof(int));
  });
}

// One DeBERTa disentangled attention launch (head dim 64) on a ragged batch, with the bucket table of `span`.
//   qkv   fp16 row-major [terms][sum(lens)][3 * heads * 64] (q | k | v, channel h * 64 + d)
//   pos_k, pos_q  fp16 row-major [terms][2 * span][heads * 64]: the position projections
//   mode  0: single-tile tensor-core kernel (<= 128 tokens), 1: multi-tile tensor-core kernel, 2: its exact variant, whose
//         operands are the two fp16 terms (terms = 2) of values scaled by sc, 3: CUDA-core kernel; terms = 1 except in mode 2
//   far_pairs  modes 1 and 2: far tile pairs take the reduced path (0: the generic path for every pair)
//   out   fp16 row-major [terms][sum(lens)][heads * 64]: the context (mode 2: the two terms of context * sc)
//   reps > 0: the launch is then repeated `reps` times between two CUDA events and *ms receives the mean time per launch
// The planar rows of no utterance hold zeros, as the model keeps them.
extern "C" int sbv2_debug_deberta_attention(const uint16_t* qkv, const uint16_t* pos_k, const uint16_t* pos_q, const int* lens, int n,
                                            int heads, int span, int mode, int far_pairs, float sc, int reps, float* ms, uint16_t* out) {
  return guarded([&] {
    SBV2_REQUIRE(qkv && pos_k && pos_q && lens && out && n > 0 && heads > 0 && mode >= 0 && mode <= 3, "bad arguments");
    SBV2_REQUIRE(mode != 2 || sc > 0.f, "the exact kernel needs the split scale");
    SBV2_REQUIRE(reps <= 0 || ms != nullptr, "timing needs *ms");
    sbv2_model owner;
    open_owner(owner);
    const LaunchCtx ctx = owner.ctx();
    std::vector<int> ystart(lens, lens + n), ylen(lens, lens + n), muls{1};
    long long rows = 0;
    for (int b = 0; b < n; ++b) {
      SBV2_REQUIRE(lens[b] >= 1 && lens[b] <= kMaxBertTokens, "utterance lengths must be in [1, 32768]");
      ystart[size_t(b)] = int(rows);
      rows += lens[b];
      SBV2_REQUIRE(rows < INT_MAX, "too many rows");
    }
    int max_rel = 0;
    const std::vector<int> tab = bert_bucket_table(span, &max_rel);
    DBuf meta;
    PinnedBuf pin;
    meta.stream = owner.stream;
    BatchGeom bg = build_geoms(&owner, meta, pin, ystart, ylen, muls);
    const Geom& G = bg.g[0];
    const int H = heads * 64, C3 = 3 * H, terms = mode == 2 ? 2 : 1, n_pos = 2 * span;
    const size_t plane = size_t(G.rows_tot) * 8, qkv_blk = size_t(C3 / 8) * plane, ctx_blk = size_t(H / 8) * plane;
    std::vector<uint16_t> hq(terms * qkv_blk, 0);
    for (int term = 0; term < terms; ++term)
      for (int b = 0; b < n; ++b)
        for (int t = 0; t < lens[b]; ++t) {
          const size_t pr = size_t(G.pstart[size_t(b)]) + t;
          const uint16_t* src = qkv + (size_t(term) * rows + ystart[size_t(b)] + t) * C3;
          for (int c = 0; c < C3; ++c) hq[term * qkv_blk + size_t(c / 8) * plane + pr * 8 + c % 8] = src[c];
        }
    std::vector<uint16_t> ho(3 * ctx_blk, 0);
    const __half* d_qkv = reinterpret_cast<const __half*>(upload(owner, hq.data(), hq.size()));
    __half* d_out = reinterpret_cast<__half*>(upload(owner, ho.data(), ho.size()));
    const int* d_tab = upload(owner, tab.data(), tab.size());
    PlanarSegs ps;
    ps.start = bg.d_ystart;
    ps.pstart = G.d_pstart;
    ps.len = G.d_len;
    ps.order = bg.d_order;
    ps.n = n;
    ps.max_len = G.max_len;
    ps.plane_stride = G.rows_tot * 8;
    std::function<void()> launch;
    if (mode == 3) {
      // the CUDA-core kernel reads fp32 tables transposed to [heads * 64][n_pos]
      std::vector<float> tk(size_t(H) * n_pos), tq(tk.size());
      for (int r = 0; r < n_pos; ++r)
        for (int c = 0; c < H; ++c) {
          tk[size_t(c) * n_pos + r] = __half2float(__ushort_as_half(pos_k[size_t(r) * H + c]));
          tq[size_t(c) * n_pos + r] = __half2float(__ushort_as_half(pos_q[size_t(r) * H + c]));
        }
      const float* d_tk = upload(owner, tk.data(), tk.size());
      const float* d_tq = upload(owner, tq.data(), tq.size());
      launch = [&, d_tk, d_tq] { launch_deberta_attention(ctx, d_out, d_qkv, d_tk, d_tq, n_pos, d_tab, max_rel, heads, 64, ps); };
    } else {
      // the tensor-core kernels read [terms][heads][8][n_pos][8]
      auto pack = [&](const uint16_t* pos) {
        std::vector<uint16_t> p(size_t(terms) * H * n_pos);
        for (int term = 0; term < terms; ++term)
          for (int r = 0; r < n_pos; ++r)
            for (int c = 0; c < H; ++c)
              p[size_t(term) * H * n_pos + (size_t(c / 8) * n_pos + r) * 8 + c % 8] = pos[(size_t(term) * n_pos + r) * H + c];
        return reinterpret_cast<const __half*>(upload(owner, p.data(), p.size()));
      };
      const __half* d_pk = pack(pos_k);
      const __half* d_pq = pack(pos_q);
      launch = [&, d_pk, d_pq] {
        if (mode == 0) launch_deberta_attention_tc(ctx, d_out, d_qkv, d_pk, d_pq, n_pos, span, heads, ps);
        else if (mode == 1) launch_deberta_attention_tc_multi(ctx, d_out, d_qkv, d_pk, d_pq, n_pos, d_tab, max_rel, heads, far_pairs != 0, ps);
        else
          launch_deberta_attention_tc_exact_multi(ctx, d_out, (long long)ctx_blk, d_qkv, (long long)qkv_blk, d_pk, d_pq, n_pos, d_tab, max_rel,
                                                  heads, sc, far_pairs != 0, ps);
      };
    }
    launch();
    if (reps > 0) {
      cudaEvent_t e0, e1;
      CUDA_CHECK(cudaEventCreate(&e0));
      CUDA_CHECK(cudaEventCreate(&e1));
      CUDA_CHECK(cudaEventRecord(e0, owner.stream));
      for (int r = 0; r < reps; ++r) launch();
      CUDA_CHECK(cudaEventRecord(e1, owner.stream));
      CUDA_CHECK(cudaEventSynchronize(e1));
      CUDA_CHECK(cudaEventElapsedTime(ms, e0, e1));
      *ms /= float(reps);
      CUDA_CHECK(cudaEventDestroy(e0));
      CUDA_CHECK(cudaEventDestroy(e1));
    }
    download(owner, ho.data(), reinterpret_cast<const uint16_t*>(d_out), ho.size());
    for (int term = 0; term < terms; ++term)
      for (int b = 0; b < n; ++b)
        for (int t = 0; t < lens[b]; ++t) {
          const size_t pr = size_t(G.pstart[size_t(b)]) + t;
          uint16_t* dst = out + (size_t(term) * rows + ystart[size_t(b)] + t) * H;
          for (int c = 0; c < H; ++c) dst[c] = ho[term * ctx_blk + size_t(c / 8) * plane + pr * 8 + c % 8];
        }
  });
}
