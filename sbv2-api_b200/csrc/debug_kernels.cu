// Unit-test hooks of the synthesizer kernels between the text encoder and the decoder: the flow's window attention
// (tensor-core and planar CUDA-core), the text encoder's fp32 attention, the inverse spline of the stochastic duration
// predictor, and the length regulator.  Linked into libsbv2_b200_debug.so only (build.py DEBUG_ONLY).  Every hook runs
// on its own stream, takes host arrays and returns host arrays before it returns; tests/test_gpu_synth_kernels.py
// compares the results with float64 evaluations of oracle/vits.py.
#include <cuda_fp16.h>

#include <algorithm>
#include <climits>

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
