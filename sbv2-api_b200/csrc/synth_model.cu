// JP-Extra synthesizer (Style-Bert-VITS2 SynthesizerTrn.infer) as a static kernel plan.
// Replaces the `ort::Session::run` of crates/sbv2_core/src/model.rs:91-103 for model.onnx.
// Graph restated in SURVEY.md §A; oracle in oracle/vits.py.
#include <algorithm>
#include <cmath>
#include <sstream>

#include "model.h"
#include "onnx_bind.h"
#include "umma_conv.h"

namespace sbv2 {
namespace {

struct ConvW {
  float* w = nullptr;  // [taps][Cin][Cout]
  float* b = nullptr;
  int cin = 0, cout = 0, k = 1;
  int tc = -1;  // index into SynthModel::text_tc (split-fp16 tensor-core layer) or -1
};
struct LNW {
  float* g = nullptr;
  float* b = nullptr;
  int c = 0;
};
struct EncLayerW {
  ConvW qkv, o, f1, f2;
  float* rel_k = nullptr;
  float* rel_v = nullptr;
  LNW n1, n2;
};
struct EncoderW {
  std::vector<EncLayerW> layers;
  ConvW spk;  // Linear gin -> hidden, applied at cond_idx
  bool has_spk = false;
  int cond_idx = 2;
  int heads = 2, head_dim = 96, window = 4, hidden = 192, filter = 768, ksize = 3;
};
struct DDSW {
  struct L {
    float* sep_w = nullptr;  // [C][3]
    float* sep_b = nullptr;
    ConvW pw;
    LNW n1, n2;
    int dil = 1;
  };
  std::vector<L> layers;
};
struct ConvFlowW {
  float* pre_w = nullptr;  // [C]
  float* pre_b = nullptr;
  DDSW dds;
  ConvW proj;  // C -> 3*bins-1
};
struct UpW {
  // ConvTranspose1d(Cin -> Cout, k, stride u, pad (k-u)/2) as u phase convolutions of k/u taps
  std::vector<float*> phase_w;  // [u] each [k/u][Cin][Cout]
  std::vector<int> phase_off;   // input row offset c of each phase
  float* b = nullptr;
  int cin = 0, cout = 0, k = 0, u = 0;
};
struct ResBlockW {
  std::vector<ConvW> c1, c2;
  std::vector<int> dil;
  int k = 3;
};
struct WNW {
  ConvW cond;  // gin -> 2*H*n_layers
  std::vector<ConvW> in_layers, res_skip;
  int k = 5;
};
struct CouplingW {
  ConvW pre, post;
  EncoderW enc;  // transformer variant
  WNW wn;        // WN variant
};

// Every flow / text layer is packed twice: [0] for batches (N blocks up to 256 channels, 256-row work items: fewest weight
// bytes per row) and [1] for few rows (16-channel N blocks, 128-row items): a batch-1 call is latency-bound, its layers
// are weight streams, and the wide packing would leave each of them to 2-12 CTAs (profiles/r2_latency_*).  An N = 16 MMA
// issues as fast as an N = 64 one (48 cycles), so the narrowest block simply gives the most CTAs per weight stream.
// Both packings give bit-identical results: the K order of every output element is the same.
constexpr int kSmallNb = 16;
constexpr int64_t kSmallFlowRows = 1024, kSmallTextRows = 512;
struct FlowTCLayer {
  ConvLayer qkv[2], o[2], f1[2], f2[2];
  __half* rel_k_p = nullptr;  // fp16 [D/8][16][8] packing of emb_rel_k for the tensor-core attention
  __half* rel_v_p = nullptr;
};
struct FlowTC {
  ConvLayer pre[2], post[2];
  std::vector<FlowTCLayer> layers;
};
// WN residual-coupling layer on the tensor cores: in_layers with the tanh * sigmoid gate fused into the epilogue
// (channels permuted per N block), res/skip 1x1 convs accumulating into the fp32 [x | skip] stream
struct WnTC {
  ConvLayer pre, post;
  std::vector<ConvLayer> in_layers, res_skip;
  ConvW cond_perm;    // cond_layer with every layer's 2H slice in the gated layers' channel order
  int gate_half = 0;
};

struct HParams {
  int n_vocab = 0, n_tones = 0, n_lang = 0, hidden = 0, inter = 0, gin = 0, n_speakers = 0, bert_dim = 0, style_dim = 0;
  int dp_filter = 0, sdp_bins = 10, sdp_flows = 0;
  bool transformer_flow = true;
  int n_flows = 0, flow_layers = 0, wn_layers = 0;
  std::vector<int> up_rates, up_kernels, res_kernels;
  std::vector<std::vector<int>> res_dils;
  int up_initial = 0;
  int hop = 1;
};

}  // namespace

}  // namespace sbv2
struct BatchBuffers;
namespace sbv2 {

struct SynthModel : sbv2_model {
  HParams hp;
  // weights
  float *emb = nullptr, *tone_emb = nullptr, *lang_emb = nullptr, *emb_g = nullptr;
  ConvW bert_proj, style_proj, enc_proj;
  EncoderW enc;
  ConvW dp_c1, dp_c2, dp_proj, dp_cond;
  LNW dp_n1, dp_n2;
  ConvW sdp_pre, sdp_proj, sdp_cond;
  DDSW sdp_dds;
  std::vector<ConvFlowW> sdp_cf;  // in module order (flows.1, .3, .5, .7)
  float *sdp_ea_m = nullptr, *sdp_ea_logs = nullptr;
  std::vector<CouplingW> flow;  // flows.0, .2, .4, .6
  ConvW dec_pre, dec_cond;
  std::vector<UpW> ups;
  std::vector<ResBlockW> resblocks;
  float* dec_post_w = nullptr;  // [1][C][k]
  int dec_post_k = 7, dec_post_c = 16;
  UmmaDecoder* umma = nullptr;  // tensor-core decoder plan (umma_decoder.cu); null -> fp32 path
  bool use_umma = true;
  std::vector<FlowTC> flow_tc;  // tensor-core transformer flow (fp16 operands, fp32 residual stream)
  bool use_tc_flow = true;
  bool use_tc_attn = true;
  uint64_t fl_qkvp_gen = 0;  // DBuf::gen of the qkv buffer that was cleared last (tails must be finite for the TC attention)
  std::vector<std::vector<HostConv>> flow_host;  // consumed at create: per coupling [pre, post, (qkv, o, f1, f2) x L]
  std::vector<std::vector<HostConv>> wn_host;    // consumed at create: per coupling [pre, post, cond, (in, res_skip) x L]
  std::vector<WnTC> wn_tc;
  bool use_tc_wn = false;
  DBuf fl_x0p, fl_hp, fl_qkvp, fl_ctxp, fl_f1p, fl_y32, fl_m32, fl_meta;
  PinnedBuf fl_pin;
  // text encoder / duration predictor convs on the tensor cores with two-term fp16 splits (~fp32 accuracy)
  std::vector<ConvLayer> text_tc, text_tc_small;  // same index; see kSmallNb
  std::vector<std::pair<ConvW*, HostConv>> text_host;  // consumed at create
  int64_t small_text_rows = kSmallTextRows, small_flow_rows = kSmallFlowRows;  // SBV2_B200_SMALL_ROWS="text,flow" overrides
  bool use_tc_text = true;
  int text_terms = 2;  // fp16 terms per operand (2: 3 cross products, 3: 6 cross products)
  int text_tc_max_cin = 0;
  DBuf tx_split, tx_meta;
  PinnedBuf tx_pin;

  uint64_t seed = 0x5b2b200ULL, rng_offset = 0;
  // workspaces
  DBuf ws[32];
  std::vector<BatchBuffers*> batch_pool;  // idle batch buffer sets
  DecoderHostWeights dec_host;  // original-layout decoder weights, consumed by umma_decoder_create
  PinnedBuf pin_in, pin_ylen, pin_ymeta;
  ~SynthModel() override;
};

}  // namespace sbv2

// Device buffers of one batch; recycled through the model's pool (cudaMalloc/cudaFree per call costs ms).
struct BatchBuffers {
  sbv2::DBuf in, zp, ymeta, wave, dur, cum, f2p, ylen_dev;
};

// One uploaded batch: host bookkeeping + device inputs/outputs.
struct sbv2_device_batch {
  int B = 0;
  int64_t Nx = 0, Ny = 0;
  std::vector<int> xlen, xstart, ylen, ystart;
  std::vector<int64_t> zp_frames;
  bool has_noise_sdp = false, has_noise_zp = false, any_sdp = false;
  BatchBuffers* bufs = nullptr;  // borrowed from / returned to the owner's pool
  sbv2_model* owner = nullptr;
  sbv2::DBuf &in, &zp, &ymeta, &wave, &dur, &cum, &f2p, &ylen_dev;
  explicit sbv2_device_batch(BatchBuffers* b, sbv2_model* o)
      : bufs(b), owner(o), in(b->in), zp(b->zp), ymeta(b->ymeta), wave(b->wave), dur(b->dur), cum(b->cum), f2p(b->f2p), ylen_dev(b->ylen_dev) {}
  // offsets (bytes) into `in`
  size_t o_x = 0, o_tone = 0, o_lang = 0, o_sid = 0, o_sdp_ratio = 0, o_ls = 0, o_ns = 0, o_nsw = 0, o_xstart = 0, o_xlen = 0,
         o_bert_off = 0, o_nsdp_off = 0, o_style = 0, o_bert = 0, o_nsdp = 0, o_zp_off = 0, o_zp_ld = 0;
  bool ran = false;
  bool decode_only = false;
  bool borrowed_host = false;  // some H2D copies read the caller's (pinned) buffers directly: synchronise before returning to it
  // silence (samples) laid out after each utterance in the waveform buffer (easy_synthesize's 22 050-sample pauses,
  // tts.rs:318-320, written on the device); empty = none
  std::vector<int64_t> pause_after;
  std::vector<long long> wstart;  // sample offset of each utterance in `wave` (filled by synth_run)
  int64_t wave_total = 0;         // samples in `wave` including pauses
  // BERT rows already on this device: gathered by ph2tok (int64 [sum t_x] at o_bert) instead of uploaded
  const float* dev_bert_rows = nullptr;
  int64_t dev_bert_n = 0;
  cudaEvent_t dev_bert_ready = nullptr;
};

namespace sbv2 {

SynthModel::~SynthModel() {
  if (umma) umma_decoder_free(umma);
  cudaSetDevice(device);
  if (stream) cudaStreamSynchronize(stream);
  for (BatchBuffers* b : batch_pool) delete b;
}

static BatchBuffers* borrow_buffers(SynthModel& M) {
  BatchBuffers* b;
  if (!M.batch_pool.empty()) {
    b = M.batch_pool.back();
    M.batch_pool.pop_back();
  } else {
    b = new BatchBuffers();
  }
  for (DBuf* d : {&b->in, &b->zp, &b->ymeta, &b->wave, &b->dur, &b->cum, &b->f2p, &b->ylen_dev}) d->stream = M.stream;
  return b;
}
namespace {

// ---------------------------------------------------------------------------------------------
// weight loading
// ---------------------------------------------------------------------------------------------
struct Loader {
  const OnnxModel& m;
  SynthModel& M;
  WeightBinder& binder;  // canonical (PyTorch) name -> initializer, incl. structurally bound anonymous weights (onnx_bind.h)

  const OnnxTensor* find(const std::string& n) const { return binder.find(n); }
  bool has(const std::string& n) const { return find(n) != nullptr; }
  const OnnxTensor& get(const std::string& n) const {
    const OnnxTensor* t = find(n);
    if (!t) fail(SBV2_ERR_UNSUPPORTED, "synthesizer graph lacks initializer '" + n + "'");
    return *t;
  }
  std::vector<float> f32(const std::string& n) const { return m.as_f32(get(n)); }
  float* vec(const std::string& n, int expect = -1) const {
    auto v = f32(n);
    if (expect >= 0 && int(v.size()) != expect)
      fail(SBV2_ERR_UNSUPPORTED, "initializer '" + n + "' has " + std::to_string(v.size()) + " elements, expected " + std::to_string(expect));
    return M.upload_f32(v);
  }
  // Conv1d weight [Cout, Cin, k] (or Linear [out, in]) -> [k][Cin][Cout]
  ConvW conv(const std::string& prefix, bool bias = true) const {
    const OnnxTensor& t = get(prefix + ".weight");
    if (t.dims.size() != 3 && t.dims.size() != 2) fail(SBV2_ERR_UNSUPPORTED, "'" + prefix + ".weight' must be 2-D or 3-D");
    ConvW c;
    c.cout = int(t.dims[0]);
    c.cin = int(t.dims[1]);
    c.k = t.dims.size() == 3 ? int(t.dims[2]) : 1;
    auto w = m.as_f32(t);
    std::vector<float> r(w.size());
    for (int co = 0; co < c.cout; ++co)
      for (int ci = 0; ci < c.cin; ++ci)
        for (int j = 0; j < c.k; ++j) r[(size_t(j) * c.cin + ci) * c.cout + co] = w[(size_t(co) * c.cin + ci) * c.k + j];
    c.w = M.upload_f32(r);
    if (bias) c.b = vec(prefix + ".bias", c.cout);
    return c;
  }
  LNW ln(const std::string& prefix) const {
    LNW l;
    const OnnxTensor& t = get(prefix + ".gamma");
    l.c = int(t.numel());
    l.g = vec(prefix + ".gamma", l.c);
    l.b = vec(prefix + ".beta", l.c);
    return l;
  }
  int count(const std::string& fmt_prefix, const std::string& suffix, int step = 1) const {
    int n = 0;
    while (has(fmt_prefix + std::to_string(n * step) + suffix)) ++n;
    return n;
  }
  EncoderW encoder(const std::string& p) const {
    EncoderW E;
    int n = count(p + ".attn_layers.", ".conv_q.weight");
    if (n == 0) fail(SBV2_ERR_UNSUPPORTED, "encoder '" + p + "' has no attention layers");
    for (int i = 0; i < n; ++i) {
      EncLayerW L;
      std::string a = p + ".attn_layers." + std::to_string(i);
      ConvW q = conv(a + ".conv_q"), k = conv(a + ".conv_k"), v = conv(a + ".conv_v");
      // fuse q|k|v along Cout
      int H = q.cout, C = q.cin;
      auto wq = f32(a + ".conv_q.weight"), wk = f32(a + ".conv_k.weight"), wv = f32(a + ".conv_v.weight");
      std::vector<float> w(size_t(C) * 3 * H), b(size_t(3) * H);
      for (int ci = 0; ci < C; ++ci)
        for (int co = 0; co < H; ++co) {
          w[size_t(ci) * 3 * H + co] = wq[size_t(co) * C + ci];
          w[size_t(ci) * 3 * H + H + co] = wk[size_t(co) * C + ci];
          w[size_t(ci) * 3 * H + 2 * H + co] = wv[size_t(co) * C + ci];
        }
      auto bq = f32(a + ".conv_q.bias"), bk = f32(a + ".conv_k.bias"), bv = f32(a + ".conv_v.bias");
      for (int co = 0; co < H; ++co) {
        b[co] = bq[co];
        b[H + co] = bk[co];
        b[2 * H + co] = bv[co];
      }
      L.qkv.w = M.upload_f32(w);
      L.qkv.b = M.upload_f32(b);
      L.qkv.cin = C;
      L.qkv.cout = 3 * H;
      L.qkv.k = 1;
      L.o = conv(a + ".conv_o");
      const OnnxTensor& rk = get(a + ".emb_rel_k");
      if (rk.dims.size() != 3 || rk.dims[0] != 1) fail(SBV2_ERR_UNSUPPORTED, "emb_rel_k must be [1, 2w+1, d] (heads_share)");
      E.window = int(rk.dims[1] - 1) / 2;
      E.head_dim = int(rk.dims[2]);
      E.heads = H / E.head_dim;
      E.hidden = H;
      L.rel_k = vec(a + ".emb_rel_k");
      L.rel_v = vec(a + ".emb_rel_v");
      L.n1 = ln(p + ".norm_layers_1." + std::to_string(i));
      L.n2 = ln(p + ".norm_layers_2." + std::to_string(i));
      L.f1 = conv(p + ".ffn_layers." + std::to_string(i) + ".conv_1");
      L.f2 = conv(p + ".ffn_layers." + std::to_string(i) + ".conv_2");
      E.filter = L.f1.cout;
      E.ksize = L.f1.k;
      E.layers.push_back(L);
    }
    if (has(p + ".spk_emb_linear.weight")) {
      E.spk = conv(p + ".spk_emb_linear");
      E.has_spk = true;
      E.cond_idx = 2;
      if (E.cond_idx >= n) fail(SBV2_ERR_UNSUPPORTED, "encoder '" + p + "': cond_layer_idx 2 needs >= 3 layers");
    }
    return E;
  }
  DDSW dds(const std::string& p) const {
    DDSW D;
    int n = count(p + ".convs_sep.", ".weight");
    int dil = 1;
    for (int i = 0; i < n; ++i) {
      DDSW::L L;
      std::string s = p + ".convs_sep." + std::to_string(i);
      const OnnxTensor& t = get(s + ".weight");
      if (t.dims.size() != 3 || t.dims[1] != 1 || t.dims[2] != 3) fail(SBV2_ERR_UNSUPPORTED, "DDSConv depthwise weight must be [C,1,3]");
      L.sep_w = vec(s + ".weight");
      L.sep_b = vec(s + ".bias");
      L.pw = conv(p + ".convs_1x1." + std::to_string(i));
      L.n1 = ln(p + ".norms_1." + std::to_string(i));
      L.n2 = ln(p + ".norms_2." + std::to_string(i));
      L.dil = dil;
      dil *= 3;
      D.layers.push_back(L);
    }
    return D;
  }
};

int attr_first(const OnnxNode& n, const char* name, int dflt) {
  auto it = n.int_attrs.find(name);
  if (it == n.int_attrs.end() || it->second.empty()) return dflt;
  return int(it->second[0]);
}

// Real exports constant-fold weight-normed convs into anonymous initializers (SURVEY.md §A.7).
// Bind them by walking Conv / ConvTranspose nodes in graph (= execution) order after conv_pre.
void bind_decoder_structurally(Loader& L) {
  const OnnxModel& m = L.m;
  if (L.has("dec.ups.0.weight")) return;  // named, or already bound through its bias (onnx_bind.h)
  size_t start = m.nodes.size();
  for (size_t i = 0; i < m.nodes.size(); ++i) {
    const auto& n = m.nodes[i];
    if (n.op_type == "Conv" && n.inputs.size() >= 2 && n.inputs[1] == "dec.conv_pre.weight") {
      start = i + 1;
      break;
    }
  }
  if (start == m.nodes.size()) fail(SBV2_ERR_UNSUPPORTED, "cannot locate dec.conv_pre in the graph to bind decoder weights");
  // sequence: (ConvTranspose, then per resblock: c1.0 c2.0 c1.1 c2.1 c1.2 c2.2) ...
  int up = -1, rb = -1, pos = 0;
  int n_res_per = 0;
  std::vector<std::string> seq;
  for (size_t i = start; i < m.nodes.size(); ++i) {
    const auto& n = m.nodes[i];
    if (n.inputs.size() < 2 || !m.find(n.inputs[1])) continue;
    if (n.op_type == "ConvTranspose") {
      if (up >= 0 && n_res_per == 0) n_res_per = (rb + 1);
      ++up;
      L.binder.alias_to("dec.ups." + std::to_string(up) + ".weight", n.inputs[1]);
      if (n.inputs.size() > 2) L.binder.alias_to("dec.ups." + std::to_string(up) + ".bias", n.inputs[2]);
      pos = 0;
    } else if (n.op_type == "Conv" && up >= 0) {
      if (n.inputs[1] == "dec.conv_post.weight") break;
      const OnnxTensor* w = m.find(n.inputs[1]);
      if (w->dims.size() != 3) continue;
      // each resblock contributes 2 * n_dil convs; a new resblock starts when the kernel size changes or after 6 convs
      int idx_in_rb = pos % 6;
      if (idx_in_rb == 0) ++rb;
      std::string which = (idx_in_rb % 2 == 0) ? "convs1" : "convs2";
      std::string nm = "dec.resblocks." + std::to_string(rb) + "." + which + "." + std::to_string(idx_in_rb / 2);
      L.binder.alias_to(nm + ".weight", n.inputs[1]);
      if (n.inputs.size() > 2) L.binder.alias_to(nm + ".bias", n.inputs[2]);
      ++pos;
    }
  }
  if (up < 0) fail(SBV2_ERR_UNSUPPORTED, "no ConvTranspose nodes found while binding decoder weights");
}

void load_weights(SynthModel& M, const OnnxModel& m) {
  WeightBinder binder(m);
  Loader L{m, M, binder};
  HParams& hp = M.hp;
  if (!L.has("enc_p.emb.weight") || !L.has("dec.conv_pre.weight"))
    fail(SBV2_ERR_UNSUPPORTED, "not a Style-Bert-VITS2 synthesizer graph (enc_p.emb.weight / dec.conv_pre.weight missing)");
  bind_decoder_structurally(L);
  // a bias whose weight could not be bound would make has(".weight") probes (spk_emb_linear ...) skip a layer silently
  binder.require_weights_for_biases("");

  auto dims = [&](const std::string& n) { return L.get(n).dims; };
  hp.n_vocab = int(dims("enc_p.emb.weight")[0]);
  hp.hidden = int(dims("enc_p.emb.weight")[1]);
  hp.n_tones = int(dims("enc_p.tone_emb.weight")[0]);
  hp.n_lang = int(dims("enc_p.language_emb.weight")[0]);
  hp.n_speakers = int(dims("emb_g.weight")[0]);
  hp.gin = int(dims("emb_g.weight")[1]);
  hp.bert_dim = int(dims("enc_p.bert_proj.weight")[1]);
  hp.style_dim = int(dims("enc_p.style_proj.weight")[1]);

  M.emb = L.vec("enc_p.emb.weight");
  M.tone_emb = L.vec("enc_p.tone_emb.weight");
  M.lang_emb = L.vec("enc_p.language_emb.weight");
  M.emb_g = L.vec("emb_g.weight");
  M.bert_proj = L.conv("enc_p.bert_proj");
  M.style_proj = L.conv("enc_p.style_proj");
  M.enc = L.encoder("enc_p.encoder");
  M.enc_proj = L.conv("enc_p.proj");
  hp.inter = M.enc_proj.cout / 2;
  if (M.enc.hidden != hp.hidden) fail(SBV2_ERR_UNSUPPORTED, "enc_p hidden size mismatch");

  // duration predictor
  M.dp_c1 = L.conv("dp.conv_1");
  M.dp_c2 = L.conv("dp.conv_2");
  M.dp_proj = L.conv("dp.proj");
  M.dp_cond = L.conv("dp.cond");
  M.dp_n1 = L.ln("dp.norm_1");
  M.dp_n2 = L.ln("dp.norm_2");
  hp.dp_filter = M.dp_c1.cout;

  // stochastic duration predictor
  M.sdp_pre = L.conv("sdp.pre");
  M.sdp_proj = L.conv("sdp.proj");
  M.sdp_cond = L.conv("sdp.cond");
  M.sdp_dds = L.dds("sdp.convs");
  M.sdp_ea_m = L.vec("sdp.flows.0.m", 2);
  M.sdp_ea_logs = L.vec("sdp.flows.0.logs", 2);
  for (int i = 1; L.has("sdp.flows." + std::to_string(i) + ".pre.weight"); i += 2) {
    std::string p = "sdp.flows." + std::to_string(i);
    ConvFlowW cf;
    const OnnxTensor& pw = L.get(p + ".pre.weight");
    if (pw.dims.size() != 3 || pw.dims[1] != 1 || pw.dims[2] != 1) fail(SBV2_ERR_UNSUPPORTED, "ConvFlow.pre must be [C,1,1]");
    cf.pre_w = L.vec(p + ".pre.weight");
    cf.pre_b = L.vec(p + ".pre.bias");
    cf.dds = L.dds(p + ".convs");
    cf.proj = L.conv(p + ".proj");
    hp.sdp_bins = (cf.proj.cout + 1) / 3;
    M.sdp_cf.push_back(cf);
  }
  hp.sdp_flows = int(M.sdp_cf.size());
  if (hp.sdp_flows < 2) fail(SBV2_ERR_UNSUPPORTED, "stochastic duration predictor needs >= 2 ConvFlows");

  // flow
  hp.transformer_flow = L.has("flow.flows.0.enc.attn_layers.0.conv_q.weight");
  for (int i = 0; L.has("flow.flows." + std::to_string(i) + ".pre.weight"); i += 2) {
    std::string p = "flow.flows." + std::to_string(i);
    CouplingW c;
    c.pre = L.conv(p + ".pre");
    c.post = L.conv(p + ".post");
    if (c.post.cout != hp.inter / 2) fail(SBV2_ERR_UNSUPPORTED, "coupling layer must be mean_only");
    if (hp.transformer_flow) {
      c.enc = L.encoder(p + ".enc");
      hp.flow_layers = int(c.enc.layers.size());
    } else {
      c.wn.cond = L.conv(p + ".enc.cond_layer");
      int n = L.count(p + ".enc.in_layers.", ".weight");
      if (n == 0) fail(SBV2_ERR_UNSUPPORTED, "flow is neither transformer nor WN coupling");
      for (int l = 0; l < n; ++l) {
        c.wn.in_layers.push_back(L.conv(p + ".enc.in_layers." + std::to_string(l)));
        c.wn.res_skip.push_back(L.conv(p + ".enc.res_skip_layers." + std::to_string(l)));
      }
      c.wn.k = c.wn.in_layers[0].k;
      hp.wn_layers = n;
    }
    M.flow.push_back(c);
  }
  hp.n_flows = int(M.flow.size());
  if (hp.n_flows == 0) fail(SBV2_ERR_UNSUPPORTED, "no coupling layers found under flow.flows");

  // decoder
  M.dec_pre = L.conv("dec.conv_pre");
  M.dec_cond = L.conv("dec.cond");
  hp.up_initial = M.dec_pre.cout;
  int n_ups = L.count("dec.ups.", ".weight");
  if (n_ups == 0) fail(SBV2_ERR_UNSUPPORTED, "decoder has no upsampling layers");
  // strides / dilations from the graph nodes when present
  std::map<std::string, const OnnxNode*> node_of_weight;
  for (const auto& n : m.nodes)
    if ((n.op_type == "Conv" || n.op_type == "ConvTranspose") && n.inputs.size() >= 2) node_of_weight[n.inputs[1]] = &n;
  auto node_for = [&](const std::string& canonical) -> const OnnxNode* {
    const OnnxTensor* t = L.find(canonical);
    auto it = node_of_weight.find(t ? t->name : canonical);
    return it == node_of_weight.end() ? nullptr : it->second;
  };
  static const int default_rates_k16[] = {8, 8, 2, 2, 2};
  hp.hop = 1;
  for (int i = 0; i < n_ups; ++i) {
    std::string p = "dec.ups." + std::to_string(i);
    const OnnxTensor& t = L.get(p + ".weight");
    if (t.dims.size() != 3) fail(SBV2_ERR_UNSUPPORTED, p + ".weight must be [Cin,Cout,k]");
    UpW U;
    U.cin = int(t.dims[0]);
    U.cout = int(t.dims[1]);
    U.k = int(t.dims[2]);
    const OnnxNode* n = node_for(p + ".weight");
    if (n) U.u = attr_first(*n, "strides", 0);
    if (U.u <= 0) {
      if (n_ups == 5 && i < 5) U.u = default_rates_k16[i];  // JP-Extra default [8,8,2,2,2]
      else fail(SBV2_ERR_UNSUPPORTED, "cannot determine the stride of " + p);
    }
    if (U.k % U.u != 0 || (U.k - U.u) % 2 != 0) fail(SBV2_ERR_UNSUPPORTED, p + ": kernel/stride combination not supported");
    auto w = m.as_f32(t);
    int pad = (U.k - U.u) / 2, taps = U.k / U.u;
    for (int r = 0; r < U.u; ++r) {  // r = output index mod u
      int s = r + pad;
      int rr = s % U.u, c = s / U.u;
      std::vector<float> pw(size_t(taps) * U.cin * U.cout);
      for (int mm = 0; mm < taps; ++mm)
        for (int ci = 0; ci < U.cin; ++ci)
          for (int co = 0; co < U.cout; ++co)
            pw[(size_t(mm) * U.cin + ci) * U.cout + co] = w[(size_t(ci) * U.cout + co) * U.k + rr + U.u * mm];
      U.phase_w.push_back(M.upload_f32(pw));
      U.phase_off.push_back(c);
    }
    U.b = L.vec(p + ".bias", U.cout);
    hp.up_rates.push_back(U.u);
    hp.up_kernels.push_back(U.k);
    hp.hop *= U.u;
    M.ups.push_back(U);
  }
  int n_rb = L.count("dec.resblocks.", ".convs1.0.weight");
  if (n_rb == 0 || n_rb % n_ups != 0) fail(SBV2_ERR_UNSUPPORTED, "unexpected number of decoder resblocks");
  int per = n_rb / n_ups;
  static const int default_dils[] = {1, 3, 5};
  for (int r = 0; r < n_rb; ++r) {
    std::string p = "dec.resblocks." + std::to_string(r);
    ResBlockW R;
    int nl = L.count(p + ".convs1.", ".weight");
    for (int l = 0; l < nl; ++l) {
      R.c1.push_back(L.conv(p + ".convs1." + std::to_string(l)));
      R.c2.push_back(L.conv(p + ".convs2." + std::to_string(l)));
      const OnnxNode* n = node_for(p + ".convs1." + std::to_string(l) + ".weight");
      int d = n ? attr_first(*n, "dilations", 0) : 0;
      if (d <= 0) d = l < 3 ? default_dils[l] : 1;
      R.dil.push_back(d);
    }
    R.k = R.c1[0].k;
    if (R.k % 2 == 0) fail(SBV2_ERR_UNSUPPORTED, "even resblock kernel size");
    if (r < per) {
      hp.res_kernels.push_back(R.k);
      hp.res_dils.push_back(R.dil);
    }
    M.resblocks.push_back(R);
  }
  {
    const OnnxTensor& t = L.get("dec.conv_post.weight");
    if (t.dims.size() != 3 || t.dims[0] != 1) fail(SBV2_ERR_UNSUPPORTED, "dec.conv_post.weight must be [1,C,k]");
    M.dec_post_c = int(t.dims[1]);
    M.dec_post_k = int(t.dims[2]);
    M.dec_post_w = L.vec("dec.conv_post.weight");
    if (L.has("dec.conv_post.bias")) fail(SBV2_ERR_UNSUPPORTED, "dec.conv_post with bias is not a JP-Extra decoder");
  }

  // original-layout copies for the tensor-core kernels' fp16 repacking
  auto host_conv = [&](const std::string& p, bool bias) {
    HostConv hc;
    const OnnxTensor& t = L.get(p + ".weight");
    hc.d0 = int(t.dims[0]);
    hc.d1 = int(t.dims[1]);
    hc.k = t.dims.size() > 2 ? int(t.dims[2]) : 1;
    hc.w = m.as_f32(t);
    if (bias) hc.b = L.f32(p + ".bias");
    return hc;
  };
  {
    // text-side convs that always run over the phoneme rows (candidates for the split-fp16 tensor-core path)
    auto reg = [&](ConvW& c, HostConv hc) {
      if (hc.d0 % 16 == 0 && hc.d1 % 16 == 0) M.text_host.emplace_back(&c, std::move(hc));
    };
    auto as_conv = [&](HostConv hc) {  // Linear [out, in] -> Conv1d k = 1
      hc.k = std::max(hc.k, 1);
      return hc;
    };
    reg(M.bert_proj, as_conv(host_conv("enc_p.bert_proj", true)));
    reg(M.enc_proj, host_conv("enc_p.proj", true));
    for (size_t l = 0; l < M.enc.layers.size(); ++l) {
      std::string a = "enc_p.encoder.attn_layers." + std::to_string(l);
      HostConv q = host_conv(a + ".conv_q", true), k = host_conv(a + ".conv_k", true), vv = host_conv(a + ".conv_v", true);
      HostConv qkv;
      qkv.d0 = q.d0 + k.d0 + vv.d0;
      qkv.d1 = q.d1;
      qkv.k = 1;
      for (const HostConv* hc : {&q, &k, &vv}) {
        qkv.w.insert(qkv.w.end(), hc->w.begin(), hc->w.end());
        qkv.b.insert(qkv.b.end(), hc->b.begin(), hc->b.end());
      }
      reg(M.enc.layers[l].qkv, std::move(qkv));
      reg(M.enc.layers[l].o, host_conv(a + ".conv_o", true));
      reg(M.enc.layers[l].f1, host_conv("enc_p.encoder.ffn_layers." + std::to_string(l) + ".conv_1", true));
      reg(M.enc.layers[l].f2, host_conv("enc_p.encoder.ffn_layers." + std::to_string(l) + ".conv_2", true));
    }
    reg(M.dp_c1, host_conv("dp.conv_1", true));
    reg(M.dp_c2, host_conv("dp.conv_2", true));
  }
  if (hp.transformer_flow) {
    for (int i = 0; i < hp.n_flows; ++i) {
      std::string p = "flow.flows." + std::to_string(2 * i);
      std::vector<HostConv> v;
      v.push_back(host_conv(p + ".pre", true));
      v.push_back(host_conv(p + ".post", true));
      for (int l = 0; l < hp.flow_layers; ++l) {
        std::string a = p + ".enc.attn_layers." + std::to_string(l);
        HostConv q = host_conv(a + ".conv_q", true), k = host_conv(a + ".conv_k", true), vv = host_conv(a + ".conv_v", true);
        HostConv qkv;
        qkv.d0 = q.d0 + k.d0 + vv.d0;
        qkv.d1 = q.d1;
        qkv.k = 1;
        for (const HostConv* hc : {&q, &k, &vv}) {
          qkv.w.insert(qkv.w.end(), hc->w.begin(), hc->w.end());
          qkv.b.insert(qkv.b.end(), hc->b.begin(), hc->b.end());
        }
        v.push_back(qkv);
        v.push_back(host_conv(a + ".conv_o", true));
        v.push_back(host_conv(p + ".enc.ffn_layers." + std::to_string(l) + ".conv_1", true));
        v.push_back(host_conv(p + ".enc.ffn_layers." + std::to_string(l) + ".conv_2", true));
      }
      M.flow_host.push_back(std::move(v));
    }
  }
  if (!hp.transformer_flow) {
    for (int i = 0; i < hp.n_flows; ++i) {
      std::string p = "flow.flows." + std::to_string(2 * i);
      std::vector<HostConv> v;
      v.push_back(host_conv(p + ".pre", true));
      v.push_back(host_conv(p + ".post", true));
      v.push_back(host_conv(p + ".enc.cond_layer", true));
      for (int l = 0; l < hp.wn_layers; ++l) {
        v.push_back(host_conv(p + ".enc.in_layers." + std::to_string(l), true));
        v.push_back(host_conv(p + ".enc.res_skip_layers." + std::to_string(l), true));
      }
      M.wn_host.push_back(std::move(v));
    }
  }
  {
    DecoderHostWeights& D = M.dec_host;
    D.pre = host_conv("dec.conv_pre", true);
    D.cond = host_conv("dec.cond", true);
    D.post = host_conv("dec.conv_post", false);
    D.gin = hp.gin;
    D.per = per;
    for (int i = 0; i < n_ups; ++i) {
      D.ups.push_back(host_conv("dec.ups." + std::to_string(i), true));
      D.up_u.push_back(M.ups[i].u);
    }
    for (int r = 0; r < n_rb; ++r) {
      std::vector<HostConv> c1, c2;
      for (size_t l = 0; l < M.resblocks[r].c1.size(); ++l) {
        c1.push_back(host_conv("dec.resblocks." + std::to_string(r) + ".convs1." + std::to_string(l), true));
        c2.push_back(host_conv("dec.resblocks." + std::to_string(r) + ".convs2." + std::to_string(l), true));
      }
      D.res_c1.push_back(c1);
      D.res_c2.push_back(c2);
      D.res_dil.push_back(M.resblocks[r].dil);
    }
  }

  std::ostringstream js;
  js << "{\"kind\":\"synthesizer\",\"n_vocab\":" << hp.n_vocab << ",\"num_tones\":" << hp.n_tones << ",\"num_languages\":" << hp.n_lang
     << ",\"hidden_channels\":" << hp.hidden << ",\"inter_channels\":" << hp.inter << ",\"gin_channels\":" << hp.gin
     << ",\"n_speakers\":" << hp.n_speakers << ",\"n_layers\":" << M.enc.layers.size() << ",\"n_heads\":" << M.enc.heads
     << ",\"filter_channels\":" << M.enc.filter << ",\"kernel_size\":" << M.enc.ksize << ",\"window_size\":" << M.enc.window
     << ",\"use_transformer_flow\":" << (hp.transformer_flow ? "true" : "false") << ",\"n_flow_layer\":" << hp.n_flows
     << ",\"n_layers_trans_flow\":" << hp.flow_layers << ",\"wn_layers\":" << hp.wn_layers << ",\"sdp_flows\":" << hp.sdp_flows
     << ",\"upsample_rates\":[";
  for (size_t i = 0; i < hp.up_rates.size(); ++i) js << (i ? "," : "") << hp.up_rates[i];
  js << "],\"upsample_kernel_sizes\":[";
  for (size_t i = 0; i < hp.up_kernels.size(); ++i) js << (i ? "," : "") << hp.up_kernels[i];
  js << "],\"resblock_kernel_sizes\":[";
  for (size_t i = 0; i < hp.res_kernels.size(); ++i) js << (i ? "," : "") << hp.res_kernels[i];
  js << "],\"hop\":" << hp.hop << ",\"structural_binding\":" << (binder.any_structural() ? "true" : "false") << "}";
  M.describe_json = js.str();
}

// ---------------------------------------------------------------------------------------------
// forward pieces
// ---------------------------------------------------------------------------------------------
enum WS { W_BERT = 0, W_H, W_QKV, W_CTX, W_Y, W_F1, W_STATS, W_G, W_STYLE, W_GG, W_DPX, W_DP1, W_DP2, W_LOGW, W_SDPX, W_SDPH,
          W_SDPT, W_SDPZ, W_NSDP, W_W, W_EPS, W_Z, W_Z2, W_M, W_HF, W_META };

struct Fwd {
  SynthModel& M;
  LaunchCtx ctx;
  // split-fp16 tensor-core path for convs over the phoneme rows (set by synth_run when enabled)
  const Geom* tg = nullptr;
  const int* tg_start = nullptr;   // device: first packed row of each utterance
  const int* tg_seg_start = nullptr;  // the Segs::start the geometry was built for
  __half* tg_split = nullptr;
  int tg_n = 0;
  bool tg_small = false;  // few phoneme rows: use the 64-wide packing of the text layers

  void conv(const ConvW& c, const float* in, int in_ld, float* out, int out_ld, const Segs& seg, int dil = 1, int act_in = ACT_NONE,
            int act_out = ACT_NONE, const float* residual = nullptr, const float* bias_utt = nullptr) {
    if (c.tc >= 0 && tg != nullptr && seg.start == tg_seg_start && residual == nullptr && act_in == ACT_NONE && dil == 1 &&
        (act_out == ACT_NONE || act_out == ACT_RELU) && out_ld % 4 == 0) {
      const ConvLayer& TL = (tg_small ? M.text_tc_small : M.text_tc)[size_t(c.tc)];
      launch_split_planar(ctx, tg_split, in, in_ld, c.cin, tg_start, *tg, tg_n, M.text_terms, TL.in_scale);
      ConvCall cc;
      cc.in = tg_split;
      cc.rm_out = out;
      cc.rm_ld = out_ld;
      cc.rm_start = tg_start;
      cc.act_out = act_out;
      cc.bias_utt = bias_utt;
      launch_umma(ctx, TL, *tg, *tg, cc, tg_n);
      return;
    }
    ConvArgs a;
    a.in = in;
    a.in_ld = in_ld;
    a.w = c.w;
    a.bias = c.b;
    a.bias_utt = bias_utt;
    a.out = out;
    a.out_ld = out_ld;
    a.residual = residual;
    a.cin = c.cin;
    a.cout = c.cout;
    a.taps = c.k;
    a.dil = dil;
    a.off = -dil * ((c.k - 1) / 2);
    a.act_in = act_in;
    a.act_out = act_out;
    a.seg = seg;
    launch_conv(ctx, a);
  }

  // attentions.Encoder: h [rows, H] in place. g_lin: [B, H] = spk_emb_linear(g) or null.
  void encoder(const EncoderW& E, float* h, const Segs& seg, int rows, const float* g /*[B,gin]*/, int gin, const Segs& bseg) {
    const int H = E.hidden;
    float* qkv = M.ws[W_QKV].as<float>();
    float* ctxb = M.ws[W_CTX].as<float>();
    float* y = M.ws[W_Y].as<float>();
    float* f1 = M.ws[W_F1].as<float>();
    for (size_t i = 0; i < E.layers.size(); ++i) {
      const EncLayerW& L = E.layers[i];
      if (E.has_spk && int(i) == E.cond_idx && g) {
        float* gg = M.ws[W_GG].as<float>();
        conv(E.spk, g, gin, gg, H, bseg);
        launch_add_utt_vec(ctx, h, h, gg, H, H, seg);
      }
      conv(L.qkv, h, H, qkv, 3 * H, seg);
      launch_rel_attention(ctx, ctxb, qkv, L.rel_k, L.rel_v, E.heads, E.head_dim, E.window, seg);
      conv(L.o, ctxb, H, y, H, seg);
      launch_layernorm(ctx, h, h, y, nullptr, L.n1.g, L.n1.b, 1e-5f, ACT_NONE, H, rows);
      conv(L.f1, h, H, f1, E.filter, seg, 1, ACT_NONE, ACT_RELU);
      // FFN uses asymmetric "same" padding ((k-1)/2, k/2); identical to symmetric for odd k
      conv(L.f2, f1, E.filter, y, H, seg);
      launch_layernorm(ctx, h, h, y, nullptr, L.n2.g, L.n2.b, 1e-5f, ACT_NONE, H, rows);
    }
  }

  // DDSConv on x [rows, C] in place; t1/t2 scratch [rows, C]
  void dds(const DDSW& D, float* x, float* t1, float* t2, int C, const Segs& seg, int rows) {
    for (const auto& L : D.layers) {
      launch_dwconv3(ctx, t1, x, L.sep_w, L.sep_b, C, L.dil, seg);
      launch_layernorm(ctx, t1, t1, nullptr, nullptr, L.n1.g, L.n1.b, 1e-5f, ACT_GELU, C, rows);
      conv(L.pw, t1, C, t2, C, seg);
      launch_layernorm(ctx, x, t2, nullptr, x, L.n2.g, L.n2.b, 1e-5f, ACT_GELU, C, rows);
    }
  }
};

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

void DBuf::ensure(size_t bytes) {
  if (bytes <= cap) return;
  if (p) {
    CUDA_CHECK(cudaStreamSynchronize(stream));
    CUDA_CHECK(cudaFree(p));
    p = nullptr;
    cap = 0;
  }
  size_t want = align_up(bytes + bytes / 4, 1 << 20);
  CUDA_CHECK(cudaMalloc(&p, want));
  cap = want;
  ++gen;
}

void PinnedBuf::ensure(size_t bytes) {
  if (bytes <= cap) return;
  if (p) {
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaFreeHost(p));
    p = nullptr;
    cap = 0;
  }
  size_t want = align_up(bytes + bytes / 4, 1 << 16);
  CUDA_CHECK(cudaMallocHost(&p, want));
  cap = want;
}

sbv2_model* create_synth_model(const OnnxModel& m, int device) {
  std::unique_ptr<SynthModel> M(new SynthModel());
  M->device = device;
  M->is_bert = false;
  CUDA_CHECK(cudaSetDevice(device));
  CUDA_CHECK(cudaStreamCreateWithFlags(&M->stream, cudaStreamNonBlocking));
  {
    const char* pe = getenv("SBV2_B200_PDL");
    M->pdl = !(pe && pe[0] == '0');  // on by default
  }
  for (auto& w : M->ws) w.stream = M->stream;
  M->metadata = m.metadata;
  load_weights(*M, m);
  // SBV2_B200_DECODER=fp32 selects the CUDA-core fp32 decoder kernels (debugging / kernel cross-checks).
  const char* env = getenv("SBV2_B200_DECODER");
  M->use_umma = !(env && std::string(env) == "fp32");
  if (M->use_umma) M->umma = umma_decoder_create(M->dec_host, M.get());
  M->dec_host = DecoderHostWeights();
  // SBV2_B200_FLOW=fp32 selects the CUDA-core fp32 flow kernels (debugging / kernel cross-checks).
  const char* fenv = getenv("SBV2_B200_FLOW");
  M->use_tc_flow = M->hp.transformer_flow && !(fenv && std::string(fenv) == "fp32") && M->hp.hidden % 16 == 0 &&
                   M->hp.hidden / 8 <= 32 && (M->hp.inter / 2) % 16 == 0;
  // SBV2_B200_FLOW_NB: largest N block of the flow / text convs.  128 (256-row work items, half the weight bytes per
  // row from L2) measured slower than 256 on the bench workload (flow 7.8 vs 7.1 ms): more items, narrower MMAs.
  int flow_nb = 256;
  if (const char* e = getenv("SBV2_B200_FLOW_NB")) flow_nb = atoi(e);
  if (M->use_tc_flow) {
    for (auto& v : M->flow_host) {
      FlowTC f;
      for (int sm = 0; sm < 2; ++sm) {
        const int mtp = sm ? 1 : 2, nbm = sm ? kSmallNb : flow_nb;
        f.pre[sm] = make_conv1d_layer(M.get(), v[0], 1, mtp, nbm);
        f.post[sm] = make_conv1d_layer(M.get(), v[1], 1, mtp, nbm);
      }
      for (size_t l = 0; 2 + 4 * l + 3 < v.size(); ++l) {
        FlowTCLayer fl;
        for (int sm = 0; sm < 2; ++sm) {
          const int mtp = sm ? 1 : 2, nbm = sm ? kSmallNb : flow_nb;
          fl.qkv[sm] = make_conv1d_layer(M.get(), v[2 + 4 * l], 1, mtp, nbm);
          fl.o[sm] = make_conv1d_layer(M.get(), v[3 + 4 * l], 1, mtp, nbm);
          fl.f1[sm] = make_conv1d_layer(M.get(), v[4 + 4 * l], 1, mtp, nbm);
          fl.f2[sm] = make_conv1d_layer(M.get(), v[5 + 4 * l], 1, mtp, nbm);
        }
        f.layers.push_back(fl);
      }
      M->flow_tc.push_back(std::move(f));
    }
    for (DBuf* b : {&M->fl_x0p, &M->fl_hp, &M->fl_qkvp, &M->fl_ctxp, &M->fl_f1p, &M->fl_y32, &M->fl_m32, &M->fl_meta}) b->stream = M->stream;
  }
  if (M->use_tc_flow) {
    const char* aenv = getenv("SBV2_B200_ATTN");
    const EncoderW& E0 = M->flow[0].enc;
    M->use_tc_attn = !(aenv && std::string(aenv) == "simt") && E0.head_dim == 96 && E0.window == 4;
    if (M->use_tc_attn) {
      for (size_t i = 0; i < M->flow_tc.size(); ++i)
        for (size_t l = 0; l < M->flow_tc[i].layers.size(); ++l) {
          const EncLayerW& Lw = M->flow[i].enc.layers[l];
          const int R = 2 * E0.window + 1, D = E0.head_dim;
          std::vector<float> hk(size_t(R) * D), hv(size_t(R) * D);
          CUDA_CHECK(cudaMemcpy(hk.data(), Lw.rel_k, hk.size() * 4, cudaMemcpyDeviceToHost));
          CUDA_CHECK(cudaMemcpy(hv.data(), Lw.rel_v, hv.size() * 4, cudaMemcpyDeviceToHost));
          auto pack = [&](const std::vector<float>& src) {
            const std::vector<__half> pk = pack_flow_rel_table(src.data(), E0.window, D);
            return static_cast<__half*>(M->upload_bytes(pk.data(), pk.size() * 2));
          };
          M->flow_tc[i].layers[l].rel_k_p = pack(hk);
          M->flow_tc[i].layers[l].rel_v_p = pack(hv);
        }
    }
  }
  if (const char* e = getenv("SBV2_B200_SMALL_ROWS")) {
    long long a = 0, b = 0;
    if (sscanf(e, "%lld,%lld", &a, &b) == 2) {
      M->small_text_rows = a;
      M->small_flow_rows = b;
    }
  }
  M->flow_host.clear();
  // WN variant on the tensor cores (SBV2_B200_FLOW=fp32 keeps the CUDA-core kernels): dilation_rate of the coupling
  // layers' WN is 1 (oracle/vits.py ResidualCouplingLayer), so every in_layer is a plain k-tap "same" convolution
  M->use_tc_wn = !M->hp.transformer_flow && !(fenv && std::string(fenv) == "fp32") && M->hp.hidden % 16 == 0 && (M->hp.inter / 2) % 16 == 0 &&
                 M->hp.gin > 0;
  if (M->use_tc_wn) {
    const int H = M->hp.hidden, nl = M->hp.wn_layers;
    for (auto& v : M->wn_host) {
      WnTC w;
      w.pre = make_conv1d_layer(M.get(), v[0], 1, 2, flow_nb);
      w.post = make_conv1d_layer(M.get(), v[1], 1, 2, flow_nb);
      std::vector<int> perm;
      for (int l = 0; l < nl; ++l) {
        w.in_layers.push_back(make_gated_conv1d_layer(M.get(), v[3 + 2 * l], 1, 2, &w.gate_half, &perm));
        w.res_skip.push_back(make_conv1d_layer(M.get(), v[4 + 2 * l], 1, 2, flow_nb));
      }
      // cond_layer (gin -> 2H * nl, k = 1) with each layer's slice permuted like the gated conv's output channels
      const HostConv& c = v[2];
      if (c.d0 != 2 * H * nl || c.k != 1) fail(SBV2_ERR_UNSUPPORTED, "WN cond_layer shape does not match the in_layers");
      std::vector<float> wp(size_t(c.d1) * c.d0), bp(size_t(c.d0));
      for (int l = 0; l < nl; ++l)
        for (int i = 0; i < 2 * H; ++i) {
          const int src = l * 2 * H + perm[size_t(i)], dst = l * 2 * H + i;
          bp[size_t(dst)] = c.b[size_t(src)];
          for (int ci = 0; ci < c.d1; ++ci) wp[size_t(ci) * c.d0 + dst] = c.w[size_t(src) * c.d1 + ci];  // [k=1][Cin][Cout]
        }
      w.cond_perm.w = M->upload_f32(wp);
      w.cond_perm.b = M->upload_f32(bp);
      w.cond_perm.cin = c.d1;
      w.cond_perm.cout = c.d0;
      w.cond_perm.k = 1;
      M->wn_tc.push_back(std::move(w));
    }
    for (DBuf* b : {&M->fl_x0p, &M->fl_hp, &M->fl_qkvp, &M->fl_ctxp, &M->fl_f1p, &M->fl_y32, &M->fl_m32, &M->fl_meta}) b->stream = M->stream;
  }
  M->wn_host.clear();
  // SBV2_B200_TEXT=fp32 keeps the text encoder / duration predictor convs on the CUDA-core fp32 kernel; =split3 uses
  // three fp16 terms per operand.  Measured against the oracle both splits give the same error (enc_x 1e-5 relative,
  // 3x the CUDA-core kernel's): the tensor core's fp32 accumulation, not the operand split, sets it.
  const char* tenv = getenv("SBV2_B200_TEXT");
  M->use_tc_text = !(tenv && std::string(tenv) == "fp32");
  M->text_terms = (tenv && std::string(tenv) == "split3") ? 3 : 2;
  if (M->use_tc_text) {
    for (auto& e : M->text_host) {
      e.first->tc = int(M->text_tc.size());
      M->text_tc.push_back(make_split_conv1d_layer(M.get(), e.second, 1, 2, M->text_terms, flow_nb));
      M->text_tc_small.push_back(make_split_conv1d_layer(M.get(), e.second, 1, 1, M->text_terms, kSmallNb));
      M->text_tc_max_cin = std::max(M->text_tc_max_cin, e.second.d1);
    }
    M->tx_split.stream = M->stream;
    M->tx_meta.stream = M->stream;
  }
  M->text_host.clear();
  CUDA_CHECK(cudaStreamSynchronize(M->stream));
  return M.release();
}

void synth_set_seed(sbv2_model* m, uint64_t seed) {
  auto* M = static_cast<SynthModel*>(m);
  M->seed = seed;
  M->rng_offset = 0;
}

// ---------------------------------------------------------------------------------------------
// upload
// ---------------------------------------------------------------------------------------------
sbv2_device_batch* synth_upload(sbv2_model* mm, const sbv2_utterance* utts, int batch, const DeviceBert* dev_bert) {
  auto* M = static_cast<SynthModel*>(mm);
  SBV2_REQUIRE(!M->is_bert, "synthesize called on a BERT model");
  SBV2_REQUIRE(utts && batch > 0, "empty batch");
  M->bind_device();
  const HParams& hp = M->hp;
  std::unique_ptr<sbv2_device_batch, void (*)(sbv2_device_batch*)> b(new sbv2_device_batch(borrow_buffers(*M), M), synth_batch_free);
  b->B = batch;
  b->xlen.resize(batch);
  b->xstart.resize(batch);
  b->zp_frames.assign(batch, 0);
  int64_t nx = 0;
  int n_nsdp = 0, n_nzp = 0;
  for (int i = 0; i < batch; ++i) {
    const sbv2_utterance& u = utts[i];
    SBV2_REQUIRE(u.t_x > 0, "t_x must be positive");
    SBV2_REQUIRE(u.t_x < (1 << 20), "t_x too large");
    SBV2_REQUIRE((u.bert || dev_bert) && u.x_tst && u.tones && u.lang_ids && u.style_vec, "null input pointer");
    SBV2_REQUIRE(u.sid >= 0 && u.sid < hp.n_speakers, "speaker id out of range");
    SBV2_REQUIRE(std::isfinite(u.sdp_ratio) && std::isfinite(u.length_scale) && std::isfinite(u.noise_scale) && std::isfinite(u.noise_scale_w),
                 "non-finite scalar input");
    for (int64_t t = 0; t < u.t_x; ++t) {
      SBV2_REQUIRE(u.x_tst[t] >= 0 && u.x_tst[t] < hp.n_vocab, "symbol id out of range");
      SBV2_REQUIRE(u.tones[t] >= 0 && u.tones[t] < hp.n_tones, "tone id out of range");
      SBV2_REQUIRE(u.lang_ids[t] >= 0 && u.lang_ids[t] < hp.n_lang, "language id out of range");
    }
    b->xlen[i] = int(u.t_x);
    b->xstart[i] = int(nx);
    nx += u.t_x;
    if (u.noise_sdp) ++n_nsdp;
    if (u.noise_zp) {
      ++n_nzp;
      SBV2_REQUIRE(u.noise_zp_frames > 0, "noise_zp_frames must be positive when noise_zp is given");
      b->zp_frames[i] = u.noise_zp_frames;
    }
    if (u.sdp_ratio != 0.f) b->any_sdp = true;
  }
  SBV2_REQUIRE(n_nsdp == 0 || n_nsdp == batch, "noise_sdp must be given for all utterances or none");
  SBV2_REQUIRE(n_nzp == 0 || n_nzp == batch, "noise_zp must be given for all utterances or none");
  b->has_noise_sdp = n_nsdp > 0;
  b->has_noise_zp = n_nzp > 0;
  b->Nx = nx;
  if (dev_bert) {
    SBV2_REQUIRE(dev_bert->rows && dev_bert->ph2tok && dev_bert->hidden == hp.bert_dim, "BERT hidden size does not match the synthesizer");
    for (int64_t t = 0; t < nx; ++t)
      SBV2_REQUIRE(dev_bert->ph2tok[t] >= 0 && dev_bert->ph2tok[t] < dev_bert->n_rows, "word2ph maps a phoneme past the last token");
    b->dev_bert_rows = dev_bert->rows;
    b->dev_bert_n = dev_bert->n_rows;
    b->dev_bert_ready = dev_bert->ready;
  }

  // blob layout
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  b->o_x = take(nx * 4);
  b->o_tone = take(nx * 4);
  b->o_lang = take(nx * 4);
  b->o_sid = take(batch * 8);
  b->o_sdp_ratio = take(batch * 4);
  b->o_ls = take(batch * 4);
  b->o_ns = take(batch * 4);
  b->o_nsw = take(batch * 4);
  b->o_xstart = take(batch * 4);
  b->o_xlen = take(batch * 4);
  b->o_bert_off = take(batch * 8);
  b->o_nsdp_off = take(batch * 8);
  b->o_style = take(size_t(batch) * hp.style_dim * 4);
  b->o_bert = take(size_t(nx) * hp.bert_dim * 4);
  b->o_nsdp = take(size_t(nx) * 2 * 4);
  const size_t total = off;

  CUDA_CHECK(cudaStreamSynchronize(M->stream));  // previous upload's copies out of the staging buffer are done
  M->pin_in.ensure(total);
  uint8_t* h = M->pin_in.as<uint8_t>();
  int32_t* hx = reinterpret_cast<int32_t*>(h + b->o_x);
  int32_t* htone = reinterpret_cast<int32_t*>(h + b->o_tone);
  int32_t* hlang = reinterpret_cast<int32_t*>(h + b->o_lang);
  int64_t* hsid = reinterpret_cast<int64_t*>(h + b->o_sid);
  float* hratio = reinterpret_cast<float*>(h + b->o_sdp_ratio);
  float* hls = reinterpret_cast<float*>(h + b->o_ls);
  float* hns = reinterpret_cast<float*>(h + b->o_ns);
  float* hnsw = reinterpret_cast<float*>(h + b->o_nsw);
  int32_t* hxs = reinterpret_cast<int32_t*>(h + b->o_xstart);
  int32_t* hxl = reinterpret_cast<int32_t*>(h + b->o_xlen);
  int64_t* hboff = reinterpret_cast<int64_t*>(h + b->o_bert_off);
  int64_t* hnoff = reinterpret_cast<int64_t*>(h + b->o_nsdp_off);
  float* hstyle = reinterpret_cast<float*>(h + b->o_style);
  float* hbert = reinterpret_cast<float*>(h + b->o_bert);
  float* hnsdp = reinterpret_cast<float*>(h + b->o_nsdp);
  for (int i = 0; i < batch; ++i) {
    const sbv2_utterance& u = utts[i];
    int s = b->xstart[i], n = b->xlen[i];
    for (int t = 0; t < n; ++t) {
      hx[s + t] = int32_t(u.x_tst[t]);
      htone[s + t] = int32_t(u.tones[t]);
      hlang[s + t] = int32_t(u.lang_ids[t]);
    }
    hsid[i] = u.sid;
    hratio[i] = u.sdp_ratio;
    hls[i] = u.length_scale;
    hns[i] = u.noise_scale;
    hnsw[i] = u.noise_scale_w;
    hxs[i] = s;
    hxl[i] = n;
    hboff[i] = int64_t(s) * hp.bert_dim;
    hnoff[i] = int64_t(s) * 2;
    memcpy(hstyle + size_t(i) * hp.style_dim, u.style_vec, size_t(hp.style_dim) * 4);
    if (u.noise_sdp) memcpy(hnsdp + size_t(s) * 2, u.noise_sdp, size_t(n) * 2 * 4);
  }
  b->in.stream = M->stream;
  b->in.ensure(total);
  // small tables first, then the BERT features utterance by utterance so that the DMA of one
  // utterance overlaps the staging memcpy of the next
  CUDA_CHECK(cudaMemcpyAsync(b->in.p, h, b->o_bert, cudaMemcpyHostToDevice, M->stream));
  CUDA_CHECK(cudaMemcpyAsync(b->in.as<uint8_t>() + b->o_nsdp, h + b->o_nsdp, size_t(nx) * 2 * 4, cudaMemcpyHostToDevice, M->stream));
  if (dev_bert) {
    // the feature region only carries the phoneme -> token-row map
    memcpy(hbert, dev_bert->ph2tok, size_t(nx) * 8);
    CUDA_CHECK(cudaMemcpyAsync(b->in.as<uint8_t>() + b->o_bert, hbert, size_t(nx) * 8, cudaMemcpyHostToDevice, M->stream));
  } else
  for (int i = 0; i < batch; ++i) {
    const size_t off_f = size_t(b->xstart[i]) * hp.bert_dim, cnt = size_t(b->xlen[i]) * hp.bert_dim * 4;
    // page-locked caller memory (sbv2_alloc_pinned / cudaHostAlloc / cudaHostRegister) is read by the DMA engine in
    // place; pageable memory goes through the staging block (one memcpy per utterance, pipelined with the copies)
    cudaPointerAttributes pa{};
    const bool pinned = cudaPointerGetAttributes(&pa, utts[i].bert) == cudaSuccess && pa.type == cudaMemoryTypeHost;
    if (!pinned) cudaGetLastError();
    const void* src = utts[i].bert;
    if (pinned) {
      b->borrowed_host = true;
    } else {
      memcpy(hbert + off_f, utts[i].bert, cnt);
      src = hbert + off_f;
    }
    CUDA_CHECK(cudaMemcpyAsync(b->in.as<uint8_t>() + b->o_bert + off_f * 4, src, cnt, cudaMemcpyHostToDevice, M->stream));
  }
  if (b->has_noise_zp) {
    size_t tot = 0;
    for (int i = 0; i < batch; ++i) tot += size_t(b->zp_frames[i]) * hp.inter;
    b->zp.stream = M->stream;
    b->zp.ensure(tot * 4);
    size_t o = 0;
    for (int i = 0; i < batch; ++i) {
      size_t n = size_t(b->zp_frames[i]) * hp.inter;
      CUDA_CHECK(cudaMemcpyAsync(b->zp.as<float>() + o, utts[i].noise_zp, n * 4, cudaMemcpyHostToDevice, M->stream));
      o += n;
    }
    b->borrowed_host = true;  // read straight from the caller's buffers (staged by the driver if pageable)
  }
  // no sync here: the copies overlap with the caller's next steps; the staging buffer is protected by
  // the synchronisation at the top of the next upload
  return b.release();
}

// ---------------------------------------------------------------------------------------------
// decoder (fp32 reference path; the tensor-core path lives in umma_conv.cu)
// ---------------------------------------------------------------------------------------------
namespace {

struct StageSegs {
  Segs seg;           // rows at this stage
  const int* dstart;  // device start array
};

void decoder_fp32(SynthModel& M, const float* z, const float* g /*[B,gin]*/, const Segs& yseg, const Segs& bseg,
                  const std::vector<int>& ystart, const std::vector<int>& ylen, float* wave, DBuf& meta_buf) {
  Fwd F{M, M.ctx()};
  const HParams& hp = M.hp;
  const int B = yseg.n;
  const int n_st = int(M.ups.size());
  // per-stage segment tables
  std::vector<int> meta(size_t(2) * B * (n_st + 1));
  std::vector<int64_t> rows(n_st + 1);
  {
    int mul = 1;
    for (int s = 0; s <= n_st; ++s) {
      if (s > 0) mul *= M.ups[s - 1].u;
      for (int i = 0; i < B; ++i) {
        meta[(size_t(2) * s) * B + i] = ystart[i] * mul;
        meta[(size_t(2) * s + 1) * B + i] = ylen[i] * mul;
      }
      rows[s] = int64_t(ystart[B - 1] + ylen[B - 1]) * mul;
    }
  }
  meta_buf.stream = M.stream;
  meta_buf.ensure(meta.size() * 4);
  CUDA_CHECK(cudaMemcpyAsync(meta_buf.p, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice, M.stream));
  CUDA_CHECK(cudaStreamSynchronize(M.stream));  // `meta` is a stack vector
  auto segs_of = [&](int s) {
    Segs g2;
    g2.n = B;
    g2.start = meta_buf.as<int>() + (size_t(2) * s) * B;
    g2.len = meta_buf.as<int>() + (size_t(2) * s + 1) * B;
    int mul = 1;
    for (int q = 0; q < s; ++q) mul *= M.ups[q].u;
    g2.max_len = yseg.max_len * mul;
    return g2;
  };
  // cond(g) -> [B, C0]
  float* gcond = M.ws[W_GG].as<float>();
  M.ws[W_GG].ensure(size_t(B) * std::max(hp.up_initial, hp.hidden) * 4);
  gcond = M.ws[W_GG].as<float>();
  F.conv(M.dec_cond, g, hp.gin, gcond, hp.up_initial, bseg);
  // buffers
  size_t max_elems = 0;
  for (int s = 0; s <= n_st; ++s) {
    int C = s == 0 ? hp.up_initial : M.ups[s - 1].cout;
    max_elems = std::max(max_elems, size_t(rows[s]) * C);
  }
  DBuf &bx = M.ws[W_QKV], &br = M.ws[W_CTX], &bt = M.ws[W_Y], &bs = M.ws[W_F1];
  bx.ensure(max_elems * 4);
  br.ensure(max_elems * 4);
  bt.ensure(max_elems * 4);
  bs.ensure(max_elems * 4);
  float* x = bx.as<float>();
  float* r = br.as<float>();
  float* t1 = bt.as<float>();
  float* xs = bs.as<float>();

  Segs s0 = segs_of(0);
  F.conv(M.dec_pre, z, hp.inter, xs, hp.up_initial, s0, 1, ACT_NONE, ACT_NONE, nullptr, gcond);
  M.debug["dec_pre"] = DebugView{xs, rows[0], hp.up_initial, 4};
  const int per = int(M.resblocks.size()) / n_st;
  for (int s = 0; s < n_st; ++s) {
    const UpW& U = M.ups[s];
    Segs sin = segs_of(s), sout = segs_of(s + 1);
    for (int ph = 0; ph < U.u; ++ph) {
      ConvArgs a;
      a.in = xs;
      a.in_ld = U.cin;
      a.w = U.phase_w[ph];
      a.bias = U.b;
      a.out = x;
      a.out_ld = U.cout;
      a.cin = U.cin;
      a.cout = U.cout;
      a.taps = U.k / U.u;
      a.dil = -1;
      a.off = U.phase_off[ph];
      a.act_in = ACT_LRELU;
      a.out_row_mul = U.u;
      a.out_row_off = ph;
      a.seg = sin;
      a.seg_out_start = sout.start;
      launch_conv(F.ctx, a);
    }
    const int C = U.cout;
    for (int j = 0; j < per; ++j) {
      const ResBlockW& R = M.resblocks[size_t(s) * per + j];
      const float* cur = x;
      for (size_t l = 0; l < R.c1.size(); ++l) {
        F.conv(R.c1[l], cur, C, t1, C, sout, R.dil[l], ACT_LRELU, ACT_NONE);
        bool last = l + 1 == R.c1.size();
        ConvArgs a;
        a.in = t1;
        a.in_ld = C;
        a.w = R.c2[l].w;
        a.bias = R.c2[l].b;
        a.out = last ? nullptr : r;
        a.out_ld = C;
        a.residual = cur;
        a.cin = C;
        a.cout = C;
        a.taps = R.c2[l].k;
        a.dil = 1;
        a.off = -((R.c2[l].k - 1) / 2);
        a.act_in = ACT_LRELU;
        a.seg = sout;
        if (last) {
          a.accum_out = xs;
          a.accum_mode = j == 0 ? ACC_SET : (j + 1 == per ? ACC_ADD_SCALE : ACC_ADD);
          a.accum_div = float(per);
          if (per == 1) {
            a.accum_mode = ACC_SET;
          }
        }
        launch_conv(F.ctx, a);
        cur = r;
      }
    }
  }
  Segs sl = segs_of(n_st);
  M.debug["dec_last"] = DebugView{xs, rows[n_st], M.dec_post_c, 4};
  launch_dec_post(F.ctx, wave, xs, M.dec_post_w, M.dec_post_c, M.dec_post_k, sl);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// run
// ---------------------------------------------------------------------------------------------
void synth_run(sbv2_model* mm, sbv2_device_batch* b) {
  auto* Mp = static_cast<SynthModel*>(mm);
  SynthModel& M = *Mp;
  M.bind_device();
  const HParams& hp = M.hp;
  Fwd F{M, M.ctx()};
  const LaunchCtx& ctx = F.ctx;
  const int B = b->B;
  const int H = hp.hidden;
  const int64_t Nx = b->Nx;
  uint8_t* in = b->in.as<uint8_t>();
  const int* d_x = reinterpret_cast<const int*>(in + b->o_x);
  const int* d_tone = reinterpret_cast<const int*>(in + b->o_tone);
  const int* d_lang = reinterpret_cast<const int*>(in + b->o_lang);
  const int64_t* d_sid = reinterpret_cast<const int64_t*>(in + b->o_sid);
  const float* d_ratio = reinterpret_cast<const float*>(in + b->o_sdp_ratio);
  const float* d_ls = reinterpret_cast<const float*>(in + b->o_ls);
  const float* d_ns = reinterpret_cast<const float*>(in + b->o_ns);
  const float* d_nsw = reinterpret_cast<const float*>(in + b->o_nsw);
  const float* d_style = reinterpret_cast<const float*>(in + b->o_style);
  Segs xseg;
  xseg.start = reinterpret_cast<const int*>(in + b->o_xstart);
  xseg.len = reinterpret_cast<const int*>(in + b->o_xlen);
  xseg.n = B;
  xseg.max_len = *std::max_element(b->xlen.begin(), b->xlen.end());
  // "batch rows" segment: one segment of B rows, for per-utterance linears
  // (start = 0, len = B) lives in the ylen_dev buffer's first two ints
  b->ylen_dev.stream = M.stream;
  b->ylen_dev.ensure(size_t(B + 2) * 4);
  {
    int two[2] = {0, B};
    CUDA_CHECK(cudaMemcpyAsync(b->ylen_dev.p, two, 8, cudaMemcpyHostToDevice, M.stream));
  }
  Segs bseg;
  bseg.start = b->ylen_dev.as<int>();
  bseg.len = b->ylen_dev.as<int>() + 1;
  bseg.n = 1;
  bseg.max_len = B;
  bseg.vectors = true;
  int* d_ylen = b->ylen_dev.as<int>() + 2;

  auto ens = [&](int id, size_t floats) { M.ws[id].ensure(floats * 4); return M.ws[id].as<float>(); };
  const int Cmax = std::max(std::max(3 * H, M.enc.filter), std::max(hp.dp_filter, 2 * hp.inter));
  float* bert = ens(W_BERT, size_t(Nx) * hp.bert_dim);
  float* h = ens(W_H, size_t(Nx) * H);
  ens(W_QKV, size_t(Nx) * 3 * H);
  ens(W_CTX, size_t(Nx) * H);
  ens(W_Y, size_t(Nx) * H);
  ens(W_F1, size_t(Nx) * Cmax);
  float* stats = ens(W_STATS, size_t(Nx) * 2 * hp.inter);
  float* g = ens(W_G, size_t(B) * hp.gin);
  float* style_emb = ens(W_STYLE, size_t(B) * H);
  ens(W_GG, size_t(B) * std::max(H, hp.up_initial));
  float* dpx = ens(W_DPX, size_t(Nx) * H);
  float* dp1 = ens(W_DP1, size_t(Nx) * hp.dp_filter);
  float* dp2 = ens(W_DP2, size_t(Nx) * hp.dp_filter);
  float* logw = ens(W_LOGW, size_t(Nx));
  float* wbuf = ens(W_W, size_t(Nx));

  // ---- speaker embedding, text encoder ------------------------------------------------------
  M.region_begin("text");
  BatchGeom tbg;
  if (M.use_tc_text && !M.text_tc.empty()) {
    std::vector<int> muls(1, 1);
    // tx_pin was last read by the previous run's text phase, which finished before that run's T_y read-back
    tbg = build_geoms(&M, M.tx_meta, M.tx_pin, b->xstart, b->xlen, muls, nullptr, /*pin_idle=*/true);
    const Geom& TG = tbg.g[0];
    const int nblk = M.text_terms == 3 ? 6 : 3;
    M.tx_split.ensure(size_t(TG.rows_tot) * nblk * M.text_tc_max_cin * 2);
    F.tg = &TG;
    F.tg_start = tbg.d_ystart;
    F.tg_seg_start = xseg.start;
    F.tg_split = M.tx_split.as<__half>();
    F.tg_n = B;
    F.tg_small = Nx <= M.small_text_rows;
    launch_zero_gaps(ctx, F.tg_split, nblk * M.text_tc_max_cin, TG, B);  // the splits only ever write utterance rows
  }
  launch_gather_rows(ctx, g, M.emb_g, d_sid, B, hp.gin, hp.n_speakers);
  if (b->dev_bert_rows) {
    // tts_util.rs:129-154 on the device: phoneme row i is the BERT row of its token (word2ph repeat), no transposes
    if (b->dev_bert_ready) CUDA_CHECK(cudaStreamWaitEvent(M.stream, b->dev_bert_ready, 0));
    launch_gather_rows(ctx, bert, b->dev_bert_rows, reinterpret_cast<const int64_t*>(in + b->o_bert), int(Nx), hp.bert_dim,
                       int(b->dev_bert_n));
  } else
    launch_cm_to_rm(ctx, reinterpret_cast<const float*>(in + b->o_bert), reinterpret_cast<const int64_t*>(in + b->o_bert_off),
                    nullptr, bert, hp.bert_dim, xseg);
  F.conv(M.bert_proj, bert, hp.bert_dim, h, H, xseg);
  F.conv(M.style_proj, d_style, hp.style_dim, style_emb, H, bseg);
  launch_embed_combine(ctx, h, d_x, d_tone, d_lang, M.emb, M.tone_emb, M.lang_emb, style_emb, H, hp.n_vocab, hp.n_tones,
                       hp.n_lang, xseg);
  F.encoder(M.enc, h, xseg, int(Nx), g, hp.gin, bseg);
  F.conv(M.enc_proj, h, H, stats, 2 * hp.inter, xseg);
  M.debug["enc_x"] = DebugView{h, Nx, H, 4};
  M.debug["stats"] = DebugView{stats, Nx, 2 * hp.inter, 4};

  // ---- duration predictor -------------------------------------------------------------------
  {
    float* gc = M.ws[W_GG].as<float>();
    F.conv(M.dp_cond, g, hp.gin, gc, H, bseg);
    launch_add_utt_vec(ctx, dpx, h, gc, H, H, xseg);
    F.conv(M.dp_c1, dpx, H, dp1, hp.dp_filter, xseg, 1, ACT_NONE, ACT_RELU);
    launch_layernorm(ctx, dp1, dp1, nullptr, nullptr, M.dp_n1.g, M.dp_n1.b, 1e-5f, ACT_NONE, hp.dp_filter, int(Nx));
    F.conv(M.dp_c2, dp1, hp.dp_filter, dp2, hp.dp_filter, xseg, 1, ACT_NONE, ACT_RELU);
    launch_layernorm(ctx, dp2, dp2, nullptr, nullptr, M.dp_n2.g, M.dp_n2.b, 1e-5f, ACT_NONE, hp.dp_filter, int(Nx));
    F.conv(M.dp_proj, dp2, hp.dp_filter, logw, 1, xseg);
    M.debug["logw_dp"] = DebugView{logw, Nx, 1, 4};
  }

  // ---- stochastic duration predictor (reverse) -----------------------------------------------
  float* zs = nullptr;
  if (b->any_sdp) {
    float* sx = ens(W_SDPX, size_t(Nx) * H);
    float* sh = ens(W_SDPH, size_t(Nx) * H);
    float* t1 = ens(W_SDPT, size_t(Nx) * H * 2);
    float* t2 = t1 + size_t(Nx) * H;
    zs = ens(W_SDPZ, size_t(Nx) * 2);
    float* nrm = ens(W_NSDP, size_t(Nx) * 2);
    float* gc = M.ws[W_GG].as<float>();
    F.conv(M.sdp_cond, g, hp.gin, gc, H, bseg);
    F.conv(M.sdp_pre, h, H, sx, H, xseg, 1, ACT_NONE, ACT_NONE, nullptr, gc);
    F.dds(M.sdp_dds, sx, t1, t2, H, xseg, int(Nx));
    F.conv(M.sdp_proj, sx, H, sh, H, xseg);  // conditioning for the flows
    float* cond = sh;
    if (b->has_noise_sdp) {
      launch_cm_to_rm(ctx, reinterpret_cast<const float*>(in + b->o_nsdp), reinterpret_cast<const int64_t*>(in + b->o_nsdp_off),
                      nullptr, nrm, 2, xseg);
    } else {
      launch_randn(ctx, nrm, Nx * 2, M.seed, M.rng_offset);
      M.rng_offset += uint64_t(Nx) * 2;
    }
    launch_sdp_init(ctx, zs, nrm, d_nsw, xseg);
    // reversed flow list with the first ConvFlow dropped: Flip, CF[n-1], Flip, ..., CF[1], Flip, EA
    float* hh = sx;  // sx no longer needed after sdp_proj
    const float inv_sqrt = 1.0f / sqrtf(float(H));
    for (int i = int(M.sdp_cf.size()) - 1; i >= 1; --i) {
      const ConvFlowW& cf = M.sdp_cf[i];
      launch_sdp_flip(ctx, zs, int(Nx));
      launch_convflow_pre(ctx, hh, zs, cf.pre_w, cf.pre_b, cond, H, int(Nx));
      F.dds(cf.dds, hh, t1, t2, H, xseg, int(Nx));
      F.conv(cf.proj, hh, H, t1, cf.proj.cout, xseg);
      launch_convflow_spline(ctx, zs, t1, cf.proj.cout, hp.sdp_bins, 5.0f, inv_sqrt, int(Nx));
    }
    launch_sdp_flip(ctx, zs, int(Nx));
    launch_sdp_affine(ctx, zs, M.sdp_ea_m, M.sdp_ea_logs, int(Nx));
    M.debug["z_sdp"] = DebugView{zs, Nx, 2, 4};
  }

  // ---- durations / alignment -------------------------------------------------------------------
  b->dur.stream = b->cum.stream = M.stream;
  b->dur.ensure(size_t(Nx) * 4);
  b->cum.ensure(size_t(Nx) * 4);
  launch_durations(ctx, logw, zs, d_ratio, d_ls, wbuf, b->dur.as<int>(), b->cum.as<int>(), d_ylen, xseg);
  M.debug["w"] = DebugView{wbuf, Nx, 1, 4};
  M.region_end("text");
  M.pin_ylen.ensure(size_t(B) * 4);
  CUDA_CHECK(cudaMemcpyAsync(M.pin_ylen.p, d_ylen, size_t(B) * 4, cudaMemcpyDeviceToHost, M.stream));
  M.wait_stream(/*yield=*/B >= 8);
  b->ylen.assign(M.pin_ylen.as<int>(), M.pin_ylen.as<int>() + B);
  b->ystart.resize(B);
  int64_t ny = 0;
  int ymax = 0;
  for (int i = 0; i < B; ++i) {
    b->ystart[i] = int(ny);
    ny += b->ylen[i];
    ymax = std::max(ymax, b->ylen[i]);
    if (b->has_noise_zp && b->zp_frames[i] < b->ylen[i])
      fail(SBV2_ERR_INVALID_ARGUMENT, "noise_zp has " + std::to_string(b->zp_frames[i]) + " frames but utterance " +
                                          std::to_string(i) + " needs T_y = " + std::to_string(b->ylen[i]));
  }
  if (ny * hp.hop > (int64_t(1) << 31) - 1) fail(SBV2_ERR_INVALID_ARGUMENT, "batch too long: more than 2^31 samples");
  b->Ny = ny;
  {
    // ymeta: ystart[B], ylen[B], zp_ld[B] (ints) then zp_off[B] (int64); staged in pinned memory — the stream is idle
    // here (the T_y read-back just synchronised it), so the previous run's copy out of the staging block is complete
    // and no second synchronisation is needed
    const size_t ibytes = align_up(size_t(3) * B * 4, 256);
    const size_t mbytes = ibytes + size_t(B) * 8;
    M.pin_ymeta.ensure(mbytes);
    int* meta = M.pin_ymeta.as<int>();
    int64_t* zoff = reinterpret_cast<int64_t*>(M.pin_ymeta.as<uint8_t>() + ibytes);
    int64_t o = 0;
    for (int i = 0; i < B; ++i) {
      meta[i] = b->ystart[i];
      meta[B + i] = b->ylen[i];
      meta[2 * B + i] = int(b->zp_frames[i]);
      zoff[i] = o;
      o += b->zp_frames[i] * hp.inter;
    }
    b->ymeta.stream = M.stream;
    b->ymeta.ensure(mbytes);
    CUDA_CHECK(cudaMemcpyAsync(b->ymeta.p, M.pin_ymeta.p, mbytes, cudaMemcpyHostToDevice, M.stream));
    b->o_zp_off = ibytes;
  }
  // waveform layout: utterances back to back, plus the caller's pauses (written as zeros on the device)
  {
    b->wstart.resize(B);
    long long w = 0;
    bool any_pause = false;
    for (int i = 0; i < B; ++i) {
      b->wstart[i] = w;
      w += (long long)b->ylen[i] * hp.hop;
      if (!b->pause_after.empty() && b->pause_after[i] > 0) {
        w += b->pause_after[i];
        any_pause = true;
      }
    }
    if (w > (int64_t(1) << 31) - 1) fail(SBV2_ERR_INVALID_ARGUMENT, "batch too long: more than 2^31 samples");
    b->wave_total = w;
    b->wave.stream = M.stream;
    b->wave.ensure(size_t(std::max<long long>(w, 1)) * 4);
    if (any_pause) CUDA_CHECK(cudaMemsetAsync(b->wave.p, 0, size_t(w) * 4, M.stream));
  }
  Segs yseg;
  yseg.start = b->ymeta.as<int>();
  yseg.len = b->ymeta.as<int>() + B;
  yseg.n = B;
  yseg.max_len = ymax;

  // ---- expand + prior sample ---------------------------------------------------------------------
  M.region_begin("flow");
  const int C = hp.inter;
  float* eps = ens(W_EPS, size_t(ny) * C);
  float* z = ens(W_Z, size_t(ny) * C);
  float* z2 = ens(W_Z2, size_t(ny) * C);
  float* mbuf = ens(W_M, size_t(ny) * C);
  b->f2p.stream = M.stream;
  b->f2p.ensure(size_t(ny) * 4);
  if (b->has_noise_zp) {
    launch_cm_to_rm(ctx, b->zp.as<float>(), reinterpret_cast<const int64_t*>(b->ymeta.as<uint8_t>() + b->o_zp_off),
                    b->ymeta.as<int>() + 2 * B, eps, C, yseg);
  } else {
    launch_randn(ctx, eps, ny * C, M.seed ^ 0x9E3779B97F4A7C15ULL, M.rng_offset);
    M.rng_offset += uint64_t(ny) * C;
  }
  launch_expand(ctx, z, b->f2p.as<int>(), stats, b->cum.as<int>(), eps, d_ns, C, xseg, yseg);
  M.debug["z_p"] = DebugView{z, ny, C, 4};

  // ---- flow (reverse) ------------------------------------------------------------------------------
  ens(W_QKV, size_t(ny) * 3 * H);
  ens(W_CTX, size_t(ny) * H);
  ens(W_Y, size_t(ny) * H);
  ens(W_F1, size_t(ny) * std::max(hp.transformer_flow ? M.flow[0].enc.filter : 2 * H, 2 * H));
  float* hf = ens(W_HF, size_t(ny) * H);
  float* zc = z;
  float* zn = z2;
  if (M.use_tc_flow) {
    // tensor-core path: fp16 planar operands, fp32 residual stream hf
    std::vector<int> muls(1, 1);
    BatchGeom bg = build_geoms(&M, M.fl_meta, M.fl_pin, b->ystart, b->ylen, muls, nullptr, /*pin_idle=*/true);  // stream idle since the T_y read-back
    const Geom& G = bg.g[0];
    PlanarSegs ps;
    ps.start = bg.d_ystart;
    ps.pstart = G.d_pstart;
    ps.len = G.d_len;
    ps.order = bg.d_order;
    ps.n = B;
    ps.max_len = ymax;
    ps.plane_stride = G.rows_tot * 8;
    const int filt = M.flow[0].enc.filter;
    M.fl_x0p.ensure(size_t(G.rows_tot) * (C / 2) * 2);
    M.fl_hp.ensure(size_t(G.rows_tot) * H * 2);
    M.fl_qkvp.ensure(size_t(G.rows_tot) * 3 * H * 2);
    if (M.fl_qkvp.gen != M.fl_qkvp_gen) {
      // rows past an utterance's end are read (and masked) by the attention: they must hold finite values
      CUDA_CHECK(cudaMemsetAsync(M.fl_qkvp.p, 0, M.fl_qkvp.cap, M.stream));
      M.fl_qkvp_gen = M.fl_qkvp.gen;
    }
    M.fl_ctxp.ensure(size_t(G.rows_tot) * H * 2);
    M.fl_f1p.ensure(size_t(G.rows_tot) * filt * 2);
    M.fl_y32.ensure(size_t(G.rows_tot) * H * 4);
    M.fl_m32.ensure(size_t(G.rows_tot) * (C / 2) * 4);
    __half* x0p = M.fl_x0p.as<__half>();
    __half* hp16 = M.fl_hp.as<__half>();
    __half* qkvp = M.fl_qkvp.as<__half>();
    __half* ctxp = M.fl_ctxp.as<__half>();
    __half* f1p = M.fl_f1p.as<__half>();
    float* y32 = M.fl_y32.as<float>();
    float* m32 = M.fl_m32.as<float>();
    launch_zero_gaps(ctx, hp16, H, G, B);
    launch_zero_gaps(ctx, f1p, filt, G, B);
    const int sm = ny <= M.small_flow_rows ? 1 : 0;  // few frames: the 64-wide packing (more CTAs per weight stream)
    auto umma = [&](const ConvLayer& L, const __half* in, __half* out, float* acc32, int act) {
      ConvCall c;
      c.in = in;
      c.out = out;
      c.accum = acc32;
      c.accum_mode = acc32 ? UACC_SET : UACC_NONE;
      c.act_out = act;
      launch_umma(ctx, L, G, G, c, B);
    };
    for (int i = hp.n_flows - 1; i >= 0; --i) {
      const CouplingW& cp = M.flow[i];
      const FlowTC& T = M.flow_tc[i];
      launch_flip_channels(ctx, zn, zc, C, ny);
      std::swap(zc, zn);
      launch_to_planar(ctx, x0p, zc, C, C / 2, bg.d_ystart, G, B, ACT_NONE);
      umma(T.pre[sm], x0p, nullptr, y32, ACT_NONE);
      launch_flow_mix(ctx, hf, hp16, nullptr, y32, nullptr, 0, H, ps);
      const EncoderW& E = cp.enc;
      for (size_t l = 0; l < E.layers.size(); ++l) {
        const EncLayerW& Lw = E.layers[l];
        const FlowTCLayer& Lt = T.layers[l];
        if (E.has_spk && int(l) == E.cond_idx) {
          float* gg = M.ws[W_GG].as<float>();
          F.conv(E.spk, g, hp.gin, gg, H, bseg);
          launch_flow_mix(ctx, hf, hp16, hf, nullptr, gg, H, H, ps);
        }
        umma(Lt.qkv[sm], hp16, qkvp, nullptr, ACT_NONE);
        if (M.use_tc_attn) launch_flow_attention_tc(ctx, ctxp, qkvp, Lt.rel_k_p, Lt.rel_v_p, E.heads, E.head_dim, E.window, ps);
        else launch_rel_attention_planar(ctx, ctxp, qkvp, Lw.rel_k, Lw.rel_v, E.heads, E.head_dim, E.window, ps);
        umma(Lt.o[sm], ctxp, nullptr, y32, ACT_NONE);
        launch_ln_planar(ctx, hf, hp16, y32, Lw.n1.g, Lw.n1.b, 1e-5f, H, ps);
        umma(Lt.f1[sm], hp16, f1p, nullptr, ACT_RELU);
        umma(Lt.f2[sm], f1p, nullptr, y32, ACT_NONE);
        launch_ln_planar(ctx, hf, hp16, y32, Lw.n2.g, Lw.n2.b, 1e-5f, H, ps);
      }
      umma(T.post[sm], hp16, nullptr, m32, ACT_NONE);
      launch_coupling_sub_planar(ctx, zc, m32, C, ps);
    }
  } else if (M.use_tc_wn) {
    // WN coupling layers on the tensor cores: fp16 planar operands, fp32 planar [x | skip] stream
    std::vector<int> muls(1, 1);
    BatchGeom bg = build_geoms(&M, M.fl_meta, M.fl_pin, b->ystart, b->ylen, muls, nullptr, /*pin_idle=*/true);
    const Geom& G = bg.g[0];
    PlanarSegs ps;
    ps.start = bg.d_ystart;
    ps.pstart = G.d_pstart;
    ps.len = G.d_len;
    ps.order = bg.d_order;
    ps.n = B;
    ps.max_len = ymax;
    ps.plane_stride = G.rows_tot * 8;
    const int nl = hp.wn_layers;
    M.fl_x0p.ensure(size_t(G.rows_tot) * (C / 2) * 2);
    M.fl_hp.ensure(size_t(G.rows_tot) * H * 2);
    M.fl_ctxp.ensure(size_t(G.rows_tot) * H * 2);
    M.fl_y32.ensure(size_t(G.rows_tot) * 2 * H * 4);
    M.fl_m32.ensure(size_t(G.rows_tot) * (C / 2) * 4);
    __half* x0p = M.fl_x0p.as<__half>();
    __half* xp = M.fl_hp.as<__half>();
    __half* actp = M.fl_ctxp.as<__half>();
    float* acc = M.fl_y32.as<float>();                            // planes [0, H/8): x, [H/8, 2H/8): skip
    float* acc_skip = acc + size_t(H / 8) * size_t(ps.plane_stride);
    float* m32 = M.fl_m32.as<float>();
    launch_zero_gaps(ctx, xp, H, G, B);
    launch_zero_gaps(ctx, actp, H, G, B);
    float* gcond = ens(W_STYLE, size_t(B) * 2 * H * nl);
    for (int i = hp.n_flows - 1; i >= 0; --i) {
      const WnTC& T = M.wn_tc[size_t(i)];
      launch_flip_channels(ctx, zn, zc, C, ny);
      std::swap(zc, zn);
      launch_to_planar(ctx, x0p, zc, C, C / 2, bg.d_ystart, G, B, ACT_NONE);
      CUDA_CHECK(cudaMemsetAsync(acc_skip, 0, size_t(H / 8) * size_t(ps.plane_stride) * 4, M.stream));  // output = zeros_like(x)
      {
        ConvCall c;
        c.in = x0p;
        c.accum = acc;
        c.accum_mode = UACC_SET;
        launch_umma(ctx, T.pre, G, G, c, B);
      }
      F.conv(T.cond_perm, g, hp.gin, gcond, 2 * H * nl, bseg);
      for (int l = 0; l < nl; ++l) {
        launch_planar_cast(ctx, xp, acc, H, G, B);
        {
          ConvCall c;
          c.in = xp;
          c.out = actp;
          c.gate_half = T.gate_half;
          c.bias_utt = gcond + size_t(l) * 2 * H;
          c.bias_utt_ld = 2 * H * nl;
          launch_umma(ctx, T.in_layers[size_t(l)], G, G, c, B);
        }
        ConvCall c;
        c.in = actp;
        c.accum = l == nl - 1 ? acc_skip : acc;  // last layer: all of res_skip goes to the output sum
        c.accum_mode = UACC_ADD;
        launch_umma(ctx, T.res_skip[size_t(l)], G, G, c, B);
      }
      launch_planar_cast(ctx, xp, acc_skip, H, G, B);
      {
        ConvCall c;
        c.in = xp;
        c.accum = m32;
        c.accum_mode = UACC_SET;
        launch_umma(ctx, T.post, G, G, c, B);
      }
      launch_coupling_sub_planar(ctx, zc, m32, C, ps);
    }
  } else
  for (int i = hp.n_flows - 1; i >= 0; --i) {
    const CouplingW& cp = M.flow[i];
    launch_flip_channels(ctx, zn, zc, C, ny);
    std::swap(zc, zn);
    // x0 = zc[:, :C/2]
    F.conv(cp.pre, zc, C, hf, H, yseg);
    if (hp.transformer_flow) {
      F.encoder(cp.enc, hf, yseg, int(ny), g, hp.gin, bseg);
      F.conv(cp.post, hf, H, mbuf, C / 2, yseg);
    } else {
      // WN: cond = cond_layer(g) [B, 2H*n]; per layer gate + res/skip
      const WNW& W = cp.wn;
      const int nl = int(W.in_layers.size());
      float* gcond = ens(W_STYLE, size_t(B) * 2 * H * nl);
      F.conv(W.cond, g, hp.gin, gcond, 2 * H * nl, bseg);
      float* a = M.ws[W_F1].as<float>();    // [ny, 2H]
      float* acts = M.ws[W_CTX].as<float>();  // [ny, H]
      float* rs = M.ws[W_QKV].as<float>();   // [ny, 2H]
      float* skip = M.ws[W_Y].as<float>();   // [ny, H]
      for (int l = 0; l < nl; ++l) {
        F.conv(W.in_layers[l], hf, H, a, 2 * H, yseg);
        launch_wn_gate(ctx, acts, a, gcond, 2 * H * nl, l * 2 * H, H, yseg);
        F.conv(W.res_skip[l], acts, H, rs, W.res_skip[l].cout, yseg);
        launch_wn_res_skip(ctx, hf, skip, rs, H, l == nl - 1, l == 0, ny);
      }
      F.conv(cp.post, skip, H, mbuf, C / 2, yseg);
    }
    launch_coupling_sub(ctx, zc, mbuf, C, ny);
  }
  M.debug["z"] = DebugView{zc, ny, C, 4};
  M.region_end("flow");

  // ---- decoder ---------------------------------------------------------------------------------------
  M.region_begin("decoder");
  if (M.use_umma && M.umma) {
    umma_decoder_run(M.umma, &M, zc, g, B, b->ystart, b->ylen, b->wave.as<float>(), &b->wstart);
  } else {
    if (b->wave_total != ny * hp.hop) fail(SBV2_ERR_UNSUPPORTED, "pauses between utterances need the tensor-core decoder");
    decoder_fp32(M, zc, g, yseg, bseg, b->ystart, b->ylen, b->wave.as<float>(), M.ws[W_META]);
  }
  M.region_end("decoder");
  b->ran = true;
}

int64_t synth_total_samples(sbv2_model* m, const sbv2_device_batch* b) { return b->Ny * static_cast<SynthModel*>(m)->hp.hop; }
int64_t synth_wave_total(const sbv2_device_batch* b) { return b->wave_total; }
void synth_set_pauses(sbv2_device_batch* b, const int64_t* pause_after) {
  b->pause_after.assign(pause_after, pause_after + b->B);
  for (int64_t v : b->pause_after) SBV2_REQUIRE(v >= 0 && v < (int64_t(1) << 28), "pause length out of range");
}
bool synth_borrows_host(const sbv2_device_batch* b) { return b->borrowed_host; }

void synth_batch_ty(const sbv2_device_batch* b, int64_t* ty) {
  for (int i = 0; i < b->B; ++i) ty[i] = b->ylen[i];
}

void synth_download(sbv2_model* mm, sbv2_device_batch* b, float** out_samples, int64_t* out_n, int32_t** out_dur, int32_t** out_f2p) {
  auto* M = static_cast<SynthModel*>(mm);
  SBV2_REQUIRE(b->ran, "batch has not been run");
  M->bind_device();
  const int64_t total = b->wave_total;
  float* host = static_cast<float*>(alloc_out(size_t(std::max<int64_t>(total, 1)) * 4, true));
  int32_t* hdur = nullptr;
  int32_t* hf2p = nullptr;
  try {
    CUDA_CHECK(cudaMemcpyAsync(host, b->wave.p, size_t(total) * 4, cudaMemcpyDeviceToHost, M->stream));
    if (out_dur && !b->decode_only) {
      hdur = static_cast<int32_t*>(alloc_out(size_t(b->Nx) * 4, true));
      CUDA_CHECK(cudaMemcpyAsync(hdur, b->dur.p, size_t(b->Nx) * 4, cudaMemcpyDeviceToHost, M->stream));
    }
    if (out_f2p && !b->decode_only) {
      hf2p = static_cast<int32_t*>(alloc_out(size_t(b->Ny) * 4, true));
      CUDA_CHECK(cudaMemcpyAsync(hf2p, b->f2p.p, size_t(b->Ny) * 4, cudaMemcpyDeviceToHost, M->stream));
    }
    M->wait_stream(/*yield=*/b->B >= 8);
  } catch (...) {
    free_out(host);
    free_out(hdur);
    free_out(hf2p);
    throw;
  }
  *out_samples = host;
  if (out_n)
    for (int i = 0; i < b->B; ++i) out_n[i] = int64_t(b->ylen[i]) * M->hp.hop;
  if (out_dur) *out_dur = hdur;
  if (out_f2p) *out_f2p = hf2p;
}

void synth_batch_free(sbv2_device_batch* b) {
  if (!b) return;
  if (b->bufs) {
    auto* M = static_cast<SynthModel*>(b->owner);
    if (M && M->batch_pool.size() < 4) M->batch_pool.push_back(b->bufs);
    else delete b->bufs;  // DBuf destructors free the device memory
  }
  delete b;
}

// HiFi-GAN decoder alone (config 3)
void synth_decode(sbv2_model* mm, const float* const* z, const int64_t* t_y, const int64_t* sid, int batch, float** out_samples,
                  int64_t* out_n) {
  auto* Mp = static_cast<SynthModel*>(mm);
  SynthModel& M = *Mp;
  SBV2_REQUIRE(!M.is_bert, "decode called on a BERT model");
  SBV2_REQUIRE(z && t_y && sid && batch > 0, "empty batch");
  M.bind_device();
  const HParams& hp = M.hp;
  std::unique_ptr<sbv2_device_batch, void (*)(sbv2_device_batch*)> bp(new sbv2_device_batch(borrow_buffers(M), &M), synth_batch_free);
  sbv2_device_batch& b = *bp;
  b.B = batch;
  b.decode_only = true;
  b.ylen.resize(batch);
  b.ystart.resize(batch);
  int64_t ny = 0;
  int ymax = 0;
  for (int i = 0; i < batch; ++i) {
    SBV2_REQUIRE(t_y[i] > 0 && t_y[i] < (1 << 22), "t_y out of range");
    SBV2_REQUIRE(sid[i] >= 0 && sid[i] < hp.n_speakers, "speaker id out of range");
    b.ylen[i] = int(t_y[i]);
    b.ystart[i] = int(ny);
    ny += t_y[i];
    ymax = std::max(ymax, b.ylen[i]);
  }
  SBV2_REQUIRE(ny * hp.hop < (int64_t(1) << 31), "batch too long");
  b.Ny = ny;
  const int C = hp.inter;
  // stage z (channel-major) + meta
  size_t meta_ints = size_t(2) * batch + 2;
  size_t o_meta = 0, o_off = align_up(meta_ints * 4, 256), o_sid = align_up(o_off + size_t(batch) * 8, 256),
         o_z = align_up(o_sid + size_t(batch) * 8, 256), total = o_z + size_t(ny) * C * 4;
  CUDA_CHECK(cudaStreamSynchronize(M.stream));
  M.pin_in.ensure(total);
  uint8_t* hbuf = M.pin_in.as<uint8_t>();
  int* hmeta = reinterpret_cast<int*>(hbuf + o_meta);
  int64_t* hoff = reinterpret_cast<int64_t*>(hbuf + o_off);
  int64_t* hsid = reinterpret_cast<int64_t*>(hbuf + o_sid);
  float* hz = reinterpret_cast<float*>(hbuf + o_z);
  for (int i = 0; i < batch; ++i) {
    hmeta[i] = b.ystart[i];
    hmeta[batch + i] = b.ylen[i];
    hoff[i] = int64_t(b.ystart[i]) * C;
    hsid[i] = sid[i];
    memcpy(hz + size_t(b.ystart[i]) * C, z[i], size_t(b.ylen[i]) * C * 4);
  }
  hmeta[2 * batch] = 0;
  hmeta[2 * batch + 1] = batch;
  b.in.stream = M.stream;
  b.in.ensure(total);
  CUDA_CHECK(cudaMemcpyAsync(b.in.p, hbuf, total, cudaMemcpyHostToDevice, M.stream));
  uint8_t* in = b.in.as<uint8_t>();
  Segs yseg;
  yseg.start = reinterpret_cast<const int*>(in + o_meta);
  yseg.len = yseg.start + batch;
  yseg.n = batch;
  yseg.max_len = ymax;
  Segs bseg;
  bseg.start = yseg.start + 2 * batch;
  bseg.len = bseg.start + 1;
  bseg.n = 1;
  bseg.max_len = batch;
  bseg.vectors = true;
  M.ws[W_Z].ensure(size_t(ny) * C * 4);
  M.ws[W_G].ensure(size_t(batch) * hp.gin * 4);
  float* zr = M.ws[W_Z].as<float>();
  float* g = M.ws[W_G].as<float>();
  LaunchCtx ctx = M.ctx();
  launch_cm_to_rm(ctx, reinterpret_cast<const float*>(in + o_z), reinterpret_cast<const int64_t*>(in + o_off), nullptr, zr, C, yseg);
  launch_gather_rows(ctx, g, M.emb_g, reinterpret_cast<const int64_t*>(in + o_sid), batch, hp.gin, hp.n_speakers);
  b.wave.stream = M.stream;
  b.wave.ensure(size_t(ny) * hp.hop * 4);
  b.wave_total = ny * hp.hop;
  M.region_begin("decoder");
  if (M.use_umma && M.umma) {
    umma_decoder_run(M.umma, &M, zr, g, batch, b.ystart, b.ylen, b.wave.as<float>());
  } else {
    decoder_fp32(M, zr, g, yseg, bseg, b.ystart, b.ylen, b.wave.as<float>(), M.ws[W_META]);
  }
  M.region_end("decoder");
  b.ran = true;
  synth_download(mm, &b, out_samples, out_n, nullptr, nullptr);
}

}  // namespace sbv2
