// DeBERTa-v2 feature encoder (deberta.onnx) as a static kernel plan.
// Replaces the `ort::Session::run` of crates/sbv2_core/src/bert.rs:11-16.  The graph is
// HF DebertaV2ForMaskedLM up to hidden_states[-3] (scripts/convert/convert_deberta.py:27-35): only
// encoder layers 0..L-3 are live; the MLM head and the last two layers are never computed.
// Two numerics modes, chosen at model creation (SBV2_B200_BERT):
//   exact (default)  every GEMM and the k=3 ConvLayer on tcgen05 with two-term fp16 operand splits (~fp32 products, the
//                    text encoder's scheme, umma_conv.h make_split_conv1d_layer), fp32 row-major activations between
//                    them, fp32 CUDA-core disentangled attention.  The features feed bert_proj -> enc_p -> ceil() in the
//                    synthesizer, and durations must match the reference bit for bit: single-term fp16 operands perturb
//                    the features by 1.4e-3 (relative) and flip ~1 duration in 1000 (tests/test_gpu_fullsize.py chain test).
//   fp16             single-term fp16 operands and planar fp16 activations (3x fewer tensor FLOPs), tensor-core
//                    disentangled attention: the throughput mode, feature error ~1e-3.
#include <algorithm>
#include <climits>
#include <cmath>
#include <sstream>

#include "model.h"
#include "onnx_bind.h"
#include "umma_conv.h"

namespace sbv2 {
namespace {

struct BertLayer {
  ConvLayer qkv, o, f1, f2;
  // the same GEMMs packed with 64-wide N blocks: a call with few tokens (one sentence, bert.rs:6-24 as the reference
  // calls it) is a pure weight stream, and 256-wide blocks would leave it to 4-16 CTAs (f2: 4 CTAs x 6 MB each)
  ConvLayer qkv_s, o_s, f1_s, f2_s;
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  float *pos_k = nullptr, *pos_q = nullptr;  // [hidden, 2*span] (transposed) projections of LN(rel_embeddings)
  __half *pos_k_p = nullptr, *pos_q_p = nullptr;  // the same as fp16 [heads][64/8][2*span][8] (tensor-core attention operands)
  // exact mode: two-term fp16 splits of the same tables, [2 terms][heads][64/8][2*span][8], values scaled by kSplitScale
  __half *pos_k_s = nullptr, *pos_q_s = nullptr;
};

struct BertModel : sbv2_model {
  int hidden = 0, heads = 0, inter = 0, vocab = 0, n_layers_total = 0, n_run = 0, span = 0, max_rel = 0;
  float eps = 1e-7f;
  float* word_emb = nullptr;
  float *emb_g = nullptr, *emb_b = nullptr;
  std::vector<BertLayer> layers;
  bool has_conv = false;
  ConvLayer conv, conv_s;
  float *conv_g = nullptr, *conv_b = nullptr;
  int* bucket_idx = nullptr;  // device [2*max_rel+1] (bert_bucket_table)
  DBuf ids, h, embp, hp, qkvp, ctxp, f1p, y32, meta, outd;
  DBuf meand;                  // bert_token_mean's output; like outd, valid until the model's next call
  const int* out_len = nullptr;  // device [batch]: valid tokens of each row of outd (in `meta`)
  int out_batch = 0;
  int64_t out_S = 0;
  uint64_t qkvp_cleared_gen = 0;  // DBuf::gen of the qkv buffer that was zero-filled last (its tail rows must be finite)
  bool use_tc_attn = true;       // SBV2_B200_BERT_ATTN=simt (read at model creation) keeps the CUDA-core attention
  bool exact = true;             // SBV2_B200_BERT=fp16 selects the single-term fp16 path
  int max_cin = 0;               // widest GEMM input (exact mode: size of the split buffer)
  DBuf x_emb, x_qkv, x_ctx, x_f1, x_y, x_split;  // exact mode: fp32 row-major activations + the split operand buffer
  DBuf x_qkvs;                   // exact mode, <= 128 tokens: q|k|v as split-planar operands of the tensor-core attention
  uint64_t x_qkvs_cleared_gen = 0;
  PinnedBuf pin_meta, pin_io;
};

std::string find_prefix(const OnnxModel& m) {
  for (const char* p : {"deberta.", "", "model.deberta.", "bert."})
    if (m.find(std::string(p) + "embeddings.word_embeddings.weight")) return p;
  fail(SBV2_ERR_UNSUPPORTED, "not a DeBERTa-v2 graph (embeddings.word_embeddings.weight missing)");
}

// HF make_log_bucket_position in float32, as torch evaluates it
// N block of the few-token weight packing.  64, not narrower: a one-sentence GEMM is bound by its per-CTA serial chain
// (K / 16 MMAs at the 48-cycle issue floor: 19 us for K = 12288) and by launch latency, not by the weight stream, so 16-wide
// blocks only multiply the CTAs that each re-read the activations (measured: 7.4 -> 8.9 ms exact, 2.8 -> 3.3 ms fp16)
constexpr int kSmallNb = 64;
constexpr float kSplitScale = 16.f;  // = ConvLayer::in_scale of the split layers (checked in the forward)
constexpr int64_t kSmallTokens = 256;  // calls with at most this many tokens use it

int log_bucket(int rel, int bucket_size, int max_position) {
  const int mid = bucket_size / 2;
  const int sign = (rel > 0) - (rel < 0);
  const int abs_pos = (rel < mid && rel > -mid) ? mid - 1 : std::abs(rel);
  if (abs_pos <= mid) return rel;
  const float log_pos = std::ceil(std::log(float(abs_pos) / float(mid)) / std::log(float(max_position - 1) / float(mid)) * float(mid - 1)) + float(mid);
  return int(log_pos) * sign;
}

}  // namespace

std::vector<int> bert_bucket_table(int span, int* max_rel) {
  if (span < 2) fail(SBV2_ERR_UNSUPPORTED, "DeBERTa position_buckets must be at least 2");
  const int hi = 2 * span - 1;
  auto idx = [&](int d) { return std::min(std::max(log_bucket(d, span, 2 * span) + span, 0), hi); };  // max_position = 2*span
  // the log buckets grow without bound, so the clamp saturates both ends; R = the first distance where both have
  // (HF span 256: idx(-512) = 0 but idx(-511) = 1, idx(d) = 511 from d = 506 on, so R = 512)
  int R = 1;
  while (idx(R) != hi || idx(-R) != 0)
    if (++R > 4 * kMaxBertTokens) fail(SBV2_ERR_UNSUPPORTED, "DeBERTa position buckets do not saturate");
  // every distance a sequence within the cap can form must read the same row as R once clamped to it
  for (int d = R; d < kMaxBertTokens; ++d)
    if (idx(d) != hi || idx(-d) != 0) fail(SBV2_ERR_INTERNAL, "DeBERTa bucket table is not saturated beyond its bound");
  std::vector<int> tab(size_t(2) * R + 1);
  for (int d = -R; d <= R; ++d) tab[size_t(d + R)] = idx(d);
  *max_rel = R;
  return tab;
}

sbv2_model* create_bert_model(const OnnxModel& m, int device) {
  std::unique_ptr<BertModel> M(new BertModel());
  M->device = device;
  M->is_bert = true;
  CUDA_CHECK(cudaSetDevice(device));
  CUDA_CHECK(cudaStreamCreateWithFlags(&M->stream, cudaStreamNonBlocking));
  {
    const char* pe = getenv("SBV2_B200_PDL");
    M->pdl = !(pe && pe[0] == '0');  // on by default
  }
  M->metadata = m.metadata;
  const std::string P = find_prefix(m);
  // real exports keep only biases / embeddings / LayerNorm parameters named: every Linear weight is an anonymous
  // transposed onnx::MatMul_N initializer, bound here through the Add that applies its bias (onnx_bind.h)
  WeightBinder binder(m);
  binder.require_weights_for_biases(P + "encoder.layer.");
  auto get = [&](const std::string& n) -> const OnnxTensor& {
    const OnnxTensor* t = binder.find(P + n);
    if (!t) fail(SBV2_ERR_UNSUPPORTED, "DeBERTa graph lacks initializer '" + P + n + "'");
    return *t;
  };
  auto f32 = [&](const std::string& n) { return m.as_f32(get(n)); };
  auto vec = [&](const std::string& n, int expect) {
    auto v = f32(n);
    if (int(v.size()) != expect) fail(SBV2_ERR_UNSUPPORTED, "initializer '" + n + "' has unexpected size");
    return M->upload_f32(v);
  };
  const OnnxTensor& we = get("embeddings.word_embeddings.weight");
  if (we.dims.size() != 2) fail(SBV2_ERR_UNSUPPORTED, "word embeddings must be 2-D");
  M->vocab = int(we.dims[0]);
  M->hidden = int(we.dims[1]);
  if (m.find(P + "embeddings.position_embeddings.weight")) fail(SBV2_ERR_UNSUPPORTED, "position_biased_input=True is not supported");
  if (M->hidden % 64 != 0 || M->hidden > 1024) fail(SBV2_ERR_UNSUPPORTED, "hidden size must be a multiple of 64 and <= 1024");
  M->heads = M->hidden / 64;
  {
    const char* e = getenv("SBV2_B200_BERT_ATTN");
    M->use_tc_attn = !(e && std::string(e) == "simt");
  }
  {
    const char* e = getenv("SBV2_B200_BERT");
    M->exact = !(e && std::string(e) == "fp16");
  }
  M->word_emb = M->upload_f32(m.as_f32(we));
  M->emb_g = vec("embeddings.LayerNorm.weight", M->hidden);
  M->emb_b = vec("embeddings.LayerNorm.bias", M->hidden);
  int L = 0;
  while (binder.has(P + "encoder.layer." + std::to_string(L) + ".attention.self.query_proj.weight")) ++L;
  if (L < 3) fail(SBV2_ERR_UNSUPPORTED, "DeBERTa graph needs at least 3 encoder layers (output is hidden_states[-3])");
  M->n_layers_total = L;
  M->n_run = L - 2;
  const OnnxTensor& rel = get("encoder.rel_embeddings.weight");
  if (rel.dims.size() != 2 || rel.dims[1] != M->hidden || rel.dims[0] % 2 != 0) fail(SBV2_ERR_UNSUPPORTED, "unexpected rel_embeddings shape");
  M->span = int(rel.dims[0] / 2);
  LaunchCtx ctx = M->ctx();
  // LN(rel_embeddings) once (norm_rel_ebd = layer_norm)
  float* rel_raw = M->upload_f32(m.as_f32(rel));
  float* rel_ln = nullptr;
  {
    float* g = vec("encoder.LayerNorm.weight", M->hidden);
    float* b = vec("encoder.LayerNorm.bias", M->hidden);
    CUDA_CHECK(cudaMalloc(&rel_ln, size_t(2) * M->span * M->hidden * 4));
    M->owned_device.push_back(rel_ln);
    launch_layernorm(ctx, rel_ln, rel_raw, nullptr, nullptr, g, b, M->eps, ACT_NONE, M->hidden, 2 * M->span);
  }
  // one segment of 2*span rows for the load-time projections
  int two[2] = {0, 2 * M->span};
  int* d_two = static_cast<int*>(M->upload_bytes(two, 8));
  Segs pseg;
  pseg.start = d_two;
  pseg.len = d_two + 1;
  pseg.n = 1;
  pseg.max_len = 2 * M->span;
  auto host_linear = [&](const std::string& n) {
    HostConv hc;
    const OnnxTensor& t = get(n + ".weight");
    if (t.dims.size() < 2) fail(SBV2_ERR_UNSUPPORTED, n + ".weight must be a matrix");
    hc.d0 = int(t.dims[0]);
    hc.d1 = int(t.dims[1]);
    hc.k = t.dims.size() > 2 ? int(t.dims[2]) : 1;
    hc.w = m.as_f32(t);
    hc.b = f32(n + ".bias");
    return hc;
  };
  // N block of the batch packing.  256 (one CTA per 128 x 256 tile).  With SBV2_B200_BERT_NB=128 two adjacent blocks form the
  // N = 256 of one CTA-pair MMA (cta_group::2, ConvCall::pair, SBV2_B200_PAIR2=1) — built, bit-identical, and measured
  // slower: 32 x 128 tokens fp16 mode 6.27 ms (256, single CTA) / 8.48 ms (128, single) / 9.12 ms (128, pairs); exact mode
  // 23.1 / 29.7 / 32.2 ms (tools/bert_pair_ab.py, profiles/r2_cta_pair_ab.log)
  int big_nb = 256;
  if (const char* e = getenv("SBV2_B200_BERT_NB")) big_nb = atoi(e);
  DBuf wt;
  wt.stream = M->stream;
  const int H = M->hidden;
  for (int l = 0; l < M->n_run; ++l) {
    const std::string lp = "encoder.layer." + std::to_string(l);
    BertLayer B;
    HostConv q = host_linear(lp + ".attention.self.query_proj"), k = host_linear(lp + ".attention.self.key_proj"),
             v = host_linear(lp + ".attention.self.value_proj");
    if (q.d0 != H || q.d1 != H) fail(SBV2_ERR_UNSUPPORTED, "unexpected attention projection shape");
    // position projections (share_att_key): pos_k = key_proj(rel_ln), pos_q = query_proj(rel_ln); fp32, once per model
    for (int which = 0; which < 2; ++which) {
      const HostConv& hc = which == 0 ? k : q;
      std::vector<float> t(size_t(H) * H);
      for (int co = 0; co < H; ++co)
        for (int ci = 0; ci < H; ++ci) t[size_t(ci) * H + co] = hc.w[size_t(co) * H + ci];
      wt.ensure(t.size() * 4 + size_t(H) * 4);
      CUDA_CHECK(cudaMemcpyAsync(wt.p, t.data(), t.size() * 4, cudaMemcpyHostToDevice, M->stream));
      CUDA_CHECK(cudaMemcpyAsync(wt.as<float>() + t.size(), hc.b.data(), size_t(H) * 4, cudaMemcpyHostToDevice, M->stream));
      float* dst = nullptr;
      CUDA_CHECK(cudaMalloc(&dst, size_t(2) * M->span * H * 4));
      M->owned_device.push_back(dst);
      ConvArgs a;
      a.in = rel_ln;
      a.in_ld = H;
      a.w = wt.as<float>();
      a.bias = wt.as<float>() + t.size();
      a.out = dst;
      a.out_ld = H;
      a.cin = H;
      a.cout = H;
      a.seg = pseg;
      launch_conv(ctx, a);
      CUDA_CHECK(cudaStreamSynchronize(M->stream));  // `t` and wt are reused
      {
        // the attention kernel reads position rows per (head, channel): keep the projections transposed, [hidden][2*span]
        const size_t np2 = size_t(2) * M->span;
        std::vector<float> hrow(np2 * H), ht(np2 * H);
        CUDA_CHECK(cudaMemcpy(hrow.data(), dst, hrow.size() * 4, cudaMemcpyDeviceToHost));
        for (size_t r = 0; r < np2; ++r)
          for (int c = 0; c < H; ++c) ht[size_t(c) * np2 + r] = hrow[r * H + c];
        CUDA_CHECK(cudaMemcpy(dst, ht.data(), ht.size() * 4, cudaMemcpyHostToDevice));
        // planar fp16 per head: [head][channel / 8][row][channel % 8]
        std::vector<__half> hp16(np2 * H);
        for (int c = 0; c < H; ++c)
          for (size_t r = 0; r < np2; ++r) hp16[(size_t(c / 8) * np2 + r) * 8 + c % 8] = __float2half_rn(hrow[r * H + c]);
        (which == 0 ? B.pos_k_p : B.pos_q_p) = static_cast<__half*>(M->upload_bytes(hp16.data(), hp16.size() * 2));
        if (M->exact) {
          std::vector<__half> hs(2 * np2 * H);
          for (int c = 0; c < H; ++c)
            for (size_t r = 0; r < np2; ++r) {
              const float x = hrow[r * H + c] * kSplitScale;
              const __half h0 = __float2half_rn(x);
              const size_t o = (size_t(c / 8) * np2 + r) * 8 + c % 8;
              hs[o] = h0;
              hs[np2 * H + o] = __float2half_rn(x - __half2float(h0));
            }
          (which == 0 ? B.pos_k_s : B.pos_q_s) = static_cast<__half*>(M->upload_bytes(hs.data(), hs.size() * 2));
        }
      }
      (which == 0 ? B.pos_k : B.pos_q) = dst;
    }
    HostConv qkv;
    qkv.d0 = 3 * H;
    qkv.d1 = H;
    for (const HostConv* hc : {&q, &k, &v}) {
      qkv.w.insert(qkv.w.end(), hc->w.begin(), hc->w.end());
      qkv.b.insert(qkv.b.end(), hc->b.begin(), hc->b.end());
    }
    auto layer = [&](const HostConv& hc, int nb_max) {
      M->max_cin = std::max(M->max_cin, hc.d1);
      return M->exact ? make_split_conv1d_layer(M.get(), hc, 1, 1, 2, nb_max) : make_conv1d_layer(M.get(), hc, 1, 1, nb_max);
    };
    const HostConv od = host_linear(lp + ".attention.output.dense"), f2 = host_linear(lp + ".output.dense");
    HostConv f1 = host_linear(lp + ".intermediate.dense");
    M->inter = f1.d0;
    B.qkv = layer(qkv, big_nb);
    B.o = layer(od, big_nb);
    B.f1 = layer(f1, big_nb);
    B.f2 = layer(f2, big_nb);
    B.qkv_s = layer(qkv, kSmallNb);
    B.o_s = layer(od, kSmallNb);
    B.f1_s = layer(f1, kSmallNb);
    B.f2_s = layer(f2, kSmallNb);
    B.ln1_g = vec(lp + ".attention.output.LayerNorm.weight", H);
    B.ln1_b = vec(lp + ".attention.output.LayerNorm.bias", H);
    B.ln2_g = vec(lp + ".output.LayerNorm.weight", H);
    B.ln2_b = vec(lp + ".output.LayerNorm.bias", H);
    M->layers.push_back(B);
  }
  if (binder.has(P + "encoder.conv.conv.weight")) {
    HostConv c = host_linear("encoder.conv.conv");
    if (c.k % 2 == 0) fail(SBV2_ERR_UNSUPPORTED, "even ConvLayer kernel size");
    M->max_cin = std::max(M->max_cin, c.d1);
    M->conv = M->exact ? make_split_conv1d_layer(M.get(), c, 1, 1, 2) : make_conv1d_layer(M.get(), c, 1, 1);
    M->conv_s = M->exact ? make_split_conv1d_layer(M.get(), c, 1, 1, 2, kSmallNb) : make_conv1d_layer(M.get(), c, 1, 1, kSmallNb);
    M->conv_g = vec("encoder.conv.LayerNorm.weight", H);
    M->conv_b = vec("encoder.conv.LayerNorm.bias", H);
    M->has_conv = true;
  }
  {
    const std::vector<int> tab = bert_bucket_table(M->span, &M->max_rel);
    M->bucket_idx = static_cast<int*>(M->upload_bytes(tab.data(), tab.size() * 4));
  }
  for (DBuf* b : {&M->ids, &M->h, &M->embp, &M->hp, &M->qkvp, &M->ctxp, &M->f1p, &M->y32, &M->meta, &M->outd, &M->meand, &M->x_emb, &M->x_qkv, &M->x_qkvs, &M->x_ctx,
                  &M->x_f1, &M->x_y, &M->x_split})
    b->stream = M->stream;
  std::ostringstream js;
  js << "{\"kind\":\"deberta-v2\",\"hidden_size\":" << H << ",\"num_attention_heads\":" << M->heads << ",\"intermediate_size\":" << M->inter
     << ",\"vocab_size\":" << M->vocab << ",\"num_hidden_layers\":" << L << ",\"live_layers\":" << M->n_run
     << ",\"position_buckets\":" << M->span << ",\"conv_layer\":" << (M->has_conv ? "true" : "false") << ",\"structural_binding\":" << (binder.any_structural() ? "true" : "false") << ",\"numerics\":\""
     << (M->exact ? "exact" : "fp16") << "\"}";
  M->describe_json = js.str();
  CUDA_CHECK(cudaStreamSynchronize(M->stream));
  return M.release();
}

int bert_hidden(const sbv2_model* m) { return static_cast<const BertModel*>(m)->hidden; }

// Forward pass; the features [batch, S, H] (zero rows where the mask is 0) stay on the device in M.outd.  Returns null
// when no token is valid.  The caller owns the synchronisation with M.stream.
const float* bert_forward_device(sbv2_model* mm, const int64_t* ids, const int64_t* mask, int batch, int64_t S) {
  auto* Mp = static_cast<BertModel*>(mm);
  BertModel& M = *Mp;
  SBV2_REQUIRE(batch > 0 && S > 0, "empty input");
  SBV2_REQUIRE(S <= kMaxBertTokens, "sequence longer than 32768 tokens");
  M.bind_device();
  const int H = M.hidden;
  // right-padded masks only: 1..1 0..0
  std::vector<int> len(batch), start(batch);
  int64_t n = 0;
  int max_len = 0;
  for (int b = 0; b < batch; ++b) {
    int l = 0;
    while (l < S && mask[b * S + l] != 0) ++l;
    for (int64_t t = l; t < S; ++t)
      if (mask[b * S + t] != 0) fail(SBV2_ERR_UNSUPPORTED, "attention_mask must be a prefix of ones (right padding)");
    len[b] = l;
    SBV2_REQUIRE(n + l <= INT_MAX, "too many tokens in one call");  // packed rows are indexed in int32
    start[b] = int(n);
    n += l;
    max_len = std::max(max_len, l);
  }
  const size_t out_elems = size_t(batch) * S * H;
  if (n == 0) return nullptr;
  LaunchCtx ctx = M.ctx();
  // ids of the valid tokens, packed
  CUDA_CHECK(cudaStreamSynchronize(M.stream));  // the previous call's copies out of / into the staging buffer are done
  M.pin_io.ensure(std::max(size_t(n) * 4, out_elems * 4));
  int* hid = M.pin_io.as<int>();
  for (int b = 0; b < batch; ++b)
    for (int t = 0; t < len[b]; ++t) {
      int64_t id = ids[b * S + t];
      SBV2_REQUIRE(id >= 0 && id < M.vocab, "token id out of range");
      hid[start[b] + t] = int(id);
    }
  M.ids.ensure(size_t(n) * 4);
  CUDA_CHECK(cudaMemcpyAsync(M.ids.p, hid, size_t(n) * 4, cudaMemcpyHostToDevice, M.stream));
  std::vector<int> muls(1, 1);
  // utterances with zero tokens still need a segment: build_geoms handles len 0
  BatchGeom bg = build_geoms(&M, M.meta, M.pin_meta, start, len, muls);
  const Geom& G = bg.g[0];
  PlanarSegs ps;
  ps.start = bg.d_ystart;
  ps.pstart = G.d_pstart;
  ps.len = G.d_len;
  ps.n = batch;
  ps.max_len = max_len;
  ps.plane_stride = G.rows_tot * 8;
  const size_t R = size_t(G.rows_tot);
  M.out_len = G.d_len;
  M.out_batch = batch;
  M.out_S = S;
  M.h.ensure(size_t(n) * H * 4);
  M.region_begin("bert");
  if (M.exact) {
    // ---- exact mode: fp32 row-major activations, two-term fp16 operand splits for every GEMM -------------------------
    M.x_emb.ensure(size_t(n) * H * 4);
    M.x_qkv.ensure(size_t(n) * 3 * H * 4);
    M.x_y.ensure(size_t(n) * H * 4);
    // split-planar operands [h0 | h1 | h0]: written by the kernel that produces the values (LayerNorm, attention, the FFN's
    // first GEMM), never by a separate pass.  sp_e: embeddings (layer 0 and the ConvLayer read it), sp_a: the residual
    // stream after a LayerNorm, sp_b: attention context, sp_c: gelu(intermediate).
    M.x_split.ensure(R * 3 * size_t(H) * 2 * 3 + R * 3 * size_t(M.inter) * 2);
    M.outd.ensure(out_elems * 4);
    float* h = M.h.as<float>();
    float* emb = M.x_emb.as<float>();
    float* qkv = M.x_qkv.as<float>();
    float* y = M.x_y.as<float>();
    __half* sp_e = M.x_split.as<__half>();
    __half* sp_a = sp_e + R * 3 * size_t(H);
    __half* sp_b = sp_a + R * 3 * size_t(H);
    __half* sp_c = sp_b + R * 3 * size_t(H);
    const float sc = M.layers[0].qkv.in_scale;  // the same for every split layer
    if (M.has_conv) launch_zero_gaps(ctx, sp_e, 3 * H, G, batch);  // k = 3 ConvLayer halo; the GEMMs have none
    // attention on the tensor cores with split operands (one tile up to 128 tokens, tile pairs beyond;
    // SBV2_B200_BERT_ATTN=simt: fp32 CUDA-core kernel); q|k|v then leave their GEMM as split planes instead of fp32 rows
    const bool tc_single = deberta_attention_tc_supported(64, M.span, max_len);
    const bool tc_exact = M.use_tc_attn && M.hidden / M.heads == 64 && sc == kSplitScale && (tc_single || deberta_attention_tc_multi_supported(64));
    __half* sp_qkv = nullptr;
    const long long qkv_blk = (long long)(3 * H / 8) * ps.plane_stride, ctx_blk = (long long)(H / 8) * ps.plane_stride;
    if (tc_exact) {
      M.x_qkvs.ensure(R * 9 * size_t(H) * 2);
      if (M.x_qkvs.gen != M.x_qkvs_cleared_gen) {
        // rows past an utterance's end are read as operands: they must hold finite values
        CUDA_CHECK(cudaMemsetAsync(M.x_qkvs.p, 0, M.x_qkvs.cap, M.stream));
        M.x_qkvs_cleared_gen = M.x_qkvs.gen;
      }
      sp_qkv = M.x_qkvs.as<__half>();
    }
    auto gemm = [&](const ConvLayer& L, const __half* in, float* out, int cout, __half* out_split, int act) {
      ConvCall c;
      c.in = in;
      c.rm_out = out;
      c.rm_ld = cout;
      c.rm_start = bg.d_ystart;
      c.split_out = out_split;
      c.split_scale = sc;
      c.act_out = act;
      c.tmap = true;
      c.splitk = true;
      c.cluster = 2;  // multicast weight stages in batches (launch_umma); split-K takes over for few tokens
      launch_umma(ctx, L, G, G, c, batch);
    };
    launch_embed_rows(ctx, h, M.word_emb, M.ids.as<int>(), H, M.vocab, n);
    launch_ln_split(ctx, emb, sp_e, sc, h, nullptr, M.emb_g, M.emb_b, M.eps, H, ps);
    const bool small = n <= kSmallTokens;
    for (int l = 0; l < M.n_run; ++l) {
      const BertLayer& B = M.layers[l];
      const float* in = l == 0 ? emb : h;
      if (tc_exact) {
        gemm(small ? B.qkv_s : B.qkv, l == 0 ? sp_e : sp_a, nullptr, 3 * H, sp_qkv, ACT_NONE);
        if (tc_single)
          launch_deberta_attention_tc_exact(ctx, sp_b, ctx_blk, sp_qkv, qkv_blk, B.pos_k_s, B.pos_q_s, 2 * M.span, M.span, M.heads, sc, ps);
        else
          launch_deberta_attention_tc_exact_multi(ctx, sp_b, ctx_blk, sp_qkv, qkv_blk, B.pos_k_s, B.pos_q_s, 2 * M.span, M.bucket_idx, M.max_rel,
                                                  M.heads, sc, true, ps);
      } else {
        gemm(small ? B.qkv_s : B.qkv, l == 0 ? sp_e : sp_a, qkv, 3 * H, nullptr, ACT_NONE);
        launch_deberta_attention_f32(ctx, nullptr, sp_b, sc, qkv, B.pos_k, B.pos_q, 2 * M.span, M.bucket_idx, M.max_rel, M.heads, 64, ps);
      }
      gemm(small ? B.o_s : B.o, sp_b, y, H, nullptr, ACT_NONE);
      launch_ln_split(ctx, h, sp_a, sc, in, y, B.ln1_g, B.ln1_b, M.eps, H, ps);
      gemm(small ? B.f1_s : B.f1, sp_a, nullptr, M.inter, sp_c, ACT_GELU);
      gemm(small ? B.f2_s : B.f2, sp_c, y, H, nullptr, ACT_NONE);
      launch_ln_split(ctx, h, sp_a, sc, h, y, B.ln2_g, B.ln2_b, M.eps, H, ps);
      if (l == 0 && M.has_conv) {
        // ConvLayer: LN(layer0_out + gelu(conv(embeddings)))
        gemm(small ? M.conv_s : M.conv, sp_e, y, H, nullptr, ACT_GELU);
        launch_ln_split(ctx, h, sp_a, sc, h, y, M.conv_g, M.conv_b, M.eps, H, ps);
      }
    }
    launch_scatter_rows(ctx, M.outd.as<float>(), h, H, int(S), ps);
    M.region_end("bert");
    M.debug["bert_h"] = DebugView{h, n, H, 4};
    return M.outd.as<float>();
  }
  M.embp.ensure(R * H * 2);
  M.hp.ensure(R * H * 2);
  M.qkvp.ensure(R * 3 * H * 2);
  M.ctxp.ensure(R * H * 2);
  M.f1p.ensure(R * M.inter * 2);
  M.y32.ensure(R * H * 4);
  M.outd.ensure(out_elems * 4);
  float* h = M.h.as<float>();
  __half* embp = M.embp.as<__half>();
  __half* hp = M.hp.as<__half>();
  __half* qkvp = M.qkvp.as<__half>();
  __half* ctxp = M.ctxp.as<__half>();
  __half* f1p = M.f1p.as<__half>();
  float* y32 = M.y32.as<float>();
  if (M.has_conv) launch_zero_gaps(ctx, embp, H, G, batch);
  launch_embed_rows(ctx, h, M.word_emb, M.ids.as<int>(), H, M.vocab, n);
  launch_ln_planar_wide(ctx, h, embp, nullptr, nullptr, M.emb_g, M.emb_b, M.eps, H, ps);
  auto umma = [&](const ConvLayer& L, const __half* in, __half* o, float* acc32, int act) {
    ConvCall c;
    c.in = in;
    c.out = o;
    c.accum = acc32;
    c.accum_mode = acc32 ? UACC_SET : UACC_NONE;
    c.act_out = act;
    c.act_on_accum = acc32 != nullptr && act != ACT_NONE;
    c.tmap = true;
    c.splitk = true;
    c.cluster = 2;  // multicast weight stages in batches (launch_umma); split-K takes over for few tokens
    launch_umma(ctx, L, G, G, c, batch);
  };
  // sequences of at most 128 tokens: disentangled attention on the tensor cores (SBV2_B200_BERT_ATTN=simt: CUDA cores)
  const bool tc_attn = M.use_tc_attn && M.hidden / M.heads == 64 && deberta_attention_tc_supported(64, M.span, max_len);
  // longer sequences: the multi-tile kernel (log-bucket position windows gathered per tile pair)
  const bool tc_multi = !tc_attn && M.use_tc_attn && M.hidden / M.heads == 64 && deberta_attention_tc_multi_supported(64);
  if ((tc_attn || tc_multi) && M.qkvp.gen != M.qkvp_cleared_gen) {
    // rows past an utterance's end are read by the tensor-core attention: they must hold finite values
    CUDA_CHECK(cudaMemsetAsync(M.qkvp.p, 0, M.qkvp.cap, M.stream));
    M.qkvp_cleared_gen = M.qkvp.gen;
  }
  const bool small = n <= kSmallTokens;
  for (int l = 0; l < M.n_run; ++l) {
    const BertLayer& B = M.layers[l];
    const __half* in = l == 0 ? embp : hp;
    umma(small ? B.qkv_s : B.qkv, in, qkvp, nullptr, ACT_NONE);
    if (tc_attn) launch_deberta_attention_tc(ctx, ctxp, qkvp, B.pos_k_p, B.pos_q_p, 2 * M.span, M.span, M.heads, ps);
    else if (tc_multi) launch_deberta_attention_tc_multi(ctx, ctxp, qkvp, B.pos_k_p, B.pos_q_p, 2 * M.span, M.bucket_idx, M.max_rel, M.heads, true, ps);
    else launch_deberta_attention(ctx, ctxp, qkvp, B.pos_k, B.pos_q, 2 * M.span, M.bucket_idx, M.max_rel, M.heads, 64, ps);
    umma(small ? B.o_s : B.o, ctxp, nullptr, y32, ACT_NONE);
    launch_ln_planar_wide(ctx, h, hp, nullptr, y32, B.ln1_g, B.ln1_b, M.eps, H, ps);
    umma(small ? B.f1_s : B.f1, hp, f1p, nullptr, ACT_GELU);
    umma(small ? B.f2_s : B.f2, f1p, nullptr, y32, ACT_NONE);
    launch_ln_planar_wide(ctx, h, hp, nullptr, y32, B.ln2_g, B.ln2_b, M.eps, H, ps);
    if (l == 0 && M.has_conv) {
      // ConvLayer: LN(layer0_out + gelu(conv(embeddings)))
      umma(small ? M.conv_s : M.conv, embp, nullptr, y32, ACT_GELU);
      launch_ln_planar_wide(ctx, h, hp, nullptr, y32, M.conv_g, M.conv_b, M.eps, H, ps);
    }
  }
  launch_scatter_rows(ctx, M.outd.as<float>(), h, H, int(S), ps);
  M.region_end("bert");
  M.debug["bert_h"] = DebugView{h, n, H, 4};
  return M.outd.as<float>();
}

const float* bert_token_mean(sbv2_model* mm, int row0, int n) {
  auto& M = *static_cast<BertModel*>(mm);
  M.bind_device();
  SBV2_REQUIRE(M.out_len && row0 >= 0 && n > 0 && row0 + n <= M.out_batch, "token mean over rows the last forward did not produce");
  M.meand.ensure(size_t(n) * M.hidden * 4);
  launch_token_mean(M.ctx(), M.meand.as<float>(), M.outd.as<float>(), M.out_len, row0, n, int(M.out_S), M.hidden);
  return M.meand.as<float>();
}

void bert_predict(sbv2_model* mm, const int64_t* ids, const int64_t* mask, int batch, int64_t S, float* out) {
  auto& M = *static_cast<BertModel*>(mm);
  const size_t out_elems = size_t(batch) * S * M.hidden;
  const float* d = bert_forward_device(mm, ids, mask, batch, S);
  if (!d) {
    memset(out, 0, out_elems * 4);
    return;
  }
  float* ho = M.pin_io.as<float>();
  CUDA_CHECK(cudaMemcpyAsync(ho, d, out_elems * 4, cudaMemcpyDeviceToHost, M.stream));
  CUDA_CHECK(cudaStreamSynchronize(M.stream));
  memcpy(out, ho, out_elems * 4);
}

}  // namespace sbv2
