// extern "C" boundary (include/sbv2_b200.h). Everything is wrapped in sbv2::guarded so no
// exception or abort crosses the ABI.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>

#include "container.h"
#include "model.h"
#include "onnx_bind.h"

namespace sbv2 {
const char* last_error_cstr();
}

using namespace sbv2;

namespace {

// One implementation of the token path: sbv2_synthesize_from_tokens_assist (and through it _batch) and
// sbv2_synthesize_from_tokens_with_durations synthesize, sbv2_predict_durations_from_tokens (query = true) stops after
// the durations kernel and writes them to out_durations.
void tokens_call(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch, const sbv2_assist_text* assists,
                 int n_assists, const int32_t* assist_of, const int64_t* pause_after, const int32_t* const* durations, bool query,
                 int32_t* out_durations, float** out_samples, int64_t* out_total, int64_t* out_n_samples) {
  SBV2_REQUIRE(synth && bert && utts && (query ? out_durations != nullptr : out_samples && out_total), "null argument");
  SBV2_REQUIRE(!synth->is_bert, "synthesize called on a BERT model");
  SBV2_REQUIRE(bert->is_bert, "bert_predict called on a synthesizer model");
  SBV2_REQUIRE(synth->device == bert->device, "the BERT and synthesizer models must live on the same device");
  SBV2_REQUIRE(batch > 0, "empty batch");
  SBV2_REQUIRE(n_assists >= 0 && (assists || n_assists == 0), "null assists with n_assists > 0");
  if (!query) {
    *out_samples = nullptr;
    *out_total = 0;
  }
  for (int a = 0; a < n_assists; ++a) {
    const sbv2_assist_text& x = assists[a];
    SBV2_REQUIRE(x.input_ids && x.attention_mask, "null assist-text input");
    SBV2_REQUIRE(x.t_tok > 0 && x.t_tok <= kMaxBertTokens, "assist text must have 1 .. 32768 tokens");
    SBV2_REQUIRE(std::isfinite(x.weight), "assist_text_weight must be finite");
    for (int64_t t = 0; t < x.t_tok; ++t)
      SBV2_REQUIRE(x.attention_mask[t] != 0, "attention_mask of an assist text must be all ones (padding is added by the library)");
  }
  // DeBERTa batch: [sentences..., used assists...] right-padded to the longest row.  An assist is used when some
  // sentence names it with a non-zero weight; used assists follow in index order and take slots 0, 1, ...
  std::vector<char> named(size_t(n_assists), 0);
  for (int i = 0; i < batch; ++i) {
    const int a = assist_of ? assist_of[i] : -1;
    SBV2_REQUIRE(a >= -1 && a < n_assists, "assist_of entry out of range");
    if (a >= 0 && assists[a].weight != 0.f) named[size_t(a)] = 1;
  }
  std::vector<int> slot_of(size_t(n_assists), -1), used;
  for (int a = 0; a < n_assists; ++a)
    if (named[size_t(a)]) {
      slot_of[size_t(a)] = int(used.size());
      used.push_back(a);
    }
  const int rows_b = batch + int(used.size());
  int64_t s_max = 0, nx = 0;
  for (int i = 0; i < batch; ++i) {
    SBV2_REQUIRE(utts[i].input_ids && utts[i].attention_mask && utts[i].word2ph && utts[i].t_tok > 0 && utts[i].t_x > 0, "empty input");
    s_max = std::max(s_max, utts[i].t_tok);
    nx += utts[i].t_x;
  }
  for (int a : used) s_max = std::max(s_max, assists[a].t_tok);
  std::vector<int64_t> ids(size_t(rows_b) * s_max, 0), mask(size_t(rows_b) * s_max, 0), ph2tok;
  std::vector<int32_t> ph_slot;
  ph2tok.reserve(size_t(nx));
  if (!used.empty()) ph_slot.reserve(size_t(nx));
  for (int i = 0; i < batch; ++i) {
    const sbv2_token_utterance& u = utts[i];
    const int32_t slot = assist_of && assist_of[i] >= 0 ? slot_of[size_t(assist_of[i])] : -1;
    int64_t n_ph = 0;
    for (int64_t t = 0; t < u.t_tok; ++t) {
      SBV2_REQUIRE(u.attention_mask[t] != 0, "attention_mask of a sentence must be all ones (padding is added by the library)");
      ids[size_t(i) * s_max + t] = u.input_ids[t];
      mask[size_t(i) * s_max + t] = 1;
      SBV2_REQUIRE(u.word2ph[t] >= 0, "negative word2ph entry");
      // tts_util.rs:129-154: token t is repeated word2ph[t] times
      for (int32_t j = 0; j < u.word2ph[t]; ++j) ph2tok.push_back(int64_t(i) * s_max + t);
      n_ph += u.word2ph[t];
    }
    SBV2_REQUIRE(n_ph == u.t_x, "sum(word2ph) must equal the number of phonemes");
    if (!used.empty()) ph_slot.insert(ph_slot.end(), size_t(n_ph), slot);
  }
  std::vector<float> coef(used.size() * 2);
  for (size_t k = 0; k < used.size(); ++k) {
    const sbv2_assist_text& x = assists[used[k]];
    for (int64_t t = 0; t < x.t_tok; ++t) {
      ids[(size_t(batch) + k) * s_max + t] = x.input_ids[t];
      mask[(size_t(batch) + k) * s_max + t] = 1;
    }
    coef[2 * k] = float(1.0 - double(x.weight));
    coef[2 * k + 1] = x.weight;
  }
  std::vector<sbv2_utterance> su;
  su.resize(size_t(batch));
  for (int i = 0; i < batch; ++i) {
    const sbv2_token_utterance& u = utts[i];
    sbv2_utterance& o = su[size_t(i)];
    o = sbv2_utterance{};
    o.x_tst = u.x_tst;
    o.tones = u.tones;
    o.lang_ids = u.lang_ids;
    o.t_x = u.t_x;
    o.sid = u.sid;
    o.style_vec = u.style_vec;
    o.sdp_ratio = u.sdp_ratio;
    o.length_scale = u.length_scale;
    o.noise_scale = u.noise_scale;
    o.noise_scale_w = u.noise_scale_w;
  }
  synth_check_durations(synth, su.data(), batch, durations);  // before DeBERTa launches anything
  const float* rows = bert_forward_device(bert, ids.data(), mask.data(), rows_b, s_max);
  SBV2_REQUIRE(rows != nullptr, "attention_mask selects no token");
  DeviceBert dev;
  if (!used.empty()) {
    dev.n_slots = int(used.size());
    dev.means = bert_token_mean(bert, batch, int(used.size()));
    dev.slot = ph_slot.data();
    dev.coef = coef.data();
  }
  cudaEvent_t ready = nullptr;
  CUDA_CHECK(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
  struct EventGuard {
    cudaEvent_t e;
    ~EventGuard() { cudaEventDestroy(e); }
  } guard{ready};
  CUDA_CHECK(cudaEventRecord(ready, bert->stream));
  dev.rows = rows;
  dev.n_rows = int64_t(rows_b) * s_max;
  dev.hidden = bert_hidden(bert);
  dev.ph2tok = ph2tok.data();
  dev.ready = ready;
  // given durations change nothing above: the DeBERTa batch and the gathered features are those of the plain call
  std::unique_ptr<sbv2_device_batch, void (*)(sbv2_device_batch*)> b(synth_upload(synth, su.data(), batch, &dev, durations),
                                                                     synth_batch_free);
  if (query) {
    synth_set_query(b.get());
    synth_run(synth, b.get());
    synth_query_durations(synth, b.get(), out_durations);  // synchronises: the BERT rows are free again
    return;
  }
  if (pause_after) synth_set_pauses(b.get(), pause_after);
  synth_run(synth, b.get());
  std::vector<int64_t> n(size_t(batch), 0);
  int32_t* dur = nullptr;
  synth_download(synth, b.get(), out_samples, n.data(), out_durations ? &dur : nullptr, nullptr);  // synchronises: the BERT rows are free again
  if (dur) {
    memcpy(out_durations, dur, size_t(synth_batch_phonemes(b.get())) * 4);
    free_out(dur);
  }
  *out_total = synth_wave_total(b.get());
  if (out_n_samples) memcpy(out_n_samples, n.data(), size_t(batch) * 8);
}

}  // namespace

extern "C" {

const char* sbv2_last_error(void) { return last_error_cstr(); }

void sbv2_free(void* p) { free_out(p); }

void* sbv2_alloc(size_t bytes) {
  void* p = nullptr;
  guarded([&] { p = alloc_out(bytes, false); });
  return p;
}

void* sbv2_alloc_pinned(size_t bytes) {
  void* p = nullptr;
  guarded([&] { p = alloc_out(bytes, true); });
  return p;
}

void sbv2_set_last_error(const char* message) { set_last_error(message ? message : ""); }

const char* sbv2_version(void) { return "sbv2_b200 0.1.0 sm_100a"; }

int sbv2_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_last_error(std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    return 0;
  }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
  }
  if (!ok) set_last_error("no sm_100 (Blackwell) device visible; this backend has no CPU fallback");
  return ok;
}

// CPU-only diagnostic: how the canonical (PyTorch) weight names of an exported graph bind to its initializers.
int sbv2_onnx_bind_report(const void* onnx_bytes, size_t n_bytes, int is_bert, char** json) {
  return guarded([&] {
    SBV2_REQUIRE(onnx_bytes && n_bytes > 0 && json, "null argument");
    (void)is_bert;
    OnnxModel m = parse_onnx(static_cast<const uint8_t*>(onnx_bytes), n_bytes);
    WeightBinder binder(m);
    const std::string s = binder.report_json();
    char* p = static_cast<char*>(alloc_out(s.size() + 1, false));
    memcpy(p, s.c_str(), s.size() + 1);
    *json = p;
  });
}

int sbv2_model_create(const void* onnx_bytes, size_t n_bytes, int is_bert, int device_ordinal, sbv2_model** out_model) {
  return guarded([&] {
    SBV2_REQUIRE(out_model, "out_model is null");
    *out_model = nullptr;
    SBV2_REQUIRE(onnx_bytes && n_bytes > 0, "empty model bytes");
    OnnxModel m = parse_onnx(static_cast<const uint8_t*>(onnx_bytes), n_bytes);
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
      cudaGetLastError();
      fail(SBV2_ERR_CUDA, "no CUDA device available (this backend has no CPU fallback)");
    }
    if (device_ordinal < 0 || device_ordinal >= n) fail(SBV2_ERR_INVALID_ARGUMENT, "device ordinal out of range");
    cudaDeviceProp prop;
    CUDA_CHECK(cudaGetDeviceProperties(&prop, device_ordinal));
    if (prop.major != 10)
      fail(SBV2_ERR_CUDA, std::string("device ") + prop.name + " is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                              "; this library contains sm_100a code only");
    *out_model = is_bert ? create_bert_model(m, device_ordinal) : create_synth_model(m, device_ordinal);
  });
}

void sbv2_model_destroy(sbv2_model* model) {
  if (!model) return;
  guarded([&] { delete model; });
}

int sbv2_model_metadata(const sbv2_model* model, const char* key, const char** value, size_t* n) {
  return guarded([&] {
    SBV2_REQUIRE(model && key && value && n, "null argument");
    auto it = model->metadata.find(key);
    if (it == model->metadata.end()) {
      *value = nullptr;
      *n = 0;
    } else {
      *value = it->second.data();
      *n = it->second.size();
    }
  });
}

int sbv2_model_describe(const sbv2_model* model, const char** json) {
  return guarded([&] {
    SBV2_REQUIRE(model && json, "null argument");
    *json = model->describe_json.c_str();
  });
}

int sbv2_bert_predict(sbv2_model* bert, const int64_t* input_ids, const int64_t* attention_mask, int64_t t_tok, float* out) {
  return guarded([&] {
    SBV2_REQUIRE(bert && input_ids && attention_mask && out, "null argument");
    SBV2_REQUIRE(bert->is_bert, "bert_predict called on a synthesizer model");
    bert_predict(bert, input_ids, attention_mask, 1, t_tok, out);
  });
}

int sbv2_bert_predict_batch(sbv2_model* bert, const int64_t* input_ids, const int64_t* attention_mask, int batch, int64_t s,
                            float* out) {
  return guarded([&] {
    SBV2_REQUIRE(bert && input_ids && attention_mask && out, "null argument");
    SBV2_REQUIRE(bert->is_bert, "bert_predict called on a synthesizer model");
    bert_predict(bert, input_ids, attention_mask, batch, s, out);
  });
}

int sbv2_bert_hidden_size(const sbv2_model* bert, int* hidden) {
  return guarded([&] {
    SBV2_REQUIRE(bert && hidden && bert->is_bert, "not a BERT model");
    *hidden = bert_hidden(bert);
  });
}

int sbv2_model_seed(sbv2_model* synth, uint64_t seed) {
  return guarded([&] {
    SBV2_REQUIRE(synth && !synth->is_bert, "not a synthesizer model");
    synth_set_seed(synth, seed);
  });
}

int sbv2_synthesize_batch(sbv2_model* synth, const sbv2_utterance* utts, int batch, float** out_samples, int64_t* out_n_samples,
                          int32_t** out_durations, int32_t** out_frame2ph) {
  return sbv2_synthesize_batch_with_durations(synth, utts, batch, nullptr, out_samples, out_n_samples, out_durations, out_frame2ph);
}

int sbv2_synthesize_batch_with_durations(sbv2_model* synth, const sbv2_utterance* utts, int batch, const int32_t* const* durations,
                                         float** out_samples, int64_t* out_n_samples, int32_t** out_durations, int32_t** out_frame2ph) {
  return guarded([&] {
    SBV2_REQUIRE(synth && out_samples && out_n_samples, "null argument");
    SBV2_REQUIRE(!synth->is_bert, "synthesize called on a BERT model");
    *out_samples = nullptr;
    if (out_durations) *out_durations = nullptr;
    if (out_frame2ph) *out_frame2ph = nullptr;
    std::unique_ptr<sbv2_device_batch, void (*)(sbv2_device_batch*)> b(synth_upload(synth, utts, batch, nullptr, durations),
                                                                       synth_batch_free);
    synth_run(synth, b.get());
    synth_download(synth, b.get(), out_samples, out_n_samples, out_durations, out_frame2ph);
  });
}

int sbv2_predict_durations_batch(sbv2_model* synth, const sbv2_utterance* utts, int batch, int32_t* out_durations) {
  return guarded([&] {
    SBV2_REQUIRE(synth && out_durations, "null argument");
    SBV2_REQUIRE(!synth->is_bert, "synthesize called on a BERT model");
    std::unique_ptr<sbv2_device_batch, void (*)(sbv2_device_batch*)> b(synth_upload(synth, utts, batch), synth_batch_free);
    synth_set_query(b.get());
    synth_run(synth, b.get());
    synth_query_durations(synth, b.get(), out_durations);
  });
}

int sbv2_synthesize_with_noise(sbv2_model* synth, const float* bert, const int64_t* x_tst, const int64_t* tones,
                               const int64_t* lang_ids, int64_t t_x, int64_t sid, const float* style_vec, float sdp_ratio,
                               float length_scale, float noise_scale, float noise_scale_w, const float* noise_sdp,
                               const float* noise_zp, int64_t noise_zp_frames, float** out_samples, int64_t* n_samples,
                               int32_t* out_durations, int32_t** out_frame2ph, int64_t* t_y) {
  return guarded([&] {
    SBV2_REQUIRE(synth && out_samples && n_samples, "null argument");
    SBV2_REQUIRE(!synth->is_bert, "synthesize called on a BERT model");
    *out_samples = nullptr;
    if (out_frame2ph) *out_frame2ph = nullptr;
    sbv2_utterance u{};
    u.bert = bert;
    u.x_tst = x_tst;
    u.tones = tones;
    u.lang_ids = lang_ids;
    u.t_x = t_x;
    u.sid = sid;
    u.style_vec = style_vec;
    u.sdp_ratio = sdp_ratio;
    u.length_scale = length_scale;
    u.noise_scale = noise_scale;
    u.noise_scale_w = noise_scale_w;
    u.noise_sdp = noise_sdp;
    u.noise_zp = noise_zp;
    u.noise_zp_frames = noise_zp_frames;
    std::unique_ptr<sbv2_device_batch, void (*)(sbv2_device_batch*)> b(synth_upload(synth, &u, 1), synth_batch_free);
    synth_run(synth, b.get());
    int32_t* dur = nullptr;
    synth_download(synth, b.get(), out_samples, n_samples, out_durations ? &dur : nullptr, out_frame2ph);
    if (out_durations && dur) {
      memcpy(out_durations, dur, size_t(t_x) * 4);
      free_out(dur);
    }
    if (t_y) synth_batch_ty(b.get(), t_y);
  });
}

int sbv2_synthesize_from_tokens(sbv2_model* synth, sbv2_model* bert, const int64_t* input_ids, const int64_t* attention_mask,
                                int64_t t_tok, const int32_t* word2ph, const int64_t* x_tst, const int64_t* tones, const int64_t* lang_ids,
                                int64_t t_x, int64_t sid, const float* style_vec, float sdp_ratio, float length_scale,
                                float noise_scale, float noise_scale_w, float** out_samples, int64_t* n_samples) {
  return guarded([&] {
    SBV2_REQUIRE(synth && bert && input_ids && attention_mask && word2ph && out_samples && n_samples, "null argument");
    SBV2_REQUIRE(!synth->is_bert, "synthesize called on a BERT model");
    SBV2_REQUIRE(bert->is_bert, "bert_predict called on a synthesizer model");
    SBV2_REQUIRE(synth->device == bert->device, "the BERT and synthesizer models must live on the same device");
    SBV2_REQUIRE(t_tok > 0 && t_x > 0, "empty input");
    *out_samples = nullptr;
    // phoneme -> token row (tts_util.rs:129-154: token i is repeated word2ph[i] times)
    std::vector<int64_t> ph2tok;
    ph2tok.reserve(size_t(t_x));
    for (int64_t i = 0; i < t_tok; ++i) {
      SBV2_REQUIRE(word2ph[i] >= 0, "negative word2ph entry");
      for (int32_t j = 0; j < word2ph[i]; ++j) ph2tok.push_back(i);
    }
    SBV2_REQUIRE(int64_t(ph2tok.size()) == t_x, "sum(word2ph) must equal the number of phonemes");
    const float* rows = bert_forward_device(bert, input_ids, attention_mask, 1, t_tok);
    SBV2_REQUIRE(rows != nullptr, "attention_mask selects no token");
    cudaEvent_t ready = nullptr;
    CUDA_CHECK(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    struct EventGuard {
      cudaEvent_t e;
      ~EventGuard() { cudaEventDestroy(e); }
    } guard{ready};
    CUDA_CHECK(cudaEventRecord(ready, bert->stream));
    DeviceBert dev;
    dev.rows = rows;
    dev.n_rows = t_tok;
    dev.hidden = bert_hidden(bert);
    dev.ph2tok = ph2tok.data();
    dev.ready = ready;
    sbv2_utterance u{};
    u.x_tst = x_tst;
    u.tones = tones;
    u.lang_ids = lang_ids;
    u.t_x = t_x;
    u.sid = sid;
    u.style_vec = style_vec;
    u.sdp_ratio = sdp_ratio;
    u.length_scale = length_scale;
    u.noise_scale = noise_scale;
    u.noise_scale_w = noise_scale_w;
    std::unique_ptr<sbv2_device_batch, void (*)(sbv2_device_batch*)> b(synth_upload(synth, &u, 1, &dev), synth_batch_free);
    synth_run(synth, b.get());
    synth_download(synth, b.get(), out_samples, n_samples, nullptr, nullptr);  // synchronises: the BERT rows are free again
  });
}

int sbv2_synthesize_from_tokens_batch(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch,
                                      const int64_t* pause_after, float** out_samples, int64_t* out_total, int64_t* out_n_samples) {
  return sbv2_synthesize_from_tokens_assist(synth, bert, utts, batch, nullptr, 0, nullptr, pause_after, out_samples, out_total,
                                            out_n_samples);
}

int sbv2_synthesize_from_tokens_assist(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch,
                                       const sbv2_assist_text* assists, int n_assists, const int32_t* assist_of,
                                       const int64_t* pause_after, float** out_samples, int64_t* out_total, int64_t* out_n_samples) {
  return sbv2_synthesize_from_tokens_with_durations(synth, bert, utts, batch, assists, n_assists, assist_of, pause_after, nullptr, nullptr,
                                                    out_samples, out_total, out_n_samples);
}

int sbv2_synthesize_from_tokens_with_durations(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch,
                                               const sbv2_assist_text* assists, int n_assists, const int32_t* assist_of,
                                               const int64_t* pause_after, const int32_t* const* durations, int32_t* out_durations,
                                               float** out_samples, int64_t* out_total, int64_t* out_n_samples) {
  return guarded([&] {
    tokens_call(synth, bert, utts, batch, assists, n_assists, assist_of, pause_after, durations, false, out_durations, out_samples,
                out_total, out_n_samples);
  });
}

int sbv2_predict_durations_from_tokens(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch,
                                       const sbv2_assist_text* assists, int n_assists, const int32_t* assist_of, int32_t* out_durations) {
  return guarded([&] {
    tokens_call(synth, bert, utts, batch, assists, n_assists, assist_of, nullptr, nullptr, true, out_durations, nullptr, nullptr, nullptr);
  });
}

int sbv2_synthesize(sbv2_model* synth, const float* bert, const int64_t* x_tst, const int64_t* tones, const int64_t* lang_ids,
                    int64_t t_x, int64_t sid, const float* style_vec, float sdp_ratio, float length_scale, float noise_scale,
                    float noise_scale_w, float** out_samples, int64_t* n_samples) {
  return sbv2_synthesize_with_noise(synth, bert, x_tst, tones, lang_ids, t_x, sid, style_vec, sdp_ratio, length_scale, noise_scale,
                                    noise_scale_w, nullptr, nullptr, 0, out_samples, n_samples, nullptr, nullptr, nullptr);
}

int sbv2_batch_upload(sbv2_model* synth, const sbv2_utterance* utts, int batch, sbv2_device_batch** out) {
  return guarded([&] {
    SBV2_REQUIRE(synth && out, "null argument");
    *out = synth_upload(synth, utts, batch);
    // inputs are borrowed for the duration of the call: copies that read the caller's buffers in place must be done
    if (synth_borrows_host(*out)) CUDA_CHECK(cudaStreamSynchronize(synth->stream));
  });
}

int sbv2_batch_run(sbv2_model* synth, sbv2_device_batch* b, int64_t* total_samples) {
  return guarded([&] {
    SBV2_REQUIRE(synth && b, "null argument");
    synth_run(synth, b);
    if (total_samples) *total_samples = synth_total_samples(synth, b);
  });
}

int sbv2_batch_download(sbv2_model* synth, sbv2_device_batch* b, float** out_samples, int64_t* out_n_samples) {
  return guarded([&] {
    SBV2_REQUIRE(synth && b && out_samples, "null argument");
    synth_download(synth, b, out_samples, out_n_samples, nullptr, nullptr);
  });
}

void sbv2_batch_free(sbv2_device_batch* b) {
  if (b) guarded([&] { synth_batch_free(b); });
}

int64_t sbv2_model_launch_count(const sbv2_model* model) { return model ? model->launches : 0; }

void* sbv2_model_stream(const sbv2_model* model) { return model ? static_cast<void*>(model->stream) : nullptr; }

int sbv2_decode_batch(sbv2_model* synth, const float* const* z, const int64_t* t_y, const int64_t* sid, int batch,
                      float** out_samples, int64_t* out_n_samples) {
  return guarded([&] {
    SBV2_REQUIRE(synth && out_samples && out_n_samples, "null argument");
    *out_samples = nullptr;
    synth_decode(synth, z, t_y, sid, batch, out_samples, out_n_samples);
  });
}

int sbv2_model_enable_timing(sbv2_model* model, int on) {
  return guarded([&] {
    SBV2_REQUIRE(model, "null argument");
    model->timing = on != 0;
  });
}

int sbv2_model_region_ms(sbv2_model* model, const char* region, float* ms) {
  return guarded([&] {
    SBV2_REQUIRE(model && region && ms, "null argument");
    model->bind_device();
    *ms = model->region_ms(region);
  });
}

// Test hook (not part of the reference API): copies a named intermediate of the last run.
int sbv2_debug_fetch(sbv2_model* model, const char* name, float** out, int64_t* rows, int64_t* cols) {
  return guarded([&] {
    SBV2_REQUIRE(model && name && out && rows && cols, "null argument");
    auto it = model->debug.find(name);
    if (it == model->debug.end()) fail(SBV2_ERR_INVALID_ARGUMENT, std::string("no debug view named ") + name);
    model->bind_device();
    const DebugView& v = it->second;
    size_t bytes = size_t(v.rows) * v.cols * 4;
    float* h = static_cast<float*>(alloc_out(bytes, false));
    CUDA_CHECK(cudaStreamSynchronize(model->stream));
    CUDA_CHECK(cudaMemcpy(h, v.ptr, bytes, cudaMemcpyDeviceToHost));
    *out = h;
    *rows = v.rows;
    *cols = v.cols;
  });
}

int sbv2_parse_sbv2file(const void* sbv2_bytes, size_t n, void** style_json, size_t* style_n, void** onnx, size_t* onnx_n) {
  return guarded([&] {
    SBV2_REQUIRE(sbv2_bytes && style_json && style_n && onnx && onnx_n, "null argument");
    Sbv2File f = parse_sbv2file(static_cast<const uint8_t*>(sbv2_bytes), n);
    void* s = alloc_out(f.style_n, false);
    void* o = alloc_out(f.onnx_n, false);
    memcpy(s, f.style_json, f.style_n);
    memcpy(o, f.onnx, f.onnx_n);
    *style_json = s;
    *style_n = f.style_n;
    *onnx = o;
    *onnx_n = f.onnx_n;
  });
}

int sbv2_load_style(const void* json_bytes, size_t n, float** out, int64_t* rows, int64_t* cols) {
  return guarded([&] {
    SBV2_REQUIRE(json_bytes && out && rows && cols, "null argument");
    StyleVectors s = load_style_json(static_cast<const uint8_t*>(json_bytes), n);
    float* p = static_cast<float*>(alloc_out(s.data.size() * 4, false));
    memcpy(p, s.data.data(), s.data.size() * 4);
    *out = p;
    *rows = s.rows;
    *cols = s.cols;
  });
}

int sbv2_load_style_npy_base64(const char* b64, size_t n, float** out, int64_t* rows, int64_t* cols) {
  return guarded([&] {
    SBV2_REQUIRE(b64 && out && rows && cols, "null argument");
    StyleVectors s = load_style_npy_base64(b64, n);
    float* p = static_cast<float*>(alloc_out(s.data.size() * 4, false));
    memcpy(p, s.data.data(), s.data.size() * 4);
    *out = p;
    *rows = s.rows;
    *cols = s.cols;
  });
}

int sbv2_get_style_vector(const float* style_vectors, int64_t rows, int64_t cols, int32_t style_id, float weight, float* out) {
  return guarded([&] {
    SBV2_REQUIRE(style_vectors && out, "null argument");
    StyleVectors s;
    s.rows = rows;
    s.cols = cols;
    s.data.assign(style_vectors, style_vectors + rows * cols);
    auto v = get_style_vector(s, style_id, weight);
    memcpy(out, v.data(), v.size() * 4);
  });
}

int sbv2_wav_from_f32(const float* samples, int64_t n, void** wav_bytes, size_t* wav_n) {
  return guarded([&] {
    SBV2_REQUIRE((samples || n == 0) && wav_bytes && wav_n, "null argument");
    auto w = wav_from_f32(samples, n);
    void* p = alloc_out(w.size(), false);
    memcpy(p, w.data(), w.size());
    *wav_bytes = p;
    *wav_n = w.size();
  });
}

int sbv2_wav_pcm16_from_f32(const float* samples, int64_t n, void** wav_bytes, size_t* wav_n) {
  return guarded([&] {
    SBV2_REQUIRE((samples || n == 0) && wav_bytes && wav_n, "null argument");
    auto w = wav_pcm16_from_f32(samples, n);
    void* p = alloc_out(w.size(), false);
    memcpy(p, w.data(), w.size());
    *wav_bytes = p;
    *wav_n = w.size();
  });
}

}  // extern "C"
