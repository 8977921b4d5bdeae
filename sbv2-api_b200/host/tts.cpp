#include "tts.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace sbv2 {
namespace host {
namespace {

[[noreturn]] void raise_from_status(int status) {
  std::string msg = sbv2_last_error();
  switch (status) {
    case SBV2_ERR_INVALID_ARGUMENT: throw Error(msg.rfind("NDArray", 0) == 0 ? ErrorKind::NdArrayError : ErrorKind::ValueError, msg);
    case SBV2_ERR_MODEL_NOT_FOUND: throw Error(ErrorKind::ModelNotFoundError, msg);
    case SBV2_ERR_PARSE:
      if (msg.rfind("style json", 0) == 0) throw Error(ErrorKind::SerdeJsonError, msg);
      if (msg.rfind("base64", 0) == 0) throw Error(ErrorKind::Base64Error, msg);
      if (msg.rfind(".sbv2", 0) == 0) throw Error(ErrorKind::IoError, msg);
      throw Error(ErrorKind::OrtError, msg);
    case SBV2_ERR_CUDA:
    case SBV2_ERR_UNSUPPORTED: throw Error(ErrorKind::OrtError, msg);
    default: throw Error(ErrorKind::OtherError, msg);
  }
}
inline void check(int status) {
  if (status != SBV2_OK) raise_from_status(status);
}

Array2 take_matrix(float* p, int64_t rows, int64_t cols) {
  Array2 a;
  a.rows = rows;
  a.cols = cols;
  a.data.assign(p, p + rows * cols);
  sbv2_free(p);
  return a;
}

}  // namespace

Session& Session::operator=(Session&& o) noexcept {
  if (this != &o) {
    sbv2_model_destroy(m_);
    m_ = o.m_;
    o.m_ = nullptr;
  }
  return *this;
}
Session::~Session() { sbv2_model_destroy(m_); }

std::optional<std::string> Session::metadata_custom(const std::string& key) const {
  const char* v = nullptr;
  size_t n = 0;
  check(sbv2_model_metadata(m_, key.c_str(), &v, &n));
  if (!v) return std::nullopt;
  return std::string(v, n);
}

namespace model {

Session load_model(const std::vector<uint8_t>& model_file, bool bert, int device_ordinal) {
  sbv2_model* m = nullptr;
  check(sbv2_model_create(model_file.data(), model_file.size(), bert ? 1 : 0, device_ordinal, &m));
  return Session(m);
}

std::vector<float> synthesize(Session& session, const Array2& bert_ori, const std::vector<int64_t>& x_tst,
                              const std::vector<int64_t>& spk_ids, const std::vector<int64_t>& tones,
                              const std::vector<int64_t>& lang_ids, const std::vector<float>& style_vector, float sdp_ratio,
                              float length_scale, float noise_scale, float noise_scale_w) {
  const int64_t t_x = int64_t(x_tst.size());
  if (spk_ids.size() != 1) throw Error(ErrorKind::OrtError, "sid must have exactly one element");
  if (int64_t(tones.size()) != t_x || int64_t(lang_ids.size()) != t_x || bert_ori.cols != t_x)
    throw Error(ErrorKind::OrtError, "x_tst, tones, language and bert must agree on x_tst_max_length");
  float* samples = nullptr;
  int64_t n = 0;
  check(sbv2_synthesize(session.get(), bert_ori.data.data(), x_tst.data(), tones.data(), lang_ids.data(), t_x, spk_ids[0],
                        style_vector.data(), sdp_ratio, length_scale, noise_scale, noise_scale_w, &samples, &n));
  std::vector<float> out(samples, samples + n);
  sbv2_free(samples);
  return out;
}

std::vector<float> synthesize_from_tokens(Session& session, Session& bert, const std::vector<int64_t>& token_ids,
                                          const std::vector<int64_t>& attention_masks, const std::vector<int32_t>& word2ph,
                                          const std::vector<int64_t>& x_tst, const std::vector<int64_t>& spk_ids,
                                          const std::vector<int64_t>& tones, const std::vector<int64_t>& lang_ids,
                                          const std::vector<float>& style_vector, float sdp_ratio, float length_scale,
                                          float noise_scale, float noise_scale_w) {
  const int64_t t_x = int64_t(x_tst.size());
  if (spk_ids.size() != 1) throw Error(ErrorKind::OrtError, "sid must have exactly one element");
  if (int64_t(tones.size()) != t_x || int64_t(lang_ids.size()) != t_x)
    throw Error(ErrorKind::OrtError, "x_tst, tones and language must agree on x_tst_max_length");
  if (token_ids.size() != attention_masks.size() || word2ph.size() != token_ids.size())
    throw Error(ErrorKind::OtherError, "word2ph length must equal the number of BERT rows");
  float* samples = nullptr;
  int64_t n = 0;
  check(sbv2_synthesize_from_tokens(session.get(), bert.get(), token_ids.data(), attention_masks.data(), int64_t(token_ids.size()),
                                    word2ph.data(), x_tst.data(), tones.data(), lang_ids.data(), t_x, spk_ids[0], style_vector.data(),
                                    sdp_ratio, length_scale, noise_scale, noise_scale_w, &samples, &n));
  std::vector<float> out(samples, samples + n);
  sbv2_free(samples);
  return out;
}

}  // namespace model

namespace bert {

Array2 predict(Session& session, const std::vector<int64_t>& token_ids, const std::vector<int64_t>& attention_masks) {
  if (token_ids.size() != attention_masks.size()) throw Error(ErrorKind::OrtError, "input_ids and attention_mask differ in length");
  int hidden = 0;
  check(sbv2_bert_hidden_size(session.get(), &hidden));
  Array2 out;
  out.rows = int64_t(token_ids.size());
  out.cols = hidden;
  out.data.resize(size_t(out.rows) * hidden);
  check(sbv2_bert_predict(session.get(), token_ids.data(), attention_masks.data(), out.rows, out.data.data()));
  return out;
}

}  // namespace bert

namespace tts_util {

Array2 expand_bert_features(const Array2& bert_content, const std::vector<int32_t>& word2ph) {
  if (int64_t(word2ph.size()) != bert_content.rows) throw Error(ErrorKind::OtherError, "word2ph length must equal the number of BERT rows");
  int64_t t_x = 0;
  for (int32_t r : word2ph) {
    if (r < 0) throw Error(ErrorKind::ValueError, "negative word2ph entry");
    t_x += r;
  }
  Array2 out;
  out.rows = bert_content.cols;
  out.cols = t_x;
  out.data.resize(size_t(out.rows) * t_x);
  int64_t col = 0;
  for (size_t i = 0; i < word2ph.size(); ++i)
    for (int32_t j = 0; j < word2ph[i]; ++j, ++col)
      for (int64_t c = 0; c < bert_content.cols; ++c) out.data[size_t(c) * t_x + col] = bert_content.data[i * bert_content.cols + c];
  return out;
}

std::vector<float> assist_mean(const Array2& assist_content) {
  if (assist_content.rows <= 0) throw Error(ErrorKind::ValueError, "assist text has no token");
  const int64_t H = assist_content.cols;
  std::vector<double> acc(size_t(H), 0.0);
  for (int64_t t = 0; t < assist_content.rows; ++t)
    for (int64_t c = 0; c < H; ++c) acc[size_t(c)] += double(assist_content.data[size_t(t * H + c)]);
  std::vector<float> mean(static_cast<size_t>(H));
  for (int64_t c = 0; c < H; ++c) mean[size_t(c)] = float(acc[size_t(c)] / double(assist_content.rows));
  return mean;
}

Array2 expand_bert_features(const Array2& bert_content, const std::vector<int32_t>& word2ph, const std::vector<float>& mean,
                            float weight) {
  if (int64_t(mean.size()) != bert_content.cols) throw Error(ErrorKind::ValueError, "assist mean and BERT rows differ in width");
  Array2 out = expand_bert_features(bert_content, word2ph);
  const float c_row = float(1.0 - double(weight)), c_mean = weight;
  for (int64_t c = 0; c < out.rows; ++c) {
    const float m = mean[size_t(c)] * c_mean;
    float* row = out.data.data() + size_t(c) * out.cols;
    for (int64_t j = 0; j < out.cols; ++j) row[j] = row[j] * c_row + m;
  }
  return out;
}

std::vector<uint8_t> array_to_vec(const std::vector<float>& audio) {
  void* p = nullptr;
  size_t n = 0;
  check(sbv2_wav_from_f32(audio.data(), int64_t(audio.size()), &p, &n));
  std::vector<uint8_t> out(static_cast<uint8_t*>(p), static_cast<uint8_t*>(p) + n);
  sbv2_free(p);
  return out;
}

}  // namespace tts_util

TTSModelHolder::TTSModelHolder(const std::vector<uint8_t>& bert_model_bytes, const std::vector<uint8_t>& tokenizer_bytes,
                               std::optional<size_t> max_loaded_models, int device_ordinal)
    : tokenizer_(tokenizer_bytes), bert_(model::load_model(bert_model_bytes, true, device_ordinal)),
      max_loaded_models_(max_loaded_models), device_(device_ordinal) {}

std::vector<std::string> TTSModelHolder::models() const {
  std::vector<std::string> out;
  for (auto& m : models_) out.push_back(m.ident);
  return out;
}

size_t TTSModelHolder::loaded_count() const {
  size_t n = 0;
  for (auto& m : models_) n += m.vits2.has_value() ? 1 : 0;
  return n;
}

TTSModel* TTSModelHolder::find_model(const std::string& ident) {
  for (auto& m : models_)
    if (m.ident == ident) return &m;
  return nullptr;
}

void TTSModelHolder::load_aivmx(const std::string& ident, const std::vector<uint8_t>& aivmx_bytes) {
  if (find_model(ident)) return;
  bool load = true;
  if (max_loaded_models_ && loaded_count() >= *max_loaded_models_) load = false;
  Session session = model::load_model(aivmx_bytes, false, device_);  // the reference loads even when `load` is false
  auto meta = session.metadata_custom("aivm_style_vectors");
  if (!meta) return;  // reference: silently skips the push when the metadata key is absent
  float* p = nullptr;
  int64_t rows = 0, cols = 0;
  check(sbv2_load_style_npy_base64(meta->data(), meta->size(), &p, &rows, &cols));
  TTSModel m;
  m.style_vectors = take_matrix(p, rows, cols);
  if (load) m.vits2.emplace(std::move(session));
  if (max_loaded_models_) m.bytes = aivmx_bytes;
  m.ident = ident;
  models_.push_back(std::move(m));
}

void TTSModelHolder::load_sbv2file(const std::string& ident, const std::vector<uint8_t>& sbv2_bytes) {
  void *style = nullptr, *onnx = nullptr;
  size_t style_n = 0, onnx_n = 0;
  check(sbv2_parse_sbv2file(sbv2_bytes.data(), sbv2_bytes.size(), &style, &style_n, &onnx, &onnx_n));
  std::vector<uint8_t> s(static_cast<uint8_t*>(style), static_cast<uint8_t*>(style) + style_n);
  std::vector<uint8_t> o(static_cast<uint8_t*>(onnx), static_cast<uint8_t*>(onnx) + onnx_n);
  sbv2_free(style);
  sbv2_free(onnx);
  load(ident, s, o);
}

void TTSModelHolder::load(const std::string& ident, const std::vector<uint8_t>& style_vectors_bytes, const std::vector<uint8_t>& vits2_bytes) {
  if (find_model(ident)) return;
  bool load = true;
  if (max_loaded_models_ && loaded_count() >= *max_loaded_models_) load = false;
  TTSModel m;
  if (load) m.vits2.emplace(model::load_model(vits2_bytes, false, device_));
  float* p = nullptr;
  int64_t rows = 0, cols = 0;
  check(sbv2_load_style(style_vectors_bytes.data(), style_vectors_bytes.size(), &p, &rows, &cols));
  m.style_vectors = take_matrix(p, rows, cols);
  m.ident = ident;
  if (max_loaded_models_) m.bytes = vits2_bytes;
  models_.push_back(std::move(m));
}

bool TTSModelHolder::unload(const std::string& ident) {
  for (size_t i = 0; i < models_.size(); ++i)
    if (models_[i].ident == ident) {
      models_.erase(models_.begin() + long(i));
      return true;
    }
  return false;
}

bool TTSModelHolder::find_and_load_model(const std::string& ident) {
  TTSModel* m = find_model(ident);
  if (!m) throw Error(ErrorKind::ModelNotFoundError, "model not found error: " + ident);
  if (m->vits2) return true;
  if (!m->bytes) throw Error(ErrorKind::OtherError, "model '" + ident + "' is not resident and its bytes were not retained");
  std::vector<uint8_t> bytes = *m->bytes;
  Array2 style = m->style_vectors;
  unload(ident);
  Session s = model::load_model(bytes, false, device_);
  if (max_loaded_models_ && loaded_count() >= *max_loaded_models_ && !models_.empty()) unload(models_.front().ident);
  TTSModel nm;
  nm.bytes = std::move(bytes);
  nm.vits2.emplace(std::move(s));
  nm.style_vectors = std::move(style);
  nm.ident = ident;
  models_.push_back(std::move(nm));
  return true;
}

std::vector<float> TTSModelHolder::get_style_vector(const std::string& ident, int32_t style_id, float weight) {
  TTSModel* m = find_model(ident);
  if (!m) throw Error(ErrorKind::ModelNotFoundError, "model not found error: " + ident);
  std::vector<float> out(size_t(m->style_vectors.cols));
  check(sbv2_get_style_vector(m->style_vectors.data.data(), m->style_vectors.rows, m->style_vectors.cols, style_id, weight, out.data()));
  return out;
}

namespace {
void check_assist(const AssistText& a) {
  if (!std::isfinite(a.weight)) throw Error(ErrorKind::ValueError, "assist_text_weight must be finite");
  if (a.token_ids.empty() || a.token_ids.size() > 32768 || a.attention_masks.size() != a.token_ids.size())
    throw Error(ErrorKind::ValueError, "assist text must have 1 .. 32768 tokens and a mask of the same length");
  for (int64_t m : a.attention_masks)
    if (m == 0) throw Error(ErrorKind::ValueError, "attention_mask of an assist text must be all ones");
}
}  // namespace

Array2 TTSModelHolder::bert_features(const std::vector<int64_t>& token_ids, const std::vector<int64_t>& attention_masks,
                                     const std::vector<int32_t>& word2ph, const AssistText* assist) {
  if (assist) check_assist(*assist);
  if (!assist || assist->weight == 0.0f) {
    Array2 content = bert::predict(bert_, token_ids, attention_masks);
    return tts_util::expand_bert_features(content, word2ph);
  }
  if (token_ids.size() != attention_masks.size()) throw Error(ErrorKind::OrtError, "input_ids and attention_mask differ in length");
  int hidden = 0;
  check(sbv2_bert_hidden_size(bert_.get(), &hidden));
  const size_t t = token_ids.size(), ta = assist->token_ids.size(), s = std::max(t, ta);
  std::vector<int64_t> ids(2 * s, 0), mask(2 * s, 0);
  std::copy(token_ids.begin(), token_ids.end(), ids.begin());
  std::copy(attention_masks.begin(), attention_masks.end(), mask.begin());
  std::copy(assist->token_ids.begin(), assist->token_ids.end(), ids.begin() + long(s));
  std::fill(mask.begin() + long(s), mask.begin() + long(s + ta), 1);
  std::vector<float> feat(2 * s * size_t(hidden));
  check(sbv2_bert_predict_batch(bert_.get(), ids.data(), mask.data(), 2, int64_t(s), feat.data()));
  Array2 content, assist_content;
  content.rows = int64_t(t);
  content.cols = hidden;
  content.data.assign(feat.begin(), feat.begin() + long(t * hidden));
  assist_content.rows = int64_t(ta);
  assist_content.cols = hidden;
  assist_content.data.assign(feat.begin() + long(s * hidden), feat.begin() + long((s + ta) * hidden));
  return tts_util::expand_bert_features(content, word2ph, tts_util::assist_mean(assist_content), assist->weight);
}

std::vector<uint8_t> TTSModelHolder::easy_synthesize(const std::string& ident, const std::vector<std::optional<ParsedText>>& lines,
                                                     int32_t style_id, int64_t speaker_id, const SynthesizeOptions& options) {
  find_and_load_model(ident);
  std::vector<float> style_vector = get_style_vector(ident, style_id, options.style_weight);
  std::vector<float> audio;
  auto synth_one = [&](const ParsedText& t) {
    TTSModel* m = find_model(ident);
    if (!m || !m->vits2) throw Error(ErrorKind::ModelNotFoundError, "model not found error: " + ident);
    return model::synthesize(*m->vits2, t.bert_ori, t.phones, {speaker_id}, t.tones, t.lang_ids, style_vector, options.sdp_ratio,
                             options.length_scale, 0.677f, 0.8f);
  };
  if (options.split_sentences) {
    // tts.rs:290-326 runs the lines one after the other; here the non-empty lines of a request go through the
    // synthesizer as ONE batch (SURVEY.md §8f row 2) and the 22 050-sample pauses are laid out around the results.
    TTSModel* m = find_model(ident);
    if (!m || !m->vits2) throw Error(ErrorKind::ModelNotFoundError, "model not found error: " + ident);
    std::vector<sbv2_utterance> utts;
    std::vector<size_t> line_of;
    for (size_t i = 0; i < lines.size(); ++i) {
      if (!lines[i]) continue;  // empty line
      const ParsedText& t = *lines[i];
      const int64_t t_x = int64_t(t.phones.size());
      if (int64_t(t.tones.size()) != t_x || int64_t(t.lang_ids.size()) != t_x || t.bert_ori.cols != t_x)
        throw Error(ErrorKind::OrtError, "x_tst, tones, language and bert must agree on x_tst_max_length");
      sbv2_utterance u{};
      u.bert = t.bert_ori.data.data();
      u.x_tst = t.phones.data();
      u.tones = t.tones.data();
      u.lang_ids = t.lang_ids.data();
      u.t_x = t_x;
      u.sid = speaker_id;
      u.style_vec = style_vector.data();
      u.sdp_ratio = options.sdp_ratio;
      u.length_scale = options.length_scale;
      u.noise_scale = 0.677f;
      u.noise_scale_w = 0.8f;
      utts.push_back(u);
      line_of.push_back(i);
    }
    // tts.rs:321-324: `concatenate` of an empty list is an error (a text of empty lines only)
    if (utts.empty()) throw Error(ErrorKind::NdArrayError, "NDArray error: nothing to concatenate");
    {
      float* samples = nullptr;
      std::vector<int64_t> n(utts.size(), 0);
      check(sbv2_synthesize_batch(m->vits2->get(), utts.data(), int(utts.size()), &samples, n.data(), nullptr, nullptr));
      size_t total = 0;
      for (size_t k = 0; k < utts.size(); ++k) total += size_t(n[k]) + (line_of[k] != lines.size() - 1 ? 22050 : 0);
      audio.reserve(total);
      const float* src = samples;
      for (size_t k = 0; k < utts.size(); ++k) {
        audio.insert(audio.end(), src, src + n[k]);
        src += n[k];
        if (line_of[k] != lines.size() - 1) audio.insert(audio.end(), 22050, 0.0f);
      }
      sbv2_free(samples);
    }
  } else {
    if (lines.size() != 1 || !lines[0]) throw Error(ErrorKind::ValueError, "split_sentences=false expects exactly one parsed text");
    audio = synth_one(*lines[0]);
  }
  return tts_util::array_to_vec(audio);
}

struct TokenBatch {
  std::vector<float> style_vector;
  std::vector<sbv2_token_utterance> utts;  // the non-empty lines in line order
  std::vector<int64_t> pause;
  sbv2_assist_text assist{};
  std::vector<int32_t> assist_of;
  std::vector<const int32_t*> durations;  // [utts] or empty: all predicted
  int64_t n_phonemes = 0;
  const sbv2_assist_text* assist_ptr() const { return assist_of.empty() ? nullptr : &assist; }
  const int32_t* assist_of_ptr() const { return assist_of.empty() ? nullptr : assist_of.data(); }
};

sbv2_model* TTSModelHolder::token_batch(const std::string& ident, const std::vector<std::optional<ParsedTokens>>& lines,
                                        int32_t style_id, int64_t speaker_id, const SynthesizeOptions& options, TokenBatch& out) {
  find_and_load_model(ident);
  out.style_vector = get_style_vector(ident, style_id, options.style_weight);
  TTSModel* m = find_model(ident);
  if (!m || !m->vits2) throw Error(ErrorKind::ModelNotFoundError, "model not found error: " + ident);
  if (!options.split_sentences && (lines.size() != 1 || !lines[0]))
    throw Error(ErrorKind::ValueError, "split_sentences=false expects exactly one parsed text");
  if (!options.durations.empty() && options.durations.size() != lines.size())
    throw Error(ErrorKind::ValueError, "durations must have one entry per line of the request");
  for (size_t i = 0; i < lines.size(); ++i) {
    if (!lines[i]) continue;  // empty line (tts.rs:293-295)
    const ParsedTokens& t = *lines[i];
    const int64_t t_x = int64_t(t.phones.size());
    if (int64_t(t.tones.size()) != t_x || int64_t(t.lang_ids.size()) != t_x)
      throw Error(ErrorKind::OrtError, "x_tst, tones and language must agree on x_tst_max_length");
    if (t.token_ids.size() != t.attention_masks.size() || t.word2ph.size() != t.token_ids.size())
      throw Error(ErrorKind::OtherError, "word2ph length must equal the number of BERT rows");
    sbv2_token_utterance u{};
    u.input_ids = t.token_ids.data();
    u.attention_mask = t.attention_masks.data();
    u.t_tok = int64_t(t.token_ids.size());
    u.word2ph = t.word2ph.data();
    u.x_tst = t.phones.data();
    u.tones = t.tones.data();
    u.lang_ids = t.lang_ids.data();
    u.t_x = t_x;
    u.sid = speaker_id;
    u.style_vec = out.style_vector.data();
    u.sdp_ratio = options.sdp_ratio;
    u.length_scale = options.length_scale;
    u.noise_scale = 0.677f;
    u.noise_scale_w = 0.8f;
    out.utts.push_back(u);
    out.n_phonemes += t_x;
    // tts.rs:318-320: half a second of silence after every line but the last one of the text
    out.pause.push_back(options.split_sentences && i != lines.size() - 1 ? 22050 : 0);
    if (!options.durations.empty()) {
      const auto& d = options.durations[i];
      if (d && int64_t(d->size()) != t_x) throw Error(ErrorKind::ValueError, "durations of a line must have one entry per phoneme");
      out.durations.push_back(d ? d->data() : nullptr);
    }
  }
  if (out.utts.empty()) throw Error(ErrorKind::NdArrayError, "NDArray error: nothing to concatenate");
  if (options.assist) {
    check_assist(*options.assist);
    out.assist.input_ids = options.assist->token_ids.data();
    out.assist.attention_mask = options.assist->attention_masks.data();
    out.assist.t_tok = int64_t(options.assist->token_ids.size());
    out.assist.weight = options.assist->weight;
    out.assist_of.assign(out.utts.size(), 0);
  }
  return m->vits2->get();
}

std::vector<uint8_t> TTSModelHolder::easy_synthesize_tokens(const std::string& ident,
                                                            const std::vector<std::optional<ParsedTokens>>& lines, int32_t style_id,
                                                            int64_t speaker_id, const SynthesizeOptions& options, TokenTiming* timing) {
  TokenBatch tb;
  sbv2_model* synth = token_batch(ident, lines, style_id, speaker_id, options, tb);
  const size_t B = tb.utts.size();
  std::vector<int32_t> dur(timing ? size_t(tb.n_phonemes) : 0);
  std::vector<int64_t> n(B, 0);
  float* samples = nullptr;
  int64_t total = 0;
  check(sbv2_synthesize_from_tokens_with_durations(synth, bert_.get(), tb.utts.data(), int(B), tb.assist_ptr(), tb.assist_of.empty() ? 0 : 1,
                                                   tb.assist_of_ptr(), tb.pause.data(), tb.durations.empty() ? nullptr : tb.durations.data(),
                                                   timing ? dur.data() : nullptr, &samples, &total, n.data()));
  if (timing) {
    // sentence k starts after the samples and pauses of the sentences before it; hop = samples / T_y, T_y = max(1, sum d)
    timing->phoneme_start.assign(size_t(tb.n_phonemes), 0);
    int64_t start = 0, p = 0;
    for (size_t k = 0; k < B; ++k) {
      int64_t ty = 0;
      for (int64_t t = 0; t < tb.utts[k].t_x; ++t) ty += dur[size_t(p + t)];
      const int64_t hop = n[k] / std::max<int64_t>(ty, 1);
      int64_t cum = 0;
      for (int64_t t = 0; t < tb.utts[k].t_x; ++t, ++p) {
        timing->phoneme_start[size_t(p)] = start + cum * hop;
        cum += dur[size_t(p)];
      }
      start += n[k] + tb.pause[k];
    }
    timing->durations = std::move(dur);
  }
  void* wav = nullptr;
  size_t wav_n = 0;
  const int st = sbv2_wav_from_f32(samples, total, &wav, &wav_n);
  sbv2_free(samples);
  check(st);
  std::vector<uint8_t> out(static_cast<uint8_t*>(wav), static_cast<uint8_t*>(wav) + wav_n);
  sbv2_free(wav);
  return out;
}

std::vector<int32_t> TTSModelHolder::predict_durations_tokens(const std::string& ident,
                                                              const std::vector<std::optional<ParsedTokens>>& lines, int32_t style_id,
                                                              int64_t speaker_id, const SynthesizeOptions& options) {
  TokenBatch tb;
  sbv2_model* synth = token_batch(ident, lines, style_id, speaker_id, options, tb);
  std::vector<int32_t> dur(size_t(tb.n_phonemes));
  check(sbv2_predict_durations_from_tokens(synth, bert_.get(), tb.utts.data(), int(tb.utts.size()), tb.assist_ptr(),
                                           tb.assist_of.empty() ? 0 : 1, tb.assist_of_ptr(), dur.data()));
  return dur;
}

}  // namespace host
}  // namespace sbv2

// ---- C ABI over the holder (so non-C++ callers and the Python tests can drive it) -----------------
namespace {
template <class F>
int holder_guard(F&& f) {
  try {
    f();
    return SBV2_OK;
  } catch (const sbv2::host::Error& e) {
    sbv2_set_last_error(e.what());
    using K = sbv2::host::ErrorKind;
    switch (e.kind) {
      case K::ModelNotFoundError: return SBV2_ERR_MODEL_NOT_FOUND;
      case K::ValueError:
      case K::NdArrayError: return SBV2_ERR_INVALID_ARGUMENT;
      case K::SerdeJsonError:
      case K::IoError:
      case K::Base64Error: return SBV2_ERR_PARSE;
      case K::OrtError: return SBV2_ERR_UNSUPPORTED;
      default: return SBV2_ERR_INTERNAL;
    }
  } catch (const std::exception& e) {
    sbv2_set_last_error(e.what());
    return SBV2_ERR_INTERNAL;
  } catch (...) {
    sbv2_set_last_error("unknown error");
    return SBV2_ERR_INTERNAL;
  }
}
}  // namespace

struct sbv2_holder {
  sbv2::host::TTSModelHolder impl;
};

extern "C" {

int sbv2_holder_new(const void* bert_onnx, size_t bert_n, const void* tokenizer, size_t tok_n, int64_t max_loaded_models,
                    int device_ordinal, sbv2_holder** out) {
  return holder_guard([&] {
    if (!out || !bert_onnx) throw sbv2::host::Error(sbv2::host::ErrorKind::ValueError, "null argument");
    *out = nullptr;
    std::vector<uint8_t> b(static_cast<const uint8_t*>(bert_onnx), static_cast<const uint8_t*>(bert_onnx) + bert_n);
    std::vector<uint8_t> t;
    if (tokenizer) t.assign(static_cast<const uint8_t*>(tokenizer), static_cast<const uint8_t*>(tokenizer) + tok_n);
    std::optional<size_t> mx;
    if (max_loaded_models >= 0) mx = size_t(max_loaded_models);
    *out = new sbv2_holder{sbv2::host::TTSModelHolder(b, t, mx, device_ordinal)};
  });
}

void sbv2_holder_free(sbv2_holder* h) { delete h; }

namespace {
void need(const void* p, const char* what) {
  if (!p) throw sbv2::host::Error(sbv2::host::ErrorKind::ValueError, std::string("null argument: ") + what);
}
}  // namespace

int sbv2_holder_load_sbv2file(sbv2_holder* h, const char* ident, const void* bytes, size_t n) {
  return holder_guard([&] {
    need(h, "holder"), need(ident, "ident"), need(bytes, "bytes");
    std::vector<uint8_t> b(static_cast<const uint8_t*>(bytes), static_cast<const uint8_t*>(bytes) + n);
    h->impl.load_sbv2file(ident, b);
  });
}

int sbv2_holder_load(sbv2_holder* h, const char* ident, const void* style_json, size_t style_n, const void* onnx, size_t onnx_n) {
  return holder_guard([&] {
    need(h, "holder"), need(ident, "ident"), need(style_json, "style_json"), need(onnx, "onnx");
    std::vector<uint8_t> s(static_cast<const uint8_t*>(style_json), static_cast<const uint8_t*>(style_json) + style_n);
    std::vector<uint8_t> o(static_cast<const uint8_t*>(onnx), static_cast<const uint8_t*>(onnx) + onnx_n);
    h->impl.load(ident, s, o);
  });
}

int sbv2_holder_load_aivmx(sbv2_holder* h, const char* ident, const void* bytes, size_t n) {
  return holder_guard([&] {
    need(h, "holder"), need(ident, "ident"), need(bytes, "bytes");
    std::vector<uint8_t> b(static_cast<const uint8_t*>(bytes), static_cast<const uint8_t*>(bytes) + n);
    h->impl.load_aivmx(ident, b);
  });
}

int sbv2_holder_unload(sbv2_holder* h, const char* ident, int* found) {
  return holder_guard([&] {
    need(h, "holder"), need(ident, "ident");
    bool f = h->impl.unload(ident);
    if (found) *found = f ? 1 : 0;
  });
}

int sbv2_holder_models(const sbv2_holder* h, char** out) {
  return holder_guard([&] {
    need(h, "holder"), need(out, "out");
    std::string s;
    for (auto& m : h->impl.models()) {
      if (!s.empty()) s += "\n";
      s += m;
    }
    char* p = static_cast<char*>(sbv2_alloc(s.size() + 1));
    memcpy(p, s.c_str(), s.size() + 1);
    *out = p;
  });
}

int sbv2_holder_loaded_count(const sbv2_holder* h, int* out) {
  return holder_guard([&] {
    need(h, "holder"), need(out, "out");
    *out = int(h->impl.loaded_count());
  });
}

int sbv2_holder_bert_hidden_size(const sbv2_holder* h, int* out) {
  return holder_guard([&] {
    need(h, "holder"), need(out, "out");
    if (sbv2_bert_hidden_size(const_cast<sbv2_holder*>(h)->impl.bert_session().get(), out) != SBV2_OK)
      throw sbv2::host::Error(sbv2::host::ErrorKind::OrtError, sbv2_last_error());
  });
}

int sbv2_holder_get_style_vector(sbv2_holder* h, const char* ident, int32_t style_id, float weight, float* out) {
  return holder_guard([&] {
    need(h, "holder"), need(ident, "ident"), need(out, "out");
    auto v = h->impl.get_style_vector(ident, style_id, weight);
    memcpy(out, v.data(), v.size() * 4);
  });
}

namespace {
// copies an assist text of the C ABI after the checks that make the copy safe (the rest: check_assist)
std::optional<sbv2::host::AssistText> assist_from_c(const sbv2_assist_text* a) {
  if (!a) return std::nullopt;
  need(a->input_ids, "assist input_ids"), need(a->attention_mask, "assist attention_mask");
  if (a->t_tok <= 0 || a->t_tok > 32768) throw sbv2::host::Error(sbv2::host::ErrorKind::ValueError, "assist text must have 1 .. 32768 tokens");
  sbv2::host::AssistText t;
  t.token_ids.assign(a->input_ids, a->input_ids + a->t_tok);
  t.attention_masks.assign(a->attention_mask, a->attention_mask + a->t_tok);
  t.weight = a->weight;
  return t;
}
}  // namespace

int sbv2_holder_bert_features(sbv2_holder* h, const int64_t* token_ids, const int64_t* attention_mask, int64_t t_tok,
                              const int32_t* word2ph, float** out, int64_t* t_x) {
  return sbv2_holder_bert_features_assist(h, token_ids, attention_mask, t_tok, word2ph, nullptr, out, t_x);
}

int sbv2_holder_bert_features_assist(sbv2_holder* h, const int64_t* token_ids, const int64_t* attention_mask, int64_t t_tok,
                                     const int32_t* word2ph, const sbv2_assist_text* assist, float** out, int64_t* t_x) {
  return holder_guard([&] {
    need(h, "holder"), need(token_ids, "token_ids"), need(attention_mask, "attention_mask"), need(word2ph, "word2ph"), need(out, "out"),
        need(t_x, "t_x");
    if (t_tok <= 0) throw sbv2::host::Error(sbv2::host::ErrorKind::ValueError, "t_tok must be positive");
    std::vector<int64_t> ids(token_ids, token_ids + t_tok), mask(attention_mask, attention_mask + t_tok);
    std::vector<int32_t> w(word2ph, word2ph + t_tok);
    const std::optional<sbv2::host::AssistText> at = assist_from_c(assist);
    auto a = h->impl.bert_features(ids, mask, w, at ? &*at : nullptr);
    float* p = static_cast<float*>(sbv2_alloc(a.data.size() * 4 + 4));
    memcpy(p, a.data.data(), a.data.size() * 4);
    *out = p;
    *t_x = a.cols;
  });
}

int sbv2_holder_easy_synthesize(sbv2_holder* h, const char* ident, const sbv2_sentence* sentences, int n_sentences,
                                int64_t total_lines, int32_t style_id, int64_t speaker_id, float sdp_ratio, float length_scale,
                                float style_weight, void** wav_bytes, size_t* wav_n) {
  return holder_guard([&] {
    using namespace sbv2::host;
    need(h, "holder"), need(ident, "ident"), need(wav_bytes, "wav_bytes"), need(wav_n, "wav_n");
    if (n_sentences > 0) need(sentences, "sentences");
    // rows of bert_ori = hidden size of the holder's DeBERTa (1024 for deberta-v2-large; model.rs:66-68 feeds what bert.rs returns)
    int hidden = 0;
    if (sbv2_bert_hidden_size(h->impl.bert_session().get(), &hidden) != SBV2_OK || hidden <= 0)
      throw Error(ErrorKind::OrtError, "cannot determine the BERT hidden size");
    std::vector<std::optional<ParsedText>> lines(size_t(total_lines > 0 ? total_lines : 0));
    for (int i = 0; i < n_sentences; ++i) {
      const sbv2_sentence& s = sentences[i];
      if (s.line_index < 0 || s.line_index >= total_lines) throw Error(ErrorKind::ValueError, "line_index out of range");
      if (!s.bert || !s.phones || !s.tones || !s.lang_ids || s.t_x <= 0) throw Error(ErrorKind::ValueError, "sentence with null or empty input");
      ParsedText t;
      t.bert_ori.rows = hidden;
      t.bert_ori.cols = s.t_x;
      t.bert_ori.data.assign(s.bert, s.bert + size_t(hidden) * size_t(s.t_x));
      t.phones.assign(s.phones, s.phones + s.t_x);
      t.tones.assign(s.tones, s.tones + s.t_x);
      t.lang_ids.assign(s.lang_ids, s.lang_ids + s.t_x);
      lines[size_t(s.line_index)] = std::move(t);
    }
    SynthesizeOptions opt;
    opt.sdp_ratio = sdp_ratio;
    opt.length_scale = length_scale;
    opt.style_weight = style_weight;
    opt.split_sentences = true;
    auto wav = h->impl.easy_synthesize(ident, lines, style_id, speaker_id, opt);
    void* p = sbv2_alloc(wav.size());
    memcpy(p, wav.data(), wav.size());
    *wav_bytes = p;
    *wav_n = wav.size();
  });
}

int sbv2_holder_easy_synthesize_tokens(sbv2_holder* h, const char* ident, const sbv2_token_sentence* sentences, int n_sentences,
                                       int64_t total_lines, int32_t style_id, int64_t speaker_id, float sdp_ratio, float length_scale,
                                       float style_weight, void** wav_bytes, size_t* wav_n) {
  return sbv2_holder_easy_synthesize_tokens_assist(h, ident, sentences, n_sentences, total_lines, style_id, speaker_id, sdp_ratio,
                                                   length_scale, style_weight, nullptr, wav_bytes, wav_n);
}

int sbv2_holder_easy_synthesize_tokens_assist(sbv2_holder* h, const char* ident, const sbv2_token_sentence* sentences, int n_sentences,
                                              int64_t total_lines, int32_t style_id, int64_t speaker_id, float sdp_ratio,
                                              float length_scale, float style_weight, const sbv2_assist_text* assist, void** wav_bytes,
                                              size_t* wav_n) {
  return sbv2_holder_easy_synthesize_tokens_timed(h, ident, sentences, n_sentences, total_lines, style_id, speaker_id, sdp_ratio,
                                                  length_scale, style_weight, assist, nullptr, nullptr, nullptr, wav_bytes, wav_n);
}

namespace {
// sentences of the C ABI -> one entry per line of the request (empty optional = empty line); `unique` rejects a
// line_index named twice (the timing arrays have one slot per sentence)
std::vector<std::optional<sbv2::host::ParsedTokens>> token_lines(const sbv2_token_sentence* sentences, int n_sentences, int64_t total_lines,
                                                                 bool unique) {
  using namespace sbv2::host;
  if (n_sentences > 0) need(sentences, "sentences");
  std::vector<std::optional<ParsedTokens>> lines(size_t(total_lines > 0 ? total_lines : 0));
  for (int i = 0; i < n_sentences; ++i) {
    const sbv2_token_sentence& s = sentences[i];
    if (s.line_index < 0 || s.line_index >= total_lines) throw Error(ErrorKind::ValueError, "line_index out of range");
    if (!s.token_ids || !s.attention_mask || !s.word2ph || !s.phones || !s.tones || !s.lang_ids || s.t_tok <= 0 || s.t_x <= 0)
      throw Error(ErrorKind::ValueError, "sentence with null or empty input");
    if (unique && lines[size_t(s.line_index)]) throw Error(ErrorKind::ValueError, "two sentences name the same line_index");
    ParsedTokens t;
    t.token_ids.assign(s.token_ids, s.token_ids + s.t_tok);
    t.attention_masks.assign(s.attention_mask, s.attention_mask + s.t_tok);
    t.word2ph.assign(s.word2ph, s.word2ph + s.t_tok);
    t.phones.assign(s.phones, s.phones + s.t_x);
    t.tones.assign(s.tones, s.tones + s.t_x);
    t.lang_ids.assign(s.lang_ids, s.lang_ids + s.t_x);
    lines[size_t(s.line_index)] = std::move(t);
  }
  return lines;
}

sbv2::host::SynthesizeOptions token_options(float sdp_ratio, float length_scale, float style_weight, const sbv2_assist_text* assist) {
  sbv2::host::SynthesizeOptions opt;
  opt.sdp_ratio = sdp_ratio;
  opt.length_scale = length_scale;
  opt.style_weight = style_weight;
  opt.split_sentences = true;
  opt.assist = assist_from_c(assist);
  return opt;
}

// first phoneme of each sentence (sentences[] order) in the line-order concatenation the holder returns
std::vector<int64_t> line_order_offsets(const sbv2_token_sentence* sentences, int n_sentences) {
  std::vector<int> order(static_cast<size_t>(n_sentences));
  for (int i = 0; i < n_sentences; ++i) order[size_t(i)] = i;
  std::sort(order.begin(), order.end(), [&](int a, int b) { return sentences[a].line_index < sentences[b].line_index; });
  std::vector<int64_t> off(static_cast<size_t>(n_sentences), 0);
  int64_t o = 0;
  for (int k : order) {
    off[size_t(k)] = o;
    o += sentences[k].t_x;
  }
  return off;
}
}  // namespace

int sbv2_holder_predict_durations_tokens(sbv2_holder* h, const char* ident, const sbv2_token_sentence* sentences, int n_sentences,
                                         int64_t total_lines, int32_t style_id, int64_t speaker_id, float sdp_ratio,
                                         float length_scale, float style_weight, const sbv2_assist_text* assist,
                                         int32_t* out_durations) {
  return holder_guard([&] {
    need(h, "holder"), need(ident, "ident"), need(out_durations, "out_durations");
    auto lines = token_lines(sentences, n_sentences, total_lines, true);
    const std::vector<int32_t> d = h->impl.predict_durations_tokens(ident, lines, style_id, speaker_id,
                                                                    token_options(sdp_ratio, length_scale, style_weight, assist));
    const std::vector<int64_t> off = line_order_offsets(sentences, n_sentences);
    int64_t o = 0;
    for (int i = 0; i < n_sentences; ++i) {
      std::copy(d.begin() + off[size_t(i)], d.begin() + off[size_t(i)] + sentences[i].t_x, out_durations + o);
      o += sentences[i].t_x;
    }
  });
}

int sbv2_holder_easy_synthesize_tokens_timed(sbv2_holder* h, const char* ident, const sbv2_token_sentence* sentences, int n_sentences,
                                             int64_t total_lines, int32_t style_id, int64_t speaker_id, float sdp_ratio,
                                             float length_scale, float style_weight, const sbv2_assist_text* assist,
                                             const int32_t* const* durations, int32_t* out_durations, int64_t* out_phoneme_start,
                                             void** wav_bytes, size_t* wav_n) {
  return holder_guard([&] {
    using namespace sbv2::host;
    need(h, "holder"), need(ident, "ident"), need(wav_bytes, "wav_bytes"), need(wav_n, "wav_n");
    const bool timed = durations || out_durations || out_phoneme_start;
    auto lines = token_lines(sentences, n_sentences, total_lines, timed);
    SynthesizeOptions opt = token_options(sdp_ratio, length_scale, style_weight, assist);
    if (durations) {
      opt.durations.resize(lines.size());
      for (int i = 0; i < n_sentences; ++i)
        if (durations[i]) opt.durations[size_t(sentences[i].line_index)].emplace(durations[i], durations[i] + sentences[i].t_x);
    }
    TokenTiming timing;
    auto wav = h->impl.easy_synthesize_tokens(ident, lines, style_id, speaker_id, opt, timed ? &timing : nullptr);
    if (timed) {
      const std::vector<int64_t> off = line_order_offsets(sentences, n_sentences);
      int64_t o = 0;
      for (int i = 0; i < n_sentences; ++i) {
        const size_t a = size_t(off[size_t(i)]), n = size_t(sentences[i].t_x);
        if (out_durations) std::copy(timing.durations.begin() + long(a), timing.durations.begin() + long(a + n), out_durations + o);
        if (out_phoneme_start)
          std::copy(timing.phoneme_start.begin() + long(a), timing.phoneme_start.begin() + long(a + n), out_phoneme_start + o);
        o += int64_t(n);
      }
    }
    void* p = sbv2_alloc(wav.size());
    memcpy(p, wav.data(), wav.size());
    *wav_bytes = p;
    *wav_n = wav.size();
  });
}

}  // extern "C"
