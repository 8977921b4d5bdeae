// C++ mirror of sbv2_core's public API for the synthesis path, written above the C ABI
// (include/sbv2_b200.h) exactly where the reference sits above `ort`:
//   model::load_model / model::synthesize   crates/sbv2_core/src/model.rs:6-111
//   bert::predict                           crates/sbv2_core/src/bert.rs:6-24
//   tts::TTSModelHolder                     crates/sbv2_core/src/tts.rs:40-349
//   tts_util::parse_text (device half), array_to_vec   tts_util.rs:120-180
// Same names, argument meaning and error behaviour; Rust's Result<T> becomes a thrown
// sbv2::host::Error carrying the reference's error variant.  The text frontend (jpreprocess,
// tokenizer) stays outside: callers hand over what `parse_text` would have produced.
#pragma once
#include <cstdint>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/sbv2_b200.h"

namespace sbv2 {
namespace host {

enum class ErrorKind { OrtError, NdArrayError, ValueError, SerdeJsonError, IoError, ModelNotFoundError, Base64Error, OtherError };

struct Error : std::runtime_error {
  ErrorKind kind;
  Error(ErrorKind k, const std::string& m) : std::runtime_error(m), kind(k) {}
};

// RAII owner of one sbv2_model (= ort::Session).
class Session {
 public:
  Session() = default;
  explicit Session(sbv2_model* m) : m_(m) {}
  Session(Session&& o) noexcept : m_(o.m_) { o.m_ = nullptr; }
  Session& operator=(Session&& o) noexcept;
  Session(const Session&) = delete;
  Session& operator=(const Session&) = delete;
  ~Session();
  sbv2_model* get() const { return m_; }
  std::optional<std::string> metadata_custom(const std::string& key) const;

 private:
  sbv2_model* m_ = nullptr;
};

struct Array2 {  // row-major f32
  int64_t rows = 0, cols = 0;
  std::vector<float> data;
};

namespace model {
Session load_model(const std::vector<uint8_t>& model_file, bool bert, int device_ordinal = 0);
// returns the [1,1,N] audio array flattened
std::vector<float> synthesize(Session& session, const Array2& bert_ori /*[1024,T_x]*/, const std::vector<int64_t>& x_tst,
                              const std::vector<int64_t>& spk_ids, const std::vector<int64_t>& tones,
                              const std::vector<int64_t>& lang_ids, const std::vector<float>& style_vector, float sdp_ratio,
                              float length_scale, float noise_scale, float noise_scale_w);
// Additive entry (SURVEY.md §8f row 1): bert::predict + tts_util word2ph expansion + synthesize in one call, the BERT
// features never leave the device.  Same result as the three separate calls.
std::vector<float> synthesize_from_tokens(Session& session, Session& bert, const std::vector<int64_t>& token_ids,
                                          const std::vector<int64_t>& attention_masks, const std::vector<int32_t>& word2ph,
                                          const std::vector<int64_t>& x_tst, const std::vector<int64_t>& spk_ids,
                                          const std::vector<int64_t>& tones, const std::vector<int64_t>& lang_ids,
                                          const std::vector<float>& style_vector, float sdp_ratio, float length_scale,
                                          float noise_scale, float noise_scale_w);
}  // namespace model

namespace bert {
Array2 predict(Session& session, const std::vector<int64_t>& token_ids, const std::vector<int64_t>& attention_masks);
}

// Style-Bert-VITS2's assist text (assist_text / assist_text_weight): another text, normalised and tokenised like the main
// text (CLS ... SEP), whose mean DeBERTa row is mixed into every phoneme feature with this weight.
struct AssistText {
  std::vector<int64_t> token_ids, attention_masks;
  float weight = 0.0f;
};

namespace tts_util {
// bert rows repeated word2ph[i] times, concatenated, transposed -> [hidden, sum(word2ph)]
Array2 expand_bert_features(const Array2& bert_content, const std::vector<int32_t>& word2ph);
// Host restatement of the device blend (include/sbv2_b200.h, sbv2_assist_text), bit for bit: the column means of an
// assist's DeBERTa rows [n_a, hidden] with one fp64 accumulator per column summed in token order ...
std::vector<float> assist_mean(const Array2& assist_content);
// ... and the expansion with every row replaced by fl(fl(row * (float)(1 - (double)weight)) + fl(mean * weight)).
// This file is compiled with -ffp-contract=off so that no fused multiply-add forms.
Array2 expand_bert_features(const Array2& bert_content, const std::vector<int32_t>& word2ph, const std::vector<float>& mean,
                            float weight);
std::vector<uint8_t> array_to_vec(const std::vector<float>& audio);
}  // namespace tts_util

struct SynthesizeOptions {
  float sdp_ratio = 0.0f;
  float length_scale = 1.0f;
  float style_weight = 1.0f;
  bool split_sentences = true;
  // applies to every line of the request (style_bert_vits2 TTSModel.infer passes it to each line); easy_synthesize_tokens only
  std::optional<AssistText> assist;
  // given phoneme durations in latent frames, per line of the request (include/sbv2_b200.h states the contract): empty =
  // all predicted, an empty optional = that line predicted; easy_synthesize_tokens only
  std::vector<std::optional<std::vector<int32_t>>> durations;
};

// Where the phonemes of a request land (easy_synthesize_tokens): both [sum t_x] over the non-empty lines in line order.
struct TokenTiming {
  std::vector<int32_t> durations;      // frames per phoneme, given or predicted
  std::vector<int64_t> phoneme_start;  // index of the phoneme's first sample in the WAV's sample data (ends at start + d * hop)
};
struct TokenBatch;  // one request's sentences as the C ABI takes them (tts.cpp)

// Output of the (out-of-scope) text frontend for one line of text.
struct ParsedText {
  Array2 bert_ori;  // [1024, T_x]
  std::vector<int64_t> phones, tones, lang_ids;
};

// The same for the device-resident chain (SURVEY.md §8f rows 1-2): the tokenizer's ids / mask and word2ph instead of
// BERT features; DeBERTa then runs inside easy_synthesize_tokens, batched over the lines of the request.
struct ParsedTokens {
  std::vector<int64_t> token_ids, attention_masks;
  std::vector<int32_t> word2ph;
  std::vector<int64_t> phones, tones, lang_ids;
};

struct TTSModel {
  std::optional<Session> vits2;
  Array2 style_vectors;
  std::string ident;
  std::optional<std::vector<uint8_t>> bytes;
};

class TTSModelHolder {
 public:
  TTSModelHolder(const std::vector<uint8_t>& bert_model_bytes, const std::vector<uint8_t>& tokenizer_bytes,
                 std::optional<size_t> max_loaded_models, int device_ordinal = 0);
  std::vector<std::string> models() const;
  void load_aivmx(const std::string& ident, const std::vector<uint8_t>& aivmx_bytes);
  void load_sbv2file(const std::string& ident, const std::vector<uint8_t>& sbv2_bytes);
  void load(const std::string& ident, const std::vector<uint8_t>& style_vectors_bytes, const std::vector<uint8_t>& vits2_bytes);
  bool unload(const std::string& ident);
  std::vector<float> get_style_vector(const std::string& ident, int32_t style_id, float weight);
  // device half of parse_text.  With an assist text of non-zero weight DeBERTa runs once over [sentence, assist] (the
  // layout of sbv2_synthesize_from_tokens_assist) and the blend is done on the host (tts_util::assist_mean and
  // expand_bert_features); weight 0 is the plain path.
  Array2 bert_features(const std::vector<int64_t>& token_ids, const std::vector<int64_t>& attention_masks,
                       const std::vector<int32_t>& word2ph, const AssistText* assist = nullptr);
  // easy_synthesize over already-parsed lines. `lines[i]` empty optional == empty line (skipped, but
  // it still counts for the "not the last line" silence rule, tts.rs:293-320).
  std::vector<uint8_t> easy_synthesize(const std::string& ident, const std::vector<std::optional<ParsedText>>& lines, int32_t style_id,
                                       int64_t speaker_id, const SynthesizeOptions& options);
  // easy_synthesize with bert::predict folded in: every non-empty line of the request goes through DeBERTa as ONE
  // right-padded batch and through the synthesizer as ONE batch (features never leave the device), the 22 050-sample
  // pauses of tts.rs:318-320 are written on the device, and the WAV is one header + one copy of the pinned result.
  // timing (optional) receives the durations used and where each phoneme starts in the WAV.
  std::vector<uint8_t> easy_synthesize_tokens(const std::string& ident, const std::vector<std::optional<ParsedTokens>>& lines,
                                              int32_t style_id, int64_t speaker_id, const SynthesizeOptions& options,
                                              TokenTiming* timing = nullptr);
  // "audio query": the durations easy_synthesize_tokens would use without given durations ([sum t_x], line order); runs
  // DeBERTa, the text encoder and the duration predictors only.
  std::vector<int32_t> predict_durations_tokens(const std::string& ident, const std::vector<std::optional<ParsedTokens>>& lines,
                                                int32_t style_id, int64_t speaker_id, const SynthesizeOptions& options);
  size_t loaded_count() const;
  Session& bert_session() { return bert_; }

 private:
  TTSModel* find_model(const std::string& ident);
  bool find_and_load_model(const std::string& ident);
  sbv2_model* token_batch(const std::string& ident, const std::vector<std::optional<ParsedTokens>>& lines, int32_t style_id,
                          int64_t speaker_id, const SynthesizeOptions& options, TokenBatch& out);
  std::vector<uint8_t> tokenizer_;
  Session bert_;
  std::vector<TTSModel> models_;
  std::optional<size_t> max_loaded_models_;
  int device_ = 0;
};

}  // namespace host
}  // namespace sbv2
