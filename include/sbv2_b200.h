/*
 * sbv2_b200.h — C ABI of the B200-native backend that replaces the ONNX Runtime session layer of
 * tuna2134/sbv2-api's `sbv2_core` (crates/sbv2_core/src/model.rs, bert.rs) and the asset readers
 * it depends on (sbv2file.rs, style.rs, tts.rs:78-123).
 *
 * Conventions
 *   - Every function returns SBV2_OK (0) on success and a non-zero sbv2_status otherwise; it never
 *     aborts and never throws across the boundary.  `sbv2_last_error()` returns a thread-local,
 *     NUL-terminated description of the last failure on the calling thread (the analogue of
 *     `ort::Error` -> `Error::OrtError`, crates/sbv2_core/src/error.rs:12-14).
 *   - Inputs are borrowed for the duration of the call.  Outputs whose size is data dependent are
 *     allocated by the library (pinned host memory) and released with `sbv2_free`.
 *   - One in-flight call per `sbv2_model` (the reference takes `&mut Session`); different models
 *     may be driven from different host threads.  One `sbv2_model` lives on one device ordinal.
 *   - There is no CPU fallback: if no sm_100 device is present `sbv2_model_create` fails.
 *   - All arrays are dense, row-major, host memory unless the name ends in `_dev`.
 */
#ifndef SBV2_B200_H_
#define SBV2_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum sbv2_status {
  SBV2_OK = 0,
  SBV2_ERR_INVALID_ARGUMENT = 1, /* maps to Error::ValueError / NdArrayError */
  SBV2_ERR_PARSE = 2,            /* malformed ONNX / .sbv2 / JSON / npy (Error::OrtError, SerdeJsonError, IoError) */
  SBV2_ERR_MODEL_NOT_FOUND = 3,  /* Error::ModelNotFoundError */
  SBV2_ERR_CUDA = 4,             /* device / driver failure (Error::OrtError) */
  SBV2_ERR_UNSUPPORTED = 5,      /* graph is not a JP-Extra synthesizer / DeBERTa-v2 encoder */
  SBV2_ERR_INTERNAL = 6
} sbv2_status;

typedef struct sbv2_model sbv2_model; /* opaque; stands for one ort::Session */

/* ---- library ------------------------------------------------------------------------------ */

/* Thread-local message of the last failing call on this thread ("" if none). */
const char* sbv2_last_error(void);
/* Releases any buffer returned through an out-pointer by this library. NULL is allowed. */
void sbv2_free(void* p);
/* Allocates a buffer that sbv2_free releases (for host layers built above this ABI). */
void* sbv2_alloc(size_t bytes);
/* Page-locked host memory (cudaHostAlloc) that sbv2_free releases.  Input buffers that live in page-locked memory —
 * from here, cudaHostAlloc or cudaHostRegister — are read by the copy engine in place; pageable inputs are staged through
 * an internal pinned block first (one extra memcpy of the BERT features per call). */
void* sbv2_alloc_pinned(size_t bytes);
/* Sets the calling thread's last-error message (for host layers built above this ABI). */
void sbv2_set_last_error(const char* message);
/* "sbv2_b200 <version> sm_100a"; static storage. */
const char* sbv2_version(void);
/* Number of CUDA devices with compute capability 10.x; 0 (and an error message) if none. */
int sbv2_device_count(void);

/* ---- model::load_model / Drop / metadata  (crates/sbv2_core/src/model.rs:6-50) -------------- */

/* Replaces `model::load_model(bytes, bert)`: parses the ONNX ModelProto in `onnx_bytes`, infers
 * the hyper-parameters from initializer shapes, converts and uploads every initializer to the
 * device once, and builds the static kernel plan.  `is_bert != 0` selects the DeBERTa-v2 feature
 * encoder (deberta.onnx, scripts/convert/convert_deberta.py), otherwise the JP-Extra synthesizer
 * (model.onnx inside a .sbv2, scripts/convert/convert_model.py). */
int sbv2_model_create(const void* onnx_bytes, size_t n_bytes, int is_bert, int device_ordinal,
                      sbv2_model** out_model);
/* Diagnostic (no device needed): JSON object describing which initializer every structurally bound weight name resolves to
 * — real exports constant-fold weight-normed convs and 3-D-input Linears into anonymous onnx::Conv_N / transposed
 * onnx::MatMul_N initializers (scripts/convert/convert_model.py:115-156, convert_deberta.py:36-52); the loaders recover
 * them through the still-named biases.  `*json` is library-allocated (sbv2_free). */
int sbv2_onnx_bind_report(const void* onnx_bytes, size_t n_bytes, int is_bert, char** json);
/* Replaces `Drop for Session` (unload / eviction, crates/sbv2_core/src/tts.rs:182-195, :238-241):
 * frees all device and pinned buffers. NULL is allowed. */
void sbv2_model_destroy(sbv2_model* model);
/* Replaces `session.metadata()?.custom(key)` (crates/sbv2_core/src/tts.rs:93-94, .aivmx style
 * vectors).  On success `*value` points to model-owned bytes (valid until destroy) and `*n` is the
 * length; a missing key yields SBV2_OK with `*value == NULL`. */
int sbv2_model_metadata(const sbv2_model* model, const char* key, const char** value, size_t* n);
/* Hyper-parameters inferred at load, as a JSON object string owned by the model. */
int sbv2_model_describe(const sbv2_model* model, const char** json);

/* ---- bert::predict  (crates/sbv2_core/src/bert.rs:6-24) ------------------------------------- */

/* input_ids, attention_mask: int64 [t_tok].  out: float32 [t_tok, hidden] (hidden = 1024 for
 * deberta-v2-large), caller-allocated.  Output = hidden_states[-3] of batch element 0
 * (scripts/convert/convert_deberta.py:34).
 * Restrictions the ONNX graph does not have: at most 32768 tokens per sequence (longer inputs return
 * SBV2_ERR_INVALID_ARGUMENT; every relative distance beyond +-512 reads the outermost position bucket, as in the graph),
 * and attention_mask must be a prefix of ones (right padding; a mask with holes returns
 * SBV2_ERR_UNSUPPORTED) — the reference's tokenizer only ever produces all-ones masks (tts_util.rs:120-128).
 * Numerics: SBV2_B200_BERT (read at sbv2_model_create) = "exact" (default: two-term fp16 operand splits, fp32 activations;
 * features reproduce HF fp32 to ~3e-4 and the synthesizer's durations exactly) or "fp16" (single-term operands, ~2x
 * faster, ~1 duration in 2000 differs downstream).  The disentangled attention runs on the tensor cores in both modes for
 * every length (SBV2_B200_BERT_ATTN=simt: CUDA-core cross-check kernels). */
int sbv2_bert_predict(sbv2_model* bert, const int64_t* input_ids, const int64_t* attention_mask,
                      int64_t t_tok, float* out);
/* Extension (the reference is batch 1): ids/mask int64 [batch, s] with right padding expressed by
 * mask zeros; out float32 [batch, s, hidden].  Row b is sbv2_bert_predict on the unpadded prefix of row b (bit for bit
 * while both calls take the same GEMM path; calls with few tokens split K over a thread-block cluster, whose fp32 sums are
 * formed in a different order — a relative difference of ~5e-5 in exact mode, far inside the mode's accuracy); padded
 * positions are written as zeros. */
int sbv2_bert_predict_batch(sbv2_model* bert, const int64_t* input_ids, const int64_t* attention_mask,
                            int batch, int64_t s, float* out);
int sbv2_bert_hidden_size(const sbv2_model* bert, int* hidden);

/* ---- model::synthesize  (crates/sbv2_core/src/model.rs:53-111) ------------------------------ */

/* One utterance, as the reference calls it.  bert: float32 [1024, t_x] (standard layout of
 * `bert_ori`, model.rs:66-68); x_tst/tones/lang: int64 [t_x]; style: float32 [256].
 * The two Gaussian noise tensors the ONNX graph draws internally are drawn here from a
 * counter-based generator seeded per model (sbv2_model_seed).
 * `*out_samples` receives float32 [n_samples] (the reference's Array3 [1,1,n]); free with sbv2_free. */
int sbv2_synthesize(sbv2_model* synth, const float* bert, const int64_t* x_tst, const int64_t* tones,
                    const int64_t* lang_ids, int64_t t_x, int64_t sid, const float* style_vec,
                    float sdp_ratio, float length_scale, float noise_scale, float noise_scale_w,
                    float** out_samples, int64_t* n_samples);
int sbv2_model_seed(sbv2_model* synth, uint64_t seed);

/* Parity entry point: same computation with the noise injected by the caller and the integer
 * alignment returned.  noise_sdp: float32 [2, t_x] (N(0,1), scaled by noise_scale_w inside);
 * noise_zp: float32 [192, noise_zp_frames] channel-major (only the first T_y frames are used; the
 * call fails with SBV2_ERR_INVALID_ARGUMENT if T_y > noise_zp_frames).
 * out_durations: int32 [t_x] (= ceil(w)), out_frame2ph: int32, library-allocated [T_y],
 * both optional (NULL to skip).  out_frame2ph[j] is the phoneme that owns frame j, or -1 for a frame
 * that belongs to no phoneme: when every duration is 0 (length_scale = 0) T_y is 1 and that frame
 * is synthesized from a zero prior mean and log-scale, as the ONNX graph does. */
int sbv2_synthesize_with_noise(sbv2_model* synth, const float* bert, const int64_t* x_tst,
                               const int64_t* tones, const int64_t* lang_ids, int64_t t_x, int64_t sid,
                               const float* style_vec, float sdp_ratio, float length_scale,
                               float noise_scale, float noise_scale_w, const float* noise_sdp,
                               const float* noise_zp, int64_t noise_zp_frames, float** out_samples,
                               int64_t* n_samples, int32_t* out_durations, int32_t** out_frame2ph,
                               int64_t* t_y);

/* SURVEY.md §8f row 1 — `parse_text` + `synthesize` of one sentence without the host round trip of the BERT features:
 * replaces bert::predict (bert.rs:6-24) -> word2ph repeat + transpose (tts_util.rs:129-154) -> model::synthesize
 * (model.rs:53-111).  The DeBERTa output stays on the device; phoneme i reads the row of its token
 * (token k is repeated word2ph[k] times, sum(word2ph) == t_x).  Both models must be on the same device.  The result is
 * bit-identical to sbv2_bert_predict + host expansion + sbv2_synthesize with the same generator state. */
int sbv2_synthesize_from_tokens(sbv2_model* synth, sbv2_model* bert, const int64_t* input_ids, const int64_t* attention_mask,
                                int64_t t_tok, const int32_t* word2ph /* [t_tok] */, const int64_t* x_tst, const int64_t* tones,
                                const int64_t* lang_ids, int64_t t_x, int64_t sid, const float* style_vec, float sdp_ratio,
                                float length_scale, float noise_scale, float noise_scale_w, float** out_samples,
                                int64_t* n_samples);

/* SURVEY.md §8f row 2 — the sentences of one request as one batch: replaces the per-line loop of
 * `easy_synthesize` (tts.rs:290-326: parse_text -> bert::predict -> synthesize per line, then concatenate with 22 050 zero
 * samples).  DeBERTa runs once over all sentences (right-padded batch), the features stay on the device, the synthesizer
 * runs once over all sentences, and `pause_after[i]` zero samples (NULL: none) are laid out after sentence i ON THE DEVICE,
 * so `*out_samples` (float32 [*out_total], pinned, sbv2_free) is the concatenated audio in one D2H copy.
 * out_n_samples (optional, int64 [batch]): synthesized samples of each sentence (without its pause).
 * Each sentence's audio is bit-identical to sbv2_synthesize_from_tokens of that sentence with the same generator state
 * only for batch == 1 (the internal noise stream is consumed batch-wise); durations do not depend on the batching. */
typedef struct sbv2_token_utterance {
  const int64_t* input_ids;      /* [t_tok] */
  const int64_t* attention_mask; /* [t_tok], all ones */
  int64_t t_tok;
  const int32_t* word2ph;        /* [t_tok], sum == t_x */
  const int64_t* x_tst;          /* [t_x] */
  const int64_t* tones;          /* [t_x] */
  const int64_t* lang_ids;       /* [t_x] */
  int64_t t_x;
  int64_t sid;
  const float* style_vec;        /* [256] */
  float sdp_ratio, length_scale, noise_scale, noise_scale_w;
} sbv2_token_utterance;
int sbv2_synthesize_from_tokens_batch(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch,
                                      const int64_t* pause_after /* [batch] or NULL */, float** out_samples,
                                      int64_t* out_total, int64_t* out_n_samples /* [batch] or NULL */);

/* Style-Bert-VITS2's assist text (`assist_text`, `assist_text_weight`; style_bert_vits2/nlp/japanese/bert_feature.py
 * extract_bert_feature): the tone of a sentence is steered toward another text by mixing that text's mean DeBERTa row into
 * the feature of every phoneme.  The assist text is normalised and tokenised by the caller exactly as the main text
 * (CLS ... SEP); an empty assist text means no blend (pass none).
 *
 * Numerics (bit for bit, on the device and in the host restatement of host/tts.hpp, tts_util::assist_mean /
 * expand_bert_features):
 *   F_a[t][c]   DeBERTa rows of the assist (hidden_states[-3], fp32), n_a = t_tok tokens, CLS and SEP included
 *   mean_a[c] = (float)((sum_{t=0..n_a-1} (double)F_a[t][c]) / (double)n_a), one fp64 accumulator per column, token order
 *   c_row     = (float)(1.0 - (double)weight), c_mean = weight
 *   row of phoneme p (token t) = fl(fl(F[t][c] * c_row) + fl(mean_a[c] * c_mean)), no fused multiply-add
 * The weight must be finite; any finite value is accepted (the reference does not clamp it).  A weight of 0 (or no
 * assist) takes the plain gather and never sends the assist through DeBERTa, so the result is bit-identical to
 * sbv2_synthesize_from_tokens_batch.
 * DeBERTa batch of one call: [sentences..., used assists...] right-padded to the longest row, where the used assists are
 * those some sentence names with a non-zero weight, in index order.  (Which rows share a call decides the GEMM path, and
 * thereby the last bits of every row: see DESIGN.md §4.) */
typedef struct sbv2_assist_text {
  const int64_t* input_ids;      /* [t_tok], the assist text through the same tokenizer */
  const int64_t* attention_mask; /* [t_tok], all ones */
  int64_t t_tok;                 /* 1 .. 32768 */
  float weight;                  /* assist_text_weight; 0 = no blend (DeBERTa is not run on it) */
} sbv2_assist_text;
/* sbv2_synthesize_from_tokens_batch with assist texts: sentence i blends assists[assist_of[i]] (-1 = none; assist_of NULL =
 * none for all).  Each sentence may carry its own assist, as it carries its own sid / style_vec / sdp_ratio.
 * SBV2_ERR_INVALID_ARGUMENT: assist_of out of [-1, n_assists), an assist with null arrays, t_tok outside 1 .. 32768, a mask
 * with a zero, or a non-finite weight (every entry of `assists` is checked, used or not). */
int sbv2_synthesize_from_tokens_assist(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch,
                                       const sbv2_assist_text* assists, int n_assists, const int32_t* assist_of /* [batch] or NULL */,
                                       const int64_t* pause_after /* [batch] or NULL */, float** out_samples, int64_t* out_total,
                                       int64_t* out_n_samples /* [batch] or NULL */);
/* Timing query of the token path (durations contract: see sbv2_predict_durations_batch below): DeBERTa, the text encoder
 * and the duration predictors, over the same DeBERTa batch as sbv2_synthesize_from_tokens_assist.
 * out_durations: int32 [sum t_x], caller-allocated. */
int sbv2_predict_durations_from_tokens(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch,
                                       const sbv2_assist_text* assists, int n_assists, const int32_t* assist_of /* [batch] or NULL */,
                                       int32_t* out_durations);
/* sbv2_synthesize_from_tokens_assist at given durations (durations[i] int32 [t_x] or NULL = predicted; durations NULL =
 * all predicted).  Given durations do not change the DeBERTa batch, so the features are those of the plain call.
 * out_durations (optional, caller-allocated int32 [sum t_x]) receives the durations used, given or predicted. */
int sbv2_synthesize_from_tokens_with_durations(sbv2_model* synth, sbv2_model* bert, const sbv2_token_utterance* utts, int batch,
                                               const sbv2_assist_text* assists, int n_assists, const int32_t* assist_of /* [batch] or NULL */,
                                               const int64_t* pause_after /* [batch] or NULL */,
                                               const int32_t* const* durations /* [batch] or NULL */,
                                               int32_t* out_durations /* [sum t_x] or NULL */, float** out_samples, int64_t* out_total,
                                               int64_t* out_n_samples /* [batch] or NULL */);

/* Batched, variable-length extension.  Per-utterance pointer arrays of length `batch`; every
 * utterance's result is bit-identical to its own batch-1 call.  Results land in one pinned block:
 * `*out_samples` float32 [sum n_samples[b]] back to back, `out_n_samples` int64 [batch] caller
 * allocated.  noise_* arrays may be NULL (internal generator) or per-utterance pointers. */
typedef struct sbv2_utterance {
  const float* bert;       /* [1024, t_x] */
  const int64_t* x_tst;    /* [t_x] */
  const int64_t* tones;    /* [t_x] */
  const int64_t* lang_ids; /* [t_x] */
  int64_t t_x;
  int64_t sid;
  const float* style_vec;  /* [256] */
  float sdp_ratio, length_scale, noise_scale, noise_scale_w;
  const float* noise_sdp;  /* [2, t_x] or NULL */
  const float* noise_zp;   /* [192, noise_zp_frames] or NULL */
  int64_t noise_zp_frames;
} sbv2_utterance;

int sbv2_synthesize_batch(sbv2_model* synth, const sbv2_utterance* utts, int batch, float** out_samples,
                          int64_t* out_n_samples, int32_t** out_durations /* [sum t_x] or NULL */,
                          int32_t** out_frame2ph /* [sum T_y] or NULL */);

/* ---- phoneme durations: timing queries and synthesis at given durations ---------------------------------------------
 *
 * A duration is an integer number of latent frames; one frame is `hop` samples (the product of the decoder's upsample
 * rates, "hop" in sbv2_model_describe: 512 for JP-Extra at 44.1 kHz).  Phoneme p of a sentence owns frames
 * [cum(p-1), cum(p)) and samples [cum(p-1)·hop, cum(p)·hop) of that sentence's audio.
 *
 * Given durations d[0..t_x) of a sentence replace the duration predictors' ceil(w):
 *   - the DP and SDP outputs are not used, so length_scale, sdp_ratio and noise_scale_w have no effect on that sentence;
 *     noise_scale still scales the prior sample;
 *   - T_y = max(1, sum d); all-zero durations give one frame synthesized from a zero prior mean and log-scale (frame2ph -1);
 *   - every entry must lie in [0, 1 000 000] (the clamp applied to predicted durations); outside it, or when the call
 *     would exceed 2^31 samples, or when explicit noise_zp has fewer than T_y frames, the call returns
 *     SBV2_ERR_INVALID_ARGUMENT before anything runs on the device.
 * Per sentence, durations are given or predicted (NULL entry of `durations`).  A sentence's result does not depend on
 * which of the others are given: with explicit noise it is bit-identical to its own batch-1 call, and predicted
 * sentences get the durations the plain call gives them.  When every sentence is given, the DP and SDP are not launched.
 *
 * Generator rule (internal noise): a timed call advances the model's counter-based generator exactly as the plain call
 * with the same inputs would — it reserves the SDP noise range whenever the plain call draws it, even when it launches
 * no SDP — and a timing query draws the SDP noise, advances by that range and draws no prior noise.  Hence
 *   seed(s); D = query(...);  seed(s); timed(D)   ==   seed(s); plain(...)   bit for bit.
 */

/* Timing query of the features path: runs the text encoder and the duration predictors and stops after the durations
 * (no flow, decoder or waveform).  out_durations: int32 [sum t_x], caller-allocated, utterances back to back; equal to
 * the out_durations of sbv2_synthesize_batch on the same inputs.  noise_sdp is honoured; noise_zp is not used. */
int sbv2_predict_durations_batch(sbv2_model* synth, const sbv2_utterance* utts, int batch, int32_t* out_durations);
/* sbv2_synthesize_batch at given durations: durations[i] is int32 [t_x] for utterance i or NULL (predicted); durations
 * itself may be NULL (all predicted, the plain call).  Outputs as sbv2_synthesize_batch. */
int sbv2_synthesize_batch_with_durations(sbv2_model* synth, const sbv2_utterance* utts, int batch,
                                         const int32_t* const* durations /* [batch] or NULL */, float** out_samples,
                                         int64_t* out_n_samples, int32_t** out_durations /* [sum t_x] or NULL */,
                                         int32_t** out_frame2ph /* [sum T_y] or NULL */);

/* Device-resident variant used by the benchmark's kernel-only timing: inputs already uploaded with
 * sbv2_batch_upload; runs the whole synthesizer and leaves the waveforms on the device. */
typedef struct sbv2_device_batch sbv2_device_batch;
int sbv2_batch_upload(sbv2_model* synth, const sbv2_utterance* utts, int batch, sbv2_device_batch** out);
int sbv2_batch_run(sbv2_model* synth, sbv2_device_batch* b, int64_t* total_samples /* optional */);
int sbv2_batch_download(sbv2_model* synth, sbv2_device_batch* b, float** out_samples, int64_t* out_n_samples);
void sbv2_batch_free(sbv2_device_batch* b);
/* Kernel launch counter of the model's stream since creation (for bench.py's gpu_launches). */
int64_t sbv2_model_launch_count(const sbv2_model* model);
/* CUDA stream the model launches on (cudaStream_t as void*), so callers can record events on it. */
void* sbv2_model_stream(const sbv2_model* model);

/* Region timing with CUDA events on the model's stream (off by default). Regions of a synthesizer
 * run: "text" (enc_p + duration predictors + durations), "flow" (expand + flow), "decoder". */
int sbv2_model_enable_timing(sbv2_model* model, int on);
int sbv2_model_region_ms(sbv2_model* model, const char* region, float* ms);
/* Test hook: float32 copy [rows, cols] of a named intermediate of the last run (sbv2_free). */
int sbv2_debug_fetch(sbv2_model* model, const char* name, float** out, int64_t* rows, int64_t* cols);

/* HiFi-GAN decoder alone (BASELINE config 3): z float32 [batch][192, t_y[b]] channel-major per
 * utterance, g = emb_g[sid]; output as sbv2_synthesize_batch. */
int sbv2_decode_batch(sbv2_model* synth, const float* const* z, const int64_t* t_y, const int64_t* sid,
                      int batch, float** out_samples, int64_t* out_n_samples);

/* ---- sbv2file::parse_sbv2file  (crates/sbv2_core/src/sbv2file.rs:15-37) ---------------------- */

/* zstd -> tar -> ("style_vectors.json", "model.onnx").  Both outputs are library-allocated. */
int sbv2_parse_sbv2file(const void* sbv2_bytes, size_t n, void** style_json, size_t* style_n,
                        void** onnx, size_t* onnx_n);

/* ---- style::load_style / get_style_vector  (crates/sbv2_core/src/style.rs:11-28) ------------- */

/* JSON {"shape":[n,d],"data":[[...]]} -> float32 [n*d] library-allocated. */
int sbv2_load_style(const void* json_bytes, size_t n, float** out, int64_t* rows, int64_t* cols);
/* .aivmx: base64(.npy float32 2-D, C or Fortran order) -> float32 [rows*cols] row-major
 * (crates/sbv2_core/src/tts.rs:95-108). */
int sbv2_load_style_npy_base64(const char* b64, size_t n, float** out, int64_t* rows, int64_t* cols);
/* mean + (v - mean) * weight with mean = row 0; out float32 [cols] caller-allocated. */
int sbv2_get_style_vector(const float* style_vectors, int64_t rows, int64_t cols, int32_t style_id,
                          float weight, float* out);

/* ---- tts_util::array_to_vec  (crates/sbv2_core/src/tts_util.rs:163-180) ---------------------- */

/* float32 mono 44.1 kHz WAV (WAVE_FORMAT_EXTENSIBLE/IEEE float, as hound writes it). */
int sbv2_wav_from_f32(const float* samples, int64_t n, void** wav_bytes, size_t* wav_n);
/* Optional (SURVEY.md 8f row 3; the reference only writes float): 16-bit PCM mono 44.1 kHz WAV, 44-byte header; samples
 * clamped to [-1, 1], scaled by 32767, rounded to nearest; NaN -> 0. */
int sbv2_wav_pcm16_from_f32(const float* samples, int64_t n, void** wav_bytes, size_t* wav_n);

/* ---- TTSModelHolder  (crates/sbv2_core/src/tts.rs:40-349) ------------------------------------ */

typedef struct sbv2_holder sbv2_holder;
/* max_loaded_models < 0 means None.  tokenizer bytes are kept but not interpreted (the text
 * frontend stays in the caller; see INTEGRATION.md). */
int sbv2_holder_new(const void* bert_onnx, size_t bert_n, const void* tokenizer, size_t tok_n,
                    int64_t max_loaded_models, int device_ordinal, sbv2_holder** out);
void sbv2_holder_free(sbv2_holder* h);
int sbv2_holder_load_sbv2file(sbv2_holder* h, const char* ident, const void* bytes, size_t n);
int sbv2_holder_load(sbv2_holder* h, const char* ident, const void* style_json, size_t style_n,
                     const void* onnx, size_t onnx_n);
int sbv2_holder_load_aivmx(sbv2_holder* h, const char* ident, const void* bytes, size_t n);
int sbv2_holder_unload(sbv2_holder* h, const char* ident, int* found);
/* '\n'-separated, NUL-terminated list of identifiers, library-allocated (sbv2_free). */
int sbv2_holder_models(const sbv2_holder* h, char** out);
/* how many models currently hold device weights (vits2.is_some()). */
int sbv2_holder_loaded_count(const sbv2_holder* h, int* out);
/* hidden size of the holder's DeBERTa = rows of every `bert` feature matrix it takes or returns (1024 for deberta-v2-large). */
int sbv2_holder_bert_hidden_size(const sbv2_holder* h, int* out);
int sbv2_holder_get_style_vector(sbv2_holder* h, const char* ident, int32_t style_id, float weight,
                                 float* out /* [256] */);
/* parse_text's device half: BERT over the token ids, then the word2ph row repeat + transpose
 * (tts_util.rs:120-154).  out: float32 [hidden, sum(word2ph)] library-allocated. */
int sbv2_holder_bert_features(sbv2_holder* h, const int64_t* token_ids, const int64_t* attention_mask,
                              int64_t t_tok, const int32_t* word2ph, float** out, int64_t* t_x);
/* The same with an assist text (NULL = none): one DeBERTa batch [sentence, assist] (the layout of
 * sbv2_synthesize_from_tokens_assist), then the blend on the host with the numerics stated there. */
int sbv2_holder_bert_features_assist(sbv2_holder* h, const int64_t* token_ids, const int64_t* attention_mask, int64_t t_tok,
                                     const int32_t* word2ph, const sbv2_assist_text* assist, float** out, int64_t* t_x);
/* easy_synthesize from already-parsed sentences (one entry per non-empty '\n'-separated line):
 * find_and_load_model, get_style_vector, per-sentence synthesize, 22050 zero samples between
 * sentences (`total_lines` is the number of lines of the original text incl. empty ones and
 * `line_index[i]` the position of sentence i, so the trailing-silence rule of tts.rs:318-320 is
 * reproduced), then WAV bytes. */
typedef struct sbv2_sentence {
  const float* bert;       /* [hidden, t_x], hidden = sbv2_holder_bert_hidden_size (1024 for deberta-v2-large) */
  const int64_t* phones;   /* [t_x] */
  const int64_t* tones;    /* [t_x] */
  const int64_t* lang_ids; /* [t_x] */
  int64_t t_x;
  int64_t line_index;
} sbv2_sentence;
int sbv2_holder_easy_synthesize(sbv2_holder* h, const char* ident, const sbv2_sentence* sentences,
                                int n_sentences, int64_t total_lines, int32_t style_id, int64_t speaker_id,
                                float sdp_ratio, float length_scale, float style_weight,
                                void** wav_bytes, size_t* wav_n);

/* The same with bert::predict folded in (SURVEY.md §8f rows 1-2): sentences carry the tokenizer's output and word2ph instead
 * of BERT features.  DeBERTa and the synthesizer each run once over all sentences of the request (features stay on the
 * device), the 22 050-sample pauses are written on the device, the WAV is one header + one copy. */
typedef struct sbv2_token_sentence {
  const int64_t* token_ids;      /* [t_tok] */
  const int64_t* attention_mask; /* [t_tok] */
  const int32_t* word2ph;        /* [t_tok], sum == t_x */
  int64_t t_tok;
  const int64_t* phones;         /* [t_x] */
  const int64_t* tones;          /* [t_x] */
  const int64_t* lang_ids;       /* [t_x] */
  int64_t t_x;
  int64_t line_index;
} sbv2_token_sentence;
int sbv2_holder_easy_synthesize_tokens(sbv2_holder* h, const char* ident, const sbv2_token_sentence* sentences,
                                       int n_sentences, int64_t total_lines, int32_t style_id, int64_t speaker_id,
                                       float sdp_ratio, float length_scale, float style_weight,
                                       void** wav_bytes, size_t* wav_n);
/* The same with an assist text (NULL = none) that applies to every line, as the reference's TTSModel.infer passes it to
 * each line of a request. */
int sbv2_holder_easy_synthesize_tokens_assist(sbv2_holder* h, const char* ident, const sbv2_token_sentence* sentences,
                                              int n_sentences, int64_t total_lines, int32_t style_id, int64_t speaker_id,
                                              float sdp_ratio, float length_scale, float style_weight,
                                              const sbv2_assist_text* assist, void** wav_bytes, size_t* wav_n);
/* Timing of a request ("audio query"): the durations easy_synthesize_tokens_timed with durations = NULL would use, int32
 * [sum t_x] caller-allocated, sentences concatenated in sentences[] order (durations contract: see
 * sbv2_predict_durations_batch).  Runs DeBERTa, the text encoder and the duration predictors only.  Each line_index may
 * appear once. */
int sbv2_holder_predict_durations_tokens(sbv2_holder* h, const char* ident, const sbv2_token_sentence* sentences, int n_sentences,
                                         int64_t total_lines, int32_t style_id, int64_t speaker_id, float sdp_ratio,
                                         float length_scale, float style_weight, const sbv2_assist_text* assist,
                                         int32_t* out_durations);
/* sbv2_holder_easy_synthesize_tokens_assist at given durations and with the timing of the result.
 *   durations: [n_sentences] in sentences[] order, each int32 [t_x] or NULL (predicted); NULL = all predicted, which
 *     returns the same WAV bytes as sbv2_holder_easy_synthesize_tokens_assist.
 *   out_durations (optional): int32 [sum t_x], the durations used, in sentences[] order.
 *   out_phoneme_start (optional): int64 [sum t_x], in sentences[] order; entry p is the index, in the WAV's sample data,
 *     of phoneme p's first sample.  It accounts for the earlier lines and the 22 050-sample pauses; the phoneme ends at
 *     start + d·hop.  Character or token spans follow from these and word2ph.
 * Each line_index may appear once. */
int sbv2_holder_easy_synthesize_tokens_timed(sbv2_holder* h, const char* ident, const sbv2_token_sentence* sentences, int n_sentences,
                                             int64_t total_lines, int32_t style_id, int64_t speaker_id, float sdp_ratio,
                                             float length_scale, float style_weight, const sbv2_assist_text* assist,
                                             const int32_t* const* durations /* [n_sentences] or NULL */,
                                             int32_t* out_durations /* [sum t_x] or NULL */,
                                             int64_t* out_phoneme_start /* [sum t_x] or NULL */, void** wav_bytes, size_t* wav_n);

#ifdef __cplusplus
}
#endif
#endif /* SBV2_B200_H_ */
