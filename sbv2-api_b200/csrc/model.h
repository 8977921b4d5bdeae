// Device-side model objects behind the C ABI.  One sbv2_model = one ort::Session of the reference.
#pragma once
#include <cuda_runtime.h>

#include "common.h"
#include "kernels.h"
#include "onnx_reader.h"

namespace sbv2 {

// Growable device buffer. Growth synchronises the owning stream first.
struct DBuf {
  void* p = nullptr;
  size_t cap = 0;
  uint64_t gen = 0;  // bumped on every (re)allocation: "was this buffer cleared?" must not rely on pointer identity
  cudaStream_t stream = nullptr;
  DBuf() = default;
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  ~DBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  void ensure(size_t bytes);
  template <class T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  ~PinnedBuf() {
    if (p) cudaFreeHost(p);
  }
  void ensure(size_t bytes);
  template <class T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

// Registry of every allocation made through sbv2_* out-pointers so sbv2_free can tell pinned from malloc.
void* alloc_out(size_t bytes, bool pinned);
void free_out(void* p);

struct DebugView {
  const void* ptr;
  int64_t rows, cols;
  int elt;  // 4 = float32, -4 = int32
};

}  // namespace sbv2

// The opaque C type. Concrete models derive from it.
struct sbv2_model {
  int device = 0;
  bool is_bert = false;
  cudaStream_t stream = nullptr;
  int64_t launches = 0;
  std::map<std::string, std::string> metadata;
  std::string describe_json;
  std::map<std::string, sbv2::DebugView> debug;
  std::vector<void*> owned_device;  // weights
  // optional region timing (CUDA events on `stream`), see sbv2_model_enable_timing
  bool timing = false;
  std::map<std::string, std::pair<cudaEvent_t, cudaEvent_t>> regions;
  void region_begin(const std::string& name);
  void region_end(const std::string& name);
  float region_ms(const std::string& name);

  virtual ~sbv2_model();
  bool pdl = true;  // programmatic dependent launch of the tensor-core kernels (SBV2_B200_PDL=0, read at model creation, disables)
  sbv2::LaunchCtx ctx() { return sbv2::LaunchCtx{stream, &launches, pdl}; }
  void bind_device() const;
  // Waits for the model's stream.  `yield` = true parks the host thread on a blocking-sync event instead of spinning in
  // cudaStreamSynchronize: the two long waits of a batched synthesize call (T_y read-back, final download) would otherwise
  // burn one host core per in-flight call — with 3 replicas on each of 8 GPUs that is more spinning threads than the
  // box has cores, and the end-to-end scaling pays for it.  Short (batch-1) calls keep spinning: waking up costs ~50 us.
  void wait_stream(bool yield);
  cudaEvent_t wait_event = nullptr;
  // uploads host data, tracked for release at destroy
  void* upload_bytes(const void* host, size_t bytes);
  float* upload_f32(const std::vector<float>& v) { return static_cast<float*>(upload_bytes(v.data(), v.size() * 4)); }
};

struct sbv2_device_batch;

namespace sbv2 {

sbv2_model* create_synth_model(const OnnxModel& m, int device);
sbv2_model* create_bert_model(const OnnxModel& m, int device);

// synthesizer entry points (synth_model.cu)
// BERT features of one utterance that are already on the synthesizer's device (sbv2_synthesize_from_tokens)
struct DeviceBert {
  const float* rows = nullptr;     // [n_rows, hidden] fp32 on the device
  int64_t n_rows = 0;
  int hidden = 0;
  const int64_t* ph2tok = nullptr;  // host, [sum t_x]: BERT row (index into `rows`) of each phoneme of the batch
  cudaEvent_t ready = nullptr;      // recorded on the producer's stream after the rows (and `means`) were written
  // assist texts (sbv2_synthesize_from_tokens_assist); n_slots == 0: plain gather
  int n_slots = 0;
  const float* means = nullptr;     // device [n_slots, hidden]: mean DeBERTa row of each assist
  const int32_t* slot = nullptr;    // host [sum t_x]: assist slot of each phoneme, -1 = the plain row
  const float* coef = nullptr;      // host [n_slots][2]: (c_row, c_mean) = ((float)(1 - (double)w), w)
};
// durations (optional, [batch]): caller-given integer durations of utterance i ([t_x], each in [0, 1e6]) or null for the
// predicted ones; they replace the DP / SDP outputs of that utterance (include/sbv2_b200.h, sbv2_synthesize_batch_with_durations)
sbv2_device_batch* synth_upload(sbv2_model* m, const sbv2_utterance* utts, int batch, const DeviceBert* dev_bert = nullptr,
                                const int32_t* const* durations = nullptr);
// Host checks of given durations (synth_upload runs them too): each entry in [0, 1e6], the given utterances' samples
// < 2^31, explicit noise_zp long enough.  Callers that launch work before synth_upload call it first.
void synth_check_durations(sbv2_model* m, const sbv2_utterance* utts, int batch, const int32_t* const* durations);
void synth_run(sbv2_model* m, sbv2_device_batch* b);
// Timing query: synth_run on a batch marked here stops after the durations kernel (no expand, flow, decoder or waveform
// buffer) and synth_query_durations copies the durations [sum t_x] into caller memory.
void synth_set_query(sbv2_device_batch* b);
void synth_query_durations(sbv2_model* m, sbv2_device_batch* b, int32_t* out);
void synth_download(sbv2_model* m, sbv2_device_batch* b, float** out_samples, int64_t* out_n, int32_t** out_dur,
                    int32_t** out_f2p);
int64_t synth_batch_phonemes(const sbv2_device_batch* b);                     // sum t_x
int64_t synth_total_samples(sbv2_model* m, const sbv2_device_batch* b);
int64_t synth_wave_total(const sbv2_device_batch* b);                        // samples of the output buffer incl. pauses
void synth_set_pauses(sbv2_device_batch* b, const int64_t* pause_after);     // before synth_run: zeros after each utterance
bool synth_borrows_host(const sbv2_device_batch* b);                         // uploads read caller memory in place
void synth_batch_ty(const sbv2_device_batch* b, int64_t* ty);
void synth_batch_free(sbv2_device_batch* b);
void synth_set_seed(sbv2_model* m, uint64_t seed);
void synth_decode(sbv2_model* m, const float* const* z, const int64_t* t_y, const int64_t* sid, int batch,
                  float** out_samples, int64_t* out_n);

// bert entry points (bert_model.cu)
void bert_predict(sbv2_model* m, const int64_t* ids, const int64_t* mask, int batch, int64_t s, float* out);
// features stay on the device ([batch, s, hidden], zero rows where the mask is 0); null when no token is valid
const float* bert_forward_device(sbv2_model* m, const int64_t* ids, const int64_t* mask, int batch, int64_t s);
int bert_hidden(const sbv2_model* m);
// launch_token_mean over rows [row0, row0 + n) of the last bert_forward_device output, on the model's stream; the result
// [n, hidden] lives in a model-owned buffer that stays valid until the model's next call
const float* bert_token_mean(sbv2_model* m, int row0, int n);

}  // namespace sbv2
