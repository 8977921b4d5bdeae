// Launch wrappers of the hand-written kernels.  All activations of the fp32 ("exact") path are
// time-major: a packed [rows, C] float32 matrix holding the utterances of a batch back to back,
// rows of utterance b being [seg_start[b], seg_start[b]+seg_len[b]).  Convolutions zero-pad at the
// boundaries of each utterance's own segment, so a batched run is bit-identical to batch-1 runs.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "common.h"

namespace sbv2 {

struct Segs {             // device pointers
  const int* start = nullptr;  // [n] first row of each utterance
  const int* len = nullptr;    // [n] rows of each utterance
  int n = 0;
  int max_len = 0;  // host-side max over len (grid sizing)
  // rows are per-utterance conditioning vectors (one segment of B rows): k = 1 convs over them run utt_linear_kernel
  // whatever B is, so an utterance's vectors do not depend on the batch it is in
  bool vectors = false;
};

enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_LRELU = 2 /*0.1*/, ACT_GELU = 3, ACT_LRELU01 = 4 /*0.01*/, ACT_TANH = 5 };
enum AccumMode { ACC_NONE = 0, ACC_SET = 1, ACC_ADD = 2, ACC_ADD_SCALE = 3 };

struct LaunchCtx {
  cudaStream_t stream = nullptr;
  int64_t* launches = nullptr;  // host counter
  bool pdl = false;             // launch the tensor-core kernels with programmatic stream serialization
  void count(int n = 1) const {
    if (launches) *launches += n;
  }
};

// Programmatic dependent launch (PDL): the grid may become resident while its predecessor in the stream drains, so its
// prologue (barrier init, TMEM allocation, launch latency) overlaps the predecessor's tail.  The kernel MUST execute
// griddepcontrol.wait (pdl_wait() in the kernels) before it reads or writes anything another kernel touches.
// Measured on the bench workload: -0.65 ms of 29 on a single stream (batch-1 latency 5.3 -> 4.9 ms) and neutral for two
// replicas per GPU once the mbarrier waits sleep instead of polling; on by default, SBV2_B200_PDL=0 disables it.
#ifdef __CUDACC__
// cluster > 1 launches thread-block clusters of that many CTAs along x (grid.x must be a multiple of it)
template <class... KArgs, class... Args>
inline void launch_pdl_cluster(bool pdl, int cluster, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                               Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (pdl) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = unsigned(cluster);
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = unsigned(n);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
  if (e != cudaSuccess) fail(SBV2_ERR_CUDA, std::string("cudaLaunchKernelEx: ") + cudaGetErrorString(e));
}
template <class... KArgs, class... Args>
inline void launch_pdl(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  launch_pdl_cluster(pdl, 1, kernel, grid, block, smem, stream, static_cast<Args&&>(args)...);
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

// out[orow(t), co] = epi( bias[co] + bias_utt[b, co] + sum_{m<taps} sum_ci W[m][ci][co] * act_in(in[t + off + m*dil, ci]) )
//   orow(t) = seg_out_start[b] + t*out_row_mul + out_row_off;   t in [0, seg.len[b])
//   epi(v)  = act_out(v + residual[orow]) ; optional accumulate into accum_out.
struct ConvArgs {
  const float* in = nullptr;
  int in_ld = 0;            // floats between consecutive rows of `in`
  const float* w = nullptr;  // [taps][Cin][Cout]
  const float* bias = nullptr;
  const float* bias_utt = nullptr;  // [n_utt][Cout] or null
  float* out = nullptr;
  int out_ld = 0;
  const float* residual = nullptr;  // same indexing as out
  float* accum_out = nullptr;       // same indexing as out
  int accum_mode = ACC_NONE;
  float accum_div = 1.f;  // ACC_ADD_SCALE: accum = (accum + v) / accum_div
  int cin = 0, cout = 0, taps = 1, dil = 1, off = 0;
  int act_in = ACT_NONE, act_out = ACT_NONE;
  int out_row_mul = 1, out_row_off = 0;
  const int* seg_out_start = nullptr;  // null: same as seg.start (times out_row_mul is NOT applied to it)
  Segs seg;
};
void launch_conv(const LaunchCtx& ctx, const ConvArgs& a);

// [C, T_b] channel-major blocks (utterance b at src + src_off[b]) -> packed [rows, C]
void launch_cm_to_rm(const LaunchCtx& ctx, const float* src, const int64_t* src_off, const int* src_ld, float* dst, int C, const Segs& seg);
// packed [rows, C] -> per-utterance [C, T_b] blocks
void launch_rm_to_cm(const LaunchCtx& ctx, const float* src, float* dst, const int64_t* dst_off, int C, const Segs& seg);

// h = (emb[x] + tone_emb[tone] + lang_emb[lang] + h + style_emb[b]) * sqrt(C)
void launch_embed_combine(const LaunchCtx& ctx, float* h, const int* x, const int* tone, const int* lang, const float* emb,
                          const float* tone_emb, const float* lang_emb, const float* style_emb, int C, int n_vocab,
                          int n_tones, int n_lang, const Segs& seg);
// gather rows: out[b, :] = table[idx[b], :]
void launch_gather_rows(const LaunchCtx& ctx, float* out, const float* table, const int64_t* idx, int n, int C, int n_rows);
// x[row, c] (+)= v[b, c]; out may alias x.
void launch_add_utt_vec(const LaunchCtx& ctx, float* out, const float* x, const float* v, int C, int v_ld, const Segs& seg);

// out = res + act(LN(a + addin)) over channels (gamma/beta, eps); res/addin optional.
void launch_layernorm(const LaunchCtx& ctx, float* out, const float* a, const float* addin, const float* res,
                      const float* gamma, const float* beta, float eps, int act, int C, int rows);

// window-relative multi-head attention (enc_p / transformer flow). qkv: [rows, 3*H*D].
void launch_rel_attention(const LaunchCtx& ctx, float* out, const float* qkv, const float* rel_k, const float* rel_v,
                          int heads, int head_dim, int window, const Segs& seg);

// depthwise dilated conv k=3 (DDSConv.convs_sep): w [C][3]
void launch_dwconv3(const LaunchCtx& ctx, float* out, const float* in, const float* w, const float* bias, int C, int dil,
                    const Segs& seg);

// SDP pieces on z [rows, 2]
void launch_sdp_init(const LaunchCtx& ctx, float* z, const float* noise_rm /*[rows,2]*/, const float* noise_scale_w_utt,
                     const Segs& seg);
void launch_sdp_flip(const LaunchCtx& ctx, float* z, int rows);
// h[t,c] = w[c]*z[t,0] + b[c] + g[t,c]   (ConvFlow.pre followed by DDSConv's "x + g")
void launch_convflow_pre(const LaunchCtx& ctx, float* h, const float* z, const float* w, const float* b, const float* g,
                         int C, int rows);
// z[t,1] <- RQS^{-1}(z[t,1]; proj[t, 0:29]) with linear tails; proj rows have ld floats
void launch_convflow_spline(const LaunchCtx& ctx, float* z, const float* proj, int ld, int num_bins, float tail_bound,
                            float inv_sqrt_filter, int rows);
void launch_sdp_affine(const LaunchCtx& ctx, float* z, const float* m, const float* logs, int rows);

// durations: logw = sdp*ratio + dp*(1-ratio); w = exp(logw)*length_scale; d = ceil(w);
// cum = inclusive scan per utterance; ylen[b] = min(max(1, sum d), INT_MAX) (the sum is formed in 64 bits)
void launch_durations(const LaunchCtx& ctx, const float* logw_dp, const float* z_sdp /*[rows,2] or null*/,
                      const float* sdp_ratio_utt, const float* length_scale_utt, float* w_out, int* dur, int* cum,
                      int* ylen, const Segs& seg);
// frame2ph + gather + prior sample: z_p[j,c] = m_p[i,c] + eps[j,c]*exp(logs_p[i,c])*noise_scale[b]
void launch_expand(const LaunchCtx& ctx, float* z_p, int* frame2ph, const float* stats /*[rows_x, 2C]: m_p | logs_p*/,
                   const int* cum, const float* eps_rm /*[rows_y, C]*/, const float* noise_scale_utt, int C,
                   const Segs& xseg, const Segs& yseg);
// Philox-based N(0,1) fill (used when the caller does not inject noise)
void launch_randn(const LaunchCtx& ctx, float* out, int64_t n, uint64_t seed, uint64_t offset);

// flow helpers on z [rows, C]
void launch_flip_channels(const LaunchCtx& ctx, float* out, const float* in, int C, int64_t rows);
// z[:, C/2:] -= m   (m: [rows, C/2])
void launch_coupling_sub(const LaunchCtx& ctx, float* z, const float* m, int C, int64_t rows);
// WN gate: acts = tanh(a[:, :H] + g[b, goff:goff+H]) * sigmoid(a[:, H:] + g[b, goff+H:goff+2H])
void launch_wn_gate(const LaunchCtx& ctx, float* acts, const float* a, const float* g_utt, int g_ld, int goff, int H,
                    const Segs& seg);
// WN res/skip update: x += rs[:, :H]; skip (+)= rs[:, H:]  (last layer: skip += rs[:, :H])
void launch_wn_res_skip(const LaunchCtx& ctx, float* x, float* skip, const float* rs, int H, int last, int first,
                        int64_t rows);

// decoder post: out[t] = tanh(sum_j sum_c w[c][j] * lrelu_0.01(x[t+j-3, c])), x [rows, C] fp32
void launch_dec_post(const LaunchCtx& ctx, float* out, const float* x, const float* w, int C, int k, const Segs& seg);

}  // namespace sbv2

// ---- transformer-flow glue around the tensor-core kernels (flow_kernels.cu) ----------------------
// Planar buffers: fp16 [C/8][rows_tot][8] or fp32 with the same indexing; utterance b occupies planar
// rows [pstart[b], pstart[b]+len[b]) and packed fp32 rows [start[b], start[b]+len[b]).
namespace sbv2 {
struct PlanarSegs {
  const int* start = nullptr;   // packed fp32 rows
  const int* pstart = nullptr;  // planar rows
  const int* len = nullptr;
  const int* order = nullptr;   // optional: utterance processed by grid slot z (longest first); null = identity
  int n = 0, max_len = 0;
  long long plane_stride = 0;   // elements between planes (= rows_tot * 8)
};
// h_out[row, :] = (src32 ? src32(planar fp32) : h_in[row, :]) + (vec ? vec[b, :] : 0); hp = fp16(h_out) planar
void launch_flow_mix(const LaunchCtx& ctx, float* h_out, __half* hp, const float* h_in, const float* src32, const float* vec,
                     int vec_ld, int C, const PlanarSegs& s);
// h = LN(h + y32) * gamma + beta (in place, fp32 packed); hp = fp16(h) planar
void launch_ln_planar(const LaunchCtx& ctx, float* h, __half* hp, const float* y32, const float* gamma, const float* beta, float eps,
                      int C, const PlanarSegs& s);
// window-relative attention on planar fp16 q|k|v (3*H*D channels) -> planar fp16 ctx (H*D channels)
void launch_rel_attention_planar(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const float* rel_k, const float* rel_v,
                                 int heads, int head_dim, int window, const PlanarSegs& s);
// same on tcgen05 tensor cores (head_dim 96, window 4); rel_k_p / rel_v_p: fp16 [D/8][16][8] packings
void launch_flow_attention_tc(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const __half* rel_k_p, const __half* rel_v_p,
                              int heads, int head_dim, int window, const PlanarSegs& s, long long* trace = nullptr);
// host: fp32 relative table [2*window+1][head_dim] -> the fp16 [D/8][16][8] packing launch_flow_attention_tc reads
std::vector<__half> pack_flow_rel_table(const float* table, int window, int head_dim);
// z[row, C/2:] -= m32 (planar fp32, C/2 channels)
void launch_coupling_sub_planar(const LaunchCtx& ctx, float* z, const float* m32, int C, const PlanarSegs& s);
}  // namespace sbv2

// ---- DeBERTa glue (bert_kernels.cu) ----------------------------------------------------------------
namespace sbv2 {
// h = LN(h + y32) * gamma + beta for any C that is a multiple of 8 and <= 1024; y32 planar fp32 or null;
// also writes the planar fp16 copy hp (and hp2 if not null).
void launch_ln_planar_wide(const LaunchCtx& ctx, float* h, __half* hp, __half* hp2, const float* y32, const float* gamma,
                           const float* beta, float eps, int C, const PlanarSegs& s);
// h[row, :] = table[ids[row], :]
void launch_embed_rows(const LaunchCtx& ctx, float* h, const float* table, const int* ids, int C, int n_vocab, int64_t rows);
// Longest sequence the DeBERTa forward accepts (tokens); longer inputs return SBV2_ERR_INVALID_ARGUMENT.
constexpr int kMaxBertTokens = 32768;
// Relative-position bucket table of HF make_log_bucket_position(delta, span, 2 * span): entry delta + R holds
// clamp(bucket(delta) + span, 0, 2*span-1) for delta = -R..R, R (*max_rel) being the saturation bound: every |delta| >= R reads
// the same row as +-R (span 256: R = 512, idx(-512) = 0, idx(-511) = 1).  So kernels clamp delta to +-R and index the table.
// Checked for every |delta| < kMaxBertTokens.
std::vector<int> bert_bucket_table(int span, int* max_rel);
// DeBERTa-v2 disentangled attention (c2p + p2c, shared keys) on planar fp16 q|k|v -> planar fp16 ctx.
// pos_k/pos_q: fp32 [2*span, heads*64] projections of the normalised relative embeddings; bucket_idx / max_rel: bert_bucket_table.
void launch_deberta_attention(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const float* pos_k_t, const float* pos_q_t,
                              int n_pos, const int* bucket_idx, int max_rel, int heads, int head_dim, const PlanarSegs& s);
// "exact" mode: the same kernel on fp32 row-major q|k|v [rows, 3*heads*64] -> fp32 row-major context [rows, heads*64]
// ctx_split != null: the context goes out as the split-planar operand [h0 | h1 | h0] (scaled by split_scale) instead
void launch_deberta_attention_f32(const LaunchCtx& ctx, float* ctx_out, __half* ctx_split, float split_scale, const float* qkv,
                                  const float* pos_k_t, const float* pos_q_t, int n_pos, const int* bucket_idx, int max_rel, int heads,
                                  int head_dim, const PlanarSegs& s);
// out = LN(a + addin) (fp32 row-major [rows, C], out optional) and the split-planar operand of the consuming GEMM in one pass
// (any C that is a multiple of 8 and <= 1024)
bool ln_split_supported(int C);
void launch_ln_split(const LaunchCtx& ctx, float* out, __half* split, float split_scale, const float* a, const float* addin,
                     const float* gamma, const float* beta, float eps, int C, const PlanarSegs& s);
// tensor-core version for sequences of at most 128 tokens (bert_attention_tc.cu); pos_*_p: fp16 [heads][D/8][n_pos][8]
bool deberta_attention_tc_supported(int head_dim, int span, int max_len);
void launch_deberta_attention_tc(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const __half* pos_k_p, const __half* pos_q_p,
                                 int n_pos, int span, int heads, const PlanarSegs& s);
// exact numerics (two-term fp16 splits of every operand), <= 128 tokens; see bert_attention_tc.cu
void launch_deberta_attention_tc_exact(const LaunchCtx& ctx, __half* ctx_s, long long ctx_blk, const __half* qkv_s, long long qkv_blk,
                                       const __half* pos_k_s, const __half* pos_q_s, int n_pos, int span, int heads, float sc,
                                       const PlanarSegs& s);
// Any length: 128-query tiles x 128-key tiles with an online softmax; position windows gathered through bucket_idx.
// far_pairs: a tile pair whose relative positions all lie at or beyond +-max_rel (|qt - kt| >= 5 for span 256) reads one
// position row, and takes the reduced path (16 gathered rows, N = 16 bias products, no skewed copies), bit-identical to
// the generic path; false forces the generic path (the debug hook compares the two).
bool deberta_attention_tc_multi_supported(int head_dim);
void launch_deberta_attention_tc_exact_multi(const LaunchCtx& ctx, __half* ctx_s, long long ctx_blk, const __half* qkv_s, long long qkv_blk,
                                             const __half* pos_k_s, const __half* pos_q_s, int n_pos, const int* bucket_idx, int max_rel,
                                             int heads, float sc, bool far_pairs, const PlanarSegs& s);
void launch_deberta_attention_tc_multi(const LaunchCtx& ctx, __half* ctx_out, const __half* qkv, const __half* pos_k_p, const __half* pos_q_p,
                                       int n_pos, const int* bucket_idx, int max_rel, int heads, bool far_pairs, const PlanarSegs& s);
// out[b, t, :] = h[start[b] + t, :] for t < len[b], zeros elsewhere (out: [n, S, C] fp32)
void launch_scatter_rows(const LaunchCtx& ctx, float* out, const float* h, int C, int S, const PlanarSegs& s);
}  // namespace sbv2
