// Tensor-core HiFi-GAN decoder plan (conv_pre, 5 x [polyphase ConvTranspose + 3 ResBlock1 (MRF)],
// conv_post) on top of the tcgen05 conv kernel of umma_conv.cu.  Every stored activation is the
// post-LeakyReLU value in planar fp16; the residual x is recovered exactly-invertibly from it
// (x = y >= 0 ? y : 10 y), the MRF mean is accumulated in fp32.
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "kernels.h"
#include "model.h"
#include "umma_conv.h"

namespace sbv2 {
extern long long* g_pair_trace;
namespace {

// decoder post: out[t] = tanh(sum_j sum_c w[c][j] * x[t+j-pad][c]); x planar fp16 already activated (lrelu 0.01).
// A block stages its 256 + k - 1 input rows in shared memory once (coalesced 16-byte loads); every thread then reads its
// k taps from there — the direct version issued k * C/8 global loads per output and was load/store-unit bound.
constexpr int POST_T = 256;
__global__ void __launch_bounds__(POST_T) post_planar_kernel(float* wave, const __half* x, long long plane_stride, const float* w, int C,
                                                             int k, const int* pstart, const int* wstart, const int* len) {
  extern __shared__ __align__(16) uint8_t post_smem[];
  const int npl = C / 8, pad = (k - 1) / 2, rows = POST_T + k - 1;
  float* ws = reinterpret_cast<float*>(post_smem);                               // [k][C]
  uint4* xs = reinterpret_cast<uint4*>(post_smem + (((size_t)k * C * 4 + 15) & ~size_t(15)));  // [npl][rows]
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * POST_T;
  if (t0 >= len[b]) return;
  for (int i = threadIdx.x; i < C * k; i += POST_T) {
    int c = i / k, j = i % k;
    ws[j * C + c] = w[i];
  }
  const long long r0 = (long long)pstart[b] + t0 - pad;  // gap rows are zero: no bounds test needed
  for (int i = threadIdx.x; i < npl * rows; i += POST_T) {
    const int pl = i / rows, r = i - pl * rows;
    xs[pl * rows + r] = *reinterpret_cast<const uint4*>(x + (size_t)pl * plane_stride + (r0 + r) * 8);
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= len[b]) return;
  float acc = 0.f;
  for (int j = 0; j < k; ++j) {
    for (int pl = 0; pl < npl; ++pl) {
      const uint4 q = xs[pl * rows + threadIdx.x + j];
      const __half2* qh = reinterpret_cast<const __half2*>(&q);
      const float* wj = ws + j * C + pl * 8;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 y = __half22float2(qh[e]);
        acc = fmaf(wj[2 * e], y.x, acc);
        acc = fmaf(wj[2 * e + 1], y.y, acc);
      }
    }
  }
  wave[(size_t)wstart[b] + t] = tanhf(acc);
}

// The JP-Extra shape (16 channels, 7 taps) with the weights in the kernel's constant parameter bank: the generic kernel
// spends one shared-memory load per FMA on the weights, here they are FFMA constant operands.
template <int C, int K>
struct PostWeights {
  float w[K][C];  // [tap][channel]
};
template <int C, int K>
__global__ void __launch_bounds__(POST_T) post_planar_const_kernel(float* wave, const __half* x, long long plane_stride,
                                                                   const __grid_constant__ PostWeights<C, K> pw, const int* pstart,
                                                                   const int* wstart, const int* len) {
  constexpr int NPL = C / 8, PAD = (K - 1) / 2, ROWS = POST_T + K - 1;
  __shared__ uint4 xs[NPL * ROWS];
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * POST_T;
  if (t0 >= len[b]) return;
  const long long r0 = (long long)pstart[b] + t0 - PAD;
  for (int i = threadIdx.x; i < NPL * ROWS; i += POST_T) {
    const int pl = i / ROWS, r = i - pl * ROWS;
    xs[pl * ROWS + r] = *reinterpret_cast<const uint4*>(x + (size_t)pl * plane_stride + (r0 + r) * 8);
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= len[b]) return;
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < K; ++j) {
#pragma unroll
    for (int pl = 0; pl < NPL; ++pl) {
      const uint4 q = xs[pl * ROWS + threadIdx.x + j];
      const __half2* qh = reinterpret_cast<const __half2*>(&q);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 y = __half22float2(qh[e]);
        acc = fmaf(pw.w[j][pl * 8 + 2 * e], y.x, acc);
        acc = fmaf(pw.w[j][pl * 8 + 2 * e + 1], y.y, acc);
      }
    }
  }
  wave[(size_t)wstart[b] + t] = tanhf(acc);
}

}  // namespace

void launch_dec_post_planar(const LaunchCtx& ctx, float* wave, const __half* x, const Geom& g, const int* d_wstart, int n_utt,
                            const float* d_w, const std::vector<float>& w_host, int C, int k, bool force_generic) {
  dim3 grid((g.max_len + POST_T - 1) / POST_T, n_utt);
  if (C == 16 && k == 7 && !force_generic) {
    PostWeights<16, 7> pw;
    for (int c = 0; c < 16; ++c)
      for (int j = 0; j < 7; ++j) pw.w[j][c] = w_host[size_t(c) * 7 + j];
    post_planar_const_kernel<16, 7><<<grid, POST_T, 0, ctx.stream>>>(wave, x, g.rows_tot * 8, pw, g.d_pstart, d_wstart, g.d_len);
  } else {
    const size_t smem = ((sizeof(float) * C * k + 15) & ~size_t(15)) + size_t(C / 8) * (POST_T + k - 1) * 16;
    post_planar_kernel<<<grid, POST_T, smem, ctx.stream>>>(wave, x, g.rows_tot * 8, d_w, C, k, g.d_pstart, d_wstart, g.d_len);
  }
  CUDA_CHECK(cudaGetLastError());
  ctx.count();
}

// ---- decoder plan -----------------------------------------------------------------------------------------
struct UmmaDecoder {
  int gin = 0, cin0 = 0, c0 = 0, n_stages = 0, per = 0, post_c = 0, post_k = 0;
  ConvLayer pre;
  float* cond_w = nullptr;  // fp32 [1][gin][c0]
  float* cond_b = nullptr;
  std::vector<ConvLayer> ups;  // [stage], polyphase groups inside
  std::vector<int> up_u, stage_c;
  std::vector<std::vector<ConvLayer>> c1, c2;  // [resblock][layer]
  std::vector<std::vector<PairLayer>> pairs;   // [resblock][layer]: fused conv1+conv2 (umma_pair.cu) where fused[rb][l]
  std::vector<std::vector<char>> fused;
  std::vector<std::vector<int>> pair_heights;  // [geometry level]: tile heights the fused pairs need
  float* post_w = nullptr;
  std::vector<float> post_w_host;  // [1][C][k], for the constant-bank kernel
  DBuf zp, xs, xu, t1, r, rj0, rj1, sum, meta, gcond;
  PinnedBuf pin_meta;
};

UmmaDecoder* umma_decoder_create(const DecoderHostWeights& w, sbv2_model* owner) {
  std::unique_ptr<UmmaDecoder> D(new UmmaDecoder());
  D->gin = w.gin;
  D->cin0 = w.pre.d1;
  D->c0 = w.pre.d0;
  D->n_stages = int(w.ups.size());
  D->per = w.per;
  D->pre = make_conv1d_layer(owner, w.pre, 1, 2);
  {
    // cond: Conv1d(gin -> c0, 1) evaluated on [B, gin] rows with the fp32 kernel
    std::vector<float> t(size_t(w.cond.d0) * w.cond.d1);
    for (int co = 0; co < w.cond.d0; ++co)
      for (int ci = 0; ci < w.cond.d1; ++ci) t[size_t(ci) * w.cond.d0 + co] = w.cond.w[size_t(co) * w.cond.d1 + ci];
    D->cond_w = owner->upload_f32(t);
    D->cond_b = owner->upload_f32(w.cond.b);
  }
  // ResBlock pairs are fused for C <= 64 (and the k = 3 pairs of C = 128): there the unfused convs are bound by HBM traffic
  // and epilogue work, not by the tensor pipe (a C = 128, k = 11 pair would stream 2 x 360 KB of weights from L2 per 118
  // output rows).  SBV2_B200_PAIR_MAXC=0 disables fusion.
  int pair_maxc = 64;
  if (const char* e = getenv("SBV2_B200_PAIR_MAXC")) pair_maxc = atoi(e);
  // N block of the C >= 256 ResBlock convs: 256 (one 128-row item streams the whole [256 x K] weight slab) or 128 (256-row
  // items, two N blocks: half the weight bytes per row)
  int wide_nb = 256;
  if (const char* e = getenv("SBV2_B200_DEC_WIDE_NB")) wide_nb = atoi(e);
  D->pair_heights.assign(size_t(D->n_stages) + 1, {});
  int C = D->c0;
  for (int s = 0; s < D->n_stages; ++s) {
    const HostConv& U = w.ups[s];
    if (U.d0 != C) fail(SBV2_ERR_UNSUPPORTED, "decoder upsample channel mismatch");
    D->ups.push_back(make_upsample_layer(owner, U, w.up_u[s], 16));
    D->up_u.push_back(w.up_u[s]);
    C = U.d1;
    D->stage_c.push_back(C);
    for (int j = 0; j < w.per; ++j) {
      size_t rb = size_t(s) * w.per + j;
      std::vector<ConvLayer> l1, l2;
      std::vector<PairLayer> lp;
      std::vector<char> lf;
      for (size_t l = 0; l < w.res_c1[rb].size(); ++l) {
        PairLayer P;
        // Per-shape choice from profiles/r2_pair_vs_unfused.log (fused vs unfused, us, 32 x ~860 frames): C = 128 pairs are
        // fused for k = 3 (426 vs 519) and k = 7 (709 vs 740) but not k = 11 (1150 vs 1019: too many weight bytes per
        // 118-row item); C = 64, k = 11 pairs only where the MRF mean rides on the epilogue (679 vs 675 plain, 778 vs 960 with
        // the mean); everything narrower is fused.
        const bool mrf_pair = l + 1 == w.res_c1[rb].size() && j + 1 == w.per;
        const bool want = (C <= pair_maxc && !(C == 64 && w.res_c1[rb][l].k == 11 && !mrf_pair)) ||
                          (C == 128 && pair_maxc >= 64 && w.res_c1[rb][l].k <= 7);
        const bool f = (w.per == 1 || w.per == 3) && want && make_pair_layer(owner, w.res_c1[rb][l], w.res_dil[rb][l], w.res_c2[rb][l], &P);
        lf.push_back(f ? 1 : 0);
        lp.push_back(P);
        if (f) {
          std::vector<int>& hs = D->pair_heights[s + 1];
          if (std::find(hs.begin(), hs.end(), P.out_rows) == hs.end()) hs.push_back(P.out_rows);
          l1.emplace_back();
          l2.emplace_back();
        } else {
          l1.push_back(make_conv1d_layer(owner, w.res_c1[rb][l], w.res_dil[rb][l], 16, C >= 256 ? wide_nb : 256));
          l2.push_back(make_conv1d_layer(owner, w.res_c2[rb][l], 1, 16, C >= 256 ? wide_nb : 256));
        }
      }
      D->c1.push_back(l1);
      D->c2.push_back(l2);
      D->pairs.push_back(lp);
      D->fused.push_back(lf);
    }
  }
  D->post_c = w.post.d1;
  D->post_k = w.post.k;
  if (D->post_c != C || D->post_c % 8 != 0) fail(SBV2_ERR_UNSUPPORTED, "decoder conv_post channel mismatch");
  D->post_w = owner->upload_f32(w.post.w);
  D->post_w_host = w.post.w;
  for (DBuf* b : {&D->zp, &D->xs, &D->xu, &D->t1, &D->r, &D->rj0, &D->rj1, &D->sum, &D->meta, &D->gcond}) b->stream = owner->stream;
  return D.release();
}

void umma_decoder_free(UmmaDecoder* d) { delete d; }

void umma_decoder_run(UmmaDecoder* D, sbv2_model* owner, const float* z, const float* g, int B, const std::vector<int>& ystart,
                      const std::vector<int>& ylen, float* wave, const std::vector<long long>* wstart) {
  LaunchCtx ctx = owner->ctx();
  std::vector<int> muls(1, 1);
  for (int s = 0; s < D->n_stages; ++s) muls.push_back(muls.back() * D->up_u[s]);
  BatchGeom bg = build_geoms(owner, D->meta, D->pin_meta, ystart, ylen, muls, &D->pair_heights, /*pin_idle=*/true, wstart);
  // buffer sizes
  size_t max_half = size_t(bg.g[0].rows_tot) * D->c0;
  for (int s = 0; s < D->n_stages; ++s) max_half = std::max(max_half, size_t(bg.g[s + 1].rows_tot) * D->stage_c[s]);
  D->zp.ensure(size_t(bg.g[0].rows_tot) * D->cin0 * 2);
  D->xs.ensure(max_half * 2);
  D->xu.ensure(max_half * 2);
  D->t1.ensure(max_half * 2);
  D->r.ensure(max_half * 2);
  const bool mrf3 = D->per == 3;  // MRF mean folded into the last conv's epilogue (fp16 r0, r1) instead of an fp32 sum buffer
  if (mrf3) {
    D->rj0.ensure(max_half * 2);
    D->rj1.ensure(max_half * 2);
  } else {
    D->sum.ensure(max_half * 4);
  }
  __half* rj[2] = {D->rj0.as<__half>(), D->rj1.as<__half>()};
  D->gcond.ensure(size_t(B) * D->c0 * 4);
  __half* zp = D->zp.as<__half>();
  __half* xs = D->xs.as<__half>();
  __half* xu = D->xu.as<__half>();
  __half* t1 = D->t1.as<__half>();
  __half* r = D->r.as<__half>();
  float* sum = D->sum.as<float>();
  float* gcond = D->gcond.as<float>();

  // cond(g) -> per-utterance bias of conv_pre
  {
    // one segment of B rows: reuse the first geometry's arrays is not possible; a tiny dedicated pair lives after wstart
    // (start = 0, len = B) — build it on the fly in the gcond buffer's tail is overkill: launch with an explicit Segs
    // whose arrays are the (ystart-independent) prefix of geometry 0: prefix[0] == 0 and we need len == B.
    static_assert(sizeof(int) == 4, "");
  }
  {
    // Segs {start=[0], len=[B]}: store in pinned+device meta tail
    // (appended by build_geoms would complicate its layout; use a small separate upload)
    int two[2] = {0, B};
    D->gcond.ensure(size_t(B) * D->c0 * 4 + 64);
    gcond = D->gcond.as<float>();
    int* d_two = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(gcond) + size_t(B) * D->c0 * 4);
    CUDA_CHECK(cudaMemcpyAsync(d_two, two, 8, cudaMemcpyHostToDevice, owner->stream));
    ConvArgs a;
    a.in = g;
    a.in_ld = D->gin;
    a.w = D->cond_w;
    a.bias = D->cond_b;
    a.out = gcond;
    a.out_ld = D->c0;
    a.cin = D->gin;
    a.cout = D->c0;
    a.seg.start = d_two;
    a.seg.len = d_two + 1;
    a.seg.n = 1;
    a.seg.max_len = B;
    launch_conv(ctx, a);
  }

  const Geom& G0 = bg.g[0];
  launch_zero_gaps(ctx, zp, D->cin0, G0, B);
  launch_to_planar(ctx, zp, z, D->cin0, D->cin0, bg.d_ystart, G0, B, ACT_NONE);
  launch_zero_gaps(ctx, xs, D->c0, G0, B);
  {
    ConvCall c;
    c.in = zp;
    c.out = xs;
    c.act_out = ACT_LRELU;
    c.bias_utt = gcond;
    launch_umma(ctx, D->pre, G0, G0, c, B);
  }
  for (int s = 0; s < D->n_stages; ++s) {
    const Geom& Gi = bg.g[s];
    const Geom& Go = bg.g[s + 1];
    const int C = D->stage_c[s];
    const int u = D->up_u[s];
    launch_zero_gaps(ctx, xu, C, Go, B);
    {
      ConvCall c;
      c.in = xs;
      c.out = xu;
      c.act_out = ACT_LRELU;
      c.out_mul = u;
      launch_umma(ctx, D->ups[s], Gi, Go, c, B);
    }
    launch_zero_gaps(ctx, t1, C, Go, B);
    launch_zero_gaps(ctx, r, C, Go, B);
    const bool last_stage = s + 1 == D->n_stages;
    for (int j = 0; j < D->per; ++j) {
      size_t rb = size_t(s) * D->per + j;
      const __half* cur = xu;
      const size_t nl = D->c1[rb].size();
      for (size_t l = 0; l < nl; ++l) {
        // destination of this pair: the stage output (last pair of the last ResBlock: MRF mean folded in), the
        // ResBlock's output rj[j], or a scratch buffer that is not the pair's input
        const bool fuse = D->fused[rb][l] != 0;
        // unfused: conv1 -> mid, conv2 (+ residual) -> dst, where dst may be the input buffer (element-wise aliasing only)
        __half* mid = cur == t1 ? r : t1;
        __half* dst = fuse ? (cur == r ? t1 : r) : (mid == t1 ? r : t1);
        int act = ACT_LRELU;
        const __half *res2 = nullptr, *res3 = nullptr;
        float out_div = 1.f;
        float* accum = nullptr;
        int accum_mode = UACC_NONE;
        if (l + 1 == nl) {
          const bool last_rb = j + 1 == D->per;
          if (mrf3 && !last_rb) {
            dst = rj[j];
          } else if (mrf3 || D->per == 1) {
            if (mrf3) {
              res2 = rj[0];
              res3 = rj[1];
              out_div = float(D->per);
            }
            launch_zero_gaps(ctx, xs, C, Go, B);
            dst = xs;
            act = last_stage ? ACT_LRELU01 : ACT_LRELU;
          } else {
            accum = sum;
            accum_mode = j == 0 ? UACC_SET : (last_rb ? UACC_FINAL : UACC_ADD);
            dst = nullptr;
            if (last_rb) {
              launch_zero_gaps(ctx, xs, C, Go, B);
              dst = xs;
              act = last_stage ? ACT_LRELU01 : ACT_LRELU;
            }
          }
        }
        if (fuse) {
          PairCall pc;
          pc.in = cur;
          pc.out = dst;
          pc.residual2 = res2;
          pc.residual3 = res3;
          pc.out_div = out_div;
          pc.act_out = act;
          launch_umma_pair(ctx, D->pairs[rb][l], Go, pc, B);
        } else {
          {
            ConvCall c;
            c.in = cur;
            c.out = mid;
            c.act_out = ACT_LRELU;
            launch_umma(ctx, D->c1[rb][l], Go, Go, c, B);
          }
          ConvCall c;
          c.in = mid;
          c.residual = cur;
          c.residual2 = res2;
          c.residual3 = res3;
          c.out_div = out_div;
          c.out = dst;
          c.act_out = act;
          c.accum = accum;
          c.accum_mode = accum_mode;
          c.accum_div = float(D->per);
          launch_umma(ctx, D->c2[rb][l], Go, Go, c, B);
        }
        cur = dst;
      }
    }
  }
  launch_dec_post_planar(ctx, wave, xs, bg.g.back(), bg.d_wstart, B, D->post_w, D->post_w_host, D->post_c, D->post_k, false);
  // the pinned geometry blob is rewritten by the next run: make sure its upload finished
  // (it did: every kernel above depends on it and the caller synchronises before returning results)
}

}  // namespace sbv2

#ifdef SBV2_DEBUG_HOOKS  // kernel unit-test / tracing entry points: only in libsbv2_b200_debug.so (build.py)
// ---- test hook: one convolution through both the fp32 kernel and the tensor-core kernel -------------------
extern "C" int sbv2_debug_conv_compare(const float* x, int64_t T, int cin, const float* w, const float* bias, int cout, int k,
                                       int dil, int mt_pref, int with_residual, float* out_umma, float* out_ref) {
  using namespace sbv2;
  return guarded([&] {
    SBV2_REQUIRE(x && w && out_umma && out_ref && T > 0, "bad arguments");
    sbv2_model owner;
    owner.device = 0;
    if (const char* pe = getenv("SBV2_B200_PDL")) owner.pdl = pe[0] != '0';
    CUDA_CHECK(cudaSetDevice(0));
    CUDA_CHECK(cudaStreamCreateWithFlags(&owner.stream, cudaStreamNonBlocking));
    LaunchCtx ctx = owner.ctx();
    HostConv hc;
    hc.d0 = cout;
    hc.d1 = cin;
    hc.k = k;
    hc.w.assign(w, w + size_t(cout) * cin * k);
    if (bias) hc.b.assign(bias, bias + cout);
    int nb_max = 256;
    if (const char* e = getenv("SBV2_B200_TEST_NBMAX")) nb_max = atoi(e);
    ConvLayer L = make_conv1d_layer(&owner, hc, dil, mt_pref, nb_max);
    // fp32 reference weights [k][cin][cout]
    std::vector<float> wr(size_t(k) * cin * cout);
    for (int co = 0; co < cout; ++co)
      for (int ci = 0; ci < cin; ++ci)
        for (int j = 0; j < k; ++j) wr[(size_t(j) * cin + ci) * cout + co] = w[(size_t(co) * cin + ci) * k + j];
    float* d_wr = owner.upload_f32(wr);
    float* d_b = bias ? static_cast<float*>(owner.upload_bytes(bias, size_t(cout) * 4)) : nullptr;
    float* d_x = static_cast<float*>(owner.upload_bytes(x, size_t(T) * cin * 4));
    DBuf meta, xin, xout, xres, ref, back;
    PinnedBuf pin;
    for (DBuf* b : {&meta, &xin, &xout, &xres, &ref, &back}) b->stream = owner.stream;
    std::vector<int> ystart{0}, ylen{int(T)}, muls{1};
    BatchGeom bg = build_geoms(&owner, meta, pin, ystart, ylen, muls);
    const Geom& G = bg.g[0];
    xin.ensure(size_t(G.rows_tot) * cin * 2);
    xout.ensure(size_t(G.rows_tot) * cout * 2);
    ref.ensure(size_t(T) * cout * 4);
    back.ensure(size_t(T) * cout * 4);
    launch_zero_gaps(ctx, xin.as<__half>(), cin, G, 1);
    launch_to_planar(ctx, xin.as<__half>(), d_x, cin, cin, bg.d_ystart, G, 1, ACT_NONE);
    ConvCall c;
    c.in = xin.as<__half>();
    c.out = xout.as<__half>();
    if (with_residual) {
      SBV2_REQUIRE(cin == cout, "residual test needs cin == cout");
      c.residual = xin.as<__half>();  // interpreted as lrelu-stored values
    }
    launch_umma(ctx, L, G, G, c, 1);
    launch_from_planar(ctx, back.as<float>(), xout.as<__half>(), cout, bg.d_ystart, G, 1);
    // reference
    ConvArgs a;
    a.in = d_x;
    a.in_ld = cin;
    a.w = d_wr;
    a.bias = d_b;
    a.out = ref.as<float>();
    a.out_ld = cout;
    a.cin = cin;
    a.cout = cout;
    a.taps = k;
    a.dil = dil;
    a.off = -dil * ((k - 1) / 2);
    a.seg.start = bg.d_ystart;      // [0]
    a.seg.len = G.d_len;            // [T]
    a.seg.n = 1;
    a.seg.max_len = int(T);
    launch_conv(ctx, a);
    CUDA_CHECK(cudaMemcpyAsync(out_umma, back.p, size_t(T) * cout * 4, cudaMemcpyDeviceToHost, owner.stream));
    CUDA_CHECK(cudaMemcpyAsync(out_ref, ref.p, size_t(T) * cout * 4, cudaMemcpyDeviceToHost, owner.stream));
    CUDA_CHECK(cudaStreamSynchronize(owner.stream));
  });
}

// ---- test hook: per-role clock64 trace of one conv launch (performance debugging) ----------------------------
namespace sbv2 {
extern long long* g_trace;
extern long long* g_pair_trace;
}
extern "C" int sbv2_debug_conv_trace(int64_t T, int cin, int cout, int k, int dil, int mt_pref, int with_residual, int accum_mode,
                                     long long* out_trace /*[n_blocks*64*8]*/, int n_blocks, float* out_ms, int* out_cfg /*[8]*/) {
  using namespace sbv2;
  return guarded([&] {
    sbv2_model owner;
    owner.device = 0;
    CUDA_CHECK(cudaSetDevice(0));
    CUDA_CHECK(cudaStreamCreateWithFlags(&owner.stream, cudaStreamNonBlocking));
    LaunchCtx ctx = owner.ctx();
    HostConv hc;
    hc.d0 = cout;
    hc.d1 = cin;
    hc.k = k;
    hc.w.assign(size_t(cout) * cin * k, 0.01f);
    hc.b.assign(cout, 0.1f);
    ConvLayer L = make_conv1d_layer(&owner, hc, dil, mt_pref);
    if (out_cfg) {
      int cfg[8] = {L.mt, L.nb, L.a_slots, L.nstages, L.sps, L.b_resident, int(L.smem), L.nkc};
      memcpy(out_cfg, cfg, sizeof(cfg));
    }
    DBuf meta, xin, xout, acc, tr;
    PinnedBuf pin;
    for (DBuf* b : {&meta, &xin, &xout, &acc, &tr}) b->stream = owner.stream;
    std::vector<int> ystart{0}, ylen{int(T)}, muls{1};
    BatchGeom bg = build_geoms(&owner, meta, pin, ystart, ylen, muls);
    const Geom& G = bg.g[0];
    xin.ensure(size_t(G.rows_tot) * cin * 2);
    xout.ensure(size_t(G.rows_tot) * cout * 2);
    acc.ensure(size_t(G.rows_tot) * cout * 4);
    CUDA_CHECK(cudaMemsetAsync(xin.p, 0, size_t(G.rows_tot) * cin * 2, owner.stream));
    CUDA_CHECK(cudaMemsetAsync(xout.p, 0, size_t(G.rows_tot) * cout * 2, owner.stream));
    CUDA_CHECK(cudaMemsetAsync(acc.p, 0, size_t(G.rows_tot) * cout * 4, owner.stream));
    const size_t tr_elems = size_t(148) * 64 * 8;
    tr.ensure(tr_elems * 8);
    CUDA_CHECK(cudaMemsetAsync(tr.p, 0, tr_elems * 8, owner.stream));
    ConvCall c;
    c.in = xin.as<__half>();
    c.out = xout.as<__half>();
    c.act_out = ACT_LRELU;
    if (with_residual) c.residual = xin.as<__half>();
    if (accum_mode) {
      c.accum = acc.as<float>();
      c.accum_mode = accum_mode;
      c.accum_div = 3.f;
      if (accum_mode != UACC_FINAL) c.out = nullptr;
    }
    for (int i = 0; i < 2; ++i) launch_umma(ctx, L, G, G, c, 1);
    cudaEvent_t e0, e1;
    CUDA_CHECK(cudaEventCreate(&e0));
    CUDA_CHECK(cudaEventCreate(&e1));
    CUDA_CHECK(cudaEventRecord(e0, owner.stream));
    for (int i = 0; i < 5; ++i) launch_umma(ctx, L, G, G, c, 1);
    CUDA_CHECK(cudaEventRecord(e1, owner.stream));
    g_trace = tr.as<long long>();
    launch_umma(ctx, L, G, G, c, 1);
    g_trace = nullptr;
    CUDA_CHECK(cudaStreamSynchronize(owner.stream));
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    if (out_ms) *out_ms = ms / 5.f;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (out_trace && n_blocks > 0)
      CUDA_CHECK(cudaMemcpy(out_trace, tr.p, size_t(std::min(n_blocks, 148)) * 64 * 8 * 8, cudaMemcpyDeviceToHost));
  });
}

// ---- test hook: one ResBlock pair through the fused kernel and through two unfused tensor-core convs ------------
// x: packed [sum(lens), C] fp32 (pre-activation); outputs are the stored (post-lrelu) values, packed the same way.
extern "C" int sbv2_debug_pair_compare(const float* x, const int* lens, int n_utt, int C, int k, int dil, const float* w1,
                                       const float* b1, const float* w2, const float* b2, int mrf, int iters, float* out_fused,
                                       float* out_ref, float* out_ms /*[2]: fused, unfused*/, int* out_cfg /*[8]*/,
                                       long long* out_trace /*[64*16] or null*/) {
  using namespace sbv2;
  return guarded([&] {
    SBV2_REQUIRE(x && lens && n_utt > 0 && w1 && w2 && out_fused && out_ref, "bad arguments");
    sbv2_model owner;
    owner.device = 0;
    CUDA_CHECK(cudaSetDevice(0));
    CUDA_CHECK(cudaStreamCreateWithFlags(&owner.stream, cudaStreamNonBlocking));
    LaunchCtx ctx = owner.ctx();
    HostConv h1, h2;
    h1.d0 = h1.d1 = h2.d0 = h2.d1 = C;
    h1.k = h2.k = k;
    h1.w.assign(w1, w1 + size_t(C) * C * k);
    h2.w.assign(w2, w2 + size_t(C) * C * k);
    h1.b.assign(b1, b1 + C);
    h2.b.assign(b2, b2 + C);
    PairLayer P;
    if (!make_pair_layer(&owner, h1, dil, h2, &P)) fail(SBV2_ERR_UNSUPPORTED, "pair does not fit the fused plan");
    if (out_cfg) {
      int cfg[8] = {P.mt, P.out_rows, P.a_slots, P.nstages, P.sps, P.b_resident, int(P.smem), P.nkc};
      memcpy(out_cfg, cfg, sizeof(cfg));
    }
    ConvLayer L1 = make_conv1d_layer(&owner, h1, dil, 16);
    ConvLayer L2 = make_conv1d_layer(&owner, h2, 1, 16);
    std::vector<int> ystart, ylen;
    int tot = 0;
    for (int i = 0; i < n_utt; ++i) {
      ystart.push_back(tot);
      ylen.push_back(lens[i]);
      tot += lens[i];
    }
    float* d_x = static_cast<float*>(owner.upload_bytes(x, size_t(tot) * C * 4));
    DBuf meta, xin, mid, of, orf, ra, rb, back;
    PinnedBuf pin;
    for (DBuf* b : {&meta, &xin, &mid, &of, &orf, &ra, &rb, &back}) b->stream = owner.stream;
    std::vector<int> muls{1};
    std::vector<std::vector<int>> heights{{P.out_rows}};
    BatchGeom bg = build_geoms(&owner, meta, pin, ystart, ylen, muls, &heights);
    const Geom& G = bg.g[0];
    const size_t bytes = size_t(G.rows_tot) * C * 2;
    for (DBuf* b : {&xin, &mid, &of, &orf, &ra, &rb}) {
      b->ensure(bytes);
      launch_zero_gaps(ctx, b->as<__half>(), C, G, n_utt);
    }
    back.ensure(size_t(tot) * C * 4);
    launch_to_planar(ctx, xin.as<__half>(), d_x, C, C, bg.d_ystart, G, n_utt, ACT_LRELU);
    if (mrf) {  // two more "ResBlock outputs": scaled copies of the input
      launch_to_planar(ctx, ra.as<__half>(), d_x, C, C, bg.d_ystart, G, n_utt, ACT_LRELU);
      launch_to_planar(ctx, rb.as<__half>(), d_x, C, C, bg.d_ystart, G, n_utt, ACT_NONE);
    }
    auto run_fused = [&] {
      PairCall pc;
      pc.in = xin.as<__half>();
      pc.out = of.as<__half>();
      if (mrf) {
        pc.residual2 = ra.as<__half>();
        pc.residual3 = rb.as<__half>();
        pc.out_div = 3.f;
      }
      launch_umma_pair(ctx, P, G, pc, n_utt);
    };
    auto run_unfused = [&] {
      ConvCall c;
      c.in = xin.as<__half>();
      c.out = mid.as<__half>();
      c.act_out = ACT_LRELU;
      launch_umma(ctx, L1, G, G, c, n_utt);
      ConvCall d;
      d.in = mid.as<__half>();
      d.residual = xin.as<__half>();
      d.out = orf.as<__half>();
      d.act_out = ACT_LRELU;
      if (mrf) {
        d.residual2 = ra.as<__half>();
        d.residual3 = rb.as<__half>();
        d.out_div = 3.f;
      }
      launch_umma(ctx, L2, G, G, d, n_utt);
    };
    run_fused();
    run_unfused();
    launch_from_planar(ctx, back.as<float>(), of.as<__half>(), C, bg.d_ystart, G, n_utt);
    CUDA_CHECK(cudaMemcpyAsync(out_fused, back.p, size_t(tot) * C * 4, cudaMemcpyDeviceToHost, owner.stream));
    CUDA_CHECK(cudaStreamSynchronize(owner.stream));
    launch_from_planar(ctx, back.as<float>(), orf.as<__half>(), C, bg.d_ystart, G, n_utt);
    CUDA_CHECK(cudaMemcpyAsync(out_ref, back.p, size_t(tot) * C * 4, cudaMemcpyDeviceToHost, owner.stream));
    CUDA_CHECK(cudaStreamSynchronize(owner.stream));
    if (iters > 0 && out_ms) {
      cudaEvent_t e0, e1, e2;
      CUDA_CHECK(cudaEventCreate(&e0));
      CUDA_CHECK(cudaEventCreate(&e1));
      CUDA_CHECK(cudaEventCreate(&e2));
      CUDA_CHECK(cudaEventRecord(e0, owner.stream));
      for (int i = 0; i < iters; ++i) run_fused();
      CUDA_CHECK(cudaEventRecord(e1, owner.stream));
      for (int i = 0; i < iters; ++i) run_unfused();
      CUDA_CHECK(cudaEventRecord(e2, owner.stream));
      CUDA_CHECK(cudaStreamSynchronize(owner.stream));
      CUDA_CHECK(cudaEventElapsedTime(&out_ms[0], e0, e1));
      CUDA_CHECK(cudaEventElapsedTime(&out_ms[1], e1, e2));
      out_ms[0] /= iters;
      out_ms[1] /= iters;
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
      cudaEventDestroy(e2);
    }
    if (out_trace) {
      DBuf tr;
      tr.stream = owner.stream;
      tr.ensure(64 * 16 * 8);
      CUDA_CHECK(cudaMemsetAsync(tr.p, 0, 64 * 16 * 8, owner.stream));
      g_pair_trace = tr.as<long long>();
      run_fused();
      g_pair_trace = nullptr;
      CUDA_CHECK(cudaStreamSynchronize(owner.stream));
      CUDA_CHECK(cudaMemcpy(out_trace, tr.p, 64 * 16 * 8, cudaMemcpyDeviceToHost));
    }
  });
}
#endif  // SBV2_DEBUG_HOOKS
