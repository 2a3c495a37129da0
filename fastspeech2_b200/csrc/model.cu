// Host-side orchestration of the two forward passes and the extern "C" surface declared in include/fs2b200.h.
// No allocation, no synchronisation: every launch goes to the caller's stream, temporaries come from the caller's workspace.
#include <mutex>
#include <new>
#include <vector>

#include "common.cuh"

namespace fs2 {

std::atomic<unsigned long long> g_launch_count{0};

// ------------------------------------------------------------------ per-device setup state
static DevState g_dev[FS2_MAX_DEVICES];
static std::mutex g_dev_mutex;
DevState* dev_state(int* err) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess || dev < 0 || dev >= FS2_MAX_DEVICES) {
    if (err) *err = e != cudaSuccess ? FS2_ERR_CUDA - (int)e : FS2_ERR_UNSUPPORTED;
    return nullptr;
  }
  DevState* d = &g_dev[dev];
  if (d->num_sms.load(std::memory_order_acquire) == 0) {
    int n = 0;
    e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess || n <= 0) {
      if (err) *err = FS2_ERR_CUDA - (int)e;
      return nullptr;
    }
    d->num_sms.store(n, std::memory_order_release);
  }
  return d;
}
int setup_once(std::atomic<bool>& done, cudaError_t (*fn)()) {
  if (done.load(std::memory_order_acquire)) return FS2_OK;
  std::lock_guard<std::mutex> lock(g_dev_mutex);
  if (done.load(std::memory_order_relaxed)) return FS2_OK;
  const cudaError_t e = fn();
  if (e != cudaSuccess) return FS2_ERR_CUDA - (int)e;
  done.store(true, std::memory_order_release);
  return FS2_OK;
}

// ------------------------------------------------------------------ per-launch profiling (off unless armed; state is per host thread)
thread_local bool g_prof_on = false;
struct ProfRec { cudaEvent_t a, b; int cls; double flops; };
static thread_local std::vector<ProfRec> g_prof;
static thread_local cudaEvent_t g_prof_pending;
void prof_before(cudaStream_t s) {
  if (!g_prof_on) return;
  cudaEventCreate(&g_prof_pending);
  cudaEventRecord(g_prof_pending, s);
}
void prof_after(cudaStream_t s, int cls, double flops) {
  if (!g_prof_on) return;
  ProfRec r;
  r.a = g_prof_pending; r.cls = cls; r.flops = flops;
  cudaEventCreate(&r.b);
  cudaEventRecord(r.b, s);
  g_prof.push_back(r);
}

// kernels / launchers defined in the other translation units
int conv1d_simt(const fs2_conv1d_args* a, cudaStream_t s);
int conv1d_tc(const fs2_conv1d_args* a, const float* wt, unsigned variant, cudaStream_t s, long long wt_batch_stride = 0);
int attention_gemm(const fs2_attention_args* a, void* ws, size_t ws_bytes, cudaStream_t s);
size_t attention_gemm_workspace(int B, int T, int H);
int attention_fused(const fs2_attention_args* a, void* ws, size_t ws_bytes, cudaStream_t s);
size_t attention_fused_workspace(int B, int T, int H);
bool conv_tc_supported(const fs2_conv1d_args* a);
int conv_tc_nb(int N);
int conv_tc_plan_query(const fs2_conv1d_args* a, int num_sms, int* out);
#ifdef FS2_DEBUG_KNOBS
extern long long* g_tc_trace;
extern int g_tc_tune[4];
extern int g_tc_pdl;
#endif

// backend dispatch of the fs2_conv1d contract
static int conv1d_dispatch(const fs2_conv1d_args* a, cudaStream_t s) {
  if (!a) return FS2_ERR_ARG;
  if (a->backend == FS2_CONV_TC) return a->w_tc ? conv1d_tc(a, a->w_tc, a->tc_variant, s) : FS2_ERR_ARG;
  if (a->backend == FS2_CONV_AUTO && a->w_tc && conv_tc_supported(a)) return conv1d_tc(a, a->w_tc, a->tc_variant, s);
  return conv1d_simt(a, s);
}
int attention_simt(const fs2_attention_args* a, cudaStream_t s);
int embed_positions(const fs2_embed_args* a, cudaStream_t s);
int add_speaker(const fs2_rowbias_args* a, cudaStream_t s);
int layernorm(const fs2_layernorm_args* a, cudaStream_t s);
int variance_head(const fs2_variance_head_args* a, cudaStream_t s);
int durations(const fs2_durations_args* a, cudaStream_t s);
int length_regulate(const fs2_length_regulate_args* a, cudaStream_t s);
int conv_post(const fs2_conv_post_args* a, cudaStream_t s);
int resstack(const fs2_resstack_args* a, cudaStream_t s);
int wav_to_int16(const fs2_wav_int16_args* a, cudaStream_t s);
int resstack_plan(const fs2_resstack_args* a, int num_sms, int* out);
int transpose_bct_to_btc(const float* in, float* out, int B, int C, int T, cudaStream_t s);
int add_positions(float* x, const float* pos, int B, int T, int D, cudaStream_t s);

// ------------------------------------------------------------------ workspace bump allocator
struct Arena {
  char* base; size_t cap, off;
  bool dry;  // dry run: only measure
  explicit Arena(void* p, size_t n) : base((char*)p), cap(n), off(0), dry(p == nullptr) {}
  float* f32(size_t n) { return (float*)take(n * sizeof(float)); }
  void* take(size_t bytes) {
    const size_t a = (off + 255) & ~(size_t)255;
    off = a + bytes;
    if (dry) return (void*)(uintptr_t)256;  // non-null dummy
    if (off > cap) return nullptr;
    return base + a;
  }
};

// contiguous [B][T][C] convolution helper
static int conv(cudaStream_t s, const float* x, int B, int T, int Cin, const float* w, const float* w_tc, const float* bias, int N,
                int taps, int dil, int pad, int out_act, float out_slope, float* y, const float* res = nullptr,
                int in_act = FS2_ACT_NONE, float in_slope = 0.f, float alpha = 1.f, int accumulate = 0,
                const int32_t* row_lens = nullptr, unsigned tc_variant = 0) {
  fs2_conv1d_args a{};
  a.w_tc = w_tc; a.backend = FS2_CONV_AUTO; a.tc_variant = tc_variant;
  a.x = x; a.x_batch_stride = (int64_t)T * Cin; a.x_row_stride = Cin;
  a.B = B; a.T = T; a.Cin = Cin;
  a.w = w; a.bias = bias; a.N = N; a.taps = taps; a.dilation = dil; a.pad_left = pad;
  a.in_act = in_act; a.in_slope = in_slope; a.out_act = out_act; a.out_slope = out_slope;
  a.res = res; a.res_batch_stride = (int64_t)T * N; a.res_row_stride = N;
  a.alpha = alpha; a.accumulate = accumulate; a.row_lens = row_lens;
  a.y = y; a.y_batch_stride = (int64_t)T * N; a.y_row_stride = N;
  return conv1d_dispatch(&a, s);
}

static int ln(cudaStream_t s, const float* x, float* y, int B, int T, int C, const float* g, const float* b, const int32_t* lens,
              int pre_relu = 0) {
  fs2_layernorm_args a{x, y, B, T, C, g, b, 1e-5f, lens, pre_relu};
  return layernorm(&a, s);
}

// K-segmented tensor-core convolution for the layers that feed the discrete decisions (encoder, predictors): the sum over taps and
// input channels is cut into (tap, 256-channel) slices; each slice is one work unit of 16 K-steps with separate accumulators for
// the hi*hi term and the cross terms (FS2_TC_VARIANT_NB64 | FS2_TC_VARIANT_SEGMENTED, one launch per conv), and the slices are added in
// fp32 round-to-nearest by the epilogue's accumulate path.  That bounds the tensor core's truncating accumulation to 16 steps per chain (a single k = 9 launch has 432) and
// brings the error back to the fp32 CUDA-core kernel's level (profiles/r02/flip_census_*.jsonl).  `w_seg`: taps * (Cin/256) tile
// buffers of 128 + 1024*N bytes (packing.pack_conv_tc_segments).  y = bias + sum_slices + res, rows >= row_lens zeroed; no output
// activation (a following ReLU is applied by the consumer: in_act of the next conv / pre_relu of the LayerNorm).
static int conv_seg(cudaStream_t s, const float* x, int B, int T, int Cin, const float* w_seg, const float* bias, int N, int taps, int pad,
                    float* y, const float* res, int in_act, float in_slope, const int32_t* row_lens) {
  fs2_conv1d_args a{};
  a.x = x; a.x_batch_stride = (int64_t)T * Cin; a.x_row_stride = Cin;
  a.B = B; a.T = T; a.Cin = Cin;
  a.w = nullptr; a.w_tc = w_seg; a.backend = FS2_CONV_TC; a.tc_variant = FS2_TC_VARIANT_NB64 | FS2_TC_VARIANT_SEGMENTED;
  a.bias = bias; a.N = N; a.taps = taps; a.dilation = 1; a.pad_left = pad;
  a.in_act = in_act; a.in_slope = in_slope; a.out_act = FS2_ACT_NONE;
  a.res = res; a.res_batch_stride = (int64_t)T * N; a.res_row_stride = N;
  a.alpha = 1.f; a.accumulate = 0; a.row_lens = row_lens;
  a.y = y; a.y_batch_stride = (int64_t)T * N; a.y_row_stride = N;
  return conv1d_tc(&a, a.w_tc, a.tc_variant, s);
}

struct FftBufs { float *x, *tmp, *qkv, *ctx, *hid; void* att_ws; size_t att_bytes; };

// The GEMM attention materialises S [B*H][T][Tk] in fp32 and keeps a score row in registers: it serves 192 <= T <= 4096 with a
// workspace of at most 8 GB; anything longer / larger runs the exact flash-style kernel, which has no length limit.
static bool attention_gemm_usable(int B, int T, int H) {
  return T >= 192 && T <= 4096 && attention_gemm_workspace(B, T, H) <= ((size_t)8 << 30);
}

// One FFT block in place on bufs.x  (transformer/Layers.py:21-30)
static int fft_block(cudaStream_t s, const fs2_acoustic_model* m, const fs2_fft_block_weights& w, const FftBufs& f, int B, int T,
                     const int32_t* lens, bool tc, unsigned tcv, bool segmented = false) {
  const int D = m->d_model, F = m->d_inner;
  const float* none = nullptr;
  if (segmented) {                                     // encoder on the tensor cores: K-segmented convs, exact attention
    if (!w.w_qkv_tc || !w.w_o_tc || !w.w_1_tc || !w.w_2_tc || m->k2 != 1) return FS2_ERR_ARG;
    FS2_TRY(conv_seg(s, f.x, B, T, D, w.w_qkv_tc, w.b_qkv, 3 * D, 1, 0, f.qkv, nullptr, FS2_ACT_NONE, 0.f, nullptr));
    fs2_attention_args at{};
    at.qkv = f.qkv; at.ctx = f.ctx; at.B = B; at.T = T; at.H = m->n_head; at.Dh = D / m->n_head; at.key_lens = lens;
    at.scale = 1.0f / sqrtf((float)(D / m->n_head));
    FS2_TRY(attention_simt(&at, s));
    FS2_TRY(conv_seg(s, f.ctx, B, T, D, w.w_o_tc, w.b_o, D, 1, 0, f.tmp, f.x, FS2_ACT_NONE, 0.f, nullptr));
    FS2_TRY(ln(s, f.tmp, f.x, B, T, D, w.ln1_g, w.ln1_b, lens));
    // conv-FFN: w_1 leaves the pre-activation hidden, the ReLU is w_2's input activation (leaky_relu with slope 0)
    FS2_TRY(conv_seg(s, f.x, B, T, D, w.w_1_tc, w.b_1, F, m->k1, (m->k1 - 1) / 2, f.hid, nullptr, FS2_ACT_NONE, 0.f, nullptr));
    FS2_TRY(conv_seg(s, f.hid, B, T, F, w.w_2_tc, w.b_2, D, 1, 0, f.tmp, f.x, FS2_ACT_LRELU, 0.f, nullptr));
    FS2_TRY(ln(s, f.tmp, f.x, B, T, D, w.ln2_g, w.ln2_b, lens));
    return FS2_OK;
  }
  FS2_TRY(conv(s, f.x, B, T, D, w.w_qkv, tc ? w.w_qkv_tc : none, w.b_qkv, 3 * D, 1, 1, 0, FS2_ACT_NONE, 0.f, f.qkv, nullptr, FS2_ACT_NONE, 0.f,
               1.f, 0, nullptr, tcv));
  fs2_attention_args at{};
  at.qkv = f.qkv; at.ctx = f.ctx; at.B = B; at.T = T; at.H = m->n_head; at.Dh = D / m->n_head; at.key_lens = lens;
  at.scale = 1.0f / sqrtf((float)(D / m->n_head));
  if (tc && f.att_ws && (m->tc_mask & FS2_TC_ATTENTION_GEMM) && attention_gemm_usable(B, T, m->n_head)) {
    FS2_TRY(attention_gemm(&at, f.att_ws, f.att_bytes, s));          // round-1 path: S materialised, two GEMM launches per head
  } else if (tc && f.att_ws && T >= 128) {                            // one fused tcgen05 kernel: S stays in tensor memory, any length
    FS2_TRY(attention_fused(&at, f.att_ws, f.att_bytes, s));
  } else {
    FS2_TRY(attention_simt(&at, s));
  }
  FS2_TRY(conv(s, f.ctx, B, T, D, w.w_o, tc ? w.w_o_tc : none, w.b_o, D, 1, 1, 0, FS2_ACT_NONE, 0.f, f.tmp, f.x, FS2_ACT_NONE, 0.f, 1.f, 0, nullptr,
               tcv));
  FS2_TRY(ln(s, f.tmp, f.x, B, T, D, w.ln1_g, w.ln1_b, lens));
  FS2_TRY(conv(s, f.x, B, T, D, w.w_1, tc ? w.w_1_tc : none, w.b_1, F, m->k1, 1, (m->k1 - 1) / 2, FS2_ACT_RELU, 0.f, f.hid, nullptr, FS2_ACT_NONE,
               0.f, 1.f, 0, nullptr, tcv));
  FS2_TRY(conv(s, f.hid, B, T, F, w.w_2, tc ? w.w_2_tc : none, w.b_2, D, m->k2, 1, (m->k2 - 1) / 2, FS2_ACT_NONE, 0.f, f.tmp, f.x, FS2_ACT_NONE,
               0.f, 1.f, 0, nullptr, tcv));
  FS2_TRY(ln(s, f.tmp, f.x, B, T, D, w.ln2_g, w.ln2_b, lens));
  return FS2_OK;
}

static bool model_ok(const fs2_acoustic_model* m) {
  return m && m->d_model > 0 && m->n_head > 0 && m->d_model % m->n_head == 0 && m->n_enc >= 0 && m->n_enc <= FS2_MAX_LAYERS &&
         m->n_dec >= 0 && m->n_dec <= FS2_MAX_LAYERS && m->n_postnet >= 0 && m->n_postnet <= FS2_MAX_POSTNET && m->d_inner > 0 &&
         m->n_mel > 0 && m->vp_filter > 0;
}

static FftBufs fft_bufs(Arena& ar, const fs2_acoustic_model* m, size_t rows, int B = 0, int T = 0, bool tc_attention = false) {
  FftBufs f;
  f.att_ws = nullptr; f.att_bytes = 0;
  if (tc_attention && (m->tc_mask & FS2_TC_ATTENTION_GEMM) && attention_gemm_usable(B, T, m->n_head)) {
    f.att_bytes = attention_gemm_workspace(B, T, m->n_head);
    f.att_ws = ar.take(f.att_bytes);
  } else if (tc_attention && T >= 128) {
    f.att_bytes = attention_fused_workspace(B, T, m->n_head);
    f.att_ws = ar.take(f.att_bytes);
  }
  f.x = ar.f32(rows * m->d_model);
  f.tmp = ar.f32(rows * m->d_model);
  f.qkv = ar.f32(rows * 3 * m->d_model);
  f.ctx = ar.f32(rows * m->d_model);
  f.hid = ar.f32(rows * m->d_inner);
  return f;
}

// VariancePredictor.forward (+ bucketize / embedding add when bins != NULL) on rows [B][T]  (model/modules.py:242-250, :80-100)
static int run_predictor(cudaStream_t s, const fs2_acoustic_model* m, const fs2_predictor_weights& w, const float* x, int B, int T,
                         const int32_t* lens, float control, const float* target, const float* bins, const float* emb, float* x_acc,
                         float* pred_out, float* h1, float* h2) {
  const int k = m->vp_kernel, D = m->d_model, VF = m->vp_filter;
  if ((m->tc_mask & FS2_TC_PREDICTORS) && w.w_c1_tc && w.w_c2_tc) {   // tensor cores, K-segmented (conv_seg); ReLU applied by the LayerNorm
    FS2_TRY(conv_seg(s, x, B, T, D, w.w_c1_tc, w.b_c1, VF, k, (k - 1) / 2, h1, nullptr, FS2_ACT_NONE, 0.f, nullptr));
    FS2_TRY(ln(s, h1, h2, B, T, VF, w.ln1_g, w.ln1_b, nullptr, 1));
    FS2_TRY(conv_seg(s, h2, B, T, VF, w.w_c2_tc, w.b_c2, VF, k, 1, h1, nullptr, FS2_ACT_NONE, 0.f, nullptr));   // padding=1 is hard-coded upstream
    FS2_TRY(ln(s, h1, h2, B, T, VF, w.ln2_g, w.ln2_b, nullptr, 1));
  } else {
    FS2_TRY(conv(s, x, B, T, D, w.w_c1, nullptr, w.b_c1, VF, k, 1, (k - 1) / 2, FS2_ACT_RELU, 0.f, h1));
    FS2_TRY(ln(s, h1, h2, B, T, VF, w.ln1_g, w.ln1_b, nullptr));
    FS2_TRY(conv(s, h2, B, T, VF, w.w_c2, nullptr, w.b_c2, VF, k, 1, 1, FS2_ACT_RELU, 0.f, h1));  // padding=1 is hard-coded upstream
    FS2_TRY(ln(s, h1, h2, B, T, VF, w.ln2_g, w.ln2_b, nullptr));
  }
  fs2_variance_head_args v{};
  v.h = h2; v.w = w.w_out; v.b = w.b_out; v.B = B; v.L = T; v.C = VF;
  v.lens = lens; v.control = control; v.target = target;
  v.bins = bins; v.n_edges = m->n_bins - 1; v.emb = emb; v.D = D; v.x = x_acc; v.pred_out = pred_out;
  return variance_head(&v, s);
}

// ------------------------------------------------------------------ phase 1
static int encode_impl(const fs2_acoustic_model* m, const fs2_encode_args* a, cudaStream_t s, Arena& ar) {
  const int B = a->B, L = a->L, D = m->d_model, VF = m->vp_filter;
  const size_t rows = (size_t)B * L;
  FftBufs f = fft_bufs(ar, m, rows);
  float* h1 = ar.f32(rows * VF);
  float* h2 = ar.f32(rows * VF);
  if (ar.dry) return FS2_OK;
  if (!f.x || !f.tmp || !f.qkv || !f.ctx || !f.hid || !h1 || !h2) return FS2_ERR_WORKSPACE;
  if (L > m->enc_pos_rows) return FS2_ERR_ARG;

  fs2_embed_args e{a->texts, m->word_emb, m->enc_pos, f.x, B, L, D, m->n_vocab};
  FS2_TRY(embed_positions(&e, s));
  for (int i = 0; i < m->n_enc; i++) FS2_TRY(fft_block(s, m, m->enc[i], f, B, L, a->src_lens, false, 0, (m->tc_mask & FS2_TC_ENCODER) != 0));
  if (m->spk_emb) {
    if (!a->speakers) return FS2_ERR_ARG;
    fs2_rowbias_args r{f.x, m->spk_emb, a->speakers, B, L, D, m->n_speakers};
    FS2_TRY(add_speaker(&r, s));
  }
  // x_adapted starts as the encoder output; pitch / energy embeddings are added in place (modules.py:117-126)
  cudaError_t ce = cudaMemcpyAsync(a->x_adapted, f.x, rows * D * sizeof(float), cudaMemcpyDeviceToDevice, s);
  if (ce != cudaSuccess) return FS2_ERR_CUDA - (int)ce;

  // duration on the un-embedded x; pitch on x; energy on x + pitch embedding.  energy uses p_control (modules.py:124).
  FS2_TRY(run_predictor(s, m, m->dur, a->x_adapted, B, L, a->src_lens, 1.f, nullptr, nullptr, nullptr, a->x_adapted, a->logd_pred, h1, h2));
  if (!m->pitch_frame_level) {
    if (!a->p_pred) return FS2_ERR_ARG;
    FS2_TRY(run_predictor(s, m, m->pitch, a->x_adapted, B, L, a->src_lens, a->p_control, a->p_target, m->pitch_bins, m->pitch_emb,
                          a->x_adapted, a->p_pred, h1, h2));
  }
  if (!m->energy_frame_level) {
    if (!a->e_pred) return FS2_ERR_ARG;
    FS2_TRY(run_predictor(s, m, m->energy, a->x_adapted, B, L, a->src_lens, a->p_control, a->e_target, m->energy_bins, m->energy_emb,
                          a->x_adapted, a->e_pred, h1, h2));
  }

  fs2_durations_args d{};
  d.src = a->d_target ? a->d_target : a->logd_pred; d.use_target = a->d_target != nullptr; d.d_control = a->d_control;
  d.B = B; d.L = L; d.d_rounded = a->d_target ? nullptr : a->d_rounded; d.cum = a->cum_dur; d.mel_lens = a->mel_lens;
  d.mel_lens32 = a->mel_lens32; d.len_stats = a->len_stats;
  FS2_TRY(durations(&d, s));
  if (a->len_stats_host) {
    ce = cudaMemcpyAsync(a->len_stats_host, a->len_stats, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
    if (ce != cudaSuccess) return FS2_ERR_CUDA - (int)ce;
  }
  return FS2_OK;
}

// ------------------------------------------------------------------ phase 2
static int decode_impl(const fs2_acoustic_model* m, const fs2_decode_args* a, cudaStream_t s, Arena& ar) {
  const int B = a->B, T = a->T, D = m->d_model;
  const size_t rows = (size_t)B * T;
  FftBufs f = fft_bufs(ar, m, rows, B, T, (m->tc_mask & FS2_TC_DECODER) != 0);
  int pc = 0;
  for (int i = 0; i < m->n_postnet; i++) pc = pc > m->post_cout[i] ? pc : m->post_cout[i];
  float* pa = ar.f32(rows * pc);
  float* pb = ar.f32(rows * pc);
  if (ar.dry) return FS2_OK;
  if (!f.x || !f.tmp || !f.qkv || !f.ctx || !f.hid || !pa || !pb || (f.att_bytes && !f.att_ws)) return FS2_ERR_WORKSPACE;
  if (T > m->dec_pos_rows) return FS2_ERR_ARG;

  const bool frame_level = m->pitch_frame_level || m->energy_frame_level;
  fs2_length_regulate_args lr{a->x_adapted, a->cum_dur, frame_level ? nullptr : m->dec_pos, f.x, B, a->L, T, D};
  FS2_TRY(length_regulate(&lr, s));
  if (frame_level) {                                   // frame-level pitch / energy (model/modules.py:139-148), then the position add
    float* h1 = f.hid;                                 // [rows][d_inner] is free here and d_inner >= 2 * vp_filter is checked below
    float* h2 = f.hid + rows * m->vp_filter;
    if ((size_t)m->d_inner < 2 * (size_t)m->vp_filter) return FS2_ERR_UNSUPPORTED;
    if (m->pitch_frame_level) {
      if (!a->p_pred_frames) return FS2_ERR_ARG;
      FS2_TRY(run_predictor(s, m, m->pitch, f.x, B, T, a->mel_mask_lens, a->p_control, a->p_target_frames, m->pitch_bins, m->pitch_emb, f.x,
                            a->p_pred_frames, h1, h2));
    }
    if (m->energy_frame_level) {
      if (!a->e_pred_frames) return FS2_ERR_ARG;
      FS2_TRY(run_predictor(s, m, m->energy, f.x, B, T, a->mel_mask_lens, a->p_control, a->e_target_frames, m->energy_bins, m->energy_emb, f.x,
                            a->e_pred_frames, h1, h2));
    }
    FS2_TRY(add_positions(f.x, m->dec_pos, B, T, D, s));
  }
  for (int i = 0; i < m->n_dec; i++) FS2_TRY(fft_block(s, m, m->dec[i], f, B, T, a->mel_mask_lens, (m->tc_mask & FS2_TC_DECODER) != 0,
                                                     (m->tc_mask & FS2_TC_DECODER_F8) ? FS2_TC_VARIANT_F8 : 0));
  const bool tcp = (m->tc_mask & FS2_TC_POSTNET) != 0;
  const unsigned tcpv = (m->tc_mask & FS2_TC_POSTNET_F8) ? FS2_TC_VARIANT_F8 : 0;
  FS2_TRY(conv(s, f.x, B, T, D, m->w_mel, tcp ? m->w_mel_tc : nullptr, m->b_mel, m->n_mel, 1, 1, 0, FS2_ACT_NONE, 0.f, a->mel, nullptr, FS2_ACT_NONE,
               0.f, 1.f, 0, nullptr, tcpv));
  // PostNet: eval BatchNorm folded into (w, b) by the packer; unmasked, tanh on all but the last (Layers.py:129-137)
  const float* cur = a->mel;
  for (int i = 0; i < m->n_postnet; i++) {
    const bool last = i == m->n_postnet - 1;
    float* dst = last ? a->postnet_mel : ((i & 1) ? pb : pa);
    FS2_TRY(conv(s, cur, B, T, m->post_cin[i], m->w_post[i], tcp ? m->w_post_tc[i] : nullptr, m->b_post[i], m->post_cout[i], m->post_k, 1,
                 (m->post_k - 1) / 2,
                 last ? FS2_ACT_NONE : FS2_ACT_TANH, 0.f, dst, last ? a->mel : nullptr, FS2_ACT_NONE, 0.f, 1.f, 0, nullptr, tcpv));
    cur = dst;
  }
  return FS2_OK;
}

// ------------------------------------------------------------------ vocoder
static int vocoder_impl(const fs2_vocoder_model* m, const fs2_vocoder_args* a, cudaStream_t s, Arena& ar) {
  const int B = a->B, T = a->T;
  size_t per_frame = (size_t)m->c0;  // floats per mel frame of the widest activation
  {
    int up = 1, ch = m->c0;
    for (int i = 0; i < m->n_stages; i++) {
      up *= m->rates[i];
      ch /= 2;
      per_frame = per_frame > (size_t)up * ch ? per_frame : (size_t)up * ch;
    }
  }
  const size_t n = (size_t)B * T * per_frame;
  float* bx = ar.f32(n);
  float* bu = ar.f32(n);
  float* bt = ar.f32(n);
  float* r1 = ar.f32(n);
  float* r2 = ar.f32(n);
  if (ar.dry) return FS2_OK;
  if (!bx || !bu || !bt || !r1 || !r2) return FS2_ERR_WORKSPACE;

  {  // conv_pre reads the (possibly strided) channels-last mel view
    fs2_conv1d_args c{};
    c.x = a->mel; c.x_batch_stride = a->mel_batch_stride; c.x_row_stride = a->mel_row_stride;
    c.B = B; c.T = T; c.Cin = m->n_mel; c.w = m->w_pre; c.w_tc = m->w_pre_tc; c.bias = m->b_pre; c.N = m->c0; c.taps = 7;
    c.dilation = 1; c.pad_left = 3; c.tc_variant = (m->f8_mask & 1) ? FS2_TC_VARIANT_F8 : 0;
    c.alpha = 1.f; c.y = bx; c.y_batch_stride = (int64_t)T * m->c0; c.y_row_stride = m->c0;
    FS2_TRY(conv1d_dispatch(&c, s));
  }
  int Ti = T, C = m->c0;
  const float inv_nk = 1.f / (float)m->n_kernels;
  for (int i = 0; i < m->n_stages; i++) {
    const int u = m->rates[i], Co = C / 2;
    if (m->up_k[i] != 2 * u || (u & 1)) return FS2_ERR_UNSUPPORTED;
    const unsigned tcv = (m->f8_mask & (2 << i)) ? FS2_TC_VARIANT_F8 : 0;
    // ---- lrelu + ConvTranspose1d as two 2-tap phase-group convolutions (hifigan/models.py:152-153)
    for (int g = 0; g < 2; g++) {
      fs2_conv1d_args c{};
      c.x = bx; c.x_batch_stride = (int64_t)Ti * C; c.x_row_stride = C; c.B = B; c.T = Ti; c.Cin = C;
      c.w = g == 0 ? m->w_up_a[i] : m->w_up_b[i];
      c.w_tc = g == 0 ? m->w_up_a_tc[i] : m->w_up_b_tc[i];
      c.bias = m->b_up[i] + (size_t)g * (u / 2) * Co;
      c.N = (u / 2) * Co; c.taps = 2; c.dilation = 1; c.pad_left = g == 0 ? 1 : 0;
      c.in_act = FS2_ACT_LRELU; c.in_slope = 0.1f; c.alpha = 1.f; c.tc_variant = tcv;
      c.y = bu + (size_t)g * (u / 2) * Co; c.y_batch_stride = (int64_t)Ti * u * Co; c.y_row_stride = (int64_t)u * Co;
      FS2_TRY(conv1d_dispatch(&c, s));
    }
    Ti *= u; C = Co;
    // ---- mean of the multi-receptive-field ResBlocks (models.py:154-160, ResBlock.forward :96-103)
    if ((m->fused_mask >> i) & 1) {                    // one persistent kernel for the whole group: intermediates never leave the SM
      if (!tcv) return FS2_ERR_ARG;
      fs2_resstack_args ra{};
      ra.x = bu; ra.y = bx; ra.B = B; ra.N = Ti; ra.C = C; ra.n_kernels = m->n_kernels; ra.n_dil = m->n_dil;
      for (int j = 0; j < m->n_kernels; j++) {
        ra.k[j] = m->rb_k[j];
        for (int d = 0; d < m->n_dil; d++) {
          const int rb = i * m->n_kernels + j;
          ra.dil[j][d] = m->rb_dil[j][d];
          ra.w1_tc[j][d] = m->w_rb1_tc[rb][d]; ra.b1[j][d] = m->b_rb1[rb][d];
          ra.w2_tc[j][d] = m->w_rb2_tc[rb][d]; ra.b2[j][d] = m->b_rb2[rb][d];
        }
      }
      FS2_TRY(resstack(&ra, s));
      continue;
    }
    for (int j = 0; j < m->n_kernels; j++) {
      const int rb = i * m->n_kernels + j, k = m->rb_k[j];
      const float* r = bu;
      const bool pairs = ((m->pair_mask >> i) & 1) && tcv && (C == 32 || C == 64) && k <= m->pair_kmax;
      for (int d = 0; d < m->n_dil; d++) {
        const int dil = m->rb_dil[j][d];
        if (pairs) {                                   // one launch per (dilated conv, conv, +x) pair: the intermediate stays on chip
          const bool lastp = d == m->n_dil - 1;
          float* dstp = lastp ? bx : (r == r1 ? r2 : r1);
          fs2_resstack_args ra{};
          ra.x = r; ra.y = dstp; ra.B = B; ra.N = Ti; ra.C = C; ra.n_kernels = 1; ra.n_dil = 1;
          ra.k[0] = k; ra.dil[0][0] = dil;
          ra.w1_tc[0][0] = m->w_rb1_tc[rb][d]; ra.b1[0][0] = m->b_rb1[rb][d];
          ra.w2_tc[0][0] = m->w_rb2_tc[rb][d]; ra.b2[0][0] = m->b_rb2[rb][d];
          ra.alpha = lastp ? inv_nk : 1.f; ra.accumulate = lastp && j > 0;
          FS2_TRY(resstack(&ra, s));
          r = dstp;
          continue;
        }
        FS2_TRY(conv(s, r, B, Ti, C, m->w_rb1[rb][d], m->w_rb1_tc[rb][d], m->b_rb1[rb][d], C, k, dil, (k * dil - dil) / 2, FS2_ACT_LRELU,
                     0.1f, bt, nullptr, FS2_ACT_LRELU, 0.1f, 1.f, 0, nullptr, tcv));
        const bool last = d == m->n_dil - 1;
        float* dst = last ? bx : (r == r1 ? r2 : r1);
        FS2_TRY(conv(s, bt, B, Ti, C, m->w_rb2[rb][d], m->w_rb2_tc[rb][d], m->b_rb2[rb][d], C, k, 1, (k - 1) / 2, FS2_ACT_NONE, 0.f, dst,
                     r, FS2_ACT_NONE, 0.f, last ? inv_nk : 1.f, last && j > 0, nullptr, tcv));
        r = dst;
      }
    }
  }
  fs2_conv_post_args p{bx, B, Ti, C, m->w_post, m->b_post, 7, 0.01f, a->wav};
  return conv_post(&p, s);
}

}  // namespace fs2

// ====================================================================== extern "C"
using namespace fs2;
#define S(x) ((cudaStream_t)(x))

extern "C" {

int fs2_abi_version(void) { return 8; }
int fs2_conv_tc_block(int N) { return conv_tc_nb(N); }
int fs2_conv_tc_plan(const fs2_conv1d_args* a, int num_sms, int32_t* out) { return conv_tc_plan_query(a, num_sms, out); }
int64_t fs2_kernel_launch_count(void) { return (int64_t)g_launch_count.load(); }
size_t fs2_struct_size(int which) {
  switch (which) {
    case 0: return sizeof(fs2_conv1d_args);
    case 1: return sizeof(fs2_layernorm_args);
    case 2: return sizeof(fs2_attention_args);
    case 3: return sizeof(fs2_embed_args);
    case 4: return sizeof(fs2_rowbias_args);
    case 5: return sizeof(fs2_variance_head_args);
    case 6: return sizeof(fs2_durations_args);
    case 7: return sizeof(fs2_length_regulate_args);
    case 8: return sizeof(fs2_conv_post_args);
    case 9: return sizeof(fs2_acoustic_model);
    case 10: return sizeof(fs2_encode_args);
    case 11: return sizeof(fs2_decode_args);
    case 12: return sizeof(fs2_vocoder_model);
    case 13: return sizeof(fs2_vocoder_args);
    case 14: return sizeof(fs2_resstack_args);
    case 15: return sizeof(fs2_wav_int16_args);
    default: return 0;
  }
}
#ifdef FS2_DEBUG_KNOBS
/* tuning / tracing knobs for scripts/tc_*.py -- compiled in only with -DFS2_DEBUG_KNOBS (FS2_DEBUG_KNOBS=1 python -m fastspeech2_b200.build):
 * the shipped library has no mutable process-wide state behind the ABI */
void fs2_debug_set_tc_trace(long long* buf) { g_tc_trace = buf; }
void fs2_debug_set_tc_pdl(int on) { g_tc_pdl = on; }
void fs2_debug_set_tc_tuning(int sa, int sb, int tps, int grid) { g_tc_tune[0] = sa; g_tc_tune[1] = sb; g_tc_tune[2] = tps; g_tc_tune[3] = grid; }
#endif
int fs2_profile_begin(void) {
  g_prof.clear();
  g_prof_on = true;
  return FS2_OK;
}
int fs2_profile_end(double* ms, double* flops, int64_t* launches) {
  g_prof_on = false;
  if (!ms || !flops || !launches) return FS2_ERR_ARG;
  for (int i = 0; i < FS2_PROF_CLASSES; i++) { ms[i] = 0; flops[i] = 0; launches[i] = 0; }
  int rc = FS2_OK;
  for (auto& r : g_prof) {
    float t = 0.f;
    cudaError_t e = cudaEventSynchronize(r.b);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&t, r.a, r.b);
    if (e != cudaSuccess) rc = FS2_ERR_CUDA - (int)e;
    const int c = (r.cls >= 0 && r.cls < FS2_PROF_CLASSES) ? r.cls : 3;
    ms[c] += t; flops[c] += r.flops; launches[c] += 1;
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  g_prof.clear();
  return rc;
}
const char* fs2_build_info(void) { return "fs2b200 sm_100a (tcgen05 split-FP16 conv + attention GEMMs, fp32 CUDA-core kernels), built " __DATE__ " " __TIME__; }

int fs2_conv1d(const fs2_conv1d_args* a, fs2_stream_t st) { return conv1d_dispatch(a, S(st)); }
int fs2_layernorm(const fs2_layernorm_args* a, fs2_stream_t st) { return layernorm(a, S(st)); }
int fs2_attention(const fs2_attention_args* a, fs2_stream_t st) {
  if (a && a->backend == 1) return attention_gemm(a, a->workspace, a->workspace_bytes, S(st));
  if (a && a->backend == 2) return attention_fused(a, a->workspace, a->workspace_bytes, S(st));
  return attention_simt(a, S(st));
}
size_t fs2_attention_workspace_bytes(int B, int T, int H) {      // enough for either tensor-core backend
  if (!(B > 0 && T > 0 && H > 0)) return 0;
  const size_t g = attention_gemm_workspace(B, T, H), f = attention_fused_workspace(B, T, H);
  return g > f ? g : f;
}
int fs2_embed_positions(const fs2_embed_args* a, fs2_stream_t st) { return embed_positions(a, S(st)); }
int fs2_add_speaker(const fs2_rowbias_args* a, fs2_stream_t st) { return add_speaker(a, S(st)); }
int fs2_variance_head(const fs2_variance_head_args* a, fs2_stream_t st) { return variance_head(a, S(st)); }
int fs2_durations(const fs2_durations_args* a, fs2_stream_t st) { return durations(a, S(st)); }
int fs2_length_regulate(const fs2_length_regulate_args* a, fs2_stream_t st) { return length_regulate(a, S(st)); }
int fs2_conv_post(const fs2_conv_post_args* a, fs2_stream_t st) { return conv_post(a, S(st)); }
int fs2_resstack(const fs2_resstack_args* a, fs2_stream_t st) { return resstack(a, S(st)); }
int fs2_wav_to_int16(const fs2_wav_int16_args* a, fs2_stream_t st) { return wav_to_int16(a, S(st)); }
int fs2_resstack_plan(const fs2_resstack_args* a, int num_sms, int32_t* out) { return out ? resstack_plan(a, num_sms, out) : FS2_ERR_ARG; }
int fs2_add_positions(float* x, const float* pos, int B, int T, int D, fs2_stream_t st) { return add_positions(x, pos, B, T, D, S(st)); }
int fs2_transpose_bct_to_btc(const float* in, float* out, int B, int C, int T, fs2_stream_t st) {
  return transpose_bct_to_btc(in, out, B, C, T, S(st));
}

size_t fs2_encode_workspace_bytes(const fs2_acoustic_model* m, int B, int L) {
  if (!model_ok(m) || B <= 0 || L <= 0) return 0;
  Arena ar(nullptr, 0);
  fs2_encode_args a{};
  a.B = B; a.L = L;
  encode_impl(m, &a, nullptr, ar);
  return ar.off + 256;
}

int fs2_acoustic_encode(const fs2_acoustic_model* m, const fs2_encode_args* a, fs2_stream_t st) {
  if (!model_ok(m) || !a || a->B <= 0 || a->L <= 0) return FS2_ERR_ARG;
  if (!a->texts || !a->src_lens || !a->logd_pred || !a->mel_lens || !a->cum_dur || !a->x_adapted ||
      !a->len_stats || !a->workspace)
    return FS2_ERR_ARG;
  if (!a->d_target && !a->d_rounded) return FS2_ERR_ARG;
  if (m->d_model / m->n_head != 128) return FS2_ERR_UNSUPPORTED;
  Arena ar(a->workspace, a->workspace_bytes);
  return encode_impl(m, a, S(st), ar);
}

size_t fs2_decode_workspace_bytes(const fs2_acoustic_model* m, int B, int T) {
  if (!model_ok(m) || B <= 0 || T <= 0) return 0;
  Arena ar(nullptr, 0);
  fs2_decode_args a{};
  a.B = B; a.T = T;
  decode_impl(m, &a, nullptr, ar);
  return ar.off + 256;
}

int fs2_acoustic_decode(const fs2_acoustic_model* m, const fs2_decode_args* a, fs2_stream_t st) {
  if (!model_ok(m) || !a || a->B <= 0 || a->L <= 0 || a->T <= 0) return FS2_ERR_ARG;
  if (!a->x_adapted || !a->cum_dur || !a->mel_mask_lens || !a->mel || !a->postnet_mel || !a->workspace) return FS2_ERR_ARG;
  if (m->d_model / m->n_head != 128) return FS2_ERR_UNSUPPORTED;
  Arena ar(a->workspace, a->workspace_bytes);
  return decode_impl(m, a, S(st), ar);
}

static bool vocoder_ok(const fs2_vocoder_model* m) {
  if (!(m && m->n_stages > 0 && m->n_stages <= FS2_MAX_STAGES && m->n_kernels > 0 && m->n_kernels <= FS2_MAX_DIL + 4 &&
        m->n_kernels * m->n_stages <= FS2_MAX_RESBLOCKS && m->n_dil > 0 && m->n_dil <= FS2_MAX_DIL && m->c0 > 0 && m->n_mel > 0))
    return false;
  if (m->c0 % (1 << m->n_stages)) return false;                          // channels halve at every stage
  for (int i = 0; i < m->n_stages; i++)
    if (m->rates[i] <= 0 || m->up_k[i] <= 0) return false;
  for (int j = 0; j < m->n_kernels; j++) {
    if (m->rb_k[j] <= 0 || !(m->rb_k[j] & 1)) return false;              // odd kernels: symmetric "same" padding (hifigan/models.py:16-17)
    for (int d = 0; d < m->n_dil; d++)
      if (m->rb_dil[j][d] <= 0) return false;
  }
  return true;
}

size_t fs2_vocoder_workspace_bytes(const fs2_vocoder_model* m, int B, int T) {
  if (!vocoder_ok(m) || B <= 0 || T <= 0) return 0;
  Arena ar(nullptr, 0);
  fs2_vocoder_args a{};
  a.B = B; a.T = T;
  vocoder_impl(m, &a, nullptr, ar);
  return ar.off + 256;
}

int fs2_vocoder_forward(const fs2_vocoder_model* m, const fs2_vocoder_args* a, fs2_stream_t st) {
  if (!vocoder_ok(m) || !a || a->B <= 0 || a->T <= 0 || !a->mel || !a->wav || !a->workspace) return FS2_ERR_ARG;
  Arena ar(a->workspace, a->workspace_bytes);
  return vocoder_impl(m, a, S(st), ar);
}

}  // extern "C"
