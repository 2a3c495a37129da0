/* fs2b200.h -- C ABI of the B200-native FastSpeech2 + HiFi-GAN inference path.
 *
 * The reference (ming024/FastSpeech2) has no FFI: its "plugin API" for this path is two nn.Module
 * classes.  This library is what a native binding underneath those two classes calls:
 *
 *   fs2_acoustic_encode  + fs2_acoustic_decode   replace  model.fastspeech2.FastSpeech2.forward
 *                                                 (model/fastspeech2.py:43-110; split at the one
 *                                                 data-dependent shape, max(mel_len), modules.py:136)
 *   fs2_vocoder_forward                           replaces hifigan.models.Generator.forward
 *                                                 (hifigan/models.py:149-165)
 *
 * plus one entry point per fused operator (used by the model-level calls and by the parity tests):
 *
 *   fs2_embed_positions   transformer/Models.py:89-91        fs2_conv1d        nn.Conv1d / nn.Linear / ConvTranspose1d call sites
 *   fs2_attention         transformer/Modules.py:14-25       fs2_layernorm     nn.LayerNorm + masked_fill (Layers.py:25,28)
 *   fs2_variance_head     model/modules.py:80-100,:246-250   fs2_durations     model/modules.py:132-135,:185-187
 *   fs2_length_regulate   model/modules.py:167-194           fs2_conv_post     hifigan/models.py:161-163
 *
 * Conventions: every pointer is a DEVICE pointer unless named *_host; activations are fp32,
 * channels-last ([B][T][C], C contiguous); the library never allocates, frees or synchronises --
 * the caller provides outputs and a workspace and owns the stream.  Return value: FS2_OK or a
 * negative error; a CUDA launch error e is returned as FS2_ERR_CUDA - e.  No exceptions, no exit().
 */
#ifndef FS2B200_H
#define FS2B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* fs2_stream_t; /* cudaStream_t */

enum {
  FS2_OK = 0,
  FS2_ERR_ARG = -1,         /* null pointer / non-positive size / misaligned pointer */
  FS2_ERR_UNSUPPORTED = -2, /* configuration outside what the kernels specialise on */
  FS2_ERR_WORKSPACE = -3,   /* workspace too small */
  FS2_ERR_CUDA = -1000      /* FS2_ERR_CUDA - cudaError_t */
};

enum { FS2_ACT_NONE = 0, FS2_ACT_RELU = 1, FS2_ACT_TANH = 2, FS2_ACT_LRELU = 3 };
enum { FS2_CONV_AUTO = 0, FS2_CONV_SIMT = 1, FS2_CONV_TC = 2 };
/* which parts of the acoustic model may use the split-FP16 tcgen05 kernel (fs2_acoustic_model.tc_mask) */
enum { FS2_TC_ENCODER = 1, FS2_TC_PREDICTORS = 2, FS2_TC_DECODER = 4, FS2_TC_POSTNET = 8,
       /* the decoder's / PostNet's w_*_tc tiles are in the f16+f8 format (see FS2_TC_VARIANT_F8) */
       FS2_TC_DECODER_F8 = 16, FS2_TC_POSTNET_F8 = 32,
       /* decoder attention through the round-1 GEMM path (scores materialised in HBM) instead of the fused kernel */
       FS2_TC_ATTENTION_GEMM = 64 };
/* fs2_conv1d_args.tc_variant bits.  F8: w_tc holds the two-MMA operand split -- fp16 hi tiles as in the three-MMA split, and in
 * place of the fp16 lo tiles E4M3 tiles [hi * 2^-12 | lo] that one K = 32 kind::f8f6f4 MMA multiplies with the activations'
 * [lo * 2^12 | hi]: y ~ a_hi.w_hi + (a_lo.w_hi + a_hi.w_lo) with the bracket at E4M3 precision (relative error ~2^-16 instead
 * of ~2^-22; 2/3 of the tensor-pipe time and shared-memory operand traffic).  Activations beyond +-448 saturate in the correction. */
enum { FS2_TC_VARIANT_F8 = 1,
       /* w_tc is tiled for 64 output channels per work item (pack_conv_tc(w, nb=64)): the hi*hi term and the two cross terms then
        * accumulate in separate tensor-memory tiles.  Used by the K-segmented encoder / predictor path (see fs2_acoustic_model). */
       FS2_TC_VARIANT_NB64 = 2,
       /* with NB64: w_tc holds taps * (C_in / 256) one-tap tile buffers back to back (packing.pack_conv_tc_segments) and the conv is
        * evaluated K-SEGMENTED inside one launch: every (tile, tap, 256-channel chunk) is a work unit with a fresh 16-step accumulator,
        * the units of a tile run back to back on one CTA and add into y in fp32 round-to-nearest (bias with the first, residual and
        * pad-row mask with the last).  Needs dilation 1, alpha 1, no output activation, C_in % 256 == 0, N % 64 == 0. */
       FS2_TC_VARIANT_SEGMENTED = 4 };

/* Tensor-core weight tiles.  For a conv weight w[taps][Cin][N] with NB = fs2_conv_tc_block(N) output channels per work item,
 * s = a per-layer power of two, hi = fp16(s*w), lo = fp16(s*w - hi), the tiled byte buffer is
 *     128-byte header (float32[0] = 1/s)  |  [N/NB][Cin/16][taps][2: hi,lo][2: 16-byte K chunk][NB][8 halfs]
 * i.e. every (K-block, tap) stage is one contiguous 64*NB-byte smem image (UMMA no-swizzle K-major, fp16), fetched by one
 * cp.async.bulk.  fastspeech2_b200/packing.py::pack_conv_tc builds it. */
int fs2_conv_tc_block(int N); /* 0 when N is not supported by the tensor-core kernel */
struct fs2_conv1d_args;
/* Launch plan the tcgen05 kernel would use for this call on a device with num_sms SMs (pure host logic, no CUDA call, pointers are
 * only checked for alignment): out[12] = {NB, MT (128-row tiles per work item), TG (accumulators per tile), slab stages, weight
 * stages, taps per weight stage, slab rows, TMEM columns, work items per utterance, work items, grid, dynamic shared memory bytes}.
 * Returns FS2_ERR_UNSUPPORTED for shapes the kernel does not take. */
int fs2_conv_tc_plan(const struct fs2_conv1d_args* a, int num_sms, int32_t* out);

#define FS2_MAX_LAYERS 12
#define FS2_MAX_POSTNET 8
#define FS2_MAX_STAGES 8
#define FS2_MAX_RESBLOCKS 32
#define FS2_MAX_DIL 4

/* ------------------------------------------------------------------ operators */

/* y[b,t,n] = (accumulate ? y : 0) + alpha * ( out_act( bias[n] + sum_{j<taps} sum_c in_act(x[b, t + j*dilation - pad_left, c]) * w[j][c][n] ) + res[b,t,n] )
 * rows outside [0,T) read as zero (Conv1d zero padding); rows t >= row_lens[b] are written as exact 0 when row_lens != NULL.
 * Strides are in elements.  Covers nn.Linear (taps=1), nn.Conv1d (any odd k, dilation), and one phase group of
 * ConvTranspose1d (two taps, y_row_stride = u*C_out; see fs2_vocoder_model).
 * Both kernels: Cin % 16 == 0, pointers 16-byte aligned, strides % 4 == 0.  The tcgen05 kernel additionally needs w_tc,
 * N % 16 == 0, x 32-byte aligned with x strides % 8 == 0 (256-bit loads), in_act in {NONE, LRELU with 0 <= slope <= 1} and
 * (taps-1)*dilation <= 256; anything else is served by the exact kernel under FS2_CONV_AUTO and refused (FS2_ERR_UNSUPPORTED)
 * under FS2_CONV_TC.  Activations beyond +-65504 saturate in the fp16 hi/lo split of the tcgen05 kernel. */
typedef struct fs2_conv1d_args {
  const float* x; int64_t x_batch_stride, x_row_stride;
  int B, T, Cin;
  const float* w;    /* [taps][Cin][N] */
  const float* bias; /* [N] or NULL */
  int N, taps, dilation, pad_left;
  const float* w_tc; /* NULL, or the same weights in the tcgen05 tile layout (see "tensor-core weight tiles" below) */
  int backend;       /* FS2_CONV_AUTO: split-FP16 tcgen05 kernel when w_tc is given and the shape qualifies, else the fp32 CUDA-core kernel */
  unsigned tc_variant; /* FS2_TC_VARIANT_* bits describing the format of w_tc */
  int in_act; float in_slope;
  int out_act; float out_slope;
  const float* res; int64_t res_batch_stride, res_row_stride; /* NULL = none */
  float alpha; int accumulate;
  const int32_t* row_lens; /* [B] or NULL */
  float* y; int64_t y_batch_stride, y_row_stride;
} fs2_conv1d_args;
int fs2_conv1d(const fs2_conv1d_args* a, fs2_stream_t stream);

/* y = LayerNorm_C(x or relu(x)) * gamma + beta over the last dim, then rows t >= row_lens[b] := 0.  x,y contiguous [B][T][C]; C%4==0, C<=1024. */
typedef struct fs2_layernorm_args {
  const float* x; float* y; int B, T, C;
  const float* gamma; const float* beta; float eps;
  const int32_t* row_lens; /* [B] or NULL */
  int pre_relu;            /* 1: LayerNorm(relu(x)) -- the predictors' conv -> ReLU -> LayerNorm (model/modules.py:242-250) when the conv left its ReLU to this op */
} fs2_layernorm_args;
int fs2_layernorm(const fs2_layernorm_args* a, fs2_stream_t stream);

/* ctx[b,t,h*Dh+j] = sum_s softmax_s( q[b,t,h,:].k[b,s,h,:] * scale , keys s >= key_lens[b] masked ) * v[b,s,h,j]
 * qkv: [B][T][3*H*Dh] rows laid out q|k|v, heads contiguous inside each.  Dh must be 128.  Query rows t >= key_lens[b] are written as 0
 * (the reference zeroes them after the following LayerNorm, transformer/Layers.py:25). */
typedef struct fs2_attention_args {
  const float* qkv; float* ctx; int B, T, H, Dh;
  const int32_t* key_lens; float scale;
  int backend;                  /* 0 = exact fp32 flash-style kernel; 1 = tensor-core GEMMs + row softmax (scores in HBM, T <= 4096); 2 = ONE fused
                                   tcgen05 kernel (QK^T, softmax, PV; scores stay in tensor memory, any T).  1 and 2 need the workspace */
  void* workspace; size_t workspace_bytes;   /* backend 1 only: >= fs2_attention_workspace_bytes(B, T, H) */
} fs2_attention_args;
int fs2_attention(const fs2_attention_args* a, fs2_stream_t stream);
size_t fs2_attention_workspace_bytes(int B, int T, int H);

/* y[b,l,:] = table[ids[b,l]] + pos[l]   (+ spk[speakers[b]] when spk != NULL: not used by the encoder, kept for tests) */
typedef struct fs2_embed_args {
  const int64_t* ids; const float* table; const float* pos; float* y; int B, L, D, n_vocab;
} fs2_embed_args;
int fs2_embed_positions(const fs2_embed_args* a, fs2_stream_t stream);

/* x[b,l,:] += table[idx[b]]  for every l < L (padded rows included, model/fastspeech2.py:68-71) */
typedef struct fs2_rowbias_args { float* x; const float* table; const int64_t* idx; int B, L, D, n_rows; } fs2_rowbias_args;
int fs2_add_speaker(const fs2_rowbias_args* a, fs2_stream_t stream);

/* pred[b,l] = (h[b,l,:].w + *b), 0 where l >= lens[b]; if bins != NULL:
 *   v = target ? target[b,l] : pred*control (pred_out then holds the scaled value),  i = #edges < v (torch.bucketize right=False),
 *   x[b,l,:] += emb[i]. */
typedef struct fs2_variance_head_args {
  const float* h; const float* w; const float* b; int B, L, C;
  const int32_t* lens; float control; const float* target;
  const float* bins; int n_edges; const float* emb; int D; float* x;
  float* pred_out;
} fs2_variance_head_args;
int fs2_variance_head(const fs2_variance_head_args* a, fs2_stream_t stream);

/* d = use_target ? src[b,l] : max(rint(exp(src[b,l]) - 1) * d_control, 0); reps = max((int)d, 0);
 * cum[b,l] = inclusive prefix sum of reps; mel_lens[b] = cum[b,L-1]; len_stats[0] = max_b mel_lens, [1] = sum_b mel_lens,
 * [2] = number of non-finite / > 1e6 durations (those contribute 0 frames; the reference raises on them).  The call zeroes len_stats.
 * max() keeps a NaN, like torch.clamp(min=0): a NaN log-duration is written to d_rounded as NaN and counted in len_stats[2]. */
typedef struct fs2_durations_args {
  const float* src; int use_target; float d_control; int B, L;
  float* d_rounded;     /* [B][L] or NULL */
  int32_t* cum;         /* [B][L] */
  int64_t* mel_lens;    /* [B] */
  int32_t* mel_lens32;  /* [B] or NULL */
  int32_t* len_stats;   /* [3] */
} fs2_durations_args;
int fs2_durations(const fs2_durations_args* a, fs2_stream_t stream);

/* y[b,t,:] = (t < cum[b,L-1] ? x[b, upper_bound(cum[b,:], t), :] : 0) + (pos ? pos[t,:] : 0),  t < T */
typedef struct fs2_length_regulate_args {
  const float* x; const int32_t* cum; const float* pos; float* y; int B, L, T, D;
} fs2_length_regulate_args;
int fs2_length_regulate(const fs2_length_regulate_args* a, fs2_stream_t stream);

/* wav[b,t] = tanh( *bias + sum_{j<taps} sum_c lrelu_slope(x[b,t+j-pad,c]) * w[j][c] )   (hifigan/models.py:161-163) */
typedef struct fs2_conv_post_args {
  const float* x; int B, T, C; const float* w; const float* bias; int taps; float in_slope; float* wav;
} fs2_conv_post_args;
int fs2_conv_post(const fs2_conv_post_args* a, fs2_stream_t stream);

/* HiFi-GAN multi-receptive-field ResBlock group of one upsample stage as ONE persistent kernel (hifigan/models.py:154-160, ResBlock.forward
 * :96-103):   y = (1/n_kernels) * sum_j R_j(x),   R_j: x <- conv_{k_j,1}( lrelu( conv_{k_j,dil_jd}( lrelu(x) ) + b1 ) ) + b2 + x  for d = 0..n_dil-1,
 * lrelu slope 0.1, "same" zero padding at the utterance ends.  x, y: contiguous [B][N][C], C in {32, 64} (the 64- / 32-channel stages);
 * every intermediate stays in shared / tensor memory (halo recompute), weights are the f16+f8 tiles of the per-layer kernel
 * (FS2_TC_VARIANT_F8 with N = C: pack_conv_tc(w, f8=True)).  (k-1)*dil/2 <= 32 per conv.  Other shapes: FS2_ERR_UNSUPPORTED.
 * x and y must not overlap (work items re-read halo rows of x): FS2_ERR_ARG. */
typedef struct fs2_resstack_args {
  const float* x; float* y; int B, N, C;
  int n_kernels, n_dil;
  int k[FS2_MAX_DIL + 4]; int dil[FS2_MAX_DIL + 4][FS2_MAX_DIL];
  const float *w1_tc[FS2_MAX_DIL + 4][FS2_MAX_DIL], *b1[FS2_MAX_DIL + 4][FS2_MAX_DIL];   /* dilated conv of each pair */
  const float *w2_tc[FS2_MAX_DIL + 4][FS2_MAX_DIL], *b2[FS2_MAX_DIL + 4][FS2_MAX_DIL];   /* dilation-1 conv of each pair */
  float alpha;     /* weight of every kernel size's result; <= 0: 1/n_kernels (the mean) */
  int accumulate;  /* 1: y += ... (also for the first kernel size) instead of y = ...; with n_kernels = n_dil = 1 the call is ONE fused
                      conv pair  y (+)= alpha * (conv_k,1(lrelu(conv_k,d(lrelu(x)))) + x)  -- the per-pair mode of the 64-channel stage */
} fs2_resstack_args;
int fs2_resstack(const fs2_resstack_args* a, fs2_stream_t stream);
/* launch plan (pure host logic): out[12] = {128-row tiles per slab, halo rows per side, output rows per work item, work items, grid,
 * weight ring stages, dynamic shared memory bytes, TMEM columns, rows per output TMA box, output boxes per tile, conv taps per weight stage,
 * independent-tile mode (single kernel size with a small halo: every 128-row tile carries its own halo)} */
int fs2_resstack_plan(const fs2_resstack_args* a, int num_sms, int32_t* out);

/* out[b,t] = t < lens[b] ? (int16) trunc(wav[b,t] * scale) : 0   -- the device half of utils.model.vocoder_infer (utils/model.py:82-90:
 * `(wavs.cpu().numpy() * max_wav_value).astype("int16")` then `wavs[i][:lengths[i]]`): 2 bytes per sample cross PCIe instead of 4, the
 * trim is fused, and the copy can be asynchronous.  lens (samples, int64, device) may be NULL; lens[b] < 0 keeps nothing, > N keeps all.
 * Values beyond int16 wrap like the reference's numpy cast: trunc to int32, keep the low 16 bits (wav = 1.0 -> -32768); NaN, +-inf and
 * values outside int32 give 0. */
typedef struct fs2_wav_int16_args {
  const float* wav; int64_t wav_batch_stride; int B; int64_t N;
  const int64_t* lens; float scale; int16_t* out; /* [B][N] contiguous */
} fs2_wav_int16_args;
int fs2_wav_to_int16(const fs2_wav_int16_args* a, fs2_stream_t stream);

/* x[b,t,:] += pos[t,:]   (decoder position add when the length regulator could not fuse it: frame-level variance configs) */
int fs2_add_positions(float* x, const float* pos, int B, int T, int D, fs2_stream_t stream);

/* out[b,t,c] = in[b,c,t]  (mel [B,80,T] -> channels-last) */
int fs2_transpose_bct_to_btc(const float* in, float* out, int B, int C, int T, fs2_stream_t stream);

/* ------------------------------------------------------------------ acoustic model (FastSpeech2.forward) */

typedef struct fs2_fft_block_weights {
  const float *w_qkv, *b_qkv;   /* [D][3D], [3D]   (w_qs|w_ks|w_vs transposed and concatenated) */
  const float *w_o, *b_o;       /* [D][D]          (fc) */
  const float *ln1_g, *ln1_b;
  const float *w_1, *b_1;       /* [k1][D][F]      (pos_ffn.w_1) */
  const float *w_2, *b_2;       /* [k2][F][D] */
  const float *ln2_g, *ln2_b;
  const float *w_qkv_tc, *w_o_tc, *w_1_tc, *w_2_tc; /* tensor-core tiles of the four weights, or NULL */
} fs2_fft_block_weights;

typedef struct fs2_predictor_weights {
  const float *w_c1, *b_c1, *ln1_g, *ln1_b; /* [k][D][F] */
  const float *w_c2, *b_c2, *ln2_g, *ln2_b; /* [k][F][F] */
  const float *w_out, *b_out;               /* [F], [1] */
  const float *w_c1_tc, *w_c2_tc;           /* tensor-core tiles of the two convs (three-MMA split format), or NULL */
} fs2_predictor_weights;

/* Encoder / predictors on the tensor cores (tc_mask bits FS2_TC_ENCODER / FS2_TC_PREDICTORS): these layers feed the discrete duration and
 * pitch / energy bucket decisions, where the truncating tensor-core accumulator of a long K loop (432 accumulation steps for the k = 9
 * conv) costs 5x the error of the fp32 CUDA-core kernel (profiles/r02/flip_census_*.jsonl).  They therefore run K-SEGMENTED: every
 * (tap, 256-input-channel) slice is its own launch of 16 K-steps whose hi*hi term has its own accumulator (FS2_TC_VARIANT_NB64), and the
 * slices are summed in fp32 round-to-nearest by the epilogue's accumulate path.  Their w_*_tc pointers then hold
 * taps * (C_in / 256) tile buffers back to back (segment (tap, kc) at index tap * (C_in/256) + kc, each 128 + 1024 * N bytes:
 * packing.pack_conv_tc_segments). */
typedef struct fs2_acoustic_model {
  int d_model, n_head, d_inner, k1, k2, n_enc, n_dec, n_mel;
  int vp_filter, vp_kernel, n_bins, n_vocab, n_speakers;
  int enc_pos_rows, dec_pos_rows;            /* rows available in the position tables */
  int tc_mask;                               /* FS2_TC_* bits; parts not selected run the fp32 CUDA-core kernels */
  int pitch_frame_level, energy_frame_level; /* 0 = phoneme-level predictor (before the length regulator), 1 = frame-level (after it): model/modules.py:117-126 vs :139-148 */
  const float *word_emb, *enc_pos, *dec_pos, *spk_emb;
  fs2_fft_block_weights enc[FS2_MAX_LAYERS], dec[FS2_MAX_LAYERS];
  fs2_predictor_weights dur, pitch, energy;
  const float *pitch_bins, *energy_bins, *pitch_emb, *energy_emb;
  const float *w_mel, *b_mel;                /* [D][n_mel] */
  int n_postnet, post_k;
  int post_cin[FS2_MAX_POSTNET], post_cout[FS2_MAX_POSTNET];
  const float *w_post[FS2_MAX_POSTNET], *b_post[FS2_MAX_POSTNET]; /* BatchNorm folded in: [k][cin][cout] */
  const float *w_mel_tc, *w_post_tc[FS2_MAX_POSTNET];             /* tensor-core tiles or NULL */
} fs2_acoustic_model;

/* Phase 1: encoder + speaker add + variance adaptor up to the duration prefix sums. */
typedef struct fs2_encode_args {
  int B, L;
  const int64_t* texts;      /* [B][L] */
  const int64_t* speakers;   /* [B] (ignored when the model has no speaker table) */
  const int32_t* src_lens;   /* [B] */
  float p_control, e_control, d_control;
  const float *p_target, *e_target, *d_target; /* [B][L] or NULL */
  float *p_pred, *e_pred, *logd_pred, *d_rounded; /* [B][L] outputs (d_rounded unused with d_target) */
  int64_t* mel_lens;         /* [B] */
  int32_t* mel_lens32;       /* [B] */
  int32_t* cum_dur;          /* [B][L] */
  float* x_adapted;          /* [B][L][D]: input of the length regulator */
  int32_t* len_stats;        /* device [3]: max and sum of mel_lens, count of non-finite durations */
  int32_t* len_stats_host;   /* pinned host [3] or NULL: async D2H copy is enqueued on the stream */
  void* workspace; size_t workspace_bytes;
} fs2_encode_args;
size_t fs2_encode_workspace_bytes(const fs2_acoustic_model* m, int B, int L);
int fs2_acoustic_encode(const fs2_acoustic_model* m, const fs2_encode_args* a, fs2_stream_t stream);

/* Phase 2: length regulator + decoder + mel_linear + PostNet (+ residual). */
typedef struct fs2_decode_args {
  int B, L, T;
  const float* x_adapted; const int32_t* cum_dur;
  const int32_t* mel_mask_lens;  /* [B]: rows t >= len are padding for the decoder masks */
  float p_control;               /* used by frame-level pitch AND energy (the reference passes p_control to both, modules.py:146) */
  const float *p_target_frames, *e_target_frames; /* [B][T] or NULL (frame-level configs, teacher forcing) */
  float *p_pred_frames, *e_pred_frames;           /* [B][T] outputs, required for the predictors configured frame-level */
  float* mel; float* postnet_mel; /* [B][T][n_mel] */
  void* workspace; size_t workspace_bytes;
} fs2_decode_args;
size_t fs2_decode_workspace_bytes(const fs2_acoustic_model* m, int B, int T);
int fs2_acoustic_decode(const fs2_acoustic_model* m, const fs2_decode_args* a, fs2_stream_t stream);

/* ------------------------------------------------------------------ vocoder (hifigan Generator.forward) */

typedef struct fs2_vocoder_model {
  int n_mel, c0, n_stages, n_kernels, n_dil;
  int rates[FS2_MAX_STAGES], up_k[FS2_MAX_STAGES];
  int rb_k[FS2_MAX_DIL + 4]; int rb_dil[FS2_MAX_DIL + 4][FS2_MAX_DIL];
  const float *w_pre, *b_pre;                                   /* [7][n_mel][c0] */
  /* ConvTranspose1d(k = 2u) as two 2-tap phase-group convolutions writing [B][T][u*C_out]:
   *   group A: output phases p < u/2 read x[q-1], x[q];  group B: phases p >= u/2 read x[q], x[q+1]. */
  const float *w_up_a[FS2_MAX_STAGES], *w_up_b[FS2_MAX_STAGES]; /* [2][C_in][(u/2)*C_out] */
  const float *b_up[FS2_MAX_STAGES];                            /* [u*C_out] (bias tiled per phase) */
  const float *w_rb1[FS2_MAX_RESBLOCKS][FS2_MAX_DIL], *b_rb1[FS2_MAX_RESBLOCKS][FS2_MAX_DIL]; /* [k][C][C] */
  const float *w_rb2[FS2_MAX_RESBLOCKS][FS2_MAX_DIL], *b_rb2[FS2_MAX_RESBLOCKS][FS2_MAX_DIL];
  const float *w_post, *b_post;                                 /* [7][C_last], [1] */
  /* tensor-core tiles (NULL = CUDA-core kernel for that conv) */
  const float *w_pre_tc, *w_up_a_tc[FS2_MAX_STAGES], *w_up_b_tc[FS2_MAX_STAGES];
  const float *w_rb1_tc[FS2_MAX_RESBLOCKS][FS2_MAX_DIL], *w_rb2_tc[FS2_MAX_RESBLOCKS][FS2_MAX_DIL];
  int f8_mask; /* bit 0: w_pre_tc, bit 1+i: every *_tc tile of stage i is in the f16+f8 format (FS2_TC_VARIANT_F8) */
  int fused_mask; /* bit i: the ResBlock group of stage i runs as one fs2_resstack launch (needs f8_mask bit 1+i and 32 / 64 channels) */
  int pair_mask;  /* bit i: in stage i every (conv_k,d ; conv_k,1 ; +x) pair with k <= pair_kmax runs as one fs2_resstack launch (the
                     HBM-bound small-kernel layers: the pair's intermediate stays on chip); same requirements as fused_mask */
  int pair_kmax;
} fs2_vocoder_model;

typedef struct fs2_vocoder_args {
  int B, T;
  const float* mel; int64_t mel_batch_stride, mel_row_stride; /* channels-last view [B][T][n_mel] */
  float* wav;                                                  /* [B][T*prod(rates)] */
  void* workspace; size_t workspace_bytes;
} fs2_vocoder_args;
size_t fs2_vocoder_workspace_bytes(const fs2_vocoder_model* m, int B, int T);
int fs2_vocoder_forward(const fs2_vocoder_model* m, const fs2_vocoder_args* a, fs2_stream_t stream);

/* ------------------------------------------------------------------ misc */
int fs2_abi_version(void);                 /* bumps when any struct above changes */
int64_t fs2_kernel_launch_count(void);     /* kernels launched by this library since load (process-wide) */
const char* fs2_build_info(void);          /* "sm_100a ..." */
size_t fs2_struct_size(int which);
/* Re-entrancy: the library keeps no mutable process-wide state behind these calls except (a) a per-device table of one-time
 * cudaFuncSetAttribute opt-ins and SM counts, filled under a mutex for the device that is CURRENT when a call is made -- make the
 * device that owns the stream current before calling -- (b) the launch counter above and (c) the profiling state below, which is
 * per host thread.  Tuning / tracing knobs exist only in builds with -DFS2_DEBUG_KNOBS.
 * Per-kernel-class device timing for bench.py's roofline (CUDA events recorded around each launch on the launch stream).
 * Classes: 0 tcgen05 kernels (conv1d implicit GEMM + fused ResBlock group), 1 attention, 2 layernorm, 3 everything else, 4 fp32 CUDA-core conv1d.  begin() arms it, end() synchronises the
 * recorded events, fills ms/flops/launches per class (arrays of FS2_PROF_CLASSES) and disarms.  Not for timed regions. */
#define FS2_PROF_CLASSES 5
int fs2_profile_begin(void);
int fs2_profile_end(double* ms, double* flops, int64_t* launches);         /* sizeof of the i-th struct above, in declaration order (binding self-check) */

#ifdef __cplusplus
}
#endif
#endif /* FS2B200_H */
