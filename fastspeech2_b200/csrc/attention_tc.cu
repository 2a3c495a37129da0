// Self-attention of the decoder FFT blocks on the tensor cores (transformer/Modules.py:14-25, key mask Models.py:79),
// built from the split-FP16 tcgen05 GEMM engine in conv_tc.cu:
//
//   1. pack_kv_tiles : per (utterance, head) re-tile K and V (fp32, inside the packed qkv rows) into the GEMM's weight-tile
//                      image (fp16 hi/lo, 128-byte header) -- K as the [d x keys] operand of S = Q K^T, V as the [keys x d]
//                      operand of O = P V.  Keys are padded to a multiple of 128 with zeros.
//   2. S = Q K^T      : conv_tc GEMM (taps = 1) with per-utterance "weights", one launch per head, fp32 scores [B*H][T][Tk].
//   3. softmax_rows   : one warp per query row, the row lives in registers: scale, key-padding mask (-inf), softmax, in place.
//                      Query rows beyond the utterance length are written as zeros (the reference zeroes them after the
//                      following LayerNorm, transformer/Layers.py:25).
//   4. O = P V        : conv_tc GEMM with C_in = Tk keys, written straight into the head's 128 columns of ctx [B][T][D].
//
// The score matrix is materialised once in fp32 (the reference writes it four times); a fused flash-style tcgen05 kernel
// that keeps S in TMEM is the planned replacement.  The exact fp32 kernel (attention_simt.cu) stays in use for the encoder.
#include "common.cuh"
#include "tc_format.cuh"

namespace fs2 {

int conv1d_tc(const fs2_conv1d_args* a, const float* wt, unsigned variant, cudaStream_t s, long long wt_batch_stride);

constexpr int AT_DH = 128;          // head width
constexpr int AT_NB = 128;          // output-channel block of the GEMM engine for N = 128*k

// Not split_f16 (tc_format.cuh): this split scales, clamps with fminf / fmaxf and then rounds, so a NaN input becomes -65504 where
// the saturating convert of split_f16 keeps the NaN.  Sharing the split would change what both attention backends return for
// non-finite K / V.
__device__ __forceinline__ void split8(const float (&f)[8], float scale, uint4& hi, uint4& lo) {
  uint32_t hw[4], lw[4];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const float a0 = fminf(fmaxf(f[2 * j] * scale, -65504.f), 65504.f);
    const float a1 = fminf(fmaxf(f[2 * j + 1] * scale, -65504.f), 65504.f);
    const __half2 h2 = __floats2half2_rn(a0, a1);
    const float2 hf = __half22float2(h2);
    const __half2 l2 = __floats2half2_rn(a0 - hf.x, a1 - hf.y);
    hw[j] = *reinterpret_cast<const uint32_t*>(&h2);
    lw[j] = *reinterpret_cast<const uint32_t*>(&l2);
  }
  hi = make_uint4(hw[0], hw[1], hw[2], hw[3]);
  lo = make_uint4(lw[0], lw[1], lw[2], lw[3]);
}

// K tiles: GEMM weights W[c = d][n = key], layout  header | [key/128][d/16][hi|lo][2 chunks][128 keys][8 halfs]
__device__ __forceinline__ void pack_k_tiles(const float* __restrict__ qkv, unsigned char* __restrict__ tiles, int B, int T, int Tk, int H,
                                             long long tile_stride, long long idx) {   // idx = (bh, key, dchunk)
  const long long total = (long long)B * H * Tk * (AT_DH / 8);
  if (idx >= total) return;
  const int dchunk = (int)(idx % (AT_DH / 8));
  const long long r = idx / (AT_DH / 8);
  const int key = (int)(r % Tk);
  const int bh = (int)(r / Tk);
  const int b = bh / H, h = bh - b * H;
  const int D = H * AT_DH;
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; j++) f[j] = 0.f;
  if (key < T) {
    const float4* src = reinterpret_cast<const float4*>(qkv + ((long long)b * T + key) * 3 * D + D + h * AT_DH + dchunk * 8);
    const float4 u = __ldg(src), v = __ldg(src + 1);
    f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w; f[4] = v.x; f[5] = v.y; f[6] = v.z; f[7] = v.w;
  }
  uint4 hi, lo;
  split8(f, KV_WSCALE, hi, lo);
  unsigned char* base = tiles + (long long)bh * tile_stride;
  if (key == 0 && dchunk == 0) *reinterpret_cast<float*>(base) = 1.f / KV_WSCALE;
  const int nblk = key / AT_NB, nn = key - nblk * AT_NB, kb = dchunk >> 1, chunk = dchunk & 1;
  const size_t b_plane = 2 * AT_NB * 16, stage = 2 * b_plane, kbl = AT_DH / 16;
  unsigned char* dst = base + TC_HDR + ((size_t)nblk * kbl + kb) * stage + ((size_t)chunk * AT_NB + nn) * 16;
  *reinterpret_cast<uint4*>(dst) = hi;
  *reinterpret_cast<uint4*>(dst + b_plane) = lo;
}

// V tiles: GEMM weights W[c = key][n = d], layout  header | [key/16][hi|lo][2 chunks of 8 keys][128 d][8 halfs (keys)]
__device__ __forceinline__ void pack_v_tiles(const float* __restrict__ qkv, unsigned char* __restrict__ tiles, int B, int T, int Tk, int H,
                                             long long tile_stride, long long idx) {   // idx = (bh, key8, d)
  const long long total = (long long)B * H * (Tk / 8) * AT_DH;
  if (idx >= total) return;
  const int d = (int)(idx % AT_DH);
  const long long r = idx / AT_DH;
  const int k8 = (int)(r % (Tk / 8));
  const int bh = (int)(r / (Tk / 8));
  const int b = bh / H, h = bh - b * H;
  const int D = H * AT_DH;
  float f[8];
#pragma unroll
  for (int e = 0; e < 8; e++) {
    const int key = k8 * 8 + e;
    f[e] = key < T ? __ldg(qkv + ((long long)b * T + key) * 3 * D + 2 * D + h * AT_DH + d) : 0.f;
  }
  uint4 hi, lo;
  split8(f, KV_WSCALE, hi, lo);
  unsigned char* base = tiles + (long long)bh * tile_stride;
  if (k8 == 0 && d == 0) *reinterpret_cast<float*>(base) = 1.f / KV_WSCALE;
  const int kb = k8 >> 1, chunk = k8 & 1;
  const size_t b_plane = 2 * AT_NB * 16, stage = 2 * b_plane;
  unsigned char* dst = base + TC_HDR + (size_t)kb * stage + ((size_t)chunk * AT_NB + d) * 16;
  *reinterpret_cast<uint4*>(dst) = hi;
  *reinterpret_cast<uint4*>(dst + b_plane) = lo;
}

// One launch writes both operand-tile sets: blocks [0, k_blocks) the K tiles, the rest the V tiles.
__global__ void pack_kv_tiles_kernel(const float* __restrict__ qkv, unsigned char* __restrict__ kt, unsigned char* __restrict__ vt, int B, int T,
                                     int Tk, int H, long long tile_stride, unsigned k_blocks) {
  if (blockIdx.x < k_blocks) pack_k_tiles(qkv, kt, B, T, Tk, H, tile_stride, (long long)blockIdx.x * blockDim.x + threadIdx.x);
  else pack_v_tiles(qkv, vt, B, T, Tk, H, tile_stride, (long long)(blockIdx.x - k_blocks) * blockDim.x + threadIdx.x);
}

// In-place row softmax of S [B*H][T][Tk] with scale and key-padding mask; one warp per row, row held in registers.
template <int CHUNKS>   // 128-key chunks per row held in registers (Tk <= 128*CHUNKS)
__global__ void softmax_rows_kernel(float* __restrict__ S, int B, int T, int Tk, int H, const int* __restrict__ key_lens, float scale) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= (long long)B * H * T) return;
  const int lane = threadIdx.x & 31;
  const int t = (int)(row % T);
  const int b = (int)(row / ((long long)T * H));
  const int len = key_lens ? min(key_lens[b], T) : T;
  float4* p = reinterpret_cast<float4*>(S + row * Tk);
  const int n4 = Tk / 4;                               // float4 per row
  if (t >= len) {
    for (int c = lane; c < n4; c += 32) p[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  float4 v[CHUNKS];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < CHUNKS; i++) {
    const int c = lane + i * 32;
    v[i] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    if (c < n4) {
      const float4 u = p[c];
      const int k0 = c * 4;
      v[i].x = k0 + 0 < len ? u.x * scale : -INFINITY;
      v[i].y = k0 + 1 < len ? u.y * scale : -INFINITY;
      v[i].z = k0 + 2 < len ? u.z * scale : -INFINITY;
      v[i].w = k0 + 3 < len ? u.w * scale : -INFINITY;
      mx = fmaxf(mx, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < CHUNKS; i++) {
    v[i].x = expf(v[i].x - mx); v[i].y = expf(v[i].y - mx); v[i].z = expf(v[i].z - mx); v[i].w = expf(v[i].w - mx);
    sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
#pragma unroll
  for (int i = 0; i < CHUNKS; i++) {
    const int c = lane + i * 32;
    if (c < n4) p[c] = make_float4(v[i].x * inv, v[i].y * inv, v[i].z * inv, v[i].w * inv);
  }
}

// K / V operand tiles of every (utterance, head) for the GEMM engine (also used by the fused kernel, attention_fused.cu)
int pack_kv_tiles(const fs2_attention_args* a, unsigned char* kt, unsigned char* vt, long long tstride, cudaStream_t s) {
  const int B = a->B, T = a->T, H = a->H;
  const int Tk = (T + 127) / 128 * 128;
  const long long nk = (long long)B * H * Tk * (AT_DH / 8), nv = (long long)B * H * (Tk / 8) * AT_DH;
  const unsigned kb = (unsigned)((nk + 255) / 256), vb = (unsigned)((nv + 255) / 256);
  prof_before(s);
  pack_kv_tiles_kernel<<<kb + vb, 256, 0, s>>>(a->qkv, kt, vt, B, T, Tk, H, tstride, kb);
  prof_after(s, 1, 0.0);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

size_t attention_gemm_workspace(int B, int T, int H) {
  const int Tk = (T + 127) / 128 * 128;
  const size_t s_bytes = ((size_t)B * H * T * Tk * sizeof(float) + 255) & ~(size_t)255;
  const size_t tile_bytes = ((size_t)B * H * kv_tile_stride(Tk) + 255) & ~(size_t)255;
  return s_bytes + 2 * tile_bytes + 256;
}

int attention_gemm(const fs2_attention_args* a, void* ws, size_t ws_bytes, cudaStream_t s) {
  if (!a || !a->qkv || !a->ctx || !ws || a->B <= 0 || a->T <= 0 || a->H <= 0) return FS2_ERR_ARG;
  if (a->Dh != AT_DH) return FS2_ERR_UNSUPPORTED;
  const int B = a->B, T = a->T, H = a->H, D = H * AT_DH;
  const int Tk = (T + 127) / 128 * 128;
  if (Tk > 128 * 32) return FS2_ERR_UNSUPPORTED;       // softmax keeps a row in registers
  if (ws_bytes < attention_gemm_workspace(B, T, H)) return FS2_ERR_WORKSPACE;
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  float* S = reinterpret_cast<float*>(base);
  const size_t s_bytes = ((size_t)B * H * T * Tk * sizeof(float) + 255) & ~(size_t)255;
  const long long tstride = kv_tile_stride(Tk);
  const size_t tile_bytes = ((size_t)B * H * tstride + 255) & ~(size_t)255;
  unsigned char* kt = reinterpret_cast<unsigned char*>(base + s_bytes);
  unsigned char* vt = kt + tile_bytes;

  FS2_TRY(pack_kv_tiles(a, kt, vt, tstride, s));
  for (int h = 0; h < H; h++) {                        // S_h = Q_h K_h^T
    fs2_conv1d_args c{};
    c.x = a->qkv + h * AT_DH; c.x_batch_stride = (int64_t)T * 3 * D; c.x_row_stride = 3 * D;
    c.B = B; c.T = T; c.Cin = AT_DH; c.N = Tk; c.taps = 1; c.dilation = 1; c.pad_left = 0; c.alpha = 1.f;
    c.y = S + (size_t)h * T * Tk; c.y_batch_stride = (int64_t)H * T * Tk; c.y_row_stride = Tk;
    FS2_TRY(conv1d_tc(&c, reinterpret_cast<const float*>(kt + (size_t)h * tstride), 0, s, (long long)H * tstride));
  }
  {
    const long long rows = (long long)B * H * T;
    const unsigned grid = (unsigned)((rows + 7) / 8);
    const int chunks = Tk / 128;
    prof_before(s);
    if (chunks <= 4) softmax_rows_kernel<4><<<grid, 256, 0, s>>>(S, B, T, Tk, H, a->key_lens, a->scale);
    else if (chunks <= 8) softmax_rows_kernel<8><<<grid, 256, 0, s>>>(S, B, T, Tk, H, a->key_lens, a->scale);
    else if (chunks <= 16) softmax_rows_kernel<16><<<grid, 256, 0, s>>>(S, B, T, Tk, H, a->key_lens, a->scale);
    else softmax_rows_kernel<32><<<grid, 256, 0, s>>>(S, B, T, Tk, H, a->key_lens, a->scale);
    prof_after(s, 1, 0.0);
    FS2_LAUNCH_CHECK();
  }
  for (int h = 0; h < H; h++) {                        // ctx_h = P_h V_h
    fs2_conv1d_args c{};
    c.x = S + (size_t)h * T * Tk; c.x_batch_stride = (int64_t)H * T * Tk; c.x_row_stride = Tk;
    c.B = B; c.T = T; c.Cin = Tk; c.N = AT_DH; c.taps = 1; c.dilation = 1; c.pad_left = 0; c.alpha = 1.f;
    c.y = a->ctx + h * AT_DH; c.y_batch_stride = (int64_t)T * D; c.y_row_stride = D;
    FS2_TRY(conv1d_tc(&c, reinterpret_cast<const float*>(vt + (size_t)h * tstride), 0, s, (long long)H * tstride));
  }
  return FS2_OK;
}

}  // namespace fs2
