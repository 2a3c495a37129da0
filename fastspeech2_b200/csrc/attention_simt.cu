// fp32 CUDA-core flash-style attention for the FFT blocks (transformer/Modules.py:14-25 with the key-padding mask of
// transformer/Models.py:79): never materialises the S x S score matrix (the reference writes 2B*S^2 floats four times).
//
// CTA = 64 queries of one (utterance, head); loops over 64-key tiles up to the utterance's valid length (keys beyond it
// are masked to -inf in the reference, i.e. contribute exactly 0).  Dh = 128.  256 threads as a 16 x 16 grid:
//   S phase : thread (ty,tx) owns queries {ty+16i} x keys {tx+16j}; Q/K rows padded to 132 floats so the interleaved
//             float4 reads are bank-conflict free.
//   PV phase: thread owns queries {ty+16i} x value columns {tx*4..+3, 64+tx*4..+3}; P is parked in the K buffer.
// Online softmax state (running max / sum) is replicated across the 16 tx lanes that share a query row.
#include "common.cuh"

namespace fs2 {

constexpr int ATT_BQ = 64, ATT_BK = 64, ATT_D = 128, ATT_LD = ATT_D + 4, ATT_PLD = ATT_BK + 4;
constexpr size_t ATT_SMEM = (size_t)(ATT_BQ * ATT_LD + ATT_BK * ATT_LD + ATT_BK * ATT_D) * sizeof(float);

__global__ void __launch_bounds__(256, 2) attention_simt_kernel(const fs2_attention_args a) {
  extern __shared__ __align__(16) float smem[];
  float* Qs = smem;                       // [64][132]
  float* Ks = Qs + ATT_BQ * ATT_LD;       // [64][132]  (reused as P [64][68])
  float* Vs = Ks + ATT_BK * ATT_LD;       // [64][128]
  float* Ps = Ks;

  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int q0 = blockIdx.x * ATT_BQ;
  const int h = blockIdx.y, b = blockIdx.z;
  const int D = a.H * ATT_D;              // model width
  const long long row_stride = 3LL * D;
  const float* base = a.qkv + (long long)b * a.T * row_stride;
  const int len = a.key_lens ? min(a.key_lens[b], a.T) : a.T;
  float* out = a.ctx + (long long)b * a.T * D + h * ATT_D;

  if (q0 >= len) {  // whole query tile is padding: the reference zeroes these rows after the LayerNorm
    for (int f = tid; f < ATT_BQ * (ATT_D / 4); f += 256) {
      const int r = f / (ATT_D / 4), c = f % (ATT_D / 4);
      if (q0 + r < a.T) reinterpret_cast<float4*>(out + (long long)(q0 + r) * D)[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    return;
  }

  // Q tile -> smem (rows beyond T read as zero)
  for (int f = tid; f < ATT_BQ * (ATT_D / 4); f += 256) {
    const int r = f / (ATT_D / 4), c = f % (ATT_D / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q0 + r < a.T) v = __ldg(reinterpret_cast<const float4*>(base + (long long)(q0 + r) * row_stride + h * ATT_D) + c);
    *reinterpret_cast<float4*>(Qs + r * ATT_LD + c * 4) = v;
  }

  float m_run[4], l_run[4], o[4][8];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    m_run[i] = -INFINITY;
    l_run[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; j++) o[i][j] = 0.f;
  }

  const int n_tiles = (len + ATT_BK - 1) / ATT_BK;
  for (int kt = 0; kt < n_tiles; kt++) {
    const int k0 = kt * ATT_BK;
    __syncthreads();  // previous tile's P/V fully consumed (and Q stores visible on the first pass)
    for (int f = tid; f < ATT_BK * (ATT_D / 4); f += 256) {
      const int r = f / (ATT_D / 4), c = f % (ATT_D / 4);
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (k0 + r < a.T) {
        const float* rowp = base + (long long)(k0 + r) * row_stride + h * ATT_D;
        kv = __ldg(reinterpret_cast<const float4*>(rowp + D) + c);
        vv = __ldg(reinterpret_cast<const float4*>(rowp + 2 * D) + c);
      }
      *reinterpret_cast<float4*>(Ks + r * ATT_LD + c * 4) = kv;
      *reinterpret_cast<float4*>(Vs + r * ATT_D + c * 4) = vv;
    }
    __syncthreads();

    // ---- S = Q K^T ----
    float s[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) s[i][j] = 0.f;
#pragma unroll 4
    for (int d = 0; d < ATT_D; d += 4) {
      float4 q[4], k[4];
#pragma unroll
      for (int i = 0; i < 4; i++) q[i] = *reinterpret_cast<const float4*>(Qs + (ty + 16 * i) * ATT_LD + d);
#pragma unroll
      for (int j = 0; j < 4; j++) k[j] = *reinterpret_cast<const float4*>(Ks + (tx + 16 * j) * ATT_LD + d);
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          s[i][j] = fmaf(q[i].x, k[j].x, s[i][j]);
          s[i][j] = fmaf(q[i].y, k[j].y, s[i][j]);
          s[i][j] = fmaf(q[i].z, k[j].z, s[i][j]);
          s[i][j] = fmaf(q[i].w, k[j].w, s[i][j]);
        }
    }
    __syncthreads();  // everyone is done reading K before it is overwritten with P

    // ---- online softmax ----
    float scale_o[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int key = k0 + tx + 16 * j;
        s[i][j] = key < len ? s[i][j] * a.scale : -INFINITY;
        mx = fmaxf(mx, s[i][j]);
      }
#pragma unroll
      for (int o2 = 8; o2 > 0; o2 >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o2));
      const float m_new = fmaxf(m_run[i], mx);  // finite: every visited tile has >= 1 valid key
      float psum = 0.f;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const float pv = expf(s[i][j] - m_new);
        psum += pv;
        Ps[(ty + 16 * i) * ATT_PLD + tx + 16 * j] = pv;
      }
#pragma unroll
      for (int o2 = 8; o2 > 0; o2 >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o2);
      scale_o[i] = expf(m_run[i] - m_new);      // exp(-inf) = 0 on the first tile
      l_run[i] = l_run[i] * scale_o[i] + psum;
      m_run[i] = m_new;
    }
    __syncthreads();

    // ---- O = O * scale + P V ----
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 8; j++) o[i][j] *= scale_o[i];
#pragma unroll 2
    for (int kk = 0; kk < ATT_BK; kk += 4) {
      float4 pr[4];
#pragma unroll
      for (int i = 0; i < 4; i++) pr[i] = *reinterpret_cast<const float4*>(Ps + (ty + 16 * i) * ATT_PLD + kk);
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const float4 v0 = *reinterpret_cast<const float4*>(Vs + (kk + u) * ATT_D + tx * 4);
        const float4 v1 = *reinterpret_cast<const float4*>(Vs + (kk + u) * ATT_D + 64 + tx * 4);
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const float pv = u == 0 ? pr[i].x : (u == 1 ? pr[i].y : (u == 2 ? pr[i].z : pr[i].w));
          o[i][0] = fmaf(pv, v0.x, o[i][0]); o[i][1] = fmaf(pv, v0.y, o[i][1]);
          o[i][2] = fmaf(pv, v0.z, o[i][2]); o[i][3] = fmaf(pv, v0.w, o[i][3]);
          o[i][4] = fmaf(pv, v1.x, o[i][4]); o[i][5] = fmaf(pv, v1.y, o[i][5]);
          o[i][6] = fmaf(pv, v1.z, o[i][6]); o[i][7] = fmaf(pv, v1.w, o[i][7]);
        }
      }
    }
  }

#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int q = q0 + ty + 16 * i;
    if (q >= a.T) continue;
    float* orow = out + (long long)q * D;
    if (q >= len) {
      *reinterpret_cast<float4*>(orow + tx * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(orow + 64 + tx * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      continue;
    }
    const float inv = 1.f / l_run[i];
    *reinterpret_cast<float4*>(orow + tx * 4) = make_float4(o[i][0] * inv, o[i][1] * inv, o[i][2] * inv, o[i][3] * inv);
    *reinterpret_cast<float4*>(orow + 64 + tx * 4) = make_float4(o[i][4] * inv, o[i][5] * inv, o[i][6] * inv, o[i][7] * inv);
  }
}

int attention_simt(const fs2_attention_args* a, cudaStream_t s) {
  if (!a || !a->qkv || !a->ctx || a->B <= 0 || a->T <= 0 || a->H <= 0) return FS2_ERR_ARG;
  if (a->Dh != ATT_D) return FS2_ERR_UNSUPPORTED;
  if (!aligned16(a->qkv) || !aligned16(a->ctx)) return FS2_ERR_ARG;
  int derr = FS2_OK;
  DevState* dv = dev_state(&derr);
  if (!dv) return derr;
  FS2_TRY(setup_once(dv->att_simt_ready,
                     [] { return cudaFuncSetAttribute(attention_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ATT_SMEM); }));
  dim3 grid((a->T + ATT_BQ - 1) / ATT_BQ, a->H, a->B);
  prof_before(s);
  attention_simt_kernel<<<grid, 256, ATT_SMEM, s>>>(*a);
  prof_after(s, 1, 4.0 * a->B * a->H * (double)a->T * a->T * ATT_D);  // dense T x T count, as the reference computes it
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

}  // namespace fs2
