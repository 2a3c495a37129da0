// HBM-bound row kernels: embedding + positions, speaker add, LayerNorm + pad mask, variance head
// (row dot + bucketize + embedding add), duration rounding + prefix sum, length-regulator gather,
// conv_post + tanh, and the [B,C,T] -> [B,T,C] transpose.  All fp32, float4 I/O, one warp per row.
#include "common.cuh"

namespace fs2 {

// ------------------------------------------------------------------ embedding + position (Models.py:89-91)
__global__ void embed_kernel(const long long* __restrict__ ids, const float* __restrict__ table,
                             const float* __restrict__ pos, float* __restrict__ y, int B, int L, int D4, int n_vocab) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= B * L) return;
  const int lane = threadIdx.x & 31;
  const int l = row % L;
  long long id = ids[row];
  if (id < 0 || id >= n_vocab) id = 0;  // the reference would raise; stay in bounds
  const float4* e = reinterpret_cast<const float4*>(table) + id * D4;
  const float4* p = reinterpret_cast<const float4*>(pos) + (long long)l * D4;
  float4* o = reinterpret_cast<float4*>(y) + (long long)row * D4;
  for (int c = lane; c < D4; c += 32) {
    const float4 a = __ldg(e + c), q = __ldg(p + c);
    o[c] = make_float4(a.x + q.x, a.y + q.y, a.z + q.z, a.w + q.w);
  }
}

int embed_positions(const fs2_embed_args* a, cudaStream_t s) {
  if (!a || !a->ids || !a->table || !a->pos || !a->y || a->B <= 0 || a->L <= 0 || a->D <= 0) return FS2_ERR_ARG;
  if (a->D % 4) return FS2_ERR_UNSUPPORTED;
  const int rows = a->B * a->L;
  embed_kernel<<<(rows + 7) / 8, 256, 0, s>>>(reinterpret_cast<const long long*>(a->ids), a->table, a->pos, a->y, a->B, a->L,
                                              a->D / 4, a->n_vocab);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ speaker add (fastspeech2.py:68-71)
__global__ void rowbias_kernel(float* __restrict__ x, const float* __restrict__ table, const long long* __restrict__ idx, int B,
                               int L, int D4, int n_rows) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= B * L) return;
  const int lane = threadIdx.x & 31;
  long long id = idx[row / L];
  if (id < 0 || id >= n_rows) id = 0;
  const float4* e = reinterpret_cast<const float4*>(table) + id * D4;
  float4* o = reinterpret_cast<float4*>(x) + (long long)row * D4;
  for (int c = lane; c < D4; c += 32) {
    const float4 a = __ldg(e + c);
    float4 v = o[c];
    v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
    o[c] = v;
  }
}

int add_speaker(const fs2_rowbias_args* a, cudaStream_t s) {
  if (!a || !a->x || !a->table || !a->idx || a->B <= 0 || a->L <= 0 || a->D <= 0) return FS2_ERR_ARG;
  if (a->D % 4) return FS2_ERR_UNSUPPORTED;
  const int rows = a->B * a->L;
  rowbias_kernel<<<(rows + 7) / 8, 256, 0, s>>>(a->x, a->table, reinterpret_cast<const long long*>(a->idx), a->B, a->L, a->D / 4,
                                                a->n_rows);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ x[b,t,:] += pos[t,:]
__global__ void add_positions_kernel(float* __restrict__ x, const float* __restrict__ pos, long long rows, int T, int D4) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int t = (int)(row % T);
  float4* o = reinterpret_cast<float4*>(x) + row * D4;
  const float4* p = reinterpret_cast<const float4*>(pos) + (long long)t * D4;
  for (int c = lane; c < D4; c += 32) {
    const float4 a = __ldg(p + c);
    float4 v = o[c];
    v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
    o[c] = v;
  }
}

int add_positions(float* x, const float* pos, int B, int T, int D, cudaStream_t s) {
  if (!x || !pos || B <= 0 || T <= 0 || D <= 0) return FS2_ERR_ARG;
  if (D % 4) return FS2_ERR_UNSUPPORTED;
  const long long rows = (long long)B * T;
  add_positions_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(x, pos, rows, T, D / 4);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ LayerNorm + pad-row zeroing
// One warp per row; the row lives in registers (C <= 1024), two-pass mean / variance like ATen's CPU kernel.
__global__ void layernorm_kernel(const float* __restrict__ x, float* __restrict__ y, int rows, int T, int C4,
                                 const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                 const int* __restrict__ row_lens, int pre_relu) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  float4* o = reinterpret_cast<float4*>(y) + (long long)row * C4;
  if (row_lens) {
    const int b = row / T, t = row - b * T;
    if (t >= row_lens[b]) {
      for (int c = lane; c < C4; c += 32) o[c] = make_float4(0.f, 0.f, 0.f, 0.f);
      return;
    }
  }
  const float4* in = reinterpret_cast<const float4*>(x) + (long long)row * C4;
  float4 v[8];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int c = lane + i * 32;
    if (c < C4) {
      v[i] = in[c];
      if (pre_relu) v[i] = make_float4(fmaxf(v[i].x, 0.f), fmaxf(v[i].y, 0.f), fmaxf(v[i].z, 0.f), fmaxf(v[i].w, 0.f));
      sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  const float inv_c = 1.f / (float)(C4 * 4);
  const float mean = warp_sum(sum) * inv_c;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int c = lane + i * 32;
    if (c < C4) {
      const float a = v[i].x - mean, b2 = v[i].y - mean, c2 = v[i].z - mean, d = v[i].w - mean;
      sq += (a * a + b2 * b2) + (c2 * c2 + d * d);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) * inv_c + eps);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int c = lane + i * 32;
    if (c < C4) {
      const float4 g = __ldg(g4 + c), bb = __ldg(b4 + c);
      o[c] = make_float4((v[i].x - mean) * rstd * g.x + bb.x, (v[i].y - mean) * rstd * g.y + bb.y,
                         (v[i].z - mean) * rstd * g.z + bb.z, (v[i].w - mean) * rstd * g.w + bb.w);
    }
  }
}

int layernorm(const fs2_layernorm_args* a, cudaStream_t s) {
  if (!a || !a->x || !a->y || !a->gamma || !a->beta || a->B <= 0 || a->T <= 0 || a->C <= 0) return FS2_ERR_ARG;
  if (a->C % 4 || a->C > 1024) return FS2_ERR_UNSUPPORTED;
  const long long rows = (long long)a->B * a->T;
  if (rows > 0x7fffffffLL) return FS2_ERR_UNSUPPORTED;
  prof_before(s);
  layernorm_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(a->x, a->y, (int)rows, a->T, a->C / 4, a->gamma, a->beta, a->eps,
                                                             a->row_lens, a->pre_relu);
  prof_after(s, 2, 0.0);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ variance head (modules.py:80-100, :246-250)
__global__ void variance_head_kernel(const fs2_variance_head_args a) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= a.B * a.L) return;
  const int lane = threadIdx.x & 31;
  const int b = row / a.L, l = row - b * a.L;
  const float4* h = reinterpret_cast<const float4*>(a.h) + (long long)row * (a.C / 4);
  const float4* w = reinterpret_cast<const float4*>(a.w);
  float acc = 0.f;
  for (int c = lane; c < a.C / 4; c += 32) {
    const float4 u = h[c], q = __ldg(w + c);
    acc += (u.x * q.x + u.y * q.y) + (u.z * q.z + u.w * q.w);
  }
  float pred = warp_sum(acc) + __ldg(a.b);
  if (a.lens && l >= a.lens[b]) pred = 0.f;  // masked_fill(mask, 0.0)
  float key = pred;
  if (a.bins) {
    if (a.target) {
      key = a.target[row];
    } else {
      pred = pred * a.control;
      key = pred;
    }
  }
  if (lane == 0) a.pred_out[row] = pred;
  if (!a.bins) return;
  // torch.bucketize(right=False): number of edges strictly below key
  int lo = 0, hi = a.n_edges;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(a.bins + mid) < key) lo = mid + 1; else hi = mid;
  }
  const float4* e = reinterpret_cast<const float4*>(a.emb) + (long long)lo * (a.D / 4);
  float4* x = reinterpret_cast<float4*>(a.x) + (long long)row * (a.D / 4);
  for (int c = lane; c < a.D / 4; c += 32) {
    const float4 q = __ldg(e + c);
    float4 v = x[c];
    v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
    x[c] = v;
  }
}

int variance_head(const fs2_variance_head_args* a, cudaStream_t s) {
  if (!a || !a->h || !a->w || !a->b || !a->pred_out || a->B <= 0 || a->L <= 0 || a->C <= 0) return FS2_ERR_ARG;
  if (a->C % 4) return FS2_ERR_UNSUPPORTED;
  if (a->bins && (!a->emb || !a->x || a->n_edges <= 0 || a->D <= 0 || a->D % 4)) return FS2_ERR_ARG;
  const int rows = a->B * a->L;
  variance_head_kernel<<<(rows + 7) / 8, 256, 0, s>>>(*a);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ durations (modules.py:132-135, :185-187)
// One CTA per utterance: round-half-even (rintf == torch.round), truncate, block-wide inclusive scan.
__global__ void durations_kernel(const fs2_durations_args a) {
  __shared__ int warp_tot[32];
  __shared__ int carry_s;
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nw = blockDim.x >> 5;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < a.L; base += blockDim.x) {
    const int l = base + tid;
    int reps = 0;
    if (l < a.L) {
      const float s = a.src[(long long)b * a.L + l];
      float d;
      if (a.use_target) {
        d = s;
      } else {
        d = rintf(expf(s) - 1.f) * a.d_control;
        d = isnan(d) ? d : fmaxf(d, 0.f);  // torch.clamp(min=0) keeps a NaN (fmaxf alone would turn it into 0 frames, uncounted)
        if (a.d_rounded) a.d_rounded[(long long)b * a.L + l] = d;
      }
      // int() truncation toward zero.  A NaN / inf / absurd duration (the reference raises on int(inf) or dies allocating) is counted
      // in len_stats[2] and contributes no frames, so the caller can fail loudly instead of sizing a gigantic output.
      const bool wild = !(d <= 1.0e6f);
      if (wild) atomicAdd(a.len_stats + 2, 1);
      reps = wild ? 0 : max((int)d, 0);
    }
    int v = reps;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += n;
    }
    if (lane == 31) warp_tot[wid] = v;
    __syncthreads();
    if (wid == 0) {
      int t = lane < nw ? warp_tot[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, t, o);
        if (lane >= o) t += n;
      }
      warp_tot[lane] = t;  // inclusive totals
    }
    __syncthreads();
    const int carry = carry_s;
    const int prefix = carry + (wid ? warp_tot[wid - 1] : 0) + v;
    if (l < a.L) a.cum[(long long)b * a.L + l] = prefix;
    __syncthreads();
    if (tid == 0) carry_s = carry + warp_tot[nw - 1];
    __syncthreads();
  }
  if (tid == 0) {
    const int total = carry_s;
    a.mel_lens[b] = total;
    if (a.mel_lens32) a.mel_lens32[b] = total;
    atomicMax(a.len_stats, total);
    atomicAdd(a.len_stats + 1, total);
  }
}

int durations(const fs2_durations_args* a, cudaStream_t s) {
  if (!a || !a->src || !a->cum || !a->mel_lens || !a->len_stats || a->B <= 0 || a->L <= 0) return FS2_ERR_ARG;
  cudaError_t e = cudaMemsetAsync(a->len_stats, 0, 3 * sizeof(int), s);
  if (e != cudaSuccess) return FS2_ERR_CUDA - (int)e;
  durations_kernel<<<a->B, 256, 0, s>>>(*a);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ length regulator gather (modules.py:167-194)
// One warp per output frame: binary search of the inclusive duration prefix sums (L2/L1 resident, 4*L bytes per utterance),
// then a coalesced float4 copy of the source phoneme row with the decoder position row added (Models.py:158-160).
__global__ void length_regulate_kernel(const fs2_length_regulate_args a) {
  const long long frame = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (frame >= (long long)a.B * a.T) return;
  const int lane = threadIdx.x & 31;
  const int b = (int)(frame / a.T), t = (int)(frame - (long long)b * a.T);
  const int* cum = a.cum + (long long)b * a.L;
  const int total = __ldg(cum + a.L - 1);
  const int D4 = a.D / 4;
  float4* o = reinterpret_cast<float4*>(a.y) + frame * D4;
  const float4* pos = a.pos ? reinterpret_cast<const float4*>(a.pos) + (long long)t * D4 : nullptr;
  if (t >= total) {
    for (int c = lane; c < D4; c += 32) o[c] = pos ? __ldg(pos + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  int lo = 0, hi = a.L - 1;  // first i with cum[i] > t
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(cum + mid) > t) hi = mid; else lo = mid + 1;
  }
  const float4* src = reinterpret_cast<const float4*>(a.x) + ((long long)b * a.L + lo) * D4;
  for (int c = lane; c < D4; c += 32) {
    float4 v = __ldg(src + c);
    if (pos) {
      const float4 q = __ldg(pos + c);
      v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
    }
    o[c] = v;
  }
}

int length_regulate(const fs2_length_regulate_args* a, cudaStream_t s) {
  if (!a || !a->x || !a->cum || !a->y || a->B <= 0 || a->L <= 0 || a->T <= 0 || a->D <= 0) return FS2_ERR_ARG;
  if (a->D % 4) return FS2_ERR_UNSUPPORTED;
  const long long frames = (long long)a->B * a->T;
  prof_before(s);
  length_regulate_kernel<<<(unsigned)((frames + 7) / 8), 256, 0, s>>>(*a);
  prof_after(s, 3, 0.0);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ conv_post + tanh (hifigan/models.py:161-163)
// C_in = 32, one output channel: 128 B per input row, HBM-bound (algorithmic traffic = one read of x).  A CTA stages
// 256 + taps - 1 activated rows in shared memory with fully coalesced float4 loads (row stride C+1 floats -> conflict-free
// column walks), then each thread reduces its own output sample from shared memory.
constexpr int CP_ROWS = 256;
__global__ void __launch_bounds__(CP_ROWS) conv_post_kernel(const fs2_conv_post_args a, int tiles_per_batch) {
  extern __shared__ float cp_smem[];
  const int C = a.C, ld = C + 1, pad = (a.taps - 1) / 2;
  float* wsm = cp_smem;                   // [taps][C]
  float* xs = cp_smem + a.taps * C;       // [CP_ROWS + taps - 1][C + 1]
  const int b = blockIdx.x / tiles_per_batch;
  const int t0 = (blockIdx.x % tiles_per_batch) * CP_ROWS;
  for (int i = threadIdx.x; i < a.taps * C; i += blockDim.x) wsm[i] = a.w[i];
  const int rows = CP_ROWS + a.taps - 1, C4 = C / 4;
  const float4* xb = reinterpret_cast<const float4*>(a.x) + (long long)b * a.T * C4;
  for (int i = threadIdx.x; i < rows * C4; i += blockDim.x) {
    const int r = i / C4, c4 = i - r * C4;
    const int t = t0 - pad + r;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t >= 0 && t < a.T) {
      v = __ldg(xb + (long long)t * C4 + c4);
      v.x = v.x > 0.f ? v.x : v.x * a.in_slope;
      v.y = v.y > 0.f ? v.y : v.y * a.in_slope;
      v.z = v.z > 0.f ? v.z : v.z * a.in_slope;
      v.w = v.w > 0.f ? v.w : v.w * a.in_slope;
    }
    float* d = xs + r * ld + c4 * 4;
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= a.T) return;
  float acc = __ldg(a.bias);
  for (int j = 0; j < a.taps; j++) {
    const float* xr = xs + (threadIdx.x + j) * ld;
    const float* wj = wsm + j * C;
#pragma unroll 8
    for (int c = 0; c < C; c++) acc = fmaf(xr[c], wj[c], acc);
  }
  a.wav[(long long)b * a.T + t] = tanhf(acc);
}

// The generator's own shape (32 channels, 7 taps, hifigan/models.py:131): no shared memory at all.  Eight lanes own one time row (one
// float4 of channels each: a warp reads 4 full 128-byte lines per load instruction, each row exactly once per group plus a 6-row halo),
// the 7 x 4 weights of a lane live in registers, and TAPS sliding accumulators carry the partial sums of the outputs a row contributes to;
// a finished output is reduced over the 8 lanes by three shuffles and every lane keeps one of 8 consecutive samples, so the stores are
// full 32-byte sectors.  (The staged kernel above issues two shared-memory loads per FMA and measured 263 us = 2.0 TB/s at
// B = 16 x 259k samples; this one is bound by the single read of x.)
constexpr int CPF_BLOCKS = 18;                         // row blocks of TAPS rows per 8-lane group
template <int TAPS>
__global__ void __launch_bounds__(256) conv_post_c32_kernel(const fs2_conv_post_args a, int groups_per_batch, long long n_groups) {
  constexpr int PAD = (TAPS - 1) / 2, ROWS = CPF_BLOCKS * TAPS - 2 * PAD;     // output rows per group (120 for 7 taps: a multiple of 8)
  static_assert(ROWS % 8 == 0, "full 8-sample stores");
  const int lane = threadIdx.x & 31, sub = lane & 7;
  long long grp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const bool live = grp < n_groups;                     // groups past the end run along with an empty row range (full-warp shuffles below)
  grp = live ? grp : 0;
  const int b = (int)(grp / groups_per_batch);
  const int t0 = (int)(grp - (long long)b * groups_per_batch) * ROWS;
  const int T = live ? a.T : 0;
  const int tend = min(t0 + ROWS, T);
  float4 w[TAPS];
#pragma unroll
  for (int j = 0; j < TAPS; j++) w[j] = __ldg(reinterpret_cast<const float4*>(a.w + j * 32) + sub);
  const float bias = __ldg(a.bias), slope = a.in_slope;
  const float4* xb = reinterpret_cast<const float4*>(a.x) + (long long)b * a.T * 8 + sub;
  float* wb = a.wav + (long long)b * a.T;
  float s[TAPS];
#pragma unroll
  for (int k = 0; k < TAPS; k++) s[k] = 0.f;
  float keep = 0.f;
#pragma unroll 1
  for (int blk = 0; blk < CPF_BLOCKS; blk++) {
    const int rb = t0 - PAD + blk * TAPS;
    float4 x[TAPS];
#pragma unroll
    for (int i = 0; i < TAPS; i++) {
      const int r = rb + i;
      x[i] = (r >= 0 && r < T) ? __ldg(xb + (long long)r * 8) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < TAPS; i++) {
      float4 v = x[i];
      v.x = v.x > 0.f ? v.x : v.x * slope; v.y = v.y > 0.f ? v.y : v.y * slope;
      v.z = v.z > 0.f ? v.z : v.z * slope; v.w = v.w > 0.f ? v.w : v.w * slope;
      // row r feeds outputs r - PAD .. r + PAD; s[k] is the partial sum of output r - PAD + k, which takes tap TAPS - 1 - k of this row
#pragma unroll
      for (int k = 0; k < TAPS; k++) {
        const float4 wj = w[TAPS - 1 - k];
        s[k] = fmaf(v.x, wj.x, fmaf(v.y, wj.y, fmaf(v.z, wj.z, fmaf(v.w, wj.w, s[k]))));
      }
      float tot = s[0];                                 // output r - PAD has received its last row
#pragma unroll
      for (int k = 0; k + 1 < TAPS; k++) s[k] = s[k + 1];
      s[TAPS - 1] = 0.f;
      tot += __shfl_xor_sync(0xffffffffu, tot, 4);
      tot += __shfl_xor_sync(0xffffffffu, tot, 2);
      tot += __shfl_xor_sync(0xffffffffu, tot, 1);
      const int t = rb + i - PAD;
      if (t >= t0 && t < tend) {
        const int o = (t - t0) & 7;
        if (o == sub) keep = tot;
        if (o == 7 || t == tend - 1) {
          if (sub <= o) wb[t - o + sub] = tanhf(keep + bias);
        }
      }
    }
  }
}

int conv_post(const fs2_conv_post_args* a, cudaStream_t s) {
  if (!a || !a->x || !a->w || !a->bias || !a->wav || a->B <= 0 || a->T <= 0 || a->C <= 0 || a->taps <= 0) return FS2_ERR_ARG;
  if (a->C == 32 && a->taps == 7 && (reinterpret_cast<uintptr_t>(a->x) & 15u) == 0 && (reinterpret_cast<uintptr_t>(a->w) & 15u) == 0) {
    constexpr int ROWS = CPF_BLOCKS * 7 - 6;
    const int gpb = (a->T + ROWS - 1) / ROWS;
    const long long n_groups = (long long)gpb * a->B, blocks = (n_groups * 8 + 255) / 256;
    if (blocks > 0x7fffffffLL) return FS2_ERR_UNSUPPORTED;
    prof_before(s);
    conv_post_c32_kernel<7><<<(unsigned)blocks, 256, 0, s>>>(*a, gpb, n_groups);
    prof_after(s, 3, 2.0 * (double)a->B * a->T * a->taps * a->C);
    FS2_LAUNCH_CHECK();
    return FS2_OK;
  }
  const size_t smem = ((size_t)a->taps * a->C + (size_t)(CP_ROWS + a->taps - 1) * (a->C + 1)) * sizeof(float);
  if (a->C % 4 || smem > 48 * 1024) return FS2_ERR_UNSUPPORTED;
  const int tiles = (a->T + CP_ROWS - 1) / CP_ROWS;
  const long long n = (long long)a->B * a->T;
  if ((long long)tiles * a->B > 0x7fffffffLL) return FS2_ERR_UNSUPPORTED;
  prof_before(s);
  conv_post_kernel<<<(unsigned)(tiles * a->B), CP_ROWS, smem, s>>>(*a, tiles);
  prof_after(s, 3, 2.0 * n * a->taps * a->C);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ [B,C,T] -> [B,T,C]
__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int T) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* ib = in + (long long)b * C * T;
  float* ob = out + (long long)b * C * T;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, t = t0 + threadIdx.x;
    if (c < C && t < T) tile[i][threadIdx.x] = ib[(long long)c * T + t];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int t = t0 + i, c = c0 + threadIdx.x;
    if (c < C && t < T) ob[(long long)t * C + c] = tile[threadIdx.x][i];
  }
}

int transpose_bct_to_btc(const float* in, float* out, int B, int C, int T, cudaStream_t s) {
  if (!in || !out || B <= 0 || C <= 0 || T <= 0) return FS2_ERR_ARG;
  dim3 grid((T + 31) / 32, (C + 31) / 32, B), block(32, 8);
  transpose_kernel<<<grid, block, 0, s>>>(in, out, C, T);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

// ------------------------------------------------------------------ waveform -> int16 + per-utterance trim (utils/model.py:82-90)
// out[b][t] = t < lens[b] ? np_int16(wav[b][t] * scale) : 0, where np_int16 is numpy's float32 -> int16 astype on x86-64: truncate
// toward zero to int32 (cvttss2si), then keep the low 16 bits.  So the conversion wraps: wav == 1.0 -- which tanhf returns exactly for
// arguments >= ~9.01 -- gives -32768, and NaN, +-inf and anything outside int32 give INT32_MIN, whose low 16 bits are 0.
// One thread converts 8 samples (16-byte store).
__device__ __forceinline__ short np_int16(float v) {
  const float t = truncf(v);
  if (!(t >= -2147483648.f && t < 2147483648.f)) return 0;
  return (short)(int)t;  // modulo 2^16
}

__global__ void wav_to_int16_kernel(const float* __restrict__ wav, long long wav_bs, const long long* __restrict__ lens, float scale, int B,
                                    long long N, short* __restrict__ out) {
  const long long per_b = (N + 7) / 8;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= per_b * B) return;
  const int b = (int)(idx / per_b);
  const long long t0 = (idx - (long long)b * per_b) * 8;
  const long long len = lens ? min(max(lens[b], 0LL), N) : N;
  const float* src = wav + (long long)b * wav_bs + t0;
  short v[8];
  if (t0 + 8 <= N && ((reinterpret_cast<uintptr_t>(src) & 15u) == 0)) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(src)), c = __ldg(reinterpret_cast<const float4*>(src) + 1);
    const float f[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = t0 + k < len ? np_int16(__fmul_rn(f[k], scale)) : (short)0;
  } else {
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = (t0 + k < N && t0 + k < len) ? np_int16(__fmul_rn(src[k], scale)) : (short)0;
  }
  short* dst = out + (long long)b * N + t0;
  if (t0 + 8 <= N && ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0)) {
    *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(v);
  } else {
    for (int k = 0; k < 8 && t0 + k < N; k++) dst[k] = v[k];
  }
}

int wav_to_int16(const fs2_wav_int16_args* a, cudaStream_t s) {
  if (!a || !a->wav || !a->out || a->B <= 0 || a->N <= 0) return FS2_ERR_ARG;
  const long long threads = ((a->N + 7) / 8) * a->B;
  wav_to_int16_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(a->wav, (long long)a->wav_batch_stride, reinterpret_cast<const long long*>(a->lens), a->scale, a->B, (long long)a->N, reinterpret_cast<short*>(a->out));
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

}  // namespace fs2
