// Fused self-attention of one FFT block on the tensor cores (transformer/Modules.py:14-25 + key mask Models.py:79, heads as
// SubLayers.py:39-44): S = Q K^T, softmax and O = P V in ONE persistent tcgen05 kernel -- the score matrix lives in tensor memory
// and never reaches HBM (the GEMM path of attention_tc.cu materialises S [B*H][T][Tk] in fp32: 535 MB per layer at B = 64).
//
//   work item = (utterance b, head h, 128 query rows); K and V come as the per-utterance operand tiles that pack_k/v_tiles_kernel
//   (attention_tc.cu) write once per layer (fp16 hi/lo, three-MMA split: attention keeps fp32-class operands).
//   pass 1: for every block of 128 keys  S = Q K_j^T (TMEM, double-buffered)  ->  row maximum (thread == query row; the two warps
//           that share a row's halves combine through shared memory once per item).
//   pass 2: S again -> p = exp2(s*c - m) (keys >= key_len masked to 0) -> fp16 hi/lo operand planes in shared memory ->
//           O += P V_j (TMEM accumulator), row sums alongside.  No rescaling of O is ever needed because the maximum is final.
//   epilogue: O / l -> ctx[b, t, h*128 .. +128]; query rows t >= key_len[b] are written as 0 (contract of fs2_attention).
//   Recomputing S costs 1/3 more MMAs than a one-pass online softmax and removes the O-rescale round trips through TMEM.
//
// Roles: warp 0 streams K / V stages (cp.async.bulk), warp 1 issues the MMAs, warps 2-9 are "row" warps (TMEM lane quarter =
// warp % 4, column half = (warp-2)/4): Q conversion, both softmax passes, the epilogue.
#include "common.cuh"
#include "tc_format.cuh"

namespace fs2 {

int pack_kv_tiles(const fs2_attention_args* a, unsigned char* kt, unsigned char* vt, long long tstride, cudaStream_t s);   // attention_tc.cu

constexpr int AF_THREADS = 320;
constexpr int AF_SB = 8;                         // K / V stage ring depth
constexpr uint32_t AF_STAGE = 8192;              // one stage: [hi | lo][2 chunks][128][16 B]

struct AfP {
  const float* qkv; float* ctx;
  const unsigned char* kt; const unsigned char* vt; long long tstride;     // per (b, h) tile buffers (128-byte header first)
  int B, T, H, Tk;                               // Tk = T rounded up to 128
  const int* key_lens; float scale;
  int n_items, qtiles;
};

// 16 fp32 values of one row -> fp16 hi / lo operand planes of K-block kb ([2 chunks][128 rows][16 B] each)
__device__ __forceinline__ void af_store16(unsigned char* kblk, int row, const float (&a)[16]) {
  uint32_t hw[2][4], lw[2][4];
  split_f16(a, hw[0], lw[0]);
  split_f16(a + 8, hw[1], lw[1]);
  unsigned char* p0 = kblk + (size_t)row * 16;
  *reinterpret_cast<uint4*>(p0) = make_uint4(hw[0][0], hw[0][1], hw[0][2], hw[0][3]);          // hi, chunk 0
  *reinterpret_cast<uint4*>(p0 + 2048) = make_uint4(hw[1][0], hw[1][1], hw[1][2], hw[1][3]);   // hi, chunk 1
  *reinterpret_cast<uint4*>(p0 + 4096) = make_uint4(lw[0][0], lw[0][1], lw[0][2], lw[0][3]);   // lo, chunk 0
  *reinterpret_cast<uint4*>(p0 + 6144) = make_uint4(lw[1][0], lw[1][1], lw[1][2], lw[1][3]);   // lo, chunk 1
}

__global__ void __launch_bounds__(AF_THREADS, 1) attention_fused_kernel(const AfP p) {
  constexpr uint32_t KBLK = 8192;                // one 16-wide K-block of an A operand: hi plane 4 KB + lo plane 4 KB (128 rows)
  constexpr uint32_t PLANES = 8 * KBLK;          // 128 x 128 operand: 64 KB
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned char* qa = smem_raw;                  // Q operand planes
  unsigned char* pa = qa + PLANES;               // P operand planes
  unsigned char* ring = pa + PLANES;
  float* xch = reinterpret_cast<float*>(ring + (size_t)AF_SB * AF_STAGE);   // [2 halves][128 rows] row max, then row sums
  uint64_t* bars = reinterpret_cast<uint64_t*>(xch + 256);
  uint64_t* fullB = bars;                        // [AF_SB]
  uint64_t* emptyB = fullB + AF_SB;              // [AF_SB]
  uint64_t* sFull = emptyB + AF_SB;              // [2] S buffer written
  uint64_t* sEmpty = sFull + 2;                  // [2] S buffer read by all row warps
  uint64_t* qReady = sEmpty + 2;                 // Q planes written (and O of the previous item drained)
  uint64_t* pReady = qReady + 1;                 // P planes of a key block written
  uint64_t* pFree = pReady + 1;                  // the PV MMAs that read them have retired
  uint64_t* oFull = pFree + 1;                   // O complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(oFull + 1);

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < AF_SB; i++) { mbar_init(&fullB[i], 1); mbar_init(&emptyB[i], 1); }
    for (int i = 0; i < 2; i++) { mbar_init(&sFull[i], 1); mbar_init(&sEmpty[i], 8); }
    mbar_init(qReady, 8); mbar_init(pReady, 8); mbar_init(pFree, 1); mbar_init(oFull, 1);
    mbar_init_fence();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t s_col[2] = {0u, 128u}, o_col = 256u;
  const int nkb = p.Tk / 128;                    // key blocks

  if (warp == 0) {
    // ===================== K / V stage producer, in the order the MMA warp consumes them =====================
    if (lane == 0) {
      Ring rb;
      auto push = [&](const unsigned char* src) {
        mbar_wait(&emptyB[rb.idx], rb.phase ^ 1);
        mbar_expect_tx(&fullB[rb.idx], AF_STAGE);
        bulk_g2s(ring + (size_t)rb.idx * AF_STAGE, src, AF_STAGE, &fullB[rb.idx]);
        rb.advance(AF_SB);
      };
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const int bh = item / p.qtiles;
        const unsigned char* kt = p.kt + (long long)bh * p.tstride + TC_HDR;   // [key block][d/16][8 KB]
        const unsigned char* vt = p.vt + (long long)bh * p.tstride + TC_HDR;   // [key/16][8 KB]
        for (int j = 0; j < nkb; j++)                                            // pass 1
          for (int kb = 0; kb < 8; kb++) push(kt + ((size_t)j * 8 + kb) * AF_STAGE);
        for (int kb = 0; kb < 8; kb++) push(kt + (size_t)kb * AF_STAGE);         // pass 2: S(0)
        for (int j = 0; j < nkb; j++) {
          if (j + 1 < nkb)
            for (int kb = 0; kb < 8; kb++) push(kt + ((size_t)(j + 1) * 8 + kb) * AF_STAGE);   // S(j+1)
          for (int kb = 0; kb < 8; kb++) push(vt + ((size_t)j * 8 + kb) * AF_STAGE);           // P V_j
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t leader = elect_one();
    const uint32_t idesc = umma_idesc_f16(128);
    const uint64_t desc_c = umma_desc(0, 2048, 128);     // A and B alike: chunk stride 128 rows * 16 B, 8-row groups 128 B apart
    const uint32_t qa16 = smem_u32(qa) >> 4, pa16 = smem_u32(pa) >> 4;
    Ring rb;
    uint32_t s_use[2] = {0, 0};                  // uses of each S buffer so far (phase of sEmpty / sFull)
    uint32_t q_phase = 0, p_phase = 0, pf_phase = 0;
    // D[tmem col] (+)= A(planes a16, 8 K-blocks) x B(next 8 ring stages), three-MMA split
    auto gemm = [&](uint32_t a16, uint32_t dcol, bool overwrite) {
      for (int kb = 0; kb < 8; kb++, rb.advance(AF_SB)) {
        mbar_wait(&fullB[rb.idx], rb.phase);
        tc_fence_after();
        if (leader) {
          const uint64_t a_hi = desc_c | (uint64_t)((a16 + kb * (KBLK >> 4)) & 0x3fff), a_lo = a_hi + (4096 >> 4);
          const uint64_t b_hi = desc_c | (uint64_t)(smem_u32(ring + (size_t)rb.idx * AF_STAGE) >> 4), b_lo = b_hi + (4096 >> 4);
          tc_mma_f16(tmem + dcol, a_lo, b_hi, idesc, (overwrite && kb == 0) ? 0u : 1u);
          tc_mma_f16(tmem + dcol, a_hi, b_hi, idesc, 1u);
          tc_mma_f16(tmem + dcol, a_hi, b_lo, idesc, 1u);
          tc_commit(&emptyB[rb.idx]);
        }
        __syncwarp();
      }
    };
    auto issue_s = [&](int j) {                  // S(j) into buffer j & 1
      const int sb = j & 1;
      if (s_use[sb] > 0) mbar_wait(&sEmpty[sb], (s_use[sb] - 1) & 1);      // the previous contents have been read
      tc_fence_after();
      gemm(qa16, s_col[sb], true);
      if (leader) tc_commit(&sFull[sb]);
      __syncwarp();
      s_use[sb]++;
    };
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      mbar_wait(qReady, q_phase); q_phase ^= 1;
      tc_fence_after();
      for (int j = 0; j < nkb; j++) issue_s(j);                             // pass 1
      issue_s(0);                                                           // pass 2
      for (int j = 0; j < nkb; j++) {
        if (j + 1 < nkb) issue_s(j + 1);
        mbar_wait(pReady, p_phase); p_phase ^= 1;
        tc_fence_after();
        gemm(pa16, o_col, j == 0);
        if (leader) { tc_commit(pFree); if (j == nkb - 1) tc_commit(oFull); }
        __syncwarp();
      }
      (void)pf_phase;
    }
  } else {
    // ===================== row warps =====================
    const int q = warp & 3, h = (warp - 2) >> 2;
    const int r128 = q * 32 + lane;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const int D = p.H * 128;
    const float c = p.scale * (1.f / KV_WSCALE) * 1.4426950408889634f;      // s*c = scaled score in log2 units (K tiles carry x16)
    uint32_t s_phase[2] = {0, 0}, pf_phase = 0, o_phase = 0;
    bool p_written = false;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const int bh = item / p.qtiles, qt = item - bh * p.qtiles;
      const int b = bh / p.H, hd = bh - b * p.H;
      const int t = qt * 128 + r128;
      const int len = p.key_lens ? min(p.key_lens[b], p.T) : p.T;
      // ---- Q rows -> operand planes (this warp: d columns 64h .. 64h+63 = K-blocks 4h .. 4h+3)
      {
        const float* src = p.qkv + ((long long)b * p.T + t) * 3 * D + hd * 128 + h * 64;
#pragma unroll
        for (int g = 0; g < 4; g++) {
          float v[16];
          if (t < p.T) {
#pragma unroll
            for (int k4 = 0; k4 < 4; k4++) {
              const float4 u = __ldg(reinterpret_cast<const float4*>(src + g * 16) + k4);
              v[4 * k4] = u.x; v[4 * k4 + 1] = u.y; v[4 * k4 + 2] = u.z; v[4 * k4 + 3] = u.w;
            }
          } else {
#pragma unroll
            for (int k = 0; k < 16; k++) v[k] = 0.f;
          }
          af_store16(qa + (size_t)(h * 4 + g) * KBLK, r128, v);
        }
        fence_proxy_async();
        tc_fence_before();                         // (also orders the previous item's O reads before the next O overwrite)
        __syncwarp();
        if (lane == 0) mbar_arrive(qReady);
      }
      // ---- pass 1: row maximum of the masked, scaled scores over this warp's key halves
      float m = -INFINITY;
      for (int j = 0; j < nkb; j++) {
        const int sb = j & 1;
        mbar_wait(&sFull[sb], s_phase[sb]); s_phase[sb] ^= 1;
        tc_fence_after();
#pragma unroll
        for (int g = 0; g < 2; g++) {
          uint32_t sv[32];
          tc_ld32(tmem + lane_base + s_col[sb] + h * 64 + g * 32, sv);
          const int key0 = j * 128 + h * 64 + g * 32;
#pragma unroll
          for (int k = 0; k < 32; k++)
            if (key0 + k < len) m = fmaxf(m, __uint_as_float(sv[k]) * c);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&sEmpty[sb]);
      }
      xch[h * 128 + r128] = m;
      row_warps_sync<256>();
      m = fmaxf(xch[r128], xch[128 + r128]);
      row_warps_sync<256>();                          // xch is reused for the row sums
      // ---- pass 2: p = exp2(s*c - m) -> P operand planes (this warp: keys 64h .. 64h+63 of the block = K-blocks 4h .. 4h+3)
      float l = 0.f;
      for (int j = 0; j < nkb; j++) {
        const int sb = j & 1;
        mbar_wait(&sFull[sb], s_phase[sb]); s_phase[sb] ^= 1;
        tc_fence_after();
        if (p_written) { mbar_wait(pFree, pf_phase); pf_phase ^= 1; }      // the previous block's PV MMAs have read the planes
#pragma unroll
        for (int g = 0; g < 2; g++) {
          uint32_t sv[32];
          tc_ld32(tmem + lane_base + s_col[sb] + h * 64 + g * 32, sv);
          const int key0 = j * 128 + h * 64 + g * 32;
#pragma unroll
          for (int half = 0; half < 2; half++) {
            float pv[16];
#pragma unroll
            for (int k = 0; k < 16; k++) {
              const float e = key0 + half * 16 + k < len ? exp2f(fmaf(__uint_as_float(sv[half * 16 + k]), c, -m)) : 0.f;
              pv[k] = e;
              l += e;
            }
            af_store16(pa + (size_t)(h * 4 + g * 2 + half) * KBLK, r128, pv);
          }
        }
        tc_fence_before();
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) { mbar_arrive(&sEmpty[sb]); mbar_arrive(pReady); }
        p_written = true;
      }
      xch[h * 128 + r128] = l;
      row_warps_sync<256>();
      l = xch[r128] + xch[128 + r128];
      // ---- epilogue: O / l (V tiles carry x16), rows beyond the utterance are zero
      mbar_wait(oFull, o_phase); o_phase ^= 1;
      tc_fence_after();
      const float inv = (t < len) ? (1.f / KV_WSCALE) / l : 0.f;
      float* dst = p.ctx + ((long long)b * p.T + t) * D + hd * 128 + h * 64;
#pragma unroll
      for (int g = 0; g < 2; g++) {
        uint32_t ov[32];
        tc_ld32(tmem + lane_base + o_col + h * 64 + g * 32, ov);
        if (t < p.T) {
#pragma unroll
          for (int k4 = 0; k4 < 8; k4++)
            reinterpret_cast<float4*>(dst + g * 32)[k4] = make_float4(__uint_as_float(ov[4 * k4]) * inv, __uint_as_float(ov[4 * k4 + 1]) * inv,
                                                                      __uint_as_float(ov[4 * k4 + 2]) * inv, __uint_as_float(ov[4 * k4 + 3]) * inv);
        }
      }
      row_warps_sync<256>();                          // xch free for the next item
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

static constexpr size_t AF_SMEM = 2 * 65536 + (size_t)AF_SB * AF_STAGE + 256 * 4 + (2 * AF_SB + 10) * 8 + 16;

size_t attention_fused_workspace(int B, int T, int H) {
  const int Tk = (T + 127) / 128 * 128;
  const size_t tile_bytes = ((size_t)B * H * kv_tile_stride(Tk) + 255) & ~(size_t)255;
  return 2 * tile_bytes + 256;
}

int attention_fused(const fs2_attention_args* a, void* ws, size_t ws_bytes, cudaStream_t s) {
  if (!a || !a->qkv || !a->ctx || !ws || a->B <= 0 || a->T <= 0 || a->H <= 0) return FS2_ERR_ARG;
  if (a->Dh != 128) return FS2_ERR_UNSUPPORTED;
  if (!aligned16(a->qkv) || !aligned16(a->ctx)) return FS2_ERR_ARG;
  if (ws_bytes < attention_fused_workspace(a->B, a->T, a->H)) return FS2_ERR_WORKSPACE;
  int derr = FS2_OK;
  DevState* dv = dev_state(&derr);
  if (!dv) return derr;
  FS2_TRY(setup_once(dv->att_fused_ready,
                     [] { return cudaFuncSetAttribute(attention_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AF_SMEM); }));
  const int Tk = (a->T + 127) / 128 * 128;
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  const long long tstride = kv_tile_stride(Tk);
  const size_t tile_bytes = ((size_t)a->B * a->H * tstride + 255) & ~(size_t)255;
  unsigned char* kt = reinterpret_cast<unsigned char*>(base);
  unsigned char* vt = kt + tile_bytes;
  FS2_TRY(pack_kv_tiles(a, kt, vt, tstride, s));
  AfP p{};
  p.qkv = a->qkv; p.ctx = a->ctx; p.kt = kt; p.vt = vt; p.tstride = tstride;
  p.B = a->B; p.T = a->T; p.H = a->H; p.Tk = Tk; p.key_lens = a->key_lens; p.scale = a->scale;
  p.qtiles = (a->T + 127) / 128;
  const long long items = (long long)a->B * a->H * p.qtiles;
  if (items > 0x7fffffffLL) return FS2_ERR_UNSUPPORTED;
  p.n_items = (int)items;
  const int num_sms = dv->num_sms.load(std::memory_order_relaxed);
  const int grid = items < num_sms ? (int)items : num_sms;
  prof_before(s);
  attention_fused_kernel<<<grid, AF_THREADS, AF_SMEM, s>>>(p);
  // algorithmic count as the reference computes it (dense T x T): 4*T*T*Dh per (b, h)
  prof_after(s, 1, 4.0 * a->B * a->H * (double)a->T * a->T * 128);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

}  // namespace fs2
