// [device code; host side and heuristics: conv_tc.cu]
// tcgen05 (5th-gen tensor core) implicit-GEMM Conv1d over channels-last activations, error-compensated split-FP16.
//
//   y[b,t,n] = epilogue( sum_{tap} sum_c act(x[b, t + tap*dil - pad, c]) * w[tap][c][n] )        (contract: fs2_conv1d)
//
// Why a split: single-pass TF32 / FP16 / BF16 operands miss the parity bars (mel 1.2e-3 vs 1e-3, waveform 5.3e-4 vs 1e-4,
// SURVEY.md section 7).  Each fp32 operand is split x = hi + lo with hi = fp16(x), lo = fp16(x - hi) (x - hi is exact in
// fp32): 22 significant bits, the same as a TF32 hi/lo split, but kind::f16 MMAs have K = 16 per instruction -- twice the
// FLOPs per instruction and per shared-memory byte of kind::tf32.  D += A_lo*B_hi + A_hi*B_hi + A_hi*B_lo, fp32 accumulate in
// TMEM.  Weights are pre-scaled by a per-layer power of two (kept in a 128-byte header of the tiled buffer) so that their lo
// parts stay in fp16's normal range; activations are used unscaled (|x| > 65504 saturates in the convert; a lo part below 2^-14 only costs an
// ABSOLUTE error < 3e-8).  Emulated end to end on the CPU (exact accumulation) this split is as accurate as fp32 convolution
// on both the synthetic and the shipped HiFi-GAN checkpoint; on the GPU the tensor core's round-toward-zero accumulator is
// what remains (profiles/r01_tc_accumulate_bias.txt), and K = 16 halves the number of accumulation steps.
//
// Persistent, warp-specialised kernel: one CTA per SM walks a list of work items (MT consecutive 128-row time tiles of
// one utterance x one block of NB <= 128 output channels); four roles overlap through mbarrier rings:
//   warp 0      weight producer: every (tap, 16-channel K-block) weight stage is ONE cp.async.bulk (TMA bulk engine) of a
//               host-pre-split, host-pre-tiled smem image  [hi|lo][16-byte K-chunk][n][8 halfs].
//   warps 2-9   activation transform: read the [MT*128 + (taps-1)*dil] x 16-channel slab of a K-block ONCE from global
//               (one 256-bit load per row and 8 channels, a 3-deep register ring of K-blocks in flight: ~60 KB of loads per SM), apply the input activation, split hi/lo and store both in the
//               UMMA no-swizzle K-major layout [16-byte K-chunk][row][8 halfs].  There a core matrix (8 rows x 16 B)
//               starting at ANY row is 128 contiguous bytes, so each conv tap is just the same slab with the descriptor start
//               address advanced by tap*dil rows: the slab is loaded and split once per K-block, not once per tap.
//   warp 1      MMA issuer (one elected thread): per weight stage MT * 3 (split terms) tcgen05.mma kind::f16, M=128, N=NB, K=16,
//               accumulating into one of two TMEM accumulator sets; tcgen05.commit releases slab / weight stages and
//               publishes the accumulators.
//   warps 10-13 epilogue: tcgen05.ld (thread == output row) -> per-warp 32x36 smem transpose so that 8 lanes cover one
//               row's 128 bytes -> bias / activation / residual / alpha / accumulate / pad-row mask -> full-line global I/O.
//               Runs on work item i while the MMAs of item i+1 fill the other accumulator set.
#pragma once
#include "common.cuh"
#include "tc_format.cuh"

namespace fs2 {

constexpr int TC_KB = 16;          // input channels per K-block (one K=16 FP16 MMA per split term)
constexpr int TC_CHUNKS = TC_KB / 8;  // 16-byte K-chunks (8 halfs) per K-block
constexpr int TC_SA_MAX = 8;       // activation slab stages (runtime p.SA)
constexpr int TC_SB_MAX = 8;       // weight stages (runtime p.SB)
constexpr int TC_TW = 8;            // transform warps
constexpr int TC_TTHREADS = TC_TW * 32;
constexpr int TC_THREADS = 64 + TC_TTHREADS + 128;   // producer + MMA warps, transform warps, 4 epilogue warps
constexpr int TC_DEPTH = 3;         // K-blocks of activation loads in flight per transform thread (register ring)
constexpr int TC_LD = 3;           // (row, K-chunk) items (2 float4 loads each) per transform thread per K-block: 256 * 3 / 2 >= 384 rows
constexpr int TC_STAGE_FLOATS = 32 * 36;   // per-epilogue-warp transpose tile

struct TcP {
  const float* x; long long xbs, xrs;
  int B, T, Cin;
  const float* wt;                 // tiled weights, see packing.pack_conv_tc
  long long wt_bstride;            // bytes between the tile buffers of consecutive utterances (0 = shared weights)
  const float* bias;
  int N;                           // total output channels
  int NB;                          // output channels per work item (MMA N), N % NB == 0, NB % 16 == 0, NB <= 128
  int taps, dil, pad;
  int in_act; float in_slope;
  int out_act; float out_slope;
  const float* res; long long rbs, rrs;
  float alpha; int accumulate;
  const int* row_lens;
  float* y; long long ybs, yrs;
  int MT;                          // 128-row tiles per work item
  int TG;                          // accumulators per tile: 1 = all split terms together, 2 = {hi*hi | the two cross terms}
  int SA, SB;                      // ring depths
  int TPS;                         // conv taps per weight stage (small NB: several taps share one bulk copy / one handshake)
  int R;                           // slab rows held in smem (>= MT*128 + (taps-1)*dil, R % 8 == 4)
  int tiles_per_batch;             // work items per utterance
  int n_items;                     // total work items = (N/NB) * B * tiles_per_batch
  int acc_stride;                  // TMEM columns between accumulators
  int tmem_cols;                   // power of two >= 2*MT*TG*acc_stride
  long long* trace;                // debug: [CTA][16 items][8] globaltimer stamps, or NULL
  unsigned variant;                // reserved for A/B experiments (unused by the shipped kernel)
  int pdl;                         // launched with programmatic stream serialisation: wait for the previous grid before touching its data
  int nseg;                        // K-segments per output tile (1 = plain conv).  > 1: the conv is the sum of nseg one-tap slices over p.Cin (= 256)
                                   // input channels each, slice s = (tap = s / seg_nkc, channel chunk = s % seg_nkc); every slice is its own work unit with a
                                   // fresh accumulator, and the units of one tile run back to back on one CTA, adding into y in fp32 (FS2_TC_VARIANT_SEGMENTED)
  int seg_nkc;                     // channel chunks per tap
  long long seg_wbytes;            // bytes between the tile buffers of consecutive slices
  int f8;                          // operand split: 0 = three kind::f16 MMAs (hi*hi + lo*hi + hi*lo), 1 = kind::f16 main term + ONE kind::f8f6f4 correction MMA
};

// debug timeline: slot 0/1 transform first-load-issue / last-store of the item, 2/3 MMA start / all issued, 4/5 epilogue start / end
// (compiled in only with -DFS2_TC_TRACE: the checks cost ~8 % of the transform warps' instructions)
#ifdef FS2_TC_TRACE
#define TC_STAMP(il, slot)                                                                       \
  do {                                                                                           \
    if (p.trace && (il) < 16) p.trace[((long long)blockIdx.x * 16 + (il)) * 8 + (slot)] = gtime(); \
  } while (0)
#else
#define TC_STAMP(il, slot) do { } while (0)
#endif

struct Item { int nblk, b, t0; };
__device__ __forceinline__ Item decode_item(const TcP& p, int item) {
  const int per_blk = p.B * p.tiles_per_batch;
  Item it;
  it.nblk = item / per_blk;
  const int rem = item - it.nblk * per_blk;
  it.b = rem / p.tiles_per_batch;
  it.t0 = (rem - it.b * p.tiles_per_batch) * p.MT * 128;
  return it;
}

template <int ACT>
__device__ __forceinline__ float tc_act(float v, float slope) {
  if (ACT == FS2_ACT_RELU) return fmaxf(v, 0.f);
  if (ACT == FS2_ACT_TANH) return tanhf(v);
  if (ACT == FS2_ACT_LRELU) return v > 0.f ? v : v * slope;
  return v;
}

// One 32-row x W-column block of one accumulator: TMEM -> regs -> smem transpose -> coalesced global I/O.
// W = 32: 8 lanes per row, 4 rows per pass, 8 passes.  W = 16: 4 lanes per row, 8 rows per pass, 4 passes.
// RES / ACC (residual add, accumulate into y) are template parameters: as runtime flags their zero-filled operands and
// predicates were ~40 % of the epilogue's instructions on plain layers.
template <int ACT, int W, bool FULL, bool RES, bool ACC>
__device__ __forceinline__ void tc_epilogue_block(const TcP& p, uint32_t taddr, float* stage, int lane, float* yptr, const float* rptr,
                                                  const float* bias, int rows_live, int rows_valid, float inv_ws) {
  constexpr int LPR = W / 4, RPI = 32 / LPR, ITERS = 32 / RPI, HALF = ITERS / 2;
  constexpr int NR = RES ? HALF : 1, NY = ACC ? HALF : 1;
  const int rr = lane / LPR;
  const long long ystep = (long long)RPI * p.yrs, rstep = (long long)RPI * p.rrs;
  // Residual loads are software-pipelined by half-blocks: the first half is requested before the TMEM load / transpose, the
  // second half before the first half is consumed (A/B: -15..-28 % on residual layers against loads at the point of use).
  float4 r0[NR], r1[NR];
#pragma unroll
  for (int k = 0; k < NR; k++) {
    r0[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    r1[k] = r0[k];
  }
  if (RES) {
#pragma unroll
    for (int k = 0; k < NR; k++)
      if (FULL || k * RPI + rr < rows_valid) r0[k] = *reinterpret_cast<const float4*>(rptr + k * rstep);
  }
  {
    uint32_t v[32];
    if (W == 32) tc_ld32(taddr, v); else tc_ld16(taddr, v);
    for (int g = 1; g < p.TG; g++) {                   // split-term accumulators are summed here, in fp32 round-to-nearest
      uint32_t u[32];
      if (W == 32) tc_ld32(taddr + g * p.acc_stride, u); else tc_ld16(taddr + g * p.acc_stride, u);
#pragma unroll
      for (int j = 0; j < W; j++) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
    }
#pragma unroll
    for (int j = 0; j < W / 4; j++)
      *reinterpret_cast<float4*>(stage + lane * 36 + j * 4) =
          make_float4(__uint_as_float(v[j * 4]), __uint_as_float(v[j * 4 + 1]), __uint_as_float(v[j * 4 + 2]), __uint_as_float(v[j * 4 + 3]));
  }
  __syncwarp();
  const float slope = p.out_slope, alpha = p.alpha;
  float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (bias) bv = __ldg(reinterpret_cast<const float4*>(bias));
  const float* sp = stage + rr * 36 + (lane % LPR) * 4;
#pragma unroll
  for (int h = 0; h < 2; h++) {
    float4 (&rv)[NR] = h == 0 ? r0 : r1;
    if (RES && h == 0) {                                // request the second half now; it lands while the first half is processed
#pragma unroll
      for (int k = 0; k < NR; k++)
        if (FULL || (HALF + k) * RPI + rr < rows_valid) r1[k] = *reinterpret_cast<const float4*>(rptr + (HALF + k) * rstep);
    }
    float4 yv[NY];
#pragma unroll
    for (int k = 0; k < NY; k++) yv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ACC) {
#pragma unroll
      for (int k = 0; k < NY; k++)
        if (FULL || (h * HALF + k) * RPI + rr < rows_valid) yv[k] = *reinterpret_cast<const float4*>(yptr + (h * HALF + k) * ystep);
    }
#pragma unroll
    for (int k = 0; k < HALF; k++) {
      const int kk = h * HALF + k;
      const int r = kk * RPI + rr;
      if (FULL || r < rows_valid) {
        const float4 a = *reinterpret_cast<const float4*>(sp + kk * RPI * 36);
        float4 o;
        o.x = tc_act<ACT>(fmaf(a.x, inv_ws, bv.x), slope);   // inv_ws is a power of two: exact
        o.y = tc_act<ACT>(fmaf(a.y, inv_ws, bv.y), slope);
        o.z = tc_act<ACT>(fmaf(a.z, inv_ws, bv.z), slope);
        o.w = tc_act<ACT>(fmaf(a.w, inv_ws, bv.w), slope);
        if (RES) {
          const float4 rk = rv[RES ? k : 0];
          o.x += rk.x; o.y += rk.y; o.z += rk.z; o.w += rk.w;
        }
        if (ACC) {
          const float4 yk = yv[ACC ? k : 0];
          o.x = o.x * alpha + yk.x; o.y = o.y * alpha + yk.y; o.z = o.z * alpha + yk.z; o.w = o.w * alpha + yk.w;
        } else {
          o.x *= alpha; o.y *= alpha; o.z *= alpha; o.w *= alpha;
        }
        if (!FULL && r >= rows_live) o = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(yptr + kk * ystep) = o;
      }
    }
  }
  __syncwarp();   // the staging tile is rewritten by the next block
}

template <int ACT, bool RES, bool ACC>
__device__ __forceinline__ void tc_epilogue_item(const TcP& p, uint32_t tmem_acc, float* stage, int q, int lane, const Item& it, float inv_ws) {
  const int NB = p.NB, n0 = it.nblk * NB;
  const int len_b = p.row_lens ? min(p.row_lens[it.b], p.T) : p.T;
  for (int mt = 0; mt < p.MT; mt++) {
    const int row0 = it.t0 + mt * 128 + q * 32;
    const int rows_valid = min(32, p.T - row0);        // rows that exist
    if (rows_valid <= 0) continue;                     // warp-uniform
    const int rows_live = min(32, len_b - row0);       // rows that are not padding (may be <= 0)
    const bool full = rows_valid == 32 && rows_live == 32;
    const uint32_t tbase = tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(mt * p.TG * p.acc_stride);
    for (int c = 0; c < NB; c += 32) {
      const int w = (NB - c) >= 32 ? 32 : 16;          // NB % 16 == 0
      const int sh = w == 32 ? 3 : 2;                  // lanes per row = 8 or 4
      const int rr = lane >> sh, cc = (lane & ((1 << sh) - 1)) * 4;
      float* yptr = p.y + (long long)it.b * p.ybs + (long long)(row0 + rr) * p.yrs + n0 + c + cc;
      const float* rptr = RES ? p.res + (long long)it.b * p.rbs + (long long)(row0 + rr) * p.rrs + n0 + c + cc : nullptr;
      const float* bias = p.bias ? p.bias + n0 + c + cc : nullptr;
      if (w == 32) {
        if (full) tc_epilogue_block<ACT, 32, true, RES, ACC>(p, tbase + c, stage, lane, yptr, rptr, bias, rows_live, rows_valid, inv_ws);
        else tc_epilogue_block<ACT, 32, false, RES, ACC>(p, tbase + c, stage, lane, yptr, rptr, bias, rows_live, rows_valid, inv_ws);
      } else {
        tc_epilogue_block<ACT, 16, false, RES, ACC>(p, tbase + c, stage, lane, yptr, rptr, bias, rows_live, rows_valid, inv_ws);
      }
    }
  }
}

template <int ACT>
__device__ __forceinline__ void tc_epilogue_dispatch(const TcP& p, uint32_t tmem_acc, float* stage, int q, int lane, const Item& it, float inv_ws) {
  if (p.res) {
    if (p.accumulate) tc_epilogue_item<ACT, true, true>(p, tmem_acc, stage, q, lane, it, inv_ws);
    else tc_epilogue_item<ACT, true, false>(p, tmem_acc, stage, q, lane, it, inv_ws);
  } else {
    if (p.accumulate) tc_epilogue_item<ACT, false, true>(p, tmem_acc, stage, q, lane, it, inv_ws);
    else tc_epilogue_item<ACT, false, false>(p, tmem_acc, stage, q, lane, it, inv_ws);
  }
}

// One K-block of one transform thread: input activation, operand split, stores into the slab planes.
//   F8 = false: plane 0 = fp16 hi, plane 1 = fp16 lo, both [16-byte K-chunk of 8 channels][row][8 halfs].
//   F8 = true : plane 0 = fp16 hi as above; plane 1 = E4M3 [chunk 0: lo * 2^12 of the 16 channels | chunk 1: hi of the 16 channels][row][16 bytes]
//               -- the A operand of one K = 32 kind::f8f6f4 MMA whose B operand is [weight hi ; weight lo].
template <bool LRELU, bool F8, int LD>
__device__ __forceinline__ void tc_convert_store(const float (&src)[LD][8], const int (&rowu)[LD], const int (&offu)[LD], const int (&off8)[LD],
                                                 unsigned char* hi, unsigned char* lo, uint32_t chunk_bytes, float in_slope) {
  const auto act = [in_slope](float v) { return LRELU ? fmaxf(v, v * in_slope) : v; };   // leaky_relu for 0 <= slope <= 1
#pragma unroll
  for (int u = 0; u < LD; u++) {
    if (rowu[u] < 0) continue;
    uint32_t hw[4], lw[4];
    if (F8) {
      uint32_t l8[2], h8[2];
      split_f16_e4m3(src[u], hw, l8, h8, act);
      *reinterpret_cast<uint4*>(hi + offu[u]) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      *reinterpret_cast<uint2*>(lo + off8[u]) = make_uint2(l8[0], l8[1]);                  // E4M3 lo of these 8 channels
      *reinterpret_cast<uint2*>(lo + off8[u] + chunk_bytes) = make_uint2(h8[0], h8[1]);    // E4M3 hi of these 8 channels
    } else {
      split_f16(src[u], hw, lw, act);
      *reinterpret_cast<uint4*>(hi + offu[u]) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
      *reinterpret_cast<uint4*>(lo + offu[u]) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
  }
}

template <int MT, int TG>
__global__ void __launch_bounds__(TC_THREADS, 1) conv_tc_kernel(const TcP p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int R = p.R, NB = p.NB, SA = p.SA, SB = p.SB;
  const uint32_t a_plane = (uint32_t)TC_CHUNKS * R * 16;          // bytes of one hi (or lo) slab
  const uint32_t b_plane = (uint32_t)TC_CHUNKS * NB * 16;         // bytes of one hi (or lo) weight tile
  float* stage_all = reinterpret_cast<float*>(smem_raw);           // [4 warps][32 x 36] epilogue transpose tiles
  unsigned char* a_base = smem_raw + 4 * TC_STAGE_FLOATS * sizeof(float);   // [SA][hi|lo][chunk][R][16 B]
  unsigned char* b_base = a_base + (size_t)SA * 2 * a_plane;       // [SB][hi|lo][chunk][NB][16 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_base + (size_t)SB * p.TPS * 2 * b_plane);
  uint64_t* fullA = bars;                  // [SA_MAX]
  uint64_t* emptyA = fullA + TC_SA_MAX;    // [SA_MAX]
  uint64_t* fullB = emptyA + TC_SA_MAX;    // [SB_MAX]
  uint64_t* emptyB = fullB + TC_SB_MAX;    // [SB_MAX]
  uint64_t* accFull = emptyB + TC_SB_MAX;  // [2]
  uint64_t* accEmpty = accFull + 2;        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accEmpty + 2);

  const int KBLOCKS = p.Cin / TC_KB;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < TC_SA_MAX; i++) { mbar_init(&fullA[i], TC_TW); mbar_init(&emptyA[i], 1); }
    for (int i = 0; i < TC_SB_MAX; i++) { mbar_init(&fullB[i], 1); mbar_init(&emptyB[i], 1); }
    for (int i = 0; i < 2; i++) { mbar_init(&accFull[i], 1); mbar_init(&accEmpty[i], 4); }
    mbar_init_fence();
  }
  if (warp == 1) tmem_alloc(tmem_slot, p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t acc_set = (uint32_t)(MT * TG * p.acc_stride);      // columns per accumulator set
  if (p.pdl) {
    grid_dep_launch();
    // Static weights were written before the stream reached this layer, so the producer warp starts prefetching weight stages
    // while the predecessor drains; per-utterance "weights" (attention K / V tiles) come from the previous kernel.  The MMA
    // warp touches no global memory.  Everything else (activation loads, residual / accumulate loads, stores) waits.
    if (warp >= 2 || (warp == 0 && p.wt_bstride != 0)) grid_dep_wait();
  }

  if (warp == 0) {
    // ===================== weight-stage producer (TMA bulk copies) =====================
    if (lane == 0) {
      const uint32_t stage_bytes = 2 * b_plane;   // one tap of one K-block (hi + lo)
      Ring rb;
      const int per_blk = p.B * p.tiles_per_batch;
      int nblk = (int)blockIdx.x / per_blk, rem = (int)blockIdx.x - nblk * per_blk;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const long long wb = p.wt_bstride ? (long long)(rem / p.tiles_per_batch) * p.wt_bstride : 0;
        for (int seg = 0; seg < p.nseg; seg++) {
        const unsigned char* wsrc = reinterpret_cast<const unsigned char*>(p.wt) + (long long)seg * p.seg_wbytes + wb + TC_HDR +
                                    (size_t)nblk * p.taps * KBLOCKS * stage_bytes;
        const unsigned char* src = wsrc;           // tiles are ordered [kb][tap]: the taps of one K-block are contiguous
        for (int kb = 0; kb < KBLOCKS; kb++) {
          for (int tap = 0; tap < p.taps; tap += p.TPS) {
            const int n = min(p.TPS, p.taps - tap);
            const uint32_t bytes = (uint32_t)n * stage_bytes;
            mbar_wait(&emptyB[rb.idx], rb.phase ^ 1);
            mbar_expect_tx(&fullB[rb.idx], bytes);
            bulk_g2s(b_base + (size_t)rb.idx * p.TPS * stage_bytes, src, bytes, &fullB[rb.idx]);
            src += bytes;
            rb.advance(SB);
          }
        }
        }
        rem += (int)gridDim.x;
        while (rem >= per_blk) { rem -= per_blk; nblk++; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp runs the (warp-uniform) loops and barrier waits so that descriptors live in uniform registers; one
    // elected lane issues the MMAs and the commits.  Per weight stage the 6*MT MMAs are fully unrolled and every operand is
    // a precomputed base plus a constant: the issue cost per MMA must stay well below the 16..64 cycles an MMA occupies
    // the tensor pipe (a generic address computation per MMA was measured to be the bottleneck).
    const uint32_t leader = elect_one();
    const uint32_t idesc = umma_idesc_f16(NB);
    const uint64_t a_const = umma_desc(0, (uint32_t)R * 16, 128), b_const = umma_desc(0, (uint32_t)NB * 16, 128);
    const uint32_t tile_cols = (uint32_t)(TG * p.acc_stride);
    const uint32_t g_cross = TG >= 2 ? (uint32_t)p.acc_stride : 0u;            // lo*hi and hi*lo
    Ring ra, rb, rt;
    uint32_t itT = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x)
    for (int seg = 0; seg < p.nseg; seg++, itT++, rt.advance(2)) {           // one work unit per (item, K-segment)
      const uint32_t buf = rt.idx;
      mbar_wait(&accEmpty[buf], rt.phase ^ 1);                    // epilogue has drained this accumulator set
      tc_fence_after();
      const uint32_t d0 = tmem + buf * acc_set;
      if (leader) TC_STAMP((int)itT, 2);
      for (int kb = 0; kb < KBLOCKS; kb++, ra.advance(SA)) {
        const uint32_t sa = ra.idx;
        mbar_wait(&fullA[sa], ra.phase);
        tc_fence_after();
        const uint64_t a_hi = a_const | (uint64_t)(smem_u32(a_base + (size_t)sa * 2 * a_plane) >> 4);
        const uint64_t a_lo = a_hi + (a_plane >> 4);
        uint32_t row_off = 0;
        for (int tap = 0; tap < p.taps; tap += p.TPS, rb.advance(SB)) {
          const uint32_t sb = rb.idx;
          const int n = min(p.TPS, p.taps - tap);
          mbar_wait(&fullB[sb], rb.phase);
          tc_fence_after();
          if (leader) {
            uint64_t b_hi = b_const | (uint64_t)(smem_u32(b_base + (size_t)sb * p.TPS * 2 * b_plane) >> 4);
            for (int j = 0; j < n; j++, b_hi += (2 * b_plane) >> 4, row_off += (uint32_t)p.dil) {
              const uint64_t b_lo = b_hi + (b_plane >> 4);
              const uint64_t ah0 = a_hi + row_off, al0 = a_lo + row_off;
              const uint32_t first = (kb | tap | j) ? 1u : 0u;
              // consecutive MMAs alternate between tiles / accumulator groups
              if (p.f8) {
#pragma unroll
                for (int mt = 0; mt < MT; mt++)          // fp16: A_hi * B_hi
                  tc_mma_f16(d0 + mt * tile_cols, ah0 + mt * 128, b_hi, idesc, first);
#pragma unroll
                for (int mt = 0; mt < MT; mt++)          // E4M3, K = 32: [A_lo | A_hi] * [B_hi ; B_lo]
                  tc_mma_f8(d0 + mt * tile_cols + g_cross, al0 + mt * 128, b_lo, idesc, TG >= 2 ? first : 1u);
              } else {
#pragma unroll
                for (int mt = 0; mt < MT; mt++)          // A_lo * B_hi
                  tc_mma_f16(d0 + mt * tile_cols + g_cross, al0 + mt * 128, b_hi, idesc, first);
#pragma unroll
                for (int mt = 0; mt < MT; mt++)          // A_hi * B_hi
                  tc_mma_f16(d0 + mt * tile_cols, ah0 + mt * 128, b_hi, idesc, TG >= 2 ? first : 1u);
#pragma unroll
                for (int mt = 0; mt < MT; mt++)          // A_hi * B_lo
                  tc_mma_f16(d0 + mt * tile_cols + g_cross, ah0 + mt * 128, b_lo, idesc, 1u);
              }
            }
            tc_commit(&emptyB[sb]);                    // weight stage free once these MMAs retire
          } else {
            row_off += (uint32_t)(n * p.dil);
          }
          __syncwarp();
        }
        if (leader) tc_commit(&emptyA[sa]);            // slab stage free
        __syncwarp();
      }
      if (leader) tc_commit(&accFull[buf]);            // accumulators of this work item complete
      if (leader) TC_STAMP((int)itT, 3);
      __syncwarp();
    }
  } else if (warp < 2 + TC_TW) {
    // ===================== transform warps (activation + fp16 hi/lo split) =====================
    // The instruction count per (row, K-chunk) unit sets the speed of the narrow / small-k layers (ncu: these warps issue
    // 40 % of the kernel's instructions and are busy 70 % of the time), so: one 256-bit load per unit, addresses from a
    // per-K-block base + a precomputed 32-bit offset, no range checks for interior work items, the fp16 clamp folded into
    // the saturating convert, the input activation resolved outside the unit loop.
    const int wt = tid - 64;                           // 0..TC_TTHREADS-1
    const int rows_needed = MT * 128 + (p.taps - 1) * p.dil;
    const int items = rows_needed * TC_CHUNKS;
    // Register ring of TC_DEPTH K-blocks: the loads of K-block seq + TC_DEPTH (possibly of a later work item) are issued as
    // soon as K-block seq has been converted and stored, so ~TC_DEPTH slabs of loads stay in flight per SM.
    constexpr int LD = MT == 4 ? 5 : TC_LD;           // (row, chunk) units per thread per K-block
    constexpr int DEPTH = MT == 4 ? 2 : TC_DEPTH;     // K-blocks in flight (register ring)
    float v[DEPTH][LD][8];
    const bool lrelu_in = p.in_act == FS2_ACT_LRELU;
    const float in_slope = p.in_slope;
    // per-thread (row, chunk) slots: fixed for the whole kernel
    int rowu[LD], offu[LD], off8[LD], goff[LD];
#pragma unroll
    for (int u = 0; u < LD; u++) {
      const int idx = u * TC_TTHREADS + wt;
      rowu[u] = idx < items ? (idx >> 1) : -1;
      offu[u] = (((idx & 1) * R) + (idx >> 1)) * 16;                  // smem byte offset inside a hi / lo plane
      off8[u] = (idx >> 1) * 16 + (idx & 1) * 8;                      // f8 split: byte offset inside one 16-channel E4M3 chunk
      goff[u] = (idx >> 1) * (int)p.xrs + (idx & 1) * 8;              // global float offset from the slab's first row
    }
    // load cursor (runs TC_DEPTH K-blocks ahead of the store cursor); no divisions on the per-K-block path
    int l_item = blockIdx.x, l_kb = 0, l_seg = 0;
    const float* l_xrow = nullptr;                     // &x[b][t0 - pad][0]; rows outside [0, T) are never dereferenced
    int l_tfirst = 0;
    bool l_interior = false;                           // warp-uniform: every slab row of the item exists
    auto l_set_item = [&]() {
      if (l_item < p.n_items) {
        const Item it = decode_item(p, l_item);
        const int s_tap = l_seg / p.seg_nkc, s_kc = l_seg - s_tap * p.seg_nkc;   // K-segment: one tap, one 256-channel chunk (0, 0 when nseg == 1)
        l_tfirst = it.t0 - p.pad + s_tap;
        l_xrow = p.x + (long long)it.b * p.xbs + (long long)l_tfirst * p.xrs + s_kc * p.Cin;
        l_interior = l_tfirst >= 0 && l_tfirst + rows_needed <= p.T;
      }
    };
    l_set_item();
    auto issue_loads = [&](float (&dst)[LD][8]) {     // loads K-block (l_item, l_kb), then advances the load cursor
      const float* xk = l_xrow + l_kb * TC_KB;
      if (l_interior) {
#pragma unroll
        for (int u = 0; u < LD; u++)
          if (rowu[u] >= 0) ldg256(dst[u], xk + goff[u]);
      } else {
#pragma unroll
        for (int u = 0; u < LD; u++) {
          const int t = l_tfirst + rowu[u];
          if (rowu[u] >= 0 && t >= 0 && t < p.T) {
            ldg256(dst[u], xk + goff[u]);
          } else {
#pragma unroll
            for (int j = 0; j < 8; j++) dst[u][j] = 0.f;              // conv zero padding
          }
        }
      }
      if (++l_kb == KBLOCKS) {
        l_kb = 0;
        if (++l_seg == p.nseg) { l_seg = 0; l_item += gridDim.x; }
        l_set_item();
      }
    };
    const int my_items = (p.n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int total = my_items * p.nseg * KBLOCKS;
#pragma unroll
    for (int d = 0; d < DEPTH; d++)
      if (d < total) issue_loads(v[d]);
    Ring ra;
#ifdef FS2_TC_TRACE
    int s_kb = 0, s_il = 0;                            // store cursor (for the debug timeline only)
#endif
    for (int base = 0; base < total; base += DEPTH) {
#pragma unroll
      for (int d = 0; d < DEPTH; d++) {
        const int seq = base + d;
        if (seq < total) {
#ifdef FS2_TC_TRACE
          if (wt == 0 && s_kb == 0) TC_STAMP(s_il, 0);
#endif
          mbar_wait(&emptyA[ra.idx], ra.phase ^ 1);
          unsigned char* hi = a_base + (size_t)ra.idx * 2 * a_plane;
          if (p.f8) {
            if (lrelu_in) tc_convert_store<true, true, LD>(v[d], rowu, offu, off8, hi, hi + a_plane, (uint32_t)R * 16, in_slope);
            else tc_convert_store<false, true, LD>(v[d], rowu, offu, off8, hi, hi + a_plane, (uint32_t)R * 16, in_slope);
          } else {
            if (lrelu_in) tc_convert_store<true, false, LD>(v[d], rowu, offu, off8, hi, hi + a_plane, (uint32_t)R * 16, in_slope);
            else tc_convert_store<false, false, LD>(v[d], rowu, offu, off8, hi, hi + a_plane, (uint32_t)R * 16, in_slope);
          }
          fence_proxy_async();                         // generic-proxy stores -> visible to the tensor core (async proxy)
          __syncwarp();
          if (lane == 0) mbar_arrive(&fullA[ra.idx]);   // one arrival per transform warp
          ra.advance(SA);
#ifdef FS2_TC_TRACE
          if (wt == 0 && s_kb == KBLOCKS - 1) TC_STAMP(s_il, 1);
          if (++s_kb == KBLOCKS) { s_kb = 0; s_il++; }
#endif
          if (seq + DEPTH < total) issue_loads(v[d]);
        }
      }
    }
  } else {
    // ===================== epilogue warps =====================
    const int q = warp & 3;                            // TMEM lane quarter this warp may access
    float* stage = stage_all + (warp - 2 - TC_TW) * TC_STAGE_FLOATS;
    const float inv_ws = __ldg(p.wt);                  // header: 1 / (power-of-two weight scale); identical for every utterance
    uint32_t itT = 0;
    Ring rt;
    if (p.nseg == 1) {
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, itT++, rt.advance(2)) {
      const uint32_t buf = rt.idx;
      const Item it = decode_item(p, item);
      mbar_wait(&accFull[buf], rt.phase);
      tc_fence_after();
      const uint32_t acc = tmem + buf * acc_set;
      if (warp == 2 + TC_TW && lane == 0) TC_STAMP((int)itT, 4);
      switch (p.out_act) {                             // uniform branch: keeps tanhf out of the other variants' inner loops
        case FS2_ACT_RELU: tc_epilogue_dispatch<FS2_ACT_RELU>(p, acc, stage, q, lane, it, inv_ws); break;
        case FS2_ACT_TANH: tc_epilogue_dispatch<FS2_ACT_TANH>(p, acc, stage, q, lane, it, inv_ws); break;
        case FS2_ACT_LRELU: tc_epilogue_dispatch<FS2_ACT_LRELU>(p, acc, stage, q, lane, it, inv_ws); break;
        default: tc_epilogue_dispatch<FS2_ACT_NONE>(p, acc, stage, q, lane, it, inv_ws); break;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&accEmpty[buf]);      // this warp's tcgen05.ld of the set have completed
      if (warp == 2 + TC_TW && lane == 0) TC_STAMP((int)itT, 5);
    }
    } else {
      // K-segmented conv: unit (item, seg) adds slice seg of the tile into y -- bias with the first slice; residual, alpha-free sum and
      // the pad-row mask with the last.  The units of one tile run back to back on this CTA and every thread re-reads what it wrote,
      // so the fp32 read-modify-write of y needs no further ordering.  No output activation (checked on the host).
      TcP u = p;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const Item it = decode_item(p, item);
        for (int seg = 0; seg < p.nseg; seg++, itT++, rt.advance(2)) {
          const uint32_t buf = rt.idx;
          const bool first = seg == 0, last = seg == p.nseg - 1;
          u.bias = first ? p.bias : nullptr;
          u.res = last ? p.res : nullptr;
          u.row_lens = last ? p.row_lens : nullptr;
          u.accumulate = (!first || p.accumulate) ? 1 : 0;
          const float seg_inv_ws = __ldg(reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(p.wt) + (long long)seg * p.seg_wbytes));
          mbar_wait(&accFull[buf], rt.phase);
          tc_fence_after();
          tc_epilogue_dispatch<FS2_ACT_NONE>(u, tmem + buf * acc_set, stage, q, lane, it, seg_inv_ws);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&accEmpty[buf]);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, p.tmem_cols);
  }
}

inline void conv_tc_launch(void (*kern)(const TcP), const TcP& p, unsigned grid, size_t smem, cudaStream_t s) {
  if (!p.pdl) {
    kern<<<grid, TC_THREADS, smem, s>>>(p);
    return;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kern, p);
}

// Each MT instantiation lives in its own translation unit (conv_tc_mt{1,2,4}.cu) so that the library builds in parallel.
cudaError_t conv_tc_prepare_mt1(int smem_bytes);
cudaError_t conv_tc_prepare_mt2(int smem_bytes);
cudaError_t conv_tc_prepare_mt4(int smem_bytes);
void conv_tc_launch_mt1(const TcP& p, unsigned grid, size_t smem, cudaStream_t s);
void conv_tc_launch_mt2(const TcP& p, unsigned grid, size_t smem, cudaStream_t s);
void conv_tc_launch_mt4(const TcP& p, unsigned grid, size_t smem, cudaStream_t s);

}  // namespace fs2
