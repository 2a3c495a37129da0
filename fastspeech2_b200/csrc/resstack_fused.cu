// One persistent tcgen05 kernel per HiFi-GAN upsample stage for the multi-receptive-field ResBlock group
//
//   y = (1/n_kernels) * sum_j ResBlock_j(x),   ResBlock_j: x <- conv_{k_j,1}(lrelu(conv_{k_j,d}(lrelu(x)))) + x  for d in dilations
//
// (hifigan/models.py:154-160 and ResBlock.forward :96-103; contract: fs2_resstack in include/fs2b200.h).  The per-layer design
// issued 18 conv launches per stage and moved every intermediate through HBM (~48 full-tensor passes); here a CTA owns one time
// tile of one utterance and keeps the whole chain on chip:
//
//   * slab = MT*128 rows starting H = max_j 6(k_j-1)... (sum of the receptive radii) rows before the tile: every conv is evaluated on
//     the full slab, garbage from the slab edges grows inward by one conv radius per layer and by construction stays inside the
//     H-row halo (halo recompute); rows outside the utterance [0, N) are forced to zero after every layer (Conv1d zero padding).
//   * activations live in shared memory ALREADY in tensor-core operand form: per 16-channel K-block an fp16 "hi" plane and an
//     E4M3 plane [lo * 2^12 | hi] (the two-MMA operand split of conv_tc_kernel.cuh, FS2_TC_VARIANT_F8), UMMA no-swizzle
//     K-major [16-byte K-chunk][row][16 B], so a conv tap is the same slab with the descriptor start advanced by tap*dilation
//     rows.  Two slabs: XA = lrelu(x) (conv1's operand), XT = lrelu(conv1 output) (conv2's operand).
//   * the residual stream x stays in TENSOR MEMORY in fp32 (MT*C columns) next to the MT accumulators (MT*C columns):
//     epilogue = tcgen05.ld acc (+ tcgen05.ld x) -> bias / residual / lrelu -> operand split -> st.shared into the other slab
//     (+ tcgen05.st x).  Thread == slab row, so consecutive lanes write consecutive 16-byte rows: conflict-free.
//   * weights stream through a cp.async.bulk ring exactly as in conv_tc_kernel.cuh (same tile images: the packer's f8 format).
//   * global I/O is TMA with tensor maps: the fp32 tile of x arrives as 3-D boxes [1][128 rows][32 channels] (128-byte swizzle;
//     rows outside [0, N) are zero-filled by the hardware = the conv's zero padding, and there is no bleed between utterances)
//     into the slab that is idle at that moment; the result leaves as boxes written from the other idle slab with a TMA store
//     (first kernel size) or TMA reduce-add (the others: the mean over kernel sizes accumulates in L2).  HBM sees x once and y once.
//   * a conv's MMAs are issued for two groups of tiles one after the other (weights streamed once per group), so the epilogue of
//     the first group overlaps the MMAs of the second and the next conv starts as soon as the tiles it reads are done.
//
// Roles: warp 0 weight producer, warp 1 MMA issuer, warps 2-9 "row" warps (TMEM lane quarter = warp % 4, column half = (warp-2)/4)
// that convert the loaded tile, run every epilogue and stage the result; lane 0 of warp 2 issues the tensor-map copies.
#include <cuda.h>

#include <type_traits>

#include "common.cuh"
#include "tc_format.cuh"

namespace fs2 {

constexpr int RS_MAXK = FS2_MAX_DIL + 4;   // kernel sizes per stage
constexpr int RS_GUARD = 1024;             // zeroed bytes in front of the first slab (taps reach up to 32 rows before row 0)
constexpr int RS_SB_MAX = 16;

struct RsConv { const unsigned char* w; const float* b; int taps, dil; };
struct RsP {
  int B, N;
  int n_kernels, n_dil;
  RsConv conv[RS_MAXK][FS2_MAX_DIL][2];
  int H, TILE, tiles_per_b, n_items;
  float alpha;
  int SB;
  int OBOX, n_oboxes;            // rows per output box (TILE = n_oboxes * OBOX, OBOX % 8 == 0)
  int TPS;                       // conv taps per weight stage (one bulk copy / one handshake)
  int accumulate;                // the first kernel size reduce-adds into y too
};

// 16 channels of one slab row -> operand planes of K-block kb (fp16 hi: two 16-byte chunks; E4M3: [lo*2^12 | hi*2]).
// `a` already carries the activation and the out-of-utterance zeroing.
__device__ __forceinline__ void rs_store16(unsigned char* kblk, uint32_t chunk_bytes, int row, const float (&a)[16]) {
  uint32_t hw[2][4], l8[2][2], h8[2][2];
  split_f16_e4m3(a, hw[0], l8[0], h8[0]);
  split_f16_e4m3(a + 8, hw[1], l8[1], h8[1]);
  unsigned char* p0 = kblk + (size_t)row * 16;
  *reinterpret_cast<uint4*>(p0) = make_uint4(hw[0][0], hw[0][1], hw[0][2], hw[0][3]);                   // plane 0, chunk 0: channels 0-7
  *reinterpret_cast<uint4*>(p0 + chunk_bytes) = make_uint4(hw[1][0], hw[1][1], hw[1][2], hw[1][3]);     // plane 0, chunk 1: channels 8-15
  *reinterpret_cast<uint4*>(p0 + 2 * chunk_bytes) = make_uint4(l8[0][0], l8[0][1], l8[1][0], l8[1][1]); // plane 1, chunk 0: E4M3 lo
  *reinterpret_cast<uint4*>(p0 + 3 * chunk_bytes) = make_uint4(h8[0][0], h8[0][1], h8[1][0], h8[1][1]); // plane 1, chunk 1: E4M3 hi
}

__device__ __forceinline__ float rs_lrelu(float v) { return fmaxf(v, 0.1f * v); }   // LRELU_SLOPE = 0.1 (hifigan/models.py:7)

// INDEP = false: the MT tiles form one contiguous slab (halo at its two ends only): whole ResBlock groups.
// INDEP = true : every 128-row tile is its own mini-slab with its own H-row halo (VT = 128 - 2H output rows per tile): single conv pairs, where
//                H is small.  The tiles of a work item are then independent, so the two MMA groups ping-pong with the row warps without
//                any cross-group wait; the result is staged in a buffer of its own and the next item's input boxes are prefetched into XT
//                as soon as the last conv's MMAs have retired, so the TMA latencies overlap the epilogue instead of the next item's start.
template <int C, int MT, bool INDEP>
__global__ void __launch_bounds__(64 + 8 * C, 1) resstack_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmy,
                                                                 const RsP p) {
  // one row warp per (TMEM lane quarter, 16-channel column group): 8 warps for 32 channels, 16 for 64 -- the epilogue is the
  // critical path between a conv's MMAs and the next conv's, so its latency is cut by spreading a row's columns over more warps
  constexpr int KB = C / 16, R = MT * 128, HC = 16, NG = 1, NRW = 4 * KB, RS_THREADS = 64 + 32 * NRW;
  constexpr int NH = C / 32;                                           // 32-channel (128-byte) column blocks of a row
  // tiles in the first MMA group.  The next conv's first group needs the epilogues of tiles 0 .. G0N: with a 3-tile slab {0} | {1,2}
  // lets it start after ONE tile's epilogue beyond the MMAs ({0,1} | {2} needed all three); with 4 tiles {0,1} | {2,3}.
  constexpr int G0N = INDEP ? MT / 2 : (MT == 3 ? 1 : 2);
  // (Tried and dropped: streaming a conv's weight stages ONCE and issuing the MMAs tile by tile -- 6.43 vs 5.67 ms on the 32-channel stage,
  // profiles/r02/resstack_bench_*.txt: the single issuing thread pays the per-stage bookkeeping four times per conv instead of twice.)
  constexpr uint32_t CHUNK = (uint32_t)R * 16, PLANE = 2 * CHUNK, KBLK = 2 * PLANE, SLAB = KB * KBLK;
  constexpr uint32_t WSTAGE = 64u * C;
  constexpr uint32_t TMEM_COLS = (2 * MT * C) <= 256 ? 256 : 512;
  constexpr uint32_t XBOX = 128 * 128;                                 // bytes of one input box [128 rows][32 ch] fp32
  static_assert(SLAB == (uint32_t)R * C * 4, "an operand slab has exactly the size of the fp32 tile it is built from");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned char* smem0 = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // swizzle atoms are 1024 bytes
  unsigned char* xa = smem0 + RS_GUARD;          // 1024-byte aligned: doubles as the swizzled staging area of the result
  unsigned char* xt = xa + SLAB;                 //                    doubles as the landing area of the fp32 input boxes
  unsigned char* stg = xt + SLAB;                // INDEP: staging area of the result boxes (otherwise XA is used)
  unsigned char* ring = INDEP ? stg + SLAB : xt + SLAB;
  const int VT = 128 - 2 * p.H;                  // INDEP: output rows per tile
  const uint32_t stage_bytes = (uint32_t)p.TPS * WSTAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)p.SB * stage_bytes);
  uint64_t* fullB = bars;                       // [RS_SB_MAX]
  uint64_t* emptyB = fullB + RS_SB_MAX;         // [RS_SB_MAX]
  uint64_t* accFull = emptyB + RS_SB_MAX;       // [MT] MMAs of one conv for tile m have retired
  uint64_t* rowsReady = accFull + 4;            // [MT] all 8 row warps have produced tile m of the next conv's operand slab (and drained its accumulator)
  uint64_t* xLoaded = rowsReady + 4;            // the round's input boxes have landed in XT
  uint64_t* xaFree = xLoaded + 1;               // the previous round's output boxes have been read out of XA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xaFree + 1);

  for (int i = tid; i < RS_GUARD / 16; i += RS_THREADS) reinterpret_cast<uint4*>(smem0)[i] = make_uint4(0, 0, 0, 0);
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < RS_SB_MAX; i++) { mbar_init(&fullB[i], 1); mbar_init(&emptyB[i], 1); }
    for (int i = 0; i < 4; i++) { mbar_init(&accFull[i], 1); mbar_init(&rowsReady[i], NRW); }
    mbar_init(xLoaded, 1); mbar_init(xaFree, 1);
    mbar_init_fence();
    tma_prefetch_map(&tmx);
    tma_prefetch_map(&tmy);
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t acc_col = 0, x_col = (uint32_t)(MT * C);     // accumulators | residual stream

  if (warp == 0) {
    // ===================== weight producer: every conv's stages once per tile group =====================
    if (lane == 0) {
      Ring rb;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x)
        for (int j = 0; j < p.n_kernels; j++)
          for (int d = 0; d < p.n_dil; d++)
            for (int c2 = 0; c2 < 2; c2++) {
              const RsConv cv = p.conv[j][d][c2];
              for (int grp = 0; grp < 2; grp++) {       // the weights are streamed once per tile group
                const unsigned char* src = cv.w + TC_HDR;   // tiles are ordered [kb][tap]: the taps of one K-block are contiguous
                for (int kb = 0; kb < KB; kb++)
                  for (int tap = 0; tap < cv.taps; tap += p.TPS) {
                    const uint32_t bytes = (uint32_t)min(p.TPS, cv.taps - tap) * WSTAGE;
                    mbar_wait(&emptyB[rb.idx], rb.phase ^ 1);
                    mbar_expect_tx(&fullB[rb.idx], bytes);
                    bulk_g2s(ring + (size_t)rb.idx * stage_bytes, src, bytes, &fullB[rb.idx]);
                    src += bytes;
                    rb.advance((uint32_t)p.SB);
                  }
              }
            }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t leader = elect_one();
    const uint32_t idesc = umma_idesc_f16(C);
    const uint64_t a_const = umma_desc(0, CHUNK, 128), b_const = umma_desc(0, (uint32_t)C * 16, 128);
    const uint32_t xa16 = smem_u32(xa) >> 4, xt16 = smem_u32(xt) >> 4;
    Ring rb;
    uint32_t ev = 0;                                        // rowsReady events consumed so far (the same for every tile)
    // the MMAs of one tile group of one conv: tiles [MLO, MLO + MCNT)
    auto issue_group = [&](auto mlo_c, auto mcnt_c, const RsConv& cv, uint32_t slab16) {
      constexpr int MLO = decltype(mlo_c)::value, MCNT = decltype(mcnt_c)::value;
      const int pad = (cv.taps - 1) * cv.dil / 2;
      for (int kb = 0; kb < KB; kb++) {
        const uint64_t a_hi = a_const | (uint64_t)((slab16 + kb * (KBLK >> 4)) & 0x3fff);
        int row_off = -pad + MLO * 128;
        for (int tap = 0; tap < cv.taps; tap += p.TPS, rb.advance((uint32_t)p.SB)) {
          const int n = min(p.TPS, cv.taps - tap);
          mbar_wait(&fullB[rb.idx], rb.phase);
          tc_fence_after();
          if (leader) {
            uint64_t b_hi = b_const | (uint64_t)(smem_u32(ring + (size_t)rb.idx * stage_bytes) >> 4);
            for (int t = 0; t < n; t++, b_hi += WSTAGE >> 4, row_off += cv.dil) {
              const uint64_t b_x8 = b_hi + ((2u * C * 16u) >> 4);
              const uint64_t ah0 = a_hi + (uint64_t)(int64_t)row_off;      // start-address field += rows (16 B each); never carries out of the field
              const uint64_t ax0 = ah0 + (PLANE >> 4);
              const uint32_t first = (kb | tap | t) ? 1u : 0u;
#pragma unroll
              for (int m = 0; m < MCNT; m++) tc_mma_f16(tmem + acc_col + (MLO + m) * C, ah0 + m * 128, b_hi, idesc, first);
#pragma unroll
              for (int m = 0; m < MCNT; m++) tc_mma_f8(tmem + acc_col + (MLO + m) * C, ax0 + m * 128, b_x8, idesc, 1u);
            }
            tc_commit(&emptyB[rb.idx]);
          } else {
            row_off += n * cv.dil;
          }
          __syncwarp();
        }
      }
      if (leader) {
#pragma unroll
        for (int m = 0; m < MCNT; m++) tc_commit(&accFull[MLO + m]);
      }
      __syncwarp();
    };
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      for (int j = 0; j < p.n_kernels; j++) {
        for (int d = 0; d < p.n_dil; d++) {
          for (int c2 = 0; c2 < 2; c2++) {
            const RsConv cv = p.conv[j][d][c2];
            const uint32_t slab16 = c2 == 0 ? xa16 : xt16;
            // Group 0 reads operand rows of tiles 0 .. G0N (one tile of halo), group 1 the rest: every tile's "ready" phase is waited
            // exactly once per conv, before the next phase of that tile can complete (it needs this conv's MMAs).
            constexpr int G0WAIT = INDEP ? G0N : (G0N + 1 < MT ? G0N + 1 : MT);   // independent tiles need no neighbour's epilogue
#pragma unroll
            for (int m = 0; m < G0WAIT; m++) mbar_wait(&rowsReady[m], ev & 1);
            tc_fence_after();
            issue_group(std::integral_constant<int, 0>{}, std::integral_constant<int, G0N>{}, cv, slab16);
#pragma unroll
            for (int m = G0WAIT; m < MT; m++) mbar_wait(&rowsReady[m], ev & 1);
            tc_fence_after();
            issue_group(std::integral_constant<int, G0N>{}, std::integral_constant<int, MT - G0N>{}, cv, slab16);
            ev++;
          }
        }
        // The round's final epilogue does not signal: a row warp's next arrival on rowsReady[m] is its conversion of the NEXT round's
        // input, which it reaches only after finishing that epilogue (program order).
      }
    }
  } else {
    // ===================== row warps: input conversion, epilogues, result staging =====================
    const int q = warp & 3, h = (warp - 2) >> 2;
    const int col0 = h * HC;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const bool io = warp == 2 && lane == 0;                 // issues every tensor-map copy (bulk groups are per thread)
    uint32_t acc_phase = 0, round_phase = 0;
    bool stores_pending = false;
    // first slab row of tile m of an item starting at output row t0
    auto tile_g0 = [&](int t0, int m) { return INDEP ? t0 + m * VT - p.H : t0 - p.H + m * 128; };
    auto load_item = [&](int it) {                          // io thread: the item's fp32 input boxes -> XT
      const int bb = it / p.tiles_per_b, tt = (it - bb * p.tiles_per_b) * p.TILE;
      mbar_expect_tx(xLoaded, (uint32_t)(MT * NH) * XBOX);
#pragma unroll
      for (int hh = 0; hh < NH; hh++)
#pragma unroll
        for (int m = 0; m < MT; m++) tma_load_3d(xt + (size_t)(hh * MT + m) * XBOX, &tmx, hh * 32, tile_g0(tt, m), bb, xLoaded);
    };
    if (INDEP && io && (int)blockIdx.x < p.n_items) load_item(blockIdx.x);
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const int b = item / p.tiles_per_b;
      const int t0 = (item - b * p.tiles_per_b) * p.TILE;
      for (int j = 0; j < p.n_kernels; j++) {
        // ---- input: TMA boxes of x -> XT (idle: the last conv that read it has retired), then residual stream -> TMEM, lrelu(x) -> XA
        if (io) {
          if (!INDEP) load_item(item);                      // (INDEP: prefetched while the previous item finished)
          if (stores_pending) tma_wait_reads();             // previous result boxes have been read out of their staging area
          mbar_arrive(xaFree);
        }
        stores_pending = true;
        mbar_wait(xLoaded, round_phase);
        if (!INDEP) mbar_wait(xaFree, round_phase);         // (INDEP: the staging area is separate; waited before it is rewritten)
#pragma unroll 1
        for (int m = 0; m < MT; m++) {
          const int r128 = q * 32 + lane, row = m * 128 + r128;
          const unsigned char* box = xt + (size_t)((col0 >> 5) * MT + m) * XBOX;
#pragma unroll
          for (int gi = 0; gi < NG; gi++) {
            const int c16 = ((col0 & 31) >> 2) + gi * 4;    // first 16-byte chunk of these 16 channels inside the 128-byte row
            float v[16];
#pragma unroll
            for (int k4 = 0; k4 < 4; k4++) {
              const float4 u = *reinterpret_cast<const float4*>(box + sw128(r128, c16 + k4));
              v[4 * k4] = u.x; v[4 * k4 + 1] = u.y; v[4 * k4 + 2] = u.z; v[4 * k4 + 3] = u.w;
            }
            uint32_t raw[16];
#pragma unroll
            for (int k = 0; k < 16; k++) raw[k] = __float_as_uint(v[k]);
            tc_st16(tmem + lane_base + x_col + m * C + col0 + gi * 16, raw);
#pragma unroll
            for (int k = 0; k < 16; k++) v[k] = rs_lrelu(v[k]);       // rows outside the utterance arrive as zeros (TMA fill)
            rs_store16(xa + (size_t)((col0 >> 4) + gi) * KBLK, CHUNK, row, v);
          }
          tc_wait_st();
          fence_proxy_async();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&rowsReady[m]);
        }
        row_warps_sync<32 * NRW>();        // every warp has finished reading the boxes: conv1's epilogue may overwrite XT
        for (int d = 0; d < p.n_dil; d++) {
          const bool last = d == p.n_dil - 1;
          for (int c2 = 0; c2 < 2; c2++) {
            const RsConv cv = p.conv[j][d][c2];
            const float inv_s = __ldg(reinterpret_cast<const float*>(cv.w));
            float4 bias[NG][4];                               // this warp's HC bias values: loaded once per conv, while its MMAs run
#pragma unroll
            for (int gi = 0; gi < NG; gi++)
#pragma unroll
              for (int k4 = 0; k4 < 4; k4++) bias[gi][k4] = __ldg(reinterpret_cast<const float4*>(cv.b + col0 + gi * 16) + k4);
            if (INDEP && c2 == 1 && last) mbar_wait(xaFree, round_phase);   // the previous item's result boxes have left the staging area
#pragma unroll 1
            for (int m = 0; m < MT; m++) {
              const int r128 = q * 32 + lane, row = m * 128 + r128;
              const int g = tile_g0(t0, m) + r128;
              const bool in = g >= 0 && g < p.N;
              mbar_wait(&accFull[m], acc_phase);
              tc_fence_after();
              if (INDEP && io && c2 == 1 && last && m == MT - 1 && item + (int)gridDim.x < p.n_items)
                load_item(item + gridDim.x);           // every MMA that read XT has retired: prefetch the next item's input boxes
#pragma unroll
              for (int gi = 0; gi < NG; gi++) {
                const int cc = col0 + gi * 16;
                uint32_t av[16], xv[16];
                tc_ld16_nowait(tmem + lane_base + acc_col + m * C + cc, av);
                if (c2 == 1) tc_ld16_nowait(tmem + lane_base + x_col + m * C + cc, xv);
                tc_wait_ld();
                float v[16];
#pragma unroll
                for (int k4 = 0; k4 < 4; k4++) {
                  const float4 bb = bias[gi][k4];
                  v[4 * k4] = fmaf(__uint_as_float(av[4 * k4]), inv_s, bb.x);
                  v[4 * k4 + 1] = fmaf(__uint_as_float(av[4 * k4 + 1]), inv_s, bb.y);
                  v[4 * k4 + 2] = fmaf(__uint_as_float(av[4 * k4 + 2]), inv_s, bb.z);
                  v[4 * k4 + 3] = fmaf(__uint_as_float(av[4 * k4 + 3]), inv_s, bb.w);
                }
                if (c2 == 0) {
                  // conv1: lrelu -> conv2's operand slab
#pragma unroll
                  for (int k = 0; k < 16; k++) v[k] = in ? rs_lrelu(v[k]) : 0.f;
                  rs_store16(xt + (size_t)(cc >> 4) * KBLK, CHUNK, row, v);
                } else {
#pragma unroll
                  for (int k = 0; k < 16; k++) v[k] += __uint_as_float(xv[k]);          // + residual
                  if (!last) {
                    uint32_t raw[16];
#pragma unroll
                    for (int k = 0; k < 16; k++) raw[k] = __float_as_uint(v[k]);
                    tc_st16(tmem + lane_base + x_col + m * C + cc, raw);
#pragma unroll
                    for (int k = 0; k < 16; k++) v[k] = in ? rs_lrelu(v[k]) : 0.f;
                    rs_store16(xa + (size_t)(cc >> 4) * KBLK, CHUNK, row, v);
                  } else if (INDEP ? (r128 >= p.H && r128 < p.H + VT) : (row >= p.H && row < p.H + p.TILE)) {
                    // result of this kernel size, alpha * x (mean over kernel sizes, models.py:154-160): staged (XA, idle since conv1 of
                    // this pair has retired; INDEP: the separate staging area) as swizzled [OBOX rows][32 channels] boxes for the TMA
                    // store / reduce-add
                    const int ro = INDEP ? r128 - p.H : row - p.H, bx = INDEP ? m : ro / p.OBOX, rb_ = INDEP ? ro : ro - bx * p.OBOX;
                    unsigned char* obox = (INDEP ? stg : xa) + (size_t)((cc >> 5) * p.n_oboxes + bx) * ((size_t)p.OBOX * 128);
                    const int c16 = (cc & 31) >> 2;
#pragma unroll
                    for (int k4 = 0; k4 < 4; k4++)
                      *reinterpret_cast<float4*>(obox + sw128(rb_, c16 + k4)) =
                          make_float4(v[4 * k4] * p.alpha, v[4 * k4 + 1] * p.alpha, v[4 * k4 + 2] * p.alpha, v[4 * k4 + 3] * p.alpha);
                  }
                }
              }
              if (c2 == 1 && last) {
                tc_fence_before();                     // accumulator / residual reads done; the next signal is the next round's input
              } else {
                if (c2 == 1) tc_wait_st();
                fence_proxy_async();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&rowsReady[m]);
              }
            }
            acc_phase ^= 1;
          }
        }
        round_phase ^= 1;
        // ---- result boxes -> y: store for the first kernel size, reduce-add (in L2) for the others; rows beyond N are clipped by the TMA
        fence_proxy_async();
        row_warps_sync<32 * NRW>();
        if (io) {
          if (!INDEP) tma_wait_all();   // the previous kernel size's boxes are complete in L2 before this one's reduce-add (a round earlier: no wait in practice)
          for (int hh = 0; hh < NH; hh++)
            for (int bx = 0; bx < p.n_oboxes; bx++) {
              const unsigned char* src = (INDEP ? stg : xa) + (size_t)(hh * p.n_oboxes + bx) * ((size_t)p.OBOX * 128);
              if (j == 0 && !p.accumulate) tma_store_3d(&tmy, hh * 32, t0 + bx * p.OBOX, b, src);
              else tma_reduce_add_3d(&tmy, hh * 32, t0 + bx * p.OBOX, b, src);
            }
          tma_commit();
        }
      }
    }
    if (io) tma_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

// ------------------------------------------------------------------ host side
static size_t rs_smem_bytes(int C, int MT, int SB, int TPS, bool indep) {
  const size_t slab = (size_t)(C / 16) * 4 * (MT * 128) * 16;
  return RS_GUARD + (indep ? 3 : 2) * slab + (size_t)SB * TPS * 64 * C + (2 * RS_SB_MAX + 10) * 8 + 16 + 1024;   // + worst-case 1024-byte alignment slack
}

// Launch plan (pure host logic): out[12] = {MT, H (halo rows per side), TILE (output rows per work item), work items, grid, weight ring
// stages, dynamic shared memory bytes, TMEM columns, rows per output box, output boxes per tile and 32-channel block, taps per weight stage,
// independent-tile mode}
int resstack_plan(const fs2_resstack_args* a, int num_sms, int* out) {
  if (!a || a->B <= 0 || a->N <= 0 || num_sms <= 0) return FS2_ERR_ARG;
  if (a->C != 32 && a->C != 64) return FS2_ERR_UNSUPPORTED;
  if (a->n_kernels <= 0 || a->n_kernels > RS_MAXK || a->n_dil <= 0 || a->n_dil > FS2_MAX_DIL) return FS2_ERR_ARG;
  int H = 0;
  for (int j = 0; j < a->n_kernels; j++) {
    const int k = a->k[j];
    if (k <= 0 || !(k & 1)) return FS2_ERR_UNSUPPORTED;
    int hj = 0;
    for (int d = 0; d < a->n_dil; d++) {
      const int dil = a->dil[j][d];
      if (dil <= 0 || (k - 1) * dil / 2 > 32) return FS2_ERR_UNSUPPORTED;      // taps reach at most 32 rows outside a tile (guard / neighbour tile)
      hj += (k - 1) * dil / 2 + (k - 1) / 2;
    }
    H = hj > H ? hj : H;
  }
  H = (H + 3) & ~3;                             // output boxes are whole swizzle atoms (multiples of 8 rows)
  // One kernel size with a small receptive radius on 32 channels: independent 128-row tiles, each with its own halo, the next work
  // item's input prefetched.  Measured (profiles/r02/pair_bench_indep.txt): 32 channels k = 3: 380 us against 476 us for the shared-halo
  // slab; 64 channels: no gain at k = 3 (549 / 556 us), a loss from k = 7 on (the per-tile halo recompute outweighs the overlap).
  const bool indep = a->n_kernels == 1 && a->C == 32 && H <= 16;
  const int MT = a->C == 32 ? 4 : 3;   // bounded by shared memory (slabs of 4*C bytes per row)
  int TILE = 0, obox = 0, n_oboxes = 0;
  if (indep) {
    obox = 128 - 2 * H; n_oboxes = MT; TILE = MT * obox;
  } else {
    // the result leaves as TMA boxes of `obox` rows (a multiple of 8, <= 256) that tile TILE exactly: widen the halo by up to 32 rows
    // until TILE splits into at most 12 boxes (e.g. 384 - 2*4 = 376 = 47 x 8 would need 47 stores; 384 - 2*8 = 368 = 2 x 184)
    for (int hc = H; hc <= H + 32 && !obox; hc += 4) {
      const int tile = MT * 128 - 2 * hc;
      if (tile < 64) break;
      for (int r = 256; r >= 8; r -= 8)
        if (tile % r == 0 && tile / r <= 12) { TILE = tile; obox = r; H = hc; break; }
    }
    if (!obox) return FS2_ERR_UNSUPPORTED;
    n_oboxes = TILE / obox;
  }
  const long long tiles_per_b = (a->N + TILE - 1) / TILE, items = tiles_per_b * a->B;
  if (items > 0x7fffffffLL) return FS2_ERR_UNSUPPORTED;
  const int TPS = a->C == 32 ? 4 : 2;           // taps per weight stage: 8 KB stages (fewer handshakes per MMA; conv_tc measured -10..-25 %)
  int SB = a->C == 32 && !indep ? 8 : 4;
  while (SB > 2 && rs_smem_bytes(a->C, MT, SB, TPS, indep) > 227 * 1024) SB--;
  if (rs_smem_bytes(a->C, MT, SB, TPS, indep) > 227 * 1024) return FS2_ERR_UNSUPPORTED;
  out[0] = MT; out[1] = H; out[2] = TILE; out[3] = (int)items; out[4] = items < num_sms ? (int)items : num_sms; out[5] = SB;
  out[6] = (int)rs_smem_bytes(a->C, MT, SB, TPS, indep); out[7] = 2 * MT * a->C <= 256 ? 256 : 512; out[8] = obox; out[9] = n_oboxes;
  out[10] = TPS; out[11] = indep ? 1 : 0;
  return FS2_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static std::atomic<void*> cached{nullptr};
  void* f = cached.load(std::memory_order_acquire);
  if (!f) {
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) return nullptr;
    cached.store(f, std::memory_order_release);
  }
  return reinterpret_cast<EncodeTiledFn>(f);
}
// fp32 [B][N][C] contiguous as a rank-3 map, boxes of [1][rows][32 channels] with the 128-byte swizzle, zero fill outside the tensor
static int make_map(CUtensorMap* tm, const float* base, int B, int N, int C, int box_rows) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return FS2_ERR_UNSUPPORTED;
  const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)N, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)C * 4, (cuuint64_t)N * C * 4};
  const cuuint32_t box[3] = {32, (cuuint32_t)box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? FS2_OK : FS2_ERR_CUDA - 1;
}

int resstack(const fs2_resstack_args* a, cudaStream_t s) {
  if (!a || !a->x || !a->y) return FS2_ERR_ARG;
  if (!aligned16(a->x) || !aligned16(a->y)) return FS2_ERR_ARG;
  if (a->B <= 0 || a->N <= 0 || a->C <= 0) return FS2_ERR_ARG;
  {  // not in place: a work item re-reads halo rows of x that its neighbours' results would already have overwritten
    const unsigned char *xb = reinterpret_cast<const unsigned char*>(a->x), *yb = reinterpret_cast<const unsigned char*>(a->y);
    const size_t bytes = (size_t)a->B * a->N * a->C * sizeof(float);
    if (xb < yb + bytes && yb < xb + bytes) return FS2_ERR_ARG;
  }
  int derr = FS2_OK;
  DevState* dv = dev_state(&derr);
  if (!dv) return derr;
  int plan[12];
  FS2_TRY(resstack_plan(a, dv->num_sms.load(std::memory_order_relaxed), plan));
  FS2_TRY(setup_once(dv->fused_ready, [] {
    const int mx = 227 * 1024;
    cudaError_t e = cudaFuncSetAttribute(resstack_kernel<32, 4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(resstack_kernel<64, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(resstack_kernel<32, 4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    return e;
  }));
  RsP p{};
  p.B = a->B; p.N = a->N;
  p.n_kernels = a->n_kernels; p.n_dil = a->n_dil;
  double flops = 0;
  for (int j = 0; j < a->n_kernels; j++)
    for (int d = 0; d < a->n_dil; d++) {
      if (!a->w1_tc[j][d] || !a->w2_tc[j][d] || !a->b1[j][d] || !a->b2[j][d]) return FS2_ERR_ARG;
      if (!aligned16(a->w1_tc[j][d]) || !aligned16(a->w2_tc[j][d]) || !aligned16(a->b1[j][d]) || !aligned16(a->b2[j][d])) return FS2_ERR_ARG;
      p.conv[j][d][0] = RsConv{reinterpret_cast<const unsigned char*>(a->w1_tc[j][d]), a->b1[j][d], a->k[j], a->dil[j][d]};
      p.conv[j][d][1] = RsConv{reinterpret_cast<const unsigned char*>(a->w2_tc[j][d]), a->b2[j][d], a->k[j], 1};
      flops += 2.0 * 2.0 * a->B * (double)a->N * a->C * a->C * a->k[j];
    }
  p.H = plan[1]; p.TILE = plan[2]; p.tiles_per_b = (a->N + p.TILE - 1) / p.TILE; p.n_items = plan[3];
  p.alpha = a->alpha > 0.f ? a->alpha : 1.f / (float)a->n_kernels; p.accumulate = a->accumulate; p.SB = plan[5]; p.OBOX = plan[8]; p.n_oboxes = plan[9]; p.TPS = plan[10];
  alignas(64) CUtensorMap tmx, tmy;
  FS2_TRY(make_map(&tmx, a->x, a->B, a->N, a->C, 128));
  FS2_TRY(make_map(&tmy, a->y, a->B, a->N, a->C, p.OBOX));
  prof_before(s);
  if (plan[11]) {
    resstack_kernel<32, 4, true><<<plan[4], 64 + 8 * 32, plan[6], s>>>(tmx, tmy, p);      // (the plan selects it for 32 channels only)
  } else {
    if (a->C == 32) resstack_kernel<32, 4, false><<<plan[4], 64 + 8 * 32, plan[6], s>>>(tmx, tmy, p);
    else resstack_kernel<64, 3, false><<<plan[4], 64 + 8 * 64, plan[6], s>>>(tmx, tmy, p);
  }
  prof_after(s, 0, flops);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

}  // namespace fs2
