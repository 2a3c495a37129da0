// Host side of the tcgen05 implicit-GEMM Conv1d: shape support, work-item / ring heuristics, launch.
// Device code: conv_tc_kernel.cuh (instantiated in conv_tc_mt{1,2,4}.cu).
#include "conv_tc_kernel.cuh"

namespace fs2 {

// ------------------------------------------------------------------ host side
#ifdef FS2_DEBUG_KNOBS
long long* g_tc_trace = nullptr;  // debug: set through fs2_debug_set_tc_trace (per-item role timeline)
#else
static constexpr long long* g_tc_trace = nullptr;
#endif

static int pow2_cols(int c) {
  int v = 32;
  while (v < c) v <<= 1;
  return v;
}

int conv_tc_nb(int N) {  // output channels per work item: NB <= 128 keeps two accumulator sets of MT=2 tiles inside TMEM
  if (N % 16) return 0;
  if (N <= 128) return N;
  for (int nb = 128; nb >= 16; nb -= 16)
    if (N % nb == 0) return nb;
  return 0;
}

bool conv_tc_supported(const fs2_conv1d_args* a) {
  if (!a || a->Cin % TC_KB || a->N % 16 || conv_tc_nb(a->N) == 0) return false;
  if ((a->x_row_stride & 7) || (a->x_batch_stride & 7) || (reinterpret_cast<uintptr_t>(a->x) & 31u)) return false;   // 256-bit loads
  if ((a->y_row_stride & 3) || (a->y_batch_stride & 3)) return false;
  if ((long long)(TC_LD * TC_TTHREADS) * a->x_row_stride > 0x7fffffffLL) return false;                                // 32-bit row offsets
  if (a->res && ((a->res_row_stride & 3) || (a->res_batch_stride & 3))) return false;
  if (a->in_act != FS2_ACT_NONE && a->in_act != FS2_ACT_LRELU) return false;
  if (a->in_act == FS2_ACT_LRELU && !(a->in_slope >= 0.f && a->in_slope <= 1.f)) return false;   // max(x, slope*x) form
  if ((a->taps - 1) * a->dilation > TC_LD * TC_TTHREADS / TC_CHUNKS - 128) return false;
  return true;
}

#ifdef FS2_DEBUG_KNOBS
int g_tc_pdl = 0;                  // programmatic dependent launch: 0 = off (default), 1 = short launches only, 2 = every launch.
                                   // Measured with the three modes interleaved step by step (scripts/pdl_ab.py,
                                   // profiles/r01_pdl_ab.txt): no gain on either forward (39.5 / 40.8 / 42.2 ms per step), so it
                                   // stays off; debug switch fs2_debug_set_tc_pdl
int g_tc_tune[4] = {0, 0, 0, 0};   // debug overrides: SA, SB, TPS, grid (0 = heuristic); set through fs2_debug_set_tc_tuning
#else                              // shipped build: no mutable process-wide state
static constexpr int g_tc_pdl = 0;
static constexpr int g_tc_tune[4] = {0, 0, 0, 0};
#endif

// Shape-derived launch plan (pure host logic, no CUDA calls): work-item shape, accumulator grouping, ring depths, shared /
// tensor memory budget, grid.  Returns FS2_OK or FS2_ERR_UNSUPPORTED.  Exposed as fs2_conv_tc_plan so that the heuristics'
// invariants are testable without a GPU (tests/test_abi.py).
static int conv_tc_plan(const fs2_conv1d_args* a, int num_sms, TcP& p, size_t& smem, int& grid) {
  const bool nb64 = (a->tc_variant & FS2_TC_VARIANT_NB64) != 0;   // 64-channel work items: separate accumulators for hi*hi and the cross terms
  p.NB = nb64 ? (a->N % 64 == 0 ? 64 : (a->N < 64 && a->N % 16 == 0 ? a->N : 0)) : conv_tc_nb(a->N);
  if (p.NB == 0) return FS2_ERR_UNSUPPORTED;
  p.acc_stride = (p.NB + 31) & ~31;
  const int halo = (a->taps - 1) * a->dilation;
  const int tiles128 = (a->T + 127) / 128;
  int mt = 2;                                          // two accumulator sets of MT tiles: 2*MT*TG*acc_stride <= 512 columns
  if (p.acc_stride <= 64 && tiles128 >= 4 && 4 * 128 + halo <= 5 * TC_TTHREADS / TC_CHUNKS) mt = 4;   // narrow layers: amortise per-item handshakes
  if (g_tc_tune[3] == -1) mt = 2;                      // debug: force MT = 2
  if (nb64 && mt > 2) mt = 2;                          // keeps TG = 2 (two accumulator sets of MT*2 tiles of 64 columns = 512)
  if (mt > tiles128) mt = tiles128 >= 2 ? 2 : 1;
  if (mt == 2 && mt * 128 + halo > TC_LD * TC_TTHREADS / TC_CHUNKS) mt = 1;   // rows one register-ring slot can hold
  // small problems (decoder projections, attention PV): prefer more, smaller work items when MT = 2 would leave SMs idle
  if (mt == 2 && 2LL * (a->N / p.NB) * a->B * ((a->T + 255) / 256) <= num_sms) mt = 1;   // measured: helps at <= 1/2 wave, hurts K-heavy layers at ~1 wave
  int R = mt * 128 + halo;
  R += (12 - (R & 7)) & 7;                             // R % 8 == 4: conflict-free transform stores (2 chunks per row)
  p.MT = mt; p.R = R;
  // narrow layers: hi*hi and the two cross terms accumulate in separate TMEM tiles (summed in fp32 round-to-nearest by the
  // epilogue) while two accumulator sets still fit in 512 columns
  p.TG = (mt == 4 ? p.acc_stride <= 32 : p.acc_stride <= 64) ? 2 : 1;
  const size_t fixed = 4 * TC_STAGE_FLOATS * sizeof(float) + (2 * TC_SA_MAX + 2 * TC_SB_MAX + 4) * 8 + 16;
  const size_t tap_bytes = (size_t)2 * TC_CHUNKS * p.NB * 16;
  // Taps per weight stage: measured (scripts/tc_tune.py, profiles/r01_tc_tune.txt) -- grouping 4 taps per bulk copy / handshake
  // is 10-25 % faster for the k = 5..11 layers at every channel width; k <= 3 layers are best with one tap per stage.
  int tps = a->taps >= 5 ? 4 : 1;
  if (g_tc_tune[2] > 0) tps = g_tc_tune[2];
  if (tps > a->taps) tps = a->taps;
  p.TPS = tps;
  const size_t a_stage = (size_t)2 * TC_CHUNKS * R * 16, b_stage = (size_t)tps * tap_bytes;
  const size_t budget = 226 * 1024;
  const int kblocks = a->Cin / TC_KB;
  // Slab ring depth, measured per shape class (scripts/tc_tune_sa.py, profiles/r01_tc_tune_sa.txt): the ring spans work items, so
  // even 2-K-block layers want 3 stages (-10..-14 % on the 32-channel stage against 2); k <= 3 layers like 5 (-4..-6 %); a
  // 4th MT=4 stage is not worth shrinking the weight ring for.
  int sa = 3, sb = tps > 1 ? 4 : TC_SB_MAX;
  if (mt < 4 && a->taps <= 3) sa = 5;
  else if (mt < 4 && kblocks >= 4) sa = 4;
  while (fixed + sa * a_stage + sb * b_stage > budget && sa > 3) sa--;
  while (fixed + sa * a_stage + sb * b_stage > budget && sb > 3) sb--;
  while (fixed + sa * a_stage + sb * b_stage > budget && sa > 2) sa--;
  while (fixed + sa * a_stage + sb * b_stage > budget && sb > 2) sb--;
  if (fixed + sa * a_stage + sb * b_stage > budget) return FS2_ERR_UNSUPPORTED;
  if (g_tc_tune[0] > 0) sa = g_tc_tune[0] > TC_SA_MAX ? TC_SA_MAX : g_tc_tune[0];
  if (g_tc_tune[1] > 0) sb = g_tc_tune[1] > TC_SB_MAX ? TC_SB_MAX : g_tc_tune[1];
  if (fixed + sa * a_stage + sb * b_stage > budget) return FS2_ERR_UNSUPPORTED;
  p.SA = sa; p.SB = sb;
  smem = fixed + sa * a_stage + sb * b_stage;
  p.tmem_cols = pow2_cols(2 * mt * p.TG * p.acc_stride);
  p.tiles_per_batch = (a->T + mt * 128 - 1) / (mt * 128);
  const long long n_items = (long long)(a->N / p.NB) * a->B * p.tiles_per_batch;
  if (n_items > 0x7fffffffLL) return FS2_ERR_UNSUPPORTED;
  p.n_items = (int)n_items;
  p.pdl = g_tc_pdl == 2 || (g_tc_pdl == 1 && n_items <= 4LL * num_sms);
  grid = n_items < num_sms ? (int)n_items : num_sms;
  if (g_tc_tune[3] > 0 && g_tc_tune[3] < grid) grid = g_tc_tune[3];
  return FS2_OK;
}

// out[12] = {NB, MT, TG, SA, SB, TPS, R, tmem_cols, tiles_per_batch, n_items, grid, dynamic smem bytes}
int conv_tc_plan_query(const fs2_conv1d_args* a, int num_sms, int* out) {
  if (!a || !out || num_sms <= 0 || a->B <= 0 || a->T <= 0 || a->Cin <= 0 || a->N <= 0 || a->taps <= 0) return FS2_ERR_ARG;
  if (!conv_tc_supported(a)) return FS2_ERR_UNSUPPORTED;
  TcP p{};
  size_t smem = 0;
  int grid = 0;
  const int rc = conv_tc_plan(a, num_sms, p, smem, grid);
  if (rc != FS2_OK) return rc;
  const int v[12] = {p.NB, p.MT, p.TG, p.SA, p.SB, p.TPS, p.R, p.tmem_cols, p.tiles_per_batch, p.n_items, grid, (int)smem};
  for (int i = 0; i < 12; i++) out[i] = v[i];
  return FS2_OK;
}

// `wt` must be the tiled layout produced by fastspeech2_b200.packing.pack_conv_tc (see fs2b200.h)
int conv1d_tc(const fs2_conv1d_args* a, const float* wt, unsigned variant, cudaStream_t s, long long wt_batch_stride) {
  if (!a || !a->x || !wt || !a->y) return FS2_ERR_ARG;
  if (a->B <= 0 || a->T <= 0 || a->Cin <= 0 || a->N <= 0 || a->taps <= 0) return FS2_ERR_ARG;
  if (!conv_tc_supported(a)) return FS2_ERR_UNSUPPORTED;
  if (!aligned16(a->x) || !aligned16(wt) || !aligned16(a->y) || (a->res && !aligned16(a->res))) return FS2_ERR_ARG;
  // K-segmented evaluation in ONE launch (FS2_TC_VARIANT_SEGMENTED): the work units are (tile, tap, 256-channel chunk)
  fs2_conv1d_args seg_args;
  int nseg = 1, seg_nkc = 1;
  if (variant & FS2_TC_VARIANT_SEGMENTED) {
    if (!(variant & FS2_TC_VARIANT_NB64) || a->Cin % 256 || a->N % 64 || a->dilation != 1 || a->alpha != 1.f || a->out_act != FS2_ACT_NONE ||
        wt_batch_stride != 0)
      return FS2_ERR_UNSUPPORTED;
    seg_nkc = a->Cin / 256; nseg = a->taps * seg_nkc;
    seg_args = *a;
    seg_args.Cin = 256; seg_args.taps = 1;          // shape of one slice: ring / tile planning happens on this
  }
  const fs2_conv1d_args* plan_args = nseg > 1 || (variant & FS2_TC_VARIANT_SEGMENTED) ? &seg_args : a;
  int derr = FS2_OK;
  DevState* dv = dev_state(&derr);                      // state of the CURRENT device: the caller's stream must belong to it
  if (!dv) return derr;
  FS2_TRY(setup_once(dv->conv_tc_ready, [] {
    const int mx = 227 * 1024;
    cudaError_t e = conv_tc_prepare_mt1(mx);
    if (e == cudaSuccess) e = conv_tc_prepare_mt2(mx);
    if (e == cudaSuccess) e = conv_tc_prepare_mt4(mx);
    return e;
  }));
  const int g_num_sms = dv->num_sms.load(std::memory_order_relaxed);
  TcP p{};
  p.x = a->x; p.xbs = a->x_batch_stride; p.xrs = a->x_row_stride;
  p.B = a->B; p.T = a->T; p.Cin = plan_args->Cin;
  p.wt = wt; p.wt_bstride = wt_batch_stride; p.bias = a->bias; p.N = a->N;
  p.taps = plan_args->taps; p.dil = a->dilation; p.pad = a->pad_left;
  p.nseg = nseg; p.seg_nkc = seg_nkc; p.seg_wbytes = TC_HDR + (long long)1024 * a->N;
  p.in_act = a->in_act; p.in_slope = a->in_slope; p.out_act = a->out_act; p.out_slope = a->out_slope;
  p.res = a->res; p.rbs = a->res_batch_stride; p.rrs = a->res_row_stride;
  p.alpha = a->alpha; p.accumulate = a->accumulate; p.row_lens = a->row_lens;
  p.y = a->y; p.ybs = a->y_batch_stride; p.yrs = a->y_row_stride;
  p.trace = g_tc_trace;
  p.variant = variant;
  p.f8 = (variant & FS2_TC_VARIANT_F8) ? 1 : 0;
  size_t smem = 0;
  int grid = 0;
  const int rc = conv_tc_plan(plan_args, g_num_sms, p, smem, grid);
  if (rc != FS2_OK) return rc;
  const int mt = p.MT;
  prof_before(s);
  if (mt == 4) conv_tc_launch_mt4(p, (unsigned)grid, smem, s);
  else if (mt == 2) conv_tc_launch_mt2(p, (unsigned)grid, smem, s);
  else conv_tc_launch_mt1(p, (unsigned)grid, smem, s);
  prof_after(s, 0, 2.0 * a->B * a->T * (double)a->Cin * a->taps * a->N);
  FS2_LAUNCH_CHECK();
  return FS2_OK;
}

}  // namespace fs2
