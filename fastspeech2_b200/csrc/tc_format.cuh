// Operand formats of the tcgen05 kernels: the activation splits the kernels write into shared memory and the packed tile
// buffers they stream with bulk copies.  Each format is defined here once; the host packers (packing.pack_conv_tc,
// pack_kv_tiles in attention_tc.cu) must produce the same layouts and scales.
#pragma once
#include "tc_ptx.cuh"

namespace fs2 {

constexpr int TC_HDR = 128;        // bytes of header in front of a packed tile buffer: float[0] = 1 / operand scale

// Operand scales of the f16 + f8 split (TcP::f8): activation lo * 2^12 and hi (unscaled) are rounded to E4M3; the packer stores
// weight hi * 2^-12 and lo (unscaled) in E4M3 (packing.pack_conv_tc), so both correction products carry the main term's scale.
// |x| <= 448 stays inside E4M3; beyond that the correction of that element saturates (the result degrades towards single-pass
// fp16 accuracy for it, never to garbage).
constexpr float TC_F8_LO_SCALE = 4096.f;
constexpr float TC_F8_HI_SCALE = 1.f;

struct NoAct { __device__ __forceinline__ float operator()(float v) const { return v; } };

// 8 values a = act(x) -> fp16 hi = fp16(a) (|a| > 65504 saturates) and lo = fp16(a - hi) (a - hi is exact in fp32); value i is half i.
// `act` lets a caller fold an input activation into the split, one pair of values at a time.
template <class Act = NoAct>
__device__ __forceinline__ void split_f16(const float* x, uint32_t (&hw)[4], uint32_t (&lw)[4], Act act = {}) {
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const float a0 = act(x[2 * j]), a1 = act(x[2 * j + 1]);
    hw[j] = cvt_f16x2_sat(a0, a1);
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hw[j]));
    lw[j] = cvt_f16x2_sat(a0 - hf.x, a1 - hf.y);
  }
}

// 8 values a = act(x) -> fp16 hi as in split_f16, and the two halves of the E4M3 correction operand [lo * 2^12 | hi]: byte i of
// lo8 / hi8 is value i.
template <class Act = NoAct>
__device__ __forceinline__ void split_f16_e4m3(const float* x, uint32_t (&hw)[4], uint32_t (&l8)[2], uint32_t (&h8)[2], Act act = {}) {
  static_assert(TC_F8_HI_SCALE == 1.f, "the E4M3 hi part is converted unscaled");
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const float a0 = act(x[2 * j]), a1 = act(x[2 * j + 1]);
    hw[j] = cvt_f16x2_sat(a0, a1);
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hw[j]));
    const uint32_t l = cvt_e4m3x2_sat((a0 - hf.x) * TC_F8_LO_SCALE, (a1 - hf.y) * TC_F8_LO_SCALE);
    const uint32_t h = cvt_e4m3x2_sat(hf.x, hf.y);
    if (j & 1) { l8[j >> 1] |= l << 16; h8[j >> 1] |= h << 16; }
    else { l8[j >> 1] = l; h8[j >> 1] = h; }
  }
}

// Packed K / V operand tiles of the decoder attention, one buffer per (utterance, head): a TC_HDR header (float[0] = 1 / KV_WSCALE),
// then fp16 hi / lo tiles of K (weights [d][key]) and V (weights [key][d]) -- 128 d x 2 planes x 2 bytes per key, keys padded to Tk, a
// multiple of 128.  Written by pack_kv_tiles (attention_tc.cu); read by attention_gemm through conv_tc and by attention_fused_kernel.
constexpr float KV_WSCALE = 16.f;  // power-of-two operand scale (|k|, |v| < 4094 stay inside fp16)
inline long long kv_tile_stride(int Tk) { return TC_HDR + (long long)Tk * 512; }

}  // namespace fs2
