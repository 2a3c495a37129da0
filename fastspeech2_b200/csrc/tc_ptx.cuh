// Device primitives shared by the tcgen05 kernels (conv_tc_kernel.cuh, resstack_fused.cu, attention_fused.cu): mbarriers, bulk
// and tensor-map copies, tensor-memory allocation / loads / stores, UMMA descriptors and MMAs, fences, operand conversions.
// Every inline PTX statement of those kernels lives here.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace fs2 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// makes the mbar_init()s of this thread visible to the async proxy (bulk copies, tcgen05.commit) before the block syncs
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// mbarrier ring cursor without runtime div/mod (an integer division per tap was on the MMA issuer's critical path)
struct Ring {
  uint32_t idx = 0, phase = 0;
  __device__ __forceinline__ void advance(uint32_t n) {
    if (++idx == n) { idx = 0; phase ^= 1u; }
  }
};

__device__ __forceinline__ void tma_prefetch_map(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, int c0, int n0, int b, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                   smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(n0), "r"(b), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, int c0, int n0, int b, const void* src) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(reinterpret_cast<uint64_t>(tm)),
               "r"(c0), "r"(n0), "r"(b), "r"(smem_u32(src))
               : "memory");
}
__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* tm, int c0, int n0, int b, const void* src) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(c0), "r"(n0), "r"(b), "r"(smem_u32(src))
               : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_reads() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// byte offset of 16-byte chunk c of row r inside a [rows][128 B] box written / read by TMA with CU_TENSOR_MAP_SWIZZLE_128B
__device__ __forceinline__ uint32_t sw128(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

// Programmatic dependent launch: the grid may start while its predecessor in the stream is still draining; everything that
// reads or writes memory the predecessor touches comes after grid_dep_wait() (returns once the predecessor has completed and
// flushed).  grid_dep_launch() lets the successor's CTAs be scheduled onto SMs as this grid's CTAs exit.
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// named barrier 1 over the first NTHREADS threads that reach it: the kernels' "row" warps, without the producer / MMA warps
template <int NTHREADS>
__device__ __forceinline__ void row_warps_sync() { asm volatile("bar.sync 1, %0;" ::"n"(NTHREADS) : "memory"); }
// 1 in one lane of the (fully active) warp, 0 in the others
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t leader;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));
  return leader;
}

// whole warp: allocates `cols` TMEM columns (a power of two >= 32), writes their base address to *slot, gives up the right to allocate more
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(cols));
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 16 (x16) or 32 (x32) consecutive columns of this thread's TMEM lane; the _nowait load's registers are valid after tc_wait_ld()
template <int N>
__device__ __forceinline__ void tc_ld16_nowait(uint32_t taddr, uint32_t (&v)[N]) {
  static_assert(N >= 16, "tc_ld16 writes 16 registers");
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[N]) {
  tc_ld16_nowait(taddr, v);
  tc_wait_ld();
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  tc_wait_ld();
}
__device__ __forceinline__ void tc_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, no-swizzle K-major: core matrix = 8 rows x 16 B stored contiguously (128 B);
// LBO = byte distance between the two 16-byte K-chunks of one K=16 (FP16) MMA, SBO = byte distance between 8-row groups.
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version (Blackwell)
  return d;                 // layout_type = SWIZZLE_NONE (0), base_offset = 0
}

// kind::f16 with FP16 operands (a_format = b_format = 0), fp32 accumulate, A and B K-major, M = 128
__device__ __forceinline__ uint32_t umma_idesc_f16(int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::f8f6f4 with E4M3 operands (K = 32 per instruction: here 16 channels x {activation-lo * weight-hi, activation-hi * weight-lo})
__device__ __forceinline__ void tc_mma_f8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// 8 consecutive floats (one 32-byte sector) in one request: SASS LDG.E.256
__device__ __forceinline__ void ldg256(float (&d)[8], const float* src) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]), "=f"(d[4]), "=f"(d[5]), "=f"(d[6]), "=f"(d[7])
               : "l"(src));
}
// fp16x2 {lo = a0, hi = a1}, round-to-nearest, |x| > 65504 saturates instead of becoming inf: SASS F2FP.SATFINITE.F16.F32.PACK_AB
__device__ __forceinline__ uint32_t cvt_f16x2_sat(float a0, float a1) {
  uint32_t h;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(a1), "f"(a0));
  return h;
}
// e4m3x2 {byte 0 = a0, byte 1 = a1}, round-to-nearest, saturating at +-448
__device__ __forceinline__ uint32_t cvt_e4m3x2_sat(float a0, float a1) {
  unsigned short h;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(h) : "f"(a1), "f"(a0));
  return (uint32_t)h;
}

__device__ __forceinline__ long long gtime() {
  long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

}  // namespace fs2
