// Shared helpers for the fs2b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "fs2b200.h"

namespace fs2 {

extern std::atomic<unsigned long long> g_launch_count;  // host-side counter, bumped once per kernel launch (any thread)

inline int cuda_status() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? FS2_OK : (FS2_ERR_CUDA - (int)e);
}

#define FS2_LAUNCH_CHECK()                 \
  do {                                     \
    ::fs2::g_launch_count++;               \
    int _st = ::fs2::cuda_status();        \
    if (_st != FS2_OK) return _st;         \
  } while (0)

#define FS2_TRY(expr)                      \
  do {                                     \
    int _st = (expr);                      \
    if (_st != FS2_OK) return _st;         \
  } while (0)

// Per-device one-time setup (SM count, >48 KB dynamic shared memory opt-ins).  cudaFuncSetAttribute applies to the CURRENT device's
// context, so the "done" flags are kept per device ordinal; dev_state() looks the current device up (thread-safe) and
// setup_once() runs a kernel family's setup the first time the family is used on that device.
constexpr int FS2_MAX_DEVICES = 64;
struct DevState {
  std::atomic<int> num_sms{0};
  std::atomic<bool> conv_tc_ready{false}, att_simt_ready{false}, fused_ready{false}, att_fused_ready{false};
};
DevState* dev_state(int* err);                       // NULL + *err on failure
// Runs fn unless `done` (a DevState flag) is set, and sets it once fn has succeeded; first calls from several threads are
// serialised.  Returns FS2_OK or the CUDA error of fn.
int setup_once(std::atomic<bool>& done, cudaError_t (*fn)());

// optional per-launch event timing (see fs2_profile_begin in fs2b200.h); armed per host thread
extern thread_local bool g_prof_on;
void prof_before(cudaStream_t s);
void prof_after(cudaStream_t s, int cls, double flops);

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

__device__ __forceinline__ float apply_act(float v, int act, float slope) {
  switch (act) {
    case FS2_ACT_RELU: return fmaxf(v, 0.f);
    case FS2_ACT_TANH: return tanhf(v);
    case FS2_ACT_LRELU: return v > 0.f ? v : v * slope;
    default: return v;
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace fs2
