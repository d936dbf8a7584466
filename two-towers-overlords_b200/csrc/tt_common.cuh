// Shared helpers for libtt_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/tt_b200.h"

namespace tt {

// thread-local error text returned by tt_last_error()
void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what, const char* file, int line);

#define TT_CUDA(call)                                                      \
  do {                                                                     \
    int _rc = ::tt::check_cuda((call), #call, __FILE__, __LINE__);         \
    if (_rc) return _rc;                                                   \
  } while (0)

#define TT_REQUIRE(cond, ...)                                              \
  do {                                                                     \
    if (!(cond)) {                                                         \
      ::tt::set_error(__VA_ARGS__);                                        \
      return 2;                                                            \
    }                                                                      \
  } while (0)

// every kernel launch of the library passes through here; the count backs bench.py's "gpu_launches"
void note_launch();
#define TT_LAUNCH_CHECK()          \
  do {                             \
    ::tt::note_launch();           \
    TT_CUDA(cudaGetLastError());   \
  } while (0)

static inline cudaStream_t as_stream(tt_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

template <typename T>
static inline T* ws_take(char*& p, size_t n_elems) {
  uintptr_t a = (reinterpret_cast<uintptr_t>(p) + 255) & ~uintptr_t(255);
  T* out = reinterpret_cast<T*>(a);
  p = reinterpret_cast<char*>(a + n_elems * sizeof(T));
  return out;
}
static inline size_t ws_round(size_t bytes) { return (bytes + 255) & ~size_t(255); }

int sm_count();

// ---- device helpers -------------------------------------------------------------------------
// Programmatic dependent launch, used between the pooled gather and the persistent chain kernel of a whole-step call:
// pdl_launch() lets the next kernel of the stream start filling SMs, which then blocks in pdl_wait() until this grid
// has completed and its writes are visible.  pdl_wait() returns at once in a kernel launched without the attribute,
// and pdl_launch() does nothing when the next kernel is launched without it.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ long long load_index(const void* p, int dtype, size_t i) {
  switch (dtype) {
    case TT_I64: return reinterpret_cast<const long long*>(p)[i];
    case TT_I32: return reinterpret_cast<const int*>(p)[i];
    case TT_U16: return reinterpret_cast<const unsigned short*>(p)[i];
    default: return reinterpret_cast<const unsigned char*>(p)[i];
  }
}

// torch.optim.Adam (single/multi-tensor, non-fused, no weight decay / amsgrad) on one element: lerp, mul + addcmul,
// sqrt / bc2_sqrt + eps, addcdiv.  Every rounding is spelled out with _rn intrinsics, so no kernel's surroundings can
// change which products the compiler contracts into FMAs: the kernels that call this helper agree bit for bit.  The
// FMAs are the ones the compiler chose for the plain expressions m + (g - m)(1 - beta1), v beta2 + (1 - beta2) g g and
// p - step_size (m / denom) in adam_dev_kernel before this helper existed, which the persistent chain kernel's Adam tail
// and tt_dp_reduce_adam match.
__device__ __forceinline__ void adam_element(float& p, float& m, float& v, float g, float beta1, float beta2, float eps,
                                             float step_size, float bc2_sqrt) {
  m = __fmaf_rn(__fsub_rn(g, m), __fsub_rn(1.f, beta1), m);
  v = __fmaf_rn(v, beta2, __fmul_rn(__fmul_rn(__fsub_rn(1.f, beta2), g), g));
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), eps);
  p = __fmaf_rn(-step_size, __fdiv_rn(m, denom), p);
}
// bias corrections of a device step count state {t, beta1^t, beta2^t, -} that was already advanced to this step
__device__ __forceinline__ float adam_step_size(const double* state, float lr) {
  return (float)((double)lr / (1.0 - state[1]));
}
__device__ __forceinline__ float adam_bc2_sqrt(const double* state) { return (float)sqrt(1.0 - state[2]); }

// fp32 -> (hi, lo) bf16 pair with hi + lo == x to ~2^-17 relative
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

}  // namespace tt
