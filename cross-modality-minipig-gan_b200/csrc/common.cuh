// Shared helpers for libmpgan_sm100 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <utility>

#include "../../include/mpgan.h"

namespace mpgan {

void set_error(const char* fmt, ...);

#define MPGAN_CHECK_LAUNCH(what)                                                 \
  do {                                                                           \
    cudaError_t e__ = cudaGetLastError();                                        \
    if (e__ != cudaSuccess) {                                                    \
      mpgan::set_error("%s: %s", what, cudaGetErrorString(e__));                 \
      return MPGAN_ERR_CUDA;                                                     \
    }                                                                            \
  } while (0)

#define MPGAN_REQUIRE(cond, code, ...)                                           \
  do {                                                                           \
    if (!(cond)) {                                                               \
      mpgan::set_error(__VA_ARGS__);                                             \
      return code;                                                               \
    }                                                                            \
  } while (0)

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// order-preserving map fp32 -> uint32 (total order; -0.0 < +0.0, NaNs sort last as in np.sort, -NaNs first).
// Integer-only on purpose: written as (b & sign) ? ~b : (b | sign), the compiler emits b | sign as the float -|f|,
// which turns a NaN into the canonical NaN and so loses its place in the order.
__device__ __forceinline__ uint32_t key_of(float f) {
  const uint32_t b = __float_as_uint(f);
  return b ^ ((uint32_t)((int32_t)b >> 31) | 0x80000000u);
}
__device__ __forceinline__ float value_of(uint32_t k) {
  const uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(b);
}

// block-wide sum of one float per thread; result valid in thread 0.  blockDim.x <= 1024, multiple of 32.
__device__ __forceinline__ float block_sum(float v, float* smem32) {
  v = warp_sum(v);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) smem32[w] = v;
  __syncthreads();
  float r = 0.f;
  if (w == 0) {
    r = (lane < (blockDim.x >> 5)) ? smem32[lane] : 0.f;
    r = warp_sum(r);
  }
  __syncthreads();
  return r;
}

// ---- programmatic dependent launch (PDL) ----
// Every kernel of the library starts with pdl_wait(); pdl_launch();  and is launched with the programmatic stream
// serialization attribute: the next kernel of the stream (or of the captured CUDA graph) is launched and scheduled
// while this one is still running and starts the moment this one has completed and flushed -- the launch latency
// between the ~1000 small dependent kernels of a training step disappears.  Correctness only needs the wait to
// precede the first global-memory access (it is the first instruction).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

inline bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("MPGAN_NO_PDL"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}

template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);   // errors surface through MPGAN_CHECK_LAUNCH
}

inline int num_sms() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  }
  return sms;
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// dispatch on activation dtype
#define MPGAN_DISPATCH_DTYPE(dtype, T, ...)                                      \
  do {                                                                           \
    if ((dtype) == MPGAN_F32) {                                                  \
      typedef float T;                                                           \
      __VA_ARGS__;                                                               \
    } else if ((dtype) == MPGAN_BF16) {                                          \
      typedef mpgan::bf16 T;                                                     \
      __VA_ARGS__;                                                               \
    } else {                                                                     \
      mpgan::set_error("bad dtype %d", (int)(dtype));                            \
      return MPGAN_ERR_UNSUPPORTED;                                              \
    }                                                                            \
  } while (0)

}  // namespace mpgan
