// Shared helpers for libctcvr.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>

#include "../../include/ctcvr.h"

namespace ctcvr {

void set_error(const char* fmt, ...);
void count_launch();   // bumps the counter behind ctcvr_launch_count()

#define CTCVR_CHECK_CUDA(expr)                                                            \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::ctcvr::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,             \
                         cudaGetErrorString(_e));                                         \
      return 1;                                                                           \
    }                                                                                     \
  } while (0)

#define CTCVR_REQUIRE(cond, ...)                                                          \
  do {                                                                                    \
    if (!(cond)) {                                                                        \
      ::ctcvr::set_error(__VA_ARGS__);                                                    \
      return 2;                                                                           \
    }                                                                                     \
  } while (0)

#define CTCVR_LAUNCH_CHECK()                                                              \
  do {                                                                                    \
    ::ctcvr::count_launch();                                                              \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess) {                                                              \
      ::ctcvr::set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__,         \
                         cudaGetErrorString(_e));                                         \
      return 1;                                                                           \
    }                                                                                     \
  } while (0)

constexpr float kNegInf = -INFINITY;

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// log(exp(a)+exp(b)), -inf safe.
__device__ __forceinline__ float log_add_exp(float a, float b) {
  float m = fmaxf(a, b);
  if (m == kNegInf) return kNegInf;
  return m + log1pf(expf(-fabsf(a - b)));
}
__device__ __forceinline__ double log_add_exp(double a, double b) {
  double m = fmax(a, b);
  if (m == -INFINITY) return -INFINITY;
  return m + log1p(exp(-fabs(a - b)));
}

// Joint activation z = act(h), h = enc_proj + pred_proj (CTCVR_ACT_* >> 8).  tanh is nn.Tanh, relu nn.ReLU (derivative
// h > 0, torch's 0 at h = 0), gelu the exact erf form of nn.GELU(): h Phi(h), derivative Phi(h) + h phi(h).
enum { ACT_TANH = 0, ACT_RELU = 1, ACT_GELU = 2 };

__device__ __forceinline__ float gelu_f32(float h) { return 0.5f * h * (1.f + erff(h * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad_f32(float h) {
  const float cdf = 0.5f * (1.f + erff(h * 0.70710678118654752f));
  return fmaf(h * 0.39894228040143268f, expf(-0.5f * h * h), cdf);
}
template <int ACT>
__device__ __forceinline__ float act_f32(float h) {
  if constexpr (ACT == ACT_RELU) return fmaxf(h, 0.f);
  else if constexpr (ACT == ACT_GELU) return gelu_f32(h);
  else return tanhf(h);
}
// act'(h) for relu / gelu (the tanh paths use 1 - z^2 from z)
template <int ACT>
__device__ __forceinline__ float act_grad_f32(float h) {
  if constexpr (ACT == ACT_RELU) return h > 0.f ? 1.f : 0.f;
  else return gelu_grad_f32(h);
}
// run-time form for the decoders (the branch is uniform across the launch)
__device__ __forceinline__ float act_rt(int act, float h) {
  if (act == ACT_RELU) return fmaxf(h, 0.f);
  if (act == ACT_GELU) return gelu_f32(h);
  return tanhf(h);
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }

}  // namespace ctcvr
