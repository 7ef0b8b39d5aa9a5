// Shared helpers for libcgan3d (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "cgan3d.h"

namespace cg {

using bf16 = __nv_bfloat16;

// thread-local last error text (cgan3d_last_error)
char *err_buf();
int fail(int code, const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *where);

#define CG_CHECK_ARG(cond, ...)                       \
  do {                                                \
    if (!(cond)) return cg::fail(CGAN3D_E_ARG, __VA_ARGS__); \
  } while (0)
#define CG_CHECK_SHAPE(cond, ...)                       \
  do {                                                  \
    if (!(cond)) return cg::fail(CGAN3D_E_SHAPE, __VA_ARGS__); \
  } while (0)
#define CG_CHECK_DTYPE(dtype, name)                                           \
  do {                                                                        \
    if ((dtype) != CGAN3D_F32 && (dtype) != CGAN3D_BF16)                      \
      return cg::fail(CGAN3D_E_DTYPE, "%s: unknown dtype %d", name, (dtype)); \
  } while (0)
#define CG_LAUNCH_CHECK(where)                          \
  do {                                                  \
    cudaError_t e__ = cudaGetLastError();               \
    if (e__ != cudaSuccess) return cg::cuda_fail(e__, where); \
  } while (0)

static inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

// with_dtype(dtype, f) calls f with the tensor element type of a checked dtype (CGAN3D_F32 -> float, else bf16) as a tag,
// so a launch is written once: [&](auto t) { using T = typename decltype(t)::type; kernel<T><<<...>>>((const T *)p, ...); }
template <typename T>
struct type_tag {
  using type = T;
};
template <typename F>
static inline auto with_dtype(int dtype, F &&f) {
  if (dtype == CGAN3D_F32) return f(type_tag<float>{});
  return f(type_tag<bf16>{});
}

__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T>
__device__ __forceinline__ T from_f(float v);
template <>
__device__ __forceinline__ float from_f<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float act_fwd(float v, int act, float slope) {
  switch (act) {
    case CGAN3D_ACT_RELU: return v > 0.f ? v : 0.f;
    case CGAN3D_ACT_LRELU: return v > 0.f ? v : v * slope;
    case CGAN3D_ACT_TANH: return tanhf(v);
    default: return v;
  }
}
// derivative w.r.t. the pre-activation value v
__device__ __forceinline__ float act_bwd(float v, int act, float slope) {
  switch (act) {
    case CGAN3D_ACT_RELU: return v > 0.f ? 1.f : 0.f;
    case CGAN3D_ACT_LRELU: return v > 0.f ? 1.f : slope;
    case CGAN3D_ACT_TANH: { float t = tanhf(v); return 1.f - t * t; }
    default: return 1.f;
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum 64 per-thread values over the 32 lanes of a warp with a recursive-halving exchange (62 shuffles instead of 64 x 5):
// afterwards v[0], v[1] of lane l hold the warp totals of channels warp_reduce64_channel(l) and +1.
__device__ __forceinline__ void warp_reduce64(float (&v)[64], int lane) {
#pragma unroll
  for (int half = 32, off = 16; half >= 2; half >>= 1, off >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float keep = hi ? v[half + i] : v[i];
      const float send = hi ? v[i] : v[half + i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
}
__device__ __forceinline__ int warp_reduce64_channel(int lane) {
  return ((lane >> 4) & 1) * 32 + ((lane >> 3) & 1) * 16 + ((lane >> 2) & 1) * 8 + ((lane >> 1) & 1) * 4 + (lane & 1) * 2;
}

// Philox4x32-10 (Salmon et al., SC'11): the four 32-bit words of counter (c0, c1, c2, c3) under the 64-bit key `seed`.
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

int num_sms();

template <typename T>
__host__ __device__ __forceinline__ T mn(T a, T b) { return a < b ? a : b; }
template <typename T>
__host__ __device__ __forceinline__ T mx(T a, T b) { return a > b ? a : b; }
static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// blocks of 256 threads for the grid-strided element-wise kernels over n items: one item per thread, at most 16 blocks per SM
static inline int ew_blocks(int64_t n) { return (int)mx<int64_t>(1, mn<int64_t>((n + 255) / 256, (int64_t)num_sms() * 16)); }

}  // namespace cg
