// BatchNorm (train/eval) + activation + residual, bias+activation, generator tail, dtype helpers.
// HBM-bound row-major [n_rows][C] kernels (channels-last activations).
// Replaces aten::native_batch_norm(+backward), relu_/leaky_relu_/tanh, add
// (reference model/blocks.py:45,50,52-53,87-88; generator.py:85; trainer/Trainer.py:171).
#include <type_traits>

#include "common.cuh"

namespace cg {

// ---------------------------------------------------------------- dropout keep law (reference model/blocks.py:68-88)
// Element e (the channels-last linear index) is kept iff u(e) >= thresh, where u(e) is word e & 3 of Philox4x32-10 at
// counter (lo32(e >> 2), hi32(e >> 2), 0, 0) under the 64-bit seed, and thresh = floor(p * 2^32) (2^32 at p = 1: nothing
// is kept).  One Philox evaluation serves four elements.  Returns the keep bits of e0 .. e0 + 7 (e0 % 8 == 0), bit k for
// e0 + k: byte e0 / 8 of the bitmask that the backward passes read.
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t e0, uint64_t seed, uint64_t thresh) {
  uint32_t bits = 0;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const uint64_t q = (e0 >> 2) + h;
    const uint4 w = philox4x32_10((uint32_t)q, (uint32_t)(q >> 32), 0, 0, seed);
    bits |= ((uint32_t)(w.x >= thresh) | (uint32_t)(w.y >= thresh) << 1 | (uint32_t)(w.z >= thresh) << 2 |
             (uint32_t)(w.w >= thresh) << 3) << (4 * h);
  }
  return bits;
}

// ---------------------------------------------------------------- column reductions
// Block of 256 threads covers `lanes = 256 / Cw` rows at a time; thread (lane, c) walks rows
// lane, lane+lanes, ... of its block's strip.  Per-thread fp32 partials over a short run are
// promoted to fp64 before the cross-thread / cross-block combine, so the result is independent
// of the block schedule to fp32 accuracy.
template <int NS, typename F>
__device__ __forceinline__ void col_reduce_body(int64_t n_rows, int C, int rows_per_block, double *sums, F f) {
  extern __shared__ double sh[];  // [NS][lanes][Cw]
  const int Cw = C <= 256 ? C : 256;
  const int lanes = blockDim.x / Cw;
  const int lane = threadIdx.x / Cw;
  const int c0 = threadIdx.x % Cw;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = min(n_rows, r0 + rows_per_block);
  for (int c = c0; c < C; c += Cw) {
    double tot[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) tot[s] = 0.0;
    if (lane < lanes) {
      float part[NS];
#pragma unroll
      for (int s = 0; s < NS; ++s) part[s] = 0.f;
      int run = 0;
      for (int64_t r = r0 + lane; r < r1; r += lanes) {
        float v[NS];
        f(r, c, v);
#pragma unroll
        for (int s = 0; s < NS; ++s) part[s] += v[s];
        if (++run == 64) {
#pragma unroll
          for (int s = 0; s < NS; ++s) { tot[s] += (double)part[s]; part[s] = 0.f; }
          run = 0;
        }
      }
#pragma unroll
      for (int s = 0; s < NS; ++s) tot[s] += (double)part[s];
    }
    __syncthreads();
    if (lane < lanes) {
#pragma unroll
      for (int s = 0; s < NS; ++s) sh[(s * lanes + lane) * Cw + c0] = tot[s];
    }
    __syncthreads();
    if (lane == 0) {
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        double a = 0.0;
        for (int l = 0; l < lanes; ++l) a += sh[(s * lanes + l) * Cw + c0];
        atomicAdd(&sums[s * C + c], a);
      }
    }
  }
}

struct ColGrid {
  int blocks, rows_per_block;
  size_t smem;
};
static ColGrid col_grid(int64_t n_rows, int C, int ns) {
  const int Cw = C <= 256 ? C : 256;
  const int lanes = 256 / Cw;
  int64_t target_blocks = (int64_t)num_sms() * 8;
  int64_t rpb = (n_rows + target_blocks - 1) / target_blocks;
  rpb = mx<int64_t>(rpb, (int64_t)lanes * 8);
  rpb = ((rpb + lanes - 1) / lanes) * lanes;
  ColGrid g;
  g.rows_per_block = (int)mn<int64_t>(rpb, 1 << 30);
  g.blocks = (int)((n_rows + g.rows_per_block - 1) / g.rows_per_block);
  g.smem = (size_t)ns * lanes * Cw * sizeof(double);
  return g;
}

template <typename T>
__global__ void __launch_bounds__(256) bn_stats_kernel(const T *__restrict__ y, int64_t n_rows, int C, int rpb,
                                                       double *sums) {
  col_reduce_body<2>(n_rows, C, rpb, sums, [&](int64_t r, int c, float v[2]) {
    const float x = to_f(y[r * C + c]);
    v[0] = x;
    v[1] = x * x;
  });
}

template <typename T>
__global__ void __launch_bounds__(256) col_sums_kernel(const T *__restrict__ x, int64_t n_rows, int C, int rpb,
                                                       double *sums) {
  col_reduce_body<1>(n_rows, C, rpb, sums, [&](int64_t r, int c, float v[1]) { v[0] = to_f(x[r * C + c]); });
}

// DROP: dz is multiplied by keep * scale first (dropout between this normalisation and its consumer, scale = 1 / (1 - p))
template <typename T, bool DROP = false>
__global__ void __launch_bounds__(256)
bn_bwd_reduce_kernel(const T *__restrict__ dz, const T *__restrict__ y, int64_t n_rows, int C, int rpb,
                     const float *__restrict__ mi, const float *__restrict__ gamma, const float *__restrict__ beta,
                     int act, float slope, double *sums, const uint8_t *__restrict__ keep_bits = nullptr, float scale = 1.f) {
  col_reduce_body<2>(n_rows, C, rpb, sums, [&](int64_t r, int c, float v[2]) {
    const float xh = (to_f(y[r * C + c]) - mi[c]) * mi[C + c];
    const float pre = gamma[c] * xh + beta[c];
    float d = to_f(dz[r * C + c]);
    if constexpr (DROP) {
      const int64_t e = r * C + c;
      d = (keep_bits[e >> 3] >> (e & 7) & 1) ? d * scale : 0.f;
    }
    const float g = d * act_bwd(pre, act, slope);
    v[0] = g;
    v[1] = g * xh;
  });
}

template <typename T>
__global__ void __launch_bounds__(256)
bias_act_bwd_kernel(const T *__restrict__ dz, const T *__restrict__ y, T *__restrict__ dy, int64_t n_rows, int C,
                    int rpb, const float *__restrict__ bias, int act, float slope, double *sums) {
  col_reduce_body<1>(n_rows, C, rpb, sums, [&](int64_t r, int c, float v[1]) {
    const float pre = to_f(y[r * C + c]) + (bias ? bias[c] : 0.f);
    const float g = to_f(dz[r * C + c]) * act_bwd(pre, act, slope);
    dy[r * C + c] = from_f<T>(g);
    v[0] = g;
  });
}


// ---------------------------------------------------------------- 8-wide vector access (C % 8 == 0 fast paths)
template <typename T>
struct V8;
template <>
struct V8<float> {
  float v[8];
  __device__ __forceinline__ void load(const float *p) {
    const float4 a = *reinterpret_cast<const float4 *>(p), b = *reinterpret_cast<const float4 *>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  __device__ __forceinline__ void store(float *p) const {
    reinterpret_cast<float4 *>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4 *>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
};
template <>
struct V8<__nv_bfloat16> {
  float v[8];
  __device__ __forceinline__ void load(const __nv_bfloat16 *p) {
    const uint4 a = *reinterpret_cast<const uint4 *>(p);
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ __forceinline__ void store(__nv_bfloat16 *p) const {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t *>(&h);
    }
    *reinterpret_cast<uint4 *>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};

// vectorised column reduction: thread (lane, c8) owns 8 adjacent channels and walks the rows grid-strided (row =
// first + i * lanes_in_grid), so every iteration of the whole grid reads one contiguous span.  load(row, raw[]) fetches
// the row's 16-byte chunks WITHOUT consuming them, so U of them are in flight per thread before eval(raw, v) runs;
// fp32 runs of 32 rows feed fp64 totals.
struct NoPost {
  __device__ __forceinline__ void operator()(double (&)[1][8]) const {}
  __device__ __forceinline__ void operator()(double (&)[2][8]) const {}
};
template <int NS, int U, int NRAW, typename FL, typename FE, typename FP = NoPost>
__device__ __forceinline__ void col_reduce8_body(int64_t n_rows, int C, double *sums, FL load, FE eval, FP post = FP()) {
  extern __shared__ double sh[];  // [lanes][NS][C]
  const int C8 = C >> 3;
  const int lanes = blockDim.x / C8;
  const int lane = threadIdx.x / C8;
  const int c0 = (threadIdx.x % C8) * 8;
  const int64_t gl = (int64_t)gridDim.x * lanes;  // lanes in the grid
  double tot[NS][8];
#pragma unroll
  for (int s = 0; s < NS; ++s)
#pragma unroll
    for (int k = 0; k < 8; ++k) tot[s][k] = 0.0;
  if (lane < lanes) {
    for (int64_t rb = (int64_t)blockIdx.x * lanes + lane; rb < n_rows; rb += 32 * gl) {
      float part[NS][8];
#pragma unroll
      for (int s = 0; s < NS; ++s)
#pragma unroll
        for (int k = 0; k < 8; ++k) part[s][k] = 0.f;
#pragma unroll 1
      for (int i0 = 0; i0 < 32; i0 += U) {
        uint4 raw[U][NRAW];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t r = rb + (int64_t)(i0 + u) * gl;
          if (r < n_rows) load(r, raw[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t r = rb + (int64_t)(i0 + u) * gl;
          if (r < n_rows) {
            float v[NS][8];
            eval(r, raw[u], v);
#pragma unroll
            for (int s = 0; s < NS; ++s)
#pragma unroll
              for (int k = 0; k < 8; ++k) part[s][k] += v[s][k];
          }
        }
      }
#pragma unroll
      for (int s = 0; s < NS; ++s)
#pragma unroll
        for (int k = 0; k < 8; ++k) tot[s][k] += (double)part[s][k];
    }
    post(tot);  // linear map of this thread's totals (commutes with the remaining summation)
#pragma unroll
    for (int s = 0; s < NS; ++s)
#pragma unroll
      for (int k = 0; k < 8; ++k) sh[((size_t)lane * NS + s) * C + c0 + k] = tot[s][k];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NS * C; i += blockDim.x) {
    double a = 0.0;
    for (int l = 0; l < lanes; ++l) a += sh[(size_t)l * NS * C + i];
    atomicAdd(&sums[i], a);
  }
}

// raw 16-byte chunk -> 8 floats
template <typename T>
__device__ __forceinline__ void unpack8(const uint4 *raw, float (&v)[8]);
template <>
__device__ __forceinline__ void unpack8<__nv_bfloat16>(const uint4 *raw, float (&v)[8]) {
  const uint32_t w[4] = {raw[0].x, raw[0].y, raw[0].z, raw[0].w};
#pragma unroll
  for (int i = 0; i < 4; ++i) { v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
}
template <>
__device__ __forceinline__ void unpack8<float>(const uint4 *raw, float (&v)[8]) {
  v[0] = __uint_as_float(raw[0].x); v[1] = __uint_as_float(raw[0].y); v[2] = __uint_as_float(raw[0].z); v[3] = __uint_as_float(raw[0].w);
  v[4] = __uint_as_float(raw[1].x); v[5] = __uint_as_float(raw[1].y); v[6] = __uint_as_float(raw[1].z); v[7] = __uint_as_float(raw[1].w);
}
template <typename T>
__device__ __forceinline__ void load8raw(const T *p, uint4 *raw) {
  constexpr int NV = (int)sizeof(T) / 2;  // 16-byte vectors per 8 elements
#pragma unroll
  for (int i = 0; i < NV; ++i) raw[i] = reinterpret_cast<const uint4 *>(p)[i];
}

static bool vec8_ok(int C, const void *a, const void *b = nullptr, const void *c = nullptr, const void *d = nullptr) {
  auto al = [](const void *p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return C % 8 == 0 && C <= 2048 && 256 % (C >> 3) == 0 && al(a) && al(b) && al(c) && al(d);
}
static ColGrid col_grid8(int64_t n_rows, int C, int ns) {
  const int lanes = 256 / (C >> 3);
  ColGrid g;
  g.rows_per_block = 0;  // rows are walked grid-strided
  // two blocks per SM = one resident wave (measured at 16x128^3x16 / 16x64^3x32 / 16x32^3x64 bf16: 2 -> 90 / 81 / 56 % of the HBM
  // peak, 4 -> 89 / 75 / 52 %, 8 -> 87 / 71 / 39 %; eight row pairs in flight per thread instead of four: slower)
  g.blocks = (int)mx<int64_t>(1, mn<int64_t>((n_rows + lanes - 1) / lanes, (int64_t)num_sms() * 2));
  g.smem = (size_t)ns * lanes * C * sizeof(double);
  return g;
}

template <typename T>
__global__ void __launch_bounds__(256) bn_stats8_kernel(const T *__restrict__ y, int64_t n_rows, int C, int rpb, double *sums) {
  const int c0 = (threadIdx.x % (C >> 3)) * 8;
  constexpr int NV = (int)sizeof(T) / 2;
  col_reduce8_body<2, 8, NV>(
      n_rows, C, sums, [&](int64_t r, uint4 *raw) { load8raw(y + r * C + c0, raw); },
      [&](int64_t, const uint4 *raw, float (&v)[2][8]) {
        float x[8];
        unpack8<T>(raw, x);
#pragma unroll
        for (int k = 0; k < 8; ++k) { v[0][k] = x[k]; v[1][k] = x[k] * x[k]; }
      });
}

// activation derivative with the activation known at compile time (ACT < 0: runtime switch)
template <int ACT>
__device__ __forceinline__ float act_bwd_t(float pre, int act, float slope) {
  if (ACT == CGAN3D_ACT_NONE) return 1.f;
  if (ACT == CGAN3D_ACT_RELU) return pre > 0.f ? 1.f : 0.f;
  if (ACT == CGAN3D_ACT_LRELU) return pre > 0.f ? 1.f : slope;
  return act_bwd(pre, act, slope);
}

// per-thread channel constants of the 8 channels a thread owns (hoisted out of the streaming loops: the per-element
// loads of mean/invstd/gamma/beta made these kernels LSU-bound instead of HBM-bound)
struct BnC8 {
  float a[8], b[8], mean[8], invstd[8], gamma[8], beta[8], nm[8];
  __device__ __forceinline__ void load(const float *mi, const float *g, const float *bt, int C, int c0) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      mean[k] = mi[c0 + k]; invstd[k] = mi[C + c0 + k]; gamma[k] = g[c0 + k]; beta[k] = bt[c0 + k];
      a[k] = gamma[k] * invstd[k];
      b[k] = beta[k] - mean[k] * a[k];
      nm[k] = -mean[k] * invstd[k];
    }
  }
};

template <typename T, int ACT, bool DROP = false, int U = 4>
__global__ void __launch_bounds__(256, 2)
bn_bwd_reduce8_kernel(const T *__restrict__ dz, const T *__restrict__ y, int64_t n_rows, int C, int rpb,
                      const float *__restrict__ mi, const float *__restrict__ gamma, const float *__restrict__ beta, int act,
                      float slope, double *sums, const uint8_t *__restrict__ keep_bits = nullptr, float scale = 1.f) {
  const int c0 = (threadIdx.x % (C >> 3)) * 8;
  struct { float a[8], b[8], invstd[8], nm[8]; } k8;  // only what the streaming loop needs (register budget: 2 blocks/SM)
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float mean = mi[c0 + k], is = mi[C + c0 + k];
    k8.invstd[k] = is;
    k8.nm[k] = -mean * is;
    k8.a[k] = gamma[c0 + k] * is;
    k8.b[k] = beta[c0 + k] - mean * k8.a[k];
  }
  constexpr int NV = (int)sizeof(T) / 2;
  // DROP: the row's keep byte (its 8 channels) travels as one more raw slot, fetched together with the row's data
  col_reduce8_body<2, U, 2 * NV + DROP>(
      n_rows, C, sums,
      [&](int64_t r, uint4 *raw) {
        load8raw(y + r * C + c0, raw);
        load8raw(dz + r * C + c0, raw + NV);
        if constexpr (DROP) raw[2 * NV].x = keep_bits[(r * C + c0) >> 3];
      },
      [&](int64_t, const uint4 *raw, float (&v)[2][8]) {
        float yy[8], dd[8];
        unpack8<T>(raw, yy);
        unpack8<T>(raw + NV, dd);
        if constexpr (DROP) {
#pragma unroll
          for (int k = 0; k < 8; ++k) dd[k] = (raw[2 * NV].x >> k & 1u) ? dd[k] * scale : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          // streams sum g and sum g*y; sum g*xhat = invstd * sum g*y - mean*invstd * sum g is applied to the totals
          const float g = dd[k] * act_bwd_t<ACT>(fmaf(k8.a[k], yy[k], k8.b[k]), act, slope);
          v[0][k] = g;
          v[1][k] = g * yy[k];
        }
      },
      [&](double (&tot)[2][8]) {
#pragma unroll
        for (int k = 0; k < 8; ++k) tot[1][k] = (double)k8.invstd[k] * tot[1][k] + (double)k8.nm[k] * tot[0][k];
      });
}

// The elementwise kernels walk the tensor with a stride that is a multiple of C, so a thread always sees the same 8 channels.
// DROP: dropout after the activation (no residual): z = keep ? act(.) * scale : 0, and thread i writes keep byte i (the
// keep bits of its 8 elements), so consecutive threads write consecutive bytes.
template <typename T, bool DROP = false>
__global__ void __launch_bounds__(256)
bn_apply8_kernel(const T *__restrict__ y, T *__restrict__ z, int64_t total8, int C, const float *__restrict__ mi,
                 const float *__restrict__ gamma, const float *__restrict__ beta, int act, float slope,
                 const T *__restrict__ residual, uint8_t *__restrict__ keep_bits = nullptr,
                 const int64_t *__restrict__ seed_dev = nullptr, uint64_t thresh = 0, float scale = 1.f) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int c0 = (int)((i * 8) % C);
  BnC8 k8;
  k8.load(mi, gamma, beta, C, c0);
  uint64_t seed = 0;
  if constexpr (DROP) seed = (uint64_t)*seed_dev;
  for (; i < total8; i += 2 * stride) {
    const int64_t e0 = i * 8, e1 = (i + stride) * 8;
    const bool two = i + stride < total8;
    V8<T> v0, v1, r0, r1;
    v0.load(y + e0);
    if (two) v1.load(y + e1);
    if (residual) { r0.load(residual + e0); if (two) r1.load(residual + e1); }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float t0 = act_fwd(fmaf(k8.a[k], v0.v[k], k8.b[k]), act, slope);
      float t1 = act_fwd(fmaf(k8.a[k], v1.v[k], k8.b[k]), act, slope);
      if (residual) { t0 += r0.v[k]; t1 += r1.v[k]; }
      v0.v[k] = t0; v1.v[k] = t1;
    }
    if constexpr (DROP) {
      const uint32_t kb0 = dropout_keep8((uint64_t)e0, seed, thresh), kb1 = two ? dropout_keep8((uint64_t)e1, seed, thresh) : 0u;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        v0.v[k] = (kb0 >> k & 1u) ? v0.v[k] * scale : 0.f;
        v1.v[k] = (kb1 >> k & 1u) ? v1.v[k] * scale : 0.f;
      }
      keep_bits[i] = (uint8_t)kb0;
      if (two) keep_bits[i + stride] = (uint8_t)kb1;
    }
    v0.store(z + e0);
    if (two) v1.store(z + e1);
  }
}

// bn_apply fused with the reflection padding of the CONSUMER (the generator's last_conv pads its input by 3,
// reference model/generator.py:77-83): one block per padded (b, x', y') line reads the mirrored source line of the raw
// conv output and writes normalise + activation straight into the padded tensor, so the un-padded activation never
// exists in HBM (one write and one read of 1 GB less per step at 16 x 128^3 x 16).
template <typename T>
__global__ void __launch_bounds__(256)
bn_apply_pad8_kernel(const T *__restrict__ y, T *__restrict__ zp, int X, int Y, int Z, int C, int p, const float *__restrict__ mi,
                     const float *__restrict__ gamma, const float *__restrict__ beta, int act, float slope) {
  extern __shared__ float s_ab[];  // a[C], b[C]: z = act(a * y + b)
  const int Xp = X + 2 * p, Yp = Y + 2 * p, Zp = Z + 2 * p, cpv = C >> 3;
  for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
    const float av = gamma[ch] * mi[C + ch];
    s_ab[ch] = av;
    s_ab[C + ch] = beta[ch] - mi[ch] * av;
  }
  __syncthreads();
  auto refl = [](int j, int n) { if (j < 0) j = -j; if (j >= n) j = 2 * (n - 1) - j; return j; };
  const int yp = blockIdx.x, xp = blockIdx.y, b = blockIdx.z;
  const int sx = refl(xp - p, X), sy = refl(yp - p, Y);
  const T *src = y + (((int64_t)b * X + sx) * Y + sy) * (int64_t)Z * C;
  T *dst = zp + (((int64_t)b * Xp + xp) * Yp + yp) * (int64_t)Zp * C;
  for (int i = threadIdx.x; i < Zp * cpv; i += blockDim.x) {
    const int z = i / cpv, c = i - z * cpv;
    V8<T> v;
    v.load(src + ((int64_t)refl(z - p, Z) * cpv + c) * 8);
    const float4 a0 = *reinterpret_cast<const float4 *>(s_ab + c * 8), a1 = *reinterpret_cast<const float4 *>(s_ab + c * 8 + 4);
    const float4 b0 = *reinterpret_cast<const float4 *>(s_ab + C + c * 8), b1 = *reinterpret_cast<const float4 *>(s_ab + C + c * 8 + 4);
    const float ka[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w}, kb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
    if (act == CGAN3D_ACT_RELU) {
#pragma unroll
      for (int k = 0; k < 8; ++k) v.v[k] = fmaxf(fmaf(ka[k], v.v[k], kb[k]), 0.f);
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) v.v[k] = act_fwd(fmaf(ka[k], v.v[k], kb[k]), act, slope);
    }
    v.store(dst + (int64_t)i * 8);
  }
}

template <typename T, int ACT, bool DROP = false>
__global__ void __launch_bounds__(256, 3)
bn_bwd_apply8_kernel(const T *__restrict__ dz, const T *__restrict__ y, T *__restrict__ dy, int64_t total8, int C, double inv_n,
                     const float *__restrict__ mi, const float *__restrict__ gamma, const float *__restrict__ beta, int act,
                     float slope, const double *__restrict__ sums, float *__restrict__ dgamma, float *__restrict__ dbeta, float acc,
                     const uint8_t *__restrict__ keep_bits = nullptr, float scale = 1.f) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (blockIdx.x == 0) {  // the parameter gradients are the reduction's totals: dbeta = sum g, dgamma = sum g * xhat
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      if (dbeta) dbeta[c] = (acc != 0.f ? dbeta[c] : 0.f) + (float)sums[c];
      if (dgamma) dgamma[c] = (acc != 0.f ? dgamma[c] : 0.f) + (float)sums[C + c];
    }
  }
  const int c0 = (int)((i * 8) % C);
  BnC8 k8;
  k8.load(mi, gamma, beta, C, c0);
  float mg[8], mgx[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { mg[k] = (float)(sums[c0 + k] * inv_n); mgx[k] = (float)(sums[C + c0 + k] * inv_n); }
  for (; i < total8; i += 2 * stride) {
    const int64_t e0 = i * 8, e1 = (i + stride) * 8;
    const bool two = i + stride < total8;
    V8<T> y0, d0, y1, d1;
    y0.load(y + e0);
    d0.load(dz + e0);
    if (two) { y1.load(y + e1); d1.load(dz + e1); }
    if constexpr (DROP) {
      const uint32_t kb0 = keep_bits[i], kb1 = two ? keep_bits[i + stride] : 0u;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        d0.v[k] = (kb0 >> k & 1u) ? d0.v[k] * scale : 0.f;
        d1.v[k] = (kb1 >> k & 1u) ? d1.v[k] * scale : 0.f;
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float xh0 = fmaf(y0.v[k], k8.invstd[k], k8.nm[k]), xh1 = fmaf(y1.v[k], k8.invstd[k], k8.nm[k]);
      const float g0 = d0.v[k] * act_bwd_t<ACT>(fmaf(k8.a[k], y0.v[k], k8.b[k]), act, slope);
      const float g1 = d1.v[k] * act_bwd_t<ACT>(fmaf(k8.a[k], y1.v[k], k8.b[k]), act, slope);
      d0.v[k] = k8.a[k] * (g0 - mg[k] - xh0 * mgx[k]);
      d1.v[k] = k8.a[k] * (g1 - mg[k] - xh1 * mgx[k]);
    }
    d0.store(dy + e0);
    if (two) d1.store(dy + e1);
  }
}

// bias + activation on 16-byte chunks (C % 8 == 0): a thread always owns the same 8 channels
template <typename T>
__global__ void __launch_bounds__(256)
bias_act8_kernel(const T *__restrict__ y, T *__restrict__ z, int64_t total8, int C, const float *__restrict__ bias, int act,
                 float slope) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int c0 = (int)((i * 8) % C);
  float b[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) b[k] = bias ? bias[c0 + k] : 0.f;
  for (; i < total8; i += stride) {
    V8<T> v;
    v.load(y + i * 8);
#pragma unroll
    for (int k = 0; k < 8; ++k) v.v[k] = act_fwd(v.v[k] + b[k], act, slope);
    v.store(z + i * 8);
  }
}

// dy = dz * act'(y + bias) and the dbias sums (fp64) in the same pass
template <typename T>
__global__ void __launch_bounds__(256)
bias_act_bwd8_kernel(const T *__restrict__ dz, const T *__restrict__ y, T *__restrict__ dy, int64_t n_rows, int C,
                     const float *__restrict__ bias, int act, float slope, double *sums) {
  const int c0 = (threadIdx.x % (C >> 3)) * 8;
  float b[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) b[k] = bias ? bias[c0 + k] : 0.f;
  constexpr int NV = (int)sizeof(T) / 2;
  col_reduce8_body<1, 4, 2 * NV>(
      n_rows, C, sums,
      [&](int64_t r, uint4 *raw) { load8raw(y + r * C + c0, raw); load8raw(dz + r * C + c0, raw + NV); },
      [&](int64_t r, const uint4 *raw, float (&v)[1][8]) {
        float yy[8], dd[8];
        unpack8<T>(raw, yy);
        unpack8<T>(raw + NV, dd);
        V8<T> o;
#pragma unroll
        for (int k = 0; k < 8; ++k) { o.v[k] = dd[k] * act_bwd(yy[k] + b[k], act, slope); v[0][k] = o.v[k]; }
        o.store(dy + r * C + c0);
      });
}

// ---------------------------------------------------------------- finalize
__global__ void bn_finalize_kernel(const double *__restrict__ sums, int64_t n, int C, float eps, float momentum,
                                   float *__restrict__ mi, float *running_mean, float *running_var,
                                   int64_t *num_batches_tracked) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0 && num_batches_tracked) *num_batches_tracked += 1;
  if (c >= C) return;
  const double mean = sums[c] / (double)n;
  double var = sums[C + c] / (double)n - mean * mean;  // biased variance used for normalisation
  if (var < 0.0) var = 0.0;
  mi[c] = (float)mean;
  mi[C + c] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean) {
    const double unbiased = n > 1 ? var * ((double)n / (double)(n - 1)) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}

__global__ void bn_eval_params_kernel(const float *__restrict__ rm, const float *__restrict__ rv, int C, float eps,
                                      float *__restrict__ mi) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  mi[c] = rm[c];
  mi[C + c] = 1.f / sqrtf(rv[c] + eps);
}

__global__ void sums_to_f32_kernel(const double *__restrict__ sums, float *__restrict__ out, int n, float scale,
                                   float beta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = (float)(sums[i] * (double)scale);
  out[i] = beta != 0.f ? out[i] * beta + v : v;
}

// ---------------------------------------------------------------- elementwise
template <typename T>
__global__ void __launch_bounds__(256)
bn_apply_kernel(const T *__restrict__ y, T *__restrict__ z, int64_t total, int C, const float *__restrict__ mi,
                const float *__restrict__ gamma, const float *__restrict__ beta, int act, float slope,
                const T *__restrict__ residual) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    float v = gamma[c] * ((to_f(y[i]) - mi[c]) * mi[C + c]) + beta[c];
    v = act_fwd(v, act, slope);
    if (residual) v += to_f(residual[i]);
    z[i] = from_f<T>(v);
  }
}

// bn_apply + dropout for any C: thread j owns the 8 elements of keep byte j (the bits past the last element are 0)
template <typename T>
__global__ void __launch_bounds__(256)
bn_apply_dropout_kernel(const T *__restrict__ y, T *__restrict__ z, uint8_t *__restrict__ keep_bits, int64_t total, int C,
                        const float *__restrict__ mi, const float *__restrict__ gamma, const float *__restrict__ beta, int act,
                        float slope, const int64_t *__restrict__ seed_dev, uint64_t thresh, float scale) {
  const uint64_t seed = (uint64_t)*seed_dev;
  const int64_t nbytes = (total + 7) >> 3;
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < nbytes; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = j * 8;
    const int n = (int)mn<int64_t>(8, total - e0);
    const uint32_t bits = dropout_keep8((uint64_t)e0, seed, thresh) & ((1u << n) - 1u);
    int c = (int)(e0 % C);
    for (int k = 0; k < n; ++k) {
      float v = gamma[c] * ((to_f(y[e0 + k]) - mi[c]) * mi[C + c]) + beta[c];  // the arithmetic of bn_apply_kernel
      v = act_fwd(v, act, slope);
      z[e0 + k] = from_f<T>((bits >> k & 1u) ? v * scale : 0.f);
      if (++c == C) c = 0;
    }
    keep_bits[j] = (uint8_t)bits;
  }
}

template <typename T, bool DROP = false>
__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const T *__restrict__ dz, const T *__restrict__ y, T *__restrict__ dy, int64_t total, int C,
                    double inv_n, const float *__restrict__ mi, const float *__restrict__ gamma,
                    const float *__restrict__ beta, int act, float slope, const double *__restrict__ sums,
                    float *__restrict__ dgamma, float *__restrict__ dbeta, float acc,
                    const uint8_t *__restrict__ keep_bits = nullptr, float scale = 1.f) {
  if (blockIdx.x == 0) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      if (dbeta) dbeta[c] = (acc != 0.f ? dbeta[c] : 0.f) + (float)sums[c];
      if (dgamma) dgamma[c] = (acc != 0.f ? dgamma[c] : 0.f) + (float)sums[C + c];
    }
  }
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const float invstd = mi[C + c];
    const float xh = (to_f(y[i]) - mi[c]) * invstd;
    const float pre = gamma[c] * xh + beta[c];
    float d = to_f(dz[i]);
    if constexpr (DROP) d = (keep_bits[i >> 3] >> (i & 7) & 1) ? d * scale : 0.f;
    const float g = d * act_bwd(pre, act, slope);
    const float mg = (float)(sums[c] * inv_n), mgx = (float)(sums[C + c] * inv_n);
    dy[i] = from_f<T>(gamma[c] * invstd * (g - mg - xh * mgx));
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
bias_act_kernel(const T *__restrict__ y, T *__restrict__ z, int64_t total, int C, const float *__restrict__ bias,
                int act, float slope) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    z[i] = from_f<T>(act_fwd(to_f(y[i]) + (bias ? bias[c] : 0.f), act, slope));
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
tanh_residual_kernel(const T *__restrict__ y, const float *__restrict__ bias, const float *__restrict__ x,
                     float *__restrict__ att, float *__restrict__ opt_hat, int64_t n) {
  const float b = bias ? bias[0] : 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float a = tanhf(to_f(y[i]) + b);
    att[i] = a;
    if (opt_hat) opt_hat[i] = x[i] - a;
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
tanh_residual_bwd_kernel(const float *__restrict__ d_opt_hat, const float *__restrict__ d_att,
                         const float *__restrict__ att, T *__restrict__ dy, int64_t n, double *dbias_sum) {
  float part = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float a = att[i];
    float up = 0.f;
    if (d_opt_hat) up -= d_opt_hat[i];
    if (d_att) up += d_att[i];
    const float g = up * (1.f - a * a);
    dy[i] = from_f<T>(g);
    part += g;
  }
  if (dbias_sum) {
    __shared__ double sh[8];
    double p = warp_sum((double)part);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = p;
    __syncthreads();
    if (threadIdx.x == 0) {
      double a = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) a += sh[w];
      atomicAdd(dbias_sum, a);
    }
  }
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) cast_kernel(const TI *__restrict__ in, TO *__restrict__ out, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = from_f<TO>(to_f(in[i]));
}

template <typename T>
__global__ void __launch_bounds__(256) axpy_kernel(const T *__restrict__ x, T *__restrict__ y, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = from_f<T>(to_f(y[i]) + to_f(x[i]));
}

static inline int ew_blocks(int64_t n) { return (int)mx<int64_t>(1, mn<int64_t>((n + 255) / 256, (int64_t)num_sms() * 16)); }

}  // namespace cg

using namespace cg;

#define CG_DTYPE_OK(d, name) \
  if ((d) != CGAN3D_F32 && (d) != CGAN3D_BF16) return fail(CGAN3D_E_DTYPE, name ": unknown dtype %d", (d))

// p -> (threshold, scale) of the keep law; false for p outside [0, 1].  scale is 0 at p = 1 (everything is dropped: the
// outputs and gradients are 0, not 0 * inf).
static bool dropout_consts(float p, uint64_t *thresh, float *scale) {
  if (!(p >= 0.f && p <= 1.f)) return false;
  *thresh = (uint64_t)floor((double)p * 4294967296.0);
  *scale = p < 1.f ? (float)(1.0 / (1.0 - (double)p)) : 0.f;
  return true;
}

// the activation as a template argument for the vec8 kernels (-1: runtime switch), then the dropout flag
template <typename F>
static void with_act_drop(int act, bool drop, F &&go) {
  auto pick_act = [&](auto drop_tag) {
    if (act == CGAN3D_ACT_RELU) go(std::integral_constant<int, CGAN3D_ACT_RELU>{}, drop_tag);
    else if (act == CGAN3D_ACT_LRELU) go(std::integral_constant<int, CGAN3D_ACT_LRELU>{}, drop_tag);
    else if (act == CGAN3D_ACT_NONE) go(std::integral_constant<int, CGAN3D_ACT_NONE>{}, drop_tag);
    else go(std::integral_constant<int, -1>{}, drop_tag);
  };
  if (drop) pick_act(std::true_type{});
  else pick_act(std::false_type{});
}

// keep_bits == nullptr: no dropout (the kernels' DROP = false instantiations)
static int bn_backward_reduce_impl(const char *name, const void *dz, const void *y, int dtype, int64_t n_rows, int C,
                                   const float *mean_invstd, const float *gamma, const float *beta, int act, float slope,
                                   double *sums, const uint8_t *keep_bits, float scale, void *stream) {
  CG_CHECK_ARG(dz && y && mean_invstd && gamma && beta && sums, "%s: NULL pointer", name);
  CG_DTYPE_OK(dtype, "bn_backward_reduce");
  CG_CHECK_SHAPE(n_rows > 0 && C > 0 && (C <= 256 || C % 256 == 0), "%s: bad sizes", name);
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(sums, 0, 2 * (size_t)C * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "bn_backward_reduce memset");
  if (vec8_ok(C, dz, y)) {
    ColGrid g8 = col_grid8(n_rows, C, 2);
    with_act_drop(act, keep_bits != nullptr, [&](auto act_tag, auto drop_tag) {
      constexpr int A = decltype(act_tag)::value;
      constexpr bool D = decltype(drop_tag)::value;
      if (dtype == CGAN3D_F32)
        // fp32 with the keep byte: two rows in flight per thread instead of four fit the 128 registers without spilling
        bn_bwd_reduce8_kernel<float, A, D, D ? 2 : 4><<<g8.blocks, 256, g8.smem, st>>>((const float *)dz, (const float *)y, n_rows, C,
                                                                            g8.rows_per_block, mean_invstd, gamma, beta, act, slope,
                                                                            sums, keep_bits, scale);
      else
        bn_bwd_reduce8_kernel<__nv_bfloat16, A, D><<<g8.blocks, 256, g8.smem, st>>>(
            (const __nv_bfloat16 *)dz, (const __nv_bfloat16 *)y, n_rows, C, g8.rows_per_block, mean_invstd, gamma, beta, act, slope,
            sums, keep_bits, scale);
    });
    CG_LAUNCH_CHECK("bn_backward_reduce(vec8)");
    return 0;
  }
  ColGrid g = col_grid(n_rows, C, 2);
  auto go = [&](auto drop_tag) {
    constexpr bool D = decltype(drop_tag)::value;
    if (dtype == CGAN3D_F32)
      bn_bwd_reduce_kernel<float, D><<<g.blocks, 256, g.smem, st>>>((const float *)dz, (const float *)y, n_rows, C,
                                                                    g.rows_per_block, mean_invstd, gamma, beta, act, slope, sums,
                                                                    keep_bits, scale);
    else
      bn_bwd_reduce_kernel<__nv_bfloat16, D><<<g.blocks, 256, g.smem, st>>>((const __nv_bfloat16 *)dz, (const __nv_bfloat16 *)y,
                                                                            n_rows, C, g.rows_per_block, mean_invstd, gamma,
                                                                            beta, act, slope, sums, keep_bits, scale);
  };
  if (keep_bits) go(std::true_type{});
  else go(std::false_type{});
  CG_LAUNCH_CHECK("bn_backward_reduce");
  return 0;
}

static int bn_backward_apply_impl(const char *name, const void *dz, const void *y, void *dy, int dtype, int64_t n_rows, int C,
                                  const float *mean_invstd, const float *gamma, const float *beta, int act, float slope,
                                  const double *sums, float *dgamma, float *dbeta, float grad_beta, const uint8_t *keep_bits,
                                  float scale, void *stream) {
  CG_CHECK_ARG(dz && y && dy && mean_invstd && gamma && beta && sums, "%s: NULL pointer", name);
  CG_CHECK_ARG(grad_beta == 0.f || grad_beta == 1.f, "%s: grad_beta must be 0 (overwrite) or 1 (accumulate)", name);
  CG_DTYPE_OK(dtype, "bn_backward_apply");
  CG_CHECK_SHAPE(n_rows > 0 && C > 0, "%s: bad sizes", name);
  cudaStream_t st = as_stream(stream);
  const int64_t total = n_rows * C;
  const double inv_n = 1.0 / (double)n_rows;
  if (vec8_ok(C, dz, y, dy)) {
    const int64_t t8 = total / 8;
    with_act_drop(act, keep_bits != nullptr, [&](auto act_tag, auto drop_tag) {
      constexpr int A = decltype(act_tag)::value;
      constexpr bool D = decltype(drop_tag)::value;
      if (dtype == CGAN3D_F32)
        bn_bwd_apply8_kernel<float, A, D><<<ew_blocks(t8), 256, 0, st>>>((const float *)dz, (const float *)y, (float *)dy, t8, C,
                                                                         inv_n, mean_invstd, gamma, beta, act, slope, sums, dgamma,
                                                                         dbeta, grad_beta, keep_bits, scale);
      else
        bn_bwd_apply8_kernel<__nv_bfloat16, A, D><<<ew_blocks(t8), 256, 0, st>>>(
            (const __nv_bfloat16 *)dz, (const __nv_bfloat16 *)y, (__nv_bfloat16 *)dy, t8, C, inv_n, mean_invstd, gamma, beta, act,
            slope, sums, dgamma, dbeta, grad_beta, keep_bits, scale);
    });
    CG_LAUNCH_CHECK("bn_backward_apply(vec8)");
    return 0;
  }
  auto go = [&](auto drop_tag) {
    constexpr bool D = decltype(drop_tag)::value;
    if (dtype == CGAN3D_F32)
      bn_bwd_apply_kernel<float, D><<<ew_blocks(total), 256, 0, st>>>((const float *)dz, (const float *)y, (float *)dy, total, C,
                                                                      inv_n, mean_invstd, gamma, beta, act, slope, sums, dgamma,
                                                                      dbeta, grad_beta, keep_bits, scale);
    else
      bn_bwd_apply_kernel<__nv_bfloat16, D><<<ew_blocks(total), 256, 0, st>>>(
          (const __nv_bfloat16 *)dz, (const __nv_bfloat16 *)y, (__nv_bfloat16 *)dy, total, C, inv_n, mean_invstd, gamma, beta,
          act, slope, sums, dgamma, dbeta, grad_beta, keep_bits, scale);
  };
  if (keep_bits) go(std::true_type{});
  else go(std::false_type{});
  CG_LAUNCH_CHECK("bn_backward_apply");
  return 0;
}

extern "C" {

int cgan3d_bn_stats(const void *y, int dtype, int64_t n_rows, int C, double *sums, void *stream) {
  CG_CHECK_ARG(y && sums, "bn_stats: NULL pointer");
  CG_DTYPE_OK(dtype, "bn_stats");
  CG_CHECK_SHAPE(n_rows >= 0 && C > 0 && (C <= 256 || C % 256 == 0), "bn_stats: bad sizes");
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(sums, 0, 2 * (size_t)C * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "bn_stats memset");
  if (n_rows == 0) return 0;
  if (vec8_ok(C, y)) {
    ColGrid g8 = col_grid8(n_rows, C, 2);
    if (dtype == CGAN3D_F32)
      bn_stats8_kernel<float><<<g8.blocks, 256, g8.smem, st>>>((const float *)y, n_rows, C, g8.rows_per_block, sums);
    else
      bn_stats8_kernel<__nv_bfloat16><<<g8.blocks, 256, g8.smem, st>>>((const __nv_bfloat16 *)y, n_rows, C, g8.rows_per_block, sums);
    CG_LAUNCH_CHECK("bn_stats(vec8)");
    return 0;
  }
  ColGrid g = col_grid(n_rows, C, 2);
  if (dtype == CGAN3D_F32)
    bn_stats_kernel<float><<<g.blocks, 256, g.smem, st>>>((const float *)y, n_rows, C, g.rows_per_block, sums);
  else
    bn_stats_kernel<__nv_bfloat16><<<g.blocks, 256, g.smem, st>>>((const __nv_bfloat16 *)y, n_rows, C, g.rows_per_block, sums);
  CG_LAUNCH_CHECK("bn_stats");
  return 0;
}

int cgan3d_col_sums(const void *x, int dtype, int64_t n_rows, int C, double *sums, void *stream) {
  CG_CHECK_ARG(x && sums, "col_sums: NULL pointer");
  CG_DTYPE_OK(dtype, "col_sums");
  CG_CHECK_SHAPE(n_rows >= 0 && C > 0 && (C <= 256 || C % 256 == 0), "col_sums: bad sizes");
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(sums, 0, (size_t)C * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "col_sums memset");
  if (n_rows == 0) return 0;
  ColGrid g = col_grid(n_rows, C, 1);
  if (dtype == CGAN3D_F32)
    col_sums_kernel<float><<<g.blocks, 256, g.smem, st>>>((const float *)x, n_rows, C, g.rows_per_block, sums);
  else
    col_sums_kernel<__nv_bfloat16><<<g.blocks, 256, g.smem, st>>>((const __nv_bfloat16 *)x, n_rows, C, g.rows_per_block, sums);
  CG_LAUNCH_CHECK("col_sums");
  return 0;
}

int cgan3d_bn_finalize(const double *sums, int64_t n_rows, int C, float eps, float momentum, float *mean_invstd,
                       float *running_mean, float *running_var, int64_t *num_batches_tracked, void *stream) {
  CG_CHECK_ARG(sums && mean_invstd, "bn_finalize: NULL pointer");
  CG_CHECK_ARG((running_mean == nullptr) == (running_var == nullptr), "bn_finalize: running stats must come in pairs");
  CG_CHECK_SHAPE(n_rows > 0 && C > 0, "bn_finalize: bad sizes");
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, as_stream(stream)>>>(sums, n_rows, C, eps, momentum, mean_invstd,
                                                                     running_mean, running_var, num_batches_tracked);
  CG_LAUNCH_CHECK("bn_finalize");
  return 0;
}

int cgan3d_bn_eval_params(const float *running_mean, const float *running_var, int C, float eps, float *mean_invstd,
                          void *stream) {
  CG_CHECK_ARG(running_mean && running_var && mean_invstd, "bn_eval_params: NULL pointer");
  CG_CHECK_SHAPE(C > 0, "bn_eval_params: bad C");
  bn_eval_params_kernel<<<(C + 127) / 128, 128, 0, as_stream(stream)>>>(running_mean, running_var, C, eps, mean_invstd);
  CG_LAUNCH_CHECK("bn_eval_params");
  return 0;
}

int cgan3d_sums_to_f32(const double *sums, float *out, int n, float scale, float beta, void *stream) {
  CG_CHECK_ARG(sums && out && n > 0, "sums_to_f32: bad args");
  sums_to_f32_kernel<<<(n + 127) / 128, 128, 0, as_stream(stream)>>>(sums, out, n, scale, beta);
  CG_LAUNCH_CHECK("sums_to_f32");
  return 0;
}

int cgan3d_bn_apply(const void *y, void *z, int dtype, int64_t n_rows, int C, const float *mean_invstd,
                    const float *gamma, const float *beta, int act, float slope, const void *residual, void *stream) {
  CG_CHECK_ARG(y && z && mean_invstd && gamma && beta, "bn_apply: NULL pointer");
  CG_DTYPE_OK(dtype, "bn_apply");
  CG_CHECK_SHAPE(n_rows >= 0 && C > 0, "bn_apply: bad sizes");
  const int64_t total = n_rows * C;
  if (total == 0) return 0;
  cudaStream_t st = as_stream(stream);
  if (vec8_ok(C, y, z, residual)) {
    const int64_t t8 = total / 8;
    if (dtype == CGAN3D_F32)
      bn_apply8_kernel<float><<<ew_blocks(t8), 256, 0, st>>>((const float *)y, (float *)z, t8, C, mean_invstd, gamma, beta, act,
                                                             slope, (const float *)residual);
    else
      bn_apply8_kernel<__nv_bfloat16><<<ew_blocks(t8), 256, 0, st>>>((const __nv_bfloat16 *)y, (__nv_bfloat16 *)z, t8, C, mean_invstd,
                                                                     gamma, beta, act, slope, (const __nv_bfloat16 *)residual);
    CG_LAUNCH_CHECK("bn_apply(vec8)");
    return 0;
  }
  if (dtype == CGAN3D_F32)
    bn_apply_kernel<float><<<ew_blocks(total), 256, 0, st>>>((const float *)y, (float *)z, total, C, mean_invstd, gamma,
                                                             beta, act, slope, (const float *)residual);
  else
    bn_apply_kernel<__nv_bfloat16><<<ew_blocks(total), 256, 0, st>>>((const __nv_bfloat16 *)y, (__nv_bfloat16 *)z, total,
                                                                     C, mean_invstd, gamma, beta, act, slope,
                                                                     (const __nv_bfloat16 *)residual);
  CG_LAUNCH_CHECK("bn_apply");
  return 0;
}

int cgan3d_bn_apply_pad(const void *y, void *z_padded, int dtype, int B, int X, int Y, int Z, int C, const float *mean_invstd,
                        const float *gamma, const float *beta, int act, float slope, int pad, void *stream) {
  CG_CHECK_ARG(y && z_padded && mean_invstd && gamma && beta, "bn_apply_pad: NULL pointer");
  CG_DTYPE_OK(dtype, "bn_apply_pad");
  CG_CHECK_SHAPE(B > 0 && X > 0 && Y > 0 && Z > 0 && C > 0 && pad > 0 && pad < X && pad < Y && pad < Z, "bn_apply_pad: bad sizes");
  if (C % 8 || !vec8_ok(C, y, z_padded) || X + 2 * pad > 65535 || B > 65535)
    return fail(CGAN3D_E_UNSUPPORTED, "bn_apply_pad: needs C %% 8 == 0 and 16-byte aligned tensors");
  cudaStream_t st = as_stream(stream);
  const dim3 grid((unsigned)(Y + 2 * pad), (unsigned)(X + 2 * pad), (unsigned)B);
  const size_t smem = 2 * (size_t)C * sizeof(float);
  if (dtype == CGAN3D_F32)
    bn_apply_pad8_kernel<float><<<grid, 256, smem, st>>>((const float *)y, (float *)z_padded, X, Y, Z, C, pad, mean_invstd, gamma, beta, act, slope);
  else
    bn_apply_pad8_kernel<__nv_bfloat16><<<grid, 256, smem, st>>>((const __nv_bfloat16 *)y, (__nv_bfloat16 *)z_padded, X, Y, Z, C, pad,
                                                                 mean_invstd, gamma, beta, act, slope);
  CG_LAUNCH_CHECK("bn_apply_pad");
  return 0;
}

int cgan3d_bn_apply_dropout(const void *y, void *z, uint8_t *keep_bits, int dtype, int64_t n_rows, int C,
                            const float *mean_invstd, const float *gamma, const float *beta, int act, float slope, float p,
                            const int64_t *seed_dev, void *stream) {
  CG_CHECK_ARG(y && z && keep_bits && mean_invstd && gamma && beta && seed_dev, "bn_apply_dropout: NULL pointer");
  CG_DTYPE_OK(dtype, "bn_apply_dropout");
  CG_CHECK_SHAPE(n_rows >= 0 && C > 0, "bn_apply_dropout: bad sizes");
  uint64_t thresh;
  float scale;
  if (!dropout_consts(p, &thresh, &scale)) return fail(CGAN3D_E_ARG, "bn_apply_dropout: p = %g is outside [0, 1]", (double)p);
  const int64_t total = n_rows * C;
  if (total == 0) return 0;
  cudaStream_t st = as_stream(stream);
  if (vec8_ok(C, y, z)) {
    const int64_t t8 = total / 8;
    if (dtype == CGAN3D_F32)
      bn_apply8_kernel<float, true><<<ew_blocks(t8), 256, 0, st>>>((const float *)y, (float *)z, t8, C, mean_invstd, gamma, beta, act,
                                                                   slope, nullptr, keep_bits, seed_dev, thresh, scale);
    else
      bn_apply8_kernel<__nv_bfloat16, true><<<ew_blocks(t8), 256, 0, st>>>((const __nv_bfloat16 *)y, (__nv_bfloat16 *)z, t8, C,
                                                                           mean_invstd, gamma, beta, act, slope, nullptr, keep_bits,
                                                                           seed_dev, thresh, scale);
    CG_LAUNCH_CHECK("bn_apply_dropout(vec8)");
    return 0;
  }
  const int64_t nbytes = (total + 7) / 8;
  if (dtype == CGAN3D_F32)
    bn_apply_dropout_kernel<float><<<ew_blocks(nbytes), 256, 0, st>>>((const float *)y, (float *)z, keep_bits, total, C, mean_invstd,
                                                                      gamma, beta, act, slope, seed_dev, thresh, scale);
  else
    bn_apply_dropout_kernel<__nv_bfloat16><<<ew_blocks(nbytes), 256, 0, st>>>((const __nv_bfloat16 *)y, (__nv_bfloat16 *)z, keep_bits,
                                                                              total, C, mean_invstd, gamma, beta, act, slope,
                                                                              seed_dev, thresh, scale);
  CG_LAUNCH_CHECK("bn_apply_dropout");
  return 0;
}

int cgan3d_bn_backward_reduce(const void *dz, const void *y, int dtype, int64_t n_rows, int C, const float *mean_invstd,
                              const float *gamma, const float *beta, int act, float slope, double *sums, void *stream) {
  return bn_backward_reduce_impl("bn_backward_reduce", dz, y, dtype, n_rows, C, mean_invstd, gamma, beta, act, slope, sums,
                                 nullptr, 1.f, stream);
}

int cgan3d_bn_backward_reduce_dropout(const void *dz, const void *y, const uint8_t *keep_bits, int dtype, int64_t n_rows, int C,
                                      const float *mean_invstd, const float *gamma, const float *beta, int act, float slope,
                                      float p, double *sums, void *stream) {
  uint64_t thresh;
  float scale;
  CG_CHECK_ARG(keep_bits, "bn_backward_reduce_dropout: NULL pointer");
  if (!dropout_consts(p, &thresh, &scale)) return fail(CGAN3D_E_ARG, "bn_backward_reduce_dropout: p = %g is outside [0, 1]", (double)p);
  return bn_backward_reduce_impl("bn_backward_reduce_dropout", dz, y, dtype, n_rows, C, mean_invstd, gamma, beta, act, slope, sums,
                                 keep_bits, scale, stream);
}

int cgan3d_bn_backward_apply(const void *dz, const void *y, void *dy, int dtype, int64_t n_rows, int C,
                             const float *mean_invstd, const float *gamma, const float *beta, int act, float slope,
                             const double *sums, float *dgamma, float *dbeta, float grad_beta, void *stream) {
  return bn_backward_apply_impl("bn_backward_apply", dz, y, dy, dtype, n_rows, C, mean_invstd, gamma, beta, act, slope, sums,
                                dgamma, dbeta, grad_beta, nullptr, 1.f, stream);
}

int cgan3d_bn_backward_apply_dropout(const void *dz, const void *y, const uint8_t *keep_bits, void *dy, int dtype, int64_t n_rows,
                                     int C, const float *mean_invstd, const float *gamma, const float *beta, int act, float slope,
                                     float p, const double *sums, float *dgamma, float *dbeta, float grad_beta, void *stream) {
  uint64_t thresh;
  float scale;
  CG_CHECK_ARG(keep_bits, "bn_backward_apply_dropout: NULL pointer");
  if (!dropout_consts(p, &thresh, &scale)) return fail(CGAN3D_E_ARG, "bn_backward_apply_dropout: p = %g is outside [0, 1]", (double)p);
  return bn_backward_apply_impl("bn_backward_apply_dropout", dz, y, dy, dtype, n_rows, C, mean_invstd, gamma, beta, act, slope,
                                sums, dgamma, dbeta, grad_beta, keep_bits, scale, stream);
}

int cgan3d_bias_act(const void *y, void *z, int dtype, int64_t n_rows, int C, const float *bias, int act, float slope,
                    void *stream) {
  CG_CHECK_ARG(y && z, "bias_act: NULL pointer");
  CG_DTYPE_OK(dtype, "bias_act");
  CG_CHECK_SHAPE(n_rows >= 0 && C > 0, "bias_act: bad sizes");
  const int64_t total = n_rows * C;
  if (total == 0) return 0;
  cudaStream_t st = as_stream(stream);
  if (vec8_ok(C, y, z)) {
    const int64_t t8 = total / 8;
    if (dtype == CGAN3D_F32)
      bias_act8_kernel<float><<<ew_blocks(t8), 256, 0, st>>>((const float *)y, (float *)z, t8, C, bias, act, slope);
    else
      bias_act8_kernel<__nv_bfloat16><<<ew_blocks(t8), 256, 0, st>>>((const __nv_bfloat16 *)y, (__nv_bfloat16 *)z, t8, C, bias, act,
                                                                     slope);
    CG_LAUNCH_CHECK("bias_act(vec8)");
    return 0;
  }
  if (dtype == CGAN3D_F32)
    bias_act_kernel<float><<<ew_blocks(total), 256, 0, st>>>((const float *)y, (float *)z, total, C, bias, act, slope);
  else
    bias_act_kernel<__nv_bfloat16><<<ew_blocks(total), 256, 0, st>>>((const __nv_bfloat16 *)y, (__nv_bfloat16 *)z, total, C,
                                                                     bias, act, slope);
  CG_LAUNCH_CHECK("bias_act");
  return 0;
}

int cgan3d_bias_act_backward(const void *dz, const void *y, void *dy, int dtype, int64_t n_rows, int C, const float *bias,
                             int act, float slope, double *dbias_sums, void *stream) {
  CG_CHECK_ARG(dz && y && dy && dbias_sums, "bias_act_backward: NULL pointer");
  CG_DTYPE_OK(dtype, "bias_act_backward");
  CG_CHECK_SHAPE(n_rows > 0 && C > 0 && (C <= 256 || C % 256 == 0), "bias_act_backward: bad sizes");
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(dbias_sums, 0, (size_t)C * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "bias_act_backward memset");
  if (vec8_ok(C, dz, y, dy)) {
    ColGrid g8 = col_grid8(n_rows, C, 1);
    if (dtype == CGAN3D_F32)
      bias_act_bwd8_kernel<float><<<g8.blocks, 256, g8.smem, st>>>((const float *)dz, (const float *)y, (float *)dy, n_rows, C, bias,
                                                                   act, slope, dbias_sums);
    else
      bias_act_bwd8_kernel<__nv_bfloat16><<<g8.blocks, 256, g8.smem, st>>>((const __nv_bfloat16 *)dz, (const __nv_bfloat16 *)y,
                                                                           (__nv_bfloat16 *)dy, n_rows, C, bias, act, slope, dbias_sums);
    CG_LAUNCH_CHECK("bias_act_backward(vec8)");
    return 0;
  }
  ColGrid g = col_grid(n_rows, C, 1);
  if (dtype == CGAN3D_F32)
    bias_act_bwd_kernel<float><<<g.blocks, 256, g.smem, st>>>((const float *)dz, (const float *)y, (float *)dy, n_rows, C,
                                                              g.rows_per_block, bias, act, slope, dbias_sums);
  else
    bias_act_bwd_kernel<__nv_bfloat16><<<g.blocks, 256, g.smem, st>>>((const __nv_bfloat16 *)dz, (const __nv_bfloat16 *)y,
                                                                      (__nv_bfloat16 *)dy, n_rows, C, g.rows_per_block,
                                                                      bias, act, slope, dbias_sums);
  CG_LAUNCH_CHECK("bias_act_backward");
  return 0;
}

int cgan3d_tanh_residual(const void *y, const float *bias, const float *x, float *attenuation, float *opt_hat, int dtype,
                         int64_t n, void *stream) {
  CG_CHECK_ARG(y && attenuation, "tanh_residual: NULL pointer");
  CG_CHECK_ARG(opt_hat == nullptr || x != nullptr, "tanh_residual: opt_hat requires x");
  CG_DTYPE_OK(dtype, "tanh_residual");
  if (n <= 0) return 0;
  cudaStream_t st = as_stream(stream);
  if (dtype == CGAN3D_F32)
    tanh_residual_kernel<float><<<ew_blocks(n), 256, 0, st>>>((const float *)y, bias, x, attenuation, opt_hat, n);
  else
    tanh_residual_kernel<__nv_bfloat16><<<ew_blocks(n), 256, 0, st>>>((const __nv_bfloat16 *)y, bias, x, attenuation,
                                                                      opt_hat, n);
  CG_LAUNCH_CHECK("tanh_residual");
  return 0;
}

int cgan3d_tanh_residual_backward(const float *d_opt_hat, const float *d_att, const float *attenuation, void *dy,
                                  int dtype, int64_t n, double *dbias_sum, void *stream) {
  CG_CHECK_ARG(attenuation && dy && (d_opt_hat || d_att), "tanh_residual_backward: NULL pointer");
  CG_DTYPE_OK(dtype, "tanh_residual_backward");
  if (n <= 0) return 0;
  cudaStream_t st = as_stream(stream);
  if (dbias_sum) {
    cudaError_t e = cudaMemsetAsync(dbias_sum, 0, sizeof(double), st);
    if (e != cudaSuccess) return cuda_fail(e, "tanh_residual_backward memset");
  }
  if (dtype == CGAN3D_F32)
    tanh_residual_bwd_kernel<float><<<ew_blocks(n), 256, 0, st>>>(d_opt_hat, d_att, attenuation, (float *)dy, n, dbias_sum);
  else
    tanh_residual_bwd_kernel<__nv_bfloat16><<<ew_blocks(n), 256, 0, st>>>(d_opt_hat, d_att, attenuation,
                                                                          (__nv_bfloat16 *)dy, n, dbias_sum);
  CG_LAUNCH_CHECK("tanh_residual_backward");
  return 0;
}

int cgan3d_cast(const void *in, int in_dtype, void *out, int out_dtype, int64_t n, void *stream) {
  CG_CHECK_ARG(in && out, "cast: NULL pointer");
  CG_DTYPE_OK(in_dtype, "cast");
  CG_DTYPE_OK(out_dtype, "cast");
  if (n <= 0) return 0;
  cudaStream_t st = as_stream(stream);
  const int nb = ew_blocks(n);
  if (in_dtype == CGAN3D_F32 && out_dtype == CGAN3D_BF16)
    cast_kernel<float, __nv_bfloat16><<<nb, 256, 0, st>>>((const float *)in, (__nv_bfloat16 *)out, n);
  else if (in_dtype == CGAN3D_BF16 && out_dtype == CGAN3D_F32)
    cast_kernel<__nv_bfloat16, float><<<nb, 256, 0, st>>>((const __nv_bfloat16 *)in, (float *)out, n);
  else if (in_dtype == CGAN3D_F32)
    cast_kernel<float, float><<<nb, 256, 0, st>>>((const float *)in, (float *)out, n);
  else
    cast_kernel<__nv_bfloat16, __nv_bfloat16><<<nb, 256, 0, st>>>((const __nv_bfloat16 *)in, (__nv_bfloat16 *)out, n);
  CG_LAUNCH_CHECK("cast");
  return 0;
}

int cgan3d_axpy(const void *x, void *y, int dtype, int64_t n, void *stream) {
  CG_CHECK_ARG(x && y, "axpy: NULL pointer");
  CG_DTYPE_OK(dtype, "axpy");
  if (n <= 0) return 0;
  cudaStream_t st = as_stream(stream);
  if (dtype == CGAN3D_F32) axpy_kernel<float><<<ew_blocks(n), 256, 0, st>>>((const float *)x, (float *)y, n);
  else axpy_kernel<__nv_bfloat16><<<ew_blocks(n), 256, 0, st>>>((const __nv_bfloat16 *)x, (__nv_bfloat16 *)y, n);
  CG_LAUNCH_CHECK("axpy");
  return 0;
}

}  // extern "C"
