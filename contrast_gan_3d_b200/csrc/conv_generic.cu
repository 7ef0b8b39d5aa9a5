// Generic CUDA-core convolution kernels (any channel count, k in {1..7}, stride 1/2).
// fp32 accumulation; storage type T = float or bf16; channels-last [B][X][Y][Z][C].
// These are the always-available correct path and the on-device checker for the tcgen05
// kernels in conv_tc.cu.  Replaces aten::convolution / convolution_backward
// (reference model/blocks.py:29-38,52).
#include "common.cuh"
#include "conv_internal.cuh"

namespace cg {

// ------------------------------------------------------------------ weight packing
template <typename T>
__global__ void pack_weights_kernel(const float *__restrict__ w, T *__restrict__ p, int Cs, int Cb, int taps) {
  int64_t total = (int64_t)taps * Cb * Cs;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int cs = (int)(i % Cs);
    int cb = (int)((i / Cs) % Cb);
    int t = (int)(i / ((int64_t)Cs * Cb));
    p[i] = from_f<T>(w[((int64_t)cs * Cb + cb) * taps + t]);
  }
}

// ------------------------------------------------------------------ gather (fprop)
// one thread: VB consecutive z outputs x COB output channels
template <typename T, int K, int S, int COB, int VB>
__global__ void __launch_bounds__(128)
gather_kernel(cgan3d_conv_geom g, const T *__restrict__ big, const T *__restrict__ wp,
              const float *__restrict__ bias, T *__restrict__ small) {
  const int ncob = g.Cs / COB;
  const int nzg = (g.Zs + VB - 1) / VB;
  const int64_t total = (int64_t)g.B * g.Xs * g.Ys * nzg * ncob;
  int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int cob = (int)(idx % ncob); idx /= ncob;
  const int zg = (int)(idx % nzg); idx /= nzg;
  const int oy = (int)(idx % g.Ys); idx /= g.Ys;
  const int ox = (int)(idx % g.Xs);
  const int b = (int)(idx / g.Xs);
  const int oz0 = zg * VB, co0 = cob * COB;
  constexpr int NZ = (VB - 1) * S + K;
  float acc[VB][COB];
#pragma unroll
  for (int v = 0; v < VB; ++v)
#pragma unroll
    for (int c = 0; c < COB; ++c) acc[v][c] = bias ? bias[co0 + c] : 0.f;
  const int iz0 = oz0 * S - g.pad;
  for (int kx = 0; kx < K; ++kx) {
    const int ix = ox * S - g.pad + kx;
    if ((unsigned)ix >= (unsigned)g.Xb) continue;
    for (int ky = 0; ky < K; ++ky) {
      const int iy = oy * S - g.pad + ky;
      if ((unsigned)iy >= (unsigned)g.Yb) continue;
      const T *xrow = big + (((int64_t)b * g.Xb + ix) * g.Yb + iy) * (int64_t)g.Zb * g.Cb;
      const T *wrow = wp + (int64_t)((kx * K + ky) * K) * g.Cb * g.Cs + co0;
      for (int ci = 0; ci < g.Cb; ++ci) {
        float xs[NZ];
#pragma unroll
        for (int j = 0; j < NZ; ++j) {
          const int iz = iz0 + j;
          xs[j] = ((unsigned)iz < (unsigned)g.Zb) ? to_f(xrow[(int64_t)iz * g.Cb + ci]) : 0.f;
        }
#pragma unroll
        for (int kz = 0; kz < K; ++kz) {
          float w[COB];
          const T *wq = wrow + (int64_t)(kz * g.Cb + ci) * g.Cs;
#pragma unroll
          for (int c = 0; c < COB; ++c) w[c] = to_f(wq[c]);
#pragma unroll
          for (int v = 0; v < VB; ++v)
#pragma unroll
            for (int c = 0; c < COB; ++c) acc[v][c] = fmaf(xs[v * S + kz], w[c], acc[v][c]);
        }
      }
    }
  }
#pragma unroll
  for (int v = 0; v < VB; ++v) {
    const int oz = oz0 + v;
    if (oz < g.Zs) {
      T *o = small + ((((int64_t)b * g.Xs + ox) * g.Ys + oy) * g.Zs + oz) * g.Cs + co0;
#pragma unroll
      for (int c = 0; c < COB; ++c) o[c] = from_f<T>(acc[v][c]);
    }
  }
}


// ------------------------------------------------------------------ gather, Cs == 1 (last_conv / critic logits)
// one thread: VB consecutive z outputs of the single output channel; input channels are consumed 8 at a time
// (one 16 B / 32 B vector load per voxel), weights [tap][Cb][1] are contiguous over ci.
template <typename T>
struct Vec8;
template <>
struct Vec8<float> {
  float v[8];
  __device__ __forceinline__ void load(const float *p) {
    const float4 a = *reinterpret_cast<const float4 *>(p), b = *reinterpret_cast<const float4 *>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
};
template <>
struct Vec8<__nv_bfloat16> {
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
};

template <typename T, int K, int S, int VB>
__global__ void __launch_bounds__(128)
gather_co1_kernel(cgan3d_conv_geom g, const T *__restrict__ big, const T *__restrict__ wp, const float *__restrict__ bias,
                  T *__restrict__ small) {
  const int nzg = (g.Zs + VB - 1) / VB;
  const int64_t total = (int64_t)g.B * g.Xs * g.Ys * nzg;
  int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int zg = (int)(idx % nzg); idx /= nzg;
  const int oy = (int)(idx % g.Ys); idx /= g.Ys;
  const int ox = (int)(idx % g.Xs);
  const int b = (int)(idx / g.Xs);
  const int oz0 = zg * VB;
  constexpr int NZ = (VB - 1) * S + K;
  float acc[VB];
#pragma unroll
  for (int v = 0; v < VB; ++v) acc[v] = bias ? bias[0] : 0.f;
  const int iz0 = oz0 * S - g.pad;
  for (int kx = 0; kx < K; ++kx) {
    const int ix = ox * S - g.pad + kx;
    if ((unsigned)ix >= (unsigned)g.Xb) continue;
    for (int ky = 0; ky < K; ++ky) {
      const int iy = oy * S - g.pad + ky;
      if ((unsigned)iy >= (unsigned)g.Yb) continue;
      const T *xrow = big + (((int64_t)b * g.Xb + ix) * g.Yb + iy) * (int64_t)g.Zb * g.Cb;
      const T *wrow = wp + (int64_t)((kx * K + ky) * K) * g.Cb;
      for (int c0 = 0; c0 < g.Cb; c0 += 8) {
        Vec8<T> wv[K];
#pragma unroll
        for (int kz = 0; kz < K; ++kz) wv[kz].load(wrow + (int64_t)kz * g.Cb + c0);
#pragma unroll
        for (int j = 0; j < NZ; ++j) {
          const int iz = iz0 + j;
          if ((unsigned)iz >= (unsigned)g.Zb) continue;
          Vec8<T> xv;
          xv.load(xrow + (int64_t)iz * g.Cb + c0);
#pragma unroll
          for (int kz = 0; kz < K; ++kz) {
            const int jv = j - kz;  // output v = (j - kz) / S when divisible
            if (jv >= 0 && jv % S == 0 && jv / S < VB) {
              float sum = 0.f;
#pragma unroll
              for (int c = 0; c < 8; ++c) sum = fmaf(xv.v[c], wv[kz].v[c], sum);
              acc[jv / S] += sum;
            }
          }
        }
      }
    }
  }
#pragma unroll
  for (int v = 0; v < VB; ++v) {
    const int oz = oz0 + v;
    if (oz < g.Zs) small[(((int64_t)b * g.Xs + ox) * g.Ys + oy) * g.Zs + oz] = from_f<T>(acc[v]);
  }
}

// Cout == 1 on a SMALL output grid (the critic's logits map): one warp per output voxel, the lanes share the
// K^3 x Cb/8 (tap, 8-channel chunk) units and shuffle-reduce -- the one-thread-per-8-outputs kernel above leaves
// almost all SMs idle at this size.
template <typename T, int K, int S>
__global__ void __launch_bounds__(128)
gather_co1_warp_kernel(cgan3d_conv_geom g, const T *__restrict__ big, const T *__restrict__ wp, const float *__restrict__ bias,
                       T *__restrict__ small, int64_t total) {
  const int64_t o = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (o >= total) return;
  int64_t t = o;
  const int oz = (int)(t % g.Zs); t /= g.Zs;
  const int oy = (int)(t % g.Ys); t /= g.Ys;
  const int ox = (int)(t % g.Xs);
  const int b = (int)(t / g.Xs);
  const int c8n = g.Cb >> 3, units = K * K * K * c8n;
  float acc = 0.f;
  for (int u = lane; u < units; u += 32) {
    const int tap = u / c8n, c0 = (u - tap * c8n) * 8;
    const int kz = tap % K, ky = (tap / K) % K, kx = tap / (K * K);
    const int ix = ox * S - g.pad + kx, iy = oy * S - g.pad + ky, iz = oz * S - g.pad + kz;
    if ((unsigned)ix >= (unsigned)g.Xb || (unsigned)iy >= (unsigned)g.Yb || (unsigned)iz >= (unsigned)g.Zb) continue;
    Vec8<T> xv, wv;
    xv.load(big + ((((int64_t)b * g.Xb + ix) * g.Yb + iy) * g.Zb + iz) * (int64_t)g.Cb + c0);
    wv.load(wp + (int64_t)tap * g.Cb + c0);
#pragma unroll
    for (int c = 0; c < 8; ++c) acc = fmaf(xv.v[c], wv.v[c], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) small[o] = from_f<T>(acc + (bias ? bias[0] : 0.f));
}

template <typename T, int K, int S>
static int launch_gather(const cgan3d_conv_geom &g, const T *big, const T *wp, const float *bias, T *small,
                         cudaStream_t st) {
  constexpr int VB = 4;
  const int nzg = (g.Zs + VB - 1) / VB;
  const bool vec_ok = g.Cb % 8 == 0 && (reinterpret_cast<uintptr_t>(big) & (8 * sizeof(T) - 1)) == 0 &&
                      (reinterpret_cast<uintptr_t>(wp) & (8 * sizeof(T) - 1)) == 0;
  if (g.Cs == 1 && vec_ok && (int64_t)g.B * g.Xs * g.Ys * g.Zs <= (1 << 17)) {
    const int64_t total = (int64_t)g.B * g.Xs * g.Ys * g.Zs;
    gather_co1_warp_kernel<T, K, S><<<(int)((total * 32 + 127) / 128), 128, 0, st>>>(g, big, wp, bias, small, total);
    CG_LAUNCH_CHECK("conv_gather(generic, Cout=1, warp per output)");
    return 0;
  }
  if (g.Cs == 1 && g.Cb % 8 == 0 && (reinterpret_cast<uintptr_t>(big) & 15) == 0 && (reinterpret_cast<uintptr_t>(wp) & 15) == 0) {
    constexpr int VB1 = 8;
    const int64_t total = (int64_t)g.B * g.Xs * g.Ys * ((g.Zs + VB1 - 1) / VB1);
    gather_co1_kernel<T, K, S, VB1><<<(int)((total + 127) / 128), 128, 0, st>>>(g, big, wp, bias, small);
    CG_LAUNCH_CHECK("conv_gather(generic, Cout=1)");
    return 0;
  }
  auto go = [&](auto cob_tag) {
    constexpr int COB = decltype(cob_tag)::value;
    int64_t total = (int64_t)g.B * g.Xs * g.Ys * nzg * (g.Cs / COB);
    int blocks = (int)((total + 127) / 128);
    gather_kernel<T, K, S, COB, VB><<<blocks, 128, 0, st>>>(g, big, wp, bias, small);
  };
  if (g.Cs % 8 == 0) go(std::integral_constant<int, 8>{});
  else if (g.Cs % 4 == 0) go(std::integral_constant<int, 4>{});
  else if (g.Cs % 2 == 0) go(std::integral_constant<int, 2>{});
  else go(std::integral_constant<int, 1>{});
  CG_LAUNCH_CHECK("conv_gather(generic)");
  return 0;
}

// ------------------------------------------------------------------ scatter (dgrad / convT fprop)
// one thread: one big-side voxel x CIB channels
template <typename T, int K, int S, int CIB>
__global__ void __launch_bounds__(128)
scatter_kernel(cgan3d_conv_geom g, const T *__restrict__ small, const T *__restrict__ wp,
               const float *__restrict__ bias, T *__restrict__ big) {
  const int ncib = g.Cb / CIB;
  const int64_t total = (int64_t)g.B * g.Xb * g.Yb * g.Zb * ncib;
  int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int cib = (int)(idx % ncib); idx /= ncib;
  const int iz = (int)(idx % g.Zb); idx /= g.Zb;
  const int iy = (int)(idx % g.Yb); idx /= g.Yb;
  const int ix = (int)(idx % g.Xb);
  const int b = (int)(idx / g.Xb);
  const int ci0 = cib * CIB;
  float acc[CIB];
#pragma unroll
  for (int c = 0; c < CIB; ++c) acc[c] = bias ? bias[ci0 + c] : 0.f;
  for (int kx = 0; kx < K; ++kx) {
    const int tx = ix + g.pad - kx;
    if (tx < 0 || (tx % S) != 0) continue;
    const int ox = tx / S;
    if (ox >= g.Xs) continue;
    for (int ky = 0; ky < K; ++ky) {
      const int ty = iy + g.pad - ky;
      if (ty < 0 || (ty % S) != 0) continue;
      const int oy = ty / S;
      if (oy >= g.Ys) continue;
      for (int kz = 0; kz < K; ++kz) {
        const int tz = iz + g.pad - kz;
        if (tz < 0 || (tz % S) != 0) continue;
        const int oz = tz / S;
        if (oz >= g.Zs) continue;
        const T *yrow = small + ((((int64_t)b * g.Xs + ox) * g.Ys + oy) * g.Zs + oz) * (int64_t)g.Cs;
        const T *wrow = wp + ((int64_t)((kx * K + ky) * K + kz) * g.Cb + ci0) * g.Cs;
        for (int co = 0; co < g.Cs; ++co) {
          const float yv = to_f(yrow[co]);
#pragma unroll
          for (int c = 0; c < CIB; ++c) acc[c] = fmaf(yv, to_f(wrow[(int64_t)c * g.Cs + co]), acc[c]);
        }
      }
    }
  }
  T *o = big + ((((int64_t)b * g.Xb + ix) * g.Yb + iy) * g.Zb + iz) * (int64_t)g.Cb + ci0;
#pragma unroll
  for (int c = 0; c < CIB; ++c) o[c] = from_f<T>(acc[c]);
}


// ------------------------------------------------------------------ scatter, strided (transposed conv / dgrad of a strided conv)
// one thread: one big-side voxel x CIB channels; filter pre-transposed to [tap][Cs][Cb] so that the CIB weights of
// one (tap, cs) are one contiguous vector load and the small-side value is a warp-broadcast scalar.
template <typename T, int K, int S, int CIB>
__global__ void __launch_bounds__(128)
scatter_tw_kernel(cgan3d_conv_geom g, const T *__restrict__ small, const T *__restrict__ wt, const float *__restrict__ bias,
                  T *__restrict__ big) {
  const int ncib = g.Cb / CIB;
  const int64_t total = (int64_t)g.B * g.Xb * g.Yb * g.Zb * ncib;
  int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int cib = (int)(idx % ncib); idx /= ncib;
  const int iz = (int)(idx % g.Zb); idx /= g.Zb;
  const int iy = (int)(idx % g.Yb); idx /= g.Yb;
  const int ix = (int)(idx % g.Xb);
  const int b = (int)(idx / g.Xb);
  const int ci0 = cib * CIB;
  float acc[CIB];
#pragma unroll
  for (int c = 0; c < CIB; ++c) acc[c] = bias ? bias[ci0 + c] : 0.f;
  for (int kx = 0; kx < K; ++kx) {
    const int tx = ix + g.pad - kx;
    if (tx < 0 || (tx % S) != 0) continue;
    const int ox = tx / S;
    if (ox >= g.Xs) continue;
    for (int ky = 0; ky < K; ++ky) {
      const int ty = iy + g.pad - ky;
      if (ty < 0 || (ty % S) != 0) continue;
      const int oy = ty / S;
      if (oy >= g.Ys) continue;
      for (int kz = 0; kz < K; ++kz) {
        const int tz = iz + g.pad - kz;
        if (tz < 0 || (tz % S) != 0) continue;
        const int oz = tz / S;
        if (oz >= g.Zs) continue;
        const T *yrow = small + ((((int64_t)b * g.Xs + ox) * g.Ys + oy) * g.Zs + oz) * (int64_t)g.Cs;
        const T *wrow = wt + (int64_t)((kx * K + ky) * K + kz) * g.Cs * g.Cb + ci0;
#pragma unroll 4
        for (int co = 0; co < g.Cs; ++co) {
          const float yv = to_f(yrow[co]);
          Vec8<T> w;
          w.load(wrow + (int64_t)co * g.Cb);
#pragma unroll
          for (int c = 0; c < CIB; ++c) acc[c] = fmaf(yv, w.v[c], acc[c]);
        }
      }
    }
  }
  T *o = big + ((((int64_t)b * g.Xb + ix) * g.Yb + iy) * g.Zb + iz) * (int64_t)g.Cb + ci0;
#pragma unroll
  for (int c = 0; c < CIB; ++c) o[c] = from_f<T>(acc[c]);
}

// [tap][Cb][Cs] -> [tap][Cs][Cb]
template <typename T>
__global__ void transpose_w_kernel(const T *__restrict__ wp, T *__restrict__ wt, int Cb, int Cs, int taps) {
  const int64_t total = (int64_t)taps * Cb * Cs;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cb = (int)(i % Cb);
    const int cs = (int)((i / Cb) % Cs);
    const int t = (int)(i / ((int64_t)Cb * Cs));
    wt[i] = wp[((int64_t)t * Cb + cb) * Cs + cs];
  }
}

template <typename T, int K, int S>
static int launch_scatter_tw(const cgan3d_conv_geom &g, const T *small, const T *wp, const float *bias, T *big, T *ws,
                             cudaStream_t st) {
  const int taps = K * K * K;
  const int64_t nw = (int64_t)taps * g.Cb * g.Cs;
  transpose_w_kernel<T><<<(int)mn<int64_t>((nw + 255) / 256, 1024), 256, 0, st>>>(wp, ws, g.Cb, g.Cs, taps);
  CG_LAUNCH_CHECK("transpose_w");
  const int64_t total = (int64_t)g.B * g.Xb * g.Yb * g.Zb * (g.Cb / 8);
  scatter_tw_kernel<T, K, S, 8><<<(int)((total + 127) / 128), 128, 0, st>>>(g, small, ws, bias, big);
  CG_LAUNCH_CHECK("conv_scatter(generic, transposed filter)");
  return 0;
}

template <typename T, int K, int S>
static int launch_scatter(const cgan3d_conv_geom &g, const T *small, const T *wp, const float *bias, T *big,
                          cudaStream_t st) {
  auto go = [&](auto tag) {
    constexpr int CIB = decltype(tag)::value;
    int64_t total = (int64_t)g.B * g.Xb * g.Yb * g.Zb * (g.Cb / CIB);
    int blocks = (int)((total + 127) / 128);
    scatter_kernel<T, K, S, CIB><<<blocks, 128, 0, st>>>(g, small, wp, bias, big);
  };
  if (g.Cb % 4 == 0) go(std::integral_constant<int, 4>{});
  else if (g.Cb % 2 == 0) go(std::integral_constant<int, 2>{});
  else go(std::integral_constant<int, 1>{});
  CG_LAUNCH_CHECK("conv_scatter(generic)");
  return 0;
}

// N consecutive channels as floats; N == 4 uses one 16 B (fp32) / 8 B (bf16) load (callers guarantee alignment: C % 4 == 0)
template <typename T, int N>
__device__ __forceinline__ void load_n(const T *p, float (&v)[N]) {
  if constexpr (N == 4 && sizeof(T) == 4) {
    const float4 a = *reinterpret_cast<const float4 *>(p);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  } else if constexpr (N == 4 && sizeof(T) == 2) {
    const uint2 a = *reinterpret_cast<const uint2 *>(p);
    v[0] = __uint_as_float(a.x << 16); v[1] = __uint_as_float(a.x & 0xffff0000u);
    v[2] = __uint_as_float(a.y << 16); v[3] = __uint_as_float(a.y & 0xffff0000u);
  } else if constexpr (N == 8) {
    Vec8<T> t;
    t.load(p);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = t.v[i];
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = to_f(p[i]);
  }
}

// ------------------------------------------------------------------ wgrad
// grid (taps, chunks); block 256 threads = lanes x (ncb x ncs) output sub-tiles of 4x4 (or 1-wide)
template <typename T, int K, int S, int CBV, int CSV>
__global__ void __launch_bounds__(256)
wgrad_kernel(cgan3d_conv_geom g, const T *__restrict__ big, const T *__restrict__ small, float *__restrict__ dw,
             int64_t vox_per_chunk, int cb_base, int cs_base, int ncb, int ncs) {
  extern __shared__ float red[];  // [ncb*CBV][ncs*CSV]
  const int tap = blockIdx.x;
  const int kz = tap % K, ky = (tap / K) % K, kx = tap / (K * K);
  const int per_lane = ncb * ncs;
  const int lanes = blockDim.x / per_lane;
  const int lane = threadIdx.x / per_lane;
  const int r = threadIdx.x % per_lane;
  const int tcb = r / ncs, tcs = r % ncs;
  const int cb0 = cb_base + tcb * CBV, cs0 = cs_base + tcs * CSV;
  const int tile_elems = ncb * CBV * ncs * CSV;
  for (int i = threadIdx.x; i < tile_elems; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  float acc[CBV][CSV];
#pragma unroll
  for (int a = 0; a < CBV; ++a)
#pragma unroll
    for (int c = 0; c < CSV; ++c) acc[a][c] = 0.f;
  // a chunk is a range of output lines (b, ox, oy); lanes stride over z inside a line, so the index decomposition
  // (integer divisions) happens once per line instead of once per voxel
  const int64_t n_lines = (int64_t)g.B * g.Xs * g.Ys;
  const int64_t l0 = blockIdx.y * vox_per_chunk;
  const int64_t l1 = min(n_lines, l0 + vox_per_chunk);
  if (lane < lanes && 2 * g.Zs <= lanes) {
    // short output lines (the critic's 7^3 logits map: 7 voxels per line against 16 lanes): lanes stride over the chunk's
    // voxels instead of idling inside one line, the index arithmetic per voxel is cheap next to a 44-deep serial line loop
    for (int64_t v = l0 * g.Zs + lane; v < l1 * g.Zs; v += lanes) {
      const int64_t l = v / g.Zs;
      const int oz = (int)(v - l * g.Zs);
      const int oy = (int)(l % g.Ys);
      const int64_t t = l / g.Ys;
      const int ox = (int)(t % g.Xs);
      const int b = (int)(t / g.Xs);
      const int ix = ox * S - g.pad + kx, iy = oy * S - g.pad + ky, iz = oz * S - g.pad + kz;
      if ((unsigned)ix >= (unsigned)g.Xb || (unsigned)iy >= (unsigned)g.Yb || (unsigned)iz >= (unsigned)g.Zb) continue;
      float xv[CBV], yv[CSV];
      load_n<T, CBV>(big + ((((int64_t)b * g.Xb + ix) * g.Yb + iy) * (int64_t)g.Zb + iz) * g.Cb + cb0, xv);
      load_n<T, CSV>(small + v * (int64_t)g.Cs + cs0, yv);
#pragma unroll
      for (int a = 0; a < CBV; ++a)
#pragma unroll
        for (int c = 0; c < CSV; ++c) acc[a][c] = fmaf(xv[a], yv[c], acc[a][c]);
    }
#pragma unroll
    for (int a = 0; a < CBV; ++a)
#pragma unroll
      for (int c = 0; c < CSV; ++c)
        atomicAdd(&red[(tcb * CBV + a) * (ncs * CSV) + tcs * CSV + c], acc[a][c]);
  } else if (lane < lanes) {
    for (int64_t l = l0; l < l1; ++l) {
      const int oy = (int)(l % g.Ys);
      const int64_t t = l / g.Ys;
      const int ox = (int)(t % g.Xs);
      const int b = (int)(t / g.Xs);
      const int ix = ox * S - g.pad + kx, iy = oy * S - g.pad + ky;
      if ((unsigned)ix >= (unsigned)g.Xb || (unsigned)iy >= (unsigned)g.Yb) continue;
      const T *xline = big + (((int64_t)b * g.Xb + ix) * g.Yb + iy) * (int64_t)g.Zb * g.Cb + cb0;
      const T *yline = small + l * (int64_t)g.Zs * g.Cs + cs0;
      for (int oz = lane; oz < g.Zs; oz += lanes) {
        const int iz = oz * S - g.pad + kz;
        if ((unsigned)iz >= (unsigned)g.Zb) continue;
        float xv[CBV], yv[CSV];
        load_n<T, CBV>(xline + (int64_t)iz * g.Cb, xv);
        load_n<T, CSV>(yline + (int64_t)oz * g.Cs, yv);
#pragma unroll
        for (int a = 0; a < CBV; ++a)
#pragma unroll
          for (int c = 0; c < CSV; ++c) acc[a][c] = fmaf(xv[a], yv[c], acc[a][c]);
      }
    }
#pragma unroll
    for (int a = 0; a < CBV; ++a)
#pragma unroll
      for (int c = 0; c < CSV; ++c)
        atomicAdd(&red[(tcb * CBV + a) * (ncs * CSV) + tcs * CSV + c], acc[a][c]);
  }
  __syncthreads();
  const int taps = K * K * K;
  for (int i = threadIdx.x; i < tile_elems; i += blockDim.x) {
    const int a = i / (ncs * CSV), c = i % (ncs * CSV);
    atomicAdd(&dw[((int64_t)(cs_base + c) * g.Cb + (cb_base + a)) * taps + tap], red[i]);
  }
}


// ------------------------------------------------------------------ wgrad, thin side (Cb == 1 or Cs == 1), stride 1
// The 7^3 first / last convolutions of the generator (343 taps x C channels of output, K = all voxels).
// One thread owns (dy, c) and all K*K (dx, dz) taps as register accumulators; a block walks output tiles
// (YT lines x ZT voxels), stages the input halo lines of one dx plane and the dY tile in shared memory (fp32) and
// slides a K-wide register window along z: per z step 2 LDS feed K FMAs.  Partial sums of all tiles a block
// processes stay in registers; one atomicAdd per (block, output) at the end.
template <typename T, int K, int S, int C, bool BIG_MULTI>
__global__ void __launch_bounds__(((K * C + 31) / 32) * 32)
wgrad_thin_kernel(cgan3d_conv_geom g, const T *__restrict__ big, const T *__restrict__ small, float *__restrict__ dw) {
  constexpr int YT = 4, ZT = S == 1 ? 64 : 32;
  constexpr int CX = BIG_MULTI ? C : 1, CY = BIG_MULTI ? 1 : C;
  constexpr int ZH = (ZT - 1) * S + K, YH = (YT - 1) * S + K;
  extern __shared__ float sm[];
  float *xs = sm;                      // [YH][ZH][CX]
  float *dys = sm + YH * ZH * CX;      // [YT][ZT][CY]
  const int tid = threadIdx.x;
  const bool active = tid < K * C;
  const int c = tid % C, dy = tid / C;
  float acc[K][K];
#pragma unroll
  for (int a = 0; a < K; ++a)
#pragma unroll
    for (int d = 0; d < K; ++d) acc[a][d] = 0.f;
  const int nyt = (g.Ys + YT - 1) / YT, nzt = (g.Zs + ZT - 1) / ZT;
  const int64_t ntiles = (int64_t)g.B * g.Xs * nyt * nzt;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    int64_t t = tile;
    const int zt = (int)(t % nzt); t /= nzt;
    const int yt = (int)(t % nyt); t /= nyt;
    const int ox = (int)(t % g.Xs);
    const int b = (int)(t / g.Xs);
    const int oy0 = yt * YT, oz0 = zt * ZT;
    __syncthreads();
    for (int i = tid; i < YT * ZT * CY; i += blockDim.x) {
      const int cc = i % CY, z = (i / CY) % ZT, y = i / (CY * ZT);
      const int oy = oy0 + y, oz = oz0 + z;
      float v = 0.f;
      if (oy < g.Ys && oz < g.Zs) v = to_f(small[((((int64_t)b * g.Xs + ox) * g.Ys + oy) * g.Zs + oz) * CY + cc]);
      dys[i] = v;
    }
#pragma unroll 1
    for (int dx = 0; dx < K; ++dx) {
      const int ix = ox * S - g.pad + dx;
      __syncthreads();
      if constexpr (CX % 8 == 0) {  // 8 channels (16 B of bf16 / 32 B of fp32) per load
        for (int i = tid; i < YH * ZH * (CX / 8); i += blockDim.x) {
          const int c8 = i % (CX / 8), z = (i / (CX / 8)) % ZH, y = i / ((CX / 8) * ZH);
          const int iy = oy0 * S - g.pad + y, iz = oz0 * S - g.pad + z;
          Vec8<T> v;
#pragma unroll
          for (int k = 0; k < 8; ++k) v.v[k] = 0.f;
          if ((unsigned)ix < (unsigned)g.Xb && (unsigned)iy < (unsigned)g.Yb && (unsigned)iz < (unsigned)g.Zb)
            v.load(big + ((((int64_t)b * g.Xb + ix) * g.Yb + iy) * g.Zb + iz) * CX + c8 * 8);
          float4 *d = reinterpret_cast<float4 *>(xs + (y * ZH + z) * CX + c8 * 8);
          d[0] = make_float4(v.v[0], v.v[1], v.v[2], v.v[3]);
          d[1] = make_float4(v.v[4], v.v[5], v.v[6], v.v[7]);
        }
      } else {
        for (int i = tid; i < YH * ZH * CX; i += blockDim.x) {
          const int cc = i % CX, z = (i / CX) % ZH, y = i / (CX * ZH);
          const int iy = oy0 * S - g.pad + y, iz = oz0 * S - g.pad + z;
          float v = 0.f;
          if ((unsigned)ix < (unsigned)g.Xb && (unsigned)iy < (unsigned)g.Yb && (unsigned)iz < (unsigned)g.Zb)
            v = to_f(big[((((int64_t)b * g.Xb + ix) * g.Yb + iy) * g.Zb + iz) * CX + cc]);
          xs[i] = v;
        }
      }
      __syncthreads();
      if (active) {
        float a[K];
#pragma unroll
        for (int d = 0; d < K; ++d) a[d] = 0.f;
#pragma unroll 1
        for (int y = 0; y < YT; ++y) {
          const float *xl = xs + ((y * S + dy) * ZH) * CX + (BIG_MULTI ? c : 0);
          const float *dl = dys + (y * ZT) * CY + (BIG_MULTI ? 0 : c);
          float w[K];
#pragma unroll
          for (int d = 0; d < K - S; ++d) w[d] = xl[d * CX];
#pragma unroll 7
          for (int z = 0; z < ZT; ++z) {
#pragma unroll
            for (int q = 0; q < S; ++q) w[K - S + q] = xl[(z * S + K - S + q) * CX];
            const float dv = dl[z * CY];
#pragma unroll
            for (int d = 0; d < K; ++d) a[d] = fmaf(w[d], dv, a[d]);
#pragma unroll
            for (int d = 0; d < K - S; ++d) w[d] = w[d + S];
          }
        }
        // fold this plane's sums into the dx-indexed accumulators without dynamic register indexing
#pragma unroll
        for (int q = 0; q < K; ++q)
          if (q == dx) {
#pragma unroll
            for (int d = 0; d < K; ++d) acc[q][d] += a[d];
          }
      }
    }
  }
  if (active) {
    constexpr int taps = K * K * K;
#pragma unroll
    for (int dx = 0; dx < K; ++dx)
#pragma unroll
      for (int dz = 0; dz < K; ++dz) atomicAdd(&dw[(int64_t)c * taps + (dx * K + dy) * K + dz], acc[dx][dz]);
  }
}

template <typename T, int K, int S, int C, bool BIG_MULTI>
static int launch_wgrad_thin(const cgan3d_conv_geom &g, const T *big, const T *small, float *dw, cudaStream_t st) {
  constexpr int YT = 4, ZT = S == 1 ? 64 : 32, CX = BIG_MULTI ? C : 1, CY = BIG_MULTI ? 1 : C;
  constexpr int threads = ((K * C + 31) / 32) * 32;
  const size_t smem = ((size_t)((YT - 1) * S + K) * ((ZT - 1) * S + K) * CX + (size_t)YT * ZT * CY) * sizeof(float);
  auto kern = wgrad_thin_kernel<T, K, S, C, BIG_MULTI>;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(wgrad_thin)");
    attr = true;
  }
  const int per_sm = (int)mx<size_t>(1, mn<size_t>(6, (size_t)200000 / (smem + 1024)));
  const int64_t ntiles = (int64_t)g.B * g.Xs * ((g.Ys + YT - 1) / YT) * ((g.Zs + ZT - 1) / ZT);
  const int grid = (int)mn<int64_t>(ntiles, (int64_t)num_sms() * per_sm);
  kern<<<grid, threads, smem, st>>>(g, big, small, dw);
  CG_LAUNCH_CHECK("conv_wgrad(thin)");
  return 0;
}

template <typename T, int K, int S>
static int launch_wgrad(const cgan3d_conv_geom &g, const T *big, const T *small, float *dw, float beta,
                        cudaStream_t st) {
  const int taps = K * K * K;
  const int64_t n_w = (int64_t)g.Cs * g.Cb * taps;
  if (beta == 0.f) {
    cudaError_t e = cudaMemsetAsync(dw, 0, n_w * sizeof(float), st);
    if (e != cudaSuccess) return cuda_fail(e, "conv_wgrad memset");
  }
  if constexpr (K >= 4) {
    if (g.Cb == 1 && g.Cs == 16) return launch_wgrad_thin<T, K, S, 16, false>(g, big, small, dw, st);
    if (g.Cb == 16 && g.Cs == 1) return launch_wgrad_thin<T, K, S, 16, true>(g, big, small, dw, st);
    if (g.Cb == 1 && g.Cs == 8) return launch_wgrad_thin<T, K, S, 8, false>(g, big, small, dw, st);
    if (g.Cb == 8 && g.Cs == 1) return launch_wgrad_thin<T, K, S, 8, true>(g, big, small, dw, st);
  }
  const int64_t n_lines = (int64_t)g.B * g.Xs * g.Ys;
  int chunks = (int)mn<int64_t>(mx<int64_t>(1, (int64_t)num_sms() * 8 / taps), n_lines);
  chunks = min(chunks, 65535);
  const int64_t vpc = (n_lines + chunks - 1) / chunks;  // lines per chunk
  auto go = [&](auto tcb_tag, auto tcs_tag) {
    constexpr int CBV = decltype(tcb_tag)::value;
    constexpr int CSV = decltype(tcs_tag)::value;
    // tile the (Cb, Cs) plane so that one voxel lane needs at most 16 x 16 threads
    constexpr int TB = 16 * CBV, TS = 16 * CSV;
    for (int cb_base = 0; cb_base < g.Cb; cb_base += TB)
      for (int cs_base = 0; cs_base < g.Cs; cs_base += TS) {
        const int ncb = min(TB, g.Cb - cb_base) / CBV, ncs = min(TS, g.Cs - cs_base) / CSV;
        const size_t smem = (size_t)ncb * CBV * ncs * CSV * sizeof(float);
        wgrad_kernel<T, K, S, CBV, CSV><<<dim3(taps, chunks), 256, smem, st>>>(g, big, small, dw, vpc, cb_base,
                                                                               cs_base, ncb, ncs);
      }
  };
  const bool b4 = g.Cb % 4 == 0, s4 = g.Cs % 4 == 0;
  const bool al16 = (reinterpret_cast<uintptr_t>(big) & 15) == 0 && (reinterpret_cast<uintptr_t>(small) & 15) == 0;
  if (g.Cb % 8 == 0 && g.Cs % 8 == 0 && al16) go(std::integral_constant<int, 8>{}, std::integral_constant<int, 8>{});
  else if (b4 && s4) go(std::integral_constant<int, 4>{}, std::integral_constant<int, 4>{});
  else if (b4) go(std::integral_constant<int, 4>{}, std::integral_constant<int, 1>{});
  else if (s4) go(std::integral_constant<int, 1>{}, std::integral_constant<int, 4>{});
  else go(std::integral_constant<int, 1>{}, std::integral_constant<int, 1>{});
  CG_LAUNCH_CHECK("conv_wgrad(generic)");
  return 0;
}

// ------------------------------------------------------------------ dispatch on (k, stride, dtype)
#define CG_KS_DISPATCH(FN, ...)                                                       \
  do {                                                                                \
    const int ks = g.k * 10 + g.stride;                                               \
    switch (ks) {                                                                     \
      case 11: return FN<T, 1, 1>(__VA_ARGS__);                                       \
      case 31: return FN<T, 3, 1>(__VA_ARGS__);                                       \
      case 32: return FN<T, 3, 2>(__VA_ARGS__);                                       \
      case 41: return FN<T, 4, 1>(__VA_ARGS__);                                       \
      case 42: return FN<T, 4, 2>(__VA_ARGS__);                                       \
      case 51: return FN<T, 5, 1>(__VA_ARGS__);                                       \
      case 71: return FN<T, 7, 1>(__VA_ARGS__);                                       \
      default: return fail(CGAN3D_E_UNSUPPORTED, "generic conv: k=%d stride=%d not built", g.k, g.stride); \
    }                                                                                 \
  } while (0)

int generic_gather(const cgan3d_conv_geom &g, int dtype, const void *big, const void *wp, const float *bias,
                   void *small, cudaStream_t st) {
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    CG_KS_DISPATCH(launch_gather, g, (const T *)big, (const T *)wp, bias, (T *)small, st);
  });
}
// [tap][Cb][Cs] -> [taps-1-tap][Cs][Cb]
template <typename T>
__global__ void flip_transpose_kernel(const T *__restrict__ wp, T *__restrict__ wf, int Cb, int Cs, int taps) {
  const int64_t total = (int64_t)taps * Cb * Cs;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cb = (int)(i % Cb);
    const int cs = (int)((i / Cb) % Cs);
    const int t = (int)(i / ((int64_t)Cb * Cs));
    wf[i] = wp[((int64_t)(taps - 1 - t) * Cb + cb) * Cs + cs];
  }
}

size_t generic_workspace_bytes(const cgan3d_conv_geom &g, int dtype, int op) {
  if (op == 1) return (size_t)g.k * g.k * g.k * g.Cb * g.Cs * (dtype == CGAN3D_F32 ? 4 : 2) + 16;
  return 0;
}

int generic_scatter(const cgan3d_conv_geom &g, int dtype, const void *small, const void *wp, const float *bias,
                    void *big, void *ws, size_t ws_bytes, cudaStream_t st) {
  const bool ws_ok = ws != nullptr && ws_bytes >= generic_workspace_bytes(g, dtype, 1) && (reinterpret_cast<uintptr_t>(ws) & 15) == 0;
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    if (g.stride == 1 && ws_ok) {
      // dgrad of a stride-1 conv == conv of the small side with the flipped filter, pad' = k-1-pad (register-tiled gather)
      const int taps = g.k * g.k * g.k;
      const int64_t total = (int64_t)taps * g.Cb * g.Cs;
      const int blocks = (int)mn<int64_t>((total + 255) / 256, 1024);
      flip_transpose_kernel<T><<<blocks, 256, 0, st>>>((const T *)wp, (T *)ws, g.Cb, g.Cs, taps);
      CG_LAUNCH_CHECK("flip_transpose");
      cgan3d_conv_geom f = g;
      f.Xb = g.Xs; f.Yb = g.Ys; f.Zb = g.Zs; f.Cb = g.Cs;
      f.Xs = g.Xb; f.Ys = g.Yb; f.Zs = g.Zb; f.Cs = g.Cb;
      f.pad = g.k - 1 - g.pad;
      return generic_gather(f, dtype, small, ws, bias, big, st);
    }
    if (g.stride > 1 && g.Cb % 8 == 0 && ws_ok)
      CG_KS_DISPATCH(launch_scatter_tw, g, (const T *)small, (const T *)wp, bias, (T *)big, (T *)ws, st);
    CG_KS_DISPATCH(launch_scatter, g, (const T *)small, (const T *)wp, bias, (T *)big, st);
  });
}
int generic_wgrad(const cgan3d_conv_geom &g, int dtype, const void *big, const void *small, float *dw, float beta,
                  cudaStream_t st) {
  return with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    CG_KS_DISPATCH(launch_wgrad, g, (const T *)big, (const T *)small, dw, beta, st);
  });
}

int pack_weights(const float *w, void *packed, int dtype, int Cs, int Cb, int k, cudaStream_t st) {
  const int taps = k * k * k;
  const int64_t total = (int64_t)taps * Cb * Cs;
  const int blocks = (int)mn<int64_t>((total + 255) / 256, 4096);
  with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    pack_weights_kernel<T><<<blocks, 256, 0, st>>>(w, (T *)packed, Cs, Cb, taps);
  });
  CG_LAUNCH_CHECK("pack_weights");
  return 0;
}

// ------------------------------------------------------------------ reflect padding
__device__ __forceinline__ int reflect_idx(int j, int n) {  // j in [-p, n+p), p < n
  if (j < 0) j = -j;
  if (j >= n) j = 2 * (n - 1) - j;
  return j;
}

template <typename T>
__global__ void reflect_pad_kernel(const T *__restrict__ in, T *__restrict__ out, int B, int X, int Y, int Z, int C,
                                   int p) {
  const int Xp = X + 2 * p, Yp = Y + 2 * p, Zp = Z + 2 * p;
  const int64_t total = (int64_t)B * Xp * Yp * Zp * C;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t t = i;
    const int c = (int)(t % C); t /= C;
    const int z = (int)(t % Zp); t /= Zp;
    const int y = (int)(t % Yp); t /= Yp;
    const int x = (int)(t % Xp);
    const int b = (int)(t / Xp);
    const int sx = reflect_idx(x - p, X), sy = reflect_idx(y - p, Y), sz = reflect_idx(z - p, Z);
    out[i] = in[((((int64_t)b * X + sx) * Y + sy) * Z + sz) * C + c];
  }
}

// sources in padded coordinates that mirror onto interior index i (at most 3 per axis)
__device__ __forceinline__ int reflect_sources(int i, int n, int p, int src[3]) {
  int cnt = 0;
  src[cnt++] = i + p;
  if (i >= 1 && i <= p) src[cnt++] = p - i;
  if (i <= n - 2 && i >= n - 1 - p) src[cnt++] = p + 2 * (n - 1) - i;
  return cnt;
}

template <typename T>
__global__ void reflect_pad_bwd_kernel(const T *__restrict__ gp, T *__restrict__ gi, int B, int X, int Y, int Z,
                                       int C, int p) {
  const int Yp = Y + 2 * p, Zp = Z + 2 * p, Xp = X + 2 * p;
  const int64_t total = (int64_t)B * X * Y * Z * C;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t t = i;
    const int c = (int)(t % C); t /= C;
    const int z = (int)(t % Z); t /= Z;
    const int y = (int)(t % Y); t /= Y;
    const int x = (int)(t % X);
    const int b = (int)(t / X);
    int sx[3], sy[3], sz[3];
    const int nx = reflect_sources(x, X, p, sx), ny = reflect_sources(y, Y, p, sy), nz = reflect_sources(z, Z, p, sz);
    float acc = 0.f;
    for (int a = 0; a < nx; ++a)
      for (int bb = 0; bb < ny; ++bb)
        for (int cc = 0; cc < nz; ++cc)
          acc += to_f(gp[((((int64_t)b * Xp + sx[a]) * Yp + sy[bb]) * Zp + sz[cc]) * C + c]);
    gi[i] = from_f<T>(acc);
  }
}

// One block per padded (b, x, y) line: the mirrored x / y sources are block-uniform, a thread only mirrors z.
// U = unit moved per thread: uint4 (16-byte chunks, C * sizeof(T) % 16 == 0) or the scalar element type.
template <typename U>
__global__ void __launch_bounds__(256)
reflect_pad_line_kernel(const U *__restrict__ in, U *__restrict__ out, int X, int Y, int Z, int upv, int p) {
  const int Yp = Y + 2 * p, Zp = Z + 2 * p, Xp = X + 2 * p;
  const int y = blockIdx.x, x = blockIdx.y, b = blockIdx.z;
  const int sx = reflect_idx(x - p, X), sy = reflect_idx(y - p, Y);
  const U *src = in + (((int64_t)b * X + sx) * Y + sy) * (int64_t)Z * upv;
  U *dst = out + (((int64_t)b * Xp + x) * Yp + y) * (int64_t)Zp * upv;
  for (int i = threadIdx.x; i < Zp * upv; i += blockDim.x) {
    const int z = i / upv, c = i - z * upv;
    dst[i] = src[reflect_idx(z - p, Z) * upv + c];
  }
}

// Short lines (the generator's 1-channel input: 134 two-byte elements per padded line): a block per line is 290 000 blocks
// of half-idle threads, 0.20 ms for 150 MB.  Here a WARP owns a line and a block walks 32 lines of one padded (b, x) plane.
template <typename U>
__global__ void __launch_bounds__(256)
reflect_pad_warpline_kernel(const U *__restrict__ in, U *__restrict__ out, int X, int Y, int Z, int upv, int p) {
  const int Yp = Y + 2 * p, Zp = Z + 2 * p, Xp = X + 2 * p;
  const int x = blockIdx.y, b = blockIdx.z, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sx = reflect_idx(x - p, X);
  const int n = Zp * upv;
  for (int k = 0; k < 4; ++k) {
    const int y = (blockIdx.x * 4 + k) * 8 + warp;
    if (y >= Yp) break;
    const int sy = reflect_idx(y - p, Y);
    const U *src = in + (((int64_t)b * X + sx) * Y + sy) * (int64_t)Z * upv;
    U *dst = out + (((int64_t)b * Xp + x) * Yp + y) * (int64_t)Zp * upv;
    for (int i = lane; i < n; i += 32) {
      const int z = i / upv, c = i - z * upv;
      dst[i] = src[reflect_idx(z - p, Z) * upv + c];
    }
  }
}

// one block per interior (b, x, y) line: no per-element index division, the mirror sources of x and y are block-uniform
template <typename T>
__global__ void __launch_bounds__(256)
reflect_pad_bwd_vec_kernel(const uint4 *__restrict__ gp, uint4 *__restrict__ gi, int B, int X, int Y, int Z, int cpv, int p, int lpb) {
  constexpr int VEC = 16 / (int)sizeof(T);
  const int Yp = Y + 2 * p, Zp = Z + 2 * p, Xp = X + 2 * p;
  const int x = blockIdx.y, b = blockIdx.z;
  int sx[3];
  const int nx = reflect_sources(x, X, p, sx);
  // lpb lines per block: a line of 128 voxels x 16 channels is ONE 16-byte chunk per thread, too little in flight
  for (int y = blockIdx.x * lpb; y < min(Y, (int)(blockIdx.x + 1) * lpb); ++y) {
  int sy[3];
  const int ny = reflect_sources(y, Y, p, sy);
  uint4 *dst = gi + (((int64_t)b * X + x) * Y + y) * (int64_t)Z * cpv;
  for (int i = threadIdx.x; i < Z * cpv; i += blockDim.x) {
    const int z = i / cpv, c = i - z * cpv;
    int sz[3];
    const int nz = reflect_sources(z, Z, p, sz);
    if (nx == 1 && ny == 1 && nz == 1) {  // interior voxel: plain copy
      dst[i] = gp[((((int64_t)b * Xp + sx[0]) * Yp + sy[0]) * Zp + sz[0]) * cpv + c];
      continue;
    }
    float acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
    for (int a = 0; a < nx; ++a)
      for (int bb = 0; bb < ny; ++bb)
        for (int cc = 0; cc < nz; ++cc) {
          const uint4 v = gp[((((int64_t)b * Xp + sx[a]) * Yp + sy[bb]) * Zp + sz[cc]) * cpv + c];
          const T *e = reinterpret_cast<const T *>(&v);
#pragma unroll
          for (int k = 0; k < VEC; ++k) acc[k] += to_f(e[k]);
        }
    uint4 o;
    T *e = reinterpret_cast<T *>(&o);
#pragma unroll
    for (int k = 0; k < VEC; ++k) e[k] = from_f<T>(acc[k]);
    dst[i] = o;
  }
  }
}

int reflect_pad(const void *in, void *out, int dtype, int B, int X, int Y, int Z, int C, int pad, cudaStream_t st) {
  const int esz = dtype == CGAN3D_F32 ? 4 : 2;
  const int Xp = X + 2 * pad, Yp = Y + 2 * pad;
  if (Xp <= 65535 && B <= 65535) {
    const dim3 grid((unsigned)Yp, (unsigned)Xp, (unsigned)B);
    if ((C * esz) % 16 == 0 && !((uintptr_t)in & 15) && !((uintptr_t)out & 15))
      reflect_pad_line_kernel<uint4><<<grid, 256, 0, st>>>((const uint4 *)in, (uint4 *)out, X, Y, Z, C * esz / 16, pad);
    else
      with_dtype(dtype, [&](auto t) {
        using T = typename decltype(t)::type;
        if ((Z + 2 * pad) * C <= 512) {  // short lines: a warp per line
          const dim3 gridw((unsigned)((Yp + 31) / 32), (unsigned)Xp, (unsigned)B);
          reflect_pad_warpline_kernel<T><<<gridw, 256, 0, st>>>((const T *)in, (T *)out, X, Y, Z, C, pad);
        } else
          reflect_pad_line_kernel<T><<<grid, 256, 0, st>>>((const T *)in, (T *)out, X, Y, Z, C, pad);
      });
    CG_LAUNCH_CHECK("reflect_pad(line)");
    return 0;
  }
  const int64_t total = (int64_t)B * (X + 2 * pad) * (Y + 2 * pad) * (Z + 2 * pad) * C;
  const int blocks = (int)mn<int64_t>((total + 255) / 256, (int64_t)num_sms() * 16);
  with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    reflect_pad_kernel<T><<<blocks, 256, 0, st>>>((const T *)in, (T *)out, B, X, Y, Z, C, pad);
  });
  CG_LAUNCH_CHECK("reflect_pad");
  return 0;
}

int reflect_pad_backward(const void *gp, void *gi, int dtype, int B, int X, int Y, int Z, int C, int pad,
                         cudaStream_t st) {
  const int esz = dtype == CGAN3D_F32 ? 4 : 2;
  const bool vec = (C * esz) % 16 == 0 && !((uintptr_t)gp & 15) && !((uintptr_t)gi & 15) && X <= 65535 && B <= 65535;
  with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    if (vec) {
      const int cpv = C * esz / 16;
      const int lpb = (int64_t)B * X * Y >= 65536 && Z * cpv <= 512 ? 4 : 1;
      const dim3 bl((unsigned)((Y + lpb - 1) / lpb), (unsigned)X, (unsigned)B);
      reflect_pad_bwd_vec_kernel<T><<<bl, 256, 0, st>>>((const uint4 *)gp, (uint4 *)gi, B, X, Y, Z, cpv, pad, lpb);
    } else {
      const int64_t total = (int64_t)B * X * Y * Z * C;
      const int blocks = (int)mn<int64_t>((total + 255) / 256, (int64_t)num_sms() * 16);
      reflect_pad_bwd_kernel<T><<<blocks, 256, 0, st>>>((const T *)gp, (T *)gi, B, X, Y, Z, C, pad);
    }
  });
  CG_LAUNCH_CHECK(vec ? "reflect_pad_bwd_vec" : "reflect_pad_backward");
  return 0;
}

}  // namespace cg
