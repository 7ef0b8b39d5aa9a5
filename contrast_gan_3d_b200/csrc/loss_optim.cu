// Fused loss reductions (ZNCC + HU in one pass, Wasserstein means), fused Adam(+clip),
// patch sampler / tiler kernels.  All HBM-bound.
// Replaces the ATen reductions behind reference model/loss.py:11-80, torch.optim.Adam +
// clamp_ (trainer/Trainer.py:135-138,157), and the CPU crop/scale of
// data/CCTADataLoader.py:83-92 / eval/CCTAContrastCorrector.py:60-81.
#include "common.cuh"

namespace cg {

// ---------------------------------------------------------------- generator losses
__device__ __forceinline__ float hinge2(float s, float lo, float hi) {
  const float a = fminf(s, lo) - lo, b = fmaxf(s, hi) - hi;
  return a * a + b * b;
}

__global__ void __launch_bounds__(256)
gen_loss_sums_kernel(const float *__restrict__ s, const float *__restrict__ t, const uint8_t *__restrict__ mask,
                     int64_t n, float lo, float hi, double *__restrict__ sums) {
  double tot[7] = {0, 0, 0, 0, 0, 0, 0};
  float part[7] = {0, 0, 0, 0, 0, 0, 0};
  int run = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float a = s[i], b = t[i];
    const float m = mask ? (mask[i] ? 1.f : 0.f) : 0.f;
    part[0] += a; part[1] += b; part[2] += a * a; part[3] += b * b; part[4] += a * b;
    part[5] += hinge2(a, lo, hi) * m; part[6] += m;
    if (++run == 64) {
#pragma unroll
      for (int k = 0; k < 7; ++k) { tot[k] += (double)part[k]; part[k] = 0.f; }
      run = 0;
    }
  }
  __shared__ double sh[7][8];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const double v = warp_sum(tot[k] + (double)part[k]);
    if ((threadIdx.x & 31) == 0) sh[k][threadIdx.x >> 5] = v;
  }
  __syncthreads();
  if (threadIdx.x < 7) {
    double a = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) a += sh[threadIdx.x][w];
    atomicAdd(&sums[threadIdx.x], a);
  }
}

// out[0] = w_sim * zncc, out[1] = w_hu * hu; coef = {mean_s, mean_t, A, Bc, hu_scale, 0,0,0}
__global__ void gen_loss_finalize_kernel(const double *__restrict__ sums, int64_t n, float w_sim, float w_hu,
                                         float *__restrict__ out, float *__restrict__ coef) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double N = (double)n;
  const double ms = sums[0] / N, mt = sums[1] / N;
  const double cc = sums[4] / N - ms * mt;
  double vs = (sums[2] - N * ms * ms) / (N - 1.0), vt = (sums[3] - N * mt * mt) / (N - 1.0);
  if (vs < 0) vs = 0;
  if (vt < 0) vt = 0;
  const double ss = sqrt(vs), st = sqrt(vt);
  const double D = ss * st + 1e-8;
  out[0] = (float)(w_sim * (-(cc / D)));
  const double M = sums[6];
  const double denom = (double)((float)M + 1e-8f);
  out[1] = (float)(w_hu * (sums[5] / denom));
  coef[0] = (float)ms;
  coef[1] = (float)mt;
  coef[2] = (float)(-(double)w_sim / (N * D));
  coef[3] = (float)((double)w_sim * (cc / (D * D)) * st * (2.0 / (N - 1.0)) / (2.0 * ss + 1e-6));
  coef[4] = (float)((double)w_hu / denom);
  coef[5] = coef[6] = coef[7] = 0.f;
}

__global__ void __launch_bounds__(256)
gen_loss_backward_kernel(const float *__restrict__ s, const float *__restrict__ t, const uint8_t *__restrict__ mask,
                         int64_t n, float lo, float hi, const float *__restrict__ coef,
                         const float *__restrict__ upstream, const float *__restrict__ d_extra, float *__restrict__ ds) {
  const float ms = coef[0], mt = coef[1], A = coef[2], Bc = coef[3], hs = coef[4];
  const float up_sim = upstream ? upstream[0] : 1.f, up_hu = upstream ? upstream[1] : 1.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float a = s[i];
    float g = up_sim * (A * (t[i] - mt) + Bc * (a - ms));
    if (mask && mask[i]) {
      if (a < lo) g += up_hu * hs * 2.f * (a - lo);
      else if (a > hi) g += up_hu * hs * 2.f * (a - hi);
    }
    if (d_extra) g += d_extra[i];
    ds[i] = g;
  }
}

// ---------------------------------------------------------------- mean / fill
template <typename T>
__global__ void __launch_bounds__(256) sum_kernel(const T *__restrict__ x, int64_t n, double *__restrict__ out) {
  double tot = 0.0;
  float part = 0.f;
  int run = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    part += to_f(x[i]);
    if (++run == 64) { tot += (double)part; part = 0.f; run = 0; }
  }
  __shared__ double sh[8];
  const double v = warp_sum(tot + (double)part);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) a += sh[w];
    atomicAdd(out, a);
  }
}

__global__ void mean_finalize_kernel(const double *__restrict__ sum, int64_t n, float scale, float *__restrict__ out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) out[0] = (float)((double)scale * sum[0] / (double)n);
}

template <typename T>
__global__ void __launch_bounds__(256) fill_kernel(T *__restrict__ x, int64_t n, const float *__restrict__ v, float scale) {
  const float val = (v ? v[0] : 1.f) * scale;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    x[i] = from_f<T>(val);
}

// ---------------------------------------------------------------- Adam (+ weight clip)
__global__ void __launch_bounds__(256)
adam_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m, float *__restrict__ v, int64_t n,
            float lr, float b1, float b2, float eps, int step, float clip) {
  __shared__ float s_step_size, s_bc2_sqrt;
  if (threadIdx.x == 0) {
    const double bc1 = 1.0 - pow((double)b1, (double)step);
    const double bc2 = 1.0 - pow((double)b2, (double)step);
    s_step_size = (float)((double)lr / bc1);
    s_bc2_sqrt = (float)sqrt(bc2);
  }
  __syncthreads();
  const float step_size = s_step_size, bc2_sqrt = s_bc2_sqrt;
  const float w1 = 1.f - b1, w2 = 1.f - b2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    float mi = m[i];
    // torch lerp_: two-branch formula for accuracy
    mi = (w1 < 0.5f) ? mi + w1 * (gi - mi) : gi - (gi - mi) * (1.f - w1);
    float vi = v[i] * b2;
    vi = vi + (w2 * gi) * gi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    float pi = p[i] + (-step_size) * (mi / denom);
    if (clip > 0.f) pi = fminf(fmaxf(pi, -clip), clip);
    m[i] = mi;
    v[i] = vi;
    p[i] = pi;
  }
}

// multi-tensor variant: one launch updates up to kAdamBatch parameter tensors (blockIdx.y = tensor); the pointer table
// travels in the kernel parameters, so there is no device-side table to upload
constexpr int kAdamBatch = 48;
struct AdamBatch {
  float *p[kAdamBatch];
  const float *g[kAdamBatch];
  float *m[kAdamBatch];
  float *v[kAdamBatch];
  int64_t n[kAdamBatch];
};
__global__ void __launch_bounds__(256)
adam_multi_kernel(const __grid_constant__ AdamBatch t, float lr, float b1, float b2, float eps, int step, float clip) {
  __shared__ float s_step_size, s_bc2_sqrt;
  if (threadIdx.x == 0) {
    const double bc1 = 1.0 - pow((double)b1, (double)step);
    const double bc2 = 1.0 - pow((double)b2, (double)step);
    s_step_size = (float)((double)lr / bc1);
    s_bc2_sqrt = (float)sqrt(bc2);
  }
  __syncthreads();
  const float step_size = s_step_size, bc2_sqrt = s_bc2_sqrt;
  const float w1 = 1.f - b1, w2 = 1.f - b2;
  const int k = blockIdx.y;
  float *__restrict__ p = t.p[k];
  const float *__restrict__ g = t.g[k];
  float *__restrict__ m = t.m[k];
  float *__restrict__ v = t.v[k];
  const int64_t n = t.n[k];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    float mi = m[i];
    mi = (w1 < 0.5f) ? mi + w1 * (gi - mi) : gi - (gi - mi) * (1.f - w1);  // torch lerp_
    float vi = v[i] * b2;
    vi = vi + (w2 * gi) * gi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    float pi = p[i] + (-step_size) * (mi / denom);
    if (clip > 0.f) pi = fminf(fmaxf(pi, -clip), clip);
    m[i] = mi;
    v[i] = vi;
    p[i] = pi;
  }
}

// Capturable variant (CUDA graphs): the learning rate and the step count live in DEVICE memory (hyper[0] = lr, hyper[1] =
// step as a float, exact up to 2^24), so a captured optimizer step stays valid when the scheduler changes the rate and as
// the bias corrections evolve.  adam_tick_kernel advances the step count once per optimizer.step().
__global__ void adam_tick_kernel(float *hyper) {
  if (threadIdx.x == 0 && blockIdx.x == 0) hyper[1] += 1.f;
}
__global__ void __launch_bounds__(256)
adam_multi_dev_kernel(const __grid_constant__ AdamBatch t, const float *__restrict__ hyper, float b1, float b2, float eps, float clip) {
  __shared__ float s_step_size, s_bc2_sqrt;
  if (threadIdx.x == 0) {
    const double lr = (double)hyper[0], step = (double)hyper[1];
    const double bc1 = 1.0 - pow((double)b1, step);
    const double bc2 = 1.0 - pow((double)b2, step);
    s_step_size = (float)(lr / bc1);
    s_bc2_sqrt = (float)sqrt(bc2);
  }
  __syncthreads();
  const float step_size = s_step_size, bc2_sqrt = s_bc2_sqrt;
  const float w1 = 1.f - b1, w2 = 1.f - b2;
  const int k = blockIdx.y;
  float *__restrict__ p = t.p[k];
  const float *__restrict__ g = t.g[k];
  float *__restrict__ m = t.m[k];
  float *__restrict__ v = t.v[k];
  const int64_t n = t.n[k];
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    float mi = m[i];
    mi = (w1 < 0.5f) ? mi + w1 * (gi - mi) : gi - (gi - mi) * (1.f - w1);  // torch lerp_
    float vi = v[i] * b2;
    vi = vi + (w2 * gi) * gi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    float pi = p[i] + (-step_size) * (mi / denom);
    if (clip > 0.f) pi = fminf(fmaxf(pi, -clip), clip);
    m[i] = mi;
    v[i] = vi;
    p[i] = pi;
  }
}

// RMSprop (torch.optim.RMSprop defaults: no momentum, not centered; reference experiments/rmsprop_conf.py:8-9):
// v = alpha v + (1 - alpha) g^2;  p -= lr g / (sqrt(v) + eps)  [+ weight clip].  The AdamBatch table is reused: m is unused.
__global__ void __launch_bounds__(256)
rmsprop_multi_kernel(const __grid_constant__ AdamBatch t, float lr, float alpha, float eps, float clip) {
  const int k = blockIdx.y;
  float *__restrict__ p = t.p[k];
  const float *__restrict__ g = t.g[k];
  float *__restrict__ v = t.v[k];
  const int64_t n = t.n[k];
  const float w = 1.f - alpha;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    float vi = v[i] * alpha;
    vi = vi + (w * gi) * gi;  // torch: square_avg.mul_(alpha).addcmul_(grad, grad, value = 1 - alpha)
    float pi = p[i] + (-lr) * (gi / (sqrtf(vi) + eps));
    if (clip > 0.f) pi = fminf(fmaxf(pi, -clip), clip);
    v[i] = vi;
    p[i] = pi;
  }
}

// ---------------------------------------------------------------- sampler / tiler
__global__ void __launch_bounds__(256)
crop_scale_kernel(const int16_t *__restrict__ vol, int X, int Y, int Z, int lbx, int lby, int lbz, int PX, int PY, int PZ,
                  int px0, int py0, int pz0, float shift, float factor, float *__restrict__ data,
                  uint8_t *__restrict__ mask) {
  const int64_t total = (int64_t)PX * PY * PZ;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int z = (int)(i % PZ), y = (int)((i / PZ) % PY), x = (int)(i / ((int64_t)PZ * PY));
    const int sx = x + lbx - px0, sy = y + lby - py0, sz = z + lbz - pz0;  // padded -> source coordinates
    float hu = 0.f;
    uint8_t mk = 0;
    if ((unsigned)sx < (unsigned)X && (unsigned)sy < (unsigned)Y && (unsigned)sz < (unsigned)Z) {
      const int16_t *q = vol + ((((int64_t)sx * Y + sy) * Z + sz) << 1);
      hu = (float)q[0];
      mk = q[1] != 0;
    }
    data[i] = (hu - shift) / factor;
    if (mask) mask[i] = mk;
  }
}

__global__ void __launch_bounds__(256)
tile_extract_kernel(const int16_t *__restrict__ vol, int X, int Y, int Z, int x0, int y0, int z0, int PX, int PY, int PZ,
                    float shift, float factor, float *__restrict__ tile) {
  const int64_t total = (int64_t)PX * PY * PZ;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int z = (int)(i % PZ), y = (int)((i / PZ) % PY), x = (int)(i / ((int64_t)PZ * PY));
    const float hu = (float)vol[((int64_t)(x0 + x) * Y + (y0 + y)) * Z + (z0 + z)];
    tile[i] = (hu - shift) / factor;
  }
}

__global__ void __launch_bounds__(256)
tile_accumulate_kernel(const float *__restrict__ tile, float *__restrict__ acc, float *__restrict__ cnt, int X, int Y, int Z,
                       int x0, int y0, int z0, int PX, int PY, int PZ) {
  const int64_t total = (int64_t)PX * PY * PZ;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int z = (int)(i % PZ), y = (int)((i / PZ) % PY), x = (int)(i / ((int64_t)PZ * PY));
    const int64_t o = ((int64_t)(x0 + x) * Y + (y0 + y)) * Z + (z0 + z);
    acc[o] += tile[i];
    cnt[o] += 1.f;
  }
}

__global__ void __launch_bounds__(256)
tile_finalize_kernel(const float *__restrict__ acc, const float *__restrict__ cnt, float *__restrict__ out, int64_t n,
                     float shift, float factor) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (acc[i] / cnt[i]) * factor + shift;
}

// One axis of the corrector's tile grid (CCTAContrastCorrector.grid_tiles): `reg` regular starts 0, s, 2s, ... <= S - P,
// then the squeezed start S - P when the last regular tile stops short of the end.  Tile t of the grid is
// (ix, iy, iz) with t = (ix * ny + iy) * nz + iz.
struct GridAxis {
  int S, P, s, reg, n;
};
static inline GridAxis grid_axis(int S, int P, int s) {
  const int reg = (S - P) / s + 1;
  return GridAxis{S, P, s, reg, reg + ((reg - 1) * s + P < S ? 1 : 0)};
}
__device__ __forceinline__ int grid_start(const GridAxis &a, int k) { return k < a.reg ? k * a.s : a.S - a.P; }

// The tiles of one axis that cover coordinate v, in ascending order: regular tiles k0 .. k0 + nreg - 1, then the
// squeezed tile (index reg) when it exists and covers v.  n <= ceil(P / s) + 1.
struct Cover {
  int k0, nreg, n;
};
__device__ __forceinline__ Cover grid_cover(const GridAxis &a, int v) {
  const int k0 = v >= a.P ? (v - a.P) / a.s + 1 : 0;
  const int k1 = mn(v / a.s, a.reg - 1);
  const int nreg = mx(0, k1 - k0 + 1);
  return Cover{k0, nreg, nreg + (a.n > a.reg && v >= a.S - a.P ? 1 : 0)};
}
__device__ __forceinline__ int cover_tile(const Cover &c, const GridAxis &a, int j) { return j < c.nreg ? c.k0 + j : a.reg; }

// tiles [n][PX][PY][PZ] of grid tiles t0 .. t0 + n - 1; blockIdx.y = tile, the same expression as tile_extract_kernel
__global__ void __launch_bounds__(256)
tile_extract_grid_kernel(const int16_t *__restrict__ vol, int Y, int Z, GridAxis gx, GridAxis gy, GridAxis gz, int t0,
                         float shift, float factor, float *__restrict__ tiles) {
  const int PX = gx.P, PY = gy.P, PZ = gz.P, total = PX * PY * PZ;
  const int t = t0 + (int)blockIdx.y;
  const int x0 = grid_start(gx, t / (gz.n * gy.n)), y0 = grid_start(gy, (t / gz.n) % gy.n), z0 = grid_start(gz, t % gz.n);
  float *tile = tiles + (int64_t)blockIdx.y * total;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int z = i % PZ, y = (i / PZ) % PY, x = i / (PZ * PY);
    const float hu = (float)vol[((int64_t)(x0 + x) * Y + (y0 + y)) * Z + (z0 + z)];
    tile[i] = (hu - shift) / factor;
  }
}

// out(v) = sum_t w(v - o_t) c_t(v) / sum_t w(v - o_t) over the grid tiles covering v, in ascending tile index; with
// to_hu the result is unscaled as in tile_finalize_kernel.  One warp per (x, y) row, lanes along z.  For GAUSS = false
// (w = 1) the operations are exactly those of tile_accumulate_kernel (tile by tile) followed by acc / cnt.
// GAUSS: w = (wx * wy) * wz, w_a(i) = expf(-(i - (P_a - 1) / 2)^2 / (2 sigma_a^2)), sigma_a = P_a / 8, tabulated per
// block in shared memory; the weighted mean is kept as a running mean, s += (w / wsum) (c - s), which gives a constant
// input back exactly (a plain sum / wsum is off by several ulp where many tiles of small weight overlap).
template <bool GAUSS>
__global__ void __launch_bounds__(256)
tile_stitch_kernel(const float *const *__restrict__ tiles, int X, int Y, int Z, GridAxis gx, GridAxis gy, GridAxis gz,
                   int to_hu, float shift, float factor, float *__restrict__ out) {
  extern __shared__ float wtab[];  // GAUSS: [PX] x weights, [PY] y weights, [PZ] z weights
  const int PY = gy.P, PZ = gz.P;
  if (GAUSS) {
    const int nw = gx.P + PY + PZ;
    for (int i = threadIdx.y * blockDim.x + threadIdx.x; i < nw; i += blockDim.x * blockDim.y) {
      const int P = i < gx.P ? gx.P : i < gx.P + PY ? PY : PZ;
      const int l = i < gx.P ? i : i < gx.P + PY ? i - gx.P : i - gx.P - PY;
      const float sig = (float)P * 0.125f, d = (float)l - 0.5f * (float)(P - 1);
      wtab[i] = expf(-(d * d) / (2.f * sig * sig));
    }
    __syncthreads();
  }
  const float *wx_t = wtab, *wy_t = wtab + gx.P, *wz_t = wtab + gx.P + PY;
  for (int row = blockIdx.x * blockDim.y + threadIdx.y; row < X * Y; row += gridDim.x * blockDim.y) {
    const int x = row / Y, y = row % Y;
    const Cover cx = grid_cover(gx, x), cy = grid_cover(gy, y);
    for (int z = threadIdx.x; z < Z; z += blockDim.x) {
      const Cover cz = grid_cover(gz, z);
      float s = 0.f, wsum = 0.f;
      for (int jx = 0; jx < cx.n; ++jx) {
        const int ix = cover_tile(cx, gx, jx), lx = x - grid_start(gx, ix);
        for (int jy = 0; jy < cy.n; ++jy) {
          const int iy = cover_tile(cy, gy, jy), ly = y - grid_start(gy, iy);
          const int tbase = (ix * gy.n + iy) * gz.n, ebase = (lx * PY + ly) * PZ;
          const float wxy = GAUSS ? wx_t[lx] * wy_t[ly] : 1.f;
          for (int jz = 0; jz < cz.n; ++jz) {
            const int iz = cover_tile(cz, gz, jz), lz = z - grid_start(gz, iz);
            const float c = tiles[tbase + iz][ebase + lz];
            if (GAUSS) {
              const float w = wxy * wz_t[lz];
              wsum += w;
              s = fmaf(w / wsum, c - s, s);
            } else {
              s += c;
              wsum += 1.f;
            }
          }
        }
      }
      const float q = GAUSS ? s : s / wsum;
      out[(int64_t)row * Z + z] = to_hu ? q * factor + shift : q;
    }
  }
}

// out = x - nearest_resize(att): the corrector's `patch - nn.Upsample(size=patch)(G(patch))` branch
// (reference eval/CCTAContrastCorrector.py:42-52,79); index law of aten::upsample_nearest3d (legacy "nearest").
__device__ __forceinline__ int nearest_src(int dst, int in_size, int out_size) {
  if (in_size == out_size) return dst;
  if (out_size == 2 * in_size) return dst >> 1;
  const float scale = (float)in_size / (float)out_size;
  const int s = (int)floorf((float)dst * scale);
  return s < in_size - 1 ? s : in_size - 1;
}
__global__ void __launch_bounds__(256)
sub_resized_kernel(const float *__restrict__ x, const float *__restrict__ att, float *__restrict__ out, int B, int X, int Y, int Z,
                   int Xa, int Ya, int Za) {
  const int64_t total = (int64_t)B * X * Y * Z;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int z = (int)(i % Z), y = (int)((i / Z) % Y), xx = (int)((i / ((int64_t)Z * Y)) % X), b = (int)(i / ((int64_t)Z * Y * X));
    const int64_t j = (((int64_t)b * Xa + nearest_src(xx, Xa, X)) * Ya + nearest_src(y, Ya, Y)) * Za + nearest_src(z, Za, Z);
    out[i] = x[i] - att[j];
  }
}

// out = (hu - shift) / factor for a contiguous int16 tensor, 8 elements per thread (one 16-byte load, two 16-byte stores):
// the device side of FactorZeroCenterScaler.__call__ (reference data/Scaler.py:41-42) for batches uploaded as raw HU
__global__ void __launch_bounds__(256)
scale_i16_kernel(const int16_t *__restrict__ hu, float *__restrict__ out, int64_t n, float shift, float factor) {
  const int64_t n8 = n >> 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 v = reinterpret_cast<const uint4 *>(hu)[i];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    float f[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      f[2 * k] = ((float)(int16_t)(w[k] & 0xFFFFu) - shift) / factor;
      f[2 * k + 1] = ((float)(int16_t)(w[k] >> 16) - shift) / factor;
    }
    reinterpret_cast<float4 *>(out)[2 * i] = make_float4(f[0], f[1], f[2], f[3]);
    reinterpret_cast<float4 *>(out)[2 * i + 1] = make_float4(f[4], f[5], f[6], f[7]);
  }
  if (blockIdx.x == 0)
    for (int64_t i = (n8 << 3) + threadIdx.x; i < n; i += blockDim.x) out[i] = ((float)hu[i] - shift) / factor;
}

// the three axes of the tile grid for a volume, patch and step, checked: 1 <= P <= S and 1 <= s <= P per axis
static int tile_grid(const char *who, int X, int Y, int Z, int PX, int PY, int PZ, int SX, int SY, int SZ, GridAxis *g) {
  CG_CHECK_SHAPE(X > 0 && Y > 0 && Z > 0 && PX > 0 && PY > 0 && PZ > 0 && PX <= X && PY <= Y && PZ <= Z,
                 "%s: patch %dx%dx%d does not fit the volume %dx%dx%d", who, PX, PY, PZ, X, Y, Z);
  CG_CHECK_SHAPE(SX >= 1 && SY >= 1 && SZ >= 1 && SX <= PX && SY <= PY && SZ <= PZ,
                 "%s: step %dx%dx%d outside 1..patch (%dx%dx%d)", who, SX, SY, SZ, PX, PY, PZ);
  CG_CHECK_SHAPE((int64_t)PX * PY * PZ <= INT32_MAX && (int64_t)X * Y <= INT32_MAX, "%s: volume or patch too large", who);
  g[0] = grid_axis(X, PX, SX);
  g[1] = grid_axis(Y, PY, SY);
  g[2] = grid_axis(Z, PZ, SZ);
  CG_CHECK_SHAPE((int64_t)g[0].n * g[1].n * g[2].n <= INT32_MAX, "%s: too many tiles", who);
  return 0;
}

}  // namespace cg

using namespace cg;

extern "C" {

int cgan3d_gen_loss_sums(const float *s, const float *t, const uint8_t *mask, int64_t n, float hu_lo, float hu_hi,
                         double *sums, void *stream) {
  CG_CHECK_ARG(s && t && sums, "gen_loss_sums: NULL pointer");
  CG_CHECK_SHAPE(n > 1, "gen_loss_sums: need at least 2 elements (unbiased std)");
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(sums, 0, 7 * sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "gen_loss_sums memset");
  const int blocks = (int)mx<int64_t>(1, mn<int64_t>((n + 255) / 256, (int64_t)num_sms() * 8));
  gen_loss_sums_kernel<<<blocks, 256, 0, st>>>(s, t, mask, n, hu_lo, hu_hi, sums);
  CG_LAUNCH_CHECK("gen_loss_sums");
  return 0;
}

int cgan3d_gen_loss_finalize(const double *sums, int64_t n, float w_sim, float w_hu, float *out, float *coef, void *stream) {
  CG_CHECK_ARG(sums && out && coef, "gen_loss_finalize: NULL pointer");
  CG_CHECK_SHAPE(n > 1, "gen_loss_finalize: need at least 2 elements");
  gen_loss_finalize_kernel<<<1, 32, 0, as_stream(stream)>>>(sums, n, w_sim, w_hu, out, coef);
  CG_LAUNCH_CHECK("gen_loss_finalize");
  return 0;
}

int cgan3d_gen_loss_backward(const float *s, const float *t, const uint8_t *mask, int64_t n, float hu_lo, float hu_hi,
                             const float *coef, const float *upstream, const float *d_extra, float *ds, void *stream) {
  CG_CHECK_ARG(s && t && coef && ds, "gen_loss_backward: NULL pointer");
  if (n <= 0) return 0;
  gen_loss_backward_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(s, t, mask, n, hu_lo, hu_hi, coef, upstream,
                                                                        d_extra, ds);
  CG_LAUNCH_CHECK("gen_loss_backward");
  return 0;
}

int cgan3d_mean(const void *x, int dtype, int64_t n, float scale, double *scratch, float *out, void *stream) {
  CG_CHECK_ARG(x && scratch && out, "mean: NULL pointer");
  CG_CHECK_DTYPE(dtype, "mean");
  CG_CHECK_SHAPE(n > 0, "mean: empty tensor");
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaMemsetAsync(scratch, 0, sizeof(double), st);
  if (e != cudaSuccess) return cuda_fail(e, "mean memset");
  const int blocks = (int)mx<int64_t>(1, mn<int64_t>((n + 255) / 256, (int64_t)num_sms() * 4));
  with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    sum_kernel<T><<<blocks, 256, 0, st>>>((const T *)x, n, scratch);
  });
  CG_LAUNCH_CHECK("mean(sum)");
  mean_finalize_kernel<<<1, 32, 0, st>>>(scratch, n, scale, out);
  CG_LAUNCH_CHECK("mean(finalize)");
  return 0;
}

int cgan3d_fill(void *x, int dtype, int64_t n, const float *value_dev, float scale, void *stream) {
  CG_CHECK_ARG(x, "fill: NULL pointer");
  CG_CHECK_DTYPE(dtype, "fill");
  if (n <= 0) return 0;
  cudaStream_t st = as_stream(stream);
  with_dtype(dtype, [&](auto t) {
    using T = typename decltype(t)::type;
    fill_kernel<T><<<ew_blocks(n), 256, 0, st>>>((T *)x, n, value_dev, scale);
  });
  CG_LAUNCH_CHECK("fill");
  return 0;
}

int cgan3d_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr, float beta1,
                     float beta2, float eps, int step, float clip, void *stream) {
  CG_CHECK_ARG(param && grad && exp_avg && exp_avg_sq, "adam_step: NULL pointer");
  CG_CHECK_ARG(step >= 1, "adam_step: step must be >= 1");
  if (n <= 0) return 0;
  adam_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step,
                                                           clip);
  CG_LAUNCH_CHECK("adam_step");
  return 0;
}

int cgan3d_adam_step_multi(int count, float *const *params, const float *const *grads, float *const *exp_avgs,
                           float *const *exp_avg_sqs, const int64_t *numels, float lr, float beta1, float beta2, float eps, int step,
                           float clip, void *stream) {
  CG_CHECK_ARG(count >= 0 && (count == 0 || (params && grads && exp_avgs && exp_avg_sqs && numels)), "adam_step_multi: NULL table");
  CG_CHECK_ARG(step >= 1, "adam_step_multi: step must be >= 1");
  for (int i0 = 0; i0 < count; i0 += kAdamBatch) {
    AdamBatch t{};
    const int nb = count - i0 < kAdamBatch ? count - i0 : kAdamBatch;
    int64_t nmax = 0;
    for (int i = 0; i < nb; ++i) {
      CG_CHECK_ARG(params[i0 + i] && grads[i0 + i] && exp_avgs[i0 + i] && exp_avg_sqs[i0 + i] && numels[i0 + i] >= 0,
                   "adam_step_multi: NULL tensor %d", i0 + i);
      t.p[i] = params[i0 + i]; t.g[i] = grads[i0 + i]; t.m[i] = exp_avgs[i0 + i]; t.v[i] = exp_avg_sqs[i0 + i];
      t.n[i] = numels[i0 + i];
      nmax = nmax > t.n[i] ? nmax : t.n[i];
    }
    if (nmax == 0) continue;
    const int bx = (int)((nmax + 255) / 256 < 64 ? (nmax + 255) / 256 : 64);
    adam_multi_kernel<<<dim3(bx, nb), 256, 0, as_stream(stream)>>>(t, lr, beta1, beta2, eps, step, clip);
    CG_LAUNCH_CHECK("adam_step_multi");
  }
  return 0;
}

int cgan3d_adam_tick(float *hyper, void *stream) {
  CG_CHECK_ARG(hyper, "adam_tick: NULL pointer");
  adam_tick_kernel<<<1, 32, 0, as_stream(stream)>>>(hyper);
  CG_LAUNCH_CHECK("adam_tick");
  return 0;
}

int cgan3d_adam_step_multi_dev(int count, float *const *params, const float *const *grads, float *const *exp_avgs,
                               float *const *exp_avg_sqs, const int64_t *numels, const float *hyper, float beta1, float beta2,
                               float eps, float clip, void *stream) {
  CG_CHECK_ARG(count >= 0 && (count == 0 || (params && grads && exp_avgs && exp_avg_sqs && numels)), "adam_step_multi_dev: NULL table");
  CG_CHECK_ARG(hyper, "adam_step_multi_dev: NULL hyper-parameter pointer");
  for (int i0 = 0; i0 < count; i0 += kAdamBatch) {
    AdamBatch t{};
    const int nb = count - i0 < kAdamBatch ? count - i0 : kAdamBatch;
    int64_t nmax = 0;
    for (int i = 0; i < nb; ++i) {
      CG_CHECK_ARG(params[i0 + i] && grads[i0 + i] && exp_avgs[i0 + i] && exp_avg_sqs[i0 + i] && numels[i0 + i] >= 0,
                   "adam_step_multi_dev: NULL tensor %d", i0 + i);
      t.p[i] = params[i0 + i]; t.g[i] = grads[i0 + i]; t.m[i] = exp_avgs[i0 + i]; t.v[i] = exp_avg_sqs[i0 + i];
      t.n[i] = numels[i0 + i];
      nmax = nmax > t.n[i] ? nmax : t.n[i];
    }
    if (nmax == 0) continue;
    const int bx = (int)((nmax + 255) / 256 < 64 ? (nmax + 255) / 256 : 64);
    adam_multi_dev_kernel<<<dim3(bx, nb), 256, 0, as_stream(stream)>>>(t, hyper, beta1, beta2, eps, clip);
    CG_LAUNCH_CHECK("adam_step_multi_dev");
  }
  return 0;
}

int cgan3d_rmsprop_step_multi(int count, float *const *params, const float *const *grads, float *const *square_avgs,
                              const int64_t *numels, float lr, float alpha, float eps, float clip, void *stream) {
  CG_CHECK_ARG(count >= 0 && (count == 0 || (params && grads && square_avgs && numels)), "rmsprop_step_multi: NULL table");
  for (int i0 = 0; i0 < count; i0 += kAdamBatch) {
    AdamBatch t{};
    const int nb = count - i0 < kAdamBatch ? count - i0 : kAdamBatch;
    int64_t nmax = 0;
    for (int i = 0; i < nb; ++i) {
      CG_CHECK_ARG(params[i0 + i] && grads[i0 + i] && square_avgs[i0 + i] && numels[i0 + i] >= 0, "rmsprop_step_multi: NULL tensor %d", i0 + i);
      t.p[i] = params[i0 + i]; t.g[i] = grads[i0 + i]; t.m[i] = nullptr; t.v[i] = square_avgs[i0 + i];
      t.n[i] = numels[i0 + i];
      nmax = nmax > t.n[i] ? nmax : t.n[i];
    }
    if (nmax == 0) continue;
    const int bx = (int)((nmax + 255) / 256 < 64 ? (nmax + 255) / 256 : 64);
    rmsprop_multi_kernel<<<dim3(bx, nb), 256, 0, as_stream(stream)>>>(t, lr, alpha, eps, clip);
    CG_LAUNCH_CHECK("rmsprop_step_multi");
  }
  return 0;
}

int cgan3d_crop_scale(const int16_t *vol, int X, int Y, int Z, int lbx, int lby, int lbz, int PX, int PY, int PZ, float shift,
                      float factor, float *data, uint8_t *mask, void *stream) {
  CG_CHECK_ARG(vol && data, "crop_scale: NULL pointer");
  CG_CHECK_SHAPE(X > 0 && Y > 0 && Z > 0 && PX > 0 && PY > 0 && PZ > 0 && factor != 0.f, "crop_scale: bad sizes");
  // symmetric zero padding up to the patch size: below = diff // 2 (batchgenerators pad_nd_image)
  const int px0 = (PX > X ? PX - X : 0) / 2, py0 = (PY > Y ? PY - Y : 0) / 2, pz0 = (PZ > Z ? PZ - Z : 0) / 2;
  const int XP = X > PX ? X : PX, YP = Y > PY ? Y : PY, ZP = Z > PZ ? Z : PZ;
  CG_CHECK_SHAPE(lbx >= 0 && lby >= 0 && lbz >= 0 && lbx + PX <= XP && lby + PY <= YP && lbz + PZ <= ZP,
                 "crop_scale: crop [%d,%d,%d]+patch outside the padded volume", lbx, lby, lbz);
  const int64_t total = (int64_t)PX * PY * PZ;
  crop_scale_kernel<<<ew_blocks(total), 256, 0, as_stream(stream)>>>(vol, X, Y, Z, lbx, lby, lbz, PX, PY, PZ, px0, py0, pz0,
                                                                     shift, factor, data, mask);
  CG_LAUNCH_CHECK("crop_scale");
  return 0;
}

int cgan3d_tile_extract(const int16_t *vol, int X, int Y, int Z, int x0, int y0, int z0, int PX, int PY, int PZ, float shift,
                        float factor, float *tile, void *stream) {
  CG_CHECK_ARG(vol && tile, "tile_extract: NULL pointer");
  CG_CHECK_SHAPE(x0 >= 0 && y0 >= 0 && z0 >= 0 && x0 + PX <= X && y0 + PY <= Y && z0 + PZ <= Z && factor != 0.f,
                 "tile_extract: tile outside the volume");
  const int64_t total = (int64_t)PX * PY * PZ;
  tile_extract_kernel<<<ew_blocks(total), 256, 0, as_stream(stream)>>>(vol, X, Y, Z, x0, y0, z0, PX, PY, PZ, shift, factor,
                                                                       tile);
  CG_LAUNCH_CHECK("tile_extract");
  return 0;
}

int cgan3d_tile_accumulate(const float *tile, float *acc, float *cnt, int X, int Y, int Z, int x0, int y0, int z0, int PX,
                           int PY, int PZ, void *stream) {
  CG_CHECK_ARG(tile && acc && cnt, "tile_accumulate: NULL pointer");
  CG_CHECK_SHAPE(x0 >= 0 && y0 >= 0 && z0 >= 0 && x0 + PX <= X && y0 + PY <= Y && z0 + PZ <= Z,
                 "tile_accumulate: tile outside the volume");
  const int64_t total = (int64_t)PX * PY * PZ;
  tile_accumulate_kernel<<<ew_blocks(total), 256, 0, as_stream(stream)>>>(tile, acc, cnt, X, Y, Z, x0, y0, z0, PX, PY, PZ);
  CG_LAUNCH_CHECK("tile_accumulate");
  return 0;
}

int cgan3d_sub_resized(const float *x, const float *att, float *out, int B, int X, int Y, int Z, int Xa, int Ya, int Za,
                       void *stream) {
  CG_CHECK_ARG(x && att && out, "sub_resized: NULL pointer");
  CG_CHECK_SHAPE(B >= 0 && X > 0 && Y > 0 && Z > 0 && Xa > 0 && Ya > 0 && Za > 0, "sub_resized: bad sizes");
  const int64_t total = (int64_t)B * X * Y * Z;
  if (total == 0) return 0;
  sub_resized_kernel<<<ew_blocks(total), 256, 0, as_stream(stream)>>>(x, att, out, B, X, Y, Z, Xa, Ya, Za);
  CG_LAUNCH_CHECK("sub_resized");
  return 0;
}

int cgan3d_scale_i16(const int16_t *hu, float *out, int64_t n, float shift, float factor, void *stream) {
  CG_CHECK_ARG(hu && out, "scale_i16: NULL pointer");
  CG_CHECK_SHAPE(n >= 0 && factor != 0.f, "scale_i16: bad size / zero factor");
  CG_CHECK_ARG(!(reinterpret_cast<uintptr_t>(hu) & 15) && !(reinterpret_cast<uintptr_t>(out) & 15), "scale_i16: pointers must be 16-byte aligned");
  if (n == 0) return 0;
  scale_i16_kernel<<<ew_blocks(n >> 3 ? n >> 3 : 1), 256, 0, as_stream(stream)>>>(hu, out, n, shift, factor);
  CG_LAUNCH_CHECK("scale_i16");
  return 0;
}

int cgan3d_tile_finalize(const float *acc, const float *cnt, float *out, int64_t n, float shift, float factor, void *stream) {
  CG_CHECK_ARG(acc && cnt && out, "tile_finalize: NULL pointer");
  if (n <= 0) return 0;
  tile_finalize_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(acc, cnt, out, n, shift, factor);
  CG_LAUNCH_CHECK("tile_finalize");
  return 0;
}

int cgan3d_tile_extract_grid(const int16_t *vol, int X, int Y, int Z, int PX, int PY, int PZ, int SX, int SY, int SZ, int t0,
                             int n, float shift, float factor, float *tiles, void *stream) {
  CG_CHECK_ARG(vol && tiles, "tile_extract_grid: NULL pointer");
  GridAxis g[3];
  if (int rc = tile_grid("tile_extract_grid", X, Y, Z, PX, PY, PZ, SX, SY, SZ, g)) return rc;
  const int ntiles = g[0].n * g[1].n * g[2].n;
  CG_CHECK_SHAPE(t0 >= 0 && n >= 0 && n <= ntiles - t0 && n <= 65535, "tile_extract_grid: tiles %d..%d outside the grid of %d (at most 65535 per call)", t0, t0 + n - 1, ntiles);
  CG_CHECK_ARG(factor != 0.f, "tile_extract_grid: zero factor");
  if (n == 0) return 0;
  const int per_tile = (int)mx<int64_t>(1, ew_blocks((int64_t)n * PX * PY * PZ) / n);
  tile_extract_grid_kernel<<<dim3(per_tile, n), 256, 0, as_stream(stream)>>>(vol, Y, Z, g[0], g[1], g[2], t0, shift, factor,
                                                                            tiles);
  CG_LAUNCH_CHECK("tile_extract_grid");
  return 0;
}

int cgan3d_tile_stitch(const float *const *tiles, int n, int X, int Y, int Z, int PX, int PY, int PZ, int SX, int SY, int SZ,
                       int blend, int to_hu, float shift, float factor, float *out, void *stream) {
  CG_CHECK_ARG(tiles && out, "tile_stitch: NULL pointer");
  GridAxis g[3];
  if (int rc = tile_grid("tile_stitch", X, Y, Z, PX, PY, PZ, SX, SY, SZ, g)) return rc;
  CG_CHECK_SHAPE(n == g[0].n * g[1].n * g[2].n, "tile_stitch: %d tiles given, the grid has %d", n, g[0].n * g[1].n * g[2].n);
  CG_CHECK_ARG(blend == CGAN3D_BLEND_AVG || blend == CGAN3D_BLEND_GAUSSIAN, "tile_stitch: unknown blend %d", blend);
  const size_t smem = blend == CGAN3D_BLEND_GAUSSIAN ? (size_t)(PX + PY + PZ) * sizeof(float) : 0;
  CG_CHECK_SHAPE(smem <= 48 * 1024, "tile_stitch: patch %dx%dx%d too large for the weight table", PX, PY, PZ);
  const dim3 block(32, 8);
  const int grid = (int)mn<int64_t>(((int64_t)X * Y + 7) / 8, (int64_t)num_sms() * 8);
  if (blend == CGAN3D_BLEND_GAUSSIAN)
    tile_stitch_kernel<true><<<grid, block, smem, as_stream(stream)>>>(tiles, X, Y, Z, g[0], g[1], g[2], to_hu, shift, factor, out);
  else
    tile_stitch_kernel<false><<<grid, block, 0, as_stream(stream)>>>(tiles, X, Y, Z, g[0], g[1], g[2], to_hu, shift, factor, out);
  CG_LAUNCH_CHECK("tile_stitch");
  return 0;
}

}  // extern "C"
