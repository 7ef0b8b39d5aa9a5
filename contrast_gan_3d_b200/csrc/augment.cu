// Spatial augmentation (batchgenerators SpatialTransform_2 / augment_spatial_2, reference experiments/basic_conf.py:88-106)
// on the device: elastic offset fields, cubic B-spline prefilter and the resampling gather.
//
//  1. elastic field: uniform [-1, 1) noise from Philox4x32-10 keyed by a per-sample seed, smoothed by the Gaussian of
//     scipy.ndimage.fourier_gaussian as three circular 1-D convolutions with periodic taps computed on the host, then
//     scaled so that max|field| = mag + 1e-8 per axis.  max and sum come from a fixed-order two-stage reduction: the
//     same seed gives bit-identical fields.
//  2. spline prefilter: scipy.ndimage.spline_filter (order 3, pole sqrt(3) - 2) of each transformed sample, including
//     SciPy's boundary handling: `nearest` pads 12 voxels by edge replication and filters with reflect boundaries,
//     `constant` filters with mirror boundaries.
//  3. resampling: c = A (mesh + offsets) - A mean(offsets) + ctr, then the 4x4x4 B-spline gather for data and the
//     order-0 lookup (index floor(c + 0.5)) for seg.  Samples that drew no transform are a zero-filled shifted copy.
#include "common.cuh"

namespace cg {
namespace {

constexpr int kMaxLine = 256;     // longest smoothed / resampled axis
constexpr int kNearestPad = 12;   // scipy.ndimage._interpolation._prepad_for_spline_filter
constexpr int kPartials = 64;     // stage-1 blocks per (sample, axis) of the field reduction
constexpr double kPole = -0.26794919243112270;  // sqrt(3) - 2

// element e of a sample's [3][PX][PY][PZ] noise: 2u - 1 with u = k * 2^-24, exact in fp32 (word 0 of counter (e, 0, 0, 0))
__device__ __forceinline__ float noise_at(uint32_t e, uint64_t seed) {
  return (float)(philox4x32_10(e, 0, 0, 0, seed).x >> 8) * 0x1p-23f - 1.f;
}

__global__ void __launch_bounds__(256) elastic_noise_kernel(const uint64_t *__restrict__ seeds, float *__restrict__ out,
                                                            int64_t per_sample) {
  const int s = blockIdx.y;
  const uint64_t seed = seeds[s];
  for (int64_t e = blockIdx.x * 256ll + threadIdx.x; e < per_sample; e += (int64_t)gridDim.x * 256)
    out[s * per_sample + e] = noise_at((uint32_t)e, seed);
}

// One circular 1-D convolution pass along one axis of every (sample, component) volume, viewed as [outer][n][inner].
// A block owns 32 lines (line L -> o = L / inner, c = L % inner), staged as a [n][33] tile: for inner == 1 (z) the
// 32 lines are one contiguous run and are transposed into the tile, otherwise lanes read 32 consecutive c.  Each
// output is y[p] = sum_k h[k] x[(p - k) mod n] with fp64 accumulation.  NOISE: the input is the Philox noise itself.
template <bool NOISE>
__global__ void __launch_bounds__(256) smooth_pass_kernel(const float *__restrict__ in, float *__restrict__ out,
                                                          const uint64_t *__restrict__ seeds,
                                                          const double *__restrict__ taps, int tap_stride,
                                                          int tap_off, int n, int inner, int lines, int64_t vol) {
  extern __shared__ double smem_d[];
  double *h = smem_d;                          // [n]
  float *T = reinterpret_cast<float *>(h + n); // [n][33] input tile
  float *R = T + n * 33;                       // [n][33] output tile
  const int sc = blockIdx.y;                   // sample * 3 + component
  const int s = sc / 3;
  const int64_t base = (int64_t)sc * vol;
  const int L0 = blockIdx.x * 32;
  const int nl = min(32, lines - L0);
  for (int k = threadIdx.x; k < n; k += 256) h[k] = taps[(int64_t)s * tap_stride + tap_off + k];
  const uint64_t seed = NOISE ? seeds[s] : 0;
  auto src = [&](int64_t idx) -> float {
    if (NOISE) return noise_at((uint32_t)((sc % 3) * vol + idx), seed);
    return in[base + idx];
  };
  if (inner == 1) {
    for (int t = threadIdx.x; t < nl * n; t += 256) T[(t % n) * 33 + t / n] = src((int64_t)L0 * n + t);
  } else {
    const int l = threadIdx.x & 31;
    if (l < nl) {
      const int L = L0 + l, o = L / inner, c = L % inner;
      for (int i = threadIdx.x >> 5; i < n; i += 8) T[i * 33 + l] = src(((int64_t)o * n + i) * inner + c);
    }
  }
  __syncthreads();
  const int col = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int p0 = w; p0 < n; p0 += 32) {
    double acc[4] = {0., 0., 0., 0.};
    int q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = min(p0 + 8 * j, n - 1);
    for (int k = 0; k < n; ++k) {
      const double hk = h[k];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc[j] = fma(hk, (double)T[q[j] * 33 + col], acc[j]);
        q[j] = q[j] == 0 ? n - 1 : q[j] - 1;
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (p0 + 8 * j < n) R[(p0 + 8 * j) * 33 + col] = (float)acc[j];
  }
  __syncthreads();
  if (inner == 1) {
    for (int t = threadIdx.x; t < nl * n; t += 256) out[base + (int64_t)L0 * n + t] = R[(t % n) * 33 + t / n];
  } else {
    const int l = threadIdx.x & 31;
    if (l < nl) {
      const int L = L0 + l, o = L / inner, c = L % inner;
      for (int i = threadIdx.x >> 5; i < n; i += 8) out[base + ((int64_t)o * n + i) * inner + c] = R[i * 33 + l];
    }
  }
}

// stage 1: block b of (sample, component) sc reduces a fixed contiguous chunk to (max|f|, sum f)
__global__ void __launch_bounds__(256) field_partials_kernel(const float *__restrict__ f, int64_t vol,
                                                             double *__restrict__ part) {
  __shared__ double ssum[256];
  __shared__ float smax[256];
  const int sc = blockIdx.y;
  const int64_t chunk = (vol + kPartials - 1) / kPartials;
  const int64_t lo = blockIdx.x * chunk, hi = min(vol, lo + chunk);
  const float *p = f + (int64_t)sc * vol;
  double sum = 0.;
  float m = 0.f;
  for (int64_t i = lo + threadIdx.x; i < hi; i += 256) {
    const float v = p[i];
    sum += (double)v;
    m = fmaxf(m, fabsf(v));
  }
  ssum[threadIdx.x] = sum;
  smax[threadIdx.x] = m;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (threadIdx.x < st) {
      ssum[threadIdx.x] += ssum[threadIdx.x + st];
      smax[threadIdx.x] = fmaxf(smax[threadIdx.x], smax[threadIdx.x + st]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    part[((int64_t)sc * kPartials + blockIdx.x) * 2] = (double)smax[0];
    part[((int64_t)sc * kPartials + blockIdx.x) * 2 + 1] = ssum[0];
  }
}

// stage 2 (one thread per (sample, component), fixed order): divisor max|f| / (mag + 1e-8), sum of the scaled field
__global__ void field_finalize_kernel(const double *__restrict__ part, const double *__restrict__ mags, int count,
                                      double *__restrict__ scale, double *__restrict__ sums) {
  const int sc = blockIdx.x * blockDim.x + threadIdx.x;
  if (sc >= count) return;
  double m = 0., s = 0.;
  for (int b = 0; b < kPartials; ++b) {
    m = fmax(m, part[((int64_t)sc * kPartials + b) * 2]);
    s += part[((int64_t)sc * kPartials + b) * 2 + 1];
  }
  const double d = m / (mags[sc] + 1e-8);  // numpy: offsets / (mx / (mag + 1e-8))
  scale[sc] = d;
  sums[sc] = s / d;
}

__global__ void __launch_bounds__(256) field_scale_kernel(const float *__restrict__ f, const double *__restrict__ scale,
                                                          int64_t vol, float *__restrict__ out) {
  const int sc = blockIdx.y;
  const double d = scale[sc];
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < vol; i += (int64_t)gridDim.x * 256)
    out[(int64_t)sc * vol + i] = (float)((double)f[(int64_t)sc * vol + i] / d);
}

// ---- cubic B-spline prefilter (scipy ndimage/src/ni_splines.c, order 3) ----------------------------------------

// in-place filter of one line c[0..n) with element stride `st`; REFLECT: half-sample symmetric (scipy `nearest` /
// `reflect`), otherwise whole-sample symmetric (`mirror` / `constant`)
template <bool REFLECT>
__device__ void spline_line(float *c, int n, int64_t st) {
  const float z = (float)kPole;
  for (int i = 0; i < n; ++i) c[i * st] *= 6.f;
  const float x0 = c[0];
  if (REFLECT) {
    const float zn = (float)pow(kPole, (double)n);
    float acc = x0 + zn * c[(n - 1) * st], zi = z;
    for (int i = 1; i < n && zi != 0.f; ++i, zi *= z) acc += zi * (c[i * st] + zn * c[(n - 1 - i) * st]);
    c[0] = acc * z / (1.f - zn * zn) + x0;
  } else {
    const float zn1 = (float)pow(kPole, (double)(n - 1));
    float acc = x0 + zn1 * c[(n - 1) * st], zi = z;
    for (int i = 1; i < n - 1 && zi != 0.f; ++i, zi *= z) acc += zi * (c[i * st] + zn1 * c[(n - 1 - i) * st]);
    c[0] = acc / (1.f - zn1 * zn1);
  }
  float prev = c[0];
  for (int i = 1; i < n; ++i) {
    prev = c[i * st] + z * prev;
    c[i * st] = prev;
  }
  float last = REFLECT ? prev * z / (z - 1.f) : (z * c[(n - 2) * st] + prev) * z / (z * z - 1.f);
  c[(n - 1) * st] = last;
  for (int i = n - 2; i >= 0; --i) {
    last = z * (last - c[i * st]);
    c[i * st] = last;
  }
}

// pass along z over every line of the padded volume; the first pass also copies the (edge-replicated) input
template <bool REFLECT>
__global__ void __launch_bounds__(128) prefilter_z_kernel(const float *__restrict__ data, const int32_t *__restrict__ samples,
                                                          int SX, int SY, int SZ, int pad, float *__restrict__ coef) {
  const int Xp = SX + 2 * pad, Yp = SY + 2 * pad, Zp = SZ + 2 * pad;
  const int line = blockIdx.x * 128 + threadIdx.x;
  if (line >= Xp * Yp) return;
  const int j = blockIdx.y;
  const int x = min(max(line / Yp - pad, 0), SX - 1), y = min(max(line % Yp - pad, 0), SY - 1);
  const float *src = data + (int64_t)samples[j] * SX * SY * SZ + ((int64_t)x * SY + y) * SZ;
  float *c = coef + (int64_t)j * Xp * Yp * Zp + (int64_t)line * Zp;
  for (int z = 0; z < Zp; ++z) c[z] = src[min(max(z - pad, 0), SZ - 1)];
  spline_line<REFLECT>(c, Zp, 1);
}

// pass along x (axis_stride = Yp * Zp, lines = Yp * Zp) or y (axis_stride = Zp, lines = Xp * Zp)
template <bool REFLECT>
__global__ void __launch_bounds__(128) prefilter_xy_kernel(float *__restrict__ coef, int Xp, int Yp, int Zp, int axis) {
  const int line = blockIdx.x * 128 + threadIdx.x;
  float *c = coef + (int64_t)blockIdx.y * Xp * Yp * Zp;
  if (axis == 0) {
    if (line >= Yp * Zp) return;
    spline_line<REFLECT>(c + line, Xp, (int64_t)Yp * Zp);
  } else {
    if (line >= Xp * Zp) return;
    spline_line<REFLECT>(c + (int64_t)(line / Zp) * Yp * Zp + line % Zp, Yp, Zp);
  }
}

// ---- resampling ------------------------------------------------------------------------------------------------

__device__ __forceinline__ void bspline_weights(float t, float w[4]) {
  const float u = 1.f - t;
  w[0] = u * u * u * (1.f / 6.f);
  w[1] = 2.f / 3.f - t * t + 0.5f * t * t * t;
  w[2] = 2.f / 3.f - u * u + 0.5f * u * u * u;
  w[3] = t * t * t * (1.f / 6.f);
}

// tap indices into an axis of n + 2 * pad coefficients for input coordinate q (n input voxels).  The fraction is taken
// before the padding offset is added, so that q keeps its fp32 resolution.
template <bool NEAREST>
__device__ __forceinline__ void taps_for(float q, int n, int pad, int idx[4], float w[4]) {
  const int np = n + 2 * pad;
  if (NEAREST) q = fminf(fmaxf(q, (float)(-2 - pad)), (float)(n + pad + 1));  // beyond: every tap clamps to one edge
  const float f = floorf(q);
  bspline_weights(q - f, w);
  const int i0 = (int)f - 1 + pad;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int i = i0 + k;
    if (NEAREST) {
      i = min(max(i, 0), np - 1);
    } else {  // mirror about 0 and n - 1 (q is inside [0, n - 1])
      i = i < 0 ? -i : i;
      i = i > np - 1 ? 2 * (np - 1) - i : i;
    }
    idx[k] = i;
  }
}

template <bool NEAREST>
__global__ void __launch_bounds__(256) spatial_resample_kernel(
    const float *__restrict__ data, const uint8_t *__restrict__ seg, int SX, int SY, int SZ, int PX, int PY, int PZ,
    const cgan3d_spatial_params_t *__restrict__ params, const float *__restrict__ field, const double *__restrict__ sums,
    const float *__restrict__ coef, float cval, int seg_fill, float *__restrict__ out, uint8_t *__restrict__ out_seg) {
  const int b = blockIdx.y;
  const int64_t P = (int64_t)PX * PY * PZ, S = (int64_t)SX * SY * SZ;
  const int64_t v = blockIdx.x * 256ll + threadIdx.x;
  if (v >= P) return;
  const int x = (int)(v / ((int64_t)PY * PZ)), y = (int)(v / PZ % PY), z = (int)(v % PZ);
  const cgan3d_spatial_params_t &pr = params[b];
  float *o = out + b * P;
  uint8_t *os = out_seg + b * P;
  const float *d = data + b * S;
  const uint8_t *sg = seg + b * S;
  if (!(pr.flags & CGAN3D_SPATIAL_TRANSFORM)) {
    const int sx = x + pr.shift[0], sy = y + pr.shift[1], sz = z + pr.shift[2];
    const bool in = sx >= 0 && sx < SX && sy >= 0 && sy < SY && sz >= 0 && sz < SZ;
    const int64_t si = ((int64_t)sx * SY + sy) * SZ + sz;
    o[v] = in ? d[si] : 0.f;
    os[v] = in ? sg[si] : (uint8_t)0;
    return;
  }
  float m0 = (float)x - 0.5f * (float)(PX - 1), m1 = (float)y - 0.5f * (float)(PY - 1), m2 = (float)z - 0.5f * (float)(PZ - 1);
  float mean[3] = {0.f, 0.f, 0.f};
  if (pr.flags & CGAN3D_SPATIAL_ELASTIC) {
    const float *f = field + (int64_t)pr.field_slot * 3 * P;
    m0 += f[v];
    m1 += f[P + v];
    m2 += f[2 * P + v];
    const double *sm = sums + pr.field_slot * 3;
    const double a0 = sm[0] / (double)P, a1 = sm[1] / (double)P, a2 = sm[2] / (double)P;
#pragma unroll
    for (int r = 0; r < 3; ++r) mean[r] = (float)(pr.A[3 * r] * a0 + pr.A[3 * r + 1] * a1 + pr.A[3 * r + 2] * a2);
  }
  float c[3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
    c[r] = fmaf(pr.A[3 * r], m0, fmaf(pr.A[3 * r + 1], m1, pr.A[3 * r + 2] * m2)) - mean[r] + pr.ctr[r];
  const bool inside = c[0] >= 0.f && c[0] <= (float)(SX - 1) && c[1] >= 0.f && c[1] <= (float)(SY - 1) &&
                      c[2] >= 0.f && c[2] <= (float)(SZ - 1);
  // seg: order 0, mode constant
  if (inside) {
    const int ix = (int)floorf(c[0] + 0.5f), iy = (int)floorf(c[1] + 0.5f), iz = (int)floorf(c[2] + 0.5f);
    os[v] = sg[((int64_t)ix * SY + iy) * SZ + iz];
  } else {
    os[v] = (uint8_t)seg_fill;
  }
  // data: order 3
  if (!NEAREST && !inside) {
    o[v] = cval;
    return;
  }
  const int pad = NEAREST ? kNearestPad : 0;
  const int Xp = SX + 2 * pad, Yp = SY + 2 * pad, Zp = SZ + 2 * pad;
  int ix[4], iy[4], iz[4];
  float wx[4], wy[4], wz[4];
  taps_for<NEAREST>(c[0], SX, pad, ix, wx);
  taps_for<NEAREST>(c[1], SY, pad, iy, wy);
  taps_for<NEAREST>(c[2], SZ, pad, iz, wz);
  const float *cf = coef + (int64_t)pr.coef_slot * Xp * Yp * Zp;
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float ay = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float *row = cf + ((int64_t)ix[i] * Yp + iy[j]) * Zp;
      const float az = wz[0] * __ldg(row + iz[0]) + wz[1] * __ldg(row + iz[1]) + wz[2] * __ldg(row + iz[2]) +
                       wz[3] * __ldg(row + iz[3]);
      ay = fmaf(wy[j], az, ay);
    }
    acc = fmaf(wx[i], ay, acc);
  }
  o[v] = acc;
}

bool dims_ok(int a, int b, int c) { return a >= 4 && b >= 4 && c >= 4 && a <= kMaxLine && b <= kMaxLine && c <= kMaxLine; }

size_t smooth_smem(int n) { return (size_t)n * sizeof(double) + 2 * (size_t)n * 33 * sizeof(float); }

template <bool NOISE>
int smooth_pass(const float *in, float *out, const uint64_t *seeds, const double *taps, int tap_stride, int tap_off,
                int n, int inner, int lines, int64_t vol, int count, cudaStream_t st) {
  static const cudaError_t opt_in = cudaFuncSetAttribute(smooth_pass_kernel<NOISE>,
                                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                         (int)smooth_smem(kMaxLine));
  if (opt_in != cudaSuccess) return cuda_fail(opt_in, "cudaFuncSetAttribute(smooth_pass)");
  smooth_pass_kernel<NOISE><<<dim3((lines + 31) / 32, count), 256, smooth_smem(n), st>>>(in, out, seeds, taps, tap_stride,
                                                                                         tap_off, n, inner, lines, vol);
  CG_LAUNCH_CHECK("smooth_pass");
  return 0;
}

size_t elastic_field_bytes(int n, int PX, int PY, int PZ) {
  return ((size_t)n * 3 * PX * PY * PZ * sizeof(float) + 255) / 256 * 256;
}

}  // namespace
}  // namespace cg

using namespace cg;

extern "C" {

int cgan3d_elastic_noise(int n, int PX, int PY, int PZ, const uint64_t *seeds, float *noise, void *stream) {
  CG_CHECK_ARG(n >= 0 && (n == 0 || (seeds && noise)), "elastic_noise: NULL pointer or negative count");
  if (!dims_ok(PX, PY, PZ)) return fail(CGAN3D_E_UNSUPPORTED, "elastic_noise: patch %dx%dx%d outside 4..%d", PX, PY, PZ, kMaxLine);
  if (n == 0) return 0;
  const int64_t per = 3ll * PX * PY * PZ;
  elastic_noise_kernel<<<dim3((unsigned)mn<int64_t>((per + 255) / 256, 1024), n), 256, 0, as_stream(stream)>>>(seeds, noise, per);
  CG_LAUNCH_CHECK("elastic_noise");
  return 0;
}

size_t cgan3d_elastic_workspace_bytes(int n, int PX, int PY, int PZ) {
  if (n <= 0 || !dims_ok(PX, PY, PZ)) return 0;
  return elastic_field_bytes(n, PX, PY, PZ) + (size_t)n * 3 * (kPartials * 2 + 1) * sizeof(double);
}

int cgan3d_elastic_field(int n, int PX, int PY, int PZ, const uint64_t *seeds, const double *mags, const double *taps,
                         float *field, double *sums, void *ws, size_t ws_bytes, void *stream) {
  CG_CHECK_ARG(n >= 0 && (n == 0 || (seeds && mags && taps && field && sums && ws)), "elastic_field: NULL pointer");
  if (!dims_ok(PX, PY, PZ)) return fail(CGAN3D_E_UNSUPPORTED, "elastic_field: patch %dx%dx%d outside 4..%d", PX, PY, PZ, kMaxLine);
  if (n == 0) return 0;
  if (ws_bytes < cgan3d_elastic_workspace_bytes(n, PX, PY, PZ))
    return fail(CGAN3D_E_WORKSPACE, "elastic_field: workspace %zu < %zu", ws_bytes, cgan3d_elastic_workspace_bytes(n, PX, PY, PZ));
  cudaStream_t st = as_stream(stream);
  const int64_t vol = (int64_t)PX * PY * PZ;
  const int count = 3 * n, tstride = PX + PY + PZ;
  float *tmp = static_cast<float *>(ws);
  double *part = reinterpret_cast<double *>(static_cast<char *>(ws) + elastic_field_bytes(n, PX, PY, PZ));
  double *scale = part + (size_t)count * kPartials * 2;
  int rc;
  // z: noise -> tmp, y: tmp -> field, x: field -> tmp
  if ((rc = smooth_pass<true>(nullptr, tmp, seeds, taps, tstride, PX + PY, PZ, 1, PX * PY, vol, count, st))) return rc;
  if ((rc = smooth_pass<false>(tmp, field, seeds, taps, tstride, PX, PY, PZ, PX * PZ, vol, count, st))) return rc;
  if ((rc = smooth_pass<false>(field, tmp, seeds, taps, tstride, 0, PX, PY * PZ, PY * PZ, vol, count, st))) return rc;
  field_partials_kernel<<<dim3(kPartials, count), 256, 0, st>>>(tmp, vol, part);
  CG_LAUNCH_CHECK("elastic_field partials");
  field_finalize_kernel<<<(count + 63) / 64, 64, 0, st>>>(part, mags, count, scale, sums);
  CG_LAUNCH_CHECK("elastic_field finalize");
  field_scale_kernel<<<dim3((unsigned)mn<int64_t>((vol + 255) / 256, 512), count), 256, 0, st>>>(tmp, scale, vol, field);
  CG_LAUNCH_CHECK("elastic_field scale");
  return 0;
}

size_t cgan3d_spline_workspace_bytes(int n, int SX, int SY, int SZ, int mode) {
  if (n <= 0 || (mode != CGAN3D_BORDER_CONSTANT && mode != CGAN3D_BORDER_NEAREST)) return 0;
  const int pad = mode == CGAN3D_BORDER_NEAREST ? kNearestPad : 0;
  return (size_t)n * (SX + 2 * pad) * (SY + 2 * pad) * (SZ + 2 * pad) * sizeof(float);
}

int cgan3d_spline_prefilter(const float *data, int SX, int SY, int SZ, int n, const int32_t *samples, int mode,
                            float *coef, size_t coef_bytes, void *stream) {
  CG_CHECK_ARG(n >= 0 && (n == 0 || (data && samples && coef)), "spline_prefilter: NULL pointer");
  if (mode != CGAN3D_BORDER_CONSTANT && mode != CGAN3D_BORDER_NEAREST)
    return fail(CGAN3D_E_UNSUPPORTED, "spline_prefilter: border mode %d (constant and nearest only)", mode);
  if (!dims_ok(SX, SY, SZ)) return fail(CGAN3D_E_UNSUPPORTED, "spline_prefilter: volume %dx%dx%d outside 4..%d", SX, SY, SZ, kMaxLine);
  if (n == 0) return 0;
  if (coef_bytes < cgan3d_spline_workspace_bytes(n, SX, SY, SZ, mode))
    return fail(CGAN3D_E_WORKSPACE, "spline_prefilter: workspace %zu < %zu", coef_bytes, cgan3d_spline_workspace_bytes(n, SX, SY, SZ, mode));
  cudaStream_t st = as_stream(stream);
  const int pad = mode == CGAN3D_BORDER_NEAREST ? kNearestPad : 0;
  const int Xp = SX + 2 * pad, Yp = SY + 2 * pad, Zp = SZ + 2 * pad;
  if (mode == CGAN3D_BORDER_NEAREST) {
    prefilter_z_kernel<true><<<dim3((Xp * Yp + 127) / 128, n), 128, 0, st>>>(data, samples, SX, SY, SZ, pad, coef);
    prefilter_xy_kernel<true><<<dim3((Xp * Zp + 127) / 128, n), 128, 0, st>>>(coef, Xp, Yp, Zp, 1);
    prefilter_xy_kernel<true><<<dim3((Yp * Zp + 127) / 128, n), 128, 0, st>>>(coef, Xp, Yp, Zp, 0);
  } else {
    prefilter_z_kernel<false><<<dim3((Xp * Yp + 127) / 128, n), 128, 0, st>>>(data, samples, SX, SY, SZ, pad, coef);
    prefilter_xy_kernel<false><<<dim3((Xp * Zp + 127) / 128, n), 128, 0, st>>>(coef, Xp, Yp, Zp, 1);
    prefilter_xy_kernel<false><<<dim3((Yp * Zp + 127) / 128, n), 128, 0, st>>>(coef, Xp, Yp, Zp, 0);
  }
  CG_LAUNCH_CHECK("spline_prefilter");
  return 0;
}

int cgan3d_spatial_resample(const float *data, const uint8_t *seg, int B, int SX, int SY, int SZ, int PX, int PY, int PZ,
                            const cgan3d_spatial_params_t *params, const float *field, const double *sums,
                            const float *coef, int mode, float cval, int seg_fill, float *out, uint8_t *out_seg,
                            void *stream) {
  CG_CHECK_ARG(B >= 0 && (B == 0 || (data && seg && params && out && out_seg)), "spatial_resample: NULL pointer");
  if (mode != CGAN3D_BORDER_CONSTANT && mode != CGAN3D_BORDER_NEAREST)
    return fail(CGAN3D_E_UNSUPPORTED, "spatial_resample: border mode %d (constant and nearest only)", mode);
  if (!dims_ok(SX, SY, SZ) || !dims_ok(PX, PY, PZ))
    return fail(CGAN3D_E_UNSUPPORTED, "spatial_resample: extents outside 4..%d", kMaxLine);
  if (B == 0) return 0;
  const int64_t P = (int64_t)PX * PY * PZ;
  dim3 grid((unsigned)((P + 255) / 256), B);
  if (mode == CGAN3D_BORDER_NEAREST)
    spatial_resample_kernel<true><<<grid, 256, 0, as_stream(stream)>>>(data, seg, SX, SY, SZ, PX, PY, PZ, params, field,
                                                                        sums, coef, cval, seg_fill, out, out_seg);
  else
    spatial_resample_kernel<false><<<grid, 256, 0, as_stream(stream)>>>(data, seg, SX, SY, SZ, PX, PY, PZ, params, field,
                                                                         sums, coef, cval, seg_fill, out, out_seg);
  CG_LAUNCH_CHECK("spatial_resample");
  return 0;
}

}  // extern "C"
