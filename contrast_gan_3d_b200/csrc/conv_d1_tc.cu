// tcgen05 kernels for the FIRST CRITIC LAYER, Conv3d(1 -> 8, k = 4, stride 2, pad 1) + its backward
// (reference model/discriminator.py:36-46: `first` ConvBlock of PatchGANDiscriminator; aten::convolution /
// convolution_backward).  One input channel means GEMM K (fprop, wgrad) or N (dgrad) of 1, so the channel-GEMM kernels do
// not apply; the layer is HBM-bound (SURVEY App. B: AI 32 FLOP/B) and all three ops stream each tensor once.
//
//  gather  (fprop):  TOEPLITZ-IN-Z as in conv_thin_tc.cu (A), on the stride-2 parity sub-grids.  Rows = flattened (x, y)
//          output positions; the 4 (x,y) parity classes are 4 TMA loads with elementStrides (1,2,2,1); inside a class the
//          2x2 taps are row shifts; K = 16 consecutive input z of one line; N = 4 output z x 8 channels; the filter of tap
//          (dx,dy) is the banded matrix T[zi][(zo,co)] = W[dx,dy,zi-2*zo,co].
//  wgrad:  both operands MN-major, K = 16 output voxels per MMA.  A (M = 64) = 8 chunks (4 dx planes x 2 line shifts) of
//          the z/y-EXPANDED input E[x'][yy][oz][(dyp,dz)] = in[x'][2yy-1+dyp][2oz-1+dz] (16-byte rows, built by a pre-pass);
//          B (N = 8) = dY.  One accumulator [64 x 8] per CTA, split-K, fp32 atomics.
//  scatter (dgrad):  all 8 output parity phases STACKED ON N.  Rows = small-grid positions g (o = g - 1), K = 16 = two
//          z-adjacent dY voxels x 8 channels (A-descriptor LBO = one row), 4 MMAs (sx, sy) per row tile; column
//          (ux,uy,uz) of row g is output voxel 2g - 1 + u.
#include "common.cuh"
#include "conv_internal.cuh"
#include "tc_common.cuh"

namespace cg {

constexpr uint32_t kSmemLimitD1 = kMaxDynSmem - 1024;

static bool d1_shape(const cgan3d_conv_geom &g) {
  return g.k == 4 && g.stride == 2 && g.pad == 1 && g.Cb == 1 && g.Cs == 8;
}

// =============================================================================================================== gather
struct D1GatherPlan {
  int B, Xi, Yi, Zi, Zc;  // input, z extent of the shifted copy: copy[row][c] = in[row][c - 1]
  int Xo, Yo, Zo;
  int Xt, Yt, Xh, Yh, nxt, nyt, nzb;
  int mtiles, rows_alloc, nslots;
  uint32_t slot_bytes, box_bytes, tmem_cols, smem_bytes;
};
constexpr int kD1Tiles = 16;
constexpr uint32_t kD1TileBytes = 1024;  // [2 z-chunks][32 n][8 z]

template <int MT>
__global__ void __launch_bounds__(192, 1)
d1_gather_tc_kernel(const __grid_constant__ CUtensorMap tmA, const bf16 *__restrict__ wT, bf16 *__restrict__ out,
                    const __grid_constant__ D1GatherPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *bres = smem;                             // 16 resident Toeplitz tiles
  uint8_t *ring = bres + kD1Tiles * kD1TileBytes;   // slab slots
  uint64_t *bars = reinterpret_cast<uint64_t *>(ring + (size_t)p.nslots * p.slot_bytes);
  uint64_t *b_ready = bars, *s_full = bars + 1, *s_empty = s_full + p.nslots;
  uint64_t *tm_full = s_empty + p.nslots, *tm_empty = tm_full + 2;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(tm_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tc::mbar_init(b_ready, 1);
    for (int i = 0; i < p.nslots; ++i) { tc::mbar_init(&s_full[i], 1); tc::mbar_init(&s_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&tm_full[i], 1); tc::mbar_init(&tm_empty[i], 4); }
    tc::fence_barrier_init();
  }
  if (warp == 5) {
    tc::tmem_alloc(tmem_ptr, p.tmem_cols);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const long long total = (long long)p.B * p.nxt * p.nyt * p.nzb;
  const int i_begin = (int)(total * blockIdx.x / gridDim.x), i_end = (int)(total * (blockIdx.x + 1) / gridDim.x);
  auto decode = [&](int it, int &b, int &x0, int &xlen, int &y0, int &ylen, int &z0) {
    const int zb = it % p.nzb; it /= p.nzb;
    const int yt = it % p.nyt; it /= p.nyt;
    const int xt = it % p.nxt;
    b = it / p.nxt;
    x0 = xt * p.Xt; xlen = min(p.Xt, p.Xo - x0);
    y0 = yt * p.Yt; ylen = min(p.Yt, p.Yo - y0);
    z0 = zb * 4;
  };

  if (warp == 4) {
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmA);
      tc::mbar_expect_tx(b_ready, kD1Tiles * kD1TileBytes);
      tc::bulk_g2s(bres, wT, kD1Tiles * kD1TileBytes, b_ready);
      uint32_t e = 0;
      for (int it = i_begin; it < i_end; ++it) {
        int b, x0, xlen, y0, ylen, z0;
        decode(it, b, x0, xlen, y0, ylen, z0);
        for (int cls = 0; cls < 4; ++cls, ++e) {  // cls = ex*2 + ey: sub-grid of input x = 2x - 1 + ex, y = 2y - 1 + ey
          const uint32_t slot = e % p.nslots, use = e / p.nslots;
          if (use > 0) tc::mbar_wait(&s_empty[slot], (use - 1) & 1);
          tc::mbar_expect_tx(&s_full[slot], 2 * p.box_bytes);
          uint8_t *dst = ring + (size_t)slot * p.slot_bytes;
          const int cx = 2 * x0 - 1 + (cls >> 1), cy = 2 * y0 - 1 + (cls & 1), cz = 2 * z0;  // copy column = z + 1
          tc::tma_load_4d(dst, &tmA, &s_full[slot], cz, cy, cx, b);
          tc::tma_load_4d(dst + (size_t)p.rows_alloc * 16, &tmA, &s_full[slot], cz + 8, cy, cx, b);
        }
      }
    }
  } else if (warp == 5) {
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(128, 32, 0, 0);
    const uint32_t ring_u32 = tc::smem_u32(ring), b_u32 = tc::smem_u32(bres);
    const uint64_t a_hi = tc::make_desc(0, (uint32_t)p.rows_alloc * 16, 128), b_hi = tc::make_desc(0, 32 * 16, 128);
    tc::mbar_wait(b_ready, 0);
    tc::tc_fence_after();
    uint32_t e = 0, acc = 0;
    for (int it = i_begin; it < i_end; ++it, ++acc) {
      const uint32_t q = acc & 1, uq = acc >> 1;
      if (uq > 0) tc::mbar_wait(&tm_empty[q], (uq - 1) & 1);
      tc::tc_fence_after();
      const uint32_t d_base = tmem_base + q * (uint32_t)(MT * 32);
      for (int cls = 0; cls < 4; ++cls, ++e) {
        const uint32_t slot = e % p.nslots;
        tc::mbar_wait(&s_full[slot], (e / p.nslots) & 1);
        tc::tc_fence_after();
        const uint32_t a_slot = (ring_u32 + slot * p.slot_bytes) >> 4;
        if (leader) {
#pragma unroll
          for (int t = 0; t < 4; ++t) {  // t = sx*2 + sy: taps dx = 2*sx + ex, dy = 2*sy + ey
            const uint64_t a0 = a_hi | (uint64_t)((a_slot + (uint32_t)((t >> 1) * p.Yh + (t & 1))) & 0x3FFF);
            const uint64_t b0 = b_hi | (uint64_t)(((b_u32 + (uint32_t)(cls * 4 + t) * kD1TileBytes) >> 4) & 0x3FFF);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
              tc::umma_bf16(d_base + mt * 32, a0 + (uint64_t)(mt * 128), b0, idesc, (uint32_t)((cls | t) != 0));
          }
          tc::umma_commit(&s_empty[slot]);
        }
        __syncwarp();
      }
      if (leader) tc::umma_commit(&tm_full[q]);
      __syncwarp();
    }
  } else {
    uint32_t acc = 0;
    for (int it = i_begin; it < i_end; ++it, ++acc) {
      int b, x0, xlen, y0, ylen, z0;
      decode(it, b, x0, xlen, y0, ylen, z0);
      const uint32_t q = acc & 1;
      tc::mbar_wait(&tm_full[q], (acc >> 1) & 1);
      tc::tc_fence_after();
      const uint32_t d_base = tmem_base + ((uint32_t)(warp * 32) << 16) + q * (uint32_t)(MT * 32);
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        const int r = mt * 128 + warp * 32 + lane;
        const int xx = r / p.Yh, yy = r - xx * p.Yh;
        const bool valid = xx < xlen && yy < ylen;
        bf16 *dst = out + ((((size_t)b * p.Xo + (x0 + xx)) * p.Yo + (y0 + yy)) * p.Zo + z0) * 8;
#pragma unroll
        for (int h = 0; h < 2; ++h) {  // 16 columns = output z (z0 + 2h, z0 + 2h + 1) x 8 channels
          uint32_t v[16];
          tc::tmem_ld16(d_base + (uint32_t)(mt * 32 + h * 16), v);
          tc::tmem_ld_wait();
          if (valid) {
            uint32_t pk[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              __nv_bfloat162 hh = __floats2bfloat162_rn(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
              pk[j] = *reinterpret_cast<uint32_t *>(&hh);
            }
            uint4 *d4 = reinterpret_cast<uint4 *>(dst + h * 16);
            if (z0 + 2 * h < p.Zo) d4[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            if (z0 + 2 * h + 1 < p.Zo) d4[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
          }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&tm_empty[q]);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 5) tc::tmem_dealloc(tmem_base, p.tmem_cols);
}

// tile (cls = ex*2+ey, t = sx*2+sy): T[zi/8][n = zo*8 + co][zi%8] = W[dx = 2sx+ex][dy = 2sy+ey][dz = zi - 2zo][co], 0 <= dz < 4
__global__ void d1_toeplitz_kernel(const bf16 *__restrict__ wp, bf16 *__restrict__ wt) {
  const int total = kD1Tiles * 2 * 32 * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int z8 = i & 7;
    int t = i >> 3;
    const int n = t & 31; t >>= 5;
    const int chunk = t & 1;
    const int tile = t >> 1;
    const int cls = tile >> 2, tt = tile & 3;
    const int dx = 2 * (tt >> 1) + (cls >> 1), dy = 2 * (tt & 1) + (cls & 1);
    const int zi = chunk * 8 + z8, zo = n >> 3, co = n & 7, dz = zi - 2 * zo;
    bf16 v = __float2bfloat16_rn(0.f);
    if (dz >= 0 && dz < 4) v = wp[(size_t)((dx * 4 + dy) * 4 + dz) * 8 + co];
    wt[i] = v;
  }
}

// copy[row][c] = in[row][c - 1] (0 outside), c in [0, Zc): makes every z window start (2*z0 - 1) a multiple of 8 columns
__global__ void __launch_bounds__(256)
d1_shift_copy_kernel(const bf16 *__restrict__ in, bf16 *__restrict__ out, long long rows, int Z, int Zc) {
  extern __shared__ uint16_t lines[];  // one warp per line (8 lines per block): line[c] = in[c - 1]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint16_t *line = lines + (size_t)warp * Zc;
  const long long r = (long long)blockIdx.x * 8 + warp;
  if (r >= rows) return;
  const uint16_t *src = reinterpret_cast<const uint16_t *>(in) + r * Z;
  for (int i = lane; i < Zc; i += 32) {
    const int z = i - 1;
    line[i] = (z >= 0 && z < Z) ? src[z] : (uint16_t)0;
  }
  __syncwarp();
  for (int j = lane; j < (Zc >> 3); j += 32) {
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = (uint32_t)line[j * 8 + 2 * k] | ((uint32_t)line[j * 8 + 2 * k + 1] << 16);
    reinterpret_cast<uint4 *>(out + r * Zc)[j] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

static bool plan_d1_gather(const cgan3d_conv_geom &g, D1GatherPlan &best) {
  if (!d1_shape(g)) return false;
  D1GatherPlan p{};
  p.B = g.B; p.Xi = g.Xb; p.Yi = g.Yb; p.Zi = g.Zb; p.Xo = g.Xs; p.Yo = g.Ys; p.Zo = g.Zs;
  p.Zc = round_up(p.Zi + 17, 8);
  p.nzb = (p.Zo + 3) / 4;
  const uint32_t fixed = kD1Tiles * kD1TileBytes + 512;
  double best_score = 0;
  bool found = false;
  for (int nyt = 1; nyt <= p.Yo && nyt <= 16; ++nyt) {
    const int Yt = (p.Yo + nyt - 1) / nyt, Yh = Yt + 1;
    if ((p.Yo + Yt - 1) / Yt != nyt || 2 * (Yh - 1) + 1 > 256) continue;
    for (int mt = 1; mt <= 4; ++mt) {
      if (Yt > mt * 128) continue;
      const int Xt = mn(p.Xo, (mt * 128 - Yt) / Yh + 1), Xh = Xt + 1;
      if (2 * (Xh - 1) + 1 > 256) continue;
      const int rows_alloc = round_up(mx(Xh * Yh, mt * 128 + Yh + 1), 8);
      const uint32_t slot = 2u * rows_alloc * 16;
      const int nslots = (int)mn<uint32_t>(8, (kSmemLimitD1 - fixed) / slot);
      if (nslots < 4) continue;
      const int nxt = (p.Xo + Xt - 1) / Xt;
      const double eff = (double)p.Xo * p.Yo / ((double)nxt * nyt * mt * 128);
      const double halo = (double)(Xh * Yh) / (Xt * Yt);
      const double score = eff / (1.0 + 0.05 * halo);
      if (score > best_score + 1e-9) {
        best_score = score; found = true;
        best = p;
        best.Xt = Xt; best.Yt = Yt; best.Xh = Xh; best.Yh = Yh; best.nxt = nxt; best.nyt = nyt; best.mtiles = mt;
        best.rows_alloc = rows_alloc; best.slot_bytes = slot; best.nslots = nslots;
      }
    }
  }
  if (!found) return false;
  best.box_bytes = 16u * best.Yh * best.Xh;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * best.mtiles * 32)) cols <<= 1;
  best.tmem_cols = cols;
  best.smem_bytes = fixed + best.nslots * best.slot_bytes;
  return true;
}

bool d1_gather_query(const cgan3d_conv_geom &g, int, TcQuery &q) {
  D1GatherPlan p;
  if (!plan_d1_gather(g, p)) return false;
  q = {(size_t)kD1Tiles * kD1TileBytes + 256 + (size_t)p.B * p.Xi * p.Yi * p.Zc * 2 + 256, false};
  return true;
}

int d1_gather_run(const cgan3d_conv_geom &g, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st) {
  D1GatherPlan p;
  if (!plan_d1_gather(g, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 critic-first conv: shape not supported");
  if ((reinterpret_cast<uintptr_t>(outp) & 15) || (reinterpret_cast<uintptr_t>(ws) & 255))
    return fail(CGAN3D_E_ARG, "tcgen05 critic-first conv: pointers must be 16-byte aligned (workspace 256)");
  bf16 *wt = reinterpret_cast<bf16 *>(ws);
  d1_toeplitz_kernel<<<32, 256, 0, st>>>(reinterpret_cast<const bf16 *>(wp), wt);
  CG_LAUNCH_CHECK("d1_toeplitz");
  bf16 *cp = reinterpret_cast<bf16 *>(reinterpret_cast<uint8_t *>(ws) + (size_t)kD1Tiles * kD1TileBytes + 256);
  const long long rows = (long long)p.B * p.Xi * p.Yi;
  d1_shift_copy_kernel<<<(unsigned)((rows + 7) / 8), 256, (size_t)8 * p.Zc * 2, st>>>(reinterpret_cast<const bf16 *>(in), cp, rows, p.Zi,
                                                                                     p.Zc);
  CG_LAUNCH_CHECK("d1_shift_copy");
  CUtensorMap tm;
  const cuuint64_t zc = (cuuint64_t)p.Zc;
  const cuuint64_t gdim[4] = {zc, (cuuint64_t)p.Yi, (cuuint64_t)p.Xi, (cuuint64_t)p.B};
  const cuuint64_t gstr[3] = {zc * 2, (cuuint64_t)p.Yi * zc * 2, (cuuint64_t)p.Xi * p.Yi * zc * 2};
  const cuuint32_t box[4] = {8, (cuuint32_t)(2 * (p.Yh - 1) + 1), (cuuint32_t)(2 * (p.Xh - 1) + 1), 1};
  const cuuint32_t estr[4] = {1, 2, 2, 1};
  int r = encode_tiled(&tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, cp, gdim, gstr, box, estr, CU_TENSOR_MAP_SWIZZLE_NONE, "critic first layer");
  if (r) return r;
  const long long total = (long long)p.B * p.nxt * p.nyt * p.nzb;
  const int grid = (int)mn<long long>(total, (long long)num_sms());
  auto launch = [&](auto mt_tag) -> int {
    constexpr int MT = decltype(mt_tag)::value;
    return tc_launch<d1_gather_tc_kernel<MT>>("d1_gather_tc_kernel", grid, 192, p.smem_bytes + 1024, 1, st, tm, wt,
                                              reinterpret_cast<bf16 *>(outp), p);
  };
  switch (p.mtiles) {
    case 1: return launch(std::integral_constant<int, 1>{});
    case 2: return launch(std::integral_constant<int, 2>{});
    case 3: return launch(std::integral_constant<int, 3>{});
    case 4: return launch(std::integral_constant<int, 4>{});
    default: return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 critic-first conv: mtiles %d not built", p.mtiles);
  }
}

// ================================================================================================================ wgrad
struct D1WgradPlan {
  int B, Xi, Yi, Zi, Xs, Ys, Zs;
  int Ye;  // lines of E per x plane (= Ys + 1)
  int Zt, nzt, Yt, nyt, rows, kblocks, stages;
  uint32_t chunk_bytes, stage_bytes, smem_bytes;
};

__global__ void __launch_bounds__(192, 1)
d1_wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmE, const __grid_constant__ CUtensorMap tmS, float *__restrict__ dw,
                   const __grid_constant__ D1WgradPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t *full = bars, *empty = bars + p.stages, *done = bars + 2 * p.stages;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); }
    tc::mbar_init(done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 5) {
    tc::tmem_alloc(tmem_ptr, 32);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // steps: (b, ox, y-tile, z-tile), split evenly
  const long long total = (long long)p.B * p.Xs * p.nyt * p.nzt;
  const int s_begin = (int)(total * blockIdx.x / gridDim.x), s_end = (int)(total * (blockIdx.x + 1) / gridDim.x);

  if (warp == 4) {
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmE);
      tc::tma_prefetch_desc(&tmS);
      for (int st = s_begin, n = 0; st < s_end; ++st, ++n) {
        int t = st;
        const int zt = t % p.nzt; t /= p.nzt;
        const int yt = t % p.nyt; t /= p.nyt;
        const int ox = t % p.Xs;
        const int b = t / p.Xs;
        const int y0 = yt * p.Yt, z0 = zt * p.Zt;
        const uint32_t s = n % p.stages, use = n / p.stages;
        if (use > 0) tc::mbar_wait(&empty[s], (use - 1) & 1);
        tc::mbar_expect_tx(&full[s], 9 * p.chunk_bytes);
        uint8_t *base = smem + (size_t)s * p.stage_bytes;
        for (int m8 = 0; m8 < 8; ++m8)  // chunk (dxi = m8 >> 1, s = m8 & 1): E plane 2*ox + dxi - 1, lines oy + s
          tc::tma_load_5d(base + (size_t)m8 * p.chunk_bytes, &tmE, &full[s], 0, z0, y0 + (m8 & 1), 2 * ox + (m8 >> 1) - 1, b);
        tc::tma_load_5d(base + (size_t)8 * p.chunk_bytes, &tmS, &full[s], 0, z0, y0, ox, b);
      }
    }
  } else if (warp == 5) {
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(64, 8, 1, 1);
    const uint64_t a_hi = tc::make_desc(0, 128, p.chunk_bytes), b_hi = tc::make_desc(0, 128, p.chunk_bytes);
    const uint32_t s0 = tc::smem_u32(smem);
    for (int st = s_begin, n = 0; st < s_end; ++st, ++n) {
      const uint32_t s = n % p.stages;
      tc::mbar_wait(&full[s], (n / p.stages) & 1);
      tc::tc_fence_after();
      if (leader) {
        uint64_t a_desc = a_hi | (uint64_t)(((s0 + s * p.stage_bytes) >> 4) & 0x3FFF);
        uint64_t b_desc = b_hi | (uint64_t)(((s0 + s * p.stage_bytes + 8 * p.chunk_bytes) >> 4) & 0x3FFF);
        tc::umma_bf16(tmem_base, a_desc, b_desc, idesc, n != 0 ? 1u : 0u);
#pragma unroll 4
        for (int kb = 1; kb < p.kblocks; ++kb) {
          a_desc += 16;
          b_desc += 16;
          tc::umma_bf16(tmem_base, a_desc, b_desc, idesc, 1u);
        }
        tc::umma_commit(&empty[s]);
      }
      __syncwarp();
    }
    if (leader) tc::umma_commit(done);
    __syncwarp();
  } else if (s_end > s_begin) {
    // M = 64 accumulator rows 16w..16w+15 live in TMEM lanes 32w..32w+15; 8 columns = output channels
    tc::mbar_wait(done, 0);
    tc::tc_fence_after();
    uint32_t v[8];
    tc::tmem_ld8(tmem_base + ((uint32_t)(warp * 32) << 16), v);
    tc::tmem_ld_wait();
    if (lane < 16) {
      const int m = warp * 16 + lane, m8 = m >> 3, j = m & 7;
      const int dx = m8 >> 1, dy = 2 * (m8 & 1) + (j >> 2), dz = j & 3;
      const int tap = (dx * 4 + dy) * 4 + dz;
#pragma unroll
      for (int c = 0; c < 8; ++c) atomicAdd(&dw[(size_t)c * 64 + tap], __uint_as_float(v[c]));
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 5) tc::tmem_dealloc(tmem_base, 32);
}

// E[b][x][yy][oz][dyp*4 + dz] = in[b][x][2*yy - 1 + dyp][2*oz - 1 + dz]  (0 outside), yy in [0, Ys], oz in [0, Zs)
// One warp per (b, x, yy) output line (8 lines per block): the two source lines are staged in shared memory.
__global__ void __launch_bounds__(256)
d1_expand_kernel(const bf16 *__restrict__ in, bf16 *__restrict__ e, long long lines_total, int Xi, int Yi, int Zi, int Ye, int Zs) {
  extern __shared__ uint16_t lines[];  // per warp: two lines, line[dyp][1 + z] = in[.., 2*yy - 1 + dyp, z]; zeros outside
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = (2 * Zs + 2 + 7) & ~7;
  uint16_t *l0 = lines + (size_t)warp * 2 * n, *l1 = l0 + n;
  const long long r = (long long)blockIdx.x * 8 + warp;
  if (r >= lines_total) return;
  const int yy = (int)(r % Ye);
  const long long bx = r / Ye;  // b * Xi + x
  const int y0 = 2 * yy - 1, y1 = 2 * yy;
  const uint16_t *base = reinterpret_cast<const uint16_t *>(in) + (size_t)bx * Yi * Zi;
  const bool in0 = y0 >= 0 && y0 < Yi, in1 = y1 < Yi;
  for (int i = lane; i < n; i += 32) {
    const int z = i - 1;
    const bool zin = z >= 0 && z < Zi;
    l0[i] = (in0 && zin) ? base[(size_t)y0 * Zi + z] : (uint16_t)0;
    l1[i] = (in1 && zin) ? base[(size_t)y1 * Zi + z] : (uint16_t)0;
  }
  __syncwarp();
  uint4 *dst = reinterpret_cast<uint4 *>(e) + (size_t)r * Zs;
  for (int oz = lane; oz < Zs; oz += 32) {
    // j = dyp*4 + dz reads line[dyp][2*oz + dz]
    const uint32_t a0 = (uint32_t)l0[2 * oz] | ((uint32_t)l0[2 * oz + 1] << 16), a1 = (uint32_t)l0[2 * oz + 2] | ((uint32_t)l0[2 * oz + 3] << 16);
    const uint32_t b0 = (uint32_t)l1[2 * oz] | ((uint32_t)l1[2 * oz + 1] << 16), b1 = (uint32_t)l1[2 * oz + 2] | ((uint32_t)l1[2 * oz + 3] << 16);
    dst[oz] = make_uint4(a0, a1, b0, b1);
  }
}

static bool plan_d1_wgrad(const cgan3d_conv_geom &g, D1WgradPlan &p) {
  if (!d1_shape(g)) return false;
  p = D1WgradPlan{};
  p.B = g.B; p.Xi = g.Xb; p.Yi = g.Yb; p.Zi = g.Zb; p.Xs = g.Xs; p.Ys = g.Ys; p.Zs = g.Zs;
  p.Ye = p.Ys + 1;
  p.nzt = (p.Zs + 255) / 256;
  p.Zt = round_up((p.Zs + p.nzt - 1) / p.nzt, 16);
  if (p.Zt > 256) { p.nzt += 1; p.Zt = round_up((p.Zs + p.nzt - 1) / p.nzt, 16); }
  p.Yt = mx(1, mn(p.Ys, 512 / p.Zt));
  p.nyt = (p.Ys + p.Yt - 1) / p.Yt;
  p.rows = p.Yt * p.Zt;
  p.kblocks = p.rows / 16;
  p.chunk_bytes = (uint32_t)p.rows * 16;
  p.stage_bytes = 9 * p.chunk_bytes;
  p.stages = (int)mn<uint32_t>(4, (kSmemLimitD1 - 512) / p.stage_bytes);
  if (p.stages < 2) return false;
  p.smem_bytes = p.stages * p.stage_bytes + 512;
  return true;
}

bool d1_wgrad_query(const cgan3d_conv_geom &g, int, TcQuery &q) {
  D1WgradPlan p;
  if (!plan_d1_wgrad(g, p)) return false;
  q = {(size_t)p.B * p.Xi * p.Ye * p.Zs * 16 + 256, false};
  return true;
}

int d1_wgrad_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, void *ws, cudaStream_t st) {
  D1WgradPlan p;
  if (!plan_d1_wgrad(g, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 critic-first wgrad: shape not supported");
  if ((reinterpret_cast<uintptr_t>(small) & 15) || (reinterpret_cast<uintptr_t>(ws) & 15))
    return fail(CGAN3D_E_ARG, "tcgen05 critic-first wgrad: pointers must be 16-byte aligned");
  if (beta == 0.f) {
    cudaError_t e = cudaMemsetAsync(dw, 0, (size_t)8 * 64 * sizeof(float), st);
    if (e != cudaSuccess) return cuda_fail(e, "tcgen05 critic-first wgrad memset");
  }
  bf16 *E = reinterpret_cast<bf16 *>(ws);
  const long long elines = (long long)p.B * p.Xi * p.Ye;
  d1_expand_kernel<<<(unsigned)((elines + 7) / 8), 256, (size_t)8 * 2 * ((2 * p.Zs + 2 + 7) & ~7) * 2, st>>>(
      reinterpret_cast<const bf16 *>(big), E, elines, p.Xi, p.Yi, p.Zi, p.Ye, p.Zs);
  CG_LAUNCH_CHECK("d1_expand");
  CUtensorMap tmE, tmS;
  int r = encode_act_map(&tmE, E, 8, p.Zs, p.Ye, p.Xi, p.B, 8, p.Zt, p.Yt, 1, 1, 0, "critic first layer, expanded input");
  if (r) return r;
  r = encode_act_map(&tmS, small, 8, p.Zs, p.Ys, p.Xs, p.B, 8, p.Zt, p.Yt, 1, 1, 0, "critic first layer, 8 channels");
  if (r) return r;
  const long long total = (long long)p.B * p.Xs * p.nyt * p.nzt;
  const int grid = (int)mn<long long>(total, (long long)num_sms());
  return tc_launch<d1_wgrad_tc_kernel>("d1_wgrad_tc_kernel", grid, 192, p.smem_bytes + 1024, 1, st, tmE, tmS, dw, p);
}

// ============================================================================================================== scatter
struct D1ScatterPlan {
  int B, Xs, Ys, Zs, Xb, Yb, Zb;
  int Xg, Yg, Zg;  // grid extents (= small + 1): grid position g <-> small-side voxel o = g - 1
  int Zt, nzt, Zh, Yt, nyt, Yh;
  int mtiles, rows_alloc, nslots;
  uint32_t slot_bytes, box_bytes, tmem_cols, smem_bytes;
};
constexpr uint32_t kD1STileBytes = 512;  // [2 sz-chunks][16 n][8 co]

template <int MT>
__global__ void __launch_bounds__(192, 1)
d1_scatter_tc_kernel(const __grid_constant__ CUtensorMap tmA, const bf16 *__restrict__ wT, bf16 *__restrict__ out,
                     const __grid_constant__ D1ScatterPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *bres = smem;          // 4 tiles (sx, sy), 2 KB
  uint8_t *ring = smem + 2048;
  uint64_t *bars = reinterpret_cast<uint64_t *>(ring + (size_t)p.nslots * p.slot_bytes);
  uint64_t *b_ready = bars, *s_full = bars + 1, *s_empty = s_full + p.nslots;
  uint64_t *tm_full = s_empty + p.nslots, *tm_empty = tm_full + 2;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(tm_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    tc::mbar_init(b_ready, 1);
    for (int i = 0; i < p.nslots; ++i) { tc::mbar_init(&s_full[i], 1); tc::mbar_init(&s_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&tm_full[i], 1); tc::mbar_init(&tm_empty[i], 4); }
    tc::fence_barrier_init();
  }
  if (warp == 5) {
    tc::tmem_alloc(tmem_ptr, p.tmem_cols);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const long long total = (long long)p.B * p.Xg * p.nyt * p.nzt;
  const int i_begin = (int)(total * blockIdx.x / gridDim.x), i_end = (int)(total * (blockIdx.x + 1) / gridDim.x);
  auto decode = [&](int it, int &b, int &gx, int &y0, int &ylen, int &z0, int &zlen) {
    const int zt = it % p.nzt; it /= p.nzt;
    const int yt = it % p.nyt; it /= p.nyt;
    gx = it % p.Xg;
    b = it / p.Xg;
    y0 = yt * p.Yt; ylen = min(p.Yt, p.Yg - y0);
    z0 = zt * p.Zt; zlen = min(p.Zt, p.Zg - z0);
  };

  if (warp == 4) {
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmA);
      tc::mbar_expect_tx(b_ready, 4 * kD1STileBytes);
      tc::bulk_g2s(bres, wT, 4 * kD1STileBytes, b_ready);
      uint32_t e = 0;
      for (int it = i_begin; it < i_end; ++it) {
        int b, gx, y0, ylen, z0, zlen;
        decode(it, b, gx, y0, ylen, z0, zlen);
        for (int sx = 0; sx < 2; ++sx, ++e) {
          const uint32_t slot = e % p.nslots, use = e / p.nslots;
          if (use > 0) tc::mbar_wait(&s_empty[slot], (use - 1) & 1);
          tc::mbar_expect_tx(&s_full[slot], p.box_bytes);
          tc::tma_load_5d(ring + (size_t)slot * p.slot_bytes, &tmA, &s_full[slot], 0, z0 - 1, y0 - 1, gx - 1 + sx, b);
        }
      }
    }
  } else if (warp == 5) {
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(128, 16, 0, 0);
    const uint32_t ring_u32 = tc::smem_u32(ring), b_u32 = tc::smem_u32(bres);
    // K = 16: chunk 0 = the row itself, chunk 1 = the next row (the z-adjacent voxel): LBO = 16 bytes
    const uint64_t a_hi = tc::make_desc(0, 16, 128), b_hi = tc::make_desc(0, 16 * 16, 128);
    tc::mbar_wait(b_ready, 0);
    tc::tc_fence_after();
    uint32_t e = 0, acc = 0;
    for (int it = i_begin; it < i_end; ++it, ++acc) {
      const uint32_t q = acc & 1, uq = acc >> 1;
      if (uq > 0) tc::mbar_wait(&tm_empty[q], (uq - 1) & 1);
      tc::tc_fence_after();
      const uint32_t d_base = tmem_base + q * (uint32_t)(MT * 16);
      for (int sx = 0; sx < 2; ++sx, ++e) {
        const uint32_t slot = e % p.nslots;
        tc::mbar_wait(&s_full[slot], (e / p.nslots) & 1);
        tc::tc_fence_after();
        const uint32_t a_slot = (ring_u32 + slot * p.slot_bytes) >> 4;
        if (leader) {
#pragma unroll
          for (int sy = 0; sy < 2; ++sy) {
            const uint64_t a0 = a_hi | (uint64_t)((a_slot + (uint32_t)(sy * p.Zh)) & 0x3FFF);
            const uint64_t b0 = b_hi | (uint64_t)(((b_u32 + (uint32_t)(sx * 2 + sy) * kD1STileBytes) >> 4) & 0x3FFF);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
              tc::umma_bf16(d_base + mt * 16, a0 + (uint64_t)(mt * 128), b0, idesc, (uint32_t)((sx | sy) != 0));
          }
          tc::umma_commit(&s_empty[slot]);
        }
        __syncwarp();
      }
      if (leader) tc::umma_commit(&tm_full[q]);
      __syncwarp();
    }
  } else {
    uint32_t acc = 0;
    for (int it = i_begin; it < i_end; ++it, ++acc) {
      int b, gx, y0, ylen, z0, zlen;
      decode(it, b, gx, y0, ylen, z0, zlen);
      const uint32_t q = acc & 1;
      tc::mbar_wait(&tm_full[q], (acc >> 1) & 1);
      tc::tc_fence_after();
      const uint32_t d_base = tmem_base + ((uint32_t)(warp * 32) << 16) + q * (uint32_t)(MT * 16);
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        const int r = mt * 128 + warp * 32 + lane;
        const int yy = r / p.Zh, zz = r - yy * p.Zh;
        uint32_t v[8];
        tc::tmem_ld8(d_base + (uint32_t)(mt * 16), v);
        tc::tmem_ld_wait();
        if (yy < ylen && zz < zlen) {
          // column n = (ux*2 + uy)*2 + uz is output voxel 2g - 1 + u
          const int ux0 = 2 * gx - 1, uy0 = 2 * (y0 + yy) - 1, uz0 = 2 * (z0 + zz) - 1;
#pragma unroll
          for (int n = 0; n < 8; ++n) {
            const int ux = ux0 + (n >> 2), uy = uy0 + ((n >> 1) & 1), uz = uz0 + (n & 1);
            if ((unsigned)ux < (unsigned)p.Xb && (unsigned)uy < (unsigned)p.Yb && (unsigned)uz < (unsigned)p.Zb)
              out[(((size_t)b * p.Xb + ux) * p.Yb + uy) * p.Zb + uz] = __float2bfloat16_rn(__uint_as_float(v[n]));
          }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&tm_empty[q]);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 5) tc::tmem_dealloc(tmem_base, p.tmem_cols);
}

// tile (sx, sy): T[sz][n = (ux*2+uy)*2+uz][co] = W[dx = ux + 2 - 2sx][dy = uy + 2 - 2sy][dz = uz + 2 - 2sz][co], n < 8, else 0
__global__ void d1_scatter_tiles_kernel(const bf16 *__restrict__ wp, bf16 *__restrict__ wt) {
  const int total = 4 * 2 * 16 * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int co = i & 7;
    int t = i >> 3;
    const int n = t & 15; t >>= 4;
    const int sz = t & 1;
    const int tile = t >> 1, sx = tile >> 1, sy = tile & 1;
    bf16 v = __float2bfloat16_rn(0.f);
    if (n < 8) {
      const int dx = (n >> 2) + 2 - 2 * sx, dy = ((n >> 1) & 1) + 2 - 2 * sy, dz = (n & 1) + 2 - 2 * sz;
      v = wp[(size_t)((dx * 4 + dy) * 4 + dz) * 8 + co];
    }
    wt[i] = v;
  }
}

static bool plan_d1_scatter(const cgan3d_conv_geom &g, D1ScatterPlan &best) {
  if (!d1_shape(g)) return false;
  D1ScatterPlan p{};
  p.B = g.B; p.Xs = g.Xs; p.Ys = g.Ys; p.Zs = g.Zs; p.Xb = g.Xb; p.Yb = g.Yb; p.Zb = g.Zb;
  p.Xg = g.Xs + 1; p.Yg = g.Ys + 1; p.Zg = g.Zs + 1;
  double best_score = 0;
  bool found = false;
  for (int nzt = 1; nzt <= 4; ++nzt) {
    const int Zt = (p.Zg + nzt - 1) / nzt, Zh = Zt + 1;
    if ((p.Zg + Zt - 1) / Zt != nzt || Zh > 256) continue;
    for (int Yt = 1; Yt <= p.Yg && Yt + 1 <= 256; ++Yt) {
      const int Yh = Yt + 1;
      const int mt = ((Yt - 1) * Zh + Zt + 127) / 128;
      if (mt > 4) break;
      const int rows_alloc = round_up(mx(Yh * Zh, mt * 128 + Zh + 2), 8);
      const uint32_t slot = (uint32_t)rows_alloc * 16;
      const int nslots = (int)mn<uint32_t>(8, (kSmemLimitD1 - 2048 - 512) / slot);
      if (nslots < 4) break;
      const int nyt = (p.Yg + Yt - 1) / Yt;
      const double eff = (double)p.Yg * p.Zg / ((double)nyt * nzt * mt * 128);
      if (eff > best_score + 1e-9) {
        best_score = eff; found = true;
        best = p;
        best.nzt = nzt; best.Zt = Zt; best.Zh = Zh; best.Yt = Yt; best.Yh = Yh; best.nyt = nyt; best.mtiles = mt;
        best.rows_alloc = rows_alloc; best.slot_bytes = slot; best.nslots = nslots;
      }
    }
  }
  if (!found) return false;
  best.box_bytes = 16u * best.Zh * best.Yh;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * best.mtiles * 16)) cols <<= 1;
  best.tmem_cols = cols;
  best.smem_bytes = 2048 + 512 + best.nslots * best.slot_bytes;
  return true;
}

bool d1_scatter_query(const cgan3d_conv_geom &g, int, TcQuery &q) {
  D1ScatterPlan p;
  if (!plan_d1_scatter(g, p)) return false;
  q = {4 * kD1STileBytes + 256, false};
  return true;
}

int d1_scatter_run(const cgan3d_conv_geom &g, const void *small, const void *wp, void *outp, void *ws, cudaStream_t st) {
  D1ScatterPlan p;
  if (!plan_d1_scatter(g, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 critic-first dgrad: shape not supported");
  if ((reinterpret_cast<uintptr_t>(small) & 15) || (reinterpret_cast<uintptr_t>(ws) & 15))
    return fail(CGAN3D_E_ARG, "tcgen05 critic-first dgrad: pointers must be 16-byte aligned");
  bf16 *wt = reinterpret_cast<bf16 *>(ws);
  d1_scatter_tiles_kernel<<<4, 256, 0, st>>>(reinterpret_cast<const bf16 *>(wp), wt);
  CG_LAUNCH_CHECK("d1_scatter_tiles");
  CUtensorMap tm;
  int r = encode_act_map(&tm, small, 8, p.Zs, p.Ys, p.Xs, p.B, 8, p.Zh, p.Yh, 1, 1, 0, "critic first layer");
  if (r) return r;
  const long long total = (long long)p.B * p.Xg * p.nyt * p.nzt;
  const int grid = (int)mn<long long>(total, (long long)num_sms());
  auto launch = [&](auto mt_tag) -> int {
    constexpr int MT = decltype(mt_tag)::value;
    return tc_launch<d1_scatter_tc_kernel<MT>>("d1_scatter_tc_kernel", grid, 192, p.smem_bytes + 1024, 1, st, tm, wt,
                                               reinterpret_cast<bf16 *>(outp), p);
  };
  switch (p.mtiles) {
    case 1: return launch(std::integral_constant<int, 1>{});
    case 2: return launch(std::integral_constant<int, 2>{});
    case 3: return launch(std::integral_constant<int, 3>{});
    case 4: return launch(std::integral_constant<int, 4>{});
    default: return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 critic-first dgrad: mtiles %d not built", p.mtiles);
  }
}

}  // namespace cg
