// tcgen05 weight-gradient kernels (bf16 operands, fp32 accumulation in TMEM, fp32 result).
// dW[cs][cb][tap] = sum_o small[o][cs] * big[stride*o - pad + tap][cb]  — reference aten::convolution_backward(weight)
// for nn.Conv3d and nn.ConvTranspose3d alike (model/blocks.py:29-38; generator.py:40-76; discriminator.py:48-67).
//
//   * GEMM view per tap: D[cs, cb] with M = 64, N = Cb, K = voxels of the small grid.  Both operands keep the
//     channels-last activation layout [C/8][row][8 ch] in shared memory, i.e. they are MN-major UMMA operands
//     (a core matrix is 8 voxels x 8 channels); rows are the flattened (y, z) positions of a small-grid slab with the
//     slab pitch Zh, and a filter tap is a ROW SHIFT of the big-side operand (as in conv_tc.cu).
//   * stride 1 (k = 3): one big-side halo slab per step, 9 (dy,dz) taps.  stride 2 (k = 3, 4): the big side is fetched
//     as 4 parity-class sub-slabs with TMA elementStrides (1,2,2,1,1) (as in conv_tc_prog.cu).
//   * Cs == 64: M = 64 rows are the 64 channels.  Cs == 32: the small-side slab is loaded TWICE, the second copy one
//     row (one voxel along z) later, so that rows 32..63 of D pair dY[r-1] with X[r+s] == the tap with shift s+1:
//     one MMA then produces two z-adjacent taps.
//     Cs == 16: four copies, shifted by (0|1 line, 0|1 voxel): one MMA produces a 2x2 block of (dy, dz) taps.
//   * A CTA owns one dx (filter x-offset) and a contiguous range of (b, y-slab, x) steps; M = 64 accumulators are
//     interleaved two per N TMEM columns; split-K over CTAs, partial sums added with red.global.add.f32.
#include "common.cuh"
#include "conv_internal.cuh"
#include "tc_common.cuh"

namespace cg {

constexpr uint32_t kSmemLimitWg = kMaxDynSmem - 1024;
constexpr int kMaxWgMma = 16, kMaxWgSrc = 4;

struct WgMma {
  uint16_t row_shift;
  uint8_t src, acc;
};
struct WgPlan {
  int B, X, Y, Z;       // small grid
  int Cb, Cs, k, stride, taps;
  int Zh, Yt, Yh, nslabs;
  int kpad, rowsA, rowsB;
  int ncopies;          // 1 (Cs == 64), 2 (Cs == 32: second copy one row later) or 4 (Cs == 16: 2x2 line/row shifts)
  int nsrc, nmma, nacc;
  int steps_per_dx, stages;
  int8_t src_cy[kMaxWgSrc], src_cz[kMaxWgSrc];
  WgMma mma[kMaxWgMma];
  int8_t acc_tap[kMaxWgMma][4];  // (dy*k+dz) produced by each 64/ncopies-row group of D (all equal when ncopies == 1); -1 = discard
  uint32_t a_bytes, b_bytes, boxA_bytes, boxB_bytes, stage_bytes, smem_bytes, tmem_cols;
};

__global__ void __launch_bounds__(192, 1)
wgrad_prog_tc_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmX, float *__restrict__ dw,
                     const __grid_constant__ WgPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *stage_mem = smem;
  uint64_t *bars = reinterpret_cast<uint64_t *>(stage_mem + (size_t)p.stages * p.stage_bytes);
  uint64_t *full = bars, *empty = bars + p.stages, *done = bars + 2 * p.stages;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // zero the staging buffers once: rows that TMA never writes (K padding, tail of the shifted reads) must read as 0
  {
    uint4 *z = reinterpret_cast<uint4 *>(stage_mem);
    const uint32_t n16 = (uint32_t)p.stages * p.stage_bytes / 16;
    for (uint32_t i = threadIdx.x; i < n16; i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { tc::mbar_init(&full[i], 1); tc::mbar_init(&empty[i], 1); }
    tc::mbar_init(done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 5) {
    tc::tmem_alloc(tmem_ptr, p.tmem_cols);
    tc::tmem_relinquish();
  }
  tc::fence_proxy_async();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // work split: blockIdx.x % k selects dx; the CTAs of one dx share its steps evenly
  const int dx = blockIdx.x % p.k;
  const int grp = blockIdx.x / p.k, ngrp = (gridDim.x - dx + p.k - 1) / p.k;
  const int s_begin = (int)((long long)p.steps_per_dx * grp / ngrp), s_end = (int)((long long)p.steps_per_dx * (grp + 1) / ngrp);
  const int kch_a = p.Cs >> 3, kch_b = p.Cb >> 3;

  if (warp == 4) {
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmY);
      tc::tma_prefetch_desc(&tmX);
      for (int st = s_begin, n = 0; st < s_end; ++st, ++n) {
        int t = st;
        const int x = t % p.X; t /= p.X;
        const int sl = t % p.nslabs;
        const int b = t / p.nslabs;
        const int y0 = sl * p.Yt;
        const uint32_t s = n % p.stages, use = n / p.stages;
        if (use > 0) tc::mbar_wait(&empty[s], (use - 1) & 1);
        tc::mbar_expect_tx(&full[s], p.boxA_bytes * kch_a * p.ncopies + p.boxB_bytes * kch_b * p.nsrc);
        uint8_t *a = stage_mem + (size_t)s * p.stage_bytes, *bb = a + p.a_bytes;
        for (int c = 0; c < p.ncopies; ++c)
          for (int cc = 0; cc < kch_a; ++cc)
            tc::tma_load_5d(a + (size_t)(c * kch_a + cc) * p.rowsA * 16, &tmY, &full[s], cc * 8, -(c & 1), y0 - (c >> 1), x, b);
        for (int sr = 0; sr < p.nsrc; ++sr)
          for (int cc = 0; cc < kch_b; ++cc)
            tc::tma_load_5d(bb + (size_t)(sr * kch_b + cc) * p.rowsB * 16, &tmX, &full[s], cc * 8, p.src_cz[sr],
                            p.stride * y0 + p.src_cy[sr], p.stride * x + dx - 1, b);
      }
    }
  } else if (warp == 5) {
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(64, p.Cb, 1, 1);
    const uint32_t a_sbo = (uint32_t)p.rowsA * 16, b_sbo = (uint32_t)p.rowsB * 16;
    const uint64_t a_hi = tc::make_desc(0, 128, a_sbo), b_hi = tc::make_desc(0, 128, b_sbo);
    const uint32_t stage0 = tc::smem_u32(stage_mem);
    const int kblocks = p.kpad >> 4;
    for (int st = s_begin, n = 0; st < s_end; ++st, ++n) {
      const uint32_t s = n % p.stages;
      tc::mbar_wait(&full[s], (n / p.stages) & 1);
      tc::tc_fence_after();
      const uint32_t a0 = (stage0 + s * p.stage_bytes) >> 4, b0 = (stage0 + s * p.stage_bytes + p.a_bytes) >> 4;
      if (leader) {
        // tap-major order: the per-tap constants stay in registers and the K loop is two descriptor adds per MMA
        for (int j = 0; j < p.nmma; ++j) {
          const WgMma &M = p.mma[j];
          const uint32_t d = tmem_base + (uint32_t)((M.acc >> 1) * p.Cb) + ((uint32_t)((M.acc & 1) * 16) << 16);
          uint64_t a_desc = a_hi | (uint64_t)(a0 & 0x3FFF);
          uint64_t b_desc = b_hi | (uint64_t)((b0 + (uint32_t)M.src * kch_b * p.rowsB + M.row_shift) & 0x3FFF);
          tc::umma_bf16(d, a_desc, b_desc, idesc, n != 0 ? 1u : 0u);
#pragma unroll 4
          for (int kb = 1; kb < kblocks; ++kb) {
            a_desc += 16;
            b_desc += 16;
            tc::umma_bf16(d, a_desc, b_desc, idesc, 1u);
          }
        }
      }
      if (leader) tc::umma_commit(&empty[s]);
      __syncwarp();
    }
    if (leader) tc::umma_commit(done);
    __syncwarp();
  } else {
    // epilogue: warps 0..3; TMEM lane 32*warp + l: l < 16 -> accumulator 2g row 16*warp + l, l >= 16 -> accumulator 2g+1
    if (s_end > s_begin) {
      tc::mbar_wait(done, 0);
      tc::tc_fence_after();
      const int m = warp * 16 + (lane & 15);                       // row of D
      const int cs = m % p.Cs;
      const int half = m / p.Cs;                                   // which shifted copy this row belongs to
      const int ngroups = (p.nacc + 1) >> 1;
      for (int g2 = 0; g2 < ngroups; ++g2) {
        const int j = g2 * 2 + (lane >> 4);
        const int t2 = j < p.nacc ? p.acc_tap[j][half] : -1;
        const int tap = dx * p.k * p.k + t2;
        for (int c0 = 0; c0 < p.Cb; c0 += 16) {
          uint32_t v[16];
          tc::tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(g2 * p.Cb + c0), v);
          tc::tmem_ld_wait();
          if (t2 >= 0) {
#pragma unroll
            for (int c = 0; c < 16; ++c)
              if (c0 + c < p.Cb) atomicAdd(&dw[((size_t)cs * p.Cb + (c0 + c)) * p.taps + tap], __uint_as_float(v[c]));
          }
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 5) tc::tmem_dealloc(tmem_base, p.tmem_cols);
}

static bool plan_wgrad(const cgan3d_conv_geom &g, WgPlan &p) {
  const int k = g.k, s = g.stride;
  if (g.pad != 1) return false;
  if (!((s == 1 && k == 3) || (s == 2 && (k == 3 || k == 4)))) return false;
  if (g.Cs != 64 && g.Cs != 32 && g.Cs != 16) return false;
  if (g.Cb % 8 || g.Cb < 8 || g.Cb > 64) return false;
  if (s == 1 && (g.Xb != g.Xs || g.Yb != g.Ys || g.Zb != g.Zs)) return false;
  p = WgPlan{};
  p.B = g.B; p.X = g.Xs; p.Y = g.Ys; p.Z = g.Zs; p.Cb = g.Cb; p.Cs = g.Cs; p.k = k; p.stride = s; p.taps = k * k * k;
  const int halo = s == 1 ? 2 : 1;
  p.Zh = p.Z + halo;
  if (s * (p.Zh - 1) + 1 > 256) return false;
  p.ncopies = 64 / g.Cs;
  p.stages = 2;
  // ---- MMA program for one (dx) plane
  int nm = 0, na = 0;
  auto add4 = [&](int src, int shift, int t0, int t1, int t2, int t3) {
    if (nm >= kMaxWgMma) { ++nm; return; }
    p.mma[nm].src = (uint8_t)src; p.mma[nm].row_shift = (uint16_t)shift; p.mma[nm].acc = (uint8_t)na;
    p.acc_tap[na][0] = (int8_t)t0; p.acc_tap[na][1] = (int8_t)t1; p.acc_tap[na][2] = (int8_t)t2; p.acc_tap[na][3] = (int8_t)t3;
    ++nm; ++na;
  };
  auto add = [&](int src, int shift, int tap0, int tap1) { add4(src, shift, tap0, tap1, tap0, tap1); };
  if (s == 1) {
    p.nsrc = 1; p.src_cy[0] = -1; p.src_cz[0] = -1;
    if (p.ncopies == 1) {
      for (int dy = 0; dy < 3; ++dy)
        for (int dz = 0; dz < 3; ++dz) add(0, dy * p.Zh + dz, dy * 3 + dz, dy * 3 + dz);
    } else if (p.ncopies == 2) {  // pairs (dz, dz+1): (0,1) and (2,-)
      for (int dy = 0; dy < 3; ++dy) { add(0, dy * p.Zh + 0, dy * 3 + 0, dy * 3 + 1); add(0, dy * p.Zh + 2, dy * 3 + 2, -1); }
    } else {  // 2x2 blocks of (dy, dz): copy (cy, cz) yields tap (dy0 + cy, dz0 + cz)
      for (int dy0 = 0; dy0 < 3; dy0 += 2)
        for (int dz0 = 0; dz0 < 3; dz0 += 2) {
          auto t = [&](int cy, int cz) { return (dy0 + cy < 3 && dz0 + cz < 3) ? (dy0 + cy) * 3 + dz0 + cz : -1; };
          add4(0, dy0 * p.Zh + dz0, t(0, 0), t(0, 1), t(1, 0), t(1, 1));
        }
    }
  } else {
    // parity classes as in conv_tc_prog.cu: class c of tap d = (d-1)&1, row shift = (d - 1 + c) / 2, slab start = 2*o - c
    p.nsrc = 4;
    auto cls = [](int d) { return (d - 1) & 1; };
    auto shf = [&](int d) { return (d - 1 + cls(d)) / 2; };
    for (int q = 0; q < 2; ++q)
      for (int r = 0; r < 2; ++r) {
        const int src = q * 2 + r;
        p.src_cy[src] = (int8_t)(-q); p.src_cz[src] = (int8_t)(-r);
        if (p.ncopies == 4) {
          // taps of this class along each axis, ordered by shift (1 or 2 of them); copy (cy, cz) <-> (dys[cy], dzs[cz])
          int dys[2], ny = 0, dzs4[2], nz4 = 0;
          for (int d = 0; d < k; ++d) { if (cls(d) == q) dys[ny++] = d; if (cls(d) == r) dzs4[nz4++] = d; }
          auto t = [&](int cy, int cz) { return (cy < ny && cz < nz4) ? dys[cy] * k + dzs4[cz] : -1; };
          add4(src, shf(dys[0]) * p.Zh + shf(dzs4[0]), t(0, 0), t(0, 1), t(1, 0), t(1, 1));
          continue;
        }
        for (int dy = 0; dy < k; ++dy) {
          if (cls(dy) != q) continue;
          // z taps of this class, ordered by shift
          int dzs[2], nz = 0;
          for (int dz = 0; dz < k; ++dz)
            if (cls(dz) == r) dzs[nz++] = dz;
          if (p.ncopies == 1) {
            for (int i = 0; i < nz; ++i) add(src, shf(dy) * p.Zh + shf(dzs[i]), dy * k + dzs[i], dy * k + dzs[i]);
          } else if (nz == 2) {  // shifts 0 and 1: one stacked MMA
            add(src, shf(dy) * p.Zh + shf(dzs[0]), dy * k + dzs[0], dy * k + dzs[1]);
          } else {
            add(src, shf(dy) * p.Zh + shf(dzs[0]), dy * k + dzs[0], -1);
          }
          if (nm > kMaxWgMma) return false;
        }
      }
  }
  p.nmma = nm; p.nacc = na;
  if (nm > kMaxWgMma) return false;
  const int ngroups = (na + 1) / 2;
  if (ngroups * g.Cb > 512) return false;
  // ---- slab height
  const int yh_extra = halo;
  bool ok = false;
  for (int Yt = mn(p.Y, 64); Yt >= 1; --Yt) {
    const int kpad = (Yt * p.Zh + 15) / 16 * 16;
    const int rowsA = kpad, rowsB = (kpad + halo * p.Zh + halo + 7) / 8 * 8;
    if (s * (Yt + yh_extra - 1) + 1 > 256) continue;
    if ((Yt + yh_extra) * p.Zh > rowsB) continue;
    const uint32_t a_bytes = (uint32_t)8 * rowsA * 16, b_bytes = (uint32_t)p.nsrc * (g.Cb / 8) * rowsB * 16;
    if (rowsB > 16383) continue;
    if ((size_t)p.stages * (a_bytes + b_bytes) + 512 > kSmemLimitWg) continue;
    p.Yt = Yt;
    ok = true;
    break;
  }
  if (!ok) return false;
  // with line-shifted copies the copy that starts one line earlier covers lines y0-1 .. y0+Yt-2: tile Y+1 lines
  const int ylines = p.Y + (p.ncopies == 4 ? 1 : 0);
  p.nslabs = (ylines + p.Yt - 1) / p.Yt;
  p.Yt = (ylines + p.nslabs - 1) / p.nslabs;  // balance the slabs
  p.Yh = p.Yt + yh_extra;
  p.kpad = (p.Yt * p.Zh + 15) / 16 * 16;
  p.rowsA = p.kpad;
  p.rowsB = (p.kpad + halo * p.Zh + halo + 7) / 8 * 8;
  p.a_bytes = (uint32_t)8 * p.rowsA * 16;
  p.b_bytes = (uint32_t)p.nsrc * (g.Cb / 8) * p.rowsB * 16;
  p.stage_bytes = p.a_bytes + p.b_bytes;
  p.boxA_bytes = 16u * p.Zh * p.Yt;
  p.boxB_bytes = 16u * p.Zh * p.Yh;
  p.smem_bytes = p.stages * p.stage_bytes + 512;
  p.steps_per_dx = p.B * p.nslabs * p.X;
  uint32_t cols = 32;
  while (cols < (uint32_t)(ngroups * g.Cb)) cols <<= 1;
  p.tmem_cols = cols;
  return true;
}

bool wgrad_prog_query(const cgan3d_conv_geom &g, int, TcQuery &q) {
  WgPlan p;
  if (!plan_wgrad(g, p)) return false;
  q = {0, false};
  return true;
}

int wgrad_prog_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st) {
  WgPlan p;
  if (!plan_wgrad(g, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 wgrad: shape not supported");
  if ((reinterpret_cast<uintptr_t>(big) & 15) || (reinterpret_cast<uintptr_t>(small) & 15))
    return fail(CGAN3D_E_ARG, "tcgen05 wgrad: pointers must be 16-byte aligned");
  if (beta == 0.f) {
    cudaError_t e = cudaMemsetAsync(dw, 0, (size_t)g.Cs * g.Cb * p.taps * sizeof(float), st);
    if (e != cudaSuccess) return cuda_fail(e, "tcgen05 wgrad memset");
  }
  CUtensorMap tmY, tmX;
  int r = encode_act_map(&tmY, small, g.Cs, g.Zs, g.Ys, g.Xs, g.B, 8, p.Zh, p.Yt, 1, 1, 0, "wgrad, small side");
  if (r) return r;
  r = encode_act_map(&tmX, big, g.Cb, g.Zb, g.Yb, g.Xb, g.B, 8, p.Zh, p.Yh, g.stride, g.stride, 0, "wgrad, big side");
  if (r) return r;
  const int grid = (int)mn<long long>((long long)p.k * p.steps_per_dx, (long long)(num_sms() / p.k) * p.k);
  return tc_launch<wgrad_prog_tc_kernel>("wgrad_prog_tc_kernel", grid, 192, p.smem_bytes + 1024, 1, st, tmY, tmX, dw, p);
}

}  // namespace cg
