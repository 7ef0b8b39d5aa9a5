// tcgen05 weight gradient of the STRIDE-2 convolutions with Cs in {32, 64} and Cb in {16, 32} (generator down/up-sampling
// layers, critic middle layers): dW[cs][cb][tap] = sum_o small[o][cs] * big[2*o - 1 + tap][cb]
// (aten::convolution_backward(weight) for nn.Conv3d and nn.ConvTranspose3d; reference model/generator.py:40-76,
// model/discriminator.py:48-67).  Second-generation layout of wgrad_tc.cu, driven by two measurements (DESIGN §4.0):
// the first kernel was bound by L2->SM traffic (16-byte TMA pieces fetch 32-byte sectors, the z-shifted operand copy and
// the per-dx CTA groups re-read both tensors) and by the flat ~65-cycle cost of its many N = 16 MMAs.
//
//   * Both operands stay channels-last and are loaded as WHOLE voxels: one TMA box per slab into a SWIZZLE_{32,64,128}B
//     MN-major layout (row = one voxel = 2*C bytes).  Swizzled UMMA operands may start at any row (the XOR pattern is a
//     function of the shared-memory address), so filter taps are still row shifts of the X operand.
//   * Cs == 32 fills M = 64 WITHOUT a second copy: the second 32-channel M block is the same dY slab one row later
//     (descriptor LBO = one row).  Block 0 / block 1 therefore pair dY[z-1] / dY[z] with the same X rows: two z-adjacent
//     taps per MMA.
//   * The 4 parity-class sub-slabs of X are adjacent N blocks: ONE MMA with N = 4*Cb covers every class at a row shift.
//     2 (Cs = 32) or 4 (Cs = 64) MMAs per K block and dx instead of 6-9.
//   * Cs == 64 runs M = 128 the same way: block 0 = dY[z-1], block 1 = dY[z].
//   * Stride 1 (the generator's ResNet layers, Cs = 64): the N blocks are the SAME X halo slab zero and two voxels later
//     (LBO = two rows), so one M = 128 MMA with N = 2*Cb yields the three dz taps of a (dx, dy) pair: 3 MMAs per K block
//     and dx instead of 9.
//   * A CTA owns one dx (filter x-offset) and a contiguous range of (b, y-slab, x) steps; split-K over CTAs, fp32 atomics.
#include "common.cuh"
#include "conv_internal.cuh"
#include "tc_common.cuh"

namespace cg {

constexpr uint32_t kSmemLimitWs = kMaxDynSmem - 2048;
constexpr int kMaxWsMma = 4;

struct WsPlan {
  int B, X, Y, Z;  // small grid
  int Cb, Cs, k, taps;
  int Zh, Yt, Yh, nslabs;
  int kpad, rowsA, rowsB;
  int stride;      // 2: N blocks = the 4 parity-class sub-slabs; 1: N blocks = 3 row-shifted views of one halo slab
  int nsrc, nblkB; // TMA sub-slabs of X per step / N blocks per MMA
  uint32_t lboB;   // bytes between N blocks
  int nmma, stages, steps_per_dx;
  uint16_t row_shift[kMaxWsMma];
  int8_t acc_tap[kMaxWsMma][2][4];  // (dy*k+dz) of [MMA][M block][N block]; -1 = discard
  uint32_t rowbytesA, rowbytesB, a_bytes, srcB_bytes, stage_bytes, boxA_bytes, boxB_bytes, smem_bytes, tmem_cols;
  int m128;  // Cs == 64: M = 128 = dY[z-1] | dY[z] (two z-adjacent taps per MMA); Cs == 32: M = 64, the same two M blocks
};

__global__ void __launch_bounds__(192, 1)
wgrad_s2_sw_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmX, float *__restrict__ dw,
                   const __grid_constant__ WsPlan p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *stage_mem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
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

  const int dx = blockIdx.x % p.k;
  const int grp = blockIdx.x / p.k, ngrp = (gridDim.x - dx + p.k - 1) / p.k;
  const int s_begin = (int)((long long)p.steps_per_dx * grp / ngrp), s_end = (int)((long long)p.steps_per_dx * (grp + 1) / ngrp);
  const int ncol = p.nblkB * p.Cb;

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
        tc::mbar_expect_tx(&full[s], p.boxA_bytes + p.nsrc * p.boxB_bytes);
        uint8_t *a = stage_mem + (size_t)s * p.stage_bytes, *bb = a + p.a_bytes;
        // dY slab, one voxel early so that M block 0 = dY[z-1] and block 1 (next row) = dY[z]
        tc::tma_load_5d(a, &tmY, &full[s], 0, -1, y0, x, b);
        if (p.stride == 2) {
          for (int src = 0; src < 4; ++src)  // parity class (q, r) = (src >> 1, src & 1): sub-slab starts at 2*o - class
            tc::tma_load_5d(bb + (size_t)src * p.srcB_bytes, &tmX, &full[s], 0, -(src & 1), 2 * y0 - (src >> 1), 2 * x + dx - 1, b);
        } else {
          tc::tma_load_5d(bb, &tmX, &full[s], 0, -1, y0 - 1, x + dx - 1, b);  // halo slab of plane x + dx - 1
        }
      }
    }
  } else if (warp == 5) {
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(p.m128 ? 128 : 64, ncol, 1, 1);
    const uint64_t a_hi = tc::make_desc_sw_mn(0, p.rowbytesA, 8 * p.rowbytesA, p.rowbytesA);
    const uint64_t b_hi = tc::make_desc_sw_mn(0, p.lboB, 8 * p.rowbytesB, p.rowbytesB);
    const uint32_t stage0 = tc::smem_u32(stage_mem);
    const int kblocks = p.kpad >> 4;
    const uint32_t a_step = (16 * p.rowbytesA) >> 4, b_step = (16 * p.rowbytesB) >> 4;
    for (int st = s_begin, n = 0; st < s_end; ++st, ++n) {
      const uint32_t s = n % p.stages;
      tc::mbar_wait(&full[s], (n / p.stages) & 1);
      tc::tc_fence_after();
      const uint32_t a0 = (stage0 + s * p.stage_bytes) >> 4, b0 = (stage0 + s * p.stage_bytes + p.a_bytes) >> 4;
      if (leader) {
        for (int j = 0; j < p.nmma; ++j) {
          const uint32_t d = p.m128 ? tmem_base + (uint32_t)(j * ncol) : tmem_base + (uint32_t)((j >> 1) * ncol) + ((uint32_t)((j & 1) * 16) << 16);
          uint64_t a_desc = a_hi | (uint64_t)(a0 & 0x3FFF);
          uint64_t b_desc = b_hi | (uint64_t)((b0 + ((uint32_t)p.row_shift[j] * p.rowbytesB >> 4)) & 0x3FFF);
          tc::umma_bf16(d, a_desc, b_desc, idesc, n != 0 ? 1u : 0u);
#pragma unroll 4
          for (int kb = 1; kb < kblocks; ++kb) {
            a_desc += a_step;
            b_desc += b_step;
            tc::umma_bf16(d, a_desc, b_desc, idesc, 1u);
          }
        }
        tc::umma_commit(&empty[s]);
      }
      __syncwarp();
    }
    if (leader) tc::umma_commit(done);
    __syncwarp();
  } else if (s_end > s_begin) {
    // epilogue: TMEM lane 32*warp + l: l < 16 -> accumulator 2g row 16*warp + l, l >= 16 -> accumulator 2g + 1
    tc::mbar_wait(done, 0);
    tc::tc_fence_after();
    float *dw_dx = dw + dx * p.k * p.k;  // this CTA's filter x-offset
    if (p.m128) {  // M = 128: TMEM lane 32*warp + l is accumulator row 32*warp + l = (block, channel)
      const int m = warp * 32 + lane;
      const int cs = m & 63, blk = m >> 6;
      for (int j = 0; j < p.nmma; ++j)
        for (int c0 = 0; c0 < ncol; c0 += 16) {
          uint32_t v[16];
          tc::tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(j * ncol + c0), v);
          tc::tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const int nn = c0 + c;
            const int src = nn / p.Cb, cb = nn - src * p.Cb;
            const int t2 = p.acc_tap[j][blk][src];
            if (t2 >= 0) atomicAdd(&dw_dx[((size_t)cs * p.Cb + cb) * p.taps + t2], __uint_as_float(v[c]));
          }
        }
    } else {
    const int m = warp * 16 + (lane & 15);
    const int cs = m % p.Cs, blk = m / p.Cs;
    const int ngroups = (p.nmma + 1) >> 1;
    for (int g2 = 0; g2 < ngroups; ++g2) {
      const int j = g2 * 2 + (lane >> 4);
      for (int c0 = 0; c0 < ncol; c0 += 16) {
        uint32_t v[16];
        tc::tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(g2 * ncol + c0), v);
        tc::tmem_ld_wait();
        if (j < p.nmma) {
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const int nn = c0 + c;
            const int src = nn / p.Cb, cb = nn - src * p.Cb;
            const int t2 = p.acc_tap[j][blk][src];
            if (t2 >= 0) atomicAdd(&dw_dx[((size_t)cs * p.Cb + cb) * p.taps + t2], __uint_as_float(v[c]));
          }
        }
      }
    }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 5) tc::tmem_dealloc(tmem_base, p.tmem_cols);
}

static bool plan_ws(const cgan3d_conv_geom &g, WsPlan &p) {
  const int k = g.k, s = g.stride;
  if (g.pad != 1) return false;
  if (s == 2) {
    if (k != 3 && k != 4) return false;
    if (g.Cs != 32 && g.Cs != 64) return false;
    if (g.Cb != 16 && g.Cb != 32) return false;
  } else if (s == 1) {
    if (k != 3 || g.Cs != 64) return false;
    if (g.Cb != 16 && g.Cb != 32 && g.Cb != 64) return false;
    if (g.Xb != g.Xs || g.Yb != g.Ys || g.Zb != g.Zs) return false;
  } else {
    return false;
  }
  p = WsPlan{};
  p.B = g.B; p.X = g.Xs; p.Y = g.Ys; p.Z = g.Zs; p.Cb = g.Cb; p.Cs = g.Cs; p.k = k; p.taps = k * k * k;
  p.stride = s;
  const int halo = s == 1 ? 2 : 1;
  p.Zh = p.Z + halo;
  if (s * (p.Zh - 1) + 1 > 256) return false;
  p.m128 = g.Cs == 64 ? 1 : 0;
  p.rowbytesA = 2u * g.Cs;
  p.rowbytesB = 2u * g.Cb;
  p.stages = 2;
  int nm = 0;
  if (s == 2) {
    p.nsrc = 4; p.nblkB = 4;
    // MMA program: sub-grid shift (sy, sz) in {0,1}^2; tap d has parity class (d-1)&1 and shift (d - 1 + class) / 2.  The two
    // M blocks cover both z shifts: block 0 holds dY[z-1] (z shift 1), block 1 holds dY[z] (z shift 0).
    auto cls = [](int d) { return (d - 1) & 1; };
    auto shf = [&](int d) { return (d - 1 + cls(d)) / 2; };
    auto find = [&](int c, int sh) { for (int d = 0; d < k; ++d) if (cls(d) == c && shf(d) == sh) return d; return -1; };
    for (int by = 0; by < 2; ++by) {
      bool any = false;
      for (int blk = 0; blk < 2; ++blk)
        for (int src = 0; src < 4; ++src) {
          int tap = -1;
          const int dy = find(src >> 1, by), dz = find(src & 1, 1 - blk);
          if (dy >= 0 && dz >= 0) tap = dy * k + dz;
          p.acc_tap[nm][blk][src] = (int8_t)tap;
          any = any || tap >= 0;
        }
      if (!any) continue;
      p.row_shift[nm] = (uint16_t)(by * p.Zh);
      ++nm;
    }
  } else {
    // M = 128: block 0 = dY[z-1], block 1 = dY[z] (the slab one row later); N blocks = the X halo slab 0 and 2 voxels later.
    // (block 1, shift s) is tap dz = s, (block 0, shift s) is tap dz = s + 1: dz = 0, 1, 2 from one MMA of N = 2*Cb, which
    // costs 84.5 cycles instead of the 96.9 of an M = 64, N = 3*Cb MMA that leaves half of the tensor rows idle.
    p.nsrc = 1; p.nblkB = 2;
    for (int dy = 0; dy < 3; ++dy) {
      for (int blk = 0; blk < 2; ++blk)
        for (int nb = 0; nb < 4; ++nb) {
          const int dz = nb < 2 ? (blk == 1 ? 2 * nb : 2 * nb + 1) : -1;
          p.acc_tap[nm][blk][nb] = (int8_t)((dz >= 0 && dz < 3) ? dy * 3 + dz : -1);
        }
      p.row_shift[nm] = (uint16_t)(dy * p.Zh);
      ++nm;
    }
  }
  p.nmma = nm;
  const int ngroups = p.m128 ? nm : (nm + 1) / 2;
  const int ncol = p.nblkB * g.Cb;
  if (ngroups * ncol > 512 || ncol > 256) return false;
  auto sizes = [&](int Yt, int &kpad, int &rowsA, int &rowsB) {
    kpad = (Yt * p.Zh + 15) / 16 * 16;
    rowsA = kpad + 8;
    rowsB = (kpad + halo * p.Zh + halo + 2 + 7) / 8 * 8;
  };
  bool ok = false;
  for (int Yt = mn(p.Y, 64); Yt >= 1; --Yt) {
    if (s * (Yt + halo - 1) + 1 > 256) continue;
    int kpad, rowsA, rowsB;
    sizes(Yt, kpad, rowsA, rowsB);
    if ((Yt + halo) * p.Zh > rowsB) continue;
    const uint32_t a_bytes = ((uint32_t)rowsA * p.rowbytesA + 1023) / 1024 * 1024;
    const uint32_t srcB = ((uint32_t)rowsB * p.rowbytesB + 1023) / 1024 * 1024;
    if ((size_t)p.stages * (a_bytes + p.nsrc * srcB) + 512 > kSmemLimitWs) continue;
    p.Yt = Yt;
    ok = true;
    break;
  }
  if (!ok) return false;
  p.nslabs = (p.Y + p.Yt - 1) / p.Yt;
  p.Yt = (p.Y + p.nslabs - 1) / p.nslabs;
  p.Yh = p.Yt + halo;
  sizes(p.Yt, p.kpad, p.rowsA, p.rowsB);
  p.a_bytes = ((uint32_t)p.rowsA * p.rowbytesA + 1023) / 1024 * 1024;
  p.srcB_bytes = ((uint32_t)p.rowsB * p.rowbytesB + 1023) / 1024 * 1024;
  p.lboB = s == 2 ? p.srcB_bytes : 2 * p.rowbytesB;
  p.stage_bytes = p.a_bytes + p.nsrc * p.srcB_bytes;
  p.boxA_bytes = p.rowbytesA * p.Zh * p.Yt;
  p.boxB_bytes = p.rowbytesB * p.Zh * p.Yh;
  p.smem_bytes = p.stages * p.stage_bytes + 512 + 1024;
  p.steps_per_dx = p.B * p.nslabs * p.X;
  uint32_t cols = 32;
  while (cols < (uint32_t)(ngroups * ncol)) cols <<= 1;
  p.tmem_cols = cols;
  return true;
}

bool wgrad_s2_query(const cgan3d_conv_geom &g, int, TcQuery &q) {
  WsPlan p;
  if (!plan_ws(g, p)) return false;
  q = {0, false};
  return true;
}

int wgrad_s2_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st) {
  WsPlan p;
  if (!plan_ws(g, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 strided wgrad: shape not supported");
  if ((reinterpret_cast<uintptr_t>(big) & 15) || (reinterpret_cast<uintptr_t>(small) & 15))
    return fail(CGAN3D_E_ARG, "tcgen05 strided wgrad: pointers must be 16-byte aligned");
  if (beta == 0.f) {
    cudaError_t e = cudaMemsetAsync(dw, 0, (size_t)g.Cs * g.Cb * p.taps * sizeof(float), st);
    if (e != cudaSuccess) return cuda_fail(e, "tcgen05 strided wgrad memset");
  }
  CUtensorMap tmY, tmX;  // whole voxels, swizzled by the row width
  int r = encode_act_map(&tmY, small, g.Cs, g.Zs, g.Ys, g.Xs, g.B, g.Cs, p.Zh, p.Yt, 1, 1, 2 * g.Cs, "strided wgrad, small side");
  if (r) return r;
  r = encode_act_map(&tmX, big, g.Cb, g.Zb, g.Yb, g.Xb, g.B, g.Cb, p.Zh, p.Yh, g.stride, g.stride, 2 * g.Cb, "strided wgrad, big side");
  if (r) return r;
  const int grid = (int)mn<long long>((long long)p.k * p.steps_per_dx, (long long)(num_sms() / p.k) * p.k);
  return tc_launch<wgrad_s2_sw_kernel>("wgrad_s2_sw_kernel", grid, 192, p.smem_bytes, 1, st, tmY, tmX, dw, p);
}

}  // namespace cg
