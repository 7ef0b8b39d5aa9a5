// tcgen05 kernels for the 7x7x7 THIN-CHANNEL convolutions of the generator (bf16 operands, fp32 accumulation in TMEM):
//   model.first      Conv3d(1 -> 16, k7, reflect)      reference model/generator.py:31-38
//   model.last_conv  Conv3d(16 -> 1, k7, reflect)+bias reference model/generator.py:77-83
// and their backward passes (aten::convolution_backward).  Together they hold 37 % of the generator's FLOPs
// (SURVEY App. A) but have GEMM N (or K) of 1, so none of the channel-GEMM kernels applies.  Each op gets its own
// mapping onto M=128 UMMA tiles:
//
//  (A) 1 -> 16 channels (fprop of `first`, dgrad of `last_conv`): TOEPLITZ-IN-Z implicit GEMM.
//      The 1-channel input is a scalar field with z contiguous, so a window of 16 consecutive z values of one (x,y)
//      line is a 32-byte K-major operand row.  GEMM rows = flattened (x', y') positions of a halo slab (TMA box
//      8z x Yh x Xh lands as [row][8 z] == the SWIZZLE_NONE core-matrix layout), K = 16 input z, N = 8 output z x 16
//      channels = 128, and the B operand of tap (dx,dy) is the banded matrix T[zi][(zo,co)] = W[dx,dy,zi-zo,co].
//      The 49 (dx,dy) taps are pure row shifts of the A descriptor (dx*Yh+dy rows), all 49 Toeplitz tiles (4 KB each)
//      stay resident in shared memory, and a TMEM lane (= output (x,y)) ends up with 8 z x 16 channels = 256
//      contiguous output bytes.  7 of every 16 K rows are non-zero: useful MMA fraction 44 %, no im2col, no expansion
//      of the input in HBM.  Zero padding (dgrad) is TMA out-of-bounds fill.
#include "common.cuh"
#include "conv_internal.cuh"
#include "tc_common.cuh"

namespace cg {

constexpr uint32_t kSmemLimitThin = kMaxDynSmem - 1024;
constexpr int kTapTilesA = 49;
constexpr int kZbA = 8;                  // output z per work item
constexpr uint32_t kTileBytesA = 4096;  // [2 z-chunks][128 n = 8 z x 16 ch][8 z] bf16
constexpr double kHaloWeightA = 0.02;   // weight of the halo overhead (Xh*Yh / Xt*Yt) in the tile score of plan_thin_a

struct ThinAPlan {
  int B, Xi, Yi, Zi;  // 1-channel input
  int Xo, Yo, Zo;     // 16-channel output
  int P;              // input coordinate = output coordinate + tap - P (P = 0: valid conv, P = 6: full correlation)
  int Xt, Yt, Xh, Yh, nxt, nyt, nzb;
  int mtiles, rows_alloc, nslots;
  uint32_t slot_bytes, box_bytes, tmem_cols, smem_bytes;
  int Zc;      // z extent of the shifted copy: copy[row][c] = in[row][c - 8 + zshift]
  int zshift;  // makes every 8-z window start on a 16-byte boundary of the copy
};

// An item covers 8 output z, N = 128.  A cta_group::2 MMA costs 59 cycles up to N = 96 and 65 at N = 128
// (profiles/r01_mma2_microbench.txt), the 14-voxel input window of 8 outputs still fits K = 16, and every window starts on a
// 16-byte boundary of ONE shifted copy of the input.
// CTA pairs (see conv_tc.cu): the two CTAs of a cluster process consecutive work items in lockstep; each holds the Toeplitz
// rows of four of the eight output z (64 of the 128 N rows), and the rank-0 CTA issues every MMA for both.
template <int MT, bool STATS>
__global__ void __launch_bounds__(192, 1)
conv7_c1_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, bf16 *__restrict__ out,
                   const __grid_constant__ ThinAPlan p, double *__restrict__ bn_sums) {
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr uint32_t NN = kZbA * 16;               // GEMM N = output z x 16 channels
  constexpr uint32_t kTileB = kTileBytesA / 2;     // this CTA's half of a Toeplitz tile
  // accumulator ring: with one M tile per item an item is only ~2 us of MMAs, so the MMA -> epilogue -> MMA hand-off
  // latency must be hidden behind several buffers (all 512 TMEM columns are used)
  constexpr uint32_t NACC = 512 / (MT * NN);
  uint8_t *bres = smem;                                    // 49 resident Toeplitz half tiles
  uint8_t *ring = bres + kTapTilesA * kTileB;              // slab slots
  uint8_t *stage = ring + (size_t)p.nslots * p.slot_bytes; // epilogue store staging: 4 warps x 32 rows x 128 B
  uint64_t *bars = reinterpret_cast<uint64_t *>(stage + 16384);
  uint64_t *b_ready = bars, *s_full = bars + 1, *s_empty = s_full + p.nslots;
  uint64_t *tm_full = s_empty + p.nslots, *tm_empty = tm_full + NACC;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(tm_empty + NACC);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tc::mbar_init(b_ready, 1);
    for (int i = 0; i < p.nslots; ++i) { tc::mbar_init(&s_full[i], 1); tc::mbar_init(&s_empty[i], 1); }
    for (int i = 0; i < (int)NACC; ++i) { tc::mbar_init(&tm_full[i], 1); tc::mbar_init(&tm_empty[i], 8); }
    tc::fence_barrier_init();
  }
  const uint32_t cta_rank = tc::cluster_ctarank();
  __syncthreads();
  tc::cluster_sync();
  if (warp == 5) { tc::tmem_alloc2(tmem_ptr, p.tmem_cols); tc::tmem_relinquish2(); }
  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // work items: the pair walks item pairs (2j, 2j+1); an odd total leaves the last odd CTA a dead copy of item 2j
  const long long total_items = (long long)p.B * p.nxt * p.nyt * p.nzb;
  const long long total = (total_items + 1) / 2;
  const int nblk = (int)gridDim.x >> 1, blk = (int)blockIdx.x >> 1;
  const int i_begin = (int)(total * blk / nblk), i_end = (int)(total * (blk + 1) / nblk);
  auto decode = [&](int it, int &b, int &x0, int &xlen, int &y0, int &ylen, int &z0) -> bool {
    bool live = true;
    it = 2 * it + (int)cta_rank;
    if (it >= total_items) { it = (int)total_items - 1; live = false; }
    const int zb = it % p.nzb; it /= p.nzb;
    const int yt = it % p.nyt; it /= p.nyt;
    const int xt = it % p.nxt;
    b = it / p.nxt;
    x0 = xt * p.Xt; xlen = min(p.Xt, p.Xo - x0);
    y0 = yt * p.Yt; ylen = min(p.Yt, p.Yo - y0);
    z0 = zb * kZbA;
    return live;
  };

  if (warp == 4) {
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmA);
      // boxes of 196 rows of 256 bytes (49 KB): this CTA's 49 half tiles, counted on the rank-0 barrier
      if (cta_rank == 0) tc::mbar_expect_tx(b_ready, 2 * kTapTilesA * kTileB);
      constexpr int rows_cta = (int)(kTapTilesA * kTileB / 256);
      for (int r0 = 0; r0 < rows_cta; r0 += 196)
        tc::tma_load_2d_2cta(bres + (size_t)r0 * 256, &tmW, b_ready, 0, (int)cta_rank * rows_cta + r0);
      uint32_t e = 0;
      for (int it = i_begin; it < i_end; ++it, ++e) {
        int b, x0, xlen, y0, ylen, z0;
        decode(it, b, x0, xlen, y0, ylen, z0);
        const uint32_t slot = e % p.nslots, use = e / p.nslots;
        if (use > 0) tc::mbar_wait(&s_empty[slot], (use - 1) & 1);
        uint8_t *dst = ring + (size_t)slot * p.slot_bytes;
        // TMA needs a 16-byte aligned start along z: the z shift of the copy makes it so.  Rows of 16 z = 32 bytes, SWIZZLE_32B
        const int c0 = z0 - p.P - p.zshift + 8;
        if (cta_rank == 0) tc::mbar_expect_tx(&s_full[slot], 2 * p.box_bytes);
        tc::tma_load_5d_2cta(dst, &tmA, &s_full[slot], c0, y0 - p.P, x0 - p.P, b, 0);
      }
    }
  } else if (warp == 5 && cta_rank != 0) {
    // odd CTA of a pair: the rank-0 CTA issues the MMAs for both
  } else if (warp == 5) {
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(256, (int)NN, 0, 0);
    const uint32_t ring_u32 = tc::smem_u32(ring), b_u32 = tc::smem_u32(bres);
    const uint64_t a_hi = tc::make_desc_sw(0, 256, 32), b_hi = tc::make_desc(0, NN / 2 * 16, 128);
    tc::mbar_wait(b_ready, 0);
    tc::tc_fence_after();
    uint32_t e = 0;
    for (int it = i_begin; it < i_end; ++it, ++e) {
      const uint32_t q = e % NACC, uq = e / NACC, slot = e % p.nslots;
      if (uq > 0) tc::mbar_wait(&tm_empty[q], (uq - 1) & 1);
      tc::mbar_wait(&s_full[slot], (e / p.nslots) & 1);
      tc::tc_fence_after();
      const uint32_t a_slot = (ring_u32 + slot * p.slot_bytes) >> 4;
      const uint32_t d_base = tmem_base + q * (uint32_t)(MT * NN);
      // lean issue loop: the seven dy taps of one dx go out back to back with descriptor adds only (a loop iteration
      // per MMA costs ~120 cycles of dependent scalar work on the single issuing warp, more than the MMA itself)
      const uint64_t a_it = a_hi | (uint64_t)(a_slot & 0x3FFF), b_it = b_hi | (uint64_t)((b_u32 >> 4) & 0x3FFF);
      for (int dx = 0; dx < 7; ++dx) {
        const uint64_t a_dx = a_it + (uint64_t)(2u * (uint32_t)(dx * p.Yh));             // 32-byte rows
        const uint64_t b_dx = b_it + (uint64_t)((uint32_t)(dx * 7) * (kTileB >> 4));
        if (leader) {
#pragma unroll
          for (int dy = 0; dy < 7; ++dy) {
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
              const uint32_t accum = dy != 0 ? 1u : (uint32_t)(dx != 0);
              tc::umma_bf16_2cta(d_base + mt * NN, a_dx + (uint64_t)(2 * dy + mt * 256), b_dx + (uint64_t)(dy * (kTileB >> 4)), idesc, accum);
            }
          }
        }
        __syncwarp();
      }
      if (leader) { tc::umma_commit_2cta(&s_empty[slot], 3); tc::umma_commit_2cta(&tm_full[q], 3); }
      __syncwarp();
    }
  } else {
    uint32_t e = 0;
    uint4 *stage_w = reinterpret_cast<uint4 *>(stage) + warp * 256;  // this warp's 32 rows x 128 B
    float ssum[STATS ? 16 : 1], ssq[STATS ? 16 : 1];  // per-channel BatchNorm partial sums of this thread's rows
    if (STATS) {
#pragma unroll
      for (int j = 0; j < 16; ++j) { ssum[j] = 0.f; ssq[j] = 0.f; }
    }
    for (int it = i_begin; it < i_end; ++it, ++e) {
      int b, x0, xlen, y0, ylen, z0_item;
      const bool live = decode(it, b, x0, xlen, y0, ylen, z0_item);
      const uint32_t q = e % NACC;
      tc::mbar_wait(&tm_full[q], (e / NACC) & 1);
      tc::tc_fence_after();
      const uint32_t d_base = tmem_base + ((uint32_t)(warp * 32) << 16) + q * (uint32_t)(MT * NN);
#pragma unroll
      for (int mth = 0; mth < MT * 2; ++mth) {  // (M tile, group of four output z)
        const int mt = mth >> 1, zh = (mth & 1) * 4;
        const int r = mt * 128 + warp * 32 + lane;
        const int xx = r / p.Yh, yy = r - xx * p.Yh;
        const bool valid = live && xx < xlen && yy < ylen;
        const int z0 = z0_item + zh;
        bf16 *dst = out + ((((size_t)b * p.Xo + (x0 + xx)) * p.Yo + (y0 + yy)) * p.Zo + z0) * 16;
        uint32_t v[4][16];  // four output z of this row: all TMEM loads in flight before one wait
#pragma unroll
        for (int zo = 0; zo < 4; ++zo) tc::tmem_ld16(d_base + (uint32_t)(mt * NN + (zh + zo) * 16), v[zo]);
        tc::tmem_ld_wait();
        // A lane owns one (x,y) row = 128 contiguous output bytes, but neighbouring lanes are a whole z line (4 KB) apart:
        // direct stores would be 32 quarter-line writes per instruction.  Stage the warp's 32 x 128 B in shared memory
        // (16-byte chunks XOR-swizzled by row, conflict-free both ways) and store full 128-byte lines, 4 rows per instruction.
        __syncwarp();
#pragma unroll
        for (int zo = 0; zo < 4; ++zo) {
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[zo][2 * j]), __uint_as_float(v[zo][2 * j + 1]));
            pk[j] = *reinterpret_cast<uint32_t *>(&h);
          }
          stage_w[lane * 8 + ((2 * zo) ^ (lane & 7))] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          stage_w[lane * 8 + ((2 * zo + 1) ^ (lane & 7))] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
          if constexpr (STATS) {
            if (valid && z0 + zo < p.Zo) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float f = __uint_as_float(v[zo][j]);
                ssum[j] += f;
                ssq[j] += f * f;
              }
            }
          }
        }
        __syncwarp();
        const unsigned long long dst_u = reinterpret_cast<unsigned long long>(dst);
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int row = it * 4 + (lane >> 3), ch = lane & 7;
          const unsigned long long d_row = __shfl_sync(0xffffffffu, dst_u, row);
          const bool v_row = __shfl_sync(0xffffffffu, (int)valid, row) != 0;
          const uint4 val = stage_w[row * 8 + (ch ^ (row & 7))];
          if (v_row && z0 + (ch >> 1) < p.Zo) reinterpret_cast<uint4 *>(d_row)[ch] = val;
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive_cluster(&tm_empty[q], 0);
    }
    if constexpr (STATS) {
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float a = warp_sum(ssum[j]), b2 = warp_sum(ssq[j]);
        if (lane == 0) { atomicAdd(&bn_sums[j], (double)a); atomicAdd(&bn_sums[16 + j], (double)b2); }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();
  if (warp == 5) tc::tmem_dealloc2(tmem_base, p.tmem_cols);
}

// Toeplitz tiles: T[(dx,dy)][zi/8][n = zo*16 + co][zi%8] = w(dx,dy,zi-zo,co) for 0 <= zi-zo < 7, else 0, as the halves
// held by the two CTAs of a pair: [half][(dx,dy)][zi/8][64 n][8], half = n / 64.
// wp is the packed filter [tap][Cb][Cs] with Cb*Cs == 16; flip = 1 reverses the taps (transposed convolution).
__global__ void toeplitz_a_kernel(const bf16 *__restrict__ wp, bf16 *__restrict__ wt, int flip) {
  constexpr int NN = kZbA * 16, Nh = NN >> 1;
  const int total = kTapTilesA * 2 * NN * 8;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int z8 = i & 7;
    int t = i >> 3;
    const int nl = t % Nh; t /= Nh;
    const int chunk = t & 1; t >>= 1;
    const int tile = t % kTapTilesA;
    const int n = (t / kTapTilesA) * Nh + nl;
    const int zi = chunk * 8 + z8, zo = n >> 4, co = n & 15, dz = zi - zo;
    bf16 v = __float2bfloat16_rn(0.f);
    if (dz >= 0 && dz < 7) {
      const int tap = tile * 7 + dz;
      v = wp[(size_t)(flip ? 342 - tap : tap) * 16 + co];
    }
    wt[i] = v;
  }
}

// TMA needs 16-byte aligned row pitches AND a 16-byte aligned start coordinate along the contiguous axis, but the z
// windows start at z0 - P.  A z-shifted, zero-margined copy of the 1-channel input makes every window start aligned:
// copy[row][c] = in[row][c - 8 + s]  (0 outside), c in [0, Zc), Zc % 8 == 0.
// One WARP per input line (8 lines per block): the line is staged in shared memory (with zero margins) and written out as
// 16-byte chunks.
__global__ void __launch_bounds__(256)
shifted_copies_kernel(const bf16 *__restrict__ in, bf16 *__restrict__ out, long long rows, int Z, int Zc, int s) {
  extern __shared__ uint16_t lines[];  // per warp: line[8 + z] = in[z], zeros in [0, 8) and beyond Z
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = (Zc + 24 + 7) & ~7;
  uint16_t *line = lines + (size_t)warp * n;
  const long long r = (long long)blockIdx.x * 8 + warp;
  if (r >= rows) return;
  const uint16_t *src = reinterpret_cast<const uint16_t *>(in) + r * Z;
  for (int i = lane; i < n; i += 32) {
    const int z = i - 8;
    line[i] = (z >= 0 && z < Z) ? src[z] : (uint16_t)0;
  }
  __syncwarp();
  for (int j = lane; j < (Zc >> 3); j += 32) {
    const int base = j * 8 + s;  // out[c] = in[c - 8 + s] = line[c + s]
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = (uint32_t)line[base + 2 * k] | ((uint32_t)line[base + 2 * k + 1] << 16);
    reinterpret_cast<uint4 *>(out + r * Zc)[j] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
//  (B) 16 -> 1 channels (fprop of `last_conv`, dgrad of `first`): filter x- AND z-offsets STACKED ON N.
//      GEMM rows = flattened (y', z') positions of one input x-plane slab (pitch Zh = Zt + 6, as in conv_tc.cu),
//      K = 16 input channels (one 32-byte SWIZZLE_32B row per voxel, one TMA per slab), and only the 7 dy taps are row
//      shifts accumulated by the tensor core.  N = 64 carries (dx, dz): D_xi[row, (dx,dz)] is the contribution of input
//      plane xi, input row `row`, to output plane xi + P - dx, output row `row - dz`.  An SS-mode tcgen05.mma costs
//      >= 72 cycles whatever its N (measured, tools/micro/mma_bench.cu), so 7 MMAs of N = 64 replace 49 of N = 16.
//      Epilogue: the slab pitch is exactly 32 rows per y-line (26 outputs + 6 halo voxels along z), so a line is one
//      32-lane TMEM group and the z shift is undone with warp shuffles alone; the x shift is undone with a 7-deep
//      register window of partial output planes per thread; one finished output plane is retired per input plane.
constexpr int kTapTilesB = 7;
constexpr uint32_t kTileBytesB = 2048;  // [64 n = dx*8 + dz][16 ci] bf16, SWIZZLE_32B rows
constexpr int kPitchB = 32, kZtB = 26;    // rows per slab line / outputs per line

struct ThinBPlan {
  int B, Xi, Yi, Zi;  // 16-channel input
  int Xo, Yo, Zo;     // 1-channel output
  int P;
  int Zt, nzt, Zh, Yt, nyt, Yh;
  int mtiles, rows_alloc, nslots;
  uint32_t slot_bytes, box_bytes, tmem_cols, smem_bytes;
};

struct SegIter {
  long long idx, end;
  int Xo;
  // pair = true: the two CTAs of a cluster share one range over COLUMN PAIRS (the caller maps pair column j to columns
  // 2j + rank), so both walk identical (x0, xlen) segments in lockstep
  __device__ __forceinline__ SegIter(long long ncols, int Xo_, bool pair = false) : Xo(Xo_) {
    const long long nblk = pair ? gridDim.x >> 1 : gridDim.x, blk = pair ? blockIdx.x >> 1 : blockIdx.x;
    const long long total = (pair ? (ncols + 1) / 2 : ncols) * Xo;
    idx = total * blk / nblk;
    end = total * (blk + 1) / nblk;
  }
  __device__ __forceinline__ bool next(int &col, int &x0, int &xlen) {
    if (idx >= end) return false;
    col = (int)(idx / Xo);
    x0 = (int)(idx - (long long)col * Xo);
    xlen = (int)mn<long long>(Xo - x0, end - idx);
    idx += xlen;
    return true;
  }
};

// CTA pairs: the two CTAs of a cluster walk column pairs in lockstep, each holds 32 of the 64 N rows of every filter tile,
// and the rank-0 CTA issues every MMA for both.
template <int MT>
__global__ void __launch_bounds__(320, 1)
conv7_to1_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, bf16 *__restrict__ out,
                    const __grid_constant__ ThinBPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *bres = smem;                                                   // 7 resident filter tiles (14 KB)
  uint8_t *ring = smem + 14336;                                            // slab slots (multiple of 256 B)
  uint64_t *bars = reinterpret_cast<uint64_t *>(ring + (size_t)p.nslots * p.slot_bytes);
  uint64_t *b_ready = bars, *s_full = bars + 1, *s_empty = s_full + p.nslots;
  uint64_t *tm_full = s_empty + p.nslots, *tm_empty = tm_full + 2;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(tm_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tc::mbar_init(b_ready, 1);
    for (int i = 0; i < p.nslots; ++i) { tc::mbar_init(&s_full[i], 1); tc::mbar_init(&s_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&tm_full[i], 1); tc::mbar_init(&tm_empty[i], 16); }
    tc::fence_barrier_init();
  }
  constexpr uint32_t kTileB = kTileBytesB / 2;  // this CTA's 32 of the 64 N rows of a tile
  const uint32_t cta_rank = tc::cluster_ctarank();
  __syncthreads();
  tc::cluster_sync();
  if (warp == 9) { tc::tmem_alloc2(tmem_ptr, p.tmem_cols); tc::tmem_relinquish2(); }
  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const long long ncols = (long long)p.B * p.nyt * p.nzt;
  auto decode = [&](int col, int &b, int &y0, int &ylen, int &z0, int &zlen) -> bool {
    bool live = true;
    col = 2 * col + (int)cta_rank;
    if (col >= ncols) { col = (int)ncols - 1; live = false; }
    const int zt = col % p.nzt; col /= p.nzt;
    const int yt = col % p.nyt;
    b = col / p.nyt;
    y0 = yt * p.Yt; ylen = min(p.Yt, p.Yo - y0);
    z0 = zt * p.Zt; zlen = min(p.Zt, p.Zo - z0);
    return live;
  };

  if (warp == 8) {
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmA);
      // SWIZZLE_32B repeats every 256 bytes, so rows 32r..32r+31 of a tile are simply its r-th kilobyte (4 map rows)
      if (cta_rank == 0) tc::mbar_expect_tx(b_ready, 2 * kTapTilesB * kTileB);
      for (int t = 0; t < kTapTilesB; ++t) tc::tma_load_2d_2cta(bres + (size_t)t * kTileB, &tmW, b_ready, 0, t * 8 + (int)cta_rank * 4);
      uint32_t e = 0;
      int col, x0, xlen;
      for (SegIter it(ncols, p.Xo, true); it.next(col, x0, xlen);) {
        int b, y0, ylen, z0, zlen;
        decode(col, b, y0, ylen, z0, zlen);
        for (int i = 0; i < xlen + 6; ++i, ++e) {
          const uint32_t slot = e % p.nslots, use = e / p.nslots;
          if (use > 0) tc::mbar_wait(&s_empty[slot], (use - 1) & 1);
          if (cta_rank == 0) tc::mbar_expect_tx(&s_full[slot], 2 * p.box_bytes);
          tc::tma_load_5d_2cta(ring + (size_t)slot * p.slot_bytes, &tmA, &s_full[slot], 0, z0 - p.P, y0 - p.P, x0 - p.P + i, b);
        }
      }
    }
  } else if (warp == 9 && cta_rank != 0) {
    // odd CTA of a pair: the rank-0 CTA issues the MMAs of both
  } else if (warp == 9) {
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(256, 64, 0, 0);
    const uint32_t ring_u32 = tc::smem_u32(ring), b_u32 = tc::smem_u32(bres);
    const uint64_t a_hi = tc::make_desc_sw(0, 256, 32), b_hi = tc::make_desc_sw(0, 256, 32);
    tc::mbar_wait(b_ready, 0);
    tc::tc_fence_after();
    uint32_t e = 0;
    int col, x0, xlen;
    for (SegIter it(ncols, p.Xo, true); it.next(col, x0, xlen);) {
      for (int i = 0; i < xlen + 6; ++i, ++e) {
        const uint32_t q = e & 1, uq = e >> 1, slot = e % p.nslots;
        if (uq > 0) tc::mbar_wait(&tm_empty[q], (uq - 1) & 1);
        tc::mbar_wait(&s_full[slot], (e / p.nslots) & 1);
        tc::tc_fence_after();
        const uint32_t a_slot = (ring_u32 + slot * p.slot_bytes) >> 4;
        const uint32_t d_base = tmem_base + q * (uint32_t)(MT * 64);
        if (leader) {
#pragma unroll
          for (int dy = 0; dy < 7; ++dy) {
            const uint64_t a0 = a_hi | (uint64_t)((a_slot + 2u * (uint32_t)(dy * kPitchB)) & 0x3FFF);  // 32-byte rows
            const uint64_t b0 = b_hi | (uint64_t)(((b_u32 + (uint32_t)dy * kTileB) >> 4) & 0x3FFF);
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
              tc::umma_bf16_2cta(d_base + mt * 64, a0 + (uint64_t)(mt * 256), b0, idesc, (uint32_t)(dy != 0));
          }
          tc::umma_commit_2cta(&s_empty[slot], 3);
          tc::umma_commit_2cta(&tm_full[q], 3);
        }
        __syncwarp();
      }
    }
  } else {
    // 8 epilogue warps: TMEM lane quadrant qd = warp & 3 (= y-line qd of every M-tile, lane = z within the line);
    // warps 0-3 own the even M-tiles, warps 4-7 the odd ones
    constexpr int NK = (MT + 1) / 2;
    const int qd = warp & 3, grp = warp >> 2;
    uint32_t e = 0;
    int col, x0, xlen;
    for (SegIter it(ncols, p.Xo, true); it.next(col, x0, xlen);) {
      int b, y0, ylen, z0, zlen;
      const bool live = decode(col, b, y0, ylen, z0, zlen);
      float win[NK][7];
      bool valid[NK];
      uint32_t off[NK];
#pragma unroll
      for (int k = 0; k < NK; ++k) {
#pragma unroll
        for (int j = 0; j < 7; ++j) win[k][j] = 0.f;
        const int mt = 2 * k + grp;
        const int yy = mt * 4 + qd;
        valid[k] = live && mt < MT && yy < ylen && lane < zlen;
        off[k] = (uint32_t)((y0 + yy) * p.Zo + (z0 + lane));
      }
      for (int i = 0; i < xlen + 6; ++i, ++e) {
        const uint32_t q = e & 1;
        tc::mbar_wait(&tm_full[q], (e >> 1) & 1);
        tc::tc_fence_after();
        const uint32_t d_base = tmem_base + ((uint32_t)(qd * 32) << 16) + q * (uint32_t)(MT * 64);
        bf16 *plane = out + ((size_t)b * p.Xo + (x0 + i - 6)) * p.Yo * p.Zo;
#pragma unroll
        for (int k = 0; k < NK; ++k) {
          const int mt = 2 * k + grp;
          if (mt >= MT) continue;
          uint32_t v[7][8];
#pragma unroll
          for (int dx = 0; dx < 7; ++dx) tc::tmem_ld8(d_base + (uint32_t)(mt * 64 + dx * 8), v[dx]);
          tc::tmem_ld_wait();
          // out[z] = sum_dz D[z + dz][(dx, dz)]: lanes z >= 26 read past the line, they are halo rows and never stored
          float t[7];
#pragma unroll
          for (int dx = 0; dx < 7; ++dx) {
            float acc = __uint_as_float(v[dx][0]);
#pragma unroll
            for (int dz = 1; dz < 7; ++dz) acc += __shfl_down_sync(0xffffffffu, __uint_as_float(v[dx][dz]), dz);
            t[dx] = acc;
          }
          // column block dx feeds output plane (this input plane) + P - dx == window slot 6 - dx
#pragma unroll
          for (int j = 0; j < 7; ++j) win[k][j] += t[6 - j];
          if (i >= 6 && valid[k]) plane[off[k]] = __float2bfloat16_rn(win[k][0]);
#pragma unroll
          for (int j = 0; j < 6; ++j) win[k][j] = win[k][j + 1];
          win[k][6] = 0.f;
        }
        tc::tc_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive_cluster(&tm_empty[q], 0);
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();
  if (warp == 9) tc::tmem_dealloc2(tmem_base, p.tmem_cols);
}

// T[dy][n = dx*8 + dz][ci] = w(dx,dy,dz,ci) for dx, dz < 7, else 0 (same flip convention as toeplitz_a_kernel), stored as
// a K-major SWIZZLE_32B operand: 32-byte rows, 16-byte chunk c of row n lives at chunk c ^ ((n >> 2) & 1).
__global__ void stack_b_kernel(const bf16 *__restrict__ wp, bf16 *__restrict__ wt, int flip) {
  const int total = kTapTilesB * 64 * 16;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int c8 = i & 7;
    int t = i >> 3;
    const int pchunk = t & 1; t >>= 1;
    const int n = t & 63;
    const int dy = t >> 6;
    const int chunk = pchunk ^ ((n >> 2) & 1);
    const int dx = n >> 3, dz = n & 7;
    bf16 v = __float2bfloat16_rn(0.f);
    if (dx < 7 && dz < 7) {
      const int tap = (dx * 7 + dy) * 7 + dz;
      v = wp[(size_t)(flip ? 342 - tap : tap) * 16 + chunk * 8 + c8];
    }
    wt[i] = v;
  }
}

// ---------------------------------------------------------------------------------------------------------------
//  (C) weight gradient of both layers:  R[c][dx,dy,dz] = sum_v S16[v, c] * Q1[v + (dx,dy,dz) - P]
//      (S16 = the 16-channel tensor, Q1 = the 1-channel one; `first`: S16 = dY, Q1 = padded input, P = pad;
//       `last_conv`: S16 = padded input, Q1 = dY, P = 6 - pad and the taps come out flipped).
//      GEMM per K-block of 16 voxels (rows = flattened (y,z) of one x-plane, both operands MN-major):
//        A: the z-EXPANDED 1-channel tensor E[v][j] = Q1[v + j*ez - P] (8 x 2 B = one 16-byte row, built by a pre-pass in
//           the workspace).  M = 64 = 8 dy line-shifts (operand chunks one slab line apart) x 8 dz (the expansion).
//        B: S16 planes.  N = 64 = 16 channels x 4 consecutive x-planes that sit in adjacent ring slots, i.e. one MMA
//           produces 4 filter x-offsets at once.  The ring has 8 slots; the 7 live planes x'-6..x' fall into 2-3 aligned
//           groups of 4, each group is one MMA whose accumulator column block is (plane - x' + 9); blocks 3..9 are the
//           7 real dx accumulators, blocks 0..2 / 10..12 are guard columns that soak up planes outside the window.
//      Split-K over CTAs (contiguous runs of x-planes of one (b, y-tile, z-tile) column), fp32 atomics at the end.
struct ThinCPlan {
  int B, Xs, Ys, Zs;  // S16 extents
  int Xe, Ye;         // planes / lines of E (= Xs + 6, Ys + 6); E rows per line = Zs
  int P, flip;
  int Zt, nzt, Yt, nyt;
  int rowsB, kblocks, e_slots;
  uint32_t slotB_bytes, slotA_bytes, boxA_bytes, boxB_bytes, smem_bytes;
};
constexpr int kRingC = 8;

__global__ void __launch_bounds__(192, 1)
wgrad7_thin_tc_kernel(const __grid_constant__ CUtensorMap tmE, const __grid_constant__ CUtensorMap tmS, float *__restrict__ dw,
                      const __grid_constant__ ThinCPlan p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *ringB = smem;                                    // 8 S16 plane slots, each [rowsB][16 ch] (SWIZZLE_32B)
  uint8_t *ringA = ringB + (size_t)kRingC * p.slotB_bytes;  // E slabs, [rowsA][8 j]
  uint64_t *bars = reinterpret_cast<uint64_t *>(ringA + (size_t)p.e_slots * p.slotA_bytes);
  uint64_t *b_full = bars, *b_empty = bars + kRingC, *a_full = b_empty + kRingC, *a_empty = a_full + p.e_slots;
  uint64_t *done = a_empty + p.e_slots;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kRingC; ++i) { tc::mbar_init(&b_full[i], 1); tc::mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < p.e_slots; ++i) { tc::mbar_init(&a_full[i], 1); tc::mbar_init(&a_empty[i], 1); }
    tc::mbar_init(done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 5) {
    tc::tmem_alloc(tmem_ptr, 256);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // every MMA accumulates (column blocks are first touched at different times), so the accumulators start at zero
  if (warp < 4) {
    for (int c0 = 0; c0 < 256; c0 += 16) tc::tmem_zero16(tmem_base + ((uint32_t)(warp * 32) << 16) + c0);
    tc::tmem_st_wait();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();

  const long long ncols = (long long)p.B * p.nyt * p.nzt;
  auto decode = [&](int col, int &b, int &y0, int &z0) {
    const int zt = col % p.nzt; col /= p.nzt;
    const int yt = col % p.nyt;
    b = col / p.nyt;
    y0 = yt * p.Yt;
    z0 = zt * p.Zt;
  };
  bool any = false;

  if (warp == 4) {
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmE);
      tc::tma_prefetch_desc(&tmS);
      // S16 plane xs lives in ring slot (xs & 7); every segment re-loads its 6 warm-up planes
      uint32_t useB[kRingC];
#pragma unroll
      for (int i = 0; i < kRingC; ++i) useB[i] = 0;
      auto load_plane = [&](int xs, int b, int y0, int z0) {
        const uint32_t slot = (uint32_t)(xs & 7);
        uint32_t n = 0;
#pragma unroll
        for (int i = 0; i < kRingC; ++i) if ((uint32_t)i == slot) { n = useB[i]; useB[i] = n + 1; }
        if (n > 0) tc::mbar_wait(&b_empty[slot], (n - 1) & 1);
        tc::mbar_expect_tx(&b_full[slot], p.boxB_bytes);
        tc::tma_load_5d(ringB + (size_t)slot * p.slotB_bytes, &tmS, &b_full[slot], 0, z0, y0, xs, b);  // [row][16 ch], SWIZZLE_32B
      };
      uint32_t ea = 0;
      int col, x0, xlen;
      for (SegIter it(ncols, p.Xe); it.next(col, x0, xlen);) {
        int b, y0, z0;
        decode(col, b, y0, z0);
        for (int xs = x0 - 6; xs < x0; ++xs) load_plane(xs, b, y0, z0);
        for (int i = 0; i < xlen; ++i, ++ea) {
          load_plane(x0 + i, b, y0, z0);
          const uint32_t slot = ea % p.e_slots, use = ea / p.e_slots;
          if (use > 0) tc::mbar_wait(&a_empty[slot], (use - 1) & 1);
          tc::mbar_expect_tx(&a_full[slot], p.boxA_bytes);
          tc::tma_load_5d(ringA + (size_t)slot * p.slotA_bytes, &tmE, &a_full[slot], 0, z0, y0, x0 + i, b);
        }
      }
    }
  } else if (warp == 5) {
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(64, 64, 1, 1);
    // B: MN-major SWIZZLE_32B, one 16-channel block per ring slot (LBO = slot stride), 8-voxel K groups 256 B apart
    const uint64_t a_hi = tc::make_desc(0, 128, (uint32_t)p.Zt * 16), b_hi = tc::make_desc_sw_mn(0, p.slotB_bytes, 256, 32);
    const uint32_t ringA_u32 = tc::smem_u32(ringA), ringB_u32 = tc::smem_u32(ringB);
    uint32_t useB[kRingC];
#pragma unroll
    for (int i = 0; i < kRingC; ++i) useB[i] = 0;
    auto wait_plane = [&](int xs) {  // mirrors the producer's per-slot use count
      const uint32_t slot = (uint32_t)(xs & 7);
      uint32_t n = 0;
#pragma unroll
      for (int i = 0; i < kRingC; ++i) if ((uint32_t)i == slot) { n = useB[i]; useB[i] = n + 1; }
      tc::mbar_wait(&b_full[slot], n & 1);
    };
    uint32_t ea = 0;
    int col, x0, xlen;
    for (SegIter it(ncols, p.Xe); it.next(col, x0, xlen);) {
      any = true;
      for (int xs = x0 - 6; xs < x0; ++xs) wait_plane(xs);
      for (int i = 0; i < xlen; ++i, ++ea) {
        const int xe = x0 + i;
        wait_plane(xe);
        const uint32_t slotA = ea % p.e_slots;
        tc::mbar_wait(&a_full[slotA], (ea / p.e_slots) & 1);
        tc::tc_fence_after();
        const uint32_t a0 = (ringA_u32 + slotA * p.slotA_bytes) >> 4;
        const int g_lo = (xe - 6) >> 2, g_hi = xe >> 2;  // aligned groups of 4 planes overlapping [xe-6, xe]
        for (int g4 = g_lo; g4 <= g_hi; ++g4) {
          const uint32_t slot0 = (uint32_t)((g4 * 4) & 7);
          const uint32_t b0 = (ringB_u32 + slot0 * p.slotB_bytes) >> 4;
          const uint32_t d = tmem_base + (uint32_t)((g4 * 4 - xe + 9) * 16);
          if (leader) {
            uint64_t a_desc = a_hi | (uint64_t)(a0 & 0x3FFF), b_desc = b_hi | (uint64_t)(b0 & 0x3FFF);
#pragma unroll 4
            for (int kb = 0; kb < p.kblocks; ++kb) {
              tc::umma_bf16(d, a_desc, b_desc, idesc, 1u);
              a_desc += 16;  // 16 rows of 16 B
              b_desc += 32;  // 16 rows of 32 B
            }
          }
          __syncwarp();
        }
        if (leader) {
          tc::umma_commit(&a_empty[slotA]);
          tc::umma_commit(&b_empty[(uint32_t)((xe - 6) & 7)]);  // plane xe-6 is not needed by later steps
        }
        __syncwarp();
      }
      // the last 6 planes of the segment are still loaded: release their slots for the next segment
      if (leader)
        for (int xs = x0 + xlen - 6; xs < x0 + xlen; ++xs) tc::umma_commit(&b_empty[(uint32_t)(xs & 7)]);
      __syncwarp();
    }
    if (leader) tc::umma_commit(done);
    __syncwarp();
  } else {
    // epilogue (warps 0..3): M = 64 accumulator rows 16w..16w+15 live in TMEM lanes 32w..32w+15
    SegIter it(ncols, p.Xe);
    if (it.idx < it.end) {
      tc::mbar_wait(done, 0);
      tc::tc_fence_after();
      const int m = warp * 16 + (lane & 15), dy = m >> 3, j = m & 7;
      for (int blk = 3; blk <= 9; ++blk) {
        uint32_t v[16];
        tc::tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(blk * 16), v);
        tc::tmem_ld_wait();
        if (lane < 16 && dy < 7 && j < 7) {
          int tap = (9 - blk) * 49 + dy * 7 + j;
          if (p.flip) tap = 342 - tap;
#pragma unroll
          for (int c = 0; c < 16; ++c) atomicAdd(&dw[(size_t)c * 343 + tap], __uint_as_float(v[c]));
        }
      }
    }
  }
  (void)any;
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 5) tc::tmem_dealloc(tmem_base, 256);
}

// E[b][xe][ye][z][j] = Q1[b][xe - P][ye - P][z + j - P]  (0 outside Q1), j = 0..7: one 16-byte row per (xe, ye, z)
// One warp per (b, xe, ye) line, 8 lines per block.
__global__ void __launch_bounds__(256)
expand_z_kernel(const bf16 *__restrict__ q, bf16 *__restrict__ e, long long lines_total, int Xq, int Yq, int Zq, int Xe, int Ye, int Ze, int P) {
  extern __shared__ uint16_t lines[];  // per warp: line[i] = Q1 line value at z = i - P (0 outside), i in [0, Ze + 8)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = (Ze + 8 + 7) & ~7;
  uint16_t *line = lines + (size_t)warp * n;
  const long long r = (long long)blockIdx.x * 8 + warp;
  if (r >= lines_total) return;
  const int ye = (int)(r % Ye);
  const int xe = (int)((r / Ye) % Xe);
  const int b = (int)(r / ((long long)Ye * Xe));
  const int xq = xe - P, yq = ye - P;
  const bool inside = xq >= 0 && xq < Xq && yq >= 0 && yq < Yq;
  const uint16_t *src = reinterpret_cast<const uint16_t *>(q) + (((size_t)b * Xq + (inside ? xq : 0)) * Yq + (inside ? yq : 0)) * Zq;
  for (int i = lane; i < Ze + 8; i += 32) {
    const int z = i - P;
    line[i] = (inside && z >= 0 && z < Zq) ? src[z] : (uint16_t)0;
  }
  __syncwarp();
  uint4 *dst = reinterpret_cast<uint4 *>(e) + (size_t)r * Ze;
  for (int z = lane; z < Ze; z += 32) {
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = (uint32_t)line[z + 2 * k] | ((uint32_t)line[z + 2 * k + 1] << 16);
    dst[z] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ---------------------------------------------------------------- host side
// op 0: gather with Cb == 1, Cs == 16 (valid conv, P = pad);  op 1: scatter with Cb == 16, Cs == 1 (P = 6 - pad)
static bool thin_a_shape(const cgan3d_conv_geom &g, int op) {
  if (g.k != 7 || g.stride != 1) return false;
  if (op == 0) return g.Cb == 1 && g.Cs == 16;
  if (op == 1) return g.Cb == 16 && g.Cs == 1;
  return false;
}

static bool plan_thin_a(const cgan3d_conv_geom &g, int op, ThinAPlan &best) {
  if (!thin_a_shape(g, op)) return false;
  ThinAPlan p{};
  p.B = g.B;
  if (op == 0) { p.Xi = g.Xb; p.Yi = g.Yb; p.Zi = g.Zb; p.Xo = g.Xs; p.Yo = g.Ys; p.Zo = g.Zs; p.P = g.pad; }
  else         { p.Xi = g.Xs; p.Yi = g.Ys; p.Zi = g.Zs; p.Xo = g.Xb; p.Yo = g.Yb; p.Zo = g.Zb; p.P = 6 - g.pad; }
  p.zshift = ((0 - p.P) % 8 + 8) % 8;
  p.Zc = round_up(p.Zi + 16, 8);
  p.nzb = (p.Zo + kZbA - 1) / kZbA;
  const int max_mt = 2;  // the accumulator ring needs at least two buffers of mtiles * N columns
  const uint32_t fixed = kTapTilesA * kTileBytesA / 2 + 16384 + 512;  // this CTA's Toeplitz half tiles, store staging, barriers
  double best_score = 0;
  bool found = false;
  for (int nyt = 1; nyt <= p.Yo; ++nyt) {
    const int Yt = (p.Yo + nyt - 1) / nyt, Yh = Yt + 6;
    if ((p.Yo + Yt - 1) / Yt != nyt) continue;
    if (Yh > 256) continue;
    for (int mt = 1; mt <= max_mt; ++mt) {
      if (Yt > mt * 128) continue;
      const int Xt = mn(p.Xo, (mt * 128 - Yt) / Yh + 1), Xh = Xt + 6;
      if (Xh > 256) continue;
      const int rows_alloc = round_up(mx(Xh * Yh, mt * 128 + 6 * Yh + 6), 32);  // 32-byte rows: slots are multiples of 1 KB
      const uint32_t slot = 2u * rows_alloc * 16;
      const int nslots = (int)mn<uint32_t>(6, (kSmemLimitThin - fixed) / slot);
      if (nslots < 2) continue;
      const int nxt = (p.Xo + Xt - 1) / Xt;
      const double eff = (double)p.Xo * p.Yo / ((double)nxt * nyt * mt * 128);
      const double halo = (double)(Xh * Yh) / (Xt * Yt);
      const double score = eff / (1.0 + kHaloWeightA * halo) * (nslots >= 3 ? 1.0 : 0.8);
      if (score > best_score + 1e-9) {
        best_score = score; found = true;
        best = p;
        best.Xt = Xt; best.Yt = Yt; best.Xh = Xh; best.Yh = Yh; best.nxt = nxt; best.nyt = nyt; best.mtiles = mt;
        best.rows_alloc = rows_alloc; best.slot_bytes = slot; best.nslots = nslots;
      }
    }
    if (nyt > 8 && found) break;
  }
  if (!found) return false;
  best.box_bytes = 32u * best.Yh * best.Xh;
  best.tmem_cols = 512;  // a ring of 512 / (mtiles * 128) accumulator buffers
  best.smem_bytes = fixed + best.nslots * best.slot_bytes;
  return true;
}

// op 0: gather with Cb == 16, Cs == 1;  op 1: scatter with Cb == 1, Cs == 16
static bool thin_b_shape(const cgan3d_conv_geom &g, int op) {
  if (g.k != 7 || g.stride != 1) return false;
  if (op == 0) return g.Cb == 16 && g.Cs == 1;
  if (op == 1) return g.Cb == 1 && g.Cs == 16;
  return false;
}

static bool plan_thin_b(const cgan3d_conv_geom &g, int op, ThinBPlan &p) {
  if (!thin_b_shape(g, op)) return false;
  p = ThinBPlan{};
  p.B = g.B;
  if (op == 0) { p.Xi = g.Xb; p.Yi = g.Yb; p.Zi = g.Zb; p.Xo = g.Xs; p.Yo = g.Ys; p.Zo = g.Zs; p.P = g.pad; }
  else         { p.Xi = g.Xs; p.Yi = g.Ys; p.Zi = g.Zs; p.Xo = g.Xb; p.Yo = g.Yb; p.Zo = g.Zb; p.P = 6 - g.pad; }
  // one y-line of the slab = 32 rows = one TMEM lane group: 26 output voxels + 6 halo voxels along z
  p.Zt = kZtB; p.Zh = kPitchB;
  p.nzt = (p.Zo + kZtB - 1) / kZtB;
  p.mtiles = mn(4, (p.Yo + 3) / 4);
  p.Yt = 4 * p.mtiles; p.Yh = p.Yt + 6;
  p.nyt = (p.Yo + p.Yt - 1) / p.Yt;
  p.rows_alloc = p.Yh * kPitchB;
  p.slot_bytes = (uint32_t)p.rows_alloc * 32;
  p.nslots = (int)mn<uint32_t>(6, (kSmemLimitThin - 14336 - 512) / p.slot_bytes);
  if (p.nslots < 2) return false;
  p.box_bytes = p.slot_bytes;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * p.mtiles * 64)) cols <<= 1;
  p.tmem_cols = cols;
  p.smem_bytes = 14336 + 512 + p.nslots * p.slot_bytes;
  return true;
}

// room for two shifted copies of the input (the workspace size callers allocate); the 8-z items read only the first
static size_t thin_a_repitch_bytes(const ThinAPlan &p) { return (size_t)2 * p.B * p.Xi * p.Yi * p.Zc * 2; }

bool thin_a_query(const cgan3d_conv_geom &g, int op, TcQuery &q) {
  ThinAPlan p;
  if (!plan_thin_a(g, op, p)) return false;
  q = {(size_t)kTapTilesA * kTileBytesA + 256 + thin_a_repitch_bytes(p) + 256, op == 0};
  return true;
}

bool thin_b_query(const cgan3d_conv_geom &g, int op, TcQuery &q) {
  ThinBPlan p;
  if (!plan_thin_b(g, op, p)) return false;
  q = {(size_t)kTapTilesB * kTileBytesB + 256, false};
  return true;
}

int thin_a_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st,
               double *bn_sums) {
  ThinAPlan p;
  if (!plan_thin_a(g, op, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 thin conv: shape not supported");
  if ((reinterpret_cast<uintptr_t>(in) & 15) || (reinterpret_cast<uintptr_t>(outp) & 15) || (reinterpret_cast<uintptr_t>(ws) & 255))
    return fail(CGAN3D_E_ARG, "tcgen05 thin conv: pointers must be 16-byte aligned (workspace 256)");
  bf16 *wt = reinterpret_cast<bf16 *>(ws);
  toeplitz_a_kernel<<<49, 256, 0, st>>>(reinterpret_cast<const bf16 *>(wp), wt, op);
  CG_LAUNCH_CHECK("toeplitz_a");
  bf16 *rp = reinterpret_cast<bf16 *>(reinterpret_cast<uint8_t *>(ws) + (size_t)kTapTilesA * kTileBytesA + 256);
  const long long rows = (long long)p.B * p.Xi * p.Yi;
  shifted_copies_kernel<<<(unsigned)((rows + 7) / 8), 256, (size_t)8 * ((p.Zc + 24 + 7) & ~7) * 2, st>>>(
      reinterpret_cast<const bf16 *>(in), rp, rows, p.Zi, p.Zc, p.zshift);
  CG_LAUNCH_CHECK("shifted_copies");
  CUtensorMap tm;  // the two shifted copies [2][B][Xi][Yi][Zc]
  const cuuint64_t zc = (cuuint64_t)p.Zc;
  const cuuint64_t gdim[5] = {zc, (cuuint64_t)p.Yi, (cuuint64_t)p.Xi, (cuuint64_t)p.B, 2};
  const cuuint64_t gstr[4] = {zc * 2, (cuuint64_t)p.Yi * zc * 2, (cuuint64_t)p.Xi * p.Yi * zc * 2, (cuuint64_t)rows * zc * 2};
  const cuuint32_t box[5] = {16, (cuuint32_t)p.Yh, (cuuint32_t)p.Xh, 1, 1};
  int r = encode_tiled(&tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, rp, gdim, gstr, box, nullptr, CU_TENSOR_MAP_SWIZZLE_32B, "thin conv");
  if (r) return r;
  CUtensorMap tmw;  // the Toeplitz tiles: 392 weight rows per CTA half, loaded as two boxes of 49 KB
  r = encode_weight_rows(&tmw, wt, kTapTilesA * kTileBytesA / 256, 196);
  if (r) return r;
  const long long total = (long long)p.B * p.nxt * p.nyt * p.nzb;
  const int grid = 2 * (int)mn<long long>((total + 1) / 2, (long long)(num_sms() / 2));
  auto launch = [&](auto mt_tag, auto st_tag) -> int {
    constexpr int MT = decltype(mt_tag)::value;
    constexpr bool ST = decltype(st_tag)::value;
    return tc_launch<conv7_c1_tc_kernel<MT, ST>>("conv7_c1_tc_kernel", grid, 192, p.smem_bytes + 1024, 2, st, tm, tmw,
                                                 reinterpret_cast<bf16 *>(outp), p, bn_sums);
  };
  if (p.mtiles == 1) return bn_sums ? launch(std::integral_constant<int, 1>{}, std::true_type{}) : launch(std::integral_constant<int, 1>{}, std::false_type{});
  if (p.mtiles == 2) return bn_sums ? launch(std::integral_constant<int, 2>{}, std::true_type{}) : launch(std::integral_constant<int, 2>{}, std::false_type{});
  return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 thin conv: mtiles %d not built", p.mtiles);
}

int thin_b_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st) {
  ThinBPlan p;
  if (!plan_thin_b(g, op, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 thin conv (16->1): shape not supported");
  if ((reinterpret_cast<uintptr_t>(in) & 15) || (reinterpret_cast<uintptr_t>(ws) & 15))
    return fail(CGAN3D_E_ARG, "tcgen05 thin conv: pointers must be 16-byte aligned");
  bf16 *wt = reinterpret_cast<bf16 *>(ws);
  stack_b_kernel<<<28, 256, 0, st>>>(reinterpret_cast<const bf16 *>(wp), wt, op);
  CG_LAUNCH_CHECK("stack_b");
  CUtensorMap tm;
  int r = encode_act_map(&tm, in, 16, p.Zi, p.Yi, p.Xi, p.B, 16, p.Zh, p.Yh, 1, 1, 32, "thin conv");
  if (r) return r;
  CUtensorMap tmw;  // the 7 filter tiles: 8 weight rows per tile, 4 per CTA half
  r = encode_weight_rows(&tmw, wt, kTapTilesB * kTileBytesB / 256, 4);
  if (r) return r;
  const long long ncols = (long long)p.B * p.nyt * p.nzt;
  const long long total = (ncols + 1) / 2 * p.Xo;
  const int grid = 2 * (int)mn<long long>(total, (long long)(num_sms() / 2));
  auto launch = [&](auto mt_tag) -> int {
    constexpr int MT = decltype(mt_tag)::value;
    return tc_launch<conv7_to1_tc_kernel<MT>>("conv7_to1_tc_kernel", grid, 320, p.smem_bytes + 1024, 2, st, tm, tmw,
                                              reinterpret_cast<bf16 *>(outp), p);
  };
  switch (p.mtiles) {
    case 1: return launch(std::integral_constant<int, 1>{});
    case 2: return launch(std::integral_constant<int, 2>{});
    case 3: return launch(std::integral_constant<int, 3>{});
    case 4: return launch(std::integral_constant<int, 4>{});
    default: return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 thin conv: mtiles %d not built", p.mtiles);
  }
}


// wgrad of the thin layers: `first` (Cb == 1, Cs == 16): S16 = small, Q1 = big;  `last_conv` (Cb == 16, Cs == 1): S16 = big
static bool plan_thin_c(const cgan3d_conv_geom &g, ThinCPlan &p) {
  if (g.k != 7 || g.stride != 1) return false;
  const bool first = g.Cb == 1 && g.Cs == 16, last = g.Cb == 16 && g.Cs == 1;
  if (!first && !last) return false;
  p = ThinCPlan{};
  p.B = g.B;
  if (first) { p.Xs = g.Xs; p.Ys = g.Ys; p.Zs = g.Zs; p.P = g.pad; p.flip = 0; }
  else       { p.Xs = g.Xb; p.Ys = g.Yb; p.Zs = g.Zb; p.P = 6 - g.pad; p.flip = 1; }
  p.Xe = p.Xs + 6; p.Ye = p.Ys + 6;
  p.nzt = (p.Zs + 255) / 256;
  p.Zt = round_up((p.Zs + p.nzt - 1) / p.nzt, 16);
  if (p.Zt > 256) { p.nzt += 1; p.Zt = round_up((p.Zs + p.nzt - 1) / p.nzt, 16); }
  p.Yt = mx(1, mn(p.Ys, 512 / p.Zt));
  if (p.Yt + 7 > 256) return false;
  p.nyt = (p.Ys + p.Yt - 1) / p.Yt;
  p.rowsB = p.Yt * p.Zt;
  p.kblocks = p.rowsB / 16;
  p.slotB_bytes = 2u * p.rowsB * 16;
  p.slotA_bytes = (uint32_t)(p.Yt + 7) * p.Zt * 16;
  p.boxB_bytes = 32u * p.Zt * p.Yt;
  p.boxA_bytes = p.slotA_bytes;
  const uint32_t fixed = kRingC * p.slotB_bytes + 512;
  if (fixed + 2 * p.slotA_bytes > kSmemLimitThin) return false;
  p.e_slots = (int)mn<uint32_t>(4, (kSmemLimitThin - fixed) / p.slotA_bytes);
  p.smem_bytes = fixed + p.e_slots * p.slotA_bytes;
  return true;
}

bool thin_c_query(const cgan3d_conv_geom &g, int, TcQuery &q) {
  ThinCPlan p;
  if (!plan_thin_c(g, p)) return false;
  q = {(size_t)p.B * p.Xe * p.Ye * p.Zs * 16 + 256, false};
  return true;
}

int thin_c_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, void *ws, cudaStream_t st) {
  ThinCPlan p;
  if (!plan_thin_c(g, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 thin wgrad: shape not supported");
  const bool first = p.flip == 0;
  const void *s16 = first ? small : big, *q1 = first ? big : small;
  const int Xq = first ? g.Xb : g.Xs, Yq = first ? g.Yb : g.Ys, Zq = first ? g.Zb : g.Zs;
  if ((reinterpret_cast<uintptr_t>(s16) & 15) || (reinterpret_cast<uintptr_t>(ws) & 15))
    return fail(CGAN3D_E_ARG, "tcgen05 thin wgrad: pointers must be 16-byte aligned");
  if (beta == 0.f) {
    cudaError_t e = cudaMemsetAsync(dw, 0, (size_t)16 * 343 * sizeof(float), st);
    if (e != cudaSuccess) return cuda_fail(e, "tcgen05 thin wgrad memset");
  }
  bf16 *E = reinterpret_cast<bf16 *>(ws);
  const long long elines = (long long)p.B * p.Xe * p.Ye;
  expand_z_kernel<<<(unsigned)((elines + 7) / 8), 256, (size_t)8 * ((p.Zs + 8 + 7) & ~7) * 2, st>>>(
      reinterpret_cast<const bf16 *>(q1), E, elines, Xq, Yq, Zq, p.Xe, p.Ye, p.Zs, p.P);
  CG_LAUNCH_CHECK("expand_z");
  CUtensorMap tmE, tmS;
  int r = encode_act_map(&tmE, E, 8, p.Zs, p.Ye, p.Xe, p.B, 8, p.Zt, p.Yt + 7, 1, 1, 0, "thin wgrad, expanded input");
  if (r) return r;
  r = encode_act_map(&tmS, s16, 16, p.Zs, p.Ys, p.Xs, p.B, 16, p.Zt, p.Yt, 1, 1, 32, "thin wgrad, 16 channels");
  if (r) return r;
  const long long total = (long long)p.B * p.nyt * p.nzt * p.Xe;
  const int grid = (int)mn<long long>(total, (long long)num_sms());
  return tc_launch<wgrad7_thin_tc_kernel>("wgrad7_thin_tc_kernel", grid, 192, p.smem_bytes + 1024, 1, st, tmE, tmS, dw, p);
}

}  // namespace cg
