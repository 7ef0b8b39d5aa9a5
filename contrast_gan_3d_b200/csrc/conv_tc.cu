// tcgen05 implicit-GEMM convolutions for sm_100a (bf16 operands, fp32 accumulation in TMEM).
//
// Kernel 1: conv_s1_tc_kernel — 3x3x3, stride 1, pad 1, Cin % 16 == 0, Cout % 16 == 0 (the 8 ResNet convs of the
// generator: 46 % of its FLOPs), used for fprop (gather) and for dgrad (scatter == gather with flipped, transposed
// filter).  Replaces aten::convolution / convolution_backward(input) at reference model/blocks.py:68-85.
//
// Design ("flattened-shift" implicit GEMM, no im2col materialisation, every input byte fetched from L2 once):
//   * One CTA owns an output slab (b, x0..x0+xlen, y0..y0+Yt, z0..z0+Zt) and marches along x.  For each input plane x
//     it TMA-loads the halo slab (Yt+2) x (Zt+2) x Cin ONCE, as Cin/8 boxes of 8 channels, into the UMMA
//     SWIZZLE_NONE K-major layout [Cin/8][row][8 ch] where row = yy*(Zt+2) + zz is the flattened halo position.
//     TMA's out-of-bounds zero fill implements the zero padding on all three axes.
//   * In that layout a filter tap (dx,dy,dz) is a pure ROW SHIFT of the A operand: the A descriptor for tap (dy,dz)
//     starts (dy*(Zt+2)+dz)*16 B further, plane dx selects one of three resident x-planes.  Output rows are the
//     flattened halo positions too; rows that fall on the halo columns are computed and discarded
//     (efficiency Yt*Zt / (mtiles*128)).
//   * Weights for one tap ([Cin/8][Cout][8] bf16, a K-major B operand) stream through a 4-stage ring with 1-D bulk
//     copies; each stage feeds mtiles*Cin/16 MMAs (M=128, N=Cout, K=16).
//   * Accumulators (mtiles x [128 x Cout] fp32) live in TMEM, double-buffered across output planes, so the
//     epilogue (tcgen05.ld -> bf16 -> 16 B global stores) of plane x overlaps the MMAs of plane x+1.
//   * Warp roles: 0-3 epilogue, 4 activation-plane TMA producer, 5 MMA issuer (+TMEM alloc), 6 weight producer.
#include "common.cuh"
#include "conv_internal.cuh"
#include "tc_common.cuh"

namespace cg {

struct TcPlan {
  int B, X, Y, Z, Cin, N;
  int Zt, nzt, Zh;
  int Yt, nslabs, Yh;
  int xseg, nxseg;
  int mtiles, rows_alloc, nitems, b_stages;
  int tps;  // filter taps per weight stage (3 = the dz taps of one (dx,dy): one barrier round trip and one commit per three taps)
  uint32_t plane_bytes, btile_bytes, box_bytes, tmem_cols, smem_bytes;
  int a_swz;  // 0: plane slab in Cin/8 chunks (SWIZZLE_NONE); 32/64/128: whole voxels, [row][Cin] in the matching swizzle mode
  int pair;   // 1: CTA pairs (cta_group::2): two columns per pair, each CTA holds half of the weight rows
};

constexpr int kPlaneSlots = 3;
constexpr int kThreads = 224;
constexpr uint32_t kSmemLimit = kMaxDynSmem - 1024;

// Work = ncols columns (b, z-tile, y-slab) x X output planes, flattened as idx = col * X + x.  CTA c owns the contiguous
// range [c*total/grid, (c+1)*total/grid): at most one plane of imbalance; a range that crosses a column boundary is
// processed as two items (each item re-loads its two halo planes).
struct ItemIter {
  int idx, end, rank;
  __device__ __forceinline__ ItemIter(const TcPlan &p) {
    // CTA pairs: the two CTAs of a cluster walk the same range of (column pair, plane) items in lockstep
    const int nblk = p.pair ? (int)gridDim.x >> 1 : (int)gridDim.x, blk = p.pair ? (int)blockIdx.x >> 1 : (int)blockIdx.x;
    const int ncols = p.pair ? (p.nitems + 1) >> 1 : p.nitems;
    rank = p.pair ? (int)blockIdx.x & 1 : 0;
    const long long total = (long long)ncols * p.X;
    idx = (int)(total * blk / nblk);
    end = (int)(total * (blk + 1) / nblk);
  }
  // live == false: the odd CTA of the last pair when the column count is odd (it computes a copy of the last column and stores nothing)
  __device__ __forceinline__ bool next(const TcPlan &p, int &b, int &z0, int &zlen, int &y0, int &ylen, int &x0, int &xlen, bool &live) {
    if (idx >= end) return false;
    int col = idx / p.X;
    x0 = idx - col * p.X;
    xlen = min(p.X - x0, end - idx);
    idx += xlen;
    live = true;
    if (p.pair) {
      col = 2 * col + rank;
      if (col >= p.nitems) { col = p.nitems - 1; live = false; }
    }
    const int sl = col % p.nslabs; col /= p.nslabs;
    const int zt = col % p.nzt;
    b = col / p.nzt;
    y0 = sl * p.Yt; ylen = min(p.Yt, p.Y - y0);
    z0 = zt * p.Zt; zlen = min(p.Zt, p.Z - z0);
    return true;
  }
};

// STATS: the epilogue also accumulates per-channel sum / sum of squares of the fp32 accumulators into bn_sums (fp64 [2*N],
// N <= 64): the BatchNorm batch statistics of reference model/blocks.py:45 without a separate pass over the output.
//
// PAIR: two CTAs of a cluster (one TPC) run as one cta_group::2 unit.  Each owns a column of the output and supplies its
// own activation planes (the A rows) plus HALF of every weight tile (the B rows), so the weight traffic per SM halves
// and one tcgen05.mma of the rank-0 CTA drives both tensor cores (50.8 instead of 77 cycles per M = 128, N = 64 slice).
// TMA loads of both CTAs count their bytes on the rank-0 barriers; its MMA commits are multicast to both CTAs.
template <int KSTEPS, int MT, bool STATS, bool PAIR>
__global__ void __launch_bounds__(kThreads, 1)
conv_s1_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const bf16 *__restrict__ wB,
                  bf16 *__restrict__ out, const TcPlan p, double *__restrict__ bn_sums) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *planes = smem;
  uint8_t *bt = planes + (size_t)kPlaneSlots * p.plane_bytes;
  const uint32_t stage_bytes = (uint32_t)p.tps * p.btile_bytes;
  uint64_t *bars = reinterpret_cast<uint64_t *>(bt + (size_t)p.b_stages * stage_bytes);
  uint64_t *plane_full = bars, *plane_empty = bars + kPlaneSlots;
  uint64_t *b_full = bars + 2 * kPlaneSlots, *b_empty = b_full + p.b_stages;
  uint64_t *tm_full = b_empty + p.b_stages, *tm_empty = tm_full + 2;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(tm_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kPlaneSlots; ++i) { tc::mbar_init(&plane_full[i], 1); tc::mbar_init(&plane_empty[i], 1); }
    for (int i = 0; i < p.b_stages; ++i) { tc::mbar_init(&b_full[i], 1); tc::mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&tm_full[i], 1); tc::mbar_init(&tm_empty[i], PAIR ? 8 : 4); }
    tc::fence_barrier_init();
  }
  const uint32_t cta_rank = PAIR ? tc::cluster_ctarank() : 0u;
  if constexpr (PAIR) {  // the peer's barriers must exist before anything signals them
    __syncthreads();
    tc::cluster_sync();
  }
  if (warp == 5) {
    if constexpr (PAIR) { tc::tmem_alloc2(tmem_ptr, p.tmem_cols); tc::tmem_relinquish2(); }
    else { tc::tmem_alloc(tmem_ptr, p.tmem_cols); tc::tmem_relinquish(); }
  }
  if (warp == 4 && lane == 0) tc::tma_prefetch_desc(&tmA);
  if (PAIR && warp == 6 && lane == 0) tc::tma_prefetch_desc(&tmW);
  tc::tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) tc::cluster_sync();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int kchunks8 = p.a_swz ? 1 : (p.Cin >> 3);
  const int taps = 27;

  if (warp == 4) {
    // ------------------------------------------------ activation-plane producer
    if (lane == 0) {
      uint32_t e = 0;
      int b, z0, zlen, y0, ylen, x0, xlen;
      bool live;
      for (ItemIter it(p); it.next(p, b, z0, zlen, y0, ylen, x0, xlen, live);) {
        for (int px = x0 - 1; px <= x0 + xlen; ++px, ++e) {
          const uint32_t slot = e % kPlaneSlots, use = e / kPlaneSlots;
          if (use > 0) tc::mbar_wait(&plane_empty[slot], (use - 1) & 1);
          uint8_t *dst = planes + (size_t)slot * p.plane_bytes;
          if constexpr (PAIR) {  // whole-voxel swizzled planes only
            if (cta_rank == 0) tc::mbar_expect_tx(&plane_full[slot], 2 * p.box_bytes);
            tc::tma_load_5d_2cta(dst, &tmA, &plane_full[slot], 0, z0 - 1, y0 - 1, px, b);
            continue;
          }
          tc::mbar_expect_tx(&plane_full[slot], p.box_bytes * kchunks8);
          if (p.a_swz) {
            tc::tma_load_5d(dst, &tmA, &plane_full[slot], 0, z0 - 1, y0 - 1, px, b);
          } else {
            for (int cc = 0; cc < kchunks8; ++cc)
              tc::tma_load_5d(dst + (size_t)cc * p.rows_alloc * 16, &tmA, &plane_full[slot], cc * 8, z0 - 1, y0 - 1, px, b);
          }
        }
      }
    }
  } else if (warp == 6) {
    // ------------------------------------------------ weight-tap producer
    if (lane == 0) {
      uint32_t t = 0;
      int b, z0, zlen, y0, ylen, x0, xlen;
      bool live;
      const int wrows = (int)(p.btile_bytes >> 8);  // 256-byte rows of the weight map per (tap, half) tile
      for (ItemIter it(p); it.next(p, b, z0, zlen, y0, ylen, x0, xlen, live);) {
        for (int i = 0; i < xlen; ++i)
          for (int tap = 0; tap < taps; tap += p.tps, ++t) {
            const uint32_t s = t % p.b_stages, use = t / p.b_stages;
            if (use > 0) tc::mbar_wait(&b_empty[s], (use - 1) & 1);
            uint8_t *dst = bt + (size_t)s * stage_bytes;
            if constexpr (PAIR) {
              if (cta_rank == 0) tc::mbar_expect_tx(&b_full[s], 2 * stage_bytes);
              for (int j = 0; j < p.tps; ++j)
                tc::tma_load_2d_2cta(dst + (size_t)j * p.btile_bytes, &tmW, &b_full[s], 0, ((tap + j) * 2 + (int)cta_rank) * wrows);
              continue;
            }
            tc::mbar_expect_tx(&b_full[s], stage_bytes);
            tc::bulk_g2s(dst, reinterpret_cast<const uint8_t *>(wB) + (size_t)tap * p.btile_bytes, stage_bytes, &b_full[s]);
          }
      }
    }
  } else if (warp == 5 && cta_rank != 0) {
    // the odd CTA of a pair issues nothing: the rank-0 CTA's MMAs read this CTA's planes and weights and write its TMEM
  } else if (warp == 5) {
    // ------------------------------------------------ MMA issuer
    // The whole warp runs the (warp-uniform) control flow so that ptxas keeps descriptors, TMEM addresses and loop
    // state in UNIFORM registers; only the tcgen05.mma / tcgen05.commit themselves are issued by one elected lane.
    // (A lane-0-only loop forces per-MMA R2UR transfers and made the issue thread, not the tensor pipe, the limit.)
    {
      const bool leader = tc::elect_one();
      const uint32_t idesc = tc::make_idesc_bf16(PAIR ? 256 : 128, p.N, 0, 0);
      const uint32_t planes_u32 = tc::smem_u32(planes), bt_u32 = tc::smem_u32(bt);
      const uint32_t a_lbo = (uint32_t)p.rows_alloc * 16, b_lbo = (uint32_t)(PAIR ? p.N >> 1 : p.N) * 16;
      auto mma = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t accum) {
        if constexpr (PAIR) tc::umma_bf16_2cta(d, ad, bd, idesc, accum);
        else tc::umma_bf16(d, ad, bd, idesc, accum);
      };
      auto commit = [&](uint64_t *bar) {
        if constexpr (PAIR) tc::umma_commit_2cta(bar, 3);
        else tc::umma_commit(bar);
      };
      const uint32_t a_row = p.a_swz ? (uint32_t)p.a_swz >> 4 : 1u;  // 16-byte units per activation row
      const uint64_t a_desc_hi = p.a_swz ? tc::make_desc_sw(0, 8u * p.a_swz, (uint32_t)p.a_swz) : tc::make_desc(0, a_lbo, 128);
      const uint64_t b_desc_hi = tc::make_desc(0, b_lbo, 128);
      const uint32_t a_kstep = p.a_swz ? 2u : (2 * a_lbo) >> 4, b_kstep = (2 * b_lbo) >> 4;  // descriptor address units (16 B)
      uint32_t e_base = 0, t = 0, acc = 0;
      const bool grouped = p.tps == 3;
      auto last_of_stage = [&](uint32_t j) { return !grouped || j == 2u; };
      int b, z0, zlen, y0, ylen, x0, xlen;
      bool live;
      for (ItemIter it(p); it.next(p, b, z0, zlen, y0, ylen, x0, xlen, live);) {
        for (int i = 0; i < xlen; ++i, ++acc) {
          const uint32_t q = acc & 1, uq = acc >> 1;
          if (uq > 0) tc::mbar_wait(&tm_empty[q], (uq - 1) & 1);
          tc::tc_fence_after();
          for (int dx = 0; dx < 3; ++dx) {
            const uint32_t e = e_base + i + dx, slot = e % kPlaneSlots;
            tc::mbar_wait(&plane_full[slot], (e / kPlaneSlots) & 1);
            tc::tc_fence_after();
            const uint32_t a_plane = (planes_u32 + slot * p.plane_bytes) >> 4;
            for (int dy = 0; dy < 3; ++dy)
              for (int dz = 0; dz < 3; ++dz) {
                const int tap = (dx * 3 + dy) * 3 + dz;
                const uint32_t s = t % p.b_stages, j = grouped ? (uint32_t)dz : 0u;  // tps is 1 or 3
                if (j == 0) {
                  tc::mbar_wait(&b_full[s], (t / p.b_stages) & 1);
                  tc::tc_fence_after();
                }
                const uint64_t b_desc0 = b_desc_hi | (uint64_t)(((bt_u32 + s * stage_bytes + j * p.btile_bytes) >> 4) & 0x3FFF);
                const uint32_t a_tap = a_plane + (uint32_t)(dy * p.Zh + dz) * a_row;
                const uint64_t a_desc0 = a_desc_hi | (uint64_t)(a_tap & 0x3FFF);
                const uint32_t d_tmem0 = tmem_base + q * (MT * p.N);
                if (leader) {
#pragma unroll
                  for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
                    for (int kk = 0; kk < KSTEPS; ++kk)
                      mma(d_tmem0 + mt * p.N, a_desc0 + (uint64_t)(mt * 128 * a_row + kk * a_kstep), b_desc0 + (uint64_t)(kk * b_kstep),
                          (uint32_t)((tap | kk) != 0));
                  }
                  if (last_of_stage(j)) commit(&b_empty[s]);
                }
                __syncwarp();
                if (last_of_stage(j)) ++t;
              }
            if (dx == 0 && leader) commit(&plane_empty[slot]);  // last use of input plane x-1
          }
          if (leader) commit(&tm_full[q]);
        }
        if (leader) {
          commit(&plane_empty[(e_base + xlen) % kPlaneSlots]);
          commit(&plane_empty[(e_base + xlen + 1) % kPlaneSlots]);
        }
        e_base += xlen + 2;
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------ epilogue (warps 0..3 <-> TMEM lanes 32*warp..)
    uint32_t acc = 0;
    float ssum[STATS ? 64 : 1], ssq[STATS ? 64 : 1];
    if (STATS) {
#pragma unroll
      for (int j = 0; j < 64; ++j) { ssum[j] = 0.f; ssq[j] = 0.f; }
    }
    int b, z0, zlen, y0, ylen, x0, xlen;
    bool live;
    for (ItemIter it(p); it.next(p, b, z0, zlen, y0, ylen, x0, xlen, live);) {
      for (int i = 0; i < xlen; ++i, ++acc) {
        const uint32_t q = acc & 1;
        tc::mbar_wait(&tm_full[q], (acc >> 1) & 1);
        tc::tc_fence_after();
        for (int mt = 0; mt < p.mtiles; ++mt) {
          const int r = mt * 128 + warp * 32 + lane;
          const int oy = r / p.Zh, oz = r - oy * p.Zh;
          const bool valid = live && oy < ylen && oz < zlen;
          bf16 *dst = out + ((((size_t)b * p.X + (x0 + i)) * p.Y + (y0 + oy)) * p.Z + (z0 + oz)) * p.N;
          const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (q * p.mtiles + mt) * p.N;
          auto store_chunk = [&](const uint32_t (&v)[16], int c0) {
            uint32_t pk[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
              pk[j] = *reinterpret_cast<uint32_t *>(&h);
            }
            tc::st_global_v8(dst + c0, pk);  // N % 16 == 0: 32-byte aligned
          };
          if (p.N <= 64) {  // up to four 16-channel chunks: all TMEM loads in flight before one wait
            uint32_t v[4][16];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc)
              if (cc * 16 < p.N) tc::tmem_ld16(taddr + cc * 16, v[cc]);
            tc::tmem_ld_wait();
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              if (cc * 16 < p.N && valid) {
                store_chunk(v[cc], cc * 16);
                if constexpr (STATS) {
#pragma unroll
                  for (int j = 0; j < 16; ++j) {
                    const float f = __uint_as_float(v[cc][j]);
                    ssum[cc * 16 + j] += f;
                    ssq[cc * 16 + j] += f * f;
                  }
                }
              }
            }
          } else {
            for (int c0 = 0; c0 < p.N; c0 += 16) {
              uint32_t v[16];
              tc::tmem_ld16(taddr + c0, v);
              tc::tmem_ld_wait();
              if (valid) store_chunk(v, c0);
            }
          }
        }
        tc::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (PAIR) tc::mbar_arrive_cluster(&tm_empty[q], 0);  // both CTAs' epilogues release the rank-0 issuer
          else tc::mbar_arrive(&tm_empty[q]);
        }
      }
    }
    if constexpr (STATS) {  // a thread saw at most a few dozen rows: fp32 partials, fp64 across threads
      warp_reduce64(ssum, lane);
      warp_reduce64(ssq, lane);
      const int ch = warp_reduce64_channel(lane);
#pragma unroll
      for (int i = 0; i < 2; ++i)
        if (ch + i < p.N) {
          atomicAdd(&bn_sums[0 + ch + i], (double)ssum[i]);
          atomicAdd(&bn_sums[p.N + 0 + ch + i], (double)ssq[i]);
        }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) {
    tc::cluster_sync();  // neither CTA may retire while the other can still signal its barriers or read its shared memory
    if (warp == 5) tc::tmem_dealloc2(tmem_base, p.tmem_cols);
  } else {
    if (warp == 5) tc::tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Kernel 1b: conv_s1_stack_kernel — the same convolution with TWO dz taps stacked on N (CTA pairs only, N <= 64).
//
// Why: a cta_group::2 MMA with N = 64 takes 59 cycles for 32 cycles of tensor work (profiles/r01_mma2_microbench.txt: the
// floor below N = 96 is the A-operand read), N = 128 takes 65 for 64.  Taps (dy, 0) and (dy, 1) read A rows one apart;
// out[r] = sum_dz G_dz[r + dz] with G_dz[m] = sum_{dx,dy} A_dx[m + dy*Zh] W[dx,dy,dz], so ONE MMA with the A rows of tap
// (dy, 0) and the weights [W(dy,0) | W(dy,1)] side by side produces G_0 in columns 0..N-1 and G_1 in columns N..2N-1 of the
// accumulator; tap (dy, 2) stays a plain N-wide MMA whose A rows are shifted by two, accumulating into the G_0 columns.
// Per (dx, dy) and K block: 65 + 59 cycles instead of 3 x 59.  The epilogue adds column group 1 of row r + 1 to column
// group 0 of row r: one warp shuffle per channel; the last lane of each warp gets its partner row from the next warp
// through shared memory after the main pass (rows r + 1 past the tile belong to rows that are never stored).
// Accumulators are 2N columns per M tile: two M tiles double-buffered fill the 512 TMEM columns at N = 64.
// The two CTAs of a pair hold the two stacked weight tiles (rank 0: W(dy,0), rank 1: W(dy,1)) — cta_group::2 takes columns
// 0..N-1 of B from rank 0 and N..2N-1 from rank 1 — and half each of W(dy,2).
constexpr int kStackThreads = 224;

template <int KSTEPS, int MT, bool STATS>
__global__ void __launch_bounds__(kStackThreads, 1)
conv_s1_stack_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, bf16 *__restrict__ out, const TcPlan p,
                     double *__restrict__ bn_sums) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *planes = smem;
  const uint32_t half_bytes = p.btile_bytes, stage_bytes = 3u * p.btile_bytes;  // per CTA: full tile (2 halves) + one half tile
  uint8_t *bt = planes + (size_t)kPlaneSlots * p.plane_bytes;
  float *xch = reinterpret_cast<float *>(bt + (size_t)p.b_stages * stage_bytes);  // [2 buffers][MT][4 warps][g0 of lane 31 | g1 of lane 0][64]
  uint64_t *bars = reinterpret_cast<uint64_t *>(xch + 2 * MT * 4 * 2 * 64);
  uint64_t *plane_full = bars, *plane_empty = bars + kPlaneSlots;
  uint64_t *b_full = bars + 2 * kPlaneSlots, *b_empty = b_full + p.b_stages;
  uint64_t *tm_full = b_empty + p.b_stages, *tm_empty = tm_full + 2;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(tm_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kPlaneSlots; ++i) { tc::mbar_init(&plane_full[i], 1); tc::mbar_init(&plane_empty[i], 1); }
    for (int i = 0; i < p.b_stages; ++i) { tc::mbar_init(&b_full[i], 1); tc::mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&tm_full[i], 1); tc::mbar_init(&tm_empty[i], 8); }
    tc::fence_barrier_init();
  }
  const uint32_t cta_rank = tc::cluster_ctarank();
  __syncthreads();
  tc::cluster_sync();  // the peer's barriers must exist before anything signals them
  if (warp == 5) { tc::tmem_alloc2(tmem_ptr, p.tmem_cols); tc::tmem_relinquish2(); }
  if (warp == 4 && lane == 0) tc::tma_prefetch_desc(&tmA);
  if (warp == 6 && lane == 0) tc::tma_prefetch_desc(&tmW);
  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int N = p.N, N2 = 2 * p.N;

  if (warp == 4) {
    // ------------------------------------------------ activation-plane producer (whole-voxel swizzled planes)
    if (lane == 0) {
      uint32_t slot = 0, use = 0;
      int b, z0, zlen, y0, ylen, x0, xlen;
      bool live;
      for (ItemIter it(p); it.next(p, b, z0, zlen, y0, ylen, x0, xlen, live);) {
        for (int px = x0 - 1; px <= x0 + xlen; ++px) {
          if (use > 0) tc::mbar_wait(&plane_empty[slot], (use - 1) & 1);
          if (cta_rank == 0) tc::mbar_expect_tx(&plane_full[slot], 2 * p.box_bytes);
          tc::tma_load_5d_2cta(planes + (size_t)slot * p.plane_bytes, &tmA, &plane_full[slot], 0, z0 - 1, y0 - 1, px, b);
          if (++slot == kPlaneSlots) { slot = 0; ++use; }
        }
      }
    }
  } else if (warp == 6) {
    // ------------------------------------------------ weight producer: one stage = the three dz taps of a (dx, dy)
    if (lane == 0) {
      uint32_t s = 0, use = 0;
      int b, z0, zlen, y0, ylen, x0, xlen;
      bool live;
      const int wrows = (int)(half_bytes >> 8);  // 256-byte rows of the weight map per half tile; a group is 6 half tiles
      for (ItemIter it(p); it.next(p, b, z0, zlen, y0, ylen, x0, xlen, live);) {
        for (int i = 0; i < xlen; ++i)
          for (int g = 0; g < 9; ++g) {
            if (use > 0) tc::mbar_wait(&b_empty[s], (use - 1) & 1);
            uint8_t *dst = bt + (size_t)s * stage_bytes;
            if (cta_rank == 0) tc::mbar_expect_tx(&b_full[s], 2 * stage_bytes);
            const int row0 = g * 6 * wrows;
            tc::tma_load_2d_2cta(dst, &tmW, &b_full[s], 0, row0 + (int)cta_rank * 2 * wrows);                       // W(dy, rank), first half of its rows
            tc::tma_load_2d_2cta(dst + half_bytes, &tmW, &b_full[s], 0, row0 + (int)cta_rank * 2 * wrows + wrows);  // ... second half
            tc::tma_load_2d_2cta(dst + 2 * half_bytes, &tmW, &b_full[s], 0, row0 + 4 * wrows + (int)cta_rank * wrows);  // this CTA's half of W(dy, 2)
            if (++s == (uint32_t)p.b_stages) { s = 0; ++use; }
          }
      }
    }
  } else if (warp == 5 && cta_rank != 0) {
    // the odd CTA of a pair issues nothing
  } else if (warp == 5) {
    // ------------------------------------------------ MMA issuer (whole warp runs the control flow, one lane issues)
    const bool leader = tc::elect_one();
    const uint32_t idesc2 = tc::make_idesc_bf16(256, N2, 0, 0), idesc1 = tc::make_idesc_bf16(256, N, 0, 0);
    const uint32_t planes_u32 = tc::smem_u32(planes), bt_u32 = tc::smem_u32(bt);
    // B, K-major SWIZZLE_NONE [Cin/8][rows][8]: the stacked tile has N rows per K chunk in each CTA, the single one N/2
    const uint32_t b_lbo2 = (uint32_t)N * 16, b_lbo1 = (uint32_t)(N >> 1) * 16;
    const uint32_t a_row = (uint32_t)p.a_swz >> 4;  // 16-byte units per activation row
    const uint64_t a_desc_hi = tc::make_desc_sw(0, 8u * p.a_swz, (uint32_t)p.a_swz);
    const uint64_t b_desc_hi2 = tc::make_desc(0, b_lbo2, 128), b_desc_hi1 = tc::make_desc(0, b_lbo1, 128);
    const uint32_t a_kstep = 2u, b_kstep2 = (2 * b_lbo2) >> 4, b_kstep1 = (2 * b_lbo1) >> 4;
    uint32_t pslot = 0, pph = 0;       // plane slot / parity of the item's first plane (x0 - 1)
    uint32_t s = 0, sph = 0, acc = 0;  // weight stage / its parity, output planes done
    int b, z0, zlen, y0, ylen, x0, xlen;
    bool live;
    for (ItemIter it(p); it.next(p, b, z0, zlen, y0, ylen, x0, xlen, live);) {
      for (int i = 0; i < xlen; ++i, ++acc) {
        const uint32_t q = acc & 1, uq = acc >> 1;
        if (uq > 0) tc::mbar_wait(&tm_empty[q], (uq - 1) & 1);
        tc::tc_fence_after();
        const uint32_t d_tmem0 = tmem_base + q * (MT * N2);
        uint32_t slot = pslot, ph = pph;
        for (int dx = 0; dx < 3; ++dx) {
          tc::mbar_wait(&plane_full[slot], ph);
          tc::tc_fence_after();
          const uint32_t a_plane = (planes_u32 + slot * p.plane_bytes) >> 4;
          for (int dy = 0; dy < 3; ++dy) {
            tc::mbar_wait(&b_full[s], sph);
            tc::tc_fence_after();
            const uint32_t bst = (bt_u32 + s * stage_bytes) >> 4;
            const uint64_t b2 = b_desc_hi2 | (uint64_t)(bst & 0x3FFF), b1 = b_desc_hi1 | (uint64_t)((bst + (2 * half_bytes >> 4)) & 0x3FFF);
            const uint64_t a0 = a_desc_hi | (uint64_t)((a_plane + (uint32_t)(dy * p.Zh) * a_row) & 0x3FFF);
            const uint64_t a2 = a_desc_hi | (uint64_t)((a_plane + (uint32_t)(dy * p.Zh + 2) * a_row) & 0x3FFF);
            if (leader) {
#pragma unroll
              for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
                for (int kk = 0; kk < KSTEPS; ++kk)
                  tc::umma_bf16_2cta(d_tmem0 + mt * N2, a0 + (uint64_t)(mt * 128 * a_row + kk * a_kstep), b2 + (uint64_t)(kk * b_kstep2), idesc2,
                                     (uint32_t)((dx | dy | kk) != 0));
              }
#pragma unroll
              for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
                for (int kk = 0; kk < KSTEPS; ++kk)
                  tc::umma_bf16_2cta(d_tmem0 + mt * N2, a2 + (uint64_t)(mt * 128 * a_row + kk * a_kstep), b1 + (uint64_t)(kk * b_kstep1), idesc1, 1u);
              }
              tc::umma_commit_2cta(&b_empty[s], 3);
            }
            __syncwarp();
            if (++s == (uint32_t)p.b_stages) { s = 0; sph ^= 1u; }
          }
          if (dx == 0 && leader) tc::umma_commit_2cta(&plane_empty[slot], 3);  // last use of input plane x - 1
          if (++slot == kPlaneSlots) { slot = 0; ph ^= 1u; }
        }
        if (leader) tc::umma_commit_2cta(&tm_full[q], 3);
        if (++pslot == kPlaneSlots) { pslot = 0; pph ^= 1u; }
      }
      // planes x0 + xlen - 1 and x0 + xlen of this item are still resident: release them, the next item starts two slots on
      if (leader) {
        tc::umma_commit_2cta(&plane_empty[pslot], 3);
        tc::umma_commit_2cta(&plane_empty[pslot + 1 >= kPlaneSlots ? pslot + 1 - kPlaneSlots : pslot + 1], 3);
      }
      pslot += 2;
      if (pslot >= kPlaneSlots) { pslot -= kPlaneSlots; pph ^= 1u; }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------ epilogue (warps 0..3 <-> TMEM lanes 32*warp..)
    const int tid = threadIdx.x;  // 0..127
    uint32_t acc = 0;
    float ssum[STATS ? 64 : 1], ssq[STATS ? 64 : 1];
    float fsum[4] = {0.f, 0.f, 0.f, 0.f}, fsq[4] = {0.f, 0.f, 0.f, 0.f};  // boundary rows: channels fch .. fch + 3 of this thread
    if (STATS) {
#pragma unroll
      for (int j = 0; j < 64; ++j) { ssum[j] = 0.f; ssq[j] = 0.f; }
    }
    const int cpt = N >> 4;                  // channels per thread in the boundary pass (16 threads per row): 4 at N = 64
    const int fch = (tid & 15) * cpt, frow = tid >> 4;  // boundary row (mt, w) = (frow >> 2, frow & 3)
    int b, z0, zlen, y0, ylen, x0, xlen;
    bool live;
    for (ItemIter it(p); it.next(p, b, z0, zlen, y0, ylen, x0, xlen, live);) {
      for (int i = 0; i < xlen; ++i, ++acc) {
        const uint32_t q = acc & 1;
        float *xq = xch + (size_t)q * (MT * 4 * 2 * 64);
        tc::mbar_wait(&tm_full[q], (acc >> 1) & 1);
        tc::tc_fence_after();
        bf16 *plane_out = out + (((size_t)b * p.X + (x0 + i)) * p.Y) * p.Z * N;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          const int r = mt * 128 + warp * 32 + lane;
          const int oy = r / p.Zh, oz = r - oy * p.Zh;
          const bool valid = live && oy < ylen && oz < zlen && lane < 31;  // lane 31 is finished in the boundary pass
          bf16 *dst = plane_out + ((size_t)(y0 + oy) * p.Z + (z0 + oz)) * N;
          const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (q * MT + mt) * N2;
          float *x0p = xq + ((mt * 4 + warp) * 2 + 0) * 64, *x1p = xq + ((mt * 4 + warp) * 2 + 1) * 64;
#pragma unroll
          for (int c2 = 0; c2 < 2; ++c2) {  // two 16-channel chunks of both column groups per TMEM wait
            if (c2 * 32 < N) {
              uint32_t v0[2][16], v1[2][16];
#pragma unroll
              for (int cc = 0; cc < 2; ++cc)
                if (c2 * 32 + cc * 16 < N) {
                  tc::tmem_ld16(taddr + c2 * 32 + cc * 16, v0[cc]);
                  tc::tmem_ld16(taddr + N + c2 * 32 + cc * 16, v1[cc]);
                }
              tc::tmem_ld_wait();
#pragma unroll
              for (int cc = 0; cc < 2; ++cc)
                if (c2 * 32 + cc * 16 < N) {
                  const int c0 = c2 * 32 + cc * 16;
                  if (lane == 0) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4)
                      *reinterpret_cast<float4 *>(x1p + c0 + j) = make_float4(__uint_as_float(v1[cc][j]), __uint_as_float(v1[cc][j + 1]),
                                                                              __uint_as_float(v1[cc][j + 2]), __uint_as_float(v1[cc][j + 3]));
                  }
                  if (lane == 31) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4)
                      *reinterpret_cast<float4 *>(x0p + c0 + j) = make_float4(__uint_as_float(v0[cc][j]), __uint_as_float(v0[cc][j + 1]),
                                                                              __uint_as_float(v0[cc][j + 2]), __uint_as_float(v0[cc][j + 3]));
                  }
                  float f[16];
#pragma unroll
                  for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v0[cc][j]) + __shfl_down_sync(0xffffffffu, __uint_as_float(v1[cc][j]), 1);
                  if (valid) {
                    uint32_t pk[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                      __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
                      pk[j] = *reinterpret_cast<uint32_t *>(&h);
                    }
                    tc::st_global_v8(dst + c0, pk);
                    if constexpr (STATS) {
#pragma unroll
                      for (int j = 0; j < 16; ++j) {
                        ssum[c0 + j] += f[j];
                        ssq[c0 + j] += f[j] * f[j];
                      }
                    }
                  }
                }
            }
          }
        }
        tc::tc_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive_cluster(&tm_empty[q], 0);  // both CTAs' epilogues release the rank-0 issuer
        asm volatile("bar.sync 1, 128;" ::: "memory");            // the boundary rows of all four warps are in shared memory
        if (frow < MT * 4) {
          const int mt = frow >> 2, w = frow & 3;
          const int mt2 = w == 3 ? mt + 1 : mt, w2 = w == 3 ? 0 : w + 1;  // the warp holding row r + 1
          const int r = mt * 128 + w * 32 + 31;
          const int oy = r / p.Zh, oz = r - oy * p.Zh;
          if (mt2 < MT && live && oy < ylen && oz < zlen) {
            const float *g0 = xq + ((mt * 4 + w) * 2 + 0) * 64 + fch, *g1 = xq + ((mt2 * 4 + w2) * 2 + 1) * 64 + fch;
            bf16 *dst = plane_out + ((size_t)(y0 + oy) * p.Z + (z0 + oz)) * N + fch;
            float f[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) f[j] = j < cpt ? g0[j] + g1[j] : 0.f;
            if (cpt == 4) {
              __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0], f[1]), h1 = __floats2bfloat162_rn(f[2], f[3]);
              uint2 pk;
              pk.x = *reinterpret_cast<uint32_t *>(&h0);
              pk.y = *reinterpret_cast<uint32_t *>(&h1);
              *reinterpret_cast<uint2 *>(dst) = pk;
            } else {
              for (int j = 0; j < cpt; ++j) dst[j] = __float2bfloat16_rn(f[j]);
            }
            if constexpr (STATS) {
#pragma unroll
              for (int j = 0; j < 4; ++j) { fsum[j] += f[j]; fsq[j] += f[j] * f[j]; }
            }
          }
        }
        // the next plane writes the OTHER exchange buffer; this one is rewritten two planes on, after the next bar.sync
      }
    }
    if constexpr (STATS) {
      // a thread saw at most a few dozen rows: fp32 partials; fp64 across the CTA in shared memory (the exchange buffers are
      // free now), then ONE global atomic per channel and CTA: with every thread adding its own partials 148 CTAs queued
      // ~1800 fp64 atomics on each of the 128 addresses at the same moment, ~18 us at the end of every launch
      double *sst = reinterpret_cast<double *>(xch);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (tid < N2) sst[tid] = 0.0;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      warp_reduce64(ssum, lane);
      warp_reduce64(ssq, lane);
      const int ch = warp_reduce64_channel(lane);
#pragma unroll
      for (int i = 0; i < 2; ++i)
        if (ch + i < N) {
          atomicAdd(&sst[ch + i], (double)ssum[i]);
          atomicAdd(&sst[N + ch + i], (double)ssq[i]);
        }
      if (frow < MT * 4) {
        for (int j = 0; j < cpt && j < 4; ++j) {
          atomicAdd(&sst[fch + j], (double)fsum[j]);
          atomicAdd(&sst[N + fch + j], (double)fsq[j]);
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (tid < N2) atomicAdd(&bn_sums[tid], sst[tid]);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();  // neither CTA may retire while the other can still signal its barriers or read its shared memory
  if (warp == 5) tc::tmem_dealloc2(tmem_base, p.tmem_cols);
}

// [tap][Cb][Cs] (generic packed) -> per (dx, dy) group: [W(.,0) full [Cin/8][N][8]] [W(.,1) full] [W(.,2) half 0 [Cin/8][N/2][8]]
// [W(.,2) half 1]; flip = dgrad (reverse taps, swap channel roles)
__global__ void repack_b_stack_kernel(const bf16 *__restrict__ wp, bf16 *__restrict__ wb, int Cb, int Cs, int flip) {
  const int Cin = flip ? Cs : Cb, N = flip ? Cb : Cs, Nh = N >> 1;
  const int64_t tile = (int64_t)Cin * N, total = 27 * tile;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int g = (int)(i / (3 * tile));
    int64_t t = i - (int64_t)g * 3 * tile;
    int dz, n, cc, c8;
    if (t < 2 * tile) {  // full tiles of dz = 0, 1
      dz = (int)(t / tile); t -= dz * tile;
      c8 = (int)(t & 7); t >>= 3;
      n = (int)(t % N);
      cc = (int)(t / N);
    } else {             // dz = 2, two halves of N
      t -= 2 * tile;
      dz = 2;
      const int h = (int)(t / (tile >> 1)); t -= (int64_t)h * (tile >> 1);
      c8 = (int)(t & 7); t >>= 3;
      n = h * Nh + (int)(t % Nh);
      cc = (int)(t / Nh);
    }
    const int tap = g * 3 + dz, ci = cc * 8 + c8;
    const int src_tap = flip ? (26 - tap) : tap;
    const int cb = flip ? n : ci, cs = flip ? ci : n;
    wb[i] = wp[((int64_t)src_tap * Cb + cb) * Cs + cs];
  }
}

// [tap][Cb][Cs] (generic packed) -> [tap'][half][Cin/8][N/nh][8]; flip = dgrad (reverse taps, swap channel roles);
// nh = 2 splits the output channels into the two halves held by the CTAs of a pair
__global__ void repack_b_kernel(const bf16 *__restrict__ wp, bf16 *__restrict__ wb, int Cb, int Cs, int taps, int flip, int nh) {
  const int Cin = flip ? Cs : Cb, N = flip ? Cb : Cs, Nl = N / nh;
  const int64_t total = (int64_t)taps * Cin * N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(i & 7);
    int64_t t = i >> 3;
    const int nl = (int)(t % Nl); t /= Nl;
    const int cc = (int)(t % (Cin >> 3)); t /= (Cin >> 3);
    const int h = (int)(t % nh);
    const int tap = (int)(t / nh);
    const int n = h * Nl + nl;
    const int ci = cc * 8 + c8;
    const int src_tap = flip ? (taps - 1 - tap) : tap;
    const int cb = flip ? n : ci, cs = flip ? ci : n;
    wb[i] = wp[((int64_t)src_tap * Cb + cb) * Cs + cs];
  }
}

// ---------------------------------------------------------------- host side
EncodeTiledFn tc_encode_fn() {
  static const EncodeTiledFn fn = [] {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      return reinterpret_cast<EncodeTiledFn>(p);
    return EncodeTiledFn{nullptr};
  }();
  return fn;
}

int encode_tiled(CUtensorMap *tm, CUtensorMapDataType dtype, int rank, const void *ptr, const cuuint64_t *gdim,
                 const cuuint64_t *gstr, const cuuint32_t *box, const cuuint32_t *estr, CUtensorMapSwizzle swizzle,
                 const char *what) {
  EncodeTiledFn enc = tc_encode_fn();
  if (!enc) return fail(CGAN3D_E_UNSUPPORTED, "cuTensorMapEncodeTiled not available");
  const cuuint32_t ones[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(tm, dtype, (cuuint32_t)rank, const_cast<void *>(ptr), gdim, gstr, box, estr ? estr : ones,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(CGAN3D_E_SHAPE, "cuTensorMapEncodeTiled (%s) failed with %d", what, (int)r);
  return 0;
}

int encode_weight_rows(CUtensorMap *tm, const void *ptr, int nrows, int box_rows) {
  const cuuint64_t gdim[2] = {64, (cuuint64_t)nrows};
  const cuuint64_t gstr[1] = {256};
  const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_INT32, 2, ptr, gdim, gstr, box, nullptr, CU_TENSOR_MAP_SWIZZLE_NONE,
                      "weight rows");
}

int encode_act_map(CUtensorMap *tm, const void *ptr, int C, int Z, int Y, int X, int B, int box_c, int nz, int ny, int ez,
                   int ey, int swizzle_bytes, const char *what) {
  const cuuint64_t gdim[5] = {(cuuint64_t)C, (cuuint64_t)Z, (cuuint64_t)Y, (cuuint64_t)X, (cuuint64_t)B};
  const cuuint64_t gstr[4] = {(cuuint64_t)C * 2, (cuuint64_t)Z * C * 2, (cuuint64_t)Y * Z * C * 2, (cuuint64_t)X * Y * Z * C * 2};
  // a box spans ez * (nz - 1) + 1 voxels along z, of which TMA loads every ez-th (likewise along y)
  const cuuint32_t box[5] = {(cuuint32_t)box_c, (cuuint32_t)(ez * (nz - 1) + 1), (cuuint32_t)(ey * (ny - 1) + 1), 1, 1};
  const cuuint32_t estr[5] = {1, (cuuint32_t)ez, (cuuint32_t)ey, 1, 1};
  const CUtensorMapSwizzle swz = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                 : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                       : CU_TENSOR_MAP_SWIZZLE_NONE;
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, ptr, gdim, gstr, box, estr, swz, what);
}

// CTA pairs need whole-voxel swizzled planes (one TMA box per plane), N/2 a multiple of 16 and 256-byte weight-map rows.
static bool pair_ok(int Cin, int N) { return Cin <= 64 && N % 32 == 0 && (Cin * N) % 256 == 0; }

static bool plan_s1(int B, int X, int Y, int Z, int Cin, int N, TcPlan &best) {
  if (N % 16 || N > 256 || N < 16) return false;
  if (Cin != 16 && Cin != 32 && Cin != 64 && Cin != 128) return false;
  TcPlan p{};
  p.B = B; p.X = X; p.Y = Y; p.Z = Z; p.Cin = Cin; p.N = N;
  p.pair = pair_ok(Cin, N) ? 1 : 0;
  p.nzt = (Z + 61) / 62;
  p.Zt = (Z + p.nzt - 1) / p.nzt;
  p.Zh = p.Zt + 2;
  p.btile_bytes = (uint32_t)Cin * N * 2 / (p.pair ? 2 : 1);
  p.tps = 3 * p.btile_bytes <= 16384 ? 3 : 1;
  const uint32_t stage_b = (uint32_t)p.tps * p.btile_bytes;
  p.b_stages = stage_b <= 8192 ? 4 : (stage_b <= 16384 ? 3 : 2);
  double best_eff = 0;
  bool found = false;
  for (int Yt = 1; Yt <= Y && Yt + 2 <= 256; ++Yt) {
    const int mt = (Yt * p.Zh + 127) / 128;
    if (2 * mt * N > 512 || mt > 4) break;
    const int rows_alloc = ((mt * 128 + 2 * p.Zh + 2) + 31) / 32 * 32;  // 2*Cin*rows_alloc is a multiple of 1024 (swizzle atom)
    const uint32_t plane_bytes = (uint32_t)(Cin / 8) * rows_alloc * 16;
    const uint32_t smem = kPlaneSlots * plane_bytes + p.b_stages * stage_b + 512;
    if (rows_alloc * 16 > 16383 * 16) break;
    if (smem > kSmemLimit) break;
    const int nslabs = (Y + Yt - 1) / Yt;
    const double eff = (double)Y * p.Zt / ((double)nslabs * mt * 128);
    if (eff > best_eff + 1e-9) {
      best_eff = eff;
      found = true;
      best = p;
      best.Yt = Yt; best.Yh = Yt + 2; best.nslabs = nslabs; best.mtiles = mt; best.rows_alloc = rows_alloc;
      best.plane_bytes = plane_bytes; best.smem_bytes = smem;
    }
  }
  if (!found) return false;
  TcPlan &q = best;
  {  // a deeper weight ring when shared memory is left over: one tap is consumed in mtiles * Cin/16 MMAs (~600 cycles for a
     // CTA pair at Cin = 64), well below the L2 latency of the next tile
    while (q.b_stages < 12 && q.smem_bytes + q.tps * q.btile_bytes <= kSmemLimit) { q.b_stages += 1; q.smem_bytes += q.tps * q.btile_bytes; }
  }
  q.a_swz = Cin <= 64 ? 2 * Cin : 0;
  q.box_bytes = (q.a_swz ? (uint32_t)q.a_swz : 16u) * q.Zh * q.Yh;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * q.mtiles * N)) cols <<= 1;
  q.tmem_cols = cols;
  q.xseg = X;
  q.nxseg = 1;
  q.nitems = B * q.nzt * q.nslabs;  // columns; the kernel splits columns x planes evenly over the grid
  return true;
}


// Tiling of the dz-stacked kernel: CTA pairs, whole-voxel swizzled planes, two M tiles of 2N accumulator columns, double
// buffered.
static bool plan_s1_stack(int B, int X, int Y, int Z, int Cin, int N, TcPlan &best) {
  if (!pair_ok(Cin, N)) return false;
  if (N > 64 || N % 32 || (Cin != 16 && Cin != 32 && Cin != 64)) return false;
  TcPlan p{};
  p.B = B; p.X = X; p.Y = Y; p.Z = Z; p.Cin = Cin; p.N = N;
  p.pair = 1;
  p.nzt = (Z + 61) / 62;
  p.Zt = (Z + p.nzt - 1) / p.nzt;
  p.Zh = p.Zt + 2;
  p.btile_bytes = (uint32_t)Cin * N;  // one half tile (N/2 rows)
  p.tps = 3;
  const uint32_t stage_b = 3u * p.btile_bytes;
  if ((p.btile_bytes & 255u) != 0) return false;
  p.b_stages = 3;
  p.a_swz = 2 * Cin;
  double best_eff = 0;
  bool found = false;
  for (int Yt = 1; Yt <= Y && Yt + 2 <= 256; ++Yt) {
    const int mt = (Yt * p.Zh + 127) / 128;
    if (mt > 2 || 2 * mt * 2 * N > 512) break;
    const int rows_alloc = ((mt * 128 + 2 * p.Zh + 2) + 31) / 32 * 32;
    const uint32_t plane_bytes = (uint32_t)rows_alloc * Cin * 2;
    const uint32_t smem = kPlaneSlots * plane_bytes + p.b_stages * stage_b + 2u * mt * 4 * 2 * 64 * 4 + 512;
    if (smem > kSmemLimit) break;
    const int nslabs = (Y + Yt - 1) / Yt;
    const double eff = (double)Y * p.Zt / ((double)nslabs * mt * 128);
    if (eff > best_eff + 1e-9) {
      best_eff = eff;
      found = true;
      best = p;
      best.Yt = Yt; best.Yh = Yt + 2; best.nslabs = nslabs; best.mtiles = mt; best.rows_alloc = rows_alloc;
      best.plane_bytes = plane_bytes; best.smem_bytes = smem;
    }
  }
  if (!found) return false;
  TcPlan &q = best;
  while (q.b_stages < 9 && q.smem_bytes + stage_b <= kSmemLimit) { q.b_stages += 1; q.smem_bytes += stage_b; }
  q.box_bytes = (uint32_t)q.a_swz * q.Zh * q.Yh;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * q.mtiles * 2 * N)) cols <<= 1;
  q.tmem_cols = cols;
  q.xseg = X;
  q.nxseg = 1;
  q.nitems = B * q.nzt * q.nslabs;
  return true;
}

bool s1_query(const cgan3d_conv_geom &g, int op, TcQuery &q) {
  if (op < 0 || op > 1 || g.k != 3 || g.stride != 1 || g.pad != 1) return false;
  if (g.Xb != g.Xs || g.Yb != g.Ys || g.Zb != g.Zs) return false;
  const int Cin = op == 0 ? g.Cb : g.Cs, N = op == 0 ? g.Cs : g.Cb;
  TcPlan p;
  if (!plan_s1(g.B, g.Xb, g.Yb, g.Zb, Cin, N, p)) return false;
  q = {(size_t)27 * g.Cb * g.Cs * 2 + 256, N <= 64};
  return true;
}

int s1_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st,
           double *bn_sums) {
  const int flip = op, Cin = flip ? g.Cs : g.Cb, N = flip ? g.Cb : g.Cs;
  TcPlan p;
  if (!plan_s1(g.B, g.Xb, g.Yb, g.Zb, Cin, N, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 conv: no tiling for this shape");
  if ((reinterpret_cast<uintptr_t>(in) & 15) || (reinterpret_cast<uintptr_t>(outp) & 31) || (reinterpret_cast<uintptr_t>(ws) & 15))
    return fail(CGAN3D_E_ARG, "tcgen05 conv: input / workspace must be 16-byte aligned, the output 32-byte aligned (256-bit stores)");
  bf16 *wb = reinterpret_cast<bf16 *>(ws);
  TcPlan ps;
  const bool stack = plan_s1_stack(g.B, g.Xb, g.Yb, g.Zb, Cin, N, ps);
  if (stack) {
    p = ps;
    repack_b_stack_kernel<<<64, 256, 0, st>>>(reinterpret_cast<const bf16 *>(wp), wb, g.Cb, g.Cs, flip);
    CG_LAUNCH_CHECK("repack_b_stack");
  } else {
    repack_b_kernel<<<64, 256, 0, st>>>(reinterpret_cast<const bf16 *>(wp), wb, g.Cb, g.Cs, 27, flip, p.pair ? 2 : 1);
    CG_LAUNCH_CHECK("repack_b");
  }
  CUtensorMap tm;
  int r = encode_act_map(&tm, in, Cin, p.Z, p.Y, p.X, p.B, p.a_swz ? Cin : 8, p.Zh, p.Yh, 1, 1, p.a_swz, "stride-1 conv");
  if (r) return r;
  CUtensorMap tmw{};
  if (p.pair) {  // one (tap, half) tile is btile_bytes / 256 weight rows
    r = encode_weight_rows(&tmw, wb, 27 * 2 * (int)(p.btile_bytes >> 8), (int)(p.btile_bytes >> 8));
    if (r) return r;
  }
  const long long work = (long long)(p.pair ? (p.nitems + 1) / 2 : p.nitems) * p.X;
  const int grid = p.pair ? 2 * (int)mn<long long>(work, (long long)(num_sms() / 2)) : (int)mn<long long>(work, (long long)num_sms());
  if (stack) {
    auto launch_k = [&](auto ks_tag, auto mt_tag, auto st_tag) -> int {
      constexpr int KS = decltype(ks_tag)::value;
      constexpr int MT = decltype(mt_tag)::value;
      constexpr bool ST = decltype(st_tag)::value;
      return tc_launch<conv_s1_stack_kernel<KS, MT, ST>>("conv_s1_stack_kernel", grid, kStackThreads, p.smem_bytes + 1024, 2, st, tm,
                                                         tmw, reinterpret_cast<bf16 *>(outp), p, bn_sums);
    };
    auto by_st = [&](auto ks_tag, auto mt_tag) -> int {
      return bn_sums ? launch_k(ks_tag, mt_tag, std::true_type{}) : launch_k(ks_tag, mt_tag, std::false_type{});
    };
    auto by_mt2 = [&](auto ks_tag) -> int {
      return p.mtiles == 1 ? by_st(ks_tag, std::integral_constant<int, 1>{}) : by_st(ks_tag, std::integral_constant<int, 2>{});
    };
    switch (Cin >> 4) {
      case 1: return by_mt2(std::integral_constant<int, 1>{});
      case 2: return by_mt2(std::integral_constant<int, 2>{});
      case 4: return by_mt2(std::integral_constant<int, 4>{});
      default: return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 stacked conv: Cin must be 16, 32 or 64");
    }
  }
  auto launch_s = [&](auto ks_tag, auto mt_tag, auto st_tag, auto pair_tag) -> int {
    constexpr int KS = decltype(ks_tag)::value;
    constexpr int MT = decltype(mt_tag)::value;
    constexpr bool ST = decltype(st_tag)::value;
    constexpr bool PR = decltype(pair_tag)::value;
    return tc_launch<conv_s1_tc_kernel<KS, MT, ST, PR>>("conv_s1_tc_kernel", grid, kThreads, p.smem_bytes + 1024, PR ? 2 : 1, st, tm, tmw,
                                                        (const bf16 *)wb, reinterpret_cast<bf16 *>(outp), p, bn_sums);
  };
  auto launch = [&](auto ks_tag, auto mt_tag) -> int {
    if (p.pair) {
      if constexpr (decltype(ks_tag)::value <= 4)
        return bn_sums ? launch_s(ks_tag, mt_tag, std::true_type{}, std::true_type{}) : launch_s(ks_tag, mt_tag, std::false_type{}, std::true_type{});
      else
        return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 conv: CTA pairs need Cin <= 64");
    }
    return bn_sums ? launch_s(ks_tag, mt_tag, std::true_type{}, std::false_type{}) : launch_s(ks_tag, mt_tag, std::false_type{}, std::false_type{});
  };
  auto by_mt = [&](auto ks_tag) -> int {
    switch (p.mtiles) {
      case 1: return launch(ks_tag, std::integral_constant<int, 1>{});
      case 2: return launch(ks_tag, std::integral_constant<int, 2>{});
      case 3: return launch(ks_tag, std::integral_constant<int, 3>{});
      case 4: return launch(ks_tag, std::integral_constant<int, 4>{});
      default: return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 conv: mtiles %d not built", p.mtiles);
    }
  };
  switch (Cin >> 4) {
    case 1: return by_mt(std::integral_constant<int, 1>{});
    case 2: return by_mt(std::integral_constant<int, 2>{});
    case 4: return by_mt(std::integral_constant<int, 4>{});
    case 8: return by_mt(std::integral_constant<int, 8>{});
    default: return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 conv: Cin must be 16, 32, 64 or 128");
  }
}

}  // namespace cg
