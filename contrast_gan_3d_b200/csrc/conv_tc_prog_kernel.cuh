// (kernel + launcher template; host planning lives in conv_tc_prog.cu, the instantiations in conv_tc_prog_ks*.cu)
// tcgen05 implicit GEMM for the STRIDED convolutions (stride 2, k = 3 or 4, pad 1): down-sampling convs of the
// generator and the critic (gather), ConvTranspose3d up-sampling and the dgrad of strided convs (scatter).
// Replaces aten::convolution / convolution_backward(input) / conv_transpose3d at reference model/generator.py:40-46,
// :60-76, model/discriminator.py:48-67 (via model/blocks.py:21-38,52).
//
// Both directions are decomposed into stride-1 "flattened-shift" sub-problems on the SMALL grid (see conv_tc.cu for the
// row-shift idea) and driven by a small host-built TAP PROGRAM:
//   * gather (small = conv_s2(big)): the big side is sampled by parity class.  For input x-plane 2*ox+dx-1 and class
//     (q, r) = parity of (y, z), one TMA load with elementStrides (1,2,2,1,1) fetches the sub-slab
//     y = 2*(y0+yy) - q, z = 2*(z0+zz) - r straight from the dense NDHWC tensor; inside a class every filter tap is a row
//     shift (0 or +1 line / +1 voxel).  One accumulator.
//   * scatter (big = conv_s2^T(small)): the 8 output parity phases (p,q,r) are 8 accumulators over the same small-grid
//     rows; each (phase, tap) pair that exists is one row-shifted MMA group on the small-side slab of plane i+xo.
//     The epilogue writes phase (p,q,r) of row (i,j,k) to big voxel (2i+p, 2j+q, 2k+r).
//   * Thin critic layers: Cin == 8 (gather) forms K = 16 from TWO z-adjacent taps of a parity class -- the second
//     8-channel K chunk is the same slab one row later (A-descriptor LBO = 16 bytes) and the filter tile holds the two
//     taps back to back; N (output channels) < 16 is padded to 16 with zero filter columns and only Nout channels are stored.
//   * Scatter, stacked mode (8*N <= 256 and the tiles fit): the 8 output phases are stacked on the MMA N dimension.  Every
//     (phase, tap) pair that reads the small-side slab at row shift (oy, oz) of plane i+xo goes into ONE MMA whose filter
//     tile has a zero block for the phases without such a tap: 8 (k = 3) or 27 (k = 4) MMA groups per row tile instead
//     of 27 / 64 -- an SS-mode MMA costs ~75-85 cycles for any N <= 128 (DESIGN §4.0).
//   * All filter tiles ([Cin/8][N][8] bf16 each) stay RESIDENT in shared memory for the whole kernel (<= 108 KB for
//     the layers of this model), so the only streamed operand is the activation slab; each slab is released as soon
//     as its taps are issued (ring of slots, no cross-plane reuse: these layers are L2/HBM-bound, SURVEY App. B).
#pragma once
#include "common.cuh"
#include "conv_internal.cuh"
#include "tc_common.cuh"

namespace cg {

constexpr int kMaxEntries = 16, kMaxTaps = 64;
constexpr uint32_t kSmemLimitProg = kMaxDynSmem - 1024;

struct ProgTap {
  uint16_t row_shift;  // rows (16 B units) added to the A descriptor start
  uint8_t btile;       // resident filter tile
  uint8_t acc;         // accumulator (output phase)
  uint8_t first;       // 1 = first MMA group into this accumulator (overwrite)
  uint8_t khalf;       // z-pair gather: 1 = the tap reads the SECOND voxel of the row (K offset of Cin elements)
  uint8_t pad[2];
};
struct ProgEntry {
  int8_t cx, cy, cz;  // TMA start coordinate = scale * tile origin + c*
  uint8_t ntaps, tap0;
  uint8_t pad[3];
};
struct ProgPlan {
  int B, Xg, Yg, Zg;     // small ("grid") side extents: rows of every MMA live on this grid
  int Xo, Yo, Zo;        // output tensor extents
  int Cin, N, nacc;      // N = MMA N (multiple of 16)
  int Nout;              // channels actually stored by this launch (<= N)
  int out_pitch, out_c0; // channels per output voxel / first channel of this launch (output-channel split: the filters of
                         // wide critic layers do not fit in shared memory, so the channels are covered by 2 or 4 launches)
  int paired;            // 1: Cin == 8, K = 16 is two z-adjacent taps (tile t holds filter taps tile_tap[t][0..1])
  uint32_t a_lbo_bytes;
  int a_swz;             // 0: activation slab in Cin/8 chunks [chunk][row][8 ch] (SWIZZLE_NONE); 32/64/128: whole voxels,
                         // [row][Cin] with 2*Cin-byte rows in the matching TMA/UMMA swizzle mode (one TMA per slab)
  int in_scale;          // 2: gather from the big side (strided TMA), 1: scatter from the small side
  int out_scale;         // 1: gather, 2: scatter (output voxel = out_scale*grid + phase)
  int Zt, nzt, Zh, Yt, nslabs, Yh;
  int mtiles, rows_alloc, nslots, nbt;
  int nentries, ntaps;
  uint32_t slot_bytes, btile_bytes, box_bytes, tmem_cols, smem_bytes;
  ProgEntry entries[kMaxEntries];
  ProgTap taps[kMaxTaps];
  int8_t tile_tap[kMaxTaps][2];  // paired mode: filter taps of the two K chunks of tile t (-1 = zero)
  int stack;                     // 1: scatter with the 8 phases stacked on N (tile t holds tap tile_phase_tap[t][phase])
  int Nmma;                      // N of one MMA (N, or 8*N when stacked)
  int acc_stride, mt_stride;     // TMEM columns between accumulators (phases) / between M-tiles
  int8_t tile_phase_tap[kMaxTaps][8];
  int pair;                      // 1: CTA pairs (cta_group::2); btile_bytes is then the HALF tile (Nmma/2 rows) held by one CTA
  int zpair;                     // 1: gather whose slab rows are z-adjacent voxel PAIRS (both z parity classes in one dense
                                 // 4*Cin-byte row): half the TMA requests of the per-class strided loads (DESIGN fact 10)
};

// STATS: the epilogue also accumulates the per-channel sum / sum of squares of the fp32 accumulators (BatchNorm batch
// statistics, reference model/blocks.py:45) into bn_sums (fp64 [2 * out_pitch], Nout <= 64).
// PAIR: CTA pairs as in conv_tc.cu -- the two CTAs of a cluster process consecutive steps in lockstep, each holds half of
// the rows of every resident filter tile, the rank-0 CTA issues the MMAs of both.
template <int KSTEPS, int MT, int STATS, bool PAIR>
__global__ void __launch_bounds__(192, 1)
conv_prog_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const bf16 *__restrict__ wB,
                    bf16 *__restrict__ out, const __grid_constant__ ProgPlan p, double *__restrict__ bn_sums) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t *bres = smem;                                         // resident filter tiles
  uint8_t *ring = bres + (((size_t)p.nbt * p.btile_bytes + 1023) & ~(size_t)1023);  // activation slab slots (1024-aligned)
  uint64_t *bars = reinterpret_cast<uint64_t *>(ring + (size_t)p.nslots * p.slot_bytes);
  uint64_t *b_ready = bars, *s_full = bars + 1, *s_empty = s_full + p.nslots;
  uint64_t *tm_full = s_empty + p.nslots, *tm_empty = tm_full + 2;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(tm_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tc::mbar_init(b_ready, 1);
    for (int i = 0; i < p.nslots; ++i) { tc::mbar_init(&s_full[i], 1); tc::mbar_init(&s_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(&tm_full[i], 1); tc::mbar_init(&tm_empty[i], PAIR ? 8 : 4); }
    tc::fence_barrier_init();
  }
  const uint32_t cta_rank = PAIR ? tc::cluster_ctarank() : 0u;
  if constexpr (PAIR) {
    __syncthreads();
    tc::cluster_sync();
  }
  if (warp == 5) {
    if constexpr (PAIR) { tc::tmem_alloc2(tmem_ptr, p.tmem_cols); tc::tmem_relinquish2(); }
    else { tc::tmem_alloc(tmem_ptr, p.tmem_cols); tc::tmem_relinquish(); }
  }
  tc::tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) tc::cluster_sync();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // contiguous, balanced range of steps (column-major over (b, z-tile, y-slab) x output plane); a CTA pair walks step
  // pairs (2j, 2j+1), an odd step count leaves the last odd CTA a dead copy of step 2j
  const long long total_steps = (long long)p.B * p.nzt * p.nslabs * p.Xg;
  const long long total = PAIR ? (total_steps + 1) / 2 : total_steps;
  const int nblk = PAIR ? (int)gridDim.x >> 1 : (int)gridDim.x, blk = PAIR ? (int)blockIdx.x >> 1 : (int)blockIdx.x;
  const int s_begin = (int)(total * blk / nblk), s_end = (int)(total * (blk + 1) / nblk);
  const int kch = (p.paired || p.a_swz) ? 1 : (p.Cin >> 3);
  auto decode = [&](int st, int &b, int &z0, int &zlen, int &y0, int &ylen, int &x) -> bool {
    bool live = true;
    if constexpr (PAIR) {
      st = 2 * st + (int)cta_rank;
      if (st >= total_steps) { st = (int)total_steps - 1; live = false; }
    }
    x = st % p.Xg; st /= p.Xg;
    const int sl = st % p.nslabs; st /= p.nslabs;
    const int zt = st % p.nzt;
    b = st / p.nzt;
    y0 = sl * p.Yt; ylen = min(p.Yt, p.Yg - y0);
    z0 = zt * p.Zt; zlen = min(p.Zt, p.Zg - z0);
    return live;
  };

  if (warp == 4) {
    // ------------------------------------------------ producer: resident filters once, then the slab stream
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmA);
      if constexpr (PAIR) {  // this CTA's half tiles, byte counts on the rank-0 barrier
        tc::tma_prefetch_desc(&tmW);
        if (cta_rank == 0) tc::mbar_expect_tx(b_ready, 2u * (uint32_t)p.nbt * p.btile_bytes);
        const int trows = (int)(p.btile_bytes >> 8);
        for (int t = 0; t < p.nbt; ++t)
          tc::tma_load_2d_2cta(bres + (size_t)t * p.btile_bytes, &tmW, b_ready, 0, ((int)cta_rank * p.nbt + t) * trows);
      } else {
        tc::mbar_expect_tx(b_ready, (uint32_t)p.nbt * p.btile_bytes);
        for (int t = 0; t < p.nbt; ++t)
          tc::bulk_g2s(bres + (size_t)t * p.btile_bytes, reinterpret_cast<const uint8_t *>(wB) + (size_t)t * p.btile_bytes,
                       p.btile_bytes, b_ready);
      }
      uint32_t e = 0;
      for (int st = s_begin; st < s_end; ++st) {
        int b, z0, zlen, y0, ylen, x;
        decode(st, b, z0, zlen, y0, ylen, x);
        for (int en = 0; en < p.nentries; ++en, ++e) {
          const ProgEntry &E = p.entries[en];
          const uint32_t slot = e % p.nslots, use = e / p.nslots;
          if (use > 0) tc::mbar_wait(&s_empty[slot], (use - 1) & 1);
          uint8_t *dst = ring + (size_t)slot * p.slot_bytes;
          const int cz = (p.zpair ? z0 : p.in_scale * z0) + E.cz, cy = p.in_scale * y0 + E.cy, cx = p.in_scale * x + E.cx;
          if constexpr (PAIR) {  // one box per slab (swizzled whole voxels, or the 8-channel critic slabs)
            if (cta_rank == 0) tc::mbar_expect_tx(&s_full[slot], 2 * p.box_bytes);
            tc::tma_load_5d_2cta(dst, &tmA, &s_full[slot], 0, cz, cy, cx, b);
            continue;
          }
          tc::mbar_expect_tx(&s_full[slot], p.box_bytes * kch);
          if (p.a_swz) {
            tc::tma_load_5d(dst, &tmA, &s_full[slot], 0, cz, cy, cx, b);
          } else {
            for (int cc = 0; cc < kch; ++cc)
              tc::tma_load_5d(dst + (size_t)cc * p.rows_alloc * 16, &tmA, &s_full[slot], cc * 8, cz, cy, cx, b);
          }
        }
      }
    }
  } else if (warp == 5 && cta_rank != 0) {
    // odd CTA of a pair: the rank-0 CTA issues the MMAs of both
  } else if (warp == 5) {
    // ------------------------------------------------ MMA issuer (warp-uniform control flow, one elected lane issues)
    const bool leader = tc::elect_one();
    const uint32_t idesc = tc::make_idesc_bf16(PAIR ? 256 : 128, p.Nmma, 0, 0);
    const uint32_t ring_u32 = tc::smem_u32(ring), b_u32 = tc::smem_u32(bres);
    const uint32_t a_lbo = p.a_lbo_bytes, b_lbo = (uint32_t)(PAIR ? p.Nmma >> 1 : p.Nmma) * 16;
    auto commit = [&](uint64_t *bar) {
      if constexpr (PAIR) tc::umma_commit_2cta(bar, 3);
      else tc::umma_commit(bar);
    };
    const uint32_t a_row = p.a_swz ? (uint32_t)p.a_swz >> 4 : 1u;  // 16-byte units per activation row
    const uint64_t a_hi = p.a_swz ? tc::make_desc_sw(0, 8u * p.a_swz, (uint32_t)p.a_swz) : tc::make_desc(0, a_lbo, 128);
    const uint64_t b_hi = tc::make_desc(0, b_lbo, 128);
    const uint32_t a_kstep = p.a_swz ? 2u : (2 * a_lbo) >> 4, b_kstep = (2 * b_lbo) >> 4;
    tc::mbar_wait(b_ready, 0);
    tc::tc_fence_after();
    uint32_t e = 0, acc = 0;
    for (int st = s_begin; st < s_end; ++st, ++acc) {
      const uint32_t q = acc & 1, uq = acc >> 1;
      if (uq > 0) tc::mbar_wait(&tm_empty[q], (uq - 1) & 1);
      tc::tc_fence_after();
      const uint32_t d_base = tmem_base + q * (uint32_t)(p.nacc * MT * p.N);
      for (int en = 0; en < p.nentries; ++en, ++e) {
        const ProgEntry &E = p.entries[en];
        const uint32_t slot = e % p.nslots;
        tc::mbar_wait(&s_full[slot], (e / p.nslots) & 1);
        tc::tc_fence_after();
        const uint32_t a_slot = (ring_u32 + slot * p.slot_bytes) >> 4;
        for (int t = 0; t < E.ntaps; ++t) {
          const ProgTap &T = p.taps[E.tap0 + t];
          const uint64_t a0 = a_hi | (uint64_t)((a_slot + T.row_shift * a_row + (uint32_t)T.khalf * (uint32_t)(p.Cin >> 3)) & 0x3FFF);
          const uint64_t b0 = b_hi | (uint64_t)(((b_u32 + (uint32_t)T.btile * p.btile_bytes) >> 4) & 0x3FFF);
          const uint32_t d0 = d_base + (uint32_t)T.acc * p.acc_stride;
          const uint32_t keep = T.first ? 0u : 1u;
          if (leader) {
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
              for (int kk = 0; kk < KSTEPS; ++kk) {
                if constexpr (PAIR)
                  tc::umma_bf16_2cta(d0 + mt * p.mt_stride, a0 + (uint64_t)(mt * 128 * a_row + kk * a_kstep), b0 + (uint64_t)(kk * b_kstep),
                                     idesc, (kk != 0) ? 1u : keep);
                else
                  tc::umma_bf16(d0 + mt * p.mt_stride, a0 + (uint64_t)(mt * 128 * a_row + kk * a_kstep), b0 + (uint64_t)(kk * b_kstep), idesc,
                                (kk != 0) ? 1u : keep);
              }
            }
          }
          __syncwarp();
        }
        if (leader) commit(&s_empty[slot]);
        __syncwarp();
      }
      if (leader) commit(&tm_full[q]);
      __syncwarp();
    }
  } else {
    // ------------------------------------------------ epilogue (warps 0..3 <-> TMEM lanes 32*warp..)
    uint32_t acc = 0;
    // STATS = channels tracked per thread (0, 32 or 64): 2 x 64 partial sums next to four 16-column TMEM chunks spilled
    float ssum[STATS ? STATS : 1], ssq[STATS ? STATS : 1];
    if (STATS) {
#pragma unroll
      for (int j = 0; j < STATS; ++j) { ssum[j] = 0.f; ssq[j] = 0.f; }
    }
    for (int st = s_begin; st < s_end; ++st, ++acc) {
      int b, z0, zlen, y0, ylen, x;
      const bool live = decode(st, b, z0, zlen, y0, ylen, x);
      const uint32_t q = acc & 1;
      tc::mbar_wait(&tm_full[q], (acc >> 1) & 1);
      tc::tc_fence_after();
      const uint32_t d_base = tmem_base + ((uint32_t)(warp * 32) << 16) + q * (uint32_t)(p.nacc * MT * p.N);
      // one 16-channel chunk of output phase `a`, M-tile `mt`: bf16 store (+ BatchNorm partial sums; cc is static)
      auto emit = [&](const uint32_t (&v)[16], int a, int mt, auto cc_tag) {
        constexpr int cc = decltype(cc_tag)::value;
        const int px = (a >> 2) & 1, py = (a >> 1) & 1, pz = a & 1;
        const int ox = p.out_scale * x + px;
        const int r = mt * 128 + warp * 32 + lane;
        const int gy = r / p.Zh, gz = r - gy * p.Zh;
        const int oy = p.out_scale * (y0 + gy) + py, oz = p.out_scale * (z0 + gz) + pz;
        if (!(live && gy < ylen && gz < zlen && ox < p.Xo && oy < p.Yo && oz < p.Zo)) return;
        bf16 *dst = out + ((((size_t)b * p.Xo + ox) * p.Yo + oy) * p.Zo + oz) * p.out_pitch + p.out_c0 + cc * 16;
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
          pk[j] = *reinterpret_cast<uint32_t *>(&h);
        }
        uint4 *d4 = reinterpret_cast<uint4 *>(dst);
        if (cc * 16 + 8 < p.Nout && (p.out_pitch & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 31) == 0) {
          tc::st_global_v8(dst, pk);  // 32-byte aligned: out_pitch and out_c0 are multiples of 16 channels
        } else {
          d4[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          if (cc * 16 + 8 < p.Nout) d4[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
        }
        if constexpr (STATS > cc * 16) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float f = __uint_as_float(v[j]);  // padded columns (>= Nout) hold exact zeros
            ssum[cc * 16 + j] += f;
            ssq[cc * 16 + j] += f * f;
          }
        }
      };
      // TMEM loads are issued four at a time before a single wait: a load -> wait -> store chain per chunk left the
      // epilogue latency-bound (ncu: tensor pipe 32 % active with neither L2 nor DRAM saturated)
      for (int mt = 0; mt < MT; ++mt) {
        const uint32_t t_mt = d_base + (uint32_t)(mt * p.mt_stride);
        if (p.nacc == 1) {  // gather: the (up to) four 16-channel chunks of the single accumulator
          uint32_t v[4][16];
          if (0 < p.Nout) tc::tmem_ld16(t_mt + 0, v[0]);
          if (16 < p.Nout) tc::tmem_ld16(t_mt + 16, v[1]);
          if (32 < p.Nout) tc::tmem_ld16(t_mt + 32, v[2]);
          if (48 < p.Nout) tc::tmem_ld16(t_mt + 48, v[3]);
          tc::tmem_ld_wait();
          if (0 < p.Nout) emit(v[0], 0, mt, std::integral_constant<int, 0>{});
          if (16 < p.Nout) emit(v[1], 0, mt, std::integral_constant<int, 1>{});
          if (32 < p.Nout) emit(v[2], 0, mt, std::integral_constant<int, 2>{});
          if (48 < p.Nout) emit(v[3], 0, mt, std::integral_constant<int, 3>{});
          if constexpr (STATS == 0) {
            for (int c0 = 64; c0 < p.Nout; c0 += 16) {  // wide layers (no fused statistics): one chunk at a time
              tc::tmem_ld16(t_mt + c0, v[0]);
              tc::tmem_ld_wait();
              const int r = mt * 128 + warp * 32 + lane;
              const int gy = r / p.Zh, gz = r - gy * p.Zh;
              if (live && gy < ylen && gz < zlen && x < p.Xo && y0 + gy < p.Yo && z0 + gz < p.Zo) {
                bf16 *dst = out + ((((size_t)b * p.Xo + x) * p.Yo + (y0 + gy)) * p.Zo + (z0 + gz)) * p.out_pitch + p.out_c0 + c0;
                uint32_t pk[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[0][2 * j]), __uint_as_float(v[0][2 * j + 1]));
                  pk[j] = *reinterpret_cast<uint32_t *>(&h);
                }
                if ((p.out_pitch & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 31) == 0) {
                  tc::st_global_v8(dst, pk);
                } else {
                  uint4 *d4 = reinterpret_cast<uint4 *>(dst);
                  d4[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                  d4[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                }
              }
            }
          }
        } else {  // scatter: 8 output phases, four at a time per 16-channel chunk
          auto phases4 = [&](auto cc_tag) {
            constexpr int cc = decltype(cc_tag)::value;
            if (cc * 16 >= p.Nout) return;
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              uint32_t v[4][16];
#pragma unroll
              for (int j = 0; j < 4; ++j) tc::tmem_ld16(t_mt + (uint32_t)((4 * g + j) * p.acc_stride + cc * 16), v[j]);
              tc::tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 4; ++j) emit(v[j], 4 * g + j, mt, cc_tag);
            }
          };
          phases4(std::integral_constant<int, 0>{});
          phases4(std::integral_constant<int, 1>{});
          phases4(std::integral_constant<int, 2>{});
          phases4(std::integral_constant<int, 3>{});
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) tc::mbar_arrive_cluster(&tm_empty[q], 0);
        else tc::mbar_arrive(&tm_empty[q]);
      }
    }
    if constexpr (STATS > 0) {  // a thread saw at most a few dozen rows: fp32 partials, fp64 across threads
      float r0[64], r1[64];
#pragma unroll
      for (int j = 0; j < 64; ++j) { r0[j] = j < STATS ? ssum[j < STATS ? j : 0] : 0.f; r1[j] = j < STATS ? ssq[j < STATS ? j : 0] : 0.f; }
      warp_reduce64(r0, lane);
      warp_reduce64(r1, lane);
      const int ch = warp_reduce64_channel(lane);
#pragma unroll
      for (int i = 0; i < 2; ++i)
        if (ch + i < p.Nout) {
          atomicAdd(&bn_sums[p.out_c0 + ch + i], (double)r0[i]);
          atomicAdd(&bn_sums[p.out_pitch + p.out_c0 + ch + i], (double)r1[i]);
        }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) {
    tc::cluster_sync();
    if (warp == 5) tc::tmem_dealloc2(tmem_base, p.tmem_cols);
  } else {
    if (warp == 5) tc::tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ---------------------------------------------------------------- launcher
// All kernel instantiations of one KSTEPS value (4 M-tile counts x 3 statistics widths x single CTA / CTA pair) are
// compiled in their own translation unit (conv_tc_prog_ks<K>.cu): in one file they took 3.5 minutes of serial nvcc time.
// conv_tc_prog.cu: enqueue repack_prog_kernel (generic packed filter -> resident tiles of plan p)
int repack_prog_launch(const bf16 *wp, bf16 *wb, int Cb, int Cs, int scatter, const ProgPlan &p, cudaStream_t st);

struct ProgLaunchArgs {
  CUtensorMap tm;
  cgan3d_conv_geom g;
  int scatter, nsplit, grid;
  const void *wp;
  void *outp, *ws;
  size_t part_bytes;
  double *bn_sums;
  cudaStream_t st;
};

template <int KS_>
int prog_launch_ks(ProgPlan &p, const ProgLaunchArgs &a) {
  const CUtensorMap &tm = a.tm;
  const cgan3d_conv_geom &g = a.g;
  const int scatter = a.scatter, nsplit = a.nsplit, grid = a.grid;
  const void *wp = a.wp;
  void *outp = a.outp, *ws = a.ws;
  const size_t part_bytes = a.part_bytes;
  double *bn_sums = a.bn_sums;
  cudaStream_t st = a.st;
  auto launch_s = [&](auto ks_tag, auto mt_tag, auto st_tag, auto pair_tag) -> int {
    constexpr int KS = decltype(ks_tag)::value;
    constexpr int MT = decltype(mt_tag)::value;
    constexpr int ST = decltype(st_tag)::value;
    constexpr bool PR = decltype(pair_tag)::value;
    for (int part = 0; part < nsplit; ++part) {  // output-channel parts (1 unless the filters exceed shared memory)
      p.out_c0 = part * p.Nout;
      bf16 *wb = reinterpret_cast<bf16 *>(reinterpret_cast<uint8_t *>(ws) + part * part_bytes);
      if (int rr = repack_prog_launch(reinterpret_cast<const bf16 *>(wp), wb, g.Cb, g.Cs, scatter, p, st)) return rr;
      CUtensorMap tmw{};
      if (PR) {  // the repacked half tiles as rows of 256 bytes
        if (int rw = encode_weight_rows(&tmw, wb, 2 * p.nbt * (int)(p.btile_bytes >> 8), (int)(p.btile_bytes >> 8))) return rw;
      }
      if (int rl = tc_launch<conv_prog_tc_kernel<KS, MT, ST, PR>>("conv_prog_tc_kernel", grid, 192, p.smem_bytes + 1024, PR ? 2 : 1, st,
                                                                 tm, tmw, (const bf16 *)wb, reinterpret_cast<bf16 *>(outp), p, bn_sums))
        return rl;
    }
    return 0;
  };
  using S0 = std::integral_constant<int, 0>;
  using S32 = std::integral_constant<int, 32>;
  using S64 = std::integral_constant<int, 64>;
  auto launch_st = [&](auto ks_tag, auto mt_tag, auto pair_tag) -> int {
    if (!bn_sums) return launch_s(ks_tag, mt_tag, S0{}, pair_tag);
    return p.Nout <= 32 ? launch_s(ks_tag, mt_tag, S32{}, pair_tag) : launch_s(ks_tag, mt_tag, S64{}, pair_tag);
  };
  auto launch = [&](auto ks_tag, auto mt_tag) -> int {
    if (p.pair) {
      if constexpr (decltype(ks_tag)::value <= 4)
        return launch_st(ks_tag, mt_tag, std::true_type{});
      else
        return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 strided conv: CTA pairs need Cin <= 64");
    }
    return launch_st(ks_tag, mt_tag, std::false_type{});
  };
  auto by_mt = [&](auto ks_tag) -> int {
    switch (p.mtiles) {
      case 1: return launch(ks_tag, std::integral_constant<int, 1>{});
      case 2: return launch(ks_tag, std::integral_constant<int, 2>{});
      case 3: return launch(ks_tag, std::integral_constant<int, 3>{});
      case 4: return launch(ks_tag, std::integral_constant<int, 4>{});
      default: return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 strided conv: mtiles %d not built", p.mtiles);
    }
  };
  return by_mt(std::integral_constant<int, KS_>{});
}

}  // namespace cg
