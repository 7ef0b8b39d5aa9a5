// Weight gradient of the generator's two thin 7x7x7 layers, second generation (replaces wgrad7_thin_tc_kernel +
// expand_z_kernel of conv_thin_tc.cu on the shapes it supports).
//   `first`     (reference model/generator.py:31-38, aten::convolution_backward weight path): S16 = dY [B,Xs,Ys,Zs,16],
//               Q1 = reflection-padded input [B,Xs+6,Ys+6,Zs+6], P = 0
//   `last_conv` (generator.py:77-83): S16 = padded input, Q1 = dY [B,Xs-6,...], P = 6, taps come out flipped
//   R[c][dx,dy,dz] = sum_v S16[v, c] * Q1[v + (dx,dy,dz) - P]
//
// What the first kernel lost (profiles/r01_ncu_full_wgrad7_last.txt: 0.198 of the bf16 peak, 3.4 GB of DRAM traffic for a
// 1.3 GB problem) and what changes here:
//   * the z-expanded operand E[v][j] = Q1[v + j] was materialised in HBM by a pre-pass (16 B per voxel written, then read
//     2.75x through the y halo).  Here it is built IN SHARED MEMORY by ten warps from the raw 1-channel lines (2 B per
//     voxel, L2 resident) that four more warps stage with cp.async: DRAM traffic = one read of S16.
//   * M was 64 (8 dy x 8 dz) with N = 64 (4 x-planes x 16 channels) and 2.5 MMAs per plane on average.  Here one E row
//     carries TWO x-planes (32-byte rows = [dx_lo][dz], SWIZZLE_32B MN-major, blocks of 16 M elements one slab LINE apart
//     = 8 dy blocks): M = 128.  N = 128 = the 8 S16 planes xe-6 .. xe+1 x 16 channels sitting in adjacent ring slots
//     (a ring of 14 planes whose first slots are mirrored behind its end, so a window never wraps): ONE M = 128, N = 128
//     MMA per 16 voxels and per PAIR of E planes, 14 of its 16 (dx_lo, plane) blocks and 49 of 64 rows useful.
//   * accumulator column = 16 * (plane - first plane of the window): the filter x-offset is dx = 6 - j + dx_lo.
// Split-K over CTAs (whole (b, y-tile) columns dealt round-robin, see SegIterW2), fp32 atomics at the end.
//
// Z-PAIR variant (template ZP = true, the default): a K row is a PAIR of z-adjacent voxels.  The S16 box is loaded as 64-byte
// rows (z parity, 16 channels) = 32 N elements per plane under SWIZZLE_64B, so the TMA engine handles half as many rows
// (its cost is per row, see the producer below) and N = 8 planes x 32 = 256; the E rows are the EVEN shifts only,
// E[l, rp][h][j] = line(h, l)[2 rp + j] — word-aligned windows of the staged line, half as many rows to build, no funnel
// shifts.  Accumulator column = 32 * plane + 16 * parity + c holds the partial sum over one z parity of the tap
// dz = j - parity; the epilogue adds lane (.., j) of the parity-0 columns to lane (.., j + 1) of the parity-1 columns.
#include "common.cuh"
#include "conv_internal.cuh"
#include "tc_common.cuh"

namespace cg {

constexpr uint32_t kSmemLimitW2 = kMaxDynSmem - 1024;
constexpr int kMaxRingW2 = 14;  // logical S16 plane slots: 8 live + 4 or 6 in flight (TMA runs 2 - 3 steps ahead of the MMAs)
constexpr int kMaxPrefW2 = 11;     // staged 32-bit words per fetch thread and step
constexpr int kBuildWarpsW2 = 10;  // warps 0-3 (also the epilogue) and 6-11 expand the operand
constexpr int kFetchWarp0W2 = 12;  // warps 12-15 fetch and stage the raw Q1 words
constexpr int kFetchersW2 = 128;
constexpr int kThreadsW2 = 512;
constexpr int kStagesW2 = 2;     // stages of the expanded operand
constexpr int kStageBufsW2 = 3;  // raw-line staging buffers (named barriers 1.. = full, 1 + kStageBufsW2.. = empty): the fetch
                                 // warps run two steps ahead of the builders
constexpr int kBuildersW2 = (kBuildWarpsW2 + kFetchersW2 / 32) * 32;  // threads on the named barrier shared by the build and fetch warps (see bar_sync_builders)

struct ThinW2Plan {
  int B, Xs, Ys, Zs;  // S16 extents
  int Xq, Yq, Zq;     // Q1 extents
  int Xe;             // E planes = Xs + 6
  int P, flip;
  int Zt, Yt, nyt, L; // z rows per line (multiple of 16, >= Zs), S16 lines per step, y tiles, E lines per step (Yt + 7)
  int LW;             // staged words per Q1 line segment
  int rows, kblocks;  // rows per S16 slot (Yt * zr), K blocks per step
  int ring, nphys, npairs;  // logical ring size; physical slots (>= ring: the first nphys - ring slots are mirrored)
  int nb16, inv_nb16;       // 16-row blocks per line and ceil(65536 / nb16)
  uint32_t slot_bytes, e2_bytes, box_bytes, stage_words, smem_bytes;
  int zp;     // z-pair variant: K rows are pairs of voxels (zr = Zt / 2 rows per line), else single voxels (zr = Zt)
  int zr;
};

// Work = ncols columns (b, y-tile) x npairs plane pairs.  Columns are dealt to the CTAs ROUND-ROBIN (CTA c takes columns
// c, c + grid, ... whole), so that at any moment the 148 CTAs stream the same planes of 148 ADJACENT y-tiles, i.e. one
// contiguous region of the 16-channel tensor: DRAM sees long sequential bursts instead of 148 scattered 8 KB pieces.  The
// columns of the last, incomplete round are split evenly by plane pairs (a range that crosses a column boundary becomes
// two segments), so every CTA gets the same number of steps to within one.
struct SegIterW2 {
  int n, rounds, r;
  long long rem_col0, idx, end;
  __device__ __forceinline__ SegIterW2(long long ncols, int n_) : n(n_), r(0) {
    rounds = (int)(ncols / gridDim.x);
    rem_col0 = (long long)rounds * gridDim.x;
    const long long total = (ncols - rem_col0) * n;
    idx = total * blockIdx.x / gridDim.x;
    end = total * (blockIdx.x + 1) / gridDim.x;
  }
  __device__ __forceinline__ long long steps() const { return (long long)rounds * n + (end - idx); }
  __device__ __forceinline__ bool next(int &col, int &p0, int &plen) {
    if (r < rounds) {
      col = r * (int)gridDim.x + (int)blockIdx.x;
      p0 = 0;
      plen = n;
      ++r;
      return true;
    }
    if (idx >= end) return false;
    const long long c = idx / n;
    col = (int)(rem_col0 + c);
    p0 = (int)(idx - c * n);
    plen = (int)mn<long long>(n - p0, end - idx);
    idx += plen;
    return true;
  }
};

// Hand-off of the staging buffers between the fetch warps (producers) and the build warps (consumers): named barriers
// 1 + buf ("full": 128 fetch threads arrive, 320 builders wait) and 1 + kStageBufsW2 + buf ("empty": the builders arrive, the
// fetchers wait).
__device__ __forceinline__ void bar_sync_id(uint32_t id) { static_assert(kBuildersW2 == 448, "barrier count"); asm volatile("bar.sync %0, 448;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void bar_arrive_id(uint32_t id) { asm volatile("bar.arrive %0, 448;" ::"r"(id) : "memory"); }

// The fetch warps walk this CTA's steps in order: (column, plane pair) advanced incrementally (SegIterW2::locate divides).
struct StepWalkW2 {
  int n, rounds, r, pair, col;
  long long rem_col0;
  __device__ __forceinline__ StepWalkW2(const SegIterW2 &it) : n(it.n), rounds(it.rounds), r(0), pair(0), rem_col0(it.rem_col0) {
    if (rounds > 0) {
      col = (int)blockIdx.x;
    } else {
      const long long c = it.idx / n;
      col = (int)(rem_col0 + c);
      pair = (int)(it.idx - c * n);
    }
    first_flat_col = (int)(rem_col0 + it.idx / n);
    first_flat_pair = (int)(it.idx % n);
  }
  int first_flat_col, first_flat_pair;
  __device__ __forceinline__ void advance() {
    if (++pair < n) return;
    pair = 0;
    if (r < rounds) {
      ++r;
      if (r < rounds) { col += (int)gridDim.x; return; }
      col = first_flat_col;
      pair = first_flat_pair;
      return;
    }
    ++col;
  }
};

template <bool ZP>
__global__ void __launch_bounds__(kThreadsW2, 1)
wgrad7_v2_kernel(const __grid_constant__ CUtensorMap tmS, const uint32_t *__restrict__ q1, float *__restrict__ dw,
                 const __grid_constant__ ThinW2Plan p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *ring = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);  // nphys S16 plane slots, [rows][16 ch], SWIZZLE_32B (TMA)
  uint8_t *e2 = ring + (size_t)p.nphys * p.slot_bytes;          // stages of the expanded operand, [L * Zt rows][2][8], SWIZZLE_32B
  uint32_t *stage = reinterpret_cast<uint32_t *>(e2 + (size_t)kStagesW2 * p.e2_bytes);  // raw Q1 line segments [2][L][LW]
  uint64_t *bars = reinterpret_cast<uint64_t *>(stage + (size_t)kStageBufsW2 * p.stage_words);
  uint64_t *s_full = bars, *s_empty = bars + kMaxRingW2, *e_full = s_empty + kMaxRingW2, *e_empty = e_full + kStagesW2, *done = e_empty + kStagesW2;
  uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr uint32_t kCols = ZP ? 256 : 128;  // accumulator columns: 8 planes x (32 | 16)
  constexpr uint32_t kNper = ZP ? 32 : 16;    // N elements per plane

  if (threadIdx.x == 0) {
    for (int i = 0; i < kMaxRingW2; ++i) { tc::mbar_init(&s_full[i], 1); tc::mbar_init(&s_empty[i], 1); }
    for (int i = 0; i < kStagesW2; ++i) { tc::mbar_init(&e_full[i], kBuildWarpsW2); tc::mbar_init(&e_empty[i], 1); }
    tc::mbar_init(done, 1);
    tc::fence_barrier_init();
  }
  if (warp == 5) {
    tc::tmem_alloc(tmem_ptr, kCols);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  if (warp < 4) {  // every MMA accumulates: start from zero
    for (int c0 = 0; c0 < (int)kCols; c0 += 16) tc::tmem_zero16(tmem_base + ((uint32_t)(warp * 32) << 16) + c0);
    tc::tmem_st_wait();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();

  const long long ncols = (long long)p.B * p.nyt;

  if (warp == 4) {
    // ------------------------------------------------ S16 plane producer (TMA).  A swizzled tensor map moves one inner row
    // (32 B of one voxel, or 64 B of a z pair) per request at ~3 cycles each, so the z-pair rows halve the engine's work
    // per plane; with everything else disabled the plane loads added 0.08 ms to the kernel.  A 16-byte cp.async producer
    // warp with the swizzle applied by hand was tried and is slower (5400 cycles per step).  Planes are numbered by the
    // order in which this CTA loads them: slot q % ring, mirrored at ring + slot when that exists.  A segment loads its 6
    // warm-up planes and then two planes per step, (ring - 8) / 2 steps ahead of the MMAs.
    if (lane == 0) {
      tc::tma_prefetch_desc(&tmS);
      // plane q of this CTA goes to slot q % ring on its (q / ring)-th use: both kept incrementally (a runtime division costs
      // this single thread ~100 cycles, and there were four per step)
      uint32_t slot = 0, use = 0;
      const uint32_t mirrored = (uint32_t)(p.nphys - p.ring);
      uint8_t *slot_ptr = ring;
      auto load_plane = [&](int xs, int b, int y0) {
        if (use > 0) tc::mbar_wait(&s_empty[slot], (use - 1) & 1);
        const bool mirror = slot < mirrored;
        tc::mbar_expect_tx(&s_full[slot], mirror ? 2 * p.box_bytes : p.box_bytes);
        tc::tma_load_5d(slot_ptr, &tmS, &s_full[slot], 0, 0, y0, xs, b);
        if (mirror) tc::tma_load_5d(slot_ptr + (size_t)p.ring * p.slot_bytes, &tmS, &s_full[slot], 0, 0, y0, xs, b);
        slot_ptr += p.slot_bytes;
        if (++slot == (uint32_t)p.ring) { slot = 0; ++use; slot_ptr = ring; }
      };
      int col, p0, plen;
      for (SegIterW2 it(ncols, p.npairs); it.next(col, p0, plen);) {
        const int b = col / p.nyt, y0 = (col - b * p.nyt) * p.Yt;
        for (int xs = 2 * p0 - 6; xs < 2 * p0; ++xs) load_plane(xs, b, y0);
        for (int i = 0; i < plen; ++i) {
          load_plane(2 * (p0 + i), b, y0);
          load_plane(2 * (p0 + i) + 1, b, y0);
        }
      }
    }
  } else if (warp == 5) {
    // ------------------------------------------------ MMA issuer
    const bool leader = tc::elect_one();
    // A: MN-major SWIZZLE_32B, 16 M elements per 32-byte row, further M blocks one slab line later (LBO), 8-row K groups 256 B
    const uint64_t a_hi = tc::make_desc_sw_mn(0, (uint32_t)p.zr * 32u, 256, 32);
    // B: MN-major, one N block per ring slot (LBO = slot stride): SWIZZLE_32B rows of 16 channels, or SWIZZLE_64B rows of
    // (z parity, 16 channels)
    const uint64_t b_hi = ZP ? tc::make_desc_sw_mn(0, p.slot_bytes, 512, 64) : tc::make_desc_sw_mn(0, p.slot_bytes, 256, 32);
    const uint32_t ring_u32 = tc::smem_u32(ring), e2_u32 = tc::smem_u32(e2);
    // planes waited for / steps issued / sequence number of the window's first plane; ws, wph = waited % ring and the parity
    // of waited / ring, w0s = w0 % ring (all incremental: no runtime divisions on this warp's critical path)
    uint32_t waited = 0, w0 = 0, ws = 0, wph = 0, w0s = 0, st = 0, eph = 0;  // st, eph: operand stage of the step and its parity
    const uint32_t ringn = (uint32_t)p.ring;
    int col, p0, plen;
    for (SegIterW2 it(ncols, p.npairs); it.next(col, p0, plen);) {
      w0 = waited;  // the segment's first window starts at its first warm-up plane
      w0s = ws;
      for (int i = 0; i < plen; ++i, w0 += 2) {
        while (waited < w0 + 8) {
          tc::mbar_wait(&s_full[ws], wph);
          ++waited;
          if (++ws == ringn) { ws = 0; wph ^= 1u; }
        }
        tc::mbar_wait(&e_full[st], eph);  // the builders fenced their plain stores into the async proxy before arriving
        tc::tc_fence_after();
        const uint32_t a0 = (e2_u32 + st * p.e2_bytes) >> 4;
        uint32_t j = 0;
        while (j < 8) {  // runs of window planes that are contiguous in the (mirrored) ring
          uint32_t slot = w0s + j;
          if (slot >= ringn) slot -= ringn;
          const uint32_t run = mn<uint32_t>(8 - j, (uint32_t)p.nphys - slot);
          const uint32_t idesc = tc::make_idesc_bf16(128, (int)(kNper * run), 1, 1);
          const uint32_t b0 = (ring_u32 + slot * p.slot_bytes) >> 4;
          const uint32_t d = tmem_base + kNper * j;
          if (leader) {
            uint64_t a_desc = a_hi | (uint64_t)(a0 & 0x3FFF), b_desc = b_hi | (uint64_t)(b0 & 0x3FFF);
#pragma unroll 4
            for (int kb = 0; kb < p.kblocks; ++kb) {
              tc::umma_bf16(d, a_desc, b_desc, idesc, 1u);
              a_desc += 32;  // 16 rows of 32 B
              b_desc += ZP ? 64 : 32;
            }
          }
          __syncwarp();
          j += run;
        }
        if (leader) {
          tc::umma_commit(&e_empty[st]);
          tc::umma_commit(&s_empty[w0s]);  // the two oldest planes leave the window (w0s is even, so is the ring)
          tc::umma_commit(&s_empty[w0s + 1]);
        }
        __syncwarp();
        w0s += 2;
        if (w0s >= ringn) w0s -= ringn;
        if (++st == (uint32_t)kStagesW2) { st = 0; eph ^= 1u; }
      }
      // the six planes still resident belong to this segment only
      if (leader)
        for (uint32_t k = 0; k < 6; ++k) tc::umma_commit(&s_empty[w0s + k >= ringn ? w0s + k - ringn : w0s + k]);
      __syncwarp();
    }
    if (leader) tc::umma_commit(done);
    __syncwarp();
  } else {
    // ------------------------------------------------ warps 0..3, 6..11: build the expanded operand (0..3 then run the
    // epilogue); warps 12..15: bring the raw Q1 words of the next steps into the staging buffers.  The roles are split
    // because the generic->async proxy fence that publishes the operand compiles to MEMBAR.ALL.CTA, which waits for every
    // outstanding global load of the executing thread: a warp that prefetches AND builds exposes the full load latency
    // (~1 us under load) in every step.  The staging area has kStageBufsW2 buffers handed over with arrive / wait named
    // barriers, so the fetch warps run two steps ahead of the builders.
    // Where the time went when measured with per-role cycle counters (`first` at C3, ~1590 cycles per step): the 8 N = 256
    // MMAs of a step read 96 KB of shared memory, the TMA fills write 23 KB (mirrors included), the builders move 36 KB, the
    // staging 10 KB: ~165 KB per step against 128 B/clk = 1290 cycles.  Shared-memory bandwidth, not the tensor pipe
    // (8 x 128 cycles), bounds the step (DESIGN fact 13); deeper rings, more operand stages and a fence on the MMA side
    // instead of the builders' changed nothing (DESIGN §4.2).
    const int ZqW = p.Zq >> 1;
    const SegIterW2 range(ncols, p.npairs);
    const uint32_t total = (uint32_t)range.steps();
    uint32_t n = 0;
    if (warp >= kFetchWarp0W2) {
      const int tid = (warp - kFetchWarp0W2) * 32 + lane;  // 0..127
      const int total_words = 2 * p.L * p.LW;
      // word i of this thread: staging index tid + 128 i = (h, l, w); rel = its offset from the step's base pointer.  Validity
      // is a bit mask over i: z range (fixed), line in [0, Yq) (changes with the column), plane in [0, Xq) (changes with the
      // step, one mask per plane h).  The words travel global -> shared as 4-byte zero-filling cp.async (src-size 0 for an
      // invalid word): no branches, no registers, and the load latency is covered by two steps of lookahead instead of
      // being exposed in this warp (first form: 11 branchy __ldg + st.shared per thread and step = 1700 cycles per step with
      // the warps never idle — the kernel's bottleneck).
      int rel[kMaxPrefW2];
      uint32_t zmask = 0, mh[2] = {0, 0};
      uint64_t lpack = 0;  // 4 bits of l per word
#pragma unroll
      for (int i = 0; i < kMaxPrefW2; ++i) {
        const int idx = tid + kFetchersW2 * i;
        rel[i] = 0;
        if (idx < total_words) {
          const int w = idx % p.LW, hl = idx / p.LW, l = hl % p.L, h = hl / p.L;
          const int wq = w - p.P / 2;  // staged word 0 holds Q1 z elements (-P, -P + 1); P is even
          if ((unsigned)wq < (unsigned)ZqW) zmask |= 1u << i;
          mh[h] |= 1u << i;
          lpack |= (uint64_t)l << (4 * i);  // L <= 15
          rel[i] = (h * p.Yq + l) * ZqW + w;
        }
      }
      StepWalkW2 walk(range);
      int cur_col = -1;
      uint32_t ymask = 0;
      const uint32_t *col_base = q1;  // Q1 word (b, x = 0, y = yb, z = -P) of the current column
      const long long plane_words = (long long)p.Yq * ZqW;
      const uint32_t stage_u32 = tc::smem_u32(stage) + (uint32_t)tid * 4u, stage_stride = p.stage_words * 4u;
      auto issue = [&](uint32_t buf) {  // raw Q1 words of this CTA's next step -> staging buffer `buf`
        if (walk.col != cur_col) {
          cur_col = walk.col;
          const int b = cur_col / p.nyt, y0 = (cur_col - b * p.nyt) * p.Yt;
          const int yb = y0 - p.P;
          col_base = q1 + ((long long)b * p.Xq * p.Yq + yb) * ZqW - p.P / 2;
          ymask = 0;
#pragma unroll
          for (int i = 0; i < kMaxPrefW2; ++i)
            if ((unsigned)(yb + (int)((lpack >> (4 * i)) & 15)) < (unsigned)p.Yq) ymask |= 1u << i;
        }
        const int xb = 2 * walk.pair - p.P;
        walk.advance();
        // base may point outside the tensor (halo): it is only dereferenced for in-range (plane, line)
        const uint32_t *base = col_base + (long long)xb * plane_words;
        const uint32_t valid = zmask & ymask & (((unsigned)xb < (unsigned)p.Xq ? mh[0] : 0u) | ((unsigned)(xb + 1) < (unsigned)p.Xq ? mh[1] : 0u));
        const uint32_t dst = stage_u32 + buf * stage_stride;
#pragma unroll
        for (int i = 0; i < kMaxPrefW2; ++i) {
          if (tid + kFetchersW2 * i < total_words) {  // uniform per (thread, i): resolved once, not data dependent
            const bool ok = (valid >> i) & 1u;
            const uint32_t *src = ok ? base + rel[i] : q1;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst + (uint32_t)(kFetchersW2 * i) * 4u), "l"(src), "r"(ok ? 4u : 0u) : "memory");
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      };
      // steps k .. k + 1 are in flight while step k is handed over; buffer (k + 2) % 3 was read by step k - 1
      const uint32_t nsb = (uint32_t)kStageBufsW2, ahead = nsb - 1;
      uint32_t issued = 0, ibuf = 0, buf = 0;
      for (; issued < ahead && issued < total; ++issued) {
        issue(ibuf);
        if (++ibuf == nsb) ibuf = 0;
      }
      for (; n < total; ++n) {
        // the group of step n is the oldest of (issued - n) <= 2 pending ones
        if (issued - n == 2) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        bar_arrive_id(1 + buf);
        if (++buf == nsb) buf = 0;
        if (issued < total) {
          if (issued >= nsb) bar_sync_id(1 + kStageBufsW2 + ibuf);  // the builders have finished reading step issued - nsb
          issue(ibuf);
          ++issued;
          if (++ibuf == nsb) ibuf = 0;
        }
      }
    } else {
      const int bw = warp < 4 ? warp : warp - 2;  // builder warp 0..9
      // E2[l * Zt + r][h][j] = line(h, l)[r + j], j = 0..7.  A warp iteration = 32 rows of one staged line (h, l): 5
      // conflict-free LDS (neighbouring lanes read overlapping words), one funnel shift per output word (odd rows start
      // in the upper half-word), one 16-byte STS (SWIZZLE_32B makes the 8 rows of a quarter-warp hit 8 different 16-byte
      // bank groups).  The 2 L ipl iterations of a step are dealt to the 6 builder warps as contiguous ranges.
      // Z-pair variant: E2[l * zr + rp][h][j] = line(h, l)[2 rp + j] = staged words rp .. rp + 3: four conflict-free LDS,
      // no shifts, 32 rows of a line per warp iteration cover 32 words.
      const int ipl = (p.zr + 31) >> 5, iters = 2 * p.L * ipl, per = (iters + kBuildWarpsW2 - 1) / kBuildWarpsW2;
      const int it0 = bw * per, it1 = mn(iters, it0 + per);
      const int hl0 = it0 / ipl, rb0 = it0 - hl0 * ipl;
      const uint32_t stage_u32 = tc::smem_u32(stage) + (uint32_t)(ZP ? lane : (lane >> 1)) * 4u, stage_stride = p.stage_words * 4u;
      const uint32_t lane_dst = (uint32_t)lane * 32u;
      const uint32_t swz = (uint32_t)((lane >> 2) & 1);  // rows advance by 32 per iteration: the swizzle phase is the lane's
      const uint32_t sh = (uint32_t)(lane & 1) << 4;
      uint32_t st = 0, use = 0, sb = 0;  // operand stage of step n and how often it has been used before; staging buffer
      // Z-pair fast path: a warp's iterations are the same in every step, so their shared-memory offsets live in registers
      // and all loads of a step are issued before the first store (the looped form below exposes the LDS -> STS latency of
      // every iteration: 240 cycles each while the tensor core is reading shared memory).
      constexpr int kFastPerW2 = 6;
      const bool fast = ZP && per <= kFastPerW2;
      uint32_t f_src[kFastPerW2], f_dst[kFastPerW2], f_ok = 0;
#pragma unroll
      for (int q = 0; q < kFastPerW2; ++q) {
        f_src[q] = f_dst[q] = 0;
        const int it = it0 + q;
        if (fast && it < it1) {
          const int hl = it / ipl, rb = it - hl * ipl, h = hl >= p.L ? 1 : 0, l = hl - h * p.L;
          if (rb * 32 + lane < p.zr) f_ok |= 1u << q;
          f_src[q] = (uint32_t)(hl * p.LW + rb * 32 + lane) * 4u;
          f_dst[q] = (uint32_t)(l * p.zr + rb * 32 + lane) * 32u + (((uint32_t)h ^ swz) << 4);
        }
      }
      for (; n < total; ++n) {
        bar_sync_id(1 + sb);  // the fetch warps have written this step's staging buffer
        if (use > 0) tc::mbar_wait(&e_empty[st], (use - 1) & 1);
        if (fast) {
          const uint32_t sbase = tc::smem_u32(stage) + sb * stage_stride, dbase = tc::smem_u32(e2) + st * p.e2_bytes;
          uint32_t a[kFastPerW2][4];
#pragma unroll
          for (int q = 0; q < kFastPerW2; ++q)
            if ((f_ok >> q) & 1u) {
              const uint32_t src = sbase + f_src[q];
              asm volatile("ld.shared.b32 %0, [%1];" : "=r"(a[q][0]) : "r"(src));
              asm volatile("ld.shared.b32 %0, [%1+4];" : "=r"(a[q][1]) : "r"(src));
              asm volatile("ld.shared.b32 %0, [%1+8];" : "=r"(a[q][2]) : "r"(src));
              asm volatile("ld.shared.b32 %0, [%1+12];" : "=r"(a[q][3]) : "r"(src));
            }
#pragma unroll
          for (int q = 0; q < kFastPerW2; ++q)
            if ((f_ok >> q) & 1u)
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dbase + f_dst[q]), "r"(a[q][0]), "r"(a[q][1]), "r"(a[q][2]), "r"(a[q][3]) : "memory");
        } else {
          const uint32_t dst_u32 = tc::smem_u32(e2) + st * p.e2_bytes + lane_dst;
          int it = it0, hl = hl0, rb = rb0;
          while (it < it1) {
            const int h = hl >= p.L ? 1 : 0, l = hl - h * p.L;
            uint32_t src = stage_u32 + sb * stage_stride + (uint32_t)(hl * p.LW + rb * (ZP ? 32 : 16)) * 4u;
            uint32_t d = dst_u32 + (uint32_t)(l * p.zr + rb * 32) * 32u + (((uint32_t)h ^ swz) << 4);
            int r = rb * 32 + lane;
#pragma unroll 2
            for (; rb < ipl && it < it1; ++rb, ++it, src += (ZP ? 128 : 64), d += 1024, r += 32) {
              if (r < p.zr) {
                uint32_t a0, a1, a2, a3, a4;
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(a0) : "r"(src));
                asm volatile("ld.shared.b32 %0, [%1+4];" : "=r"(a1) : "r"(src));
                asm volatile("ld.shared.b32 %0, [%1+8];" : "=r"(a2) : "r"(src));
                asm volatile("ld.shared.b32 %0, [%1+12];" : "=r"(a3) : "r"(src));
                if (ZP) {
                  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(d), "r"(a0), "r"(a1), "r"(a2), "r"(a3) : "memory");
                } else {
                  asm volatile("ld.shared.b32 %0, [%1+16];" : "=r"(a4) : "r"(src));
                  const uint32_t o0 = __funnelshift_r(a0, a1, sh), o1 = __funnelshift_r(a1, a2, sh), o2 = __funnelshift_r(a2, a3, sh),
                                 o3 = __funnelshift_r(a3, a4, sh);
                  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(d), "r"(o0), "r"(o1), "r"(o2), "r"(o3) : "memory");
                }
              }
            }
            rb = 0;
            ++hl;
          }
        }
        if (n + (uint32_t)kStageBufsW2 < total) bar_arrive_id(1 + kStageBufsW2 + sb);  // this warp has read the staging buffer: the fetch warps may refill it
        if (++sb == (uint32_t)kStageBufsW2) sb = 0;
        tc::fence_proxy_async();  // generic-proxy writes -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&e_full[st]);
        if (++st == (uint32_t)kStagesW2) { st = 0; ++use; }
      }
    }
    // epilogue: TMEM lane m = (dy = m >> 4, dx_lo = (m >> 3) & 1, dz = m & 7); column = 16 * j + c, dx = 6 - j + dx_lo
    if (n > 0 && warp < 4) {
      tc::mbar_wait(done, 0);
      tc::tc_fence_after();
      const int m = warp * 32 + lane, dy = m >> 4, dxl = (m >> 3) & 1, dz = m & 7;
      for (int j = 0; j < 8; ++j) {
        uint32_t v[16];
        tc::tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + kNper * (uint32_t)j, v);
        if (ZP) {
          // columns 16..31 of the plane: the odd-z partial sums, tap dz = (lane's j) - 1: take them from lane + 1
          uint32_t v1[16];
          tc::tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + kNper * (uint32_t)j + 16u, v1);
          tc::tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 16; ++c)
            v[c] = __float_as_uint(__uint_as_float(v[c]) + __shfl_down_sync(0xffffffffu, __uint_as_float(v1[c]), 1));
        } else {
          tc::tmem_ld_wait();
        }
        const int dx = 6 - j + dxl;
        if (dy < 7 && dz < 7 && dx >= 0 && dx < 7) {
          int tap = dx * 49 + dy * 7 + dz;
          if (p.flip) tap = 342 - tap;
#pragma unroll
          for (int c = 0; c < 16; ++c) atomicAdd(&dw[(size_t)c * 343 + tap], __uint_as_float(v[c]));
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 5) tc::tmem_dealloc(tmem_base, kCols);
}

// ---------------------------------------------------------------- host side
static bool plan_w2(const cgan3d_conv_geom &g, ThinW2Plan &p) {
  if (g.k != 7 || g.stride != 1) return false;
  const bool first = g.Cb == 1 && g.Cs == 16, last = g.Cb == 16 && g.Cs == 1;
  if (!first && !last) return false;
  p = ThinW2Plan{};
  p.B = g.B;
  if (first) { p.Xs = g.Xs; p.Ys = g.Ys; p.Zs = g.Zs; p.Xq = g.Xb; p.Yq = g.Yb; p.Zq = g.Zb; p.P = g.pad; p.flip = 0; }
  else       { p.Xs = g.Xb; p.Ys = g.Yb; p.Zs = g.Zb; p.Xq = g.Xs; p.Yq = g.Ys; p.Zq = g.Zs; p.P = 6 - g.pad; p.flip = 1; }
  if ((p.P & 1) || (p.Zq & 1)) return false;  // staged words hold aligned element pairs
  p.Xe = p.Xs + 6;
  p.npairs = (p.Xe + 1) / 2;
  p.Zt = (p.Zs + 15) / 16 * 16;
  if (p.Zt > 256) return false;
  p.LW = (p.Zt + 8) / 2 + 1;
  p.nb16 = p.Zt / 16;
  p.inv_nb16 = (65536 + p.nb16 - 1) / p.nb16;
  p.zp = (p.Zs & 1) ? 0 : 1;  // an odd extent keeps one voxel per K row
  p.zr = p.zp ? p.Zt / 2 : p.Zt;
  // pass 0 only takes a tile whose ring is the deep one (14 logical slots, >= 4 mirrored); pass 1 takes what fits
  for (int pass = p.zp ? 0 : 1; pass < 2 && p.Yt == 0; ++pass)
  for (int Yt = mn(p.Ys, 8); Yt >= 1; --Yt) {
    const int L = Yt + 7;
    if (2 * L * p.LW > kFetchersW2 * kMaxPrefW2) continue;
    if ((Yt * p.zr) % 16) continue;  // whole K blocks of 16 rows
    const uint32_t slot = (uint32_t)Yt * p.Zt * 32u;
    const uint32_t e2b = ((uint32_t)L * p.zr * 32u + 1023u) / 1024u * 1024u;
    const uint32_t stage_words = ((uint32_t)(2 * L * p.LW) + 3u) & ~3u;
    const uint32_t fixed = (uint32_t)kStagesW2 * e2b + (uint32_t)kStageBufsW2 * stage_words * 4 + 512;
    if (slot % 1024) continue;
    int nphys = (int)((kSmemLimitW2 - mn(kSmemLimitW2, fixed)) / slot);
    if (nphys > kMaxRingW2 + 6) nphys = kMaxRingW2 + 6;
    // ring of 14 (TMA three steps ahead) when at least four of its slots can be mirrored, else 12; a mirrored slot keeps the
    // window of 8 planes contiguous, so most steps need ONE N = 128 MMA per K block
    const int ring = nphys >= kMaxRingW2 + 4 ? kMaxRingW2 : 12;
    if (nphys < ring + 2 && Yt > 1) continue;
    if (nphys < ring) continue;
    if (pass == 0 && ring < kMaxRingW2) continue;
    if (nphys > ring + 6) nphys = ring + 6;  // windows start at even slots <= ring - 2: six mirrors make every window contiguous
    p.Yt = Yt; p.L = L; p.nphys = nphys; p.ring = ring;
    p.slot_bytes = slot; p.e2_bytes = e2b; p.stage_words = stage_words;
    p.smem_bytes = fixed + (uint32_t)nphys * slot;
    break;
  }
  if (p.Yt == 0) return false;
  p.nyt = (p.Ys + p.Yt - 1) / p.Yt;
  p.rows = p.Yt * p.zr;
  p.kblocks = p.rows / 16;
  p.box_bytes = p.slot_bytes;
  return true;
}

bool thin_w2_query(const cgan3d_conv_geom &g, int, TcQuery &q) {
  ThinW2Plan p;
  if (!plan_w2(g, p)) return false;
  q = {0, false};
  return true;
}

int thin_w2_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st) {
  ThinW2Plan p;
  if (!plan_w2(g, p)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 thin wgrad v2: shape not supported");
  const bool first = p.flip == 0;
  const void *s16 = first ? small : big, *q1 = first ? big : small;
  if ((reinterpret_cast<uintptr_t>(s16) & 15) || (reinterpret_cast<uintptr_t>(q1) & 3))
    return fail(CGAN3D_E_ARG, "tcgen05 thin wgrad v2: the 16-channel tensor must be 16-byte aligned, the 1-channel tensor 4-byte aligned");
  if (beta == 0.f) {
    cudaError_t e = cudaMemsetAsync(dw, 0, (size_t)16 * 343 * sizeof(float), st);
    if (e != cudaSuccess) return cuda_fail(e, "tcgen05 thin wgrad v2 memset");
  }
  CUtensorMap tmS;  // rows of one voxel (16 channels, 32 B) or of a z-adjacent voxel pair (64 B)
  const int vox = p.zp ? 2 : 1;
  const int r = encode_act_map(&tmS, s16, 16 * vox, p.Zs / vox, p.Ys, p.Xs, p.B, 16 * vox, p.zr, p.Yt, 1, 1, 32 * vox, "thin wgrad v2");
  if (r) return r;
  const long long total = (long long)p.B * p.nyt * p.npairs;
  const int grid = (int)mn<long long>(total, (long long)num_sms());
  if (p.zp)
    return tc_launch<wgrad7_v2_kernel<true>>("wgrad7_v2_kernel", grid, kThreadsW2, p.smem_bytes + 1024, 1, st, tmS,
                                             reinterpret_cast<const uint32_t *>(q1), dw, p);
  return tc_launch<wgrad7_v2_kernel<false>>("wgrad7_v2_kernel", grid, kThreadsW2, p.smem_bytes + 1024, 1, st, tmS,
                                            reinterpret_cast<const uint32_t *>(q1), dw, p);
}

}  // namespace cg
