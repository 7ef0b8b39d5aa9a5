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
#include "conv_tc_prog_kernel.cuh"

namespace cg {

extern template int prog_launch_ks<1>(ProgPlan &, const ProgLaunchArgs &);
extern template int prog_launch_ks<2>(ProgPlan &, const ProgLaunchArgs &);
extern template int prog_launch_ks<4>(ProgPlan &, const ProgLaunchArgs &);
extern template int prog_launch_ks<8>(ProgPlan &, const ProgLaunchArgs &);

// [tap][Cb][Cs] (generic packed) -> resident tiles [tile][K/8][N][8]; gather: Cin=Cb, Nout=Cs; scatter: Cin=Cs, Nout=Cb.
// Normal mode: tile == filter tap, K = Cin.  Paired mode (Cin == 8): K chunk h of tile t holds filter tap tile_tap[t][h].
// Columns n >= Nout are zero.
__global__ void repack_prog_kernel(const bf16 *__restrict__ wp, bf16 *__restrict__ wb, int Cb, int Cs, int scatter,
                                   const __grid_constant__ ProgPlan p) {
  // CTA pairs: [half][tile][K/8][N/2][8], half = n / (N/2)
  const int K = p.paired ? 16 : p.Cin, N = p.Nmma, nh = p.pair ? 2 : 1, Nl = N / nh;
  const int64_t total = (int64_t)p.nbt * K * N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(i & 7);
    int64_t t = i >> 3;
    const int nl = (int)(t % Nl); t /= Nl;
    const int cc = (int)(t % (K >> 3)); t /= (K >> 3);
    const int tile = (int)(t % p.nbt);
    const int n = (int)(t / p.nbt) * Nl + nl;
    const int nn = p.stack ? n % p.N : n;  // stacked: row n = phase * N + channel
    const int tap = p.stack ? p.tile_phase_tap[tile][n / p.N] : (p.paired ? p.tile_tap[tile][cc] : tile);
    const int ci = p.paired ? c8 : cc * 8 + c8;
    bf16 v = __float2bfloat16_rn(0.f);
    if (nn < p.Nout && tap >= 0) {
      const int no = nn + p.out_c0;
      const int cb = scatter ? no : ci, cs = scatter ? ci : no;
      v = wp[((int64_t)tap * Cb + cb) * Cs + cs];
    }
    wb[i] = v;
  }
}

int repack_prog_launch(const bf16 *wp, bf16 *wb, int Cb, int Cs, int scatter, const ProgPlan &p, cudaStream_t st) {
  repack_prog_kernel<<<64, 256, 0, st>>>(wp, wb, Cb, Cs, scatter, p);
  CG_LAUNCH_CHECK("repack_prog");
  return 0;
}

// ---------------------------------------------------------------- host: program + tiling
static bool build_program(const cgan3d_conv_geom &g, int scatter, ProgPlan &p) {
  const int k = g.k;
  if (g.stride != 2 || g.pad != 1 || (k != 3 && k != 4)) return false;
  int ne = 0, nt = 0;
  if (!scatter) {
    // classes by parity of (d - pad): class 0 <-> even offset (slab starts at 2*o), class 1 <-> odd offset (starts at 2*o-1)
    auto cls = [&](int d) { return (d - 1) & 1; };
    auto shift = [&](int d) { return (d - 1 + cls(d)) / 2; };  // rows of the sub-slab, >= 0
    bool first = true;
    if (p.zpair) {
      // rows are z pairs (2j, 2j + 1) of one y class, the slab starts at pair z0 - 1: tap dz reads input z = 2*o + dz - 1,
      // i.e. dz = 0 -> pair o - 1, second voxel; dz = 1 -> pair o, first voxel; dz = 2 -> pair o, second voxel
      if (k != 3) return false;
      for (int dx = 0; dx < k; ++dx)
        for (int q = 0; q < 2; ++q) {
          ProgEntry E{};
          E.cx = (int8_t)(dx - 1); E.cy = (int8_t)(-q); E.cz = (int8_t)(-1);
          E.tap0 = (uint8_t)nt; E.ntaps = 0;
          for (int dy = 0; dy < k; ++dy) {
            if (cls(dy) != q) continue;
            for (int dz = 0; dz < k; ++dz) {
              if (nt >= kMaxTaps) return false;
              ProgTap T{};
              T.row_shift = (uint16_t)(shift(dy) * p.Zh + (dz == 0 ? 0 : 1));
              T.khalf = (uint8_t)(dz == 1 ? 0 : 1);
              T.btile = (uint8_t)((dx * k + dy) * k + dz);
              T.acc = 0; T.first = first ? 1 : 0;
              first = false;
              p.taps[nt++] = T; E.ntaps++;
            }
          }
          if (E.ntaps == 0) continue;
          if (ne >= kMaxEntries) return false;
          p.entries[ne++] = E;
        }
      p.nacc = 1;
      p.nentries = ne;
      p.ntaps = nt;
      return true;
    }
    for (int dx = 0; dx < k; ++dx)
      for (int q = 0; q < 2; ++q)
        for (int r = 0; r < 2; ++r) {
          ProgEntry E{};
          E.cx = (int8_t)(dx - 1); E.cy = (int8_t)(-q); E.cz = (int8_t)(-r);
          E.tap0 = (uint8_t)nt; E.ntaps = 0;
          for (int dy = 0; dy < k; ++dy) {
            if (cls(dy) != q) continue;
            if (p.paired) {
              // the (1 or 2) z taps of this class become the two K chunks of one MMA: rows r + shift and r + shift + 1
              int dzs[2] = {-1, -1}, nz = 0;
              for (int dz = 0; dz < k; ++dz)
                if (cls(dz) == r) dzs[nz++] = dz;
              if (nz == 2 && shift(dzs[1]) != shift(dzs[0]) + 1) return false;
              if (nt >= kMaxTaps) return false;
              ProgTap T{};
              T.row_shift = (uint16_t)(shift(dy) * p.Zh + shift(dzs[0]));
              T.btile = (uint8_t)nt;
              p.tile_tap[nt][0] = (int8_t)((dx * k + dy) * k + dzs[0]);
              p.tile_tap[nt][1] = (int8_t)(nz == 2 ? (dx * k + dy) * k + dzs[1] : -1);
              T.acc = 0; T.first = first ? 1 : 0;
              first = false;
              p.taps[nt++] = T; E.ntaps++;
              continue;
            }
            for (int dz = 0; dz < k; ++dz) {
              if (cls(dz) != r) continue;
              if (nt >= kMaxTaps) return false;
              ProgTap T{};
              T.row_shift = (uint16_t)(shift(dy) * p.Zh + shift(dz));
              T.btile = (uint8_t)((dx * k + dy) * k + dz);
              T.acc = 0; T.first = first ? 1 : 0;
              first = false;
              p.taps[nt++] = T; E.ntaps++;
            }
          }
          if (E.ntaps == 0) continue;
          if (ne >= kMaxEntries) return false;
          p.entries[ne++] = E;
        }
    p.nacc = 1;
  } else {
    // big index I = 2*i + ph receives small index i + off through tap d iff (ph + 1 - d) is even, off = (ph + 1 - d) / 2
    int offmin = 0, offmax = 0;
    for (int ph = 0; ph < 2; ++ph)
      for (int d = 0; d < k; ++d)
        if (((ph + 1 - d) & 1) == 0) { const int o = (ph + 1 - d) / 2; offmin = min(offmin, o); offmax = max(offmax, o); }
    if (p.stack) {
      // tap of phase ph that reads the slab at offset off along one axis: d = ph + 1 - 2*off (if 0 <= d < k)
      auto tap1 = [&](int ph, int off) { const int d = ph + 1 - 2 * off; return (d >= 0 && d < k) ? d : -1; };
      bool first = true;
      for (int xo = offmin; xo <= offmax; ++xo) {
        ProgEntry E{};
        E.cx = (int8_t)xo; E.cy = (int8_t)offmin; E.cz = (int8_t)offmin;
        E.tap0 = (uint8_t)nt; E.ntaps = 0;
        for (int oy = offmin; oy <= offmax; ++oy)
          for (int oz = offmin; oz <= offmax; ++oz) {
            bool any = false;
            int8_t taps8[8];
            for (int ph = 0; ph < 8; ++ph) {
              const int dx = tap1(ph >> 2, xo), dy = tap1((ph >> 1) & 1, oy), dz = tap1(ph & 1, oz);
              taps8[ph] = (int8_t)((dx >= 0 && dy >= 0 && dz >= 0) ? (dx * k + dy) * k + dz : -1);
              any = any || taps8[ph] >= 0;
            }
            if (!any) continue;
            if (nt >= kMaxTaps) return false;
            ProgTap T{};
            T.row_shift = (uint16_t)((oy - offmin) * p.Zh + (oz - offmin));
            T.btile = (uint8_t)nt;
            T.acc = 0; T.first = first ? 1 : 0;
            first = false;
            for (int ph = 0; ph < 8; ++ph) p.tile_phase_tap[nt][ph] = taps8[ph];
            p.taps[nt++] = T; E.ntaps++;
          }
        if (E.ntaps == 0) continue;
        if (ne >= kMaxEntries) return false;
        p.entries[ne++] = E;
      }
      p.nacc = 8;
      p.nentries = ne;
      p.ntaps = nt;
      return true;
    }
    bool seen[8] = {false, false, false, false, false, false, false, false};
    for (int xo = offmin; xo <= offmax; ++xo) {
      ProgEntry E{};
      E.cx = (int8_t)xo; E.cy = (int8_t)offmin; E.cz = (int8_t)offmin;
      E.tap0 = (uint8_t)nt; E.ntaps = 0;
      for (int px = 0; px < 2; ++px)
        for (int dx = 0; dx < k; ++dx) {
          if (((px + 1 - dx) & 1) || (px + 1 - dx) / 2 != xo) continue;
          for (int py = 0; py < 2; ++py)
            for (int dy = 0; dy < k; ++dy) {
              if ((py + 1 - dy) & 1) continue;
              for (int pz = 0; pz < 2; ++pz)
                for (int dz = 0; dz < k; ++dz) {
                  if ((pz + 1 - dz) & 1) continue;
                  if (nt >= kMaxTaps) return false;
                  const int oy = (py + 1 - dy) / 2, oz = (pz + 1 - dz) / 2;
                  ProgTap T{};
                  T.row_shift = (uint16_t)((oy - offmin) * p.Zh + (oz - offmin));
                  T.btile = (uint8_t)((dx * k + dy) * k + dz);
                  T.acc = (uint8_t)((px * 2 + py) * 2 + pz);
                  T.first = seen[T.acc] ? 0 : 1;
                  seen[T.acc] = true;
                  p.taps[nt++] = T; E.ntaps++;
                }
            }
        }
      if (E.ntaps == 0) continue;
      if (ne >= kMaxEntries) return false;
      p.entries[ne++] = E;
    }
    p.nacc = 8;
  }
  p.nentries = ne;
  p.ntaps = nt;
  return true;
}

static bool plan_prog_split(const cgan3d_conv_geom &g, int scatter, ProgPlan &best, int nsplit);

// tries 1, 2, 4 output-channel splits; *nsplit_out receives the number of launches
static bool plan_prog(const cgan3d_conv_geom &g, int scatter, ProgPlan &best, int *nsplit_out = nullptr) {
  for (int ns = 1; ns <= 4; ns *= 2)
    if (plan_prog_split(g, scatter, best, ns)) {
      if (nsplit_out) *nsplit_out = ns;
      return true;
    }
  return false;
}

static bool plan_prog_split(const cgan3d_conv_geom &g, int scatter, ProgPlan &best, int nsplit) {
  if (g.stride != 2 || g.pad != 1 || (g.k != 3 && g.k != 4)) return false;
  const int Cin = scatter ? g.Cs : g.Cb, Nfull = scatter ? g.Cb : g.Cs;
  if (Nfull % nsplit || (nsplit > 1 && (Nfull / nsplit) % 16)) return false;
  const int Nout = Nfull / nsplit;
  const int paired = (!scatter && Cin == 8) ? 1 : 0;
  if (!paired && Cin != 16 && Cin != 32 && Cin != 64 && Cin != 128) return false;
  if (Nout % 8 || Nout < 8 || Nout > 256 || (Nout > 8 && Nout % 16)) return false;
  const int N = Nout < 16 ? 16 : Nout;
  const int nacc = scatter ? 8 : 1;
  // every big-side voxel must belong to a phase of some small-grid row (holds for transposed convs and for the dgrad of
  // convs over even extents; an odd extent with k = 4 has one more plane than 2*small)
  if (scatter && (g.Xb > 2 * g.Xs || g.Yb > 2 * g.Ys || g.Zb > 2 * g.Zs)) return false;
  const int halo = (scatter && g.k == 4) ? 2 : 1;  // extra rows/lines of the slab beyond the tile
  const int taps = g.k * g.k * g.k;
  ProgPlan p{};
  p.B = g.B; p.Xg = g.Xs; p.Yg = g.Ys; p.Zg = g.Zs;
  p.Xo = scatter ? g.Xb : g.Xs; p.Yo = scatter ? g.Yb : g.Ys; p.Zo = scatter ? g.Zb : g.Zs;
  p.Cin = Cin; p.N = N; p.nacc = nacc; p.Nout = Nout; p.paired = paired; p.out_pitch = Nfull; p.out_c0 = 0;
  p.in_scale = scatter ? 1 : 2; p.out_scale = scatter ? 2 : 1;
  p.nbt = paired ? taps / 2 + (g.k == 3 ? 9 : 0) : taps;  // upper bound; build_program fixes the exact count
  p.btile_bytes = (uint32_t)(paired ? 16 : Cin) * N * 2;
  p.Nmma = N; p.acc_stride = 0; p.mt_stride = N;  // acc_stride of the unstacked layout depends on mtiles (set below)
  // CTA pairs: one TMA box per slab (swizzled whole voxels or the 8-channel critic slabs) and N/2 a multiple of 16
  const bool pair_base = paired || Cin <= 64;
  p.pair = (pair_base && N % 32 == 0) ? 1 : 0;
  if (p.pair) p.btile_bytes /= 2;
  if (scatter && 8 * N <= 256) {
    const int ncombo = g.k == 3 ? 8 : 27;
    const uint32_t tile = (uint32_t)Cin * 8 * N * 2 / (pair_base ? 2 : 1);
    if ((ncombo * tile + 1023) / 1024 * 1024 + 40000 <= kSmemLimitProg) {
      p.stack = 1; p.Nmma = 8 * N; p.nbt = ncombo; p.btile_bytes = tile; p.pair = pair_base ? 1 : 0;
    }
  }
  const uint32_t b_total = (p.nbt * p.btile_bytes + 1023) / 1024 * 1024;
  if (b_total + 40000 > kSmemLimitProg) return false;
  const bool zpair = !scatter && !paired && (Cin == 16 || Cin == 32) && g.k == 3 && g.Zb % 2 == 0;
  p.zpair = zpair ? 1 : 0;
  const int a_swz = zpair ? 4 * Cin : ((!paired && Cin <= 64) ? 2 * Cin : 0);
  double best_score = 0;
  bool found = false;
  for (int nzt = 1; nzt <= 4; ++nzt) {
    const int Zt = (p.Zg + nzt - 1) / nzt, Zh = Zt + halo;
    if (2 * (Zh - 1) + 1 > 256) continue;
    for (int Yt = 1; Yt <= p.Yg; ++Yt) {
      const int Yh = Yt + halo;
      if (2 * (Yh - 1) + 1 > 256) break;
      const int mt = (Yt * Zh + 127) / 128;
      if (mt > 4 || 2 * nacc * mt * N > 512) break;
      const int rows_alloc = ((mt * 128 + halo * Zh + halo) + 7) / 8 * 8;
      if (rows_alloc > 16383 || Yh * Zh > rows_alloc) continue;
      const uint32_t slot = a_swz ? ((uint32_t)rows_alloc * a_swz + 1023) / 1024 * 1024 : (uint32_t)(paired ? 1 : Cin / 8) * rows_alloc * 16;
      const int nslots = (int)mn<uint32_t>(8, (kSmemLimitProg - b_total - 512) / slot);
      if (nslots < 3) break;
      const int nslabs = (p.Yg + Yt - 1) / Yt;
      const double eff = (double)p.Yg * p.Zg / ((double)nslabs * nzt * mt * 128);
      const double halo_cost = (double)(Yh * Zh) / (Yt * Zt);
      const double score = eff / (0.5 + 0.5 * halo_cost);
      if (score > best_score + 1e-9) {
        best_score = score; found = true;
        best = p;
        best.nzt = nzt; best.Zt = Zt; best.Zh = Zh; best.Yt = Yt; best.Yh = Yh; best.nslabs = nslabs; best.mtiles = mt;
        best.rows_alloc = rows_alloc; best.slot_bytes = slot; best.nslots = nslots;
      }
    }
  }
  if (!found) return false;
  ProgPlan &q = best;
  const int es = q.in_scale;
  q.a_swz = a_swz;
  if (q.stack) { q.acc_stride = q.N; q.mt_stride = 8 * q.N; }
  else { q.acc_stride = q.mtiles * q.N; q.mt_stride = q.N; }
  q.box_bytes = (a_swz ? (uint32_t)a_swz : 16u) * q.Zh * q.Yh;
  (void)es;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * nacc * q.mtiles * N)) cols <<= 1;
  q.tmem_cols = cols;
  q.smem_bytes = b_total + q.nslots * q.slot_bytes + 512;
  q.a_lbo_bytes = paired ? 16u : (uint32_t)q.rows_alloc * 16;
  if (!build_program(g, scatter, q)) return false;
  if (paired || q.stack) {
    if ((uint32_t)q.ntaps * q.btile_bytes > b_total) return false;
    q.nbt = q.ntaps;
  }
  return true;
}

// bytes of one output-channel part's repacked filter tiles in the workspace
static size_t prog_part_bytes(const ProgPlan &p) { return ((size_t)p.nbt * p.btile_bytes * (p.pair ? 2 : 1) + 255) / 256 * 256; }

bool prog_query(const cgan3d_conv_geom &g, int op, TcQuery &q) {
  if (op != 0 && op != 1) return false;
  ProgPlan p;
  int nsplit = 1;
  if (!plan_prog(g, op, p, &nsplit)) return false;
  q = {prog_part_bytes(p) * nsplit + 256, (op == 0 ? g.Cs : g.Cb) <= 64};
  return true;
}

int prog_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st,
             double *bn_sums) {
  const int scatter = op;
  ProgPlan p;
  int nsplit = 1;
  if (!plan_prog(g, scatter, p, &nsplit)) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 strided conv: no tiling for this shape");
  const size_t part_bytes = prog_part_bytes(p);
  if ((reinterpret_cast<uintptr_t>(in) & 15) || (reinterpret_cast<uintptr_t>(outp) & 15) || (reinterpret_cast<uintptr_t>(ws) & 15))
    return fail(CGAN3D_E_ARG, "tcgen05 strided conv: pointers must be 16-byte aligned");
  // input tensor: gather reads the big side with element strides 2 on z and y; scatter reads the small side densely
  const int Xi = scatter ? g.Xs : g.Xb, Yi = scatter ? g.Ys : g.Yb, Zi = scatter ? g.Zs : g.Zb, Ci = p.Cin;
  if ((reinterpret_cast<uintptr_t>(outp) & 15) || (p.Nout * 2) % 16 || (p.out_pitch * 2) % 16) return fail(CGAN3D_E_ARG, "tcgen05 strided conv: output rows must be 16-byte aligned");
  const int es = p.in_scale;
  CUtensorMap tm;
  // z-pair gather: the innermost dimension is a PAIR of z-adjacent voxels (dense along z, element stride 2 only on y)
  const int zp = p.zpair ? 2 : 1;
  int r = encode_act_map(&tm, in, Ci * zp, Zi / zp, Yi, Xi, g.B, p.a_swz ? Ci * zp : 8, p.Zh, p.Yh, p.zpair ? 1 : es, es, p.a_swz,
                         "strided conv");
  if (r) return r;
  const long long total = (long long)p.B * p.nzt * p.nslabs * p.Xg;
  const int grid = p.pair ? 2 * (int)mn<long long>((total + 1) / 2, (long long)(num_sms() / 2)) : (int)mn<long long>(total, (long long)num_sms());
  ProgLaunchArgs la{};
  la.tm = tm; la.g = g; la.scatter = scatter; la.nsplit = nsplit; la.grid = grid; la.wp = wp; la.outp = outp; la.ws = ws;
  la.part_bytes = part_bytes; la.bn_sums = bn_sums; la.st = st;
  switch (p.paired ? 1 : (p.Cin >> 4)) {
    case 1: return prog_launch_ks<1>(p, la);
    case 2: return prog_launch_ks<2>(p, la);
    case 4: return prog_launch_ks<4>(p, la);
    case 8: return prog_launch_ks<8>(p, la);
    default: return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 strided conv: Cin must be 16, 32, 64 or 128");
  }
}

}  // namespace cg
