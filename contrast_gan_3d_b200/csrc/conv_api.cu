// C-ABI entry points for the convolutions: argument validation + implementation choice.
#include "common.cuh"
#include "conv_internal.cuh"

namespace cg {

static int check_geom(const cgan3d_conv_geom *g, int dtype) {
  CG_CHECK_ARG(g != nullptr, "conv: geometry is NULL");
  CG_CHECK_DTYPE(dtype, "conv");
  CG_CHECK_SHAPE(g->B >= 0 && g->Xb > 0 && g->Yb > 0 && g->Zb > 0 && g->Cb > 0 && g->Cs > 0, "conv: bad sizes");
  CG_CHECK_SHAPE(g->k >= 1 && g->k <= 7 && (g->stride == 1 || g->stride == 2) && g->pad >= 0 && g->pad < g->k,
                 "conv: k=%d stride=%d pad=%d unsupported", g->k, g->stride, g->pad);
  // small side must be a legal output extent of the base conv; for stride 2 two big extents map to the same
  // small extent (that is what ConvTranspose3d's output_padding selects), so check the range, not equality.
  const int dims_b[3] = {g->Xb, g->Yb, g->Zb}, dims_s[3] = {g->Xs, g->Ys, g->Zs};
  for (int i = 0; i < 3; ++i) {
    const int num = dims_b[i] + 2 * g->pad - g->k;
    CG_CHECK_SHAPE(num >= 0, "conv: kernel larger than padded input on axis %d", i);
    CG_CHECK_SHAPE(dims_s[i] == num / g->stride + 1, "conv: small extent %d != floor((%d+2*%d-%d)/%d)+1 on axis %d",
                   dims_s[i], dims_b[i], g->pad, g->k, g->stride, i);
  }
  return 0;
}

enum class TcFamily { None, ThinA, ThinB, D1Gather, D1Scatter, S1, Prog, ThinW2, ThinC, D1Wgrad, WgradS2, WgradProg };

struct TcRoute {
  TcFamily family = TcFamily::None;
  TcQuery q{};
};

// The tcgen05 kernel family that runs (g, dtype, op), with what its planner reports: the first family in the op's list
// whose planner accepts the shape, or None (the generic CUDA-core kernels then run; every family is bf16 only).  The
// families' shape domains overlap in two places, and there the order decides: the v2 thin weight gradient before the
// round-1 one (even padding and extents), wgrad_s2 before wgrad_prog.
static TcRoute tc_route(const cgan3d_conv_geom &g, int dtype, int op) {
  using F = TcFamily;
  struct Entry {
    F family;
    bool (*query)(const cgan3d_conv_geom &, int, TcQuery &);
  };
  static const Entry kOrder[3][5] = {
      {{F::ThinA, thin_a_query}, {F::ThinB, thin_b_query}, {F::D1Gather, d1_gather_query}, {F::S1, s1_query}, {F::Prog, prog_query}},
      {{F::ThinA, thin_a_query}, {F::ThinB, thin_b_query}, {F::D1Scatter, d1_scatter_query}, {F::S1, s1_query}, {F::Prog, prog_query}},
      {{F::ThinW2, thin_w2_query}, {F::ThinC, thin_c_query}, {F::D1Wgrad, d1_wgrad_query}, {F::WgradS2, wgrad_s2_query},
       {F::WgradProg, wgrad_prog_query}}};
  TcRoute r;
  if (!cgan3d_device_supports_tc() || tc_encode_fn() == nullptr || dtype != CGAN3D_BF16 || op < 0 || op > 2) return r;
  for (const Entry &e : kOrder[op])
    if (e.query(g, op, r.q)) {
      r.family = e.family;
      break;
    }
  return r;
}

static int pick(const TcRoute &r, int impl, bool *use_tc) {
  const bool can = r.family != TcFamily::None;
  if (impl == 2 && !can) return fail(CGAN3D_E_UNSUPPORTED, "conv: tcgen05 path does not support this shape/op");
  *use_tc = (impl == 2) || (impl == 0 && can);
  return 0;
}

static int check_workspace(const TcRoute &r, const void *ws, size_t ws_bytes) {
  const size_t need = r.q.workspace_bytes;
  if (need && (ws == nullptr || ws_bytes < need))
    return fail(CGAN3D_E_WORKSPACE, "tcgen05 conv: workspace %zu < %zu", ws_bytes, need);
  return 0;
}

// gather (op 0: in = big side, out = small side) or scatter (op 1: the other way round) on the routed family
static int tc_conv(const TcRoute &r, const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *out, void *ws,
                   size_t ws_bytes, cudaStream_t st, double *bn_sums) {
  if (int e = check_workspace(r, ws, ws_bytes)) return e;
  switch (r.family) {
    case TcFamily::ThinA: return thin_a_run(g, op, in, wp, out, ws, st, bn_sums);
    case TcFamily::ThinB: return thin_b_run(g, op, in, wp, out, ws, st);
    case TcFamily::D1Gather: return d1_gather_run(g, in, wp, out, ws, st);
    case TcFamily::D1Scatter: return d1_scatter_run(g, in, wp, out, ws, st);
    case TcFamily::S1: return s1_run(g, op, in, wp, out, ws, st, bn_sums);
    case TcFamily::Prog: return prog_run(g, op, in, wp, out, ws, st, bn_sums);
    default: return fail(CGAN3D_E_UNSUPPORTED, "conv: tcgen05 path does not support this shape/op");
  }
}

static int run_conv(const cgan3d_conv_geom &g, int dtype, int op, const void *in, const void *wp, const float *bias, void *out,
                    void *ws, size_t ws_bytes, int impl, cudaStream_t st) {
  const TcRoute r = tc_route(g, dtype, op);
  bool tc = false;
  if (int e = pick(r, impl, &tc)) return e;
  if (!tc) return op == 0 ? generic_gather(g, dtype, in, wp, bias, out, st) : generic_scatter(g, dtype, in, wp, bias, out, ws, ws_bytes, st);
  if (bias) return fail(CGAN3D_E_UNSUPPORTED, "tcgen05 conv: bias is applied by the bias_act pass");
  return tc_conv(r, g, op, in, wp, out, ws, ws_bytes, st, nullptr);
}

}  // namespace cg

using namespace cg;

extern "C" {

int cgan3d_pack_weights(const float *w, void *packed, int dtype, int Cs, int Cb, int k, void *stream) {
  CG_CHECK_ARG(w && packed, "pack_weights: NULL pointer");
  CG_CHECK_DTYPE(dtype, "pack_weights");
  CG_CHECK_SHAPE(Cs > 0 && Cb > 0 && k > 0 && k <= 7, "pack_weights: bad sizes");
  return pack_weights(w, packed, dtype, Cs, Cb, k, as_stream(stream));
}

size_t cgan3d_conv_workspace_bytes(const cgan3d_conv_geom *g, int dtype, int op) {
  if (!g || check_geom(g, dtype) != 0) return 0;
  const size_t a = tc_route(*g, dtype, op).q.workspace_bytes, b = generic_workspace_bytes(*g, dtype, op);
  return a > b ? a : b;
}

int cgan3d_conv_select(const cgan3d_conv_geom *g, int dtype, int op) {
  int r = check_geom(g, dtype);
  if (r) return r;
  return tc_route(*g, dtype, op).family != TcFamily::None ? 2 : 1;
}

int cgan3d_conv_gather(const cgan3d_conv_geom *g, int dtype, const void *big, const void *wpacked, const float *bias,
                       void *small, void *workspace, size_t workspace_bytes, int impl, void *stream) {
  int r = check_geom(g, dtype);
  if (r) return r;
  CG_CHECK_ARG(big && wpacked && small, "conv_gather: NULL pointer");
  if (g->B == 0) return 0;
  return run_conv(*g, dtype, 0, big, wpacked, bias, small, workspace, workspace_bytes, impl, as_stream(stream));
}

int cgan3d_conv_fuses_bnstats(const cgan3d_conv_geom *g, int dtype, int op) {
  if (!g || check_geom(g, dtype) != 0) return 0;
  return tc_route(*g, dtype, op).q.fuses_bnstats ? 1 : 0;
}

int cgan3d_conv_bnstats(const cgan3d_conv_geom *g, int dtype, int op, const void *in, const void *wpacked, void *out,
                        double *sums, void *workspace, size_t workspace_bytes, void *stream) {
  int r = check_geom(g, dtype);
  if (r) return r;
  CG_CHECK_ARG(in && wpacked && out && sums, "conv_bnstats: NULL pointer");
  CG_CHECK_ARG(op == 0 || op == 1, "conv_bnstats: op must be 0 (gather) or 1 (scatter)");
  const TcRoute rt = tc_route(*g, dtype, op);
  if (!rt.q.fuses_bnstats) return fail(CGAN3D_E_UNSUPPORTED, "conv_bnstats: this layer / device cannot fuse the statistics");
  const int C = op == 0 ? g->Cs : g->Cb;
  cudaError_t e = cudaMemsetAsync(sums, 0, (size_t)2 * C * sizeof(double), as_stream(stream));
  if (e != cudaSuccess) return cuda_fail(e, "conv_bnstats memset");
  if (g->B == 0) return 0;
  return tc_conv(rt, *g, op, in, wpacked, out, workspace, workspace_bytes, as_stream(stream), sums);
}

int cgan3d_conv_scatter(const cgan3d_conv_geom *g, int dtype, const void *small, const void *wpacked,
                        const float *bias, void *big, void *workspace, size_t workspace_bytes, int impl,
                        void *stream) {
  int r = check_geom(g, dtype);
  if (r) return r;
  CG_CHECK_ARG(big && wpacked && small, "conv_scatter: NULL pointer");
  if (g->B == 0) return 0;
  return run_conv(*g, dtype, 1, small, wpacked, bias, big, workspace, workspace_bytes, impl, as_stream(stream));
}

int cgan3d_conv_wgrad(const cgan3d_conv_geom *g, int dtype, const void *big, const void *small, float *dw, float beta,
                      void *workspace, size_t workspace_bytes, int impl, void *stream) {
  int r = check_geom(g, dtype);
  if (r) return r;
  CG_CHECK_ARG(big && small && dw, "conv_wgrad: NULL pointer");
  CG_CHECK_ARG(beta == 0.f || beta == 1.f, "conv_wgrad: beta must be 0 or 1");
  const TcRoute rt = tc_route(*g, dtype, 2);
  bool tc = false;
  if ((r = pick(rt, impl, &tc))) return r;
  if (!tc) return generic_wgrad(*g, dtype, big, small, dw, beta, as_stream(stream));
  if ((r = check_workspace(rt, workspace, workspace_bytes))) return r;
  const cudaStream_t st = as_stream(stream);
  switch (rt.family) {
    case TcFamily::ThinW2: return thin_w2_run(*g, big, small, dw, beta, st);
    case TcFamily::ThinC: return thin_c_run(*g, big, small, dw, beta, workspace, st);
    case TcFamily::D1Wgrad: return d1_wgrad_run(*g, big, small, dw, beta, workspace, st);
    case TcFamily::WgradS2: return wgrad_s2_run(*g, big, small, dw, beta, st);
    case TcFamily::WgradProg: return wgrad_prog_run(*g, big, small, dw, beta, st);
    default: return fail(CGAN3D_E_UNSUPPORTED, "conv: tcgen05 path does not support this shape/op");
  }
}

int cgan3d_reflect_pad(const void *in, void *out, int dtype, int B, int X, int Y, int Z, int C, int pad,
                       void *stream) {
  CG_CHECK_ARG(in && out, "reflect_pad: NULL pointer");
  CG_CHECK_DTYPE(dtype, "reflect_pad");
  CG_CHECK_SHAPE(pad >= 0 && pad < X && pad < Y && pad < Z && C > 0 && B >= 0,
                 "reflect_pad: pad %d must be smaller than every extent (%d,%d,%d)", pad, X, Y, Z);
  if (B == 0) return 0;
  return reflect_pad(in, out, dtype, B, X, Y, Z, C, pad, as_stream(stream));
}

int cgan3d_reflect_pad_backward(const void *padded_grad, void *in_grad, int dtype, int B, int X, int Y, int Z, int C,
                                int pad, void *stream) {
  CG_CHECK_ARG(padded_grad && in_grad, "reflect_pad_backward: NULL pointer");
  CG_CHECK_DTYPE(dtype, "reflect_pad_backward");
  CG_CHECK_SHAPE(pad >= 0 && pad < X && pad < Y && pad < Z && C > 0 && B >= 0, "reflect_pad_backward: bad pad");
  if (B == 0) return 0;
  return reflect_pad_backward(padded_grad, in_grad, dtype, B, X, Y, Z, C, pad, as_stream(stream));
}

}  // extern "C"
