// Internal (non-ABI) entry points shared by the convolution translation units.
#pragma once
#include <cuda.h>
#include <type_traits>

#include "common.cuh"

namespace cg {

int pack_weights(const float *w, void *packed, int dtype, int Cs, int Cb, int k, cudaStream_t st);
int generic_gather(const cgan3d_conv_geom &g, int dtype, const void *big, const void *wp, const float *bias,
                   void *small, cudaStream_t st);
int generic_scatter(const cgan3d_conv_geom &g, int dtype, const void *small, const void *wp, const float *bias,
                    void *big, void *ws, size_t ws_bytes, cudaStream_t st);
size_t generic_workspace_bytes(const cgan3d_conv_geom &g, int dtype, int op);
int generic_wgrad(const cgan3d_conv_geom &g, int dtype, const void *big, const void *small, float *dw, float beta,
                  cudaStream_t st);
int reflect_pad(const void *in, void *out, int dtype, int B, int X, int Y, int Z, int C, int pad, cudaStream_t st);
int reflect_pad_backward(const void *gp, void *gi, int dtype, int B, int X, int Y, int Z, int C, int pad,
                         cudaStream_t st);

// cuTensorMapEncodeTiled, looked up once through the runtime's driver entry point (conv_tc.cu); nullptr when the driver
// does not export it.  Only encode_tiled calls it; the tcgen05 route (conv_api.cu) uses it to test availability.
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tc_encode_fn();

// Every tensor map of the library: no interleave, L2_128B promotion, zero fill out of bounds.  estr == nullptr: all element
// strides 1.  `what` names the map in the error message.
int encode_tiled(CUtensorMap *tm, CUtensorMapDataType dtype, int rank, const void *ptr, const cuuint64_t *gdim,
                 const cuuint64_t *gstr, const cuuint32_t *box, const cuuint32_t *estr, CUtensorMapSwizzle swizzle,
                 const char *what);
// Repacked CTA-pair weight tiles viewed as nrows INT32 rows of 256 bytes, loaded box_rows rows at a time.
int encode_weight_rows(CUtensorMap *tm, const void *ptr, int nrows, int box_rows);
// Channels-last bf16 activations [B][X][Y][Z][C]: a box of box_c channels x nz voxels x ny lines of one x-plane, the voxels
// taken every ez-th along z and every ey-th along y.  swizzle_bytes: 0 (none), 32, 64 or 128.
int encode_act_map(CUtensorMap *tm, const void *ptr, int C, int Z, int Y, int X, int B, int box_c, int nz, int ny, int ez,
                   int ey, int swizzle_bytes, const char *what);

// Dynamic shared memory every tcgen05 kernel is opted into: 227 KB, the most a block may have on sm_100.  Each planner
// budgets a margin below it (kMaxDynSmem - 1024, or - 2048 for the strided wgrad).
constexpr uint32_t kMaxDynSmem = 232448;

// Launch a tcgen05 kernel with `smem` bytes of dynamic shared memory, as clusters of `cluster` CTAs along x when cluster > 1.
// The opt-in to kMaxDynSmem runs once per kernel: a function-local static is initialised once, thread-safely, and the
// template is instantiated per kernel, so kernels with the same signature do not share it.
template <auto Kernel, typename... Args>
int tc_launch(const char *name, int grid, int block, size_t smem, int cluster, cudaStream_t st, const Args &...args) {
  static const cudaError_t opt_in = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem);
  if (opt_in != cudaSuccess) {
    char where[128];
    snprintf(where, sizeof(where), "cudaFuncSetAttribute(%s)", name);
    return cuda_fail(opt_in, where);
  }
  cudaLaunchAttribute attr{};
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = (unsigned)cluster;
  attr.val.clusterDim.y = 1;
  attr.val.clusterDim.z = 1;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  if (cluster > 1) {
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
  }
  const cudaError_t e = cudaLaunchKernelEx(&cfg, Kernel, args...);
  if (e != cudaSuccess) return cuda_fail(e, name);
  CG_LAUNCH_CHECK(name);
  return 0;
}

// ---------------------------------------------------------------- tcgen05 kernel families (bf16 only)
// Each family exports a query and a launcher.  tc_route (conv_api.cu) picks the family, and the entry points there check
// the rules the families share.  A query returns true when the family's planner accepts the shape and then fills TcQuery;
// op: 0 gather, 1 scatter, 2 wgrad (families that serve one op ignore it).  A launcher takes a shape its query accepted, a
// workspace of at least the reported size and, where the family fuses them, bn_sums (fp64 [2*Cout], zeroed by the
// caller): the epilogue adds the per-channel sum / sum of squares of the fp32 accumulators.  The launchers check the
// pointer alignment their kernels need.
struct TcQuery {
  size_t workspace_bytes;  // what cgan3d_conv_workspace_bytes reports for the family; 0: none used
  bool fuses_bnstats;      // the launcher takes bn_sums
};

// conv_thin_tc.cu (7x7x7 thin-channel layers).  A: 1 -> 16 channels (gather of Cb == 1, scatter of Cs == 1);
// B: 16 -> 1 channels (the other two); C: round-1 weight gradient of both, for the shapes wgrad7_v2.cu does not plan
bool thin_a_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int thin_a_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st,
               double *bn_sums);
bool thin_b_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int thin_b_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st);
bool thin_c_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int thin_c_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, void *ws, cudaStream_t st);

// wgrad7_v2.cu: weight gradient of the thin layers, the z-expansion built in shared memory (no workspace)
bool thin_w2_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int thin_w2_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st);

// conv_d1_tc.cu (first critic layer: 1 -> 8 channels, k4 s2)
bool d1_gather_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int d1_gather_run(const cgan3d_conv_geom &g, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st);
bool d1_scatter_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int d1_scatter_run(const cgan3d_conv_geom &g, const void *small, const void *wp, void *outp, void *ws, cudaStream_t st);
bool d1_wgrad_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int d1_wgrad_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, void *ws, cudaStream_t st);

// conv_tc.cu (3x3x3 stride-1 convolutions, Cin in {16, 32, 64, 128})
bool s1_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int s1_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st,
           double *bn_sums);

// conv_tc_prog.cu (strided convolutions)
bool prog_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int prog_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, cudaStream_t st,
             double *bn_sums);

// wgrad_s2_tc.cu (stride-2 layers with Cs in {32, 64}, Cb in {16, 32}, and the stride-1 ResNet layers with Cs == 64)
bool wgrad_s2_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int wgrad_s2_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st);

// wgrad_tc.cu (the weight-gradient shapes wgrad_s2_tc.cu does not plan)
bool wgrad_prog_query(const cgan3d_conv_geom &g, int op, TcQuery &q);
int wgrad_prog_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st);

}  // namespace cg
