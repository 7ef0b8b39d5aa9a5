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

// tcgen05 implicit-GEMM path (conv_tc.cu). op: 0 gather, 1 scatter, 2 wgrad.
bool tc_supported(const cgan3d_conv_geom &g, int dtype, int op);
size_t tc_workspace_bytes(const cgan3d_conv_geom &g, int dtype, int op);
// bn_sums (optional, fp64 [2*Cout], zeroed by the caller): the epilogue adds the per-channel sum / sum of squares of the
// fp32 accumulators (BatchNorm batch statistics fused into the convolution); see tc_fuses_bnstats.
int tc_gather(const cgan3d_conv_geom &g, const void *big, const void *wp, const float *bias, void *small,
              void *ws, size_t ws_bytes, cudaStream_t st, double *bn_sums = nullptr);
int tc_scatter(const cgan3d_conv_geom &g, const void *small, const void *wp, const float *bias, void *big,
               void *ws, size_t ws_bytes, cudaStream_t st, double *bn_sums = nullptr);
bool tc_fuses_bnstats(const cgan3d_conv_geom &g, int dtype, int op);
int tc_wgrad(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, void *ws,
             size_t ws_bytes, cudaStream_t st);

// cuTensorMapEncodeTiled, looked up once through the runtime's driver entry point (conv_tc.cu); nullptr when the driver
// does not export it.  Only encode_tiled calls it; tc_supported uses it to test availability.
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

// conv_tc_prog.cu (strided convolutions)
bool tc_prog_supported(const cgan3d_conv_geom &g, int dtype, int op);
size_t tc_prog_workspace_bytes(const cgan3d_conv_geom &g, int dtype, int op);
int tc_prog_run(const cgan3d_conv_geom &g, int scatter, const void *in, const void *wp, void *outp, void *ws, size_t ws_bytes,
                cudaStream_t st, double *bn_sums = nullptr);
bool tc_prog_fuses_bnstats(const cgan3d_conv_geom &g, int scatter);

// conv_thin_tc.cu (7x7x7 thin-channel layers)
bool thin_supported(const cgan3d_conv_geom &g, int dtype, int op);
size_t thin_workspace_bytes(const cgan3d_conv_geom &g, int dtype, int op);
int thin_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, size_t ws_bytes,
             cudaStream_t st, double *bn_sums = nullptr);
bool thin_fuses_bnstats(const cgan3d_conv_geom &g, int op);
int thin_wgrad_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, void *ws, size_t ws_bytes,
                   cudaStream_t st);

// wgrad7_v2.cu: weight gradient of the thin layers, the z-expansion built in shared memory (no workspace)
bool thin_w2_supported(const cgan3d_conv_geom &g);
int thin_w2_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st);

// conv_d1_tc.cu (first critic layer: 1 -> 8 channels, k4 s2)
bool d1_supported(const cgan3d_conv_geom &g, int dtype, int op);
size_t d1_workspace_bytes(const cgan3d_conv_geom &g, int dtype, int op);
int d1_run(const cgan3d_conv_geom &g, int op, const void *in, const void *wp, void *outp, void *ws, size_t ws_bytes, cudaStream_t st);
int d1_wgrad_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, void *ws, size_t ws_bytes,
                 cudaStream_t st);

// wgrad_s2_tc.cu (stride-2 layers with Cs in {32, 64}, Cb in {16, 32}, and the stride-1 ResNet layers with Cs == 64)
bool tc_wgrad_s2_supported(const cgan3d_conv_geom &g);
int tc_wgrad_s2_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st);

// wgrad_tc.cu (the weight-gradient shapes wgrad_s2_tc.cu does not plan)
bool tc_wgrad_supported(const cgan3d_conv_geom &g);
int tc_wgrad_run(const cgan3d_conv_geom &g, const void *big, const void *small, float *dw, float beta, cudaStream_t st);

}  // namespace cg
