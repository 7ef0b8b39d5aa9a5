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
// does not export it.  Every tensor map of the library uses CU_TENSOR_MAP_L2_PROMOTION_L2_128B.
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tc_encode_fn();

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
