/*
 * cgan3d.h — C ABI of the B200-native contrast-gan-3D hot path (libcgan3d.so).
 *
 * The reference (xqz-u/contrast-gan-3D) has no FFI: its hot path is stock ATen ops reached
 * through nn.Module.forward / autograd (SURVEY.md §8b).  Each entry point below replaces
 * the ATen call(s) made at the cited reference line(s); the Python host
 * (contrast_gan_3d_b200/) binds them with ctypes and wraps them in autograd.Functions
 * behind the reference's unchanged nn.Module / Trainer API.
 *
 * Conventions
 *  - All pointers are DEVICE pointers owned by the caller (PyTorch); the library never
 *    allocates persistent device memory.  Workspaces are passed in, sizes come from the
 *    *_workspace_bytes queries.
 *  - Every function only ENQUEUES work on `stream` (a cudaStream_t passed as void*); no
 *    hidden synchronisation, callable from any host thread (autograd engine threads).
 *  - Return value: 0 = ok; negative = argument/shape error detected before launch
 *    (CGAN3D_E_*); positive = cudaError_t passthrough.  cgan3d_last_error() returns a
 *    thread-local message.  There is no CPU fallback: an unsupported shape is an error.
 *  - Activation layout: channels-last [B][X][Y][Z][C] (X,Y,Z = the reference's W,H,D; C
 *    innermost).  For C == 1 this is bit-identical to the reference's [B,1,W,H,D].
 *  - dtype codes: CGAN3D_F32 = 0, CGAN3D_BF16 = 1 (storage type; accumulation is fp32).
 *  - Conv weights cross the ABI in the torch layout of the *base convolution*
 *    W[Cs][Cb][k][k][k] fp32, where Cb = channels of the big (un-strided) side and Cs =
 *    channels of the small (strided) side.  nn.Conv3d: Cs=Cout, Cb=Cin.
 *    nn.ConvTranspose3d: weight [Cin,Cout,k,k,k] is already [Cs][Cb] with Cs=Cin.
 */
#ifndef CGAN3D_H
#define CGAN3D_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGAN3D_VERSION 100

#define CGAN3D_F32 0
#define CGAN3D_BF16 1

#define CGAN3D_ACT_NONE 0
#define CGAN3D_ACT_RELU 1
#define CGAN3D_ACT_LRELU 2
#define CGAN3D_ACT_TANH 3

#define CGAN3D_E_ARG (-1)         /* null pointer / negative size */
#define CGAN3D_E_SHAPE (-2)       /* geometry inconsistent or unsupported */
#define CGAN3D_E_DTYPE (-3)       /* unknown dtype code */
#define CGAN3D_E_WORKSPACE (-4)   /* workspace too small */
#define CGAN3D_E_UNSUPPORTED (-5) /* kernel variant not built for this shape */

/* Geometry of the base convolution  small[o] = sum_k big[o*stride - pad + k] * W[k].
 * big side: [B][Xb][Yb][Zb][Cb]; small side: [B][Xs][Ys][Zs][Cs].                       */
typedef struct cgan3d_conv_geom {
  int32_t B;
  int32_t Xb, Yb, Zb, Cb;
  int32_t Xs, Ys, Zs, Cs;
  int32_t k, stride, pad;
} cgan3d_conv_geom;

int cgan3d_version(void);
const char *cgan3d_last_error(void);
/* Bit i set = capability i present: 0 generic CUDA-core kernels, 1 tcgen05 implicit GEMM. */
uint32_t cgan3d_capabilities(void);
/* 1 if the device behind the current context can run the tcgen05 kernels (sm_100). */
int cgan3d_device_supports_tc(void);

/* ---- weights ---------------------------------------------------------------------- */
/* W fp32 [Cs][Cb][k^3]  ->  packed `dtype` [k^3][Cb][Cs] used by all conv kernels.
 * Replaces nothing in the reference (layout plumbing).                                  */
int cgan3d_pack_weights(const float *w, void *packed, int dtype, int Cs, int Cb, int k, void *stream);

/* ---- convolutions (replace aten::convolution / convolution_backward) ----------------
 * gather:  small = conv(big)          nn.Conv3d fprop   (reference model/blocks.py:29-38,52;
 *                                     generator.py:77-83; discriminator.py:69-80)
 *                                     nn.ConvTranspose3d dgrad
 * scatter: big = conv^T(small)        nn.Conv3d dgrad;  nn.ConvTranspose3d fprop
 *                                     (reference generator.py:63-74 via blocks.py:21-23)
 * wgrad:   dW = big (*) small         weight gradient of either module (fp32, torch layout;
 *                                     beta = 0 overwrite, 1 accumulate)
 * `bias` (fp32 [C_out_side]) may be NULL.  impl: 0 = auto (tcgen05 when supported, else
 * generic), 1 = force generic CUDA-core kernel, 2 = force tcgen05 (error if unsupported).   */
size_t cgan3d_conv_workspace_bytes(const cgan3d_conv_geom *g, int dtype, int op /*0 gather,1 scatter,2 wgrad*/);
int cgan3d_conv_gather(const cgan3d_conv_geom *g, int dtype, const void *big, const void *wpacked,
                       const float *bias, void *small, void *workspace, size_t workspace_bytes, int impl,
                       void *stream);
int cgan3d_conv_scatter(const cgan3d_conv_geom *g, int dtype, const void *small, const void *wpacked,
                        const float *bias, void *big, void *workspace, size_t workspace_bytes, int impl,
                        void *stream);
int cgan3d_conv_wgrad(const cgan3d_conv_geom *g, int dtype, const void *big, const void *small, float *dw,
                      float beta, void *workspace, size_t workspace_bytes, int impl, void *stream);
/* Convolution + BatchNorm batch statistics in one launch (tcgen05 path only): same result in `out` as conv_gather
 * (op 0, in = big side) / conv_scatter (op 1, in = small side) without bias, and sums[0..C) = sum, sums[C..2C) = sum of
 * squares over all output voxels of each output channel (fp64, taken from the fp32 accumulators before the storage
 * rounding).  Replaces aten::convolution + the statistics half of aten::native_batch_norm (reference
 * model/blocks.py:52-53).  cgan3d_conv_fuses_bnstats returns 1 when the layer supports it on this device; otherwise
 * call conv_gather / conv_scatter followed by cgan3d_bn_stats.                                                        */
int cgan3d_conv_fuses_bnstats(const cgan3d_conv_geom *g, int dtype, int op);
int cgan3d_conv_bnstats(const cgan3d_conv_geom *g, int dtype, int op, const void *in, const void *wpacked, void *out,
                        double *sums, void *workspace, size_t workspace_bytes, void *stream);
/* which implementation `impl=0` would choose: 1 generic, 2 tcgen05 */
int cgan3d_conv_select(const cgan3d_conv_geom *g, int dtype, int op);

/* ---- reflect padding (aten::reflection_pad3d fwd/bwd; reference generator.py:31-38 via
 *      Conv3d(padding_mode="reflect")) -------------------------------------------------- */
int cgan3d_reflect_pad(const void *in, void *out, int dtype, int B, int X, int Y, int Z, int C, int pad,
                       void *stream);
/* adjoint: in_grad[i] = sum of padded_grad over all padded positions that mirror onto i */
int cgan3d_reflect_pad_backward(const void *padded_grad, void *in_grad, int dtype, int B, int X, int Y, int Z,
                                int C, int pad, void *stream);

/* ---- batch norm + activation (aten::native_batch_norm fwd/bwd, relu_/leaky_relu_,
 *      residual add; reference model/blocks.py:45,50,52-53,87-88) ------------------------ */
/* per-channel sums over n_rows rows of C channels: sums[0..C) = sum x, sums[C..2C) = sum x^2 (fp64) */
int cgan3d_bn_stats(const void *y, int dtype, int64_t n_rows, int C, double *sums, void *stream);
/* mean/invstd (fp32 [C] each, written to mean_invstd[0..2C)) from sums; updates running stats with
 * momentum (unbiased var) when running_mean != NULL and increments *num_batches_tracked (int64 device
 * scalar, may be NULL).                                                                    */
int cgan3d_bn_finalize(const double *sums, int64_t n_rows, int C, float eps, float momentum, float *mean_invstd,
                       float *running_mean, float *running_var, int64_t *num_batches_tracked, void *stream);
/* z = act(gamma * (y - mean) * invstd + beta) [+ residual];  scale_shift path for eval mode:
 * pass mean_invstd computed from running stats (cgan3d_bn_eval_params).                    */
int cgan3d_bn_eval_params(const float *running_mean, const float *running_var, int C, float eps,
                          float *mean_invstd, void *stream);
int cgan3d_bn_apply(const void *y, void *z, int dtype, int64_t n_rows, int C, const float *mean_invstd,
                    const float *gamma, const float *beta, int act, float slope, const void *residual,
                    void *stream);
/* bn_apply fused with the consumer's reflection padding (nn.Conv3d(padding_mode="reflect"), reference
 * model/generator.py:77-83 after model/blocks.py:45-53): z_padded[B, X+2p, Y+2p, Z+2p, C] = reflect_pad(act(bn(y)), p).
 * C % 8 == 0; otherwise CGAN3D_E_UNSUPPORTED (the caller pads separately).                            */
int cgan3d_bn_apply_pad(const void *y, void *z_padded, int dtype, int B, int X, int Y, int Z, int C,
                        const float *mean_invstd, const float *gamma, const float *beta, int act, float slope,
                        int pad, void *stream);
/* bn_apply followed by the ResNet block's dropout (nn.Dropout(p) between block0 and block1, reference
 * model/blocks.py:68-88, in train mode): z = keep ? act(gamma * (y - mean) * invstd + beta) / (1 - p) : 0 in fp32, rounded
 * once; no residual.  keep_bits (ceil(n_rows * C / 8) bytes) receives bit e & 7 of byte e >> 3 = keep(e) for the
 * channels-last linear index e.  Keep law: keep(e) <=> u >= floor(p * 2^32), u = word e & 3 of Philox4x32-10 with key
 * (lo32 seed, hi32 seed) and counter (lo32(e >> 2), hi32(e >> 2), 0, 0); p in [0, 1] (as fp32), p = 1 writes zeros.  The
 * 64-bit seed is read from device memory (*seed_dev), so the call can be captured in a CUDA graph.                    */
int cgan3d_bn_apply_dropout(const void *y, void *z, uint8_t *keep_bits, int dtype, int64_t n_rows, int C,
                            const float *mean_invstd, const float *gamma, const float *beta, int act, float slope, float p,
                            const int64_t *seed_dev, void *stream);
/* backward of bn_apply (train mode): given dz, y -> dy, dgamma, dbeta.
 * Pass 1 (reduce): sums[0..C) = sum g, sums[C..2C) = sum g*xhat, g = dz * act'(.)          */
int cgan3d_bn_backward_reduce(const void *dz, const void *y, int dtype, int64_t n_rows, int C,
                              const float *mean_invstd, const float *gamma, const float *beta, int act,
                              float slope, double *sums, void *stream);
/* the same through bn_apply_dropout (the dropout backward of reference model/blocks.py:68-88 fused in):
 * g = dz * keep / (1 - p) * act'(.), keep read from the bitmask that bn_apply_dropout wrote                             */
int cgan3d_bn_backward_reduce_dropout(const void *dz, const void *y, const uint8_t *keep_bits, int dtype, int64_t n_rows,
                                      int C, const float *mean_invstd, const float *gamma, const float *beta, int act,
                                      float slope, float p, double *sums, void *stream);
/* Pass 2: dy = gamma*invstd*(g - sum_g/n - xhat*sum_gx/n); the same launch writes the parameter gradients dgamma = sum
 * g*xhat, dbeta = sum g (fp32 [C], may be NULL): grad_beta = 0 overwrites them, 1 accumulates into them (the caller's
 * gradient buffer: a layer applied twice per backward, reference trainer/Trainer.py:114-116).                          */
int cgan3d_bn_backward_apply(const void *dz, const void *y, void *dy, int dtype, int64_t n_rows, int C,
                             const float *mean_invstd, const float *gamma, const float *beta, int act,
                             float slope, const double *sums, float *dgamma, float *dbeta, float grad_beta,
                             void *stream);
/* pass 2 through bn_apply_dropout (reference model/blocks.py:68-88): g as in cgan3d_bn_backward_reduce_dropout */
int cgan3d_bn_backward_apply_dropout(const void *dz, const void *y, const uint8_t *keep_bits, void *dy, int dtype,
                                     int64_t n_rows, int C, const float *mean_invstd, const float *gamma,
                                     const float *beta, int act, float slope, float p, const double *sums, float *dgamma,
                                     float *dbeta, float grad_beta, void *stream);
/* bias + activation without norm (critic first layer, blocks.py:34 bias=True under Identity norm):
 * z = act(y + bias); backward: dy = dz * act'(y + bias), dbias = sum dy                     */
int cgan3d_bias_act(const void *y, void *z, int dtype, int64_t n_rows, int C, const float *bias, int act,
                    float slope, void *stream);
int cgan3d_bias_act_backward(const void *dz, const void *y, void *dy, int dtype, int64_t n_rows, int C,
                             const float *bias, int act, float slope, double *dbias_sums, void *stream);
/* column sums (fp64) of a [n_rows][C] tensor: conv bias gradient */
int cgan3d_col_sums(const void *x, int dtype, int64_t n_rows, int C, double *sums, void *stream);
int cgan3d_sums_to_f32(const double *sums, float *out, int n, float scale, float beta, void *stream);

/* ---- generator tail: attenuation = tanh(y + bias); opt_hat = x - attenuation
 *      (reference generator.py:85, trainer/Trainer.py:170-171) --------------------------- */
int cgan3d_tanh_residual(const void *y, const float *bias, const float *x, float *attenuation, float *opt_hat,
                         int dtype, int64_t n, void *stream);
/* dy = -d_opt_hat * (1 - att^2) [+ d_att * (1 - att^2)] */
int cgan3d_tanh_residual_backward(const float *d_opt_hat, const float *d_att, const float *attenuation,
                                  void *dy, int dtype, int64_t n, double *dbias_sum, void *stream);

/* ---- dtype / layout helpers ----------------------------------------------------------- */
int cgan3d_cast(const void *in, int in_dtype, void *out, int out_dtype, int64_t n, void *stream);
int cgan3d_axpy(const void *x, void *y, int dtype, int64_t n, void *stream); /* y += x */

/* ---- losses (reference model/loss.py) ------------------------------------------------- */
/* One pass over opt_hat (s), subopt (t), mask (uint8):  sums[0..7) fp64 =
 * {sum s, sum t, sum s^2, sum t^2, sum s*t, sum hinge^2*mask, sum mask}; hinge per loss.py:64-69. */
int cgan3d_gen_loss_sums(const float *s, const float *t, const uint8_t *mask, int64_t n, float hu_lo, float hu_hi,
                         double *sums, void *stream);
/* Finalize on device: out[0] = zncc loss (loss.py:37-41), out[1] = HU loss (loss.py:70-71),
 * coef[0..6) = coefficients for the backward pass.                                          */
int cgan3d_gen_loss_finalize(const double *sums, int64_t n, float w_sim, float w_hu, float *out, float *coef,
                             void *stream);
/* ds = upstream[0] * d(w_sim*zncc)/ds + upstream[1] * d(w_hu*hu)/ds (+ d_extra if not NULL); upstream is a device
 * float[2] or NULL (= {1,1}).  StableStd backward per loss.py:20-29. */
int cgan3d_gen_loss_backward(const float *s, const float *t, const uint8_t *mask, int64_t n, float hu_lo,
                             float hu_hi, const float *coef, const float *upstream, const float *d_extra,
                             float *ds, void *stream);
/* mean of a tensor (Wasserstein terms, loss.py:77-79): out[0] = scale * sum(x)/n (fp32) */
int cgan3d_mean(const void *x, int dtype, int64_t n, float scale, double *scratch, float *out, void *stream);
/* fill with constant (gradient of a mean) */
int cgan3d_fill(void *x, int dtype, int64_t n, const float *value_dev, float scale, void *stream);

/* ---- optimizer (torch.optim.Adam single-tensor math + the critic weight clip,
 *      reference trainer/Trainer.py:135-138,157) ------------------------------------------ */
int cgan3d_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr,
                     float beta1, float beta2, float eps, int step, float clip /* <=0: none */, void *stream);
/* Same update for `count` parameter tensors in one launch per 48 tensors (torch.optim.Adam's foreach path,
 * reference trainer/Trainer.py:134,158 via optimizer.step()).  The five tables are HOST arrays of `count` device
 * pointers / element counts; all tensors share lr, betas, eps, step and clip.                                  */
int cgan3d_adam_step_multi(int count, float *const *params, const float *const *grads, float *const *exp_avgs,
                           float *const *exp_avg_sqs, const int64_t *numels, float lr, float beta1, float beta2,
                           float eps, int step, float clip, void *stream);

/* Capturable form of the same update (CUDA graphs): lr and the step count are read from DEVICE memory, hyper[0] = lr,
 * hyper[1] = step (float, exact to 2^24), so a captured optimizer.step() stays valid across scheduler changes
 * (torch.optim.Adam(capturable=True) semantics; reference trainer/Trainer.py:134-140,157-159).  cgan3d_adam_tick adds 1
 * to hyper[1]; call it once per optimizer step before the update launches.                                        */
int cgan3d_adam_tick(float *hyper, void *stream);
int cgan3d_adam_step_multi_dev(int count, float *const *params, const float *const *grads, float *const *exp_avgs,
                               float *const *exp_avg_sqs, const int64_t *numels, const float *hyper, float beta1,
                               float beta2, float eps, float clip, void *stream);

/* torch.optim.RMSprop (defaults: alpha 0.99, eps 1e-8, no momentum, not centered; reference
 * experiments/rmsprop_conf.py:8-9) for `count` tensors per launch, with the optional critic weight clip.             */
int cgan3d_rmsprop_step_multi(int count, float *const *params, const float *const *grads, float *const *square_avgs,
                              const int64_t *numels, float lr, float alpha, float eps, float clip, void *stream);

/* ---- patch sampler (reference data/CCTADataLoader.py:76-95, data/Scaler.py:41-42) ----------
 * vol: int16 [X][Y][Z][2] (HU, centerline mask) on device.  Pads symmetrically with 0 up to the
 * patch size (below = d//2), crops at lower bounds lb (computed on the host by the index law),
 * writes data = (HU - shift)/factor fp32 and mask uint8 for one patch [PX][PY][PZ].             */
int cgan3d_crop_scale(const int16_t *vol, int X, int Y, int Z, int lbx, int lby, int lbz, int PX, int PY, int PZ,
                      float shift, float factor, float *data, uint8_t *mask, void *stream);
/* out[i] = (hu[i] - shift) / factor for a contiguous int16 tensor (batches uploaded as raw HU and scaled on the device;
 * FactorZeroCenterScaler.__call__, reference data/Scaler.py:41-42, bit-identical in fp32).  16-byte aligned pointers. */
int cgan3d_scale_i16(const int16_t *hu, float *out, int64_t n, float shift, float factor, void *stream);
/* tile extraction / stitching for whole-volume inference (eval/CCTAContrastCorrector.py:60-81) */
int cgan3d_tile_extract(const int16_t *vol, int X, int Y, int Z, int x0, int y0, int z0, int PX, int PY, int PZ,
                        float shift, float factor, float *tile, void *stream);
int cgan3d_tile_accumulate(const float *tile, float *acc, float *cnt, int X, int Y, int Z, int x0, int y0, int z0,
                           int PX, int PY, int PZ, void *stream);
int cgan3d_tile_finalize(const float *acc, const float *cnt, float *out, int64_t n, float shift, float factor,
                         void *stream);
/* out[B][X][Y][Z] = x - nearest_resize(att[B][Xa][Ya][Za] -> [X][Y][Z]): the corrector's `patch - nn.Upsample(size=
 * inference_patch_size)(G(patch))` branch, taken when the generator does not round-trip the patch size
 * (eval/CCTAContrastCorrector.py:42-52,79); aten::upsample_nearest3d index law (src = floor(dst * in/out)).        */
int cgan3d_sub_resized(const float *x, const float *att, float *out, int B, int X, int Y, int Z, int Xa, int Ya, int Za,
                       void *stream);

/* ---- spatial augmentation (batchgenerators SpatialTransform_2, reference experiments/basic_conf.py:88-106) ------
 * Three stages per batch: elastic offset fields for the samples that drew elastic deformation, cubic B-spline
 * coefficients for the samples that drew any transform, and one resampling launch for the whole batch.  Data order 3
 * with border mode constant or nearest, seg order 0 constant, 3-D only; anything else is CGAN3D_E_UNSUPPORTED.
 * Extents are 4..256 per axis.  Every parameter array is a device pointer.                                          */
#define CGAN3D_BORDER_CONSTANT 0
#define CGAN3D_BORDER_NEAREST 1
#define CGAN3D_SPATIAL_TRANSFORM 1 /* sample drew elastic, rotation or scaling: resample, else shifted copy */
#define CGAN3D_SPATIAL_ELASTIC 2   /* sample adds field[field_slot] to the mesh */

/* per-sample record of the resampling stage (72 bytes) */
typedef struct {
  int32_t flags;      /* CGAN3D_SPATIAL_* */
  int32_t coef_slot;  /* index of the sample's coefficient volume (TRANSFORM) */
  int32_t field_slot; /* index of the sample's offset field and sums (ELASTIC) */
  int32_t shift[3];   /* lower bounds of the zero-filled copy (no TRANSFORM): out[x] = in[x + shift] */
  float A[9];         /* row-major linear map: diag(scale) * rotation^T */
  float ctr[3];       /* centre of the patch in input voxels */
} cgan3d_spatial_params_t;

/* uniform [-1, 1) noise [n][3][PX][PY][PZ] fp32 of the elastic stage: Philox4x32-10 keyed by seeds[i], counter = the
 * element's linear index within its sample.  The elastic field generates exactly these values internally.          */
int cgan3d_elastic_noise(int n, int PX, int PY, int PZ, const uint64_t *seeds, float *noise, void *stream);
size_t cgan3d_elastic_workspace_bytes(int n, int PX, int PY, int PZ);
/* field[i][d] = g / (max|g| / (mags[i][d] + 1e-8)), g = circular convolution of the noise with taps[i] (per sample:
 * PX x-taps, PY y-taps, PZ z-taps, fp64, the real inverse FFT of fourier_gaussian's kernel) along z, y and x;
 * sums[i][d] = sum of field[i][d] (fp64).  Fixed-order reductions: the output depends on the seeds only.           */
int cgan3d_elastic_field(int n, int PX, int PY, int PZ, const uint64_t *seeds, const double *mags, const double *taps,
                         float *field, double *sums, void *ws, size_t ws_bytes, void *stream);
/* coefficient volumes of scipy.ndimage.spline_filter(order=3) of data[samples[j]] (fp32 [B][SX][SY][SZ]); for
 * CGAN3D_BORDER_NEAREST of the input edge-padded by 12 voxels, as map_coordinates does.                            */
size_t cgan3d_spline_workspace_bytes(int n, int SX, int SY, int SZ, int mode);
int cgan3d_spline_prefilter(const float *data, int SX, int SY, int SZ, int n, const int32_t *samples, int mode,
                            float *coef, size_t coef_bytes, void *stream);
/* out[b] (fp32 [B][PX][PY][PZ]) and out_seg[b] (uint8) from data / seg [B][SX][SY][SZ]: per sample either
 * map_coordinates at c = A (mesh + field) - A mean(field) + ctr (data order 3 in `mode`, cval outside; seg order 0,
 * seg_fill outside [0, S-1]) or the zero-filled copy at params[b].shift.                                           */
int cgan3d_spatial_resample(const float *data, const uint8_t *seg, int B, int SX, int SY, int SZ, int PX, int PY, int PZ,
                            const cgan3d_spatial_params_t *params, const float *field, const double *sums,
                            const float *coef, int mode, float cval, int seg_fill, float *out, uint8_t *out_seg,
                            void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CGAN3D_H */
