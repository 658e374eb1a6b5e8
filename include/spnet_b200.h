/* spnet_b200.h — C ABI of libspnet_b200.so, the sm_100a kernel library behind the
 * B200-native SPNet hot path (Xception-SPNet forward/backward + YOLO-ellipse loss).
 *
 * The reference (drscotthawley/SPNet) is pure Python on Keras 2.1.3 / TF 1.14 and has no
 * FFI of its own; this is the boundary its maintainer would bind with ctypes (see
 * INTEGRATION.md). Each entry point names the reference code it replaces.
 *
 * Conventions (SURVEY.md §8b):
 *   - the caller owns all memory: device pointers + explicit shapes; the library never
 *     allocates, frees or synchronises;
 *   - every call is asynchronous on `stream`, safe to capture in a CUDA graph;
 *   - returns 0, or a negative code (SPNET_ERR_*) with a per-thread message available from
 *     spnet_last_error(); never throws;
 *   - `stats` / `colstats` arguments are ORDER-INDEPENDENT ACCUMULATORS: int64 buffers of 2 words per entry
 *     (fixed-point limbs, quantum 2^-56; csrc/common.cuh stat_add / stat_get), 2*C entries (sum | second sum),
 *     zero-initialised once by the caller and reset by the finalize call that consumes them. Integer atomics
 *     make the cross-CTA sums bit-identical from run to run, whatever order the CTAs arrive in;
 *   - activations are NHWC; `dtype` is 0 (fp32) or 1 (bf16) for activation tensors;
 *     parameters, BatchNorm statistics, losses and weight gradients are fp32;
 *   - sm_100a only (spnet_check_device() reports anything else); no CPU fallback.
 *
 * This header is parsed by spnet_b200/_lib.py to build the ctypes signatures: keep one
 * prototype per statement, parameters as `type name`.
 */
#ifndef SPNET_B200_H
#define SPNET_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define SPNET_ERR_ARG (-1)
#define SPNET_ERR_CUDA (-2)
#define SPNET_ERR_ARCH (-3)

/* ---- library ---- */
int spnet_version(void);
const char* spnet_last_error(void);
int spnet_check_device(void);

/* ---- loss / output head ----
 * custom_loss (spnet/models.py:564-589) and my_loss (:594-633) in one launch.
 * out6 = [total, center, size, angle, noobj, class]; grad (nullable) = dL/dy_pred.
 * hybrid: cf.loss_type != 'same' (BCE-with-logits on noobj). sel_sigmoid: y_pred's noobj
 * columns are pre-activations of a SelectiveSigmoid layer (:277-298). */
int spnet_yolo_ellipse_loss(const float* y_true, const float* y_pred, int batch, int ncols, int hybrid, int sel_sigmoid, float* out6, float* grad, cudaStream_t stream);
/* SelectiveSigmoid.call (spnet/models.py:293-295); selective_activation.py:6-9 */
int spnet_selective_sigmoid_fwd(const float* x, float* y, int rows, int ncols, int start, int end, int skip, cudaStream_t stream);
int spnet_selective_sigmoid_bwd(const float* y, const float* dy, float* dx, int rows, int ncols, int start, int end, int skip, cudaStream_t stream);
/* denorm_Y (spnet/utils.py:186-188) + integer part of cleanup_antinode_vars (:56-64) +
 * existence test (:109-118). denorm [n,ncols] f32, ints [n,ncols/8,5] i32 (cx,cy,a,b,noobj),
 * exists [n,ncols/8] u8. */
int spnet_decode_detections(const float* y, const float* means, const float* ranges, int n, int ncols, float* denorm, int* ints, unsigned char* exists, cudaStream_t stream);

/* Grid-cell / slot assignment on the device: true_to_pred_grid (spnet/utils.py:191-244) + norm_Y (:179-184) for n
 * images in one launch, bit-exact (float64 divide, truncation toward zero, clamp, first-come slot order). ann
 * [n,max_obj,8] float64 rows as parse_meta_file (:260-286) returns them, counts [n] i32; defaults / means / ranges
 * [nx*ny*ppc*8] fp32 from setup_means_and_ranges (:144-176); Y [n,nx*ny*ppc*8] fp32; err [n] i32 = 0 or 1 + index
 * of the antinode that tripped the reference's `assert slot < preds_per_cell` (:240).
 * spnet_yolo_ellipse_loss_ann: the same assignment fused in front of custom_loss - one launch from raw annotations
 * to loss value, 5-term breakdown and dL/dy_pred; y_true_out nullable. */
int spnet_assign_grid(const double* ann, const int* counts, int n, int max_obj, int nx, int ny, int ppc, const float* defaults, const float* means, const float* ranges, float* Y, int* err, cudaStream_t stream);
int spnet_yolo_ellipse_loss_ann(const double* ann, const int* counts, int max_obj, int nx, int ny, int ppc, const float* defaults, const float* means, const float* ranges, const float* y_pred, int batch, int hybrid, int sel_sigmoid, float* y_true_out, float* out6, float* grad, int* err, cudaStream_t stream);
/* load_X_one_proc's (v/255 - 0.5)*2 (spnet/utils.py:340-342) on the device: uint8 frames cross PCIe, lut [256] fp32
 * holds the 256 possible results as numpy computes them (bit-exact by construction). */
int spnet_normalize_u8(const unsigned char* in, const float* lut, float* out, long long n, cudaStream_t stream);

/* ---- Evaluation metrics (spnet/diagnostics.py: calc_errors :13-60; compute_iou :85-120 for every (image, slot)
 *      pair, analytic ellipse raster with an anti-aliasing margin instead of cv2). yp / yt: denormalised fp32
 *      [n, ncols]; counters int32 [7] (caller zeroes), pix_err fp32 [n]; iou fp32 [n, ncols/8] (-1 = skipped pair),
 *      counts nullable int32 [n, ncols/8, 2]. ---- */
int spnet_calc_errors(const float* yp, const float* yt, int n, int ncols, int* counters, float* pix_err, cudaStream_t stream);
int spnet_ellipse_iou(const float* yp, const float* yt, int n, int ncols, int nx, int ny, float margin, float* iou, int* counts, cudaStream_t stream);

/* ---- AugmentOnTheFly on the device (spnet/callbacks.py:272-341; cutout_inplace / salt_n_pepa_inplace of
 *      spnet/augmentation.py:117-135,159-180): x = augmented copy of the pristine frames x_orig, fp32 [n,H,W,C],
 *      one launch per epoch, counter-based random draws keyed by (seed, frame). ---- */
int spnet_augment_on_the_fly(const float* x_orig, float* x, int n, int H, int W, int C, long long seed, int max_regions, int minsize, int maxsize, float sp_prob, float sp_amount, float salt_vs_pepper, cudaStream_t stream);

/* ---- SeparableConv2D depthwise half (keras.applications.Xception; spnet/models.py:359) ---- */
int spnet_dwconv3x3_fwd(const void* in, const float* k, const float* in_a, const float* in_b, int relu, void* out, int dtype, int B, int H, int W, int C, cudaStream_t stream);
int spnet_dwconv3x3_bwd_fused(const void* gout, const void* in, const float* k, const float* in_a, const float* in_b, int relu, const float* bn_mean, const float* bn_rstd, long long* stats, const void* add_src, const void* add_strided, void* gin, float* dk, long long* dk_acc, int dtype, int B, int H, int W, int C, cudaStream_t stream);

/* ---- GEMMs: pointwise 1x1, strided 1x1 residual convs, block1_conv2 (im2col), Dense head
 *      (spnet/models.py:359,388). See gemm_tc.cu / gemm_simt.cu for operand conventions. out_mode 3 (slabs): split s
 *      of the K range stores its [M, N] partial product at D + s * slab_stride elements - split-K with a fixed
 *      summation order (spnet_slab_reduce), or a batch of GEMMs stacked along K in ONE launch (the weight gradients
 *      of Xception's 24 identical middle-flow layers, written straight into the flat gradient buffer). ---- */
int spnet_gemm_bf16(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, void* D, long long ldd, long long slab_stride, int out_mode, int M, int N, int K, int splits, long long* colstats, cudaStream_t stream);
int spnet_gemm_simt(const void* A, long long sa_r, long long sa_k, const void* B, long long sb_r, long long sb_k, void* D, long long ldd, long long slab_stride, int dtype, int out_mode, int M, int N, int K, int splits, long long* colstats, cudaStream_t stream);

/* ---- Conv2D k x k, stride 1, as implicit GEMM on tcgen05 (gemm_tc.cu, no im2col buffer): Xception
 *      block1_conv2 (keras.applications.Xception; spnet/models.py:359) and the InceptionResNetV2 branch
 *      convolutions (spnet/models.py:18,357-359). NHWC bf16 activations with pixel stride ld (a channel slice
 *      of a wider buffer is fine), Keras kernel [KH,KW,Cin,Cout] bf16; pt / pl = top / left zero padding.
 *      fwd: optional fused BatchNorm column statistics; wgrad: fp32 reduce-add into dW. ---- */
int spnet_conv_tc_fwd(const void* X, long long ldx, int NB, int H, int W, int Cin, const void* Wt, void* Y, long long ldy, int OH, int OW, int Cout, int KH, int KW, int pt, int pl, long long* colstats, cudaStream_t stream);
int spnet_conv_tc_dgrad(const void* dY, long long ldy, int NB, int OH, int OW, int Cout, const void* Wt, void* dX, long long ldx, int H, int W, int Cin, int KH, int KW, int pt, int pl, cudaStream_t stream);
int spnet_conv_tc_wgrad(const void* X, long long ldx, int NB, int H, int W, int Cin, const void* dY, long long ldy, int OH, int OW, int Cout, float* dW, int KH, int KW, int pt, int pl, cudaStream_t stream);
/* 'valid' stride-1 convolution of a DENSE NHWC bf16 tensor (pixel stride = Cin) with the KW taps of a filter row folded
 * into the channel axis (they are KW*Cin contiguous elements): KH * ceil(KW*Cin/64) k-blocks per tile and no im2col buffer.
 * Replaces the im2col + GEMM route of Xception's block1_conv2 (3x3, 32 -> 64; keras.applications.xception, called from
 * spnet/models.py:359). Y [NB, H-KH+1, W-KW+1, Cout] bf16 (pixel stride ldy), Wt the Keras kernel [KH, KW, Cin, Cout];
 * colstats as for spnet_conv_tc_fwd. The weight gradient is reduce-added into dW (fp32, caller zeroes it). */
int spnet_conv_tc_fwd_kwfold(const void* X, int NB, int H, int W, int Cin, const void* Wt, void* Y, long long ldy, int Cout, int KH, int KW, long long* colstats, cudaStream_t stream);
int spnet_conv_tc_wgrad_kwfold(const void* X, int NB, int H, int W, int Cin, const void* dY, long long ldy, int Cout, float* dW, int KH, int KW, cudaStream_t stream);

/* ---- BatchNormalization (43 layers; spnet/models.py:326-336 + Xception) ---- */
int spnet_bn_finalize(long long* stats, long long count, const float* gamma, const float* beta, float eps, float momentum, int unbiased_moving_var, float* a, float* b, float* save_mean, float* save_rstd, float* moving_mean, float* moving_var, int C, cudaStream_t stream);
int spnet_bn_inference_affine(const float* gamma, const float* beta, const float* moving_mean, const float* moving_var, float eps, float* a, float* b, float* save_mean, float* save_rstd, int C, cudaStream_t stream);
int spnet_bn_apply(const void* z, const float* a, const float* b, int act, const void* x, void* out, int dtype, long long rows, int C, cudaStream_t stream);
int spnet_bn_bwd_reduce(void* g, const void* z, const float* save_mean, const float* save_rstd, const float* relu_a, const float* relu_b, int act, long long* stats, int dtype, long long rows, int C, cudaStream_t stream);
int spnet_colstats(const void* z, long long* stats, int dtype, long long rows, int C, cudaStream_t stream);
int spnet_bn_bwd_finalize(long long* stats, long long count, float* dgamma, float* dbeta, float* c1, float* c2, int C, cudaStream_t stream);
int spnet_bn_bwd_dz(const void* g, const void* z, const float* a, const float* save_mean, const float* save_rstd, const float* c1, const float* c2, void* out, int dtype, long long rows, int C, cudaStream_t stream);

/* ---- MaxPooling2D(3,2,'same') + BN-apply + residual Add (Xception blocks 2-4, 13) ---- */
int spnet_maxpool3s2_add_fwd(const void* z, const float* a, const float* b, const void* res, const float* ra, const float* rb, void* out, unsigned char* argmax, int dtype, int B, int H, int W, int C, cudaStream_t stream);
int spnet_maxpool3s2_bwd(const void* gout, const unsigned char* argmax, void* gin, int dtype, int B, int H, int W, int C, cudaStream_t stream);
int spnet_gather_s2(const void* in, void* out, int dtype, int B, int H, int W, int C, int off_h, int off_w, cudaStream_t stream);
int spnet_scatter_s2(const void* in, void* out, int dtype, int B, int H, int W, int C, int off_h, int off_w, cudaStream_t stream);

/* ---- SPNet stem (spnet/models.py:319-340), block1_conv1, block1_conv2 im2col ---- */
int spnet_conv_small_fwd(int which, const void* in, const float* w, const float* in_a, const float* in_b, int act, void* out, void* skip, long long* stats, int dtype, int B, int H, int W, cudaStream_t stream);
int spnet_conv_small_wgrad(int which, const void* in, const float* in_a, const float* in_b, int act, const void* g, float* dw, long long* dw_acc, int dtype, int B, int H, int W, cudaStream_t stream);
int spnet_conv_small_dgrad(int which, const void* g, const float* w, const void* mask_z, const float* mask_a, const float* mask_b, int act, void* gin, int dtype, int B, int H, int W, cudaStream_t stream);
int spnet_stem_k3_to_k4(const float* k3, float* k4, int cout, cudaStream_t stream);
int spnet_stem_k4grad_to_k3grad(const float* g4, float* g3, int cout, cudaStream_t stream);
int spnet_stem_out_fwd(const void* c3, const float* a, const float* b, const void* skip, void* out, int dtype, long long pixels, float rate, const unsigned long long* seed, cudaStream_t stream);
int spnet_stem_out_bwd(const void* g, void* gout, int dtype, long long pixels, float rate, const unsigned long long* seed, cudaStream_t stream);
int spnet_bn3_bwd_reduce(const void* g, const void* z, const float* save_mean, const float* save_rstd, long long* stats, int dtype, long long pixels, cudaStream_t stream);
int spnet_bn3_bwd_dz(const void* g, const void* z, const float* a, const float* save_mean, const float* save_rstd, const float* c1, const float* c2, void* out, int dtype, long long pixels, cudaStream_t stream);
int spnet_im2col3x3(const void* in, const float* a, const float* b, int relu, void* col, int dtype, int B, int H, int W, int C, cudaStream_t stream);
int spnet_col2im3x3(const void* gcol, const void* z, const float* a, const float* b, int relu, void* gin, int dtype, int B, int H, int W, int C, cudaStream_t stream);

/* ---- dense-convolution backbone pieces (keras.applications.InceptionResNetV2 via spnet/models.py:18,357-359):
 *      generic im2col / col2im around the GEMMs, 'valid' max-pool, AveragePooling2D(3,1,'same'), channel-slice
 *      copies (Concatenate), the scaled residual of the Inception-ResNet blocks, bias gradient ---- */
int spnet_im2col(const void* in, void* col, int dtype, int B, int H, int W, int C, int KH, int KW, int sh, int sw, int pt, int pl, int OH, int OW, cudaStream_t stream);
int spnet_col2im(const void* gcol, void* gin, int accumulate, int dtype, int B, int H, int W, int C, int KH, int KW, int sh, int sw, int pt, int pl, int OH, int OW, cudaStream_t stream);
int spnet_maxpool3s2_valid_fwd(const void* z, void* out, unsigned char* argmax, int dtype, int B, int H, int W, int C, cudaStream_t stream);
int spnet_maxpool3s2_valid_bwd(const void* gout, const unsigned char* argmax, void* gin, int dtype, int B, int H, int W, int C, cudaStream_t stream);
int spnet_avgpool3s1(const void* in, void* out, int bwd, int accumulate, int dtype, int B, int H, int W, int C, cudaStream_t stream);
int spnet_copy2d(const void* src, long long ld_src, void* dst, long long ld_dst, int accumulate, int dtype, long long rows, int cols, cudaStream_t stream);
int spnet_residual_fwd(const void* x, const void* u, const float* bias, float scale, int relu, void* y, int dtype, long long rows, int C, cudaStream_t stream);
int spnet_residual_bwd(const void* gy, const void* y, float scale, int relu, void* gx, int accumulate_gx, void* gu, int dtype, long long rows, int C, cudaStream_t stream);
int spnet_colsum_rows(const void* g, float* out, int dtype, long long rows, int C, cudaStream_t stream);

/* ---- optimiser: keras Adam (spnet/models.py:494) + L2 of add_regularization (:47-71) ---- */
/* frozen8 (nullable): one byte per 8 parameters, non-zero = not trainable (layer.trainable = False, spnet/models.py:361-372);
 * g_bf16 (nullable): read the gradients from this bf16 buffer (data-parallel all-reduce in bf16) instead of g. */
int spnet_adam_keras_step(float* p, const float* g, float* m, float* v, long long n, long long n_l2, float l2, const float* lr_t_dev, float beta1, float beta2, float eps, float grad_scale, void* p_bf16, const unsigned char* frozen8, const void* g_bf16, cudaStream_t stream);
/* *out (an order-independent accumulator, 1 entry = 2 int64 words) += scale * sum(p^2); spnet_acc_to_f32 converts
 * accumulators to fp32 (and clears them). spnet_slab_reduce: second half of a split-K GEMM with a fixed summation
 * order (spnet_gemm_bf16 out_mode 3): out = [out +] bias + slab_0 + slab_1 + ... */
int spnet_sumsq(const float* p, long long n, float scale, long long* out, cudaStream_t stream);
int spnet_acc_to_f32(long long* acc, float* out, long long n, int accumulate, int clear, cudaStream_t stream);
int spnet_slab_reduce(const float* slabs, int nslabs, long long slab_stride, long long lds, const float* bias, float* out, long long ldo, int rows, int cols, int accumulate, cudaStream_t stream);
int spnet_cast_f32_to_bf16(const float* src, void* dst, long long n, cudaStream_t stream);
int spnet_cast_bf16_to_f32(const void* src, float* dst, long long n, cudaStream_t stream);
int spnet_bias_fill(const float* bias, float* out, int rows, int cols, cudaStream_t stream);
int spnet_colsum(const float* g, float* out, int rows, int cols, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SPNET_B200_H */
