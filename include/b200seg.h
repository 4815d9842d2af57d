/* b200seg.h -- C ABI of libb200seg.so: the sm_100a kernels behind the reference's model classes.
 *
 * The reference (SEAME-pt/Team02-ObjectDetection) has no FFI layer of its own: its hot path is
 * reached through the torch.nn.Module protocol (src/unet.py:32-51, :137-147) and every operator
 * below replaces one ATen dispatch that path makes (SURVEY.md section 2.1).  The Python mirror of
 * src/unet.py (team02-objectdetection_b200/b200seg/unet.py) binds these with ctypes; see
 * INTEGRATION.md for the stub.
 *
 * Conventions (SURVEY.md section 8b):
 *   - plain C: raw device pointers, ints, floats; no torch / C++ types.
 *   - activations are NHWC ("channels innermost"), dtype B200SEG_F32 or B200SEG_BF16; the channel
 *     count of an NHWC tensor must be a multiple of 16 bytes / sizeof(dtype) unless stated.
 *   - every entry point takes the CUDA stream to launch on, never synchronises, never allocates,
 *     keeps no pointer after it returns, and is CUDA-graph capturable.
 *   - return 0 on success; <0 argument/shape error (nothing launched); >0 a cudaError_t from the
 *     launch.  b200seg_last_error() returns a thread-local message for the last non-zero return.
 *   - no CPU fallback: a host pointer is undefined behaviour, a missing GPU is an error.
 */
#ifndef B200SEG_H_
#define B200SEG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* b200seg_stream_t;

enum { B200SEG_F32 = 0, B200SEG_BF16 = 1 };
/* target (label map) dtypes of the validation-metrics entry points */
enum { B200SEG_I64 = 2, B200SEG_U8 = 3 };
/* logits layout of b200seg_seg_metrics */
enum { B200SEG_NCHW = 0, B200SEG_NHWC = 1 };
enum { B200SEG_ACT_NONE = 0, B200SEG_ACT_RELU = 1, B200SEG_ACT_RELU6 = 2 };

int b200seg_version(void);
const char* b200seg_last_error(void);
/* number of SMs / compute capability major*10+minor of the current device (sanity: 148 / 100). */
int b200seg_device_info(int* sm_count, int* cc);

/* ---------------------------------------------------------------------------------------------
 * Direct 3x3 convolution for tiny Cin (the stem, torchvision mobilenetv2.py:125-127 called from
 * unet.py:15/34; and UNet.inc's first conv, unet.py:58,127).  pad 1, stride 1 or 2.
 *   x  : NCHW [B,Cin,H,W] (f32 or bf16)  -- the model's public input layout
 *   w  : f32 [3][3][Cin][Cout] with the eval-mode BatchNorm scale already folded in
 *   b  : f32 [Cout] folded shift (conv bias and BN), may be NULL
 *   y  : NHWC [B,Ho,Wo,Cout]; Cout % 8 == 0, Cin <= 4
 * replaces aten::convolution + native_batch_norm + hardtanh/relu. */
int b200seg_conv3x3_smallcin(const void* x, int x_dtype, const float* w, const float* b, void* y,
                             int y_dtype, int B, int Cin, int H, int W, int Cout, int stride, int act,
                             b200seg_stream_t s);

/* features.0 + features.1 of the MobileNetV2 encoder as one kernel (eval, BatchNorm folded; unet.py:15,34 ->
 * tv:models/mobilenetv2.py:42-57): stem 3x3 stride 2 (3->32) + ReLU6 -> depthwise 3x3 + ReLU6 -> linear 1x1 (32->16); the two
 * 32-channel half-resolution maps stay in shared memory.  Replaces three aten::convolution (+BN +hardtanh) calls.
 *   x NCHW [B,3,H,W] (f32 | bf16); w_stem f32 [3][3][3][32], b_stem f32 [32]; w_dw bf16 [9][32], b_dw f32 [32];
 *   w_pw bf16 [16][32], b_pw f32 [16]; y NHWC bf16 [B,H/2,W/2,16].  b200seg_stem_mb1_supported: 1 when the shape qualifies. */
int b200seg_stem_mb1_supported(int x_dtype, int H, int W, int Cstem, int Cout);
int b200seg_stem_mb1(const void* x, int x_dtype, const float* w_stem, const float* b_stem, const void* w_dw,
                     const float* b_dw, const void* w_pw, const float* b_pw, void* y, int B, int H, int W,
                     b200seg_stream_t s);

/* Depthwise 3x3 (+folded BN shift +act), NHWC, pad 1, stride 1|2 (mobilenetv2.py:42-51).
 *   w : f32 [9][C] (tap-major, BN scale folded);  b : f32 [C] or NULL. */
int b200seg_dwconv3x3(const void* x, const float* w, const float* b, void* y, int dtype, int B, int H,
                      int W, int C, int stride, int act, b200seg_stream_t s);

/* Same operator for bf16 activations with bf16 taps w [9][C]: the stencil runs on the sm_100a mixed-precision FMA
 * (f32 += bf16 * bf16 read from either half of a packed register), so no unpack instructions are issued; results equal
 * b200seg_dwconv3x3 for bf16-representable taps.  variant: register-blocking choice (0 = default). */
int b200seg_dwconv3x3_bf16w(const void* x, const void* w, const float* b, void* y, int B, int H, int W, int C, int stride,
                            int act, int variant, b200seg_stream_t s);

/* Dense convolution on the 5th-gen tensor cores: TMA -> smem ring -> tcgen05.mma -> TMEM ->
 * epilogue(bias, act, +residual) -> TMA store.  bf16 in / fp32 accumulate / bf16 out.
 * taps = 1 (pointwise, mobilenetv2.py:38,53; unet.py:113,116) or 9 (3x3 pad 1 stride 1, unet.py:58,61).
 *   x   : NHWC bf16 [B,H,W,Cin]          Cin % 8 == 0
 *   w   : bf16 [Cout][taps][Cin]         (K-major "OHWI"; BN scale folded)
 *   b   : f32 [Cout] or NULL
 *   res : NHWC bf16 [B,H,W,Cout] or NULL (added after act: the inverted-residual shortcut,
 *         mobilenetv2.py:61-62)
 *   y   : NHWC bf16 [B,H,W,Cout]         Cout % 8 == 0
 *   flags: bit0 = store straight from registers instead of smem+TMA (debug / odd pitches) */
int b200seg_conv_tc(const void* x, const void* w, const float* b, const void* res, void* y, int B, int H,
                    int W, int Cin, int Cout, int taps, int act, int flags, b200seg_stream_t s);
/* Same convolution of cat([skip, x], channel) without materialising the concatenation (the first 3x3 conv of a decoder
 * stage, unet.py:100-103 + 58): K chunks of the skip are loaded from skip, the rest from x, by TMA.
 *   skip : NHWC bf16 [B,H,W,Cs], Cs % 8 == 0 (Cs = 0: skip unused, identical to b200seg_conv_tc)
 *   x    : NHWC bf16 [B,H,W,Cu], Cu % 8 == 0
 *   w    : bf16 [Cout][taps][Cs + Cu], the packing of the concatenated input
 * Bit-identical to b200seg_conv_tc on the concatenated tensor when Cs % 64 == 0, and with Cs % 16 == 0 on maps narrower
 * than 96 columns; otherwise the fp32 accumulation visits the K groups in another order. */
int b200seg_conv_tc_cat(const void* skip, const void* x, const void* w, const float* b, const void* res, void* y, int B,
                        int H, int W, int Cs, int Cu, int Cout, int taps, int act, int flags, b200seg_stream_t s);

/* 3x3 convolution (pad 1, stride 1) with few output channels (Cout <= 32, or 65..80 for the data gradient of up4.conv.0:
 * N = 240, two accumulators = 480 TMEM columns) on wide maps as a ROW-STACKED implicit GEMM: the
 * three vertical taps are stacked along the MMA N axis (one accumulator of 3*Cout columns per input row), the epilogue sums
 * the three accumulators that meet in an output row.  2.1x fewer tensor-pipe cycles and 3x fewer operand reads than
 * b200seg_conv_tc for the same operands and results (unet.py:58,61 -- up4's double_conv -- and their data gradients).
 * b200seg_conv_rs_supported returns 1 when the shape qualifies.  flags: tuning only (0 = heuristics). */
int b200seg_conv_rs_supported(int H, int W, int Cin, int Cout);
int b200seg_conv_rs(const void* x, const void* w, const float* b, const void* res, void* y, int B, int H, int W, int Cin,
                    int Cout, int act, int flags, b200seg_stream_t s);
/* Two-source input as in b200seg_conv_tc_cat: skip NHWC bf16 [B,H,W,Cs], x NHWC bf16 [B,H,W,Cu], w [Cout][9][Cs + Cu]. */
int b200seg_conv_rs_cat_supported(int H, int W, int Cs, int Cu, int Cout);
int b200seg_conv_rs_cat(const void* skip, const void* x, const void* w, const float* b, const void* res, void* y, int B,
                        int H, int W, int Cs, int Cu, int Cout, int act, int flags, b200seg_stream_t s);

/* Depthwise 3x3 on the tensor cores (bf16): the same TMA/tcgen05 pipeline as b200seg_conv_tc run over
 * 64-channel chunks with BLOCK-DIAGONAL weights, so the 9-tap stencil costs no CUDA-core FMAs or
 * bf16<->f32 conversions and the kernel is bounded by HBM instead of instruction issue
 * (mobilenetv2.py:42-51; pad 1, stride 1|2 -- stride 2 uses TMA element strides).
 *   x     : NHWC bf16 [B,H,W,C], C % 8 == 0
 *   wdiag : bf16 [C][9][64], wdiag[c][t][k] = w[c][t] * bn_scale[c] if k == c % 64 else 0
 *   b     : f32 [C] or NULL;   y : NHWC bf16 [B,Ho,Wo,C] */
int b200seg_dwconv3x3_tc(const void* x, const void* wdiag, const float* b, void* y, int B, int H, int W,
                         int C, int stride, int act, int flags, b200seg_stream_t s);

/* Same contract on the FP32 SIMT pipes (no tensor cores) for the fp32 parity configuration
 * (BASELINE config 1: 1e-4 relative needs true fp32 products, SURVEY finding 10c).  dtype selects
 * the storage type of x/res/y; w is f32 [Cout][taps][Cin]. */
int b200seg_conv_simt(const void* x, const float* w, const float* b, const void* res, void* y, int dtype,
                      int B, int H, int W, int Cin, int Cout, int taps, int act, b200seg_stream_t s);

/* up.forward (unet.py:100-103): y[..., :Cs] = skip ; y[..., Cs:] = bilinear_x2(x, align_corners=False).
 *   skip NHWC [B,2h,2w,Cs], x NHWC [B,h,w,Cu], y NHWC [B,2h,2w,Cs+Cu].  Cs = 0 (skip may be NULL): the upsample alone,
 *   which b200seg_conv_tc_cat / b200seg_conv_rs_cat then read next to the skip tensor. */
int b200seg_upsample2x_concat(const void* skip, const void* x, void* y, int dtype, int B, int h, int w,
                              int Cs, int Cu, b200seg_stream_t s);

/* final_upsample (unet.py:30,49): bilinear x2 align_corners=True of NHWC logits [B,h,w,ldc]
 * (first C channels valid) into NCHW [B,C,2h,2w] of out_dtype -- the model's public output. */
int b200seg_upsample2x_ac_nchw(const void* logits, int dtype, int ldc, void* out, int out_dtype, int B,
                               int h, int w, int C, b200seg_stream_t s);
/* Same, fused with the per-pixel argmax inference.py:64 takes: writes uint8 [B,2h,2w]. */
int b200seg_upsample2x_ac_argmax(const void* logits, int dtype, int ldc, uint8_t* mask, int B, int h,
                                 int w, int C, b200seg_stream_t s);

/* One fused torchvision InvertedResidual block with expand ratio > 1, eval mode, BatchNorm folded, bf16
 * (tv:models/mobilenetv2.py:38-62 -- ConvBNReLU6 1x1 expand, ConvBNReLU6 depthwise 3x3 stride s, ConvBN 1x1
 * project, + x when stride 1 and Cin == Cout; reached through unet.py:15-19,34-42).  The expanded activation
 * stays in shared memory / TMEM.
 *   x [B,H,W,Cin] bf16;  w_exp [Ce][Cin] bf16;  w_proj [Cout][Ce] bf16;  y [B,Ho,Wo,Cout] bf16
 *   b_exp, b_dw: f32 [ceil64(Ce)] zero padded;  w_dw: bf16 [9][ceil64(Ce)] zero padded (the stencil runs on the
 *   mixed-precision FMA, f32 += bf16 * bf16);  b_proj: f32 [ceil16(Cout)]
 *   flags: tuning only (0 = heuristics). */
int b200seg_mbconv(const void* x, const void* w_exp, const float* b_exp, const void* w_dw, const float* b_dw,
                   const void* w_proj, const float* b_proj, int residual, void* y, int B, int H, int W, int Cin,
                   int Ce, int Cout, int stride, int flags, b200seg_stream_t s);

/* The output tail of MobileNetV2UNet.forward in one kernel, eval mode, bf16 (unet.py:47-49, :108-121, :30):
 * outconv(32, C) = 1x1 32->16 (+folded BN) + ReLU -> 1x1 16->C + bias, then final_upsample (bilinear x2,
 * align_corners=True) to NCHW logits (mask == NULL) or to the uint8 argmax mask of inference.py:64 (out == NULL).
 *   x [B,h,w,32] bf16;  w0 bf16 [16][32], b0 f32 [16];  w3 bf16 [16][16] (rows >= C zero), b3 f32 [16];  C <= 16. */
int b200seg_tail_fused(const void* x, const void* w0, const float* b0, const void* w3, const float* b3, void* out,
                       int out_dtype, uint8_t* mask, int B, int h, int w, int C, b200seg_stream_t s);

/* Validation metrics (the commented-out validation loop of train.py:46-74) accumulated on the device.  Both entry points
 * ADD into the caller's state (zero it to start):
 *   confusion int64 [C][C]  row = target class, column = predicted class (argmax, first maximum wins like torch.argmax)
 *   counts    int64 [2]     [0] += pixels whose target is in [0,C) and not ignore_index; [1] += pixels whose target is
 *                           neither in range nor ignore_index (nn.CrossEntropyLoss raises on those; the Python layer
 *                           reports a NaN loss).  A pixel whose target equals ignore_index contributes nothing, also when
 *                           ignore_index is a class index.
 *   loss_sum  f64 [1]       += sum over the counted pixels of logsumexp(z) - z[target] (f32 per pixel and per CTA)
 *   target    [B,2h,2w] (tail) or [B,H,W] of target_dtype B200SEG_I64 (16-byte aligned for the tail) or B200SEG_U8
 *             (2-byte aligned for the tail); a uint8 label equal to ignore_index is ignored like an int64 one.
 * b200seg_tail_fused_metrics: the output tail above (same operands, C <= 16) with the metrics taken in its epilogue from the
 *   same interpolated logits the mask mode compares, so the confusion equals the histogram of that mask exactly; no
 *   logits tensor is written.
 * b200seg_seg_metrics: the same metrics over existing logits (f32 | bf16), C <= 64.  layout B200SEG_NCHW: [B,C,H,W]
 *   (ldc ignored); B200SEG_NHWC: [B,H,W,ldc] with the first C channels valid (UNet's padded logits buffer). */
int b200seg_tail_fused_metrics(const void* x, const void* w0, const float* b0, const void* w3, const float* b3,
                               const void* target, int target_dtype, long long ignore_index, int64_t* confusion,
                               int64_t* counts, double* loss_sum, int B, int h, int w, int C, b200seg_stream_t s);
int b200seg_seg_metrics(const void* logits, int dtype, int layout, int ldc, const void* target, int target_dtype,
                        long long ignore_index, int64_t* confusion, int64_t* counts, double* loss_sum, int B, int C, int H,
                        int W, b200seg_stream_t s);

/* NHWC [B,H,W,ldc] (first C valid) -> NCHW [B,C,H,W] (UNet returns logits at input resolution). */
int b200seg_nhwc_to_nchw(const void* x, int dtype, int ldc, void* out, int out_dtype, int B, int H, int W,
                         int C, b200seg_stream_t s);

/* MaxPool2d(2) NHWC (unet.py:85). */
int b200seg_maxpool2x2(const void* x, void* y, int dtype, int B, int H, int W, int C, b200seg_stream_t s);

/* nn.CrossEntropyLoss() forward fused with its gradient (main.py:99, train.py:37-38):
 *   logits NCHW f32 [B,C,H,W] (any C >= 1), target int64 [B,H,W] in [0,C) or ignore_index
 *   loss_sum : f32[1], accumulates sum of -log softmax[target] over the non-ignored pixels (caller zeroes)
 *   dlogits  : NCHW f32 (softmax - onehot) * grad_scale / counts[0], or NULL for forward only
 *   counts   : device f32[2] from b200seg_ce_count (counts[0] = non-ignored targets: the divisor of the 'mean'
 *              reduction), or NULL: dlogits is scaled by grad_scale alone. */
int b200seg_softmax_ce(const float* logits, const int64_t* target, float* loss_sum, float* dlogits,
                       float grad_scale, const float* counts, int B, int C, int H, int W, b200seg_stream_t s);
/* d(logits) *= gout[0] in place (the incoming gradient of the scalar loss, train.py:38); a no-op on the device when it is 1 */
int b200seg_scale_unless_one(float* x, long long n, const float* s, b200seg_stream_t st);
/* counts[0] += number of targets in [0,C); counts[1] += number of targets that are neither in range nor ignore_index
 * (torch raises on those; the Python binding turns a non-zero counts[1] into a NaN loss). Caller zeroes counts. */
int b200seg_ce_count(const int64_t* target, float* counts, long long N, int C, long long ignore_index,
                     b200seg_stream_t s);

/* nn.CrossEntropyLoss(weight, ignore_index, reduction, label_smoothing) with int64 or uint8 targets, fused forward and
 * gradient.  A pixel is counted when its target t is in [0,C) and t != ignore_index (a uint8 label equals ignore_index only
 * when ignore_index is in [0,255]).  For a counted pixel, with lse = logsumexp(z), w the class weights (all ones when
 * weight is NULL), Wsum = sum_c w_c, eps = label_smoothing in [0,1]:
 *   loss = (1-eps) w_t (lse - z_t) + eps/C sum_c w_c (lse - z_c)
 *   grad = (1-eps) w_t (softmax - onehot_t) + eps/C (Wsum softmax - w)
 * Other pixels: loss 0 and gradient 0, but a bad label (neither counted nor ignore_index) has a NaN loss.
 *   logits NCHW f32 [B,C,H,W] (any C >= 1); target [B,H,W] of target_dtype B200SEG_I64 | B200SEG_U8; weight device f32 [C]
 *   or NULL.
 * b200seg_softmax_ce_ex: exactly one of
 *   loss_sum f64[1] ('mean' / 'sum'): += sum of the pixel losses (caller zeroes); dlogits (or NULL) = grad / denom[0], or
 *            grad alone when denom is NULL ('sum');
 *   loss_map f32 [B,H,W] ('none'): the pixel losses; dlogits and denom must be NULL.
 * b200seg_ce_count_ex: denom f64[2] += (sum of w_t over the counted pixels = the 'mean' divisor, number of bad labels);
 *   caller zeroes.  N = B*H*W.
 * b200seg_softmax_ce_ex_bwd: the backward of the loss map: dlogits = grad * gout (gout f32 [B,H,W]) in one pass over the
 *   logits.
 * 16-byte aligned logits, dlogits, loss_map, gout and target (uint8: 4-byte) with H*W % 4 == 0 and C <= 16 take the
 * 4-pixel vector path; anything else the one-pixel kernels. */
int b200seg_softmax_ce_ex(const float* logits, const void* target, int target_dtype, long long ignore_index,
                          const float* weight, float label_smoothing, double* loss_sum, float* loss_map, float* dlogits,
                          const double* denom, int B, int C, int H, int W, b200seg_stream_t s);
int b200seg_ce_count_ex(const void* target, int target_dtype, long long ignore_index, const float* weight, double* denom,
                        long long N, int C, b200seg_stream_t s);
int b200seg_softmax_ce_ex_bwd(const float* logits, const void* target, int target_dtype, long long ignore_index,
                              const float* weight, float label_smoothing, const float* gout, float* dlogits, int B, int C,
                              int H, int W, b200seg_stream_t s);

/* Any class count (outconv(in_ch, out_ch), unet.py:108-121, takes any out_ch; the fast kernels above hold <= 16
 * channels in registers): final_upsample to NCHW logits (mask == NULL) or to the uint8 argmax mask (out == NULL) from
 * NHWC logits with pixel pitch ldc >= C; its adjoint (dlogits NHWC [B,h,w,ldc], channels >= C zeroed); and the argmax
 * of NHWC logits at input resolution (plain UNet has no final upsample; inference.py:64). */
int b200seg_upsample2x_ac_generic(const void* logits, int dtype, int ldc, void* out, int out_dtype, uint8_t* mask, int B,
                                  int h, int w, int C, b200seg_stream_t s);
int b200seg_final_bwd_generic(const float* dout, void* dlogits, int dtype, int B, int h, int w, int C, int ldc,
                              b200seg_stream_t s);
int b200seg_nhwc_argmax(const void* x, int dtype, int ldc, uint8_t* mask, long long P, int C, b200seg_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * Training path (train.py:35-39: model.train() forward, loss.backward()).  Activations NHWC viewed as
 * [P = B*H*W pixels, C]; per-channel statistics are accumulated across CTAs in f64 buffers the caller
 * zeroes.  Reduction outputs come in `nslot` copies `slot_stride` doubles apart (CTA i adds into copy i % nslot;
 * the consumer -- bn_finalize / f64_to_f32 -- sums the copies): one copy serialises ~1200 atomics per address.
 * dgrad of the dense convs reuses b200seg_conv_simt / b200seg_conv_tc with transposed weights.
 * --------------------------------------------------------------------------------------------- */
/* native_batch_norm (training): sum[c] += sum_p (z-k), sumsq[c] += sum_p (z-k)^2 with the per-channel shift k = z at
 * pixel 0 (shifted sums: no catastrophic cancellation for nearly constant channels); bn_finalize adds k back. */
int b200seg_bn_stats(const void* z, int dtype, long long P, int C, double* sum, double* sumsq, int nslot,
                     long long slot_stride, b200seg_stream_t s);
/* mean/biased var -> invstd; scale = gamma*invstd, shift = beta - mean*scale; running stats updated with
 * momentum and the unbiased variance (nn.BatchNorm2d defaults); running_* may be NULL. */
int b200seg_bn_finalize(const void* z, int dtype, const double* sum, const double* sumsq, int nslot,
                        long long slot_stride, long long n, const float* gamma,
                        const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                        float* mean, float* invstd, float* scale, float* shift, int C, b200seg_stream_t s);
/* a = act(z*scale + shift) (+ res)   -- BN apply + ReLU/ReLU6 (+ inverted-residual shortcut) */
int b200seg_bn_apply(const void* z, const float* scale, const float* shift, const void* res, void* a, int dtype,
                     long long P, int C, int act, b200seg_stream_t s);
/* b200seg_bn_finalize + b200seg_bn_apply in one launch: every block derives the per-channel constants from the slot sums
 * of b200seg_bn_stats (st_sums: f64 [nslot][2][C] = sum | sum of squares, shifted by z at pixel 0) and the first row of
 * blocks publishes sv = f32 [4][C] (mean, invstd, scale, shift) and updates the running statistics (train.py:24,36). */
int b200seg_bn_finalize_apply(const void* z, const double* st_sums, int nslot, const float* gamma, const float* beta, float eps,
                              float momentum, float* running_mean, float* running_var, float* sv, const void* res, void* a,
                              int dtype, long long P, int C, int act, b200seg_stream_t s);
/* native_batch_norm_backward + hardtanh/threshold_backward, pass 1: sg[c] += sum g, sgx[c] += sum g*xhat,
 * g = da * act'(z*scale+shift), xhat = (z-mean)*invstd.   (d beta = sg, d gamma = sgx) */
int b200seg_bn_bwd_reduce(const void* da, const void* z, const float* scale, const float* shift, const float* mean,
                          const float* invstd, int dtype, long long P, int C, int act, double* sg, double* sgx,
                          int nslot, long long slot_stride, b200seg_stream_t s);
/* pass 2: dz = scale * (g - sg/P - xhat * sgx/P); sg/sgx are the pass-1 sums converted to f32 (f64 arithmetic in
 * the per-element loop would run at 1/64 rate) */
int b200seg_bn_bwd_apply(const void* da, const void* z, const float* scale, const float* shift, const float* mean,
                         const float* invstd, const float* sg, const float* sgx, void* dz, int dtype, long long P,
                         int C, int act, b200seg_stream_t s);
/* pass 2 reading the f64 slot sums of pass 1 directly (red: [nslot][2][C] = sum g | sum g*xhat; sv as above): no f64 -> f32
 * launch between the two passes. */
int b200seg_bn_bwd_apply_slots(const void* da, const void* z, const float* sv, const double* red, int nslot, void* dz,
                               int dtype, long long P, int C, int act, b200seg_stream_t s);
/* Train-mode BatchNorm2d forward / backward of the small and mid-size layers in ONE launch per direction: a thread-block cluster
 * owns 16 channels, reduces through distributed shared memory and applies in the same kernel (nn.BatchNorm2d in model.train(),
 * train.py:24,36, and its backward, train.py:38).  bf16, C % 16 == 0, tensors up to ~40 MB (b200seg_bn_cluster_supported);
 * larger layers use the grid-wide kernels above.  sv: f32 [4][C] = mean, invstd, scale, shift; red: zeroed f64 [nslot][2][C],
 * slot 0 receives sum g (d beta) and sum g*xhat (d gamma). */
int b200seg_bn_cluster_supported(int dtype, long long P, int C);
int b200seg_bn_cluster_bwd_supported(int dtype, long long P, int C);
int b200seg_bn_cluster_fwd(const void* z, long long P, int C, const float* gamma, const float* beta, float eps, float momentum,
                           float* running_mean, float* running_var, float* sv, const void* res, void* a, int act,
                           b200seg_stream_t s);
int b200seg_bn_cluster_bwd(const void* da, const void* z, const float* sv, long long P, int C, int act, double* red, void* dz,
                           b200seg_stream_t s);
/* dz = da * act'(a_out) for a layer without BatchNorm */
int b200seg_act_bwd(const void* da, const void* a_out, void* dz, int dtype, long long N, int act, b200seg_stream_t s);
/* out[slot][c] += sum_p x[p][c]  (bias gradients) ; out[i] = scale * sum_slot in[slot*slot_stride + i] as f32 */
int b200seg_colsum(const void* x, int dtype, long long P, int C, double* out, int nslot, long long slot_stride,
                   b200seg_stream_t s);
int b200seg_f64_to_f32(const double* in, float* out, int n, int nslot, long long slot_stride, float scale,
                       b200seg_stream_t s);
/* convolution_backward (weight): dw f32 [Cout][taps][Cin] += sum_p dz[p][co] * x[p shifted by tap][ci]; caller zeroes dw */
int b200seg_conv_wgrad(const void* x, const void* dz, float* dw, int dtype, int B, int H, int W, int Cin, int Cout,
                       int taps, b200seg_stream_t s);
/* same on the tensor cores (bf16 x / dz, Cin % 8 == 0, Cout % 8 == 0): the pixel axis is the MMA reduction axis,
 * the NHWC tiles are read as MN-major UMMA operands, partial tiles are added with red.global.add.v4.f32 */
int b200seg_conv_wgrad_tc(const void* x, const void* dz, float* dw, int B, int H, int W, int Cin, int Cout, int taps,
                          b200seg_stream_t s);
/* depthwise backward: dx (+= acc_in) from dz with taps w f32 [9][C]; dw f64 [9][C] += ... (caller zeroes) */
int b200seg_dw_dgrad(const void* dz, const float* w, const void* acc_in, void* dx, int dtype, int B, int H, int W,
                     int C, int stride, b200seg_stream_t s);
int b200seg_dw_wgrad(const void* x, const void* dz, double* dw, int nslot, int dtype, int B, int H, int W, int C,
                     int stride, b200seg_stream_t s);   /* dw: nslot copies of [9][C], summed by f64_to_f32 */
/* stem / first-conv weight gradient: x NCHW, dz NHWC, dw f32 [3][3][Cin][Cout] += ... (caller zeroes) */
int b200seg_smallcin_wgrad(const void* x, int x_dtype, const void* dz, int dtype, float* dw, int B, int Cin, int H,
                           int W, int Cout, int stride, b200seg_stream_t s);
/* adjoint of b200seg_upsample2x_concat: dskip = dcat[..., :Cs] (+ acc_skip), dx = bilinear^T(dcat[..., Cs:]) */
int b200seg_upcat_bwd(const void* dcat, const void* acc_skip, void* dskip, void* dx, int dtype, int B, int h, int w,
                      int Cs, int Cu, b200seg_stream_t s);
/* adjoint of b200seg_upsample2x_ac_nchw: dout NCHW f32 [B,C,2h,2w] -> dlogits NHWC [B,h,w,16] */
int b200seg_final_bwd(const float* dout, void* dlogits, int dtype, int B, int h, int w, int C, b200seg_stream_t s);
/* adjoint of b200seg_nhwc_to_nchw, and of b200seg_maxpool2x2 (gradient to the first maximum, += acc_in) */
int b200seg_nchw_to_nhwc_pad(const float* x, void* y, int dtype, int B, int C, int H, int W, int ldc,
                             b200seg_stream_t s);
int b200seg_maxpool_bwd(const void* x, const void* dy, const void* acc_in, void* dx, int dtype, int B, int H, int W,
                        int C, b200seg_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * Fused multi-tensor Adam (SURVEY 8f): torch.optim.Adam(params, lr) of main.py:100 / train.py:39 for all tensors
 * in one launch.  table: device array of {float* p; const float* g; float* m; float* v; long long n;} (40 bytes
 * each); block b updates elements [chunk_index[b]*CHUNK, +CHUNK) of tensor chunk_tensor[b], CHUNK =
 * b200seg_adam_chunk().  bias_corr1/2 = 1 - beta^t for the step count t >= 1 (host side, as torch computes them).
 * --------------------------------------------------------------------------------------------- */
int b200seg_adam_multi(const void* table, const int* chunk_tensor, const int* chunk_index, int n_chunks, float lr,
                       double one_minus_beta1, float beta2, double one_minus_beta2, float eps, float weight_decay,
                       double bias_corr1, double bias_corr2, b200seg_stream_t s);
int b200seg_adam_chunk(void);
/* Weight repack of the training step for all layers in one launch (csrc/adam.cu).  table: device array of
 * {const float* w (OIHW); void* fwd; void* dgrad; int cout, cin, kk (= taps), cout_pad, kind, pad;} (48 bytes);
 * kind 0: bf16 fwd [cout_pad][kk][cin] + dgrad [cin][kk flipped][cout_pad]; 1: the same in f32; 2: stem f32
 * [kk][cin][cout]; 3: depthwise f32 [kk][cout].  Block b handles elements [chunk_index[b]*CHUNK, +CHUNK) of the padded
 * OIHW tensor chunk_tensor[b], CHUNK = b200seg_pack_chunk(). */
int b200seg_pack_weights_multi(const void* table, const int* chunk_tensor, const int* chunk_index, int n_chunks,
                               b200seg_stream_t s);
int b200seg_pack_chunk(void);
/* Eval-mode weight preparation (model.eval(), inference.py:25) for all layers in one launch: BatchNorm folded into the
 * convolution in fp32 (w' = w*g/sqrt(rv+eps), b' = beta + (b - rm)*g/sqrt(rv+eps)) and written in the operand layout of
 * the forward kernels.  table: device array of {const float* w (OIHW), cbias, gamma, beta, rmean, rvar (NULL gamma = no
 * BN); void* out_w; float* out_b (or NULL); int cout, cin, kk, ldw, kind; float eps; long long pad;} (96 bytes), one row
 * per output operand.  kind 0/1: dense bf16/f32 [cout_pad][kk][cin]; 2: stem f32 [kk][cin][cout]; 3: depthwise f32
 * [kk][ldw]; 4: depthwise block-diagonal bf16 [C][kk][64]; 5: depthwise bf16 [kk][ldw].  Outputs are caller-zeroed (padding
 * is never written).  Chunking as above, CHUNK = b200seg_fold_chunk() over cout*cin*kk (+ cout shift elements). */
int b200seg_fold_pack_eval_multi(const void* table, const int* chunk_tensor, const int* chunk_index, int n_chunks,
                                 b200seg_stream_t s);
int b200seg_fold_chunk(void);
/* Gradient finalize (loss.backward() -> p.grad, train.py:38): every parameter gradient of one bucket from the backward
 * kernels' staging layouts into the parameters' own layout inside the flat gradient arena, one launch, pre-scaled (1/world
 * for the data-parallel mean).  table: device array of {float* dst; const void* src; long long n; long long slot_stride;
 * int kind, cout, cin, kk, nslot, pad; float scale; int pad;} (64 bytes).  kind 0: f64 slot sums -> f32 [n]; 1: dense f32
 * [cout_pad][kk][cin] -> OIHW; 2: stem f32 [kk][cin][cout] -> OIHW; 3: depthwise f64 slot sums [kk][C] -> [C][kk].  Block b
 * handles elements [chunk_index[b]*CHUNK, +CHUNK) of tensor chunk_tensor[b], CHUNK = b200seg_grad_chunk(). */
int b200seg_grad_finalize_multi(const void* table, const int* chunk_tensor, const int* chunk_index, int n_chunks,
                                b200seg_stream_t s);
int b200seg_grad_chunk(void);

/* ---------------------------------------------------------------------------------------------
 * Frame pre-processing of inference.py:28-46 for a batch (SURVEY 8f): uint8 HWC BGR frames [B,Hs,Ws,3] ->
 * cv2.resize(INTER_LINEAR, bit-exact fixed point) to HxW -> RGB -> /255 -> (x - mean) / std -> NCHW [B,3,H,W] of
 * out_dtype; rgb (nullable) receives the resized RGB uint8 image [B,H,W,3] (the function's second return value).
 * --------------------------------------------------------------------------------------------- */
int b200seg_preprocess_u8(const uint8_t* frames, int B, int Hs, int Ws, void* out, int out_dtype, uint8_t* rgb, int H,
                          int W, float mean0, float mean1, float mean2, float std0, float std1, float std2,
                          b200seg_stream_t s);

/* Dataset label remap on the device (the class_map loops of BDD100KDataset.py:23-35,66-69, CarlaDataset.py, SEAMEDataset.py, followed
 * by `.long()`): out[i] = lut256[in[i]], uint8 labels -> int64 targets.  Unmapped source classes map to whatever the table holds
 * (0 = background in the reference). */
int b200seg_remap_labels(const uint8_t* in, int64_t* out, const uint8_t* lut256, long long n, b200seg_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * Object boxes from the class mask (inference.py:48-146, overlay_predictions), bit-equal to cv2 4.13 for every primitive:
 * cv2.resize(mask [B,Hm,Wm] uint8, (W, H), INTER_NEAREST) -> per selected class classes[0..K-1] (1 <= K <= 16, distinct,
 * in [0, 255]; a HOST array) the binary plane resized == class -> cv2.morphologyEx(MORPH_CLOSE, ones(close, close)) (close
 * odd, 1..15; 1 = no close) -> cv2.connectedComponentsWithStats(connectivity=8).  Rows of the components with area >=
 * min_area, per frame in (class position, cv2 label) order: stats int32 [B,max_objects,7] = class, label, left, top,
 * width, height, area and centroid float64 [B,max_objects,2]; rows past the count are zero.  count int32 [B] = components
 * with area >= min_area (may exceed max_objects: the rows past capacity are dropped).  labels (nullable) int32 [B,K,H,W]
 * receives the cv2 label image of every plane.  workspace: device memory of at least b200seg_detect_workspace_bytes(B, K,
 * H, W) bytes, 256-byte aligned.  Enqueues its kernels on s: no allocation, no synchronisation (capturable).
 * --------------------------------------------------------------------------------------------- */
int b200seg_detect_workspace_bytes(int B, int K, int H, int W, long long* bytes);
int b200seg_detect_objects(const uint8_t* mask, int B, int Hm, int Wm, int H, int W, const int* classes, int K, int close,
                           int min_area, int max_objects, void* workspace, long long workspace_bytes, int* count, int* stats,
                           double* centroid, int* labels, b200seg_stream_t s);
/* cv2.addWeighted(frames, alpha, palette[resized mask], beta, gamma) on uint8 BGR frames [B,H,W,3]: the mask [B,Hm,Wm] is
 * resized INTER_NEAREST to HxW, palette is a device array of npal (0..256) BGR uint8 colours, mask values >= npal blend with
 * black; out[B,H,W,3] = saturate(rint(fmaf(frame, alpha, fmaf(colour, beta, gamma)))). */
int b200seg_overlay(const uint8_t* frames, const uint8_t* mask, int B, int Hm, int Wm, int H, int W, const uint8_t* palette,
                    int npal, float alpha, float beta, float gamma, uint8_t* out, b200seg_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* B200SEG_H_ */
