/* b2u.h -- C ABI of libb200unet.so: the B200 (sm_100a) kernels behind the UNet segmentation hot path of
 * clolckliang/unet-pytorch.
 *
 * The reference has no FFI layer (it is pure Python on torch.nn); the boundary this library plugs into is the
 * set of torch.nn calls made by nets/unet.py, nets/vgg.py, nets/unet_training.py and utils/utils_metrics.py.
 * Every entry point below names the reference call it replaces (path:line under the reference repo).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless stated otherwise; the library never allocates, frees or retains
 *     caller memory (workspaces are passed in; sizes come from the *_workspace functions);
 *   - activations/gradients are NHWC bf16 ("void*"), C a multiple of 8 (64 for the tensor-core convs);
 *     logits and parameters are fp32 in the reference's own layouts (NCHW, OIHW);
 *   - `stream` is a cudaStream_t (CUstream); launches are asynchronous on it;
 *   - return value 0 = ok, otherwise a B2U_ERR_* code; b2u_last_error() gives the message (thread-local).
 *
 * libb200unet_fp32.so (csrc/validation_fp32.cu) is the fp32 VALIDATION build of this same header: the entry points the
 * host engines use, with every "void*" activation / gradient / packed operand as fp32 instead of bf16 and CUDA-core
 * contractions (BASELINE tolerance "<= 1e-5 for an fp32 validation build"); test tooling only, never the product path.
 */
#ifndef B2U_H_
#define B2U_H_
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2U_OK 0
#define B2U_ERR_SHAPE 1
#define B2U_ERR_CUDA 2
#define B2U_ERR_DRIVER 3
#define B2U_ERR_NCCL 4
#define B2U_ERR_ARG 5

const char* b2u_last_error(void);
int b2u_version(void);
int b2u_num_sms(void);
/* number of kernel launches made by this library since load / the last reset (process-wide) */
long long b2u_launch_count(void);
void b2u_reset_launch_count(void);

/* ---- layout / packing ------------------------------------------------------------------------------------ */
/* first conv of the encoder (nets/vgg.py:53 with in_channels=3): NCHW fp32 image -> im2col rows [N,H,W,64] bf16,
 * column k = (r*3+s)*Cin + c, zero padded; the conv itself then is a 1x1 b2u_conv_fprop with K = 64. */
int b2u_im2col_first(const float* x_nchw, void* col, int N, int Cin, int H, int W, void* stream);
/* nn.Conv2d.weight (OIHW fp32, nets/vgg.py:53, nets/unet.py:11-12) -> bf16 K-major operands:
 * wf[Cout][taps*Cin] for fprop, wd[Cin][taps*Cout] (taps flipped) for dgrad; either may be NULL. */
int b2u_pack_weights(const float* w_oihw, void* wf, void* wd, int Cout, int Cin, int taps, void* stream);
int b2u_pack_weights_first(const float* w_oihw, void* wf, int Cout, int Cin, void* stream);
/* every conv of the model in one launch; table (DEVICE memory): n x {const float* w; void* wf; void* wd; long long start;
 * int Cout, Cin, taps, first, C0, C0_pad, Ctot_pad, Cout_pad} (64 B each); start = first work block of the layer,
 * (Cout/32)*(Cin/32) blocks per layer (first layer: ceil(Cout/32)); operands may be channel-padded to multiples of 64 */
int b2u_pack_weights_multi(const void* table, int n, long long total_blocks, void* stream);
int b2u_nhwc_bf16_to_nchw_f32(const void* x, float* y, int N, int C, int H, int W, void* stream);
int b2u_nchw_f32_to_nhwc_bf16(const float* x, void* y, int N, int C, int H, int W, void* stream);
/* same with the channel dimension zero-padded to Cpad (the 3-channel image feeding a 1x1 first conv) */
int b2u_nchw_f32_to_nhwc_bf16_padded(const float* x, void* y, int N, int C, int H, int W, int Cpad, void* stream);
/* device-side input pipeline: raw uint8 HWC image -> `preprocess_input` (/255) + CHW fp32 (utils/dataloader.py:41,
 * utils/utils.py:64-66), uint8 label map -> int64 (dataloader.py:43); 4 B/pixel over PCIe instead of 20 */
int b2u_u8hwc_to_nchw_f32(const unsigned char* x, float* y, int N, int H, int W, int C, float scale, void* stream);
int b2u_u8_to_i64(const unsigned char* x, long long* y, long long n, void* stream);
/* the predictor's letterbox (utils/utils.py:22-34 resize_image + preprocess_input + transpose, unet.py:116-120) for a batch
 * of uint8 RGB images of different sizes, bit-exact with PIL's Image.resize(..., BICUBIC) on a (128,128,128) canvas and
 * numpy's float32 / 255.0.  An item is 64 B: {const uint8* src ([ih][iw][3], device); int ih, iw, nh, nw, dy, dx; int kx,
 * ky; int64 coef_x, coef_y, tmp}.  The caller sets src .. dx in a HOST table (nw, nh = int(iw * scale), int(ih * scale),
 * dx, dy = (W - nw) / 2, (H - nh) / 2, as resize_image computes them); b2u_letterbox_workspace fills kx .. tmp and returns
 * the workspace bytes (0 and an error message if an item does not fit the H x W canvas).  b2u_letterbox_bicubic then
 * reads that table from DEVICE memory and writes fp32 NCHW [count][3][H][W]; ws must hold the bytes the plan returned. */
size_t b2u_letterbox_workspace(void* host_items, int count, int H, int W);
int b2u_letterbox_bicubic(const void* items, int count, float* out, int H, int W, void* ws, size_t ws_bytes, void* stream);

/* ---- tensor-core convolutions (tcgen05 implicit GEMM) ------------------------------------------------------ */
/* y = [relu](conv(cat(x0, x1), w) + bias).  Replaces nn.Conv2d(k=3,p=1 | k=1)+ReLU (nets/vgg.py:53-57,
 * nets/unet.py:11-12,18-21) and, with x1 != NULL, torch.cat([skip, up], 1) + conv (nets/unet.py:17-18).
 * taps = 9 (3x3, pad 1) or 1.  C0, C1, Cout multiples of 64.  bn_override: 0 = choose the tiling; bits 0..15 force the
 * N tile (64/128/192/256), bit 16 forces one 8x16-pixel M tile per CTA step, bit 17 caps the stack at two M tiles (the
 * unmasked N = 64 layers default to four) (tests exercise every variant). */
int b2u_conv_fprop(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* bias, void* y, int N,
                   int H, int W, int Cout, int taps, int relu, int bn_override, void* stream);
/* b2u_conv_fprop that also emits the BatchNorm statistics of its output (conv -> nn.BatchNorm2d chains,
 * nets/TraditionalUnet.py:9-14, nets/resnet.py:77-95, nets/LightWeightUnet.py:8-11, nets/UltraLightweightUnet*.py):
 * stat_partial [b2u_conv_stat_rows(...)][2][Cout] fp32 = per M tile, the sums of z and z^2 over its in-image pixels, taken
 * from the bf16 values as stored; b2u_bn_fwd_train_stats consumes them instead of re-reading z */
int b2u_conv_stat_rows(int N, int H, int W, int Cout, int taps, int bn_override);
int b2u_conv_fprop_stats(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* bias, void* y, int N,
                         int H, int W, int Cout, int taps, int relu, int bn_override, float* stat_partial, int stat_rows,
                         void* stream);
/* b2u_conv_dgrad that also emits, per M tile, the column sums (and sums of squares) of the gradient it stores, after the
 * ReLU mask: stat_partial [b2u_conv_dgrad_stat_rows(...)][2][C0 + C1] fp32.  dx is the pre-activation gradient of the conv
 * below, so the sums are that conv's bias gradient (autograd of nn.Conv2d's bias, nets/vgg.py:53): b2u_bias_from_stats folds
 * them into db[C] and the separate pass over dz (b2u_bias_grad) is not needed. */
int b2u_conv_dgrad_stat_rows(int N, int H, int W, int Ctot, int taps, int bn_override, int masked);
int b2u_conv_dgrad_stats(const void* dz, int Cz, const void* wd, void* dx0, int C0, void* dx1, int C1, const void* mask,
                         int N, int H, int W, int taps, int bn_override, float* stat_partial, int stat_rows, void* stream);
int b2u_bias_from_stats(float* stat_partial /* second-quantity slots are used as scratch */, int rows, int C, float* db, void* stream);
/* ReLU backward from a BIT mask (r2).  b2u_conv_fprop_relu_bits = b2u_conv_fprop (or, with low != NULL and x1 == NULL,
 * b2u_decoder_conv_fprop) with ReLU, which also writes bits_out [N,H,W,Cout/64] 64-bit words: bit c % 64 of word c / 64 =
 * (y[n,h,w,c] > 0) -- what autograd's ReLU backward (nn.ReLU, nets/vgg.py:57, nets/unet.py:14) needs to know about y.
 * b2u_conv_dgrad_bits = b2u_conv_dgrad with one output whose mask is that tensor: 8 bytes per pixel and 64-channel block
 * instead of 128 bytes of y, and the launch tiles like an unmasked one (four stacked M tiles for the 64-channel layers).
 * stat_partial (nullable): per-tile column sums as in b2u_conv_dgrad_stats, rows = b2u_conv_dgrad_stat_rows(masked = 0). */
int b2u_conv_fprop_relu_bits(const void* x0, int C0, const void* x1, int C1, const void* low, const void* wf, const float* bias,
                             void* y, void* up_out, unsigned long long* bits_out, int N, int H, int W, int Cout, int taps,
                             int bn_override, void* stream);
int b2u_conv_dgrad_bits(const void* dz, int Cz, const void* wd, void* dx0, int C0, const unsigned long long* mask_bits,
                        int N, int H, int W, int taps, int bn_override, float* stat_partial, int stat_rows, void* stream);
/* First conv of a decoder stage with the up-sampling and the concat folded into its operand load: replaces
 * self.conv1(torch.cat([inputs1, self.up(inputs2)], 1)) of unetUp.forward (nets/unet.py:16-18; likewise Up.forward of
 * nets/TraditionalUnet.py:36-43) = nn.UpsamplingBilinear2d(scale_factor=2) + torch.cat + nn.Conv2d(k=3,p=1) [+ReLU].
 * skip: [N,H,W,C0]; low: the LOW-RESOLUTION tensor [N,H/2,W/2,C1], interpolated (bilinear, align_corners=True) by producer
 * warps directly into the tensor core's A-operand stage -- neither the concat nor the up-sampled tensor is read from HBM.
 * up_out (nullable): receives the up-sampled tensor [N,H,W,C1] as a by-product (training keeps it as the operand of this
 * conv's weight gradient; inference passes NULL and the tensor never exists).  scale (nullable): folded eval-mode
 * BatchNorm as in b2u_conv_fprop_scaled.  stat_partial/stat_rows (nullable/0): as in b2u_conv_fprop_stats, with the row
 * count of b2u_conv_stat_rows(..., bn_override | 1 << 18): this kernel cuts the image into 8 (w) x 16 (h) pixel tiles (one
 * halo box per channel block serves all nine taps), the plain convs into 16 x 8. */
int b2u_decoder_conv_fprop(const void* skip, int C0, const void* low, int C1, const void* wf, const float* scale,
                           const float* bias, void* y, void* up_out, int N, int H, int W, int Cout, int relu, int bn_override,
                           float* stat_partial, int stat_rows, void* stream);
/* dgrad of the same conv (autograd of nn.Conv2d, utils/utils_fit.py:92): dz has Cz channels; the C0+C1 input-channel
 * gradients go to dx0 / dx1 (dx1 NULL: single input).  mask (NHWC bf16, C0 channels, single output only) applies the
 * ReLU backward of the tensor that fed the conv: dx0 = 0 where mask <= 0. */
int b2u_conv_dgrad(const void* dz, int Cz, const void* wd, void* dx0, int C0, void* dx1, int C1, const void* mask,
                   int N, int H, int W, int taps, int bn_override, void* stream);
/* wgrad: dw (OIHW fp32, overwritten) = sum over pixels of dz (x) cat(x0, x1); db (nullable, [Cout]) = sum over pixels
 * of dz, from the same pass.  first_cin > 0: x0 is the im2col tensor of b2u_im2col_first and dw is
 * [Cout][first_cin][3][3].  flags bit1: never use the swapped-role Cout = 64 kernel (tests); any other bit set returns
 * B2U_ERR_ARG. */
size_t b2u_conv_wgrad_workspace(int N, int H, int W, int Cin_tot, int Cout, int taps);
int b2u_conv_wgrad(const void* x0, int C0, const void* x1, int C1, const void* dz, int Cout, float* dw, float* db, void* ws,
                   size_t ws_bytes, int N, int H, int W, int taps, int first_cin, int flags, void* stream);
/* db[c] = sum over pixels of dz[.,c]  (bias gradient of nn.Conv2d) */
size_t b2u_bias_grad_workspace(int C);
int b2u_bias_grad(const void* dz, float* db, void* ws, size_t ws_bytes, long long P, int C, void* stream);

/* ---- gradient wrt the input image (x.grad of the drop-in modules, autograd of the first layer's nn.Conv2d) ------ */
/* dx (NCHW fp32 [N][Cin][H][W], overwritten) = data gradient of the first 3x3 s1 p1 conv (nets/vgg.py:53,
 * nets/TraditionalUnet.py:9), the one run over b2u_im2col_first rows: dz [N,H,W,Cz] = the gradient wrt its output (ReLU-masked
 * or from the BatchNorm backward), w = its fp32 OIHW weight [Cout][Cin][3][3] (Cout <= Cz, Cz % 16 == 0, 9 Cin <= 64).  The
 * gradient wrt the image is that of the hi columns of the two-term split alone.  Any H, W; dz (and x below) 16-byte aligned
 * (B2U_ERR_ARG otherwise). */
int b2u_first_conv_dgrad_input(const void* dz, int Cz, const float* w, float* dx, int N, int Cin, int H, int W, int Cout,
                               void* stream);
/* the same for the 7x7 s2 p3 ResNet stem (nets/resnet.py:109) run over b2u_im2col_stem rows: dz [N,ceil(H/2),ceil(W/2),Cz],
 * w [Cout][Cin][7][7] (49 Cin <= 192); H, W = the image's */
int b2u_stem_dgrad_input(const void* dz, int Cz, const float* w, float* dx, int N, int Cin, int H, int W, int Cout, void* stream);
/* channels [0, C) of an NHWC tensor [N,H,W,Cpad] -> NCHW fp32 [N][C][H][W]: the gradient wrt an image that entered through
 * b2u_nchw_f32_to_nhwc_bf16_padded (channels [C, 2C) hold the lo half of its split and carry the same gradient) */
int b2u_nhwc_bf16_padded_to_nchw_f32(const void* x, float* y, int N, int C, int H, int W, int Cpad, void* stream);

/* ---- pooling / upsampling ---------------------------------------------------------------------------------- */
/* nn.MaxPool2d(2, 2) (nets/vgg.py:51).  H, W = dims of the un-pooled tensor. */
int b2u_maxpool2x2_fwd(const void* x, void* y, int N, int H, int W, int C, void* stream);
/* dz = (route(dpool to the first max of each window) + dskip) * (y > 0 if relu_mask); dskip may be NULL */
int b2u_maxpool2x2_bwd(const void* dpool, const void* dskip, const void* y, void* dz, int N, int H, int W, int C,
                       int relu_mask, void* stream);
/* nn.UpsamplingBilinear2d(scale_factor=2) = bilinear, align_corners=True (nets/unet.py:13).  H, W = low-res dims. */
int b2u_upsample2x_fwd(const void* x, void* y, int N, int H, int W, int C, void* stream);
/* adjoint; ylow (nullable) = the ReLU output that was upsampled: dlow = 0 where ylow <= 0 */
int b2u_upsample2x_bwd(const void* dup, const void* ylow, void* dlow, int N, int H, int W, int C, void* stream);

/* ---- batch normalisation (nn.BatchNorm2d [+ nn.ReLU], nets/TraditionalUnet.py:9-14, nets/resnet.py:65-71) ---------- */
/* z, y, dy, dz: NHWC bf16 with C channels (C % 8 == 0), P = N*H*W pixels; gamma/beta/running/save: fp32 [C].
 * train: batch statistics (biased variance), running stats updated with `momentum` (unbiased variance), torch semantics. */
size_t b2u_bn_workspace(int C);
/* residual (nullable): y = [relu](bn(z) + residual), the tail of a ResNet bottleneck (nets/resnet.py:92-95) */
int b2u_bn_fwd_train(const void* z, const void* residual, void* y, const float* gamma, const float* beta,
                     float* running_mean, float* running_var, float* save_mean, float* save_invstd, void* ws,
                     size_t ws_bytes, long long P, int C, float eps, float momentum, int relu, void* stream);
int b2u_bn_fwd_train_stats(const void* z, const void* residual, void* y, const float* gamma, const float* beta,
                           float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                           const float* stat_partial, int stat_rows, void* ws, size_t ws_bytes, long long P, int C, float eps,
                           float momentum, int relu, void* stream);
int b2u_bn_fwd_eval(const void* z, const void* residual, void* y, const float* gamma, const float* beta,
                    const float* running_mean, const float* running_var, void* ws, size_t ws_bytes, long long P, int C,
                    float eps, int relu, void* stream);
/* SyncBatchNorm building blocks (nn.SyncBatchNorm.convert_sync_batchnorm, train.py:335-336): the statistics and apply
 * passes as separate calls so the caller can exchange statistics across ranks in between.  Forward: b2u_bn_moments writes
 * this rank's [2][C] fp32 (mean, biased variance); the caller all-gathers them into [world][2][C] and
 * b2u_bn_fwd_train_moments combines them (every rank holds P rows).  Backward: the caller all-reduces the [2][C] sums of
 * b2u_bn_bwd_sums; P_stat = rows over all ranks.  b2u_bn_bwd_sums returns this rank's (dbeta, dgamma), which stay local
 * (DDP averages them), like torch */
int b2u_bn_moments(const void* z, float* moments, void* ws, size_t ws_bytes, long long P, int C, void* stream);
int b2u_bn_fwd_train_moments(const void* z, const void* residual, void* y, const float* gamma, const float* beta,
                             float* running_mean, float* running_var, float* save_mean, float* save_invstd,
                             const float* moments, int world, void* ws, size_t ws_bytes, long long P, int C, float eps,
                             float momentum, int relu, void* stream);
int b2u_bn_bwd_sums(const void* dy, const void* y, const void* z, const float* gamma, const float* beta, const float* save_mean,
                    const float* save_invstd, float* sums, void* ws, size_t ws_bytes, long long P, int C, int relu,
                    void* stream);
int b2u_bn_bwd_apply_sums(const void* dy, const void* y, const void* z, const float* gamma, const float* beta,
                          const float* save_mean, const float* save_invstd, void* dz, void* gout, const float* sums,
                          long long P_stat, void* ws, size_t ws_bytes, long long P, int C, int relu, void* stream);
/* eval-mode conv -> nn.BatchNorm2d (-> ReLU) as ONE kernel: b2u_bn_fold gives scale = gamma / sqrt(rv + eps) and
 * bias = (conv_bias - rm) * scale + beta; b2u_conv_fprop_scaled applies y = [relu](acc * scale + bias) in the conv epilogue
 * (model.eval() inference of the BatchNorm nets: no z tensor, no BatchNorm pass) */
int b2u_bn_fold(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                const float* conv_bias, float* scale, float* bias, int C, float eps, void* stream);
int b2u_conv_fprop_scaled(const void* x0, int C0, const void* x1, int C1, const void* wf, const float* scale, const float* bias,
                          void* y, int N, int H, int W, int Cout, int taps, int relu, int bn_override, void* stream);
/* dy = gradient wrt y; dz (may alias dy) = gradient wrt z; gout (nullable) = ReLU-masked dy = gradient wrt the residual;
 * dgamma/dbeta nullable.  y = the forward output, required only when a residual was added before the ReLU; with
 * y == NULL the ReLU mask is recomputed from z, gamma, beta and the saved statistics exactly as the forward evaluated
 * it (one tensor read less per pass) */
int b2u_bn_bwd(const void* dy, const void* y, const void* z, const float* gamma, const float* beta, const float* save_mean,
               const float* save_invstd, void* dz, void* gout, float* dgamma, float* dbeta, void* ws, size_t ws_bytes,
               long long P, int C, int relu, void* stream);

/* ---- ResNet50 encoder helpers (nets/resnet.py:100-176) ------------------------------------------------------ */
/* 7x7 stride-2 pad-3 stem (nets/resnet.py:109): NCHW fp32 -> im2col rows [N,ceil(H/2),ceil(W/2),192] bf16 */
int b2u_im2col_stem(const float* x_nchw, void* col, int N, int Cin, int H, int W, void* stream);
int b2u_pack_weights_im2col(const float* w_oihw, void* wf, int Cout, int Cin, int taps, int Kpad, void* stream);
/* wgrad of a conv that was run through an im2col tensor: x0 = im2col rows [N,H,W,Kpad], dw = [Cout][cin][taps] */
int b2u_conv_wgrad_im2col(const void* x0, int Kpad, const void* dz, int Cout, float* dw, void* ws, size_t ws_bytes, int N,
                          int H, int W, int cin, int taps, void* stream);
/* stride-2 convs = stride-1 conv + keep even pixels (3x3) / keep even pixels + 1x1 conv (downsample branch) */
int b2u_subsample2(const void* x, void* y, int N, int H, int W, int C, void* stream);
int b2u_zero_insert2(const void* y, void* x, int N, int H, int W, int C, void* stream);
/* nn.MaxPool2d(3, 2, padding=0, ceil_mode=True) (nets/resnet.py:113); H, W = input dims */
int b2u_maxpool3x3s2_fwd(const void* x, void* y, int N, int H, int W, int C, void* stream);
int b2u_maxpool3x3s2_bwd(const void* dy, const void* x, void* dx, int N, int H, int W, int C, void* stream);
/* out = a + b over n bf16 elements (gradient accumulation at tensors with two consumers) */
int b2u_add_bf16(const void* a, const void* b, void* out, long long n, void* stream);
/* out = relu(a + b): the residual join `x += residual; relu(x)` of ResidualBlock (nets/LightWeightUnet.py:52-53);
 * dx = dy * (y > 0): its gradient towards both inputs */
int b2u_add_relu_bf16(const void* a, const void* b, void* out, long long n, void* stream);
int b2u_relu_bwd_bf16(const void* dy, const void* y, void* dx, long long n, void* stream);
/* F.interpolate(x, size=(Ho, Wo), mode="bilinear", align_corners=True) on fp32 NCHW maps and its adjoint: the resize the
 * losses / f_score apply to logits smaller than the labels (nets/unet_training.py:12-13, 24-25, 41-42;
 * utils/utils_metrics.py:15-16).  x: [NC][Hi][Wi], y: [NC][Ho][Wo] */
int b2u_resize_bilinear_f32_fwd(const float* x, float* y, long long NC, int Hi, int Wi, int Ho, int Wo, void* stream);
int b2u_resize_bilinear_f32_bwd(const float* dy, float* dx, long long NC, int Hi, int Wi, int Ho, int Wo, void* stream);

/* ---- depthwise conv, squeeze-excite, per-(image,channel) scaling (Lightweight / UltraLightweight UNets) ---------- */
/* nn.Conv2d(C, C, 3, padding=1, groups=C) (nets/UltraLightweightUnet_large.py:9-10): w fp32 [C][9]; flip=1 uses the
 * taps reversed and is the data gradient */
int b2u_dwconv3x3_fwd(const void* x, const float* w, const float* bias, void* y, int N, int H, int W, int C, int flip,
                      void* stream);
size_t b2u_dwconv3x3_wgrad_workspace(int C);
int b2u_dwconv3x3_wgrad(const void* x, const void* dy, float* dw, float* db, void* ws, size_t ws_bytes, int N, int H, int W,
                        int C, void* stream);
/* out[n][c] = scale * sum over image n's pixels of a (b NULL: AdaptiveAvgPool2d(1) with scale 1/HW) or of a*b */
int b2u_spatial_reduce_workspace_floats(int N, int C);
int b2u_spatial_reduce(const void* a, const void* b, float* out, void* ws, size_t ws_bytes, int N, long long HW, int C,
                       float scale, void* stream);
/* y = x * s[n][c] + a[n][c] (a nullable): SE excitation `x * y` (:52), its backward, nn.Dropout2d masks */
int b2u_scale_nc(const void* x, const float* s, const float* a, void* y, int N, long long HW, int C, void* stream);
/* SE block's Linear-ReLU-Linear-Sigmoid (nets/UltraLightweightUnet_large.py:41-46) and its gradients */
int b2u_se_fc_fwd(const float* pooled, const float* w1, const float* b1, const float* w2, const float* b2, float* hidden,
                  float* scale, int N, int C, int Cp, int R, void* stream);
int b2u_se_fc_bwd(const float* dscale, const float* pooled, const float* hidden, const float* scale, const float* w1,
                  const float* w2, float* dpooled, float* dw1, float* db1, float* dw2, float* db2, float* scratch, int N,
                  int C, int Cp, int R, float dp_scale, void* stream);

/* ---- classifier head (nn.Conv2d(64, num_classes, 1), nets/unet.py:58,76), 1 <= ncls <= 255 ------------------ */
int b2u_head_fwd(const void* x, const float* w, const float* b, float* logits_nchw, int N, int H, int W, int Cin,
                 int ncls, void* stream);
/* workspace bytes of b2u_head_bwd for ncls classes; b2u_head_bwd_workspace() = the size for up to 32 classes */
size_t b2u_head_bwd_workspace_cls(int ncls);
size_t b2u_head_bwd_workspace(void);
int b2u_head_bwd(const float* dlogits_nchw, const void* x, const float* w, void* dx, float* dw, float* db, void* ws,
                 size_t ws_bytes, int N, int H, int W, int Cin, int ncls, int relu_mask, void* stream);

/* ---- losses and metrics ------------------------------------------------------------------------------------ */
/* CE_Loss / Focal_Loss / Dice_loss (nets/unet_training.py:9-56) and f_score (utils/utils_metrics.py:12-31) in one
 * pass.  out (device, b2u_loss_out_len(C) floats): [0] CE, [1] Focal, [2] Dice loss, [3] f_score, then backward
 * coefficients.  target: int64 [N,H,W]; onehot (nullable): fp32 [N,H,W,C+1].  1 <= C <= 255. */
size_t b2u_loss_workspace(int C);
int b2u_loss_out_len(int C);
int b2u_loss_fwd(const float* logits, const long long* target, const float* onehot, const float* cls_w, float* out,
                 double* stats, void* ws, size_t ws_bytes, int N, int C, int H, int W, float beta, float smooth,
                 float focal_alpha, float focal_gamma, float thr, void* stream);
/* dlogits = gscale[0] dCE + gscale[1] dFocal + gscale[2] dDice (gscale: 3 floats on device).
 * out_mode 0: fp32 NCHW (autograd of the drop-in losses); 1: bf16 NHWC [N,H,W,64 G], G = ceil(C / 32) groups, group g =
 * [hi(32) | lo(32)] two-term bf16 split of the dlogits of classes 32g .. 32g + 31 (classes >= C zero), the dz operand of
 * b2u_conv_dgrad / b2u_conv_wgrad (taps = 1) for the head's backward on the tensor cores (both halves meet the same
 * weights, see b2u_pack_head_dgrad). */
int b2u_loss_bwd(const float* logits, const long long* target, const float* onehot, const float* cls_w, const float* fin,
                 const float* gscale, void* dlogits, int out_mode, int N, int C, int H, int W, float focal_alpha,
                 float focal_gamma, void* stream);
/* final.weight [C][64] fp32 -> [64][64 G] bf16 dgrad operand wd[ci][co]: columns 64g + r, r in [0,32) and [32,64), both
 * = class 32g + r % 32 (zero past C) */
int b2u_pack_head_dgrad(const float* w, void* wd, int ncls, void* stream);
/* the same 1x1 classifier forward on the tensor cores: wf = bf16 [64 G][64] from b2u_pack_head_fprop (in group g, rows
 * 64g + [0,32) = bf16(W), rows 64g + [32,64) = bf16(W - bf16(W)) of classes 32g..; the epilogue adds the halves), fp32
 * NCHW logits written directly; bias: [ncls] */
int b2u_pack_head_fprop(const float* w, void* wf, int ncls, void* stream);
int b2u_head_fwd_tc(const void* x, const void* wf, const float* bias, float* logits, int N, int H, int W, int ncls,
                    void* stream);
/* per-pixel class decision of the inference loop (unet.py:246-250: argmax(softmax(z)) == argmax(z)) */
int b2u_argmax_u8(const float* logits, unsigned char* mask, int N, int C, int H, int W, void* stream);
/* the predictor's tail (unet.py:135-148, 324-340): softmax, crop of the letterbox bars (cy, cx, ch, cw), cv2.resize(...,
 * INTER_LINEAR) of the probabilities to oh x ow, argmax -> uint8 mask [N][oh][ow]; nothing but the mask leaves the GPU */
int b2u_softmax_resize_argmax_u8(const float* logits, unsigned char* mask, int N, int C, int H, int W, int cy, int cx,
                                 int ch, int cw, int oh, int ow, void* stream);
/* the same tail for a batch whose images have their own crop and original size: logits [count][C][H][W]; items = count x
 * {int cy, cx, ch, cw, oh, ow; int64 mask_off} (32 B each) in DEVICE memory, every crop inside H x W; image i's mask
 * [oh][ow] goes to masks + mask_off (16-byte aligned offsets let the masks go straight to b2u_fast_hist_batch);
 * max_oh, max_ow: the largest oh, ow of the batch.  Each pixel's class equals b2u_softmax_resize_argmax_u8's. */
int b2u_softmax_resize_argmax_u8_batch(const float* logits, const void* items, int count, int C, int H, int W,
                                       unsigned char* masks, int max_oh, int max_ow, void* stream);
/* detect_image's rendering (unet.py:150-203) for a batch: items = count x {const uint8* src ([ih][iw][3] RGB); const uint8*
 * mask ([ih][iw], from the batched tail); int64 out_off; int ih, iw} (32 B each) in DEVICE memory; palette: [C][3] uint8,
 * device.  mix_type 0 writes Image.blend(src, palette[mask], 0.7) (Pillow's float32 arithmetic without FMA, truncated),
 * 1 palette[mask], 2 src where mask != 0 else 0, each to out + out_off as [ih][iw][3]; -1 writes no image (out, palette may
 * be NULL).  counts (nullable): [count][C] uint64, cleared by the call, then the per-image pixel count of each class.
 * max_pixels: the largest ih * iw of the batch; 1 <= C <= 255.  One kernel launch per batch. */
int b2u_render_batch(const void* items, int count, const unsigned char* palette, int C, int mix_type, unsigned char* out,
                     unsigned long long* counts, long long max_pixels, void* stream);
/* fast_hist (utils/utils_metrics.py:34-43): hist (n*n+1 uint64, accumulated) ; dtype 0=u8 1=i32 2=i64; 1 <= n <= 256 */
int b2u_fast_hist(const void* a, const void* b, long long len, int n, int dtype, unsigned long long* hist, void* stream);
/* compute_mIoU's loop over an evaluation set (utils/utils_metrics.py:74-95) in ONE launch: items = count x {const uint8* a;
 * const uint8* b; int64 len; int64 first_chunk} (32 B each) in DEVICE memory, every pointer 16-byte aligned; first_chunk = running
 * sum of b2u_fast_hist_chunks(len) over the previous items, total_chunks = the sum over all of them; hist as above */
int b2u_fast_hist_batch(const void* items, int count, long long total_chunks, int n, unsigned long long* hist, void* stream);
long long b2u_fast_hist_chunks(long long len);
/* get_miou.py:45-65 without the mask round trip: pred = argmax_c logits (fp32 NCHW; lowest index on ties, unet.py:246-250),
 * optionally stored as a uint8 mask [N][H][W], and (gt, pred) counted into hist (n*n+1 uint64, accumulated) in the same pass;
 * gt: uint8 [N][H][W] (values >= n ignored, 1 <= n <= 256) or NULL (mask only); H*W %% 4 == 0 */
int b2u_argmax_hist(const float* logits, const unsigned char* gt, unsigned char* pred, int N, int C, int H, int W, int n,
                    unsigned long long* hist, void* stream);

/* ---- optimizer (torch.optim.Adam / SGD step of train.py:402-405 on flat fp32 buffers) ----------------------- */
int b2u_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int step, float grad_scale, void* stream);
int b2u_sgd_step(float* param, const float* grad, float* momentum_buf, long long n, float lr, float momentum,
                 float weight_decay, int nesterov, int first_step, float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2U_H_ */
