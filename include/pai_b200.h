/* pai_b200 -- C-ABI of the B200-native Pix2Pix / PatchGAN / SSIM-PSNR hot path.
 *
 * The reference (cristianpjensen/thesis-pai-reconstruction) is pure Python/PyTorch and has no
 * FFI of its own; every entry point below names the reference call site whose arithmetic it
 * replaces.  The host side (thesis-pai-reconstruction_b200/pai_b200/lib.py) binds these with
 * ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch); the library allocates
 *     nothing persistent and never synchronises the stream
 *   - activations / gradients: NHWC bf16, `ld` = elements between consecutive pixels (>= channels,
 *     so a tensor may be a channel slice of a wider concat buffer)
 *   - `stream` is a cudaStream_t passed as void*
 *   - return 0 on success, negative on error; pai_last_error() describes the last failure of the
 *     calling thread.  There is no CPU fallback anywhere.
 */
#ifndef PAI_B200_H
#define PAI_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define PAI_ACT_NONE 0
#define PAI_ACT_LEAKY 1 /* LeakyReLU(slope) */
#define PAI_ACT_RELU 2
#define PAI_ACT_TANH 3

#define PAI_DTYPE_F32 0
#define PAI_DTYPE_BF16 1

const char* pai_last_error(void);
int pai_version(void);
/* The tensor-core kernels are persistent: one CTA (195 KB of shared memory) per SM.  A collective that must run
 * CONCURRENTLY with them (the NCCL gradient all-reduce overlapped with the backward pass, pai_b200/dp.py; Lightning DDP's
 * bucketed overlap for main.py:123-135) needs SMs of its own, or its CTAs and ours wait for each other for the whole
 * duration of a kernel.  pai_reserve_sms(n) makes every persistent launch of this process use (#SMs - n) CTAs. */
int pai_reserve_sms(int n);

/* ---------------------------------------------------------------------------------------------
 * 4x4 convolutions as tcgen05 implicit GEMM.
 *
 * pai_conv4x4_fprop: nn.Conv2d(cin, cout, kernel_size=4, stride=stride, padding=1)
 *   (models/pix2pix.py:63-69,141-147 stride 2; models/wrapper.py:196-203,229-233 stride 2 and 1)
 *     y[n,oh,ow,co] = act(bias[co] + sum_{ky,kx,ci} x[n, stride*oh-1+ky, stride*ow-1+kx, ci] * W[co,ci,ky,kx])
 *   x: [n,h,w,cin] bf16, cin % 64 == 0; stride 2 needs x_ld == cin and even h, w.
 *   w_packed: bf16 [cout_pad][16*cin], w_packed[co][(ky*4+kx)*cin + ci] = W[co,ci,ky,kx];
 *             rows cout..cout_pad-1 zero, cout_pad % n_tile == 0.
 *   y: [n,ho,wo,*] (ho = h/2 | h-1), bf16 or fp32 (y_f32), pixel stride y_ld.
 *   splitk_ws: NULL, or a ZEROED fp32 buffer of n*ho*wo*cout elements.  When given and the layer has too few
 *             output tiles to occupy the GPU (the <= 8x8 U-Net levels), the K loop is split over SMs, partial
 *             sums meet in the workspace and a second small kernel applies bias/activation into y.
 *   The same routine is the data-gradient of ConvTranspose2d(4,2,1) (models/pix2pix.py:99-105) when
 *   fed dL/dy and the ConvT weight [Cin_T,Cout_T,4,4] read as a Conv weight [out=Cin_T, in=Cout_T].
 */
int pai_conv4x4_fprop(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                      int cout_pad, int stride, const float* bias, int act, float slope, void* y, int y_ld,
                      int y_f32, int n_tile, float* splitk_ws, void* stream);

/* The same convolution with TWO bf16 outputs of the same accumulator, each with its own activation and pixel stride
 * (cout %% 64 == 0, no split-K): eval-mode encoder blocks whose BatchNorm is folded into the weights write the next
 * encoder's LeakyReLU input AND the decoder's ReLU concat slot (models/pix2pix.py:62,98,212) from one GEMM. */
int pai_conv4x4_fprop_dual(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                           int cout_pad, int stride, const float* bias, int act, float slope, void* y, int y_ld, void* y2,
                           int y2_ld, int act2, int n_tile, void* stream);

/* pai_convT4x4s2_fprop: nn.ConvTranspose2d(cin, cout, kernel_size=4, stride=2, padding=1)
 *   (models/pix2pix.py:99-105,186-192), run as 4 sub-pixel phases:
 *     y[n,2a+py,2b+px,co] = act(bias[co] + sum_ci sum_{(ky,dy) in T[py]} sum_{(kx,dx) in T[px]}
 *                               x[n,a+dy,b+dx,ci] * W[ci,co,ky,kx]),  T[0]={(1,0),(3,-1)}, T[1]={(0,+1),(2,0)}
 *   w_packed: bf16 [4][cout_pad][4*cin]: w_packed[py*2+px][co][(ty*2+tx)*cin+ci] = W[ci,co,T[py][ty].k,T[px][tx].k]
 *   Also the data-gradient of Conv2d(4,2,1) when fed dL/dy and the Conv weight [Cout,Cin,4,4]
 *   read as a ConvT weight [in=Cout, out=Cin].
 */
int pai_convT4x4s2_fprop(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                         int cout_pad, const float* bias, int act, float slope, void* y, int y_ld, int y_f32,
                         int n_tile, float* splitk_ws, void* stream);
/* BatchNorm statistics from the GEMM epilogue ("BN fused into the epilogue" of the north star): the convolution writes
 * its raw bf16 output (+bias, no activation) AND every CTA adds the per-channel sum / sum of squares of the values it
 * stores to its own row of bn_partials [bn_rows >= #SMs][2*cout] (fp32, zeroed by the caller) -- the separate
 * statistics pass over the output (pai_bn_stats) disappears.  Needs cout %% 64 == 0 and a layer large enough not to be
 * split along K (more than 74 * 128 output pixels); otherwise an error is returned and nothing is launched. */
int pai_conv4x4_fprop_bnstats(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                              int cout_pad, int stride, const float* bias, void* y, int y_ld, int n_tile,
                              float* bn_partials, int bn_rows, void* stream);
int pai_convT4x4s2_fprop_bnstats(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                                 int cout_pad, const float* bias, void* y, int y_ld, int n_tile, float* bn_partials,
                                 int bn_rows, void* stream);
/* Data gradient of a stride-2 4x4 Conv2d FUSED with the activation backward of the layer below it (PatchGAN blocks,
 * models/wrapper.py:196-206: Conv -> LeakyReLU):  gx = convT(gy, w) * act'(saved_act)  where saved_act [n, 2h, 2w, cin] is
 * the stored LeakyReLU / ReLU output of the layer below (its sign is the sign of the pre-activation; slope = 0 for ReLU),
 * laid out exactly like gx (same gx_ld).  colsum_partials (optional, [rows >= #SMs][2*cin] fp32, zeroed by the caller)
 * receives per-CTA partial column sums of gx in its first cin entries per row = the bias gradient of the layer below.
 * Replaces pai_convT4x4s2_fprop + pai_act_bwd (one write and two reads of the gradient tensor less). */
int pai_conv4x4_dgrad_act(const void* gy, int n, int h, int w, int cout, int gy_ld, const void* w_packed_dgrad, int cin,
                          int cin_pad, const void* saved_act, float slope, void* gx, int gx_ld, int n_tile,
                          float* colsum_partials, int rows, void* stream);

/* Weight gradients (autograd of the two modules above; SURVEY.md Appendix B).
 * pai_conv4x4_wgrad:   dw[ky*4+kx][co][ci] += sum_{n,oh,ow} gy[n,oh,ow,co] * x[n,stride*oh-1+ky,stride*ow-1+kx,ci]
 * pai_convT4x4s2_wgrad: dw[ky*4+kx][ci][co] += sum_{n,a,b} x[n,a,b,ci] * gy[n,2a-1+ky,2b-1+kx,co]
 *   dw is fp32 and is ACCUMULATED into (zero it first); channel counts: both % 64 == 0.  x: [n,h,w,cin]; gy: the module's output gradient.
 */
int pai_conv4x4_wgrad(const void* x, int n, int h, int w, int cin, int x_ld, const void* gy, int cout, int gy_ld,
                      int stride, float* dw, int splitk, void* stream);
int pai_convT4x4s2_wgrad(const void* x, int n, int h, int w, int cin, int x_ld, const void* gy, int cout, int gy_ld,
                         float* dw, int splitk, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SSIM / PSNR / MSE metric and loss path (torchmetrics==0.11.4 functionals as bound by
 * models/utils.py:38-47 with data_range=1.0; callers models/wrapper.py:53-63,150-156,166-173 and
 * report.py:78-96,146,188-217).  11x11 Gaussian window (sigma 1.5), c1=1e-4, c2=9e-4, reflect pad 5.
 *
 * pai_ssim_psnr_fwd: pred/target are [n,h,w] single-channel planes (dtype PAI_DTYPE_F32|BF16);
 *   denormalize != 0 applies models/utils.py:11 clamp(0.5*x+0.5, 0, 1) to both on load.
 *   ssim_sum[n]   = sum of the SSIM map over rows/cols 5..dim-6 (per-image SSIM = / ((h-10)*(w-10)))
 *   band_sum[n,16] (nullable) = per depth band d, the sum over rows d*h/16+5 .. (d+1)*h/16-6, cols 5..w-6
 *                   (report.py:188-217 depth_ssim = / ((h/16-10)*(w-10)))
 *   sse[n]        = sum (p-t)^2  (PSNR = 10 log10(numel/sse), MSE = sse/numel, RMSE = sqrt)
 *   full_map[n,h,w] (nullable) = the reflect-padded SSIM image of return_full_image=True.
 * pai_ssim_psnr_bwd: grad_pred[n,h,w] (same dtype as pred) = d/dpred of
 *   sum_i g_ssim_sum[i]*ssim_sum[i] + g_sse[i]*sse[i]  (g_sse nullable), chained through the
 *   de-normalisation when denormalize != 0.  workspace: pai_ssim_bwd_workspace_bytes(n,h,w) bytes.
 */
int pai_ssim_psnr_fwd(const void* pred, const void* target, int dtype, int n, int h, int w, int denormalize,
                      float* ssim_sum, float* band_sum, float* sse, float* full_map, void* stream);
int pai_ssim_psnr_bwd(const void* pred, const void* target, int dtype, int n, int h, int w, int denormalize,
                      const float* g_ssim_sum, const float* g_sse, void* workspace, void* grad_pred, void* stream);
long long pai_ssim_bwd_workspace_bytes(int n, int h, int w);

/* ---------------------------------------------------------------------------------------------
 * BatchNorm2d (eps, momentum; models/pix2pix.py:70,106) split around the convolution kernels, the
 * non-inplace pre-activations LeakyReLU(0.2)/ReLU (models/pix2pix.py:62,98) and the zero-copy skip
 * concat (models/pix2pix.py:212).  x: [m pixels][c] bf16, `ld` elements between pixels.
 *   pai_bn_stats      sums[0:c] = sum_x, sums[c:2c] = sum_x^2 (fp32; zeroed by the call)
 *   pai_bn_finalize   training: batch mean / biased var from sums, running stats updated with
 *                     `momentum` and the unbiased variance; eval: running stats are used.
 *                     scale_shift[4c] = [gamma*invstd | beta - mean*gamma*invstd | mean | invstd]
 *   pai_bn_apply_act  out1 = act1(scale*x + shift) and optionally out2 = act2(...) (each may be a
 *                     channel slot of a wider buffer); scale_shift NULL = identity
 *   pai_bn_bwd_reduce dz = g1*act1'(z) + g2*act2'(z) (g2 nullable), z = scale*x + shift;
 *                     sums[0:c] = sum dz (= dbeta), sums[c:2c] = sum dz*xhat (= dgamma)
 *   pai_bn_bwd_apply  dx = gamma*invstd*(dz - mean(dz) - xhat*mean(dz*xhat)); scale_shift NULL = no
 *                     normalisation (dx = dz: plain activation backward, sums[0:c] of the reduce = dbias)
 *   pai_act_bwd       layers without BatchNorm (enc0, bottleneck, PatchGAN blocks): dx = dz and
 *                     sums2c[0:c] = sum dz (= dbias) in ONE pass; x only supplies the sign of the pre-activation
 *   pai_colsum        sums2c[0:c] = column sums of x (bias gradients); sums2c[c:2c] is scratch
 */
int pai_bn_stats(const void* x, long long m, int c, int ld, float* sums, void* stream);
int pai_bn_finalize(const float* sums, long long m, int c, const float* gamma, const float* beta, float eps,
                    float momentum, int training, float* running_mean, float* running_var, float* scale_shift,
                    void* stream);
/* The same from `nparts` rows of partial sums [nparts][2*c] (summed first): the per-CTA rows written by
 * pai_conv4x4_fprop_bnstats / pai_convT4x4s2_fprop_bnstats. */
int pai_bn_finalize_partials(const float* sums, int nparts, long long m, int c, const float* gamma, const float* beta,
                             float eps, float momentum, int training, float* running_mean, float* running_var,
                             float* scale_shift, void* stream);
int pai_bn_apply_act(const void* x, long long m, int c, int ld, const float* scale_shift, void* out1, int ld1,
                     int act1, void* out2, int ld2, int act2, float slope, void* stream);
int pai_bn_bwd_reduce(const void* x, long long m, int c, int ld, const float* scale_shift, const void* g1, int ldg1,
                      int act1, const void* g2, int ldg2, int act2, float slope, float* sums, void* stream);
int pai_bn_bwd_apply(const void* x, long long m, int c, int ld, const float* scale_shift, const void* g1, int ldg1,
                     int act1, const void* g2, int ldg2, int act2, float slope, const float* sums,
                     const float* gamma, void* dx, int lddx, void* stream);
int pai_act_bwd(const void* x, long long m, int c, int ld, const void* g1, int ldg1, int act1, const void* g2, int ldg2,
                int act2, float slope, float* sums2c, void* dx, int lddx, void* stream);
int pai_colsum(const void* x, long long m, int c, int ld, float* sums2c, void* stream);
/* Small layers (the <= 8x8 levels: m * 16 B per operand must fit 200 KB of shared memory, pai_bn_small_ok): one block
 * per 8 channels holds its slice of ALL pixels, so the whole training-mode BatchNorm is one launch.
 *   pai_bn_small_fwd  = pai_bn_stats + pai_bn_finalize (running statistics, scale_shift[4c]) + pai_bn_apply_act, and
 *                       the Dropout2d scaling of models/pix2pix.py:107 on out1 when `mask` [n][c] (fp32, 0 or 1/(1-p))
 *                       is given (pixels_per_image = h*w of the layer)
 *   pai_bn_small_bwd  = pai_scale_channels (Dropout2d backward on g1, when `mask` is given) + pai_bn_bwd_reduce +
 *                       pai_bn_bwd_apply; sums[2c] as in pai_bn_bwd_reduce (plain 2c floats, written not accumulated)
 *   operands of pai_bn_small_ok: 1 for fwd, 2 (+1 with g2) for bwd */
int pai_bn_small_ok(long long m, int c, int operands);
int pai_bn_small_fwd(const void* x, long long m, int c, int ld, const float* gamma, const float* beta, float eps,
                     float momentum, float* running_mean, float* running_var, float* scale_shift, void* out1, int ld1,
                     int act1, void* out2, int ld2, int act2, float slope, const float* mask, int pixels_per_image,
                     void* stream);
int pai_bn_small_bwd(const void* x, long long m, int c, int ld, const float* scale_shift, const void* g1, int ldg1,
                     int act1, const void* g2, int ldg2, int act2, float slope, const float* mask, int pixels_per_image,
                     const float* gamma, float* sums, void* dx, int lddx, void* stream);

/* ---------------------------------------------------------------------------------------------
 * The four degenerate (1- or 2-channel-wide, HBM-bound) layers: enc0 Conv2d(1,64,4,2,1)
 * (models/pix2pix.py:141-147), D0 Conv2d(2,64,4,2,1) on cat([x,y],1) (models/wrapper.py:229,237),
 * dec7 ConvTranspose2d(128,1,4,2,1) (models/pix2pix.py:186-192) and D4 Conv2d(512,1,4,1,1)
 * (models/wrapper.py:233).  Planes are single-channel fp32 [n,ih,iw]; the wide operand is NHWC bf16
 * on the [n,oh,ow] grid; (dy,dx) of tap t=(ky,kx) is (ky-1,kx-1), or (1-ky,1-kx) when flip.
 *   pai_smallc_conv_fprop  out[n,oy,ox,c] = act(bias[c] + sum_{t,j} plane_j[n,s*oy+dy,s*ox+dx] * w[c][t][j])
 *                          (enc0 / D0 forward; dec7 and D4 data gradients)
 *   pai_smallc_conv_wgrad  dw[c][t][j] += sum_{n,y,x} a[n,y,x,c] * plane_j[n,s*y+dy,s*x+dx]   (dw fp32, accumulated)
 */
int pai_smallc_conv_fprop(const float* plane0, const float* plane1, int cin, int n, int ih, int iw, int oh, int ow,
                          int stride, int flip, const float* w, const float* bias, int c, void* out1, int ld1,
                          int act1, void* out2, int ld2, int act2, float slope, void* stream);
int pai_smallc_conv_wgrad(const void* a, int lda, int c, const float* plane0, const float* plane1, int cin, int n,
                          int ih, int iw, int oh, int ow, int stride, int flip, float* dw, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Degenerate layers as tensor-core GEMMs.  A convolution whose input (enc0, D0) or output (dec7, D0's
 * data gradient) is 1-2 channels wide becomes  im2col / col2im of the thin side  +  a pointwise GEMM:
 *   pai_im2col4x4      col[n,oy,ox, t*cin+j] = plane_j[n, s*oy+dy_t, s*ox+dx_t] (bf16 rows of 64 channels; only the first
 *                      16*cin are written -- consumers pass k_valid = 16*cin / ignore the other wgrad columns)
 *   pai_pointwise_gemm y[r, co] = act(bias[co] + sum_ci x[r, ci] * w_packed[co][ci])  (1x1 conv over m rows;
 *                      k_valid > 0 (cin == 64 only): just the first k_valid columns of x hold data (pai_im2col4x4
 *                      output), the rest is never read by the tensor core and may be uninitialised;
 *                      optional second bf16 output y2 with its own activation; m % 128 == 0)
 *   pai_pointwise_wgrad dw[cu][cs] += sum_r u[r, cu] * s[r, cs]                         (m % 64 == 0)
 *   pai_col2im4x4s2    out[n,2a+py,2b+px] = act(bias + sum of the 4 (tap, neighbour) partial products of
 *                      p[n,h,w,16])  -- the transposed 4x4 stride-2 conv with one output channel.
 */
int pai_im2col4x4(const float* plane0, const float* plane1, int cin, int n, int ih, int iw, int oh, int ow, int stride,
                  int flip, void* col, void* stream);
int pai_pointwise_gemm(const void* x, long long m, int cin, int x_ld, const void* w_packed, int cout, int cout_pad,
                       const float* bias, int act, float slope, void* y, int y_ld, int y_f32, void* y2, int y2_ld,
                       int act2, int n_tile, int k_valid, void* stream);
int pai_pointwise_wgrad(const void* u, long long m, int cu, int u_ld, const void* s, int cs, int s_ld, float* dw,
                        int splitk, void* stream);
int pai_col2im4x4s2(const float* p, int ldp, int n, int h, int w, const float* bias, int act, float* out,
                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * The same degenerate layers as SINGLE-PASS tcgen05 kernels (csrc/thin.cu): the thin operand of the GEMM is built in
 * shared memory by the CTA itself, so no im2col / col2im carrier ever exists in HBM and the wide tensor is read or
 * written exactly once (these layers are HBM-bound).
 *   pai_thin_conv4x4s2_fprop   Conv2d(cin in {1,2}, cout, 4, 2, 1) from fp32 planes [n,ih,iw] (enc0 models/pix2pix.py:141-147,
 *                              D0 on cat([x,y]) models/wrapper.py:229,237; also the data gradient of dec7
 *                              ConvTranspose2d(C,1,4,2,1) models/pix2pix.py:186-192 fed the output-gradient plane):
 *                              out[n,oy,ox,co] = act(bias[co] + sum_{t,j} plane_j[n,2oy-1+ky,2ox-1+kx] * w_packed[co][t*cin+j])
 *                              w_packed bf16 [cout][64] (zero padded columns), cout in {64,128,192,256}; optional second
 *                              bf16 output with its own activation / pixel stride.
 *   pai_thin_conv4x4s2_wgrad   dw[c][t*cin+j] += sum_pix u[pix,c] * plane_j[n,2oy-1+ky,2ox-1+kx]   (dw fp32 [c][16*cin], zeroed by
 *                              the caller; c in {64,128}; iw %% 128 == 0): weight gradients of enc0 / D0 (u = dL/d pre-activation)
 *                              and of dec7 (u = its input, plane = output gradient).
 *   pai_thin_convT4x4s2_plane  ConvTranspose2d(c, 1, 4, 2, 1) (+bias, optional Tanh) from NHWC bf16 [n,h,128,c] to an fp32 plane
 *                              [n,2h,256] (dec7 forward models/pix2pix.py:186-195; data gradient of D0 w.r.t. one input plane):
 *                              w_taps bf16 [16][c], w_taps[ky*4+kx][ci] = W[ci,0,ky,kx]; rows are streamed once.
 *   pai_col2im4x4s1            out[n,oy,ox] = sum_{ky,kx} p[n,oy-1+ky,ox-1+kx, ky*4+kx] over an [n,h,w,ldp] fp32 tensor of per-tap
 *                              partial products -> [n,h-1,w-1]: the PatchGAN head Conv2d(512,1,4,1,1) (models/wrapper.py:233)
 *                              after ONE pointwise GEMM over its input instead of 16 shifted ones.
 */
int pai_thin_conv4x4s2_fprop(const float* plane0, const float* plane1, int cin, int n, int ih, int iw,
                             const void* w_packed, int cout, const float* bias, void* out1, int ld1, int act1, void* out2,
                             int ld2, int act2, float slope, void* stream);
int pai_thin_conv4x4s2_wgrad(const void* u, int u_ld, int c, const float* plane0, const float* plane1, int cin, int n,
                             int ih, int iw, float* dw, void* stream);
int pai_thin_convT4x4s2_plane(const void* x, int n, int h, int w, int c, int x_ld, const void* w_taps, const float* bias,
                              int act, float* out, void* stream);
int pai_col2im4x4s1(const float* p, int ldp, int n, int h, int w, float* out, void* stream);

/* report.py's image outputs on the device (report.py:122-141,220-233):
 *   pai_to_uint8   torchvision ConvertImageDtype(torch.uint8) (models/utils.py:12): (x * 255.999) truncated; values outside
 *                  [0, 1] wrap modulo 256 like the float -> int32 -> uint8 conversion of the x86 host the reference runs on
 *   pai_afmhot_u8  matplotlib's "afmhot" colormap (r, g, b = clip(2v, 2v - 0.5, 2v - 1)) with its 256-entry look-up
 *                  (index = min(int(x * 256), 255), entry i evaluated at v = i / 255) followed by pai_to_uint8:
 *                  img [n, h*w] in [0, 1] -> out [n, 3, h*w] uint8 */
int pai_to_uint8(const float* x, long long count, unsigned char* out, void* stream);
int pai_afmhot_u8(const float* img, int n, long long hw, unsigned char* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optimizer step: torch.optim.Adam(lr=2e-4, betas=(0.5,0.999), eps=1e-7) of
 * UnetWrapper.configure_optimizers / training_step (models/wrapper.py:97-115,136,160), fused with
 * the bf16 operand repack of the implicit-GEMM kernels.  step_size = lr / (1 - beta1^t),
 * inv_bias_correction2_sqrt = 1 / sqrt(1 - beta2^t); parameters, gradients and moments are fp32.
 *   pai_adam_pack_conv4x4  w [a, b, 4, 4] (Conv2d: a = Cout, b = Cin; ConvTranspose2d: a = Cin, b = Cout):
 *                          Adam update in place (skipped when grad == NULL: pack only), then
 *                          pack1[a, (ky*4+kx)*b + b'] and pack2[py*2+px, b', (ty*2+tx)*a + a'] (either may
 *                          be NULL; pack2 has b_pad rows per phase; padding rows are left untouched)
 *   pai_adam_pack_conv4x4_multi  the same for `count` weights in ONE launch (host arrays, one entry per weight;
 *                          grads are required): a launch per weight keeps every small layer at the latency of one
 *                          thread block
 *   pai_adam_multi         the same update for `count` small dense tensors in one launch (host arrays of
 *                          device pointers)
 *   pai_adam_prepare       device-side step counter for CUDA-graph capture of the training step: ++*step and
 *                          dyn[0..1] = {lr / (1 - beta1^t), 1 / sqrt(1 - beta2^t)} (double arithmetic).  When the
 *                          `dyn` argument of the two update functions is non-NULL they read these two scalars from
 *                          the device instead of their step_size / inv_bias_correction2_sqrt arguments.
 */
int pai_adam_pack_conv4x4(float* w, const float* grad, float* exp_avg, float* exp_avg_sq, int a, int b, float beta1,
                          float beta2, float step_size, float inv_bias_correction2_sqrt, float eps, void* pack1,
                          void* pack2, int b_pad, const float* dyn, void* stream);
int pai_adam_pack_conv4x4_multi(int count, float* const* ws, const float* const* grads, float* const* exp_avgs,
                                float* const* exp_avg_sqs, const int* as, const int* bs, void* const* pack1s,
                                void* const* pack2s, const int* b_pads, float beta1, float beta2, float step_size,
                                float inv_bias_correction2_sqrt, float eps, const float* dyn, void* stream);
int pai_adam_multi(int count, float* const* params, const float* const* grads, float* const* exp_avgs,
                   float* const* exp_avg_sqs, const int* numels, float beta1, float beta2, float step_size,
                   float inv_bias_correction2_sqrt, float eps, const float* dyn, void* stream);
int pai_adam_prepare(int* step, float lr, float beta1, float beta2, float* dyn, void* stream);
/* Exponential moving average of the weights (callbacks/ema.py:24-34, torch_ema's rule, decay 0.9999 main.py:131):
 * shadow_k <- shadow_k - one_minus_decay * (shadow_k - param_k) for `count` fp32 tensors in one launch (host arrays of
 * device pointers; 12 B per parameter instead of three elementwise passes per tensor). */
int pai_ema_multi(int count, float* const* shadows, const float* const* params, const int* numels, float one_minus_decay,
                  void* stream);
/* Weight gradient from the wgrad kernels' accumulation layout dw[16][ab] (tap-major, ab = A*B) to the parameter layout
 * grad[ab][16] (= [A, B, 4, 4], models/pix2pix.py:63,99); zero_src != 0 also zeroes dw for the next accumulation. */
int pai_wgrad_finish(float* dw_tap_major, long long ab, float* grad, int zero_src, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Layers of the Residual / Attention / Trans U-Net variants (models/res_unet.py, attention_unet.py,
 * trans_unet.py).  Dense 3x3 and 1x1 convolutions run on the implicit-GEMM kernels:
 *   pai_conv3x3_fprop   nn.Conv2d(cin, cout, 3, padding=1): y[n,oy,ox,co] = act(bias[co] + sum x[n,oy-1+ky,ox-1+kx,ci] *
 *                       W[co,ci,ky,kx]); w_packed bf16 [cout_pad][9*cin], w_packed[co][(ky*3+kx)*cin+ci].  Its data
 *                       gradient is the same routine on dL/dy with w_packed[ci][((2-ky)*3+(2-kx))*cout+co].
 *   pai_conv3x3_wgrad   dw[ky*3+kx][co][ci] += sum gy[n,oy,ox,co] * x[n,oy-1+ky,ox-1+kx,ci]   (fp32, accumulated)
 *   (1x1 convolutions are pai_pointwise_gemm / pai_pointwise_wgrad.)
 * The rest are HBM-bound streams over NHWC bf16 tensors (c % 8 == 0); 1-channel tensors are fp32 planes:
 *   pai_maxpool2_fwd/bwd      nn.MaxPool2d(2); the gradient goes to the first maximum of the window
 *   pai_upsample2_fwd/bwd     nn.Upsample(scale_factor=2) (nearest); the gradient sums the 2x2 block
 *   pai_add_act               out = act(a + b) (b nullable)                (residual add; its backward is pai_act_bwd)
 *   pai_scale_rows_fwd/bwd    out[p,:] = act(x[p,:] * s[p]);  gx = g*act'*s,  gs[p] = sum_c g*act'*x   (x * attention)
 *   pai_conv_plane_to_wide    out[p,c] = act(bias[c] + sum_t plane[p+off_t] * w[c][t]), k x k taps, off_t = (ky-pad, kx-pad),
 *                             negated when flip (Conv2d(1,C,k) forward; data gradient of Conv2d(C,1,k))
 *   pai_conv_wide_to_plane    out[p] = act(bias + sum_t sum_c x[p+off_t,c] * w[t][c])       (Conv2d(C,1,k) forward)
 *   pai_conv_plane_wide_wgrad dw[c][t] += sum_p wide[p,c] * plane[p+off_t]                  (k = 1 or 3)
 *   pai_gconv4_3x3_fprop      Conv2d(c, c, 3, padding=1, groups=c/4): w fp32 [c][9][4]
 *   pai_gconv4_3x3_wgrad      dw[co][t][j] += sum_p gy[p,co] * x[p+off_t, 4*(co/4)+j]
 */
int pai_conv3x3_fprop(const void* x, int n, int h, int w, int cin, int x_ld, const void* w_packed, int cout,
                      int cout_pad, const float* bias, int act, float slope, void* y, int y_ld, int y_f32, int n_tile,
                      float* splitk_ws, void* stream);
int pai_conv3x3_wgrad(const void* x, int n, int h, int w, int cin, int x_ld, const void* gy, int cout, int gy_ld,
                      float* dw, void* stream);
int pai_maxpool2_fwd(const void* x, int n, int h, int w, int c, int ldx, void* y, int ldy, void* stream);
int pai_maxpool2_bwd(const void* x, int n, int h, int w, int c, int ldx, const void* gy, int ldgy, void* gx, int ldgx,
                     void* stream);
int pai_upsample2_fwd(const void* x, int n, int h, int w, int c, int ldx, void* y, int ldy, void* stream);
int pai_upsample2_bwd(const void* gy, int n, int h, int w, int c, int ldgy, void* gx, int ldgx, void* stream);
int pai_add_act(const void* a, int lda, const void* b, int ldb, long long m, int c, int act, float slope, void* out,
                int ldo, void* stream);
int pai_scale_rows_fwd(const void* x, int ldx, const float* s, long long m, int c, int act, void* out, int ldo,
                       void* stream);
int pai_scale_rows_bwd(const void* x, int ldx, const float* s, const void* g, int ldg, long long m, int c, int act,
                       void* gx, int ldgx, float* gs, void* stream);
/* nn.Dropout2d (models/pix2pix.py:107, models/attention_unet.py, models/res_unet.py): out[n, p, :] = x[n, p, :] * mask[n, :]
 * with mask [n, c] fp32 = 0 or 1/(1 - p) drawn by the caller; in place when out == x; the backward is the same call on
 * the gradient. */
int pai_scale_channels(const void* x, int ldx, const float* mask, int n, long long hw, int c, void* out, int ldo,
                       void* stream);
int pai_conv_plane_to_wide(const float* plane, int n, int h, int w, int k, int pad, int flip, const float* wt,
                           const float* bias, int c, int act, float slope, void* out, int ldo, void* stream);
int pai_conv_wide_to_plane(const void* x, int n, int h, int w, int c, int ldx, int k, int pad, const float* wt,
                           const float* bias, int act, float* out, void* stream);
int pai_conv_plane_wide_wgrad(const float* plane, const void* wide, int ldw, int n, int h, int w, int c, int k, int pad,
                              int flip, float* dw, void* stream);
int pai_gconv4_3x3_fprop(const void* x, int n, int h, int w, int c, int ldx, const float* wt, const float* bias, void* y,
                         int ldy, void* stream);
int pai_gconv4_3x3_wgrad(const void* x, int ldx, const void* gy, int ldg, int n, int h, int w, int c, float* dw,
                         void* stream);

int pai_subsample2(const void* x, int n, int h, int w, int c, int ldx, void* y, int ldy, int scatter, void* stream);

/* ---------------------------------------------------------------------------------------------
 * ViT bottleneck of the Trans U-Net (models/trans_unet.py:120-175): nn.LayerNorm, and
 * nn.TransformerEncoderLayer(d, 8 heads, dim_feedforward=2048, activation="gelu") (post-norm).  Linear layers are
 * pai_pointwise_gemm / pai_pointwise_wgrad.  Tokens are rows of a dense [m, d] bf16 matrix.
 *   pai_layernorm_fwd/bwd  y = (x - mean)/sqrt(var + eps) * gamma + beta over the last dimension; mean / rstd [m] fp32
 *                          are saved for the backward, which also yields dgamma / dbeta (fp32 [d])
 *   pai_gelu_fwd/bwd       exact (erf) GELU
 *   pai_attn_fwd/bwd       multi-head self-attention core over the SEQUENCE axis of qkv [s*b, 3*heads*head_dim]
 *                          (row = s_idx*b + b_idx; the reference's missing batch_first makes s = images of the batch,
 *                          b = patches, SURVEY.md Q4): probs [b*heads, s, s] fp32 = softmax(Q K^T / sqrt(head_dim)),
 *                          out [s*b, heads*head_dim] = probs V; the backward needs an fp32 work buffer like probs.
 *   pai_subsample2         y[n,a,b,:] = x[n,2a,2b,:] (scatter = 0) or its adjoint into a zeroed y (scatter = 1)
 */
int pai_layernorm_fwd(const void* x, long long m, int d, const float* gamma, const float* beta, float eps, void* y,
                      float* mean, float* rstd, void* stream);
int pai_layernorm_bwd(const void* x, const void* g, long long m, int d, const float* gamma, const float* mean,
                      const float* rstd, void* dx, float* dgamma, float* dbeta, void* stream);
int pai_gelu_fwd(const void* x, long long n, void* y, void* stream);
int pai_gelu_bwd(const void* x, const void* g, long long n, void* dx, void* stream);
int pai_attn_fwd(const void* qkv, int s, int b, int heads, int head_dim, float* probs, void* out, void* stream);
int pai_attn_bwd(const void* qkv, const void* dout, int s, int b, int heads, int head_dim, const float* probs,
                 float* ds_work, void* dqkv, void* stream);

/* Train-mode dropout of nn.TransformerEncoderLayer(d, 8, dropout=p) (torch's TransformerEncoderLayer._sa_block /
 * _ff_block), fused into the kernels above.  The mask is regenerated from a counter-based RNG (Philox4x32-10) in
 * every kernel that applies it, forward and backward, and never stored.  Element idx of site `site` under the
 * 64-bit key *key (a device pointer, so a CUDA graph replay can draw a new key):
 *   r = word (idx & 3) of philox4x32_10(counter = (lo32(idx >> 2), hi32(idx >> 2), site, 0), key = (lo32, hi32)),
 *   dropped iff r < llround(p * 2^32) (double precision, clamped to 2^32 - 1); kept elements are scaled by 1/(1-p).
 * Site = layer * 4 + k; idx is the element's linear index in the tensor of site k:
 *   k = 0  attention probabilities [b*heads, s, s] (MultiheadAttention's dropout_p)     pai_attn_fwd/bwd_dropout
 *   k = 1  attention block output [s*b, d] before norm1(x + .) (dropout1)               pai_add_dropout_layernorm_fwd,
 *   k = 3  feed-forward output [s*b, d] before norm2(x + .) (dropout2)                    pai_layernorm_bwd_dropout
 *   k = 2  after the GELU, [s*b, dim_feedforward] (dropout)                             pai_gelu_dropout_fwd/bwd
 * Every entry point rejects a null key and p outside (0, 1) before any CUDA call.
 *   pai_dropout_mask               out_u8[idx] = 1 (kept) / 0 (dropped), idx < n: the mask the kernels apply
 *   pai_attn_fwd_dropout           out = (P o M / (1-p)) V; probs keeps the undropped softmax P
 *   pai_attn_bwd_dropout           dP = (dO V^T) o M / (1-p), dS = P o (dP - rowsum(P o dP)), dV = (P o M / (1-p))^T dO
 *   pai_add_dropout_layernorm_fwd  z = x + y o M / (1-p) (bf16, saved for the backward), out = LayerNorm(z); d % 4 == 0
 *   pai_layernorm_bwd_dropout      pai_layernorm_bwd of (z, g) -> dz, dgamma, dbeta, and dy = dz o M / (1-p)
 *   pai_gelu_dropout_fwd/bwd       y = GELU(x) o M / (1-p);  dx = g o M / (1-p) o GELU'(x); n % 4 == 0
 */
int pai_dropout_mask(const long long* key, int site, long long n, float p, void* out_u8, void* stream);
int pai_attn_fwd_dropout(const void* qkv, int s, int b, int heads, int head_dim, const long long* key, int site, float p,
                         float* probs, void* out, void* stream);
int pai_attn_bwd_dropout(const void* qkv, const void* dout, int s, int b, int heads, int head_dim, const long long* key,
                         int site, float p, const float* probs, float* ds_work, void* dqkv, void* stream);
int pai_add_dropout_layernorm_fwd(const void* x, const void* y, long long m, int d, const long long* key, int site, float p,
                                  const float* gamma, const float* beta, float eps, void* z, void* out, float* mean,
                                  float* rstd, void* stream);
int pai_layernorm_bwd_dropout(const void* z, const void* g, long long m, int d, const float* gamma, const float* mean,
                              const float* rstd, const long long* key, int site, float p, void* dz, void* dy,
                              float* dgamma, float* dbeta, void* stream);
int pai_gelu_dropout_fwd(const void* x, long long n, const long long* key, int site, float p, void* y, void* stream);
int pai_gelu_dropout_bwd(const void* x, const void* g, long long n, const long long* key, int site, float p, void* dx,
                         void* stream);

/* ---------------------------------------------------------------------------------------------
 * fp32 check path (north star: "1e-5 with the fp32 accumulate check path").  Slow, exact twins of the tensor-core
 * layers on fp32 NCHW tensors in the reference's own layouts: one thread per output element, fp32 FMA accumulation,
 * no bf16 rounding.  Forward and backward; used by tests through pai_b200.engine.check_path(), never by training / bench.
 *   pai_check_conv2d_f32     nn.Conv2d (transposed = 0, weight [cout,cin,k,k]) or nn.ConvTranspose2d (transposed = 1,
 *                            weight [cin,cout,k,k]) with square kernel k, stride, zero padding pad; pre_act is the
 *                            activation the reference applies in front of the conv (models/pix2pix.py:62,98,
 *                            models/wrapper.py:205), evaluated on load;  y [n,cout,ho,wo]
 *   pai_check_batchnorm_f32  nn.BatchNorm2d over [n,c,hw]; training = batch statistics (+ running-stat update,
 *                            unbiased variance), eval = running statistics
 *   pai_check_act_f32        elementwise PAI_ACT_* (the final Tanh, models/pix2pix.py:195)
 */
int pai_check_conv2d_f32(const float* x, int n, int cin, int h, int w, const float* wt, int cout, int k, int stride,
                         int pad, const float* bias, int pre_act, float slope, int transposed, float* y, void* stream);
int pai_check_batchnorm_f32(const float* x, int n, int c, int hw, const float* gamma, const float* beta,
                            float* running_mean, float* running_var, int training, float eps, float momentum, float* y,
                            void* stream);
int pai_check_act_f32(const float* x, long long count, int act, float slope, float* y, void* stream);
/* Backward twins (autograd of the three layers above, fp32, double-precision reductions):
 *   pai_check_conv2d_wgrad_f32   dW (same layout as wt) and, if dbias != NULL, dbias[cout] = sum of g, for the layer
 *                                y = conv(pre_act(x)); g = dL/dy [n,cout,ho,wo].  (The data gradient is pai_check_conv2d_f32
 *                                on g with transposed flipped, followed by pai_check_act_bwd_f32 for the pre-activation.)
 *   pai_check_batchnorm_bwd_f32  train-mode BatchNorm2d: dx, dgamma, dbeta from x and g
 *   pai_check_act_bwd_f32        dx = g * act'(x) */
int pai_check_conv2d_wgrad_f32(const float* x, int n, int cin, int h, int w, const float* g, int cout, int k, int stride,
                               int pad, int pre_act, float slope, int transposed, float* dw, float* dbias, void* stream);
int pai_check_batchnorm_bwd_f32(const float* x, const float* g, int n, int c, int hw, const float* gamma, float eps,
                                float* dx, float* dgamma, float* dbeta, void* stream);
int pai_check_act_bwd_f32(const float* x, const float* g, long long count, int act, float slope, float* dx, void* stream);

/* ---------------------------------------------------------------------------------------------
 * dataset.py's per-image transform (dataset.py:51-61,126-134) for a batch of decoded grayscale uint8 images [n,ih,iw]:
 * transforms.Resize((oh, ow), antialias=True) (ATen _upsample_bilinear2d_aa; round_u8 != 0 rounds back to uint8 levels
 * as torchvision does for uint8 tensors) -> ConvertImageDtype(float32) -> Normalize(0.5, 0.5) (normalize != 0; applied
 * to the ONE channel -- the reference passes 3-channel statistics and fails on GRAY images, SURVEY.md Q2).
 * out: fp32 [n,oh,ow].  Decoding PNG/JPEG files stays on the host. */
int pai_resize_aa_normalize_u8(const unsigned char* img, int n, int ih, int iw, int oh, int ow, int normalize,
                               int round_u8, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PAI_B200_H */
