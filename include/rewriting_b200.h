/* rewriting_b200.h — the C-ABI drop-in boundary of librw_b200.so.
 *
 * Every entry point takes plain device pointers, sizes and a cudaStream_t, returns
 * 0 on success or a negative rw_status (never throws, never allocates device
 * memory: scratch is a caller-provided workspace), and runs asynchronously on the
 * given stream.  Pointers are borrowed; the caller (PyTorch in the shipped host
 * code) owns all storage.  This is the surface the reference's two pybind11
 * extension modules plus its library-call "kernels" are replaced by:
 *
 *   reference interface (file:line, relative to davidbau/rewriting)      -> entry point here
 *   -------------------------------------------------------------------------------------------
 *   fused.fused_bias_act(input,bias,refer,act,grad,alpha,scale)
 *       utils/stylegan2/op/fused_bias_act.cpp:11-21                        -> rw_fused_bias_act
 *   upfirdn2d_op.upfirdn2d(input,kernel,up_x,up_y,down_x,down_y,pads)
 *       utils/stylegan2/op/upfirdn2d.cpp:4-22                              -> rw_upfirdn2d
 *   ApplyStyle  style[:,:,None,None]*fmap  utils/stylegan2/models.py:616-620 -> rw_prep_keys
 *   DemodulatedConv2dF.forward (F.conv2d / F.conv_transpose2d + demod)
 *       utils/stylegan2/models.py:313-329                                  -> rw_prep_weights,
 *                                                                              rw_demod,
 *                                                                              rw_modconv_fwd,
 *                                                                              rw_modconv_up_fwd
 *   BlurF -> NoiseInjectionF -> FusedLeakyReLUF of an upsampling StyledConv
 *       utils/stylegan2/models.py:275-281,535-546,622-626                  -> rw_blur_up_act
 *   NoiseInjectionF.forward  utils/stylegan2/models.py:539-546             -> rw_add_noise
 *   ToRGBF.forward           utils/stylegan2/models.py:639-655             -> rw_torgb
 *   autograd of the conv (dgrad / wgrad)                                    -> rw_modconv_fwd on
 *                                                                              gradient planes,
 *                                                                              rw_conv_wgrad
 *   RunningSecondMoment.add -> mom2.addbmm_(a[:,:,None], a[:,None,:])
 *       utils/runningstats.py:1086-1097,1181-1190                          -> rw_split_rows,
 *                                                                              rw_second_moment_accum
 *   projected_conv(weight, direction)  rewrite/ganrewrite.py:806-813       -> rw_project_rank
 *   ProgressiveGanRewriter.insert hot loop rewrite/ganrewrite.py:279-294   -> rw_insert_loop
 *
 * Layout vocabulary
 *   key planes  : the style-modulated key k = style*x as two bf16 planes (hi, lo; k ~= hi+lo)
 *                 in "padded-flat" channels-last order: row index = (b*(H+1) + y)*(W+1) + x,
 *                 y in [0,H], x in [0,W]; row H and column W are zero.  rows = B*(H+1)*(W+1).
 *   weight planes: scale*W as bf16 hi/lo, [Cout][tap][Cin] (tap = u*3+v) — or [Cin][tap'][Cout]
 *                 with flipped taps for dgrad.
 */
#ifndef REWRITING_B200_H_
#define REWRITING_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* rw_stream_t; /* == cudaStream_t */

enum rw_status {
  RW_STATUS_OK = 0,
  RW_STATUS_BAD_ARG = -1,
  RW_STATUS_CUDA = -2,
  RW_STATUS_NO_DRIVER_SYMBOL = -3,
  RW_STATUS_UNSUPPORTED = -4
};

/* ---- library ---- */
int rw_version(void);
const char* rw_last_error(void);
int rw_set_device(int device);
int rw_device_sm_count(void);

/* ---- operand preparation ---- */
int rw_prep_keys(const float* x, const float* style, int B, int C, int H, int W, void* kp_hi,
                 void* kp_lo, float* k_out, rw_stream_t stream);
int rw_split_rows(const float* a, long long n, void* hi, void* lo, rw_stream_t stream);
int rw_prep_weights(const float* w, int Cout, int Cin, float scale, int transpose_io,
                    int flip_taps, void* wt_hi, void* wt_lo, float* wsq, rw_stream_t stream);
int rw_demod(const float* style, const float* wsq, int B, int Cout, int Cin, float eps,
             float* demod, rw_stream_t stream);

/* ---- fused modulated 3x3 convolution (tcgen05) ---- */
/* out[b,o,y,x] = act( conv3x3(k, scale*W)[b,o,y,x] * scale_bo[b,o] + noise_w[0]*noise[b,y*W+x] + bias[o] )
 * scale_bo / noise / bias may be NULL; noise_w is a DEVICE scalar (the nn.Parameter's storage,
 * so no host sync per layer); act: 0 none, 1 leaky_relu(0.2)*sqrt(2). */
int rw_modconv_fwd(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                   const float* scale_bo, const float* noise, long long noise_bstride,
                   const float* noise_w, const float* bias, int act, int B, int Cin, int Cout,
                   int H, int W, float* out, rw_stream_t stream);
/* t[b,o,:,:] = conv_transpose2d(k, (scale*W)^T, stride 2, pad 0)[b,o] * scale_bo[b,o]; out is
 * [B,Cout,2H+1,2W+1].  One launch: the four polyphase components are tile-interleaved (exact
 * algorithmic FLOPs, A tiles shared through L2). */
int rw_modconv_up_fwd(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                      const float* scale_bo, int B, int Cin, int Cout, int H, int W, float* t_out,
                      rw_stream_t stream);
/* ---- generation fast path: producers write the consumer's operands directly ----
 * rw_modconv_fwd_fused = rw_modconv_fwd whose epilogue can additionally emit
 *   next_{hi,lo}[rows][Cout] : key planes of the NEXT layer, split_bf16(next_scale[b,o] * y)
 *   rgb_part[P][B][3][H*W] : this layer's ToRGB partial sums, one per epilogue column group,
 *                            with rgb_w[B,3,Cout]; P = rw_modconv_rgb_parts(Cout) (Cout/64 for
 *                            Cout % 128 == 0, 2 for the 64- and 32-channel layers)
 * `out` (fp32 NCHW) becomes optional.  rw_modconv_up_fwd_cl writes the conv_transpose output
 * channels-last per phase, t_cl[4][rows][Cout]; rw_blur_up_fused turns it into the next layer's
 * planes (and/or fp32 NCHW); rw_rgb_combine = sum of partials + bias + 2x-upsampled skip. */
int rw_modconv_fwd_fused(const void* kp_hi, const void* kp_lo, const void* wt_hi,
                         const void* wt_lo, const float* scale_bo, const float* noise,
                         long long noise_bstride, const float* noise_w, const float* bias, int act,
                         int B, int Cin, int Cout, int H, int W, float* out,
                         const float* next_scale, void* next_hi, void* next_lo,
                         const float* rgb_w, float* rgb_part, rw_stream_t stream);
/* number of ToRGB partials rw_modconv_fwd_fused writes for Cout output channels; < 1 when the
 * row-GEMM does not take Cout */
int rw_modconv_rgb_parts(int Cout);
int rw_modconv_up_fwd_cl(const void* kp_hi, const void* kp_lo, const void* wt_hi,
                         const void* wt_lo, const float* scale_bo, int B, int Cin, int Cout, int H,
                         int W, float* t_cl, rw_stream_t stream);
int rw_blur_up_fused(const float* t_cl, int B, int C, int Hin, int Win, const float* kernel4x4,
                     const float* noise, long long noise_bstride, const float* noise_w,
                     const float* bias, int act, const float* next_scale, void* next_hi,
                     void* next_lo, float* y_out, rw_stream_t stream);
/* The whole upsampling StyledConv of the fast path in ONE kernel (csrc/upconv_tc.cu):
 * conv_transpose2d(stride 2) -> 4x4 blur (pad 1,1) -> * demod -> + noise_w*noise + bias ->
 * leaky-ReLU*sqrt(2) -> * next_scale -> the next layer's bf16 hi/lo planes (pad row/column zeroed).
 * Replaces the reference chain models.py:313-329 (DemodulatedConv2dF, upsample branch) -> :275-281
 * (BlurF / upfirdn2d_kernel.cu:52-137) -> :535-546 (NoiseInjectionF) -> fused_bias_act_kernel.cu
 * :27-47, without ever writing the (2H+1)x(2W+1) fp32 conv_transpose output.
 * wt_{hi,lo}: rw_prep_weights(transpose_io = 2) planes [Cout/16][2 channel halves][9 taps][8][Cin]
 * (opaque to the caller: produced and consumed by this library only).  W must be a power
 * of two in [4, 128], Cin % 64 == 0, Cout % 16 == 0, the 4x4 kernel rank one (separable). */
int rw_modconv_up_fused(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                        const float* demod, const float* kernel4x4, const float* noise,
                        long long noise_bstride, const float* noise_w, const float* bias,
                        const float* next_scale, void* next_hi, void* next_lo, int B, int Cin,
                        int Cout, int H, int W, rw_stream_t stream);

/* The same kernel as the LAYER-level op (the autograd forward of an upsampling StyledConv,
 * reference models.py:232-289 with upsample=True): writes this layer's activation y
 * [B, Cout, 2H, 2W] fp32 NCHW instead of the next layer's planes.  demod may be NULL (no
 * demodulation), noise / noise_w NULL together (no noise injection), act = 0 skips bias + leaky-ReLU
 * (bias may then be NULL). */
int rw_modconv_up_fused_y(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                          const float* demod, const float* kernel4x4, const float* noise,
                          long long noise_bstride, const float* noise_w, const float* bias, int act,
                          float* y, int B, int Cin, int Cout, int H, int W, rw_stream_t stream);
/* all modulation linears in one launch: out_l[b,c] = latent[b,lat_l,:] . (W_l[c,:]*scale) + bias_l[c]
 * (HOST arrays of n device pointers / ints; n <= 32) */
int rw_styles(const float* latent, int B, int n_latent, int K, float scale, int n,
              const float* const* w, const float* const* bias, float* const* out, const int* lat,
              const int* chans, rw_stream_t stream);
/* EqualLinear (utils/stylegan2/models.py:487-511): out[b,c] = sum_k x[b,k]*(w[c,k]*scale) +
 * bias[c]*bias_mul, then lrelu(0.2)*sqrt(2) when act != 0 (the mapping network's
 * fused_lrelu layers, lr_mul = 0.01).  One launch per layer instead of sgemm + bias_act + two
 * elementwise kernels. */
int rw_equal_linear(const float* x, int B, int K, const float* w, const float* bias, int Cout,
                    float scale, float bias_mul, int act, float* out, rw_stream_t stream);
/* PixelNormL (models.py:609-614): out = z * rsqrt(mean(z^2, dim 1) + 1e-8), z [B,K] */
int rw_pixel_norm(const float* z, int B, int K, float* out, rw_stream_t stream);
/* Everything that depends only on the styles, for all layers in one launch (n <= 32 jobs):
 * kind 0: out[b,o] = rsqrt(sum_i style[b,i]^2 * w[o,i] + eps)  (w = wsq of rw_prep_weights; the
 *         demodulation factor of models.py:325-327);
 * kind 1: out[b,c,i] = (wscale*w[c,i])*style[b,i]  (ToRGB's modulated 1x1 weights, cout = 3). */
int rw_demod_multi(int B, float eps, int n, const float* const* style, const float* const* w,
                   float* const* out, const int* cout, const int* cin, const int* kind,
                   const float* wscale, rw_stream_t stream);
int rw_rgb_combine(const float* part, int nparts, int B, int H, int W, const float* bias,
                   const float* prev, const float* kernel4x4, float* out, rw_stream_t stream);
/* same, and/or the image as NHWC bytes  clamp(x*127.5 + 127.5, 0, 255)  (uint8 truncation): the
 * output side of the sampling loops (metrics/sample.py:33-37, utils/get_samples.py:121-127 move
 * fp32 NCHW images to the host one by one); `out` may be NULL when only the bytes are wanted */
int rw_rgb_combine_u8(const float* part, int nparts, int B, int H, int W, const float* bias,
                      const float* prev, const float* kernel4x4, float* out,
                      unsigned char* out_u8_nhwc, rw_stream_t stream);
/* y = act( upfirdn2d(t, k4x4, pad=(1,1)) + noise_w*noise + bias ), t [B,C,2H+1,2W+1] -> y [B,C,2H,2W] */
int rw_blur_up_act(const float* t, int B, int C, int Hin, int Win, const float* kernel4x4,
                   const float* noise, long long noise_bstride, const float* noise_w,
                   const float* bias, int act, float* y, rw_stream_t stream);
int rw_add_noise(const float* x, const float* noise, long long noise_bstride,
                 const float* noise_w, int B, int C, int HW, float* y, rw_stream_t stream);
int rw_torgb(const float* x, const float* style, const float* w, const float* bias,
             const float* skip, int B, int C, int H, int W, float scale, float* out,
             rw_stream_t stream);

/* ---- operator-level ops of the reference ---- */
int rw_fused_bias_act(const float* x, const float* bias, const float* ref, int act, int grad,
                      float alpha, float scale, long long n, int step_b, int size_b, float* y,
                      rw_stream_t stream);
int rw_upfirdn2d(const float* in, const float* kernel, int major, int in_h, int in_w, int kh,
                 int kw, int up_x, int up_y, int down_x, int down_y, int pad_x0, int pad_x1,
                 int pad_y0, int pad_y1, float* out, int out_h, int out_w, rw_stream_t stream);

/* ---- key second moment / weight gradient (tcgen05 col-GEMM) ---- */
size_t rw_gram_workspace_bytes(int Cm, int Cn, long long rows, int ntaps);
/* mom2[C,C] += sum_r a_r a_r^T over `rows` rows of the hi/lo planes [rows][C] */
int rw_second_moment_accum(const void* hi, const void* lo, long long rows, int C, float* mom2,
                           void* workspace, size_t workspace_bytes, rw_stream_t stream);
/* dW[o][tap][i] = sum_p G[p,o] * K[p + shift(tap), i]  for a 3x3 conv over the padded-flat grid
 * (up=0) or the conv_transpose phases (up=1: G planes are given per phase, see host code). */
int rw_conv_wgrad(const void* g_hi, const void* g_lo, const void* kp_hi, const void* kp_lo,
                  long long rows, int Cout, int Cin, int Wp, float* dw_toi, void* workspace,
                  size_t workspace_bytes, rw_stream_t stream);

/* backward of the upsampling layer: gradient phase planes [rows][4*Cout] (rw_prep_phase_keys from the
 * gradient wrt the conv_transpose output [B,Cout,2H+1,2W+1], times demod), then
 *   dk[b,i,y,x] = sum_{o,u,v} g[b,o,2y+u,2x+v] * scale*W[o,i,u,v]      (rw_modconv_up_dgrad, weights
 *                 as [Cin][tap][Cout] planes, taps NOT flipped)
 *   dW[o][tap][i] = sum_p G_phase(tap)[p + shift(tap), o] * K[p, i]     (rw_conv_up_wgrad) */
int rw_prep_phase_keys(const float* g, const float* scale_bc, int B, int C, int H, int W,
                       void* hi, void* lo, rw_stream_t stream);
int rw_modconv_up_dgrad(const void* gph_hi, const void* gph_lo, const void* wt_hi,
                        const void* wt_lo, const float* scale_bi, int B, int Cin, int Cout, int H,
                        int W, float* dk, rw_stream_t stream);
int rw_conv_up_wgrad(const void* gph_hi, const void* gph_lo, const void* kp_hi, const void* kp_lo,
                     long long rows, int Cout, int Cin, int Wp, float* dw_toi, void* workspace,
                     size_t workspace_bytes, rw_stream_t stream);

/* ---- StyledConv backward: the HBM-bound passes between the tensor-core kernels ----
 * (autograd of FusedLeakyReLUF / NoiseInjectionF / BlurF / ApplyStyle / the demodulation:
 *  utils/stylegan2/op/fused_act.py:19-86, utils/stylegan2/models.py:275-281,320-328,535-546,616-620)
 *
 * rw_act_grad_reduce: one pass over (gy, y) of a [B,C,HW] layer output y = act(t + nw*noise + bias):
 *   g_pre = dL/d(pre-activation) (written unless g_pre == NULL; equal to gy when act == 0),
 *   s_sum[b,c] = sum_p g_pre, s_dot[b,c] = sum_p g_pre*t (t recovered from y), s_noise[b,c] =
 *   sum_p g_pre*noise[b,p].  noise / bias may be NULL.
 * rw_blur_adj_phase_keys: gradient phase planes [rows][4*C] (the layout of rw_prep_phase_keys) of
 *   scale[b,c] * blur^T(g_pre), g_pre [B,C,2H,2W]; the [B,C,2H+1,2W+1] tensor is never stored.
 * rw_dgrad_finish: gs_raw[b,i] = sum_p dk*x; dk <- dk*style[b,i] in place ([B,C,HW] planes).
 * rw_wgrad_finish: gw[o,i,tap] = scale*dw_toi[o,tap,i] - scale^2*w[o,i,tap]*sum_b s_dot[b,o]*
 *   demod[b,o]^2*style[b,i]^2 (s_dot == NULL: no demodulation term).
 * rw_style_grad_finish: g_style[b,i] = gs_raw[b,i] - style[b,i]*sum_o s_dot[b,o]*demod[b,o]^2*
 *   wsq[o,i] (gs_raw == NULL: 0). */
int rw_act_grad_reduce(const float* gy, const float* y, const float* noise,
                       long long noise_bstride, const float* noise_w, const float* bias, int act,
                       int B, int C, int HW, float* g_pre, float* s_sum, float* s_dot,
                       float* s_noise, rw_stream_t stream);
int rw_blur_adj_phase_keys(const float* g_pre, const float* scale_bc, const float* kernel4x4, int B,
                           int C, int H, int W, void* hi, void* lo, rw_stream_t stream);
int rw_dgrad_finish(float* dk, const float* x, const float* style, int B, int C, int HW,
                    float* gs_raw, rw_stream_t stream);
int rw_wgrad_finish(const float* dw_toi, const float* w, const float* s_dot, const float* demod,
                    const float* style, int B, int Cout, int Cin, float scale, float* gw,
                    rw_stream_t stream);
int rw_style_grad_finish(const float* gs_raw, const float* style, const float* s_dot,
                         const float* demod, const float* wsq, int B, int Cout, int Cin,
                         float* g_style, rw_stream_t stream);

/* ---- rank-r edit ---- */
/* out = base + sign * P_d(w);  P_d(w)[o,:,t] = sum_r (w[o,:,t] . d_r) d_r;  base may be NULL */
int rw_project_rank(const float* w, const float* base, const float* d, int rank, int Cout,
                    int Cin, int taps, float sign, float* out, rw_stream_t stream);

typedef struct rw_insert_args {
  float* W;               /* [Cout,Cin,3,3], updated in place */
  float* m;               /* Adam exp_avg     */
  float* v;               /* Adam exp_avg_sq  */
  const float* w_ortho;   /* W0 - P_d(W0) or NULL (low_rank_insert off) */
  const float* d;         /* [rank,Cin] orthonormal rows */
  const float* key_cl;    /* key crop, zero-bordered channels-last [B][h+2][w+2][Cin] */
  const float* style;     /* [B,Cin] */
  const float* target;    /* goal activations v* [B,Cout,h,w] */
  const float* noise;     /* [B,h*w] or NULL */
  const float* bias;      /* [Cout] or NULL */
  float* loss_out;        /* [nsteps,Cout] per-channel sums of |v*-y| */
  float noise_w, lr, beta1, beta2, eps;
  int rank, B, Cin, Cout, h, w;
  int has_noise_act;      /* 1: target = dconv->noise->activate, 0: dconv only */
  int it0, nsteps, niter_total, piter, project_gradient;
  /* appended in round 2 (zero = the StyleGAN2 behaviour of round 1): */
  int plain_conv;          /* 1: y = conv(k, W) with no style demodulation and no 1/sqrt(9 Cin)
                              weight scale — the `layerN.conv` target of ProgressiveGanRewriter
                              (ganrewrite.py:25-96; `style` is then ignored and may be NULL) */
  float one_minus_beta1;   /* torch.optim.Adam forms 1-beta in double and rounds once to float */
  float one_minus_beta2;   /* (0 -> computed in the kernel as 1.0f - beta) */
  double beta1_exact;      /* the betas as the Python doubles torch forms its bias corrections */
  double beta2_exact;      /* 1 - beta**step from (0 -> the float fields above, widened) */
} rw_insert_args;
int rw_insert_loop(const rw_insert_args* args, rw_stream_t stream);

/* out[rows][N] = A[rows][K] . W[N][K]^T on the tensor-core row-GEMM (3-term split bf16 planes from
 * rw_split_rows; K % 64 == 0, N % 128 == 0): the key algebra between key capture and the
 * direction d — ZCA . k and ZCA . v of ganrewrite.py:107-110, 339-374 — without a cuBLAS call */
int rw_rowgemm(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, int rows, int K,
               int N, float* out, rw_stream_t stream);

/* ---- ProgGAN generator leaves (reference utils/proggan.py:128-181): the target of
 * ProgressiveGanRewriter is a plain `layerN.conv` (ganrewrite.py:25-96) ----
 * rw_pixel_norm_nchw: PixelNormLayer, x / sqrt(mean_c x^2 + 1e-8), optionally fused with the
 *   following DoubleResolutionLayer (nearest 2x, up2 = 1: out is [B,C,2H,2W]);
 * rw_nearest_up2: DoubleResolutionLayer alone on [planes,H,W];
 * rw_conv3x3_bias_act: 3x3 conv (pad 1) over key planes on the tensor-core row-GEMM with
 *   + bias[o] and leaky-ReLU(0.2) * act_gain in the epilogue — NormConvBlock's conv -> WScaleLayer
 *   -> LeakyReLU when the WScale factor is folded into the weight planes (rw_prep_weights scale). */
int rw_pixel_norm_nchw(const float* x, int B, int C, int H, int W, int up2, float* out,
                       rw_stream_t stream);
int rw_nearest_up2(const float* x, long long planes, int H, int W, float* out, rw_stream_t stream);
int rw_conv3x3_bias_act(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                        const float* bias, int act, float act_gain, int B, int Cin, int Cout, int H,
                        int W, float* out, rw_stream_t stream);

/* ---- bring-up hooks (tests/tools only) ---- */
/* rw_modconv_up_fused with demod = next_scale = ones_bo, additionally dumping the raw tap products
 * P[b][y][x][tap][Cout] of the tensor-core stage */
int rw_debug_upconv_taps(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                         const float* ones_bo, const float* kernel4x4, const float* noise,
                         long long noise_bstride, const float* noise_w, const float* bias,
                         void* next_hi, void* next_lo, int B, int Cin, int Cout, int H, int W,
                         float* taps_out, rw_stream_t stream);
int rw_debug_rowgemm(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo,
                     int rows, int K, int N, float* out, rw_stream_t stream);
int rw_debug_colgemm(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                     int rows, int Cm, int Cn, int lbo_bytes, int sbo_bytes, float* out,
                     void* workspace, size_t workspace_bytes, rw_stream_t stream);

/* rw_modconv_up_fused instrumented with clock64(): prof_out[grid][8 epilogue warps][16] = cycles in
 * {wait for the MMAs, TMEM drain, combine + mailbox + barrier, shuffles, edge-lane fix-ups,
 * horizontal FIR, vertical FIR + activation + stores}, the step count, and the last phase split into
 * {FIR + activation + bf16 split, wait for the staging slots, stmatrix + fence + pair barrier, TMA store issue} and
 * the third of those into {stmatrix, fence.proxy.async, pair barrier} */
int rw_debug_upconv_profile(const void* kp_hi, const void* kp_lo, const void* wt_hi,
                            const void* wt_lo, const float* demod, const float* kernel4x4,
                            const float* noise, long long noise_bstride, const float* noise_w,
                            const float* bias, const float* next_scale, void* next_hi, void* next_lo,
                            int B, int Cin, int Cout, int H, int W, long long* prof_out,
                            rw_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* REWRITING_B200_H_ */
