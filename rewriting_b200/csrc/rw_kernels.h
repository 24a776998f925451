// rw_kernels.h — internal launch interfaces between the C-ABI (api.cu) and the
// kernel translation units.  Not part of the public boundary (see
// include/rewriting_b200.h for that).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rw {

// ---------------------------------------------------------------------------
// row-GEMM (conv_tc.cu)
// ---------------------------------------------------------------------------
struct ConvTcParams {
  int rows;          // padded-flat rows = B * Hp * Wp  (GEMM M)
  int Cin;           // GEMM K per tap
  int Cout;          // GEMM N
  // Up to 4 "phases" share one launch (the 4 polyphase components of a stride-2
  // conv_transpose): tile index = (m, n, phase) with phase fastest, so the CTAs that
  // run concurrently read the same A tiles (L2 hits instead of 4 DRAM passes).
  int nphase;
  int ph_ntaps[4];
  int ph_shift[4][9];   // row shift applied to the A operand for this tap
  int ph_kofs[4][9];    // column offset of this tap inside the weight matrix
  int ph_acol[4][9];    // column offset of this tap inside the A planes (0 unless A holds
                        // several channel-concatenated tensors, e.g. the 4 gradient phases)
  int a_cols;           // total columns of the A planes (0 -> Cin)
  int ph_Hv[4], ph_Wv[4];       // valid output extent inside the padded grid
  long long ph_out_ofs[4];      // element offset of this phase's output origin
  int Hp, Wp;        // padded grid of one image
  int B;             // batch (only needed for the rgb partial layout)
  // epilogue
  const float* scale_bo;  // [B, Cout] per-sample per-channel scale (demod / style) or null
  const float* bias;      // [Cout] or null
  const float* noise;     // [B, noise_bstride] or null, indexed y*Wv + x
  long long noise_bstride;
  const float* noise_w;   // device scalar (read by the kernel: no host sync per layer)
  int act;                // 1 -> leaky_relu(0.2) * act_gain
  float act_gain;         // 0 -> sqrt(2) (FusedLeakyReLU); ProgGAN's nn.LeakyReLU uses 1
  float* out;             // may be null when only planes / rgb partials are wanted
  long long out_sb, out_sc, out_sy, out_sx;  // element strides: batch, channel, y, x
  // out_mode 0: strided (NCHW-like) store at valid positions only
  // out_mode 1: channels-last rows  out[(ph*rows + p)*Cout + o]  for every row p < rows
  int out_mode;
  // fused producer outputs (generation fast path): the NEXT layer's key planes
  //   next_{hi,lo}[p][o] = split_bf16(next_scale[b,o] * y)   (zero at pad positions)
  void* next_hi;
  void* next_lo;
  const float* next_scale;   // [B, Cout] style of the consuming layer
  // and this layer's ToRGB partial sums over the tile's 128 output channels
  //   rgb_part[nt][b][c][y*Wv+x] = sum_{o in tile} rgb_w[b][c][o] * y[b,o,y,x]
  float* rgb_part;
  const float* rgb_w;        // [B, 3, Cout] modulated 1x1 weights
};

int conv_tc_launch(const ConvTcParams& p, const void* a_hi, const void* a_lo, const void* w_hi,
                   const void* w_lo, int wk_total, cudaStream_t stream);
// N tile of a Cout-channel launch (128, or 64 / 32 for the narrow layers; 0 = unsupported) and the
// number of ToRGB partial groups the fused epilogue writes (2 * Cout / N tile)
int conv_tc_tile_n(int Cout);
int conv_tc_rgb_parts(int Cout);

// ---------------------------------------------------------------------------
// fused upsampling StyledConv (upconv_tc.cu): conv_transpose + blur + demod + noise + bias +
// leaky-ReLU + next-layer style -> bf16 hi/lo planes, one kernel, no fp32 intermediate
// ---------------------------------------------------------------------------
struct UpFusedParams {
  int B, Cin, Cout, H, W;      // input resolution H x W (W a power of two, 4..128)
  const float* demod;          // [B, Cout]
  const float* bias;           // [Cout]
  const float* noise;          // [B, noise_bstride], indexed Y * 2W + X at OUTPUT resolution
  long long noise_bstride;
  const float* noise_w;        // device scalar
  const float* k4;             // 4x4 blur kernel (rank one)
  const float* next_scale;     // [B, Cout] style of the consuming layer
  void* next_hi;               // [B][2H+1][2W+1][Cout] bf16 planes (pad row / column zeroed)
  void* next_lo;
  // layer-level mode (the autograd op's forward): y_out != null writes the layer's own output
  // y [B][Cout][2H][2W] fp32 instead of the next layer's planes; demod / noise / noise_w may then
  // be null (= 1 / no noise) and act = 0 skips bias + leaky-ReLU
  float* y_out;
  int act;
  int ncg, nbands, nitems;     // filled by the launcher
  float* debug_p;              // bring-up: raw tap products P[b][y][x][tap][Cout] (y < H), or null
  int debug_nostore;           // bring-up (profiling variant only): skip the plane stores
  long long* debug_prof;       // bring-up: per (CTA, epilogue warp) cycle counters [grid][8][16], or null
};
// weights: bf16 hi/lo planes [Cout/16][channel half][9 taps][8][Cin]  (rw_prep_weights, transpose_io = 2)
int upconv_fused_launch(const UpFusedParams& p, const void* a_hi, const void* a_lo,
                        const void* w_hi, const void* w_lo, cudaStream_t stream);

// ---------------------------------------------------------------------------
// col-GEMM (gram_tc.cu):  out[m, n] = sum_r A[r + shift_a, m] * B[r + shift_b, n]
// ---------------------------------------------------------------------------
struct GramTcParams {
  int rows;            // contraction length (rows r in [0, rows))
  int rows_a, rows_b;  // allocated rows of the A / B planes (for the TMA bounds)
  int Cm, Cn;          // channels of A (-> M) and B (-> N)
  int shift_a, shift_b;
  int ntaps;              // >= 1; grid.z
  int tap_shift_a[9];     // extra row shift of the A operand per tap
  int tap_acol[9];        // column offset inside the A planes per tap
  int a_cols;             // total columns of the A planes (0 -> Cm)
  int tap_shift_b[9];     // extra row shift of the B operand per tap
  int tap_col_ofs[9];     // column offset of this tap's block inside a partial row
  int splits;          // row-range splits (partials reduced deterministically afterwards)
  float* partial;      // [splits][Cm][ldp] fp32 workspace
  long long ldp;       // leading dimension (elements) of one partial matrix row
  int upper_only;      // 1: skip tiles strictly below the diagonal (symmetric A==B)
};

int gram_tc_launch(const GramTcParams& p, const void* a_hi, const void* a_lo, const void* b_hi,
                   const void* b_lo, cudaStream_t stream);

// out[m*ldo+n] (= or +=) sum_s partial[s][m][n]; optional symmetric mirror of the
// upper triangle into the lower one.
int reduce_partials_launch(const float* partial, int splits, int M, int N, long long ldp,
                           float* out, long long ldo, int accumulate, int mirror_upper,
                           cudaStream_t stream);

// ---------------------------------------------------------------------------
// SIMT kernels (simt.cu)
// ---------------------------------------------------------------------------
int prep_phase_keys_launch(const float* g, const float* scale_bc, int B, int C, int H, int W,
                           void* hi, void* lo, cudaStream_t stream);
int prep_keys_launch(const float* x, const float* style, int B, int C, int H, int W, void* kp_hi,
                     void* kp_lo, float* k_out, cudaStream_t stream);
int split_rows_launch(const float* a, long long n, void* hi, void* lo, cudaStream_t stream);
int prep_weights_launch(const float* w, int Cout, int Cin, float scale, int transpose_io,
                        int flip_taps, void* wt_hi, void* wt_lo, float* wsq, cudaStream_t stream);
int demod_launch(const float* style, const float* wsq, int B, int Cout, int Cin, float eps,
                 float* demod, cudaStream_t stream);
int blur_up_act_launch(const float* t, int B, int C, int Hin, int Win, const float* kernel4x4,
                       const float* noise, long long noise_bstride, const float* noise_w,
                       const float* bias, int act, float* y, cudaStream_t stream);
int blur_up_fused_launch(const float* t_cl, int B, int C, int Hin, int Win, const float* k4,
                         const float* noise, long long noise_bstride, const float* noise_w,
                         const float* bias, int act, const float* next_scale, void* next_hi,
                         void* next_lo, float* y_out, cudaStream_t stream);
int rgb_combine_launch(const float* part, int nparts, int B, int H, int W, const float* bias,
                       const float* prev, const float* k4, float* out, unsigned char* out_u8,
                       cudaStream_t stream);
int styles_launch(const float* latent, int B, int n_latent, int K, float scale, float bias_mul,
                  int act, int n, const float* const* w, const float* const* bias,
                  float* const* out, const int* lat, const int* chans, cudaStream_t stream);
int pixel_norm_launch(const float* z, int B, int K, float* out, cudaStream_t stream);
int pixel_norm_nchw_launch(const float* x, int B, int C, int H, int W, int up2, float* out,
                           cudaStream_t stream);
int nearest_up2_launch(const float* x, long long planes, int H, int W, float* out,
                       cudaStream_t stream);
int demod_multi_launch(int B, float eps, int n, const float* const* style,
                       const float* const* wsq, float* const* out, const int* cout,
                       const int* cin, const int* kind, const float* wscale,
                       cudaStream_t stream);
int upfirdn2d_launch(const float* in, const float* kernel, int major, int in_h, int in_w, int kh,
                     int kw, int up_x, int up_y, int down_x, int down_y, int px0, int px1, int py0,
                     int py1, float* out, int out_h, int out_w, cudaStream_t stream);
int bias_act_launch(const float* x, const float* bias, const float* ref, int act, int grad,
                    float alpha, float scale, long long n, int step_b, int size_b, float* y,
                    cudaStream_t stream);
int torgb_launch(const float* x, const float* style, const float* w, const float* bias,
                 const float* skip, int B, int C, int H, int W, float scale, float* out,
                 cudaStream_t stream);
int add_noise_launch(const float* x, const float* noise, long long noise_bstride, const float* noise_w,
                     int B, int C, int HW, float* y, cudaStream_t stream);

// StyledConv backward, HBM-bound passes (bwd.cu)
int act_grad_reduce_launch(const float* gy, const float* y, const float* noise,
                           long long noise_bstride, const float* noise_w, const float* bias,
                           int act, int B, int C, int HW, float* g_pre, float* s_sum,
                           float* s_dot, float* s_noise, cudaStream_t stream);
int blur_adj_phase_launch(const float* g_pre, const float* scale_bc, const float* k4, int B, int C,
                          int H, int W, void* hi, void* lo, cudaStream_t stream);
int dgrad_finish_launch(float* dk, const float* x, const float* style, int B, int C, int HW,
                        float* gs_raw, cudaStream_t stream);
int wgrad_finish_launch(const float* dwt, const float* w, const float* s_dot, const float* dm,
                        const float* style, int B, int Cout, int Cin, float sc, float* gw,
                        cudaStream_t stream);
int style_grad_finish_launch(const float* gs_raw, const float* style, const float* s_dot,
                             const float* dm, const float* wsq, int B, int Cout, int Cin,
                             float* g_style, cudaStream_t stream);

// rewrite (rewrite.cu)
int project_rank_launch_signed(const float* w, const float* base, const float* d, int rank,
                               int Cout, int Cin, int taps, float sign, float* out,
                               cudaStream_t stream);
void gram_tc_set_desc(int lbo, int sbo);

struct InsertLoopParams {
  float* W;             // [Cout, Cin, 3, 3] updated in place
  float* m;             // Adam first moment  (same shape)
  float* v;             // Adam second moment (same shape)
  const float* w_ortho; // W0 - P_d(W0), or null when low_rank_insert is off
  const float* d;       // [rank, Cin] orthonormal rows
  int rank;
  const float* key;     // key crop, zero-bordered channels-last [B][h+2][w+2][Cin]
  const float* style;   // [B, Cin]
  const float* target;  // [B, Cout, h, w] goal activations v*
  const float* noise;   // [B, h*w] or null
  float noise_w;
  const float* bias;    // [Cout]
  int B, Cin, Cout, h, w;
  int has_noise_act;    // 1: target ends after `activate`; 0: ends after dconv
  float lr, beta1, beta2, eps;
  int it0, niter_total, nsteps;  // run iterations it0 .. it0+nsteps-1
  int piter;
  int project_gradient; // low_rank_gradient
  float* loss_out;      // [nsteps, Cout] per-channel partial |v*-y| sums
  int plain_conv;       // 1: no demodulation, weight scale 1 (ProgGAN `layerN.conv`)
  float one_minus_beta1, one_minus_beta2;   // 1-beta as torch forms it (double, rounded once)
  double beta1_exact, beta2_exact;          // betas for the bias corrections (python doubles)
};
int insert_loop_launch(const InsertLoopParams& p, cudaStream_t stream);

}  // namespace rw
