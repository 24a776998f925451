// simt.cu — HBM-bound CUDA-core kernels around the tensor-core path: operand
// preparation (style modulation + bf16 hi/lo split + NCHW -> padded-flat
// channels-last), demodulation factors, the up-path blur epilogue, ToRGB, and the
// two operator-level ops of the reference (`fused_bias_act`, `upfirdn2d`).
//
// Reference semantics (cited per kernel) are utils/stylegan2/models.py and
// utils/stylegan2/op/*.  All kernels are coalesced / vectorised; none uses
// tensor cores (these are byte-movement bound, SURVEY.md §8d).
#include <cstdlib>

#include "rw_common.cuh"
#include "rw_kernels.h"

namespace rw {

namespace {

// ---------------------------------------------------------------------------
// prep_keys: k = style[b,c] * x[b,c,y,x]   (ApplyStyle, models.py:616-620)
//   -> optional fp32 NCHW copy (the API-visible key) and bf16 hi/lo planes in
//   the padded-flat layout  [(b, y in 0..H, x in 0..W)][c]  with zero pad row /
//   pad column.
// grid: (ceil(Hp*Wp/32), C/CB, B), block 256; CB = 64 channels per block, 32 when C % 64 != 0
// ---------------------------------------------------------------------------
template <int CB>
__global__ void __launch_bounds__(256)
prep_keys_kernel(const float* __restrict__ x, const float* __restrict__ style, int C, int H, int W,
                 __nv_bfloat16* __restrict__ kp_hi, __nv_bfloat16* __restrict__ kp_lo,
                 float* __restrict__ k_out) {
  __shared__ float tile[CB][33];
  const int Hp = H + 1, Wp = W + 1;
  const int img = Hp * Wp;
  const int p0 = blockIdx.x * 32;
  const int c0 = blockIdx.y * CB;
  const int b = blockIdx.z;
  const int t = threadIdx.x;
  {
    const int pl = t & 31;
    const int p = p0 + pl;
    const int yy = p / Wp, xx = p - yy * Wp;
    const bool valid = (p < img) && (yy < H) && (xx < W);
#pragma unroll
    for (int i = 0; i < CB / 8; ++i) {
      const int cl = (t >> 5) + 8 * i;
      float v = 0.f;
      if (valid) {
        const size_t gi = ((static_cast<size_t>(b) * C + c0 + cl) * H + yy) * W + xx;
        const float s = style ? __ldg(style + static_cast<size_t>(b) * C + c0 + cl) : 1.f;
        v = s * __ldg(x + gi);
        if (k_out) k_out[gi] = v;
      }
      tile[cl][pl] = v;
    }
  }
  __syncthreads();
  {
    const int pl = t / (CB / 8);        // position (0..31 used)
    const int cg = (t % (CB / 8)) * 8;  // 8 channels per thread
    const int p = p0 + pl;
    if (pl < 32 && p < img) {
      __align__(16) __nv_bfloat16 h[8];
      __align__(16) __nv_bfloat16 l[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) split_bf16(tile[cg + j][pl], h[j], l[j]);
      const size_t row = static_cast<size_t>(b) * img + p;
      *reinterpret_cast<uint4*>(kp_hi + row * C + c0 + cg) = *reinterpret_cast<const uint4*>(h);
      *reinterpret_cast<uint4*>(kp_lo + row * C + c0 + cg) = *reinterpret_cast<const uint4*>(l);
    }
  }
}

// ---------------------------------------------------------------------------
// prep_phase_keys: gradient planes of a stride-2 conv_transpose output.
//   g [B,C,2H+1,2W+1] fp32 (gradient wrt the conv_transpose output), scale_bc [B,C] (demod)
//   -> planes [rows = B*(H+1)*(W+1)][4*C]: column block ph = a*2+b holds
//      scale * g[b, c, 2m+a, 2n+b]  at row (b, m, n)   (zero where 2m+a > 2H or 2n+b > 2W)
// so that dgrad / wgrad of the polyphase conv are again row-shift GEMMs over ONE matrix.
// grid: (ceil(Hp*Wp/32), C/64, B*4), block 256 — same smem transpose as prep_keys.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
prep_phase_keys_kernel(const float* __restrict__ g, const float* __restrict__ scale, int C, int H,
                       int W, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  __shared__ float tile[64][33];
  const int Hp = H + 1, Wp = W + 1, Ht = 2 * H + 1, Wt = 2 * W + 1;
  const int img = Hp * Wp;
  const int p0 = blockIdx.x * 32;
  const int c0 = blockIdx.y * 64;
  const int b = blockIdx.z >> 2, ph = blockIdx.z & 3;
  const int pa = ph >> 1, pb = ph & 1;
  const int t = threadIdx.x;
  {
    const int pl = t & 31;
    const int p = p0 + pl;
    const int m = p / Wp, n = p - m * Wp;
    const int ty = 2 * m + pa, tx = 2 * n + pb;
    const bool valid = (p < img) && (ty < Ht) && (tx < Wt);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int cl = (t >> 5) + 8 * i;
      float v = 0.f;
      if (valid) {
        const size_t gi = ((static_cast<size_t>(b) * C + c0 + cl) * Ht + ty) * Wt + tx;
        const float s = scale ? __ldg(scale + static_cast<size_t>(b) * C + c0 + cl) : 1.f;
        v = s * __ldg(g + gi);
      }
      tile[cl][pl] = v;
    }
  }
  __syncthreads();
  {
    const int pl = t >> 3;
    const int cg = (t & 7) * 8;
    const int p = p0 + pl;
    if (p < img) {
      __align__(16) __nv_bfloat16 h[8];
      __align__(16) __nv_bfloat16 l[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) split_bf16(tile[cg + j][pl], h[j], l[j]);
      const size_t row = static_cast<size_t>(b) * img + p;
      const size_t off = row * (4 * static_cast<size_t>(C)) + static_cast<size_t>(ph) * C + c0 + cg;
      *reinterpret_cast<uint4*>(hi + off) = *reinterpret_cast<const uint4*>(h);
      *reinterpret_cast<uint4*>(lo + off) = *reinterpret_cast<const uint4*>(l);
    }
  }
}

// ---------------------------------------------------------------------------
// split_rows: fp32 -> bf16 hi/lo planes, same shape (generic RunningSecondMoment
// input [N, C], runningstats.py:1086)
// ---------------------------------------------------------------------------
__global__ void split_rows_kernel(const float* __restrict__ a, long long n,
                                  __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const long long i4 = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i4 + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(a + i4);
    __align__(8) __nv_bfloat16 h[4];
    __align__(8) __nv_bfloat16 l[4];
    split_bf16(v.x, h[0], l[0]);
    split_bf16(v.y, h[1], l[1]);
    split_bf16(v.z, h[2], l[2]);
    split_bf16(v.w, h[3], l[3]);
    *reinterpret_cast<uint2*>(hi + i4) = *reinterpret_cast<const uint2*>(h);
    *reinterpret_cast<uint2*>(lo + i4) = *reinterpret_cast<const uint2*>(l);
  } else {
    for (long long i = i4; i < n; ++i) split_bf16(a[i], hi[i], lo[i]);
  }
}

// ---------------------------------------------------------------------------
// prep_weights: W[Cout][Cin][3][3] fp32 -> (scale*W) as bf16 hi/lo planes
//   transpose_io = 0: Wt[o][tap][i]            (forward conv / conv_transpose)
//   transpose_io = 1: Wt[i][tap'][o]           (dgrad), tap' = 8 - tap if flip
//   transpose_io = 2: Wt[o/16][o%16/8][tap][o%8][i]   (fused upsampling conv, upconv_tc.cu)
// and wsq[o][i] = sum_taps (scale*W)^2   (for demod, models.py:325-327)
// one thread per (o, i)
// ---------------------------------------------------------------------------
__global__ void prep_weights_kernel(const float* __restrict__ w, int Cout, int Cin, float scale,
                                    int transpose_io, int flip_taps,
                                    __nv_bfloat16* __restrict__ wt_hi,
                                    __nv_bfloat16* __restrict__ wt_lo, float* __restrict__ wsq) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= Cout * Cin) return;
  const int o = idx / Cin, i = idx - o * Cin;
  const float* src = w + static_cast<size_t>(idx) * 9;
  float ss = 0.f;
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const float v = scale * src[tap];
    ss += v * v;
    __nv_bfloat16 h, l;
    split_bf16(v, h, l);
    size_t dst;
    if (!transpose_io) {
      dst = (static_cast<size_t>(o) * 9 + tap) * Cin + i;
    } else if (transpose_io == 2) {     // [Cout/16][half][tap][8][Cin]: the fused up-conv's N = 144
      // tiles; an epilogue warp reads the 72 columns of its channel half with two wide TMEM loads
      dst = (((static_cast<size_t>(o >> 4) * 2 + ((o >> 3) & 1)) * 9 + tap) * 8 + (o & 7)) * Cin + i;
    } else {
      const int tp = flip_taps ? 8 - tap : tap;
      dst = (static_cast<size_t>(i) * 9 + tp) * Cout + o;
    }
    wt_hi[dst] = h;
    wt_lo[dst] = l;
  }
  if (wsq) wsq[idx] = ss;
}

// ---------------------------------------------------------------------------
// demod[b,o] = rsqrt(sum_i style[b,i]^2 * wsq[o,i] + eps)      one warp per (b,o)
// ---------------------------------------------------------------------------
__global__ void demod_kernel(const float* __restrict__ style, const float* __restrict__ wsq, int B,
                             int Cout, int Cin, float eps, float* __restrict__ demod) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= B * Cout) return;
  const int b = gw / Cout, o = gw - b * Cout;
  const float* s = style + static_cast<size_t>(b) * Cin;
  const float* q = wsq + static_cast<size_t>(o) * Cin;
  float acc = 0.f;
  for (int i = lane; i < Cin; i += 32) {
    const float sv = __ldg(s + i);
    acc = fmaf(sv * sv, __ldg(q + i), acc);
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0) demod[gw] = rsqrtf(acc + eps);
}

// ---------------------------------------------------------------------------
// blur_up_act: second half of an upsampling StyledConv.
//   t [B,C,2H+1,2W+1] (conv_transpose output, already demodulated)
//   y = act( FIR4x4(pad(t,1,1)) + noise_w*noise + bias )          [B,C,2H,2W]
// (BlurF pad=(1,1): models.py:275-281,468-485; then NoiseInjectionF, FusedLeakyReLUF)
// block = 32x8 outputs, smem tile with 3-pixel halo.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
blur_up_act_kernel(const float* __restrict__ t, int C, int Ht, int Wt, const float* __restrict__ k4,
                   const float* __restrict__ noise, long long noise_bstride,
                   const float* __restrict__ noise_w, const float* __restrict__ bias, int act,
                   float* __restrict__ y) {
  constexpr int TX = 32, TY = 8;
  __shared__ float tile[TY + 3][TX + 3];
  __shared__ float kf[16];
  const int Ho = Ht - 1, Wo = Wt - 1;
  const int bc = blockIdx.z;
  const int b = bc / C, c = bc - b * C;
  const int ox0 = blockIdx.x * TX, oy0 = blockIdx.y * TY;
  const int tid = threadIdx.y * TX + threadIdx.x;
  // upfirdn2d correlates the padded signal with the *flipped* kernel
  if (tid < 16) kf[tid] = __ldg(k4 + 15 - tid);
  const float* src = t + static_cast<size_t>(bc) * Ht * Wt;
  for (int i = tid; i < (TY + 3) * (TX + 3); i += TX * TY) {
    const int ly = i / (TX + 3), lx = i - ly * (TX + 3);
    const int iy = oy0 + ly - 1, ix = ox0 + lx - 1;  // pad 1 on the low side
    float v = 0.f;
    if (iy >= 0 && iy < Ht && ix >= 0 && ix < Wt) v = __ldg(src + static_cast<size_t>(iy) * Wt + ix);
    tile[ly][lx] = v;
  }
  __syncthreads();
  const int ox = ox0 + threadIdx.x, oy = oy0 + threadIdx.y;
  if (ox >= Wo || oy >= Ho) return;
  float acc = 0.f;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int bb = 0; bb < 4; ++bb)
      acc = fmaf(tile[threadIdx.y + a][threadIdx.x + bb], kf[a * 4 + bb], acc);
  if (noise) acc += __ldg(noise_w) * __ldg(noise + static_cast<size_t>(b) * noise_bstride +
                                    static_cast<size_t>(oy) * Wo + ox);
  if (bias) acc += __ldg(bias + c);
  if (act) acc = (acc > 0.f ? acc : 0.2f * acc) * 1.4142135623730951f;
  y[(static_cast<size_t>(bc) * Ho + oy) * Wo + ox] = acc;
}

// ---------------------------------------------------------------------------
// upfirdn2d (generic, minor == 1 as called by the reference):
//   zero-insert upsample, pad/crop, correlate with flipped kernel, decimate.
// (op/upfirdn2d.py:152-186 defines the semantics; upfirdn2d_kernel.cu:52-137
//  is the reference's tiled implementation.)  One thread per output sample.
// ---------------------------------------------------------------------------
__global__ void upfirdn2d_kernel(const float* __restrict__ in, const float* __restrict__ kern,
                                 int in_h, int in_w, int kh, int kw, int up_x, int up_y,
                                 int down_x, int down_y, int px0, int py0, float* __restrict__ out,
                                 int out_h, int out_w, long long total) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int ox = static_cast<int>(idx % out_w);
  const long long r = idx / out_w;
  const int oy = static_cast<int>(r % out_h);
  const long long mj = r / out_h;
  const float* src = in + mj * in_h * in_w;
  float acc = 0.f;
  for (int ky = 0; ky < kh; ++ky) {
    const int uy = oy * down_y + ky - py0;
    if (uy < 0 || uy % up_y != 0) continue;
    const int iy = uy / up_y;
    if (iy >= in_h) continue;
    for (int kx = 0; kx < kw; ++kx) {
      const int ux = ox * down_x + kx - px0;
      if (ux < 0 || ux % up_x != 0) continue;
      const int ix = ux / up_x;
      if (ix >= in_w) continue;
      acc = fmaf(__ldg(src + static_cast<size_t>(iy) * in_w + ix),
                 __ldg(kern + (kh - 1 - ky) * kw + (kw - 1 - kx)), acc);
    }
  }
  out[idx] = acc;
}

// ---------------------------------------------------------------------------
// bias_act: y = act(x + b[(i/step_b)%size_b]) * scale with the reference's
// act/grad switch (op/fused_bias_act_kernel.cu:19-49): act 1 = linear,
// 3 = lrelu(alpha); grad 0 = forward, 1 = gate by sign of `ref`, 2 = zero.
// ---------------------------------------------------------------------------
__global__ void bias_act_kernel(const float* __restrict__ x, const float* __restrict__ b,
                                const float* __restrict__ ref, int act, int grad, float alpha,
                                float scale, long long n, int step_b, int size_b,
                                float* __restrict__ y) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += stride) {
    float v = x[i];
    if (b) v += __ldg(b + (i / step_b) % size_b);
    const float r = ref ? ref[i] : 0.f;
    float o;
    if (grad == 2) {
      o = 0.f;
    } else if (act == 3) {
      const float g = (grad == 1) ? r : v;
      o = (g > 0.f) ? v : v * alpha;
    } else {
      o = v;
    }
    y[i] = o * scale;
  }
}

// ---------------------------------------------------------------------------
// torgb: out[b,c,p] = sum_i (scale * w[c,i] * style[b,i]) * x[b,i,p] + bias[c] (+ skip[b,c,p])
// (ToRGBF + ModulatedConv2d(demodulate=False, k=1): models.py:394-425,628-655)
// block = 256 pixels of one sample; modulated weights staged in smem.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
torgb_kernel(const float* __restrict__ x, const float* __restrict__ style,
             const float* __restrict__ w, const float* __restrict__ bias,
             const float* __restrict__ skip, int C, int HW, float scale, float* __restrict__ out) {
  extern __shared__ float wm[];  // [3][C]
  const int b = blockIdx.y;
  for (int i = threadIdx.x; i < 3 * C; i += blockDim.x) {
    const int ci = i % C;
    wm[i] = (scale * __ldg(w + i)) * __ldg(style + static_cast<size_t>(b) * C + ci);
  }
  __syncthreads();
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const float* xb = x + static_cast<size_t>(b) * C * HW + p;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 4
  for (int i = 0; i < C; ++i) {
    const float v = __ldg(xb + static_cast<size_t>(i) * HW);
    a0 = fmaf(wm[i], v, a0);
    a1 = fmaf(wm[C + i], v, a1);
    a2 = fmaf(wm[2 * C + i], v, a2);
  }
  float* ob = out + static_cast<size_t>(b) * 3 * HW + p;
  const float* sb = skip ? skip + static_cast<size_t>(b) * 3 * HW + p : nullptr;
  a0 += __ldg(bias + 0);
  a1 += __ldg(bias + 1);
  a2 += __ldg(bias + 2);
  if (sb) { a0 += sb[0]; a1 += sb[HW]; a2 += sb[2 * static_cast<size_t>(HW)]; }
  ob[0] = a0;
  ob[HW] = a1;
  ob[2 * static_cast<size_t>(HW)] = a2;
}

// y[b,c,p] = x[b,c,p] + noise_w * noise[b,p]     (NoiseInjectionF, models.py:535-546)
__global__ void add_noise_kernel(const float* __restrict__ x, const float* __restrict__ noise,
                                 long long noise_bstride, const float* __restrict__ noise_w_p,
                                 int C, int HW,
                                 long long total, float* __restrict__ y) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const float noise_w = __ldg(noise_w_p);
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += stride) {
    const int p = static_cast<int>(i % HW);
    const long long b = i / (static_cast<long long>(HW) * C);
    y[i] = x[i] + noise_w * __ldg(noise + b * noise_bstride + p);
  }
}

// ---------------------------------------------------------------------------
// blur_up_fused: generation fast path for an upsampling StyledConv.
//   t_cl  [4 phases][rows_in][C] fp32 channels-last (conv_tc out_mode 1; phase = (ty&1)*2+(tx&1),
//         row = (b*(H+1) + ty/2)*(W+1) + tx/2) — the conv_transpose output, demodulated
//   v = act( FIR4x4(pad(t,1,1)) + noise_w*noise + bias )                       (as blur_up_act)
//   -> next layer's key planes  split_bf16(next_scale[b,c] * v)  over the padded-flat grid of
//      the OUTPUT resolution (pad row / column written as zeros), optional fp32 NCHW copy.
// block: 4*QD channels (QD = 16, or 8 when C % 64 != 0) x (8 x 16) outputs, 16*QD threads;
// thread = (pixel group, channel quad); float4 smem reads.
// ---------------------------------------------------------------------------
constexpr int BF_TY = 8, BF_TX = 16, BF_C = 64;
constexpr int BF_PW = BF_TX + 3, BF_PH = BF_TY + 3;

template <int QD>
__global__ void __launch_bounds__(16 * QD, 4)
blur_up_fused_kernel(const float* __restrict__ t_cl, int B, int C, int H, int W,
                     const float* __restrict__ k4, const float* __restrict__ noise,
                     long long noise_bstride, const float* __restrict__ noise_w,
                     const float* __restrict__ bias, int act,
                     const float* __restrict__ next_scale, __nv_bfloat16* __restrict__ next_hi,
                     __nv_bfloat16* __restrict__ next_lo, float* __restrict__ y_out) {
  extern __shared__ float4 tile4[];      // [BF_PH*BF_PW][QD quads]
  __shared__ float kf[16];
  constexpr int kC = 4 * QD;
  const int Ho = 2 * H, Wo = 2 * W;
  const int Hp_in = H + 1, Wp_in = W + 1;
  const long long rows_in = static_cast<long long>(B) * Hp_in * Wp_in;
  const int cblocks = C / kC;
  const int b = blockIdx.z / cblocks;
  const int c0 = (blockIdx.z - b * cblocks) * kC;
  const int ox0 = blockIdx.x * BF_TX, oy0 = blockIdx.y * BF_TY;
  const int tid = threadIdx.x;
  if (tid < 16) kf[tid] = __ldg(k4 + 15 - tid);   // flipped kernel (upfirdn2d correlates)
  for (int i = tid; i < BF_PH * BF_PW * QD; i += 16 * QD) {
    const int qd = i % QD;
    const int pos = i / QD;
    const int ly = pos / BF_PW, lx = pos - ly * BF_PW;
    const int ty = oy0 + ly - 1, tx = ox0 + lx - 1;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ty >= 0 && ty <= Ho && tx >= 0 && tx <= Wo) {
      const int ph = (ty & 1) * 2 + (tx & 1);
      const long long row = (static_cast<long long>(b) * Hp_in + (ty >> 1)) * Wp_in + (tx >> 1);
      v = __ldg(reinterpret_cast<const float4*>(t_cl + (ph * rows_in + row) * C + c0) + qd);
    }
    tile4[i] = v;
  }
  __syncthreads();
  const int qd = tid % QD;
  const int grp = tid / QD;                 // 16 groups of 8 pixels
  const int ly = grp >> 1;
  const int lx0 = (grp & 1) * 8;
  const int oy = oy0 + ly;
  if (oy > Ho) return;
  const int c = c0 + qd * 4;
  const float nw = noise ? __ldg(noise_w) : 0.f;
  float4 bs = make_float4(0.f, 0.f, 0.f, 0.f);
  if (bias) bs = __ldg(reinterpret_cast<const float4*>(bias + c));
  float4 sc = make_float4(1.f, 1.f, 1.f, 1.f);
  if (next_scale) sc = __ldg(reinterpret_cast<const float4*>(next_scale + static_cast<size_t>(b) * C + c));
  const size_t out_row0 = (static_cast<size_t>(b) * (Ho + 1) + oy) * (Wo + 1);

  // 8 consecutive outputs of one row: slide over 11 input columns per filter row, so every
  // smem value is read once (44 LDS.128 instead of 128) — the kernel is smem-bound otherwise.
  float4 a[8];
#pragma unroll
  for (int px = 0; px < 8; ++px) a[px] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int fy = 0; fy < 4; ++fy) {
    float4 tv[11];
#pragma unroll
    for (int i = 0; i < 11; ++i) tv[i] = tile4[((ly + fy) * BF_PW + lx0 + i) * QD + qd];
#pragma unroll
    for (int fx = 0; fx < 4; ++fx) {
      const float kk = kf[fy * 4 + fx];
#pragma unroll
      for (int px = 0; px < 8; ++px) {
        a[px].x = fmaf(tv[px + fx].x, kk, a[px].x);
        a[px].y = fmaf(tv[px + fx].y, kk, a[px].y);
        a[px].z = fmaf(tv[px + fx].z, kk, a[px].z);
        a[px].w = fmaf(tv[px + fx].w, kk, a[px].w);
      }
    }
  }
#pragma unroll
  for (int px = 0; px < 8; ++px) {
    const int ox = ox0 + lx0 + px;
    if (ox > Wo) break;
    float4 v = a[px];
    const bool real = (oy < Ho) && (ox < Wo);
    if (real) {
      if (noise) {
        const float nz = nw * __ldg(noise + static_cast<size_t>(b) * noise_bstride +
                                    static_cast<size_t>(oy) * Wo + ox);
        v.x += nz; v.y += nz; v.z += nz; v.w += nz;
      }
      v.x += bs.x; v.y += bs.y; v.z += bs.z; v.w += bs.w;
      if (act) {
        v.x = (v.x > 0.f ? v.x : 0.2f * v.x) * 1.4142135623730951f;
        v.y = (v.y > 0.f ? v.y : 0.2f * v.y) * 1.4142135623730951f;
        v.z = (v.z > 0.f ? v.z : 0.2f * v.z) * 1.4142135623730951f;
        v.w = (v.w > 0.f ? v.w : 0.2f * v.w) * 1.4142135623730951f;
      }
      if (y_out) {
        const size_t hw = static_cast<size_t>(Ho) * Wo;
        float* yp = y_out + (static_cast<size_t>(b) * C + c) * hw + static_cast<size_t>(oy) * Wo + ox;
        yp[0] = v.x; yp[hw] = v.y; yp[2 * hw] = v.z; yp[3 * hw] = v.w;
      }
    }
    if (next_hi) {
      const float k0 = real ? sc.x * v.x : 0.f, k1 = real ? sc.y * v.y : 0.f;
      const float k2 = real ? sc.z * v.z : 0.f, k3 = real ? sc.w * v.w : 0.f;
      const __nv_bfloat162 h01 = __floats2bfloat162_rn(k0, k1), h23 = __floats2bfloat162_rn(k2, k3);
      const float2 f01 = __bfloat1622float2(h01), f23 = __bfloat1622float2(h23);
      const __nv_bfloat162 l01 = __floats2bfloat162_rn(k0 - f01.x, k1 - f01.y);
      const __nv_bfloat162 l23 = __floats2bfloat162_rn(k2 - f23.x, k3 - f23.y);
      const size_t off = (out_row0 + ox) * C + c;
      *reinterpret_cast<uint2*>(next_hi + off) =
          make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
      *reinterpret_cast<uint2*>(next_lo + off) =
          make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
    }
  }
}

// ---------------------------------------------------------------------------
// blur_up_pipe: blur_up_fused for the generation fast path's configuration (noise + bias +
// leaky-ReLU, output = the next layer's key planes only), rebuilt after an ncu capture of the
// one-tile-per-CTA kernel on layer 13 (profiles/: 0.84 ms, DRAM 31 %, issue slots 58 % busy, ALU
// the top pipe — 607 M warp instructions, of which the 16-tap FIR was only a third):
//  * persistent CTAs (2 per SM) walk the tile list with a static stride; tile i+1 is prefetched
//    with cp.async (16 B, zero-fill outside the image) into the second buffer while tile i is
//    filtered;
//  * index arithmetic hoisted: the (ly, lx) of a thread's 14 staging slots come from a small
//    shared table, the tile coordinate advances as a mixed-radix counter (no division in the
//    loop), channel-block fastest so that both 256-byte halves of a row move together;
//  * no per-pixel null-pointer branches (the generic kernel keeps those), leaky-ReLU as
//    max(v, 0.2 v);
//  * a rank-one 4x4 FIR (the model's [1,3,3,1] x [1,3,3,1]) is applied separably: 176 + 128
//    instead of 512 FMAs per thread.  Detected on the device (exact rank-one test), other
//    kernels take the 16-tap loop.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void st_shared_zero16(uint32_t dst) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};\n" ::"r"(dst), "f"(0.f) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

constexpr int BF_NPOS = BF_PH * BF_PW;                 // 209 staged positions per tile
static_assert((BF_TY & 1) == 0 && (BF_TX & 1) == 0 && BF_TX == 16 && BF_PW == 19,
              "the staging code below relies on odd tile origins and a 16 + 3 column split");

// mixed-radix tile coordinate: digit 0 = channel block, 1 = tile x, 2 = tile y, 3 = sample
struct BlurCoord {
  int d[4];
};

__device__ __forceinline__ BlurCoord blur_coord(unsigned t, const int (&radix)[4]) {
  BlurCoord c;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    c.d[i] = static_cast<int>(t % static_cast<unsigned>(radix[i]));
    t /= static_cast<unsigned>(radix[i]);
  }
  c.d[3] = static_cast<int>(t);
  return c;
}

__device__ __forceinline__ void blur_coord_add(BlurCoord& c, const BlurCoord& step,
                                               const int (&radix)[4]) {
  int carry = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    int v = c.d[i] + step.d[i] + carry;
    carry = v >= radix[i] ? 1 : 0;
    c.d[i] = v - (carry ? radix[i] : 0);
  }
  c.d[3] += step.d[3] + carry;
}

__global__ void __launch_bounds__(256, 2)
blur_up_pipe_kernel(const float* __restrict__ t_cl, int B, int C, int H, int W,
                    const float* __restrict__ k4, const float* __restrict__ noise,
                    long long noise_bstride, const float* __restrict__ noise_w,
                    const float* __restrict__ bias, const float* __restrict__ next_scale,
                    __nv_bfloat16* __restrict__ next_hi, __nv_bfloat16* __restrict__ next_lo,
                    int tiles_x, int tiles_y, unsigned ntiles) {
  extern __shared__ float4 tile4[];      // 2 x [BF_NPOS][16 quads]
  __shared__ float kf[16];
  __shared__ int sep_flag;
  // per-tile side data, staged with the tile so that the filter phase issues no global load
  // (ncu: the 8 noise loads per thread, each consumed at once, were the top stall):
  // [0,128) noise of the 8 x 16 outputs, [128,192) bias, [192,256) next-layer style
  __shared__ __align__(16) float side[2][256];
  constexpr int TILE_ELEMS = BF_NPOS * 16;
  const int Ho = 2 * H, Wo = 2 * W;
  const int Hp_in = H + 1, Wp_in = W + 1;
  const int rows_in = B * Hp_in * Wp_in;                 // 4 * rows_in < 2^31 (checked on the host)
  const int radix[4] = {C / BF_C, tiles_x, tiles_y, B};
  const int tid = threadIdx.x;
  if (tid < 16) kf[tid] = __ldg(k4 + 15 - tid);   // flipped kernel (upfirdn2d correlates)
  if (tid == 0) {
    // rank one  <=>  k[i][j] * k[0][0] == k[i][0] * k[0][j]  (exact for [1,3,3,1] (x) [1,3,3,1])
    bool sep = __ldg(k4 + 15) != 0.f;
    for (int a = 0; a < 4; ++a)
      for (int bb = 0; bb < 4; ++bb)
        sep = sep && (__ldg(k4 + 15 - (a * 4 + bb)) * __ldg(k4 + 15) ==
                      __ldg(k4 + 15 - a * 4) * __ldg(k4 + 15 - bb));
    sep_flag = sep ? 1 : 0;
  }
  __syncthreads();
  const uint32_t smem0 = smem_u32(tile4);
  const int qd = tid & 15;
  const int p0 = tid >> 4;

  // Staging of one tile = 11 x 19 positions x 16 channel quads.  Thread (lx = tid >> 4, qd) owns
  // column lx of all 11 rows: the tile origin (8k - 1, 16k - 1) is odd, so the row parity of slot
  // ly is a compile-time constant and the two phase pointers just advance by one input row every
  // second slot.  The last 3 columns (33 positions) are spread over the threads afterwards.
  auto issue = [&](const BlurCoord& tc, int buf) {
    const int oy0 = tc.d[2] * BF_TY - 1, ox0 = tc.d[1] * BF_TX - 1;
    const int m = tc.d[2] * (BF_TY / 2);                 // ty = 2m - 1 + ly
    const int rowb = tc.d[3] * Hp_in;
    const float* base = t_cl + tc.d[0] * BF_C + qd * 4;
    const uint32_t tile_s = smem0 + static_cast<uint32_t>(buf) * TILE_ELEMS * 16u;
    const unsigned rstride = static_cast<unsigned>(Wp_in) * static_cast<unsigned>(C);
    {
      const int lx = p0;                                  // 0..15
      const int tx = ox0 + lx;
      const bool vx = static_cast<unsigned>(tx) <= static_cast<unsigned>(Wo);
      const int pb = tx & 1, txh = tx >> 1;
      // odd rows (ly even): phase 2+pb, input row m-1 + ly/2 ; even rows (ly odd): phase pb, row m + ly/2
      const unsigned i1 = static_cast<unsigned>((2 + pb) * rows_in + (rowb + m - 1) * Wp_in + txh);
      const unsigned i0 = static_cast<unsigned>(pb * rows_in + (rowb + m) * Wp_in + txh);
      const float* p1 = base + static_cast<unsigned long long>(i1) * static_cast<unsigned>(C);
      const float* pe = base + static_cast<unsigned long long>(i0) * static_cast<unsigned>(C);
      const uint32_t dst = tile_s + static_cast<uint32_t>(lx * 16 + qd) * 16u;
#pragma unroll
      for (int l = 0; l < BF_PH; ++l) {
        const int ty = oy0 + l;
        const bool valid = vx && (static_cast<unsigned>(ty) <= static_cast<unsigned>(Ho));
        const float* src = ((l & 1) ? pe : p1) + static_cast<size_t>(l >> 1) * rstride;
        const uint32_t d = dst + static_cast<uint32_t>(l * BF_PW * 16) * 16u;
        if (valid) cp_async16(d, src); else st_shared_zero16(d);
      }
    }
#pragma unroll
    for (int e0 = 0; e0 < 3 * BF_PH * 16; e0 += 256) {     // columns 16..18: 528 quads
      const int e = e0 + tid;
      if (e < 3 * BF_PH * 16) {
        const int r = e >> 4;                              // 0..32 = ly * 3 + (lx - 16)
        const int l = r / 3, lx = 16 + (r - l * 3);
        const int ty = oy0 + l, tx = ox0 + lx;
        const bool valid = (static_cast<unsigned>(ty) <= static_cast<unsigned>(Ho)) &&
                           (static_cast<unsigned>(tx) <= static_cast<unsigned>(Wo));
        const unsigned idx = static_cast<unsigned>((((ty & 1) << 1) | (tx & 1)) * rows_in +
                                                   (rowb + (ty >> 1)) * Wp_in + (tx >> 1));
        const float* src = base + static_cast<unsigned long long>(idx) * static_cast<unsigned>(C);
        const uint32_t d = tile_s + static_cast<uint32_t>((l * BF_PW + lx) * 16 + qd) * 16u;
        if (valid) cp_async16(d, src); else st_shared_zero16(d);
      }
    }
    {
      const uint32_t side_s = smem_u32(&side[buf][0]);
      if (tid < BF_TY * BF_TX) {
        const int oy = tc.d[2] * BF_TY + (tid >> 4), ox = tc.d[1] * BF_TX + (tid & 15);
        if (oy < Ho && ox < Wo)
          cp_async4(side_s + tid * 4u, noise + static_cast<size_t>(tc.d[3]) * noise_bstride +
                                           static_cast<size_t>(oy) * Wo + ox);
        else
          side[buf][tid] = 0.f;
      } else if (tid < BF_TY * BF_TX + 16) {
        const int q4 = (tid - BF_TY * BF_TX) * 4;
        cp_async16(side_s + (128 + q4) * 4u, bias + tc.d[0] * BF_C + q4);
      } else if (tid < BF_TY * BF_TX + 32) {
        const int q4 = (tid - BF_TY * BF_TX - 16) * 4;
        cp_async16(side_s + (192 + q4) * 4u,
                   next_scale + static_cast<size_t>(tc.d[3]) * C + tc.d[0] * BF_C + q4);
      }
    }
    cp_async_commit();
  };

  unsigned t = blockIdx.x;
  BlurCoord cur = blur_coord(t, radix);
  const BlurCoord step = blur_coord(gridDim.x, radix);
  if (t < ntiles) issue(cur, 0);
  const float nw = __ldg(noise_w);
  const int grp = tid >> 4;                 // 16 groups of 8 pixels
  const int ly = grp >> 1;
  const int lx0 = (grp & 1) * 8;
  const bool sep = sep_flag != 0;
  // horizontal taps of the rank-one kernel, k[fy][fx] = k[fy][0] * (k[0][fx] / k[0][0]); computed
  // once (the division was 10 % of the kernel's instructions when it sat inside the tile loop)
  const float inv = sep ? 1.f / kf[0] : 0.f;
  const float kx0 = 1.f, kx1 = kf[1] * inv, kx2 = kf[2] * inv, kx3 = kf[3] * inv;
  int buf = 0;
  for (; t < ntiles; t += gridDim.x, buf ^= 1) {
    BlurCoord nxt = cur;
    blur_coord_add(nxt, step, radix);
    if (t + gridDim.x < ntiles) {
      issue(nxt, buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();                         // tile t has landed for every thread
    const float4* tl = tile4 + buf * TILE_ELEMS;
    const int b = cur.d[3];
    const int oy = cur.d[2] * BF_TY + ly;
    const int oxb = cur.d[1] * BF_TX + lx0;
    if (oy <= Ho && oxb <= Wo) {
      const int c = cur.d[0] * BF_C + qd * 4;
      float4 a[8];
      if (sep) {
        // vertical pass over the 11 columns this thread needs, then 4 horizontal taps per output
        float4 v[11];
#pragma unroll
        for (int i = 0; i < 11; ++i) v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int fy = 0; fy < 4; ++fy) {
          const float ky = kf[fy * 4];
#pragma unroll
          for (int i = 0; i < 11; ++i) {
            const float4 tv = tl[((ly + fy) * BF_PW + lx0 + i) * 16 + qd];
            v[i].x = fmaf(tv.x, ky, v[i].x);
            v[i].y = fmaf(tv.y, ky, v[i].y);
            v[i].z = fmaf(tv.z, ky, v[i].z);
            v[i].w = fmaf(tv.w, ky, v[i].w);
          }
        }
#pragma unroll
        for (int px = 0; px < 8; ++px) {
          a[px].x = fmaf(v[px + 3].x, kx3, fmaf(v[px + 2].x, kx2, fmaf(v[px + 1].x, kx1, v[px].x * kx0)));
          a[px].y = fmaf(v[px + 3].y, kx3, fmaf(v[px + 2].y, kx2, fmaf(v[px + 1].y, kx1, v[px].y * kx0)));
          a[px].z = fmaf(v[px + 3].z, kx3, fmaf(v[px + 2].z, kx2, fmaf(v[px + 1].z, kx1, v[px].z * kx0)));
          a[px].w = fmaf(v[px + 3].w, kx3, fmaf(v[px + 2].w, kx2, fmaf(v[px + 1].w, kx1, v[px].w * kx0)));
        }
      } else {
#pragma unroll
        for (int px = 0; px < 8; ++px) a[px] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int fy = 0; fy < 4; ++fy) {
          float4 tv[11];
#pragma unroll
          for (int i = 0; i < 11; ++i) tv[i] = tl[((ly + fy) * BF_PW + lx0 + i) * 16 + qd];
#pragma unroll
          for (int fx = 0; fx < 4; ++fx) {
            const float kk = kf[fy * 4 + fx];
#pragma unroll
            for (int px = 0; px < 8; ++px) {
              a[px].x = fmaf(tv[px + fx].x, kk, a[px].x);
              a[px].y = fmaf(tv[px + fx].y, kk, a[px].y);
              a[px].z = fmaf(tv[px + fx].z, kk, a[px].z);
              a[px].w = fmaf(tv[px + fx].w, kk, a[px].w);
            }
          }
        }
      }
      const float4 bs = *reinterpret_cast<const float4*>(&side[buf][128 + qd * 4]);
      const float4 sc = *reinterpret_cast<const float4*>(&side[buf][192 + qd * 4]);
      const bool rowreal = oy < Ho;
      const float* nrow = &side[buf][ly * BF_TX + lx0];
      const size_t off0 = ((static_cast<size_t>(b) * (Ho + 1) + oy) * (Wo + 1) + oxb) * C + c;
      __nv_bfloat16* ph = next_hi + off0;
      __nv_bfloat16* pl = next_lo + off0;
#pragma unroll
      for (int px = 0; px < 8; ++px) {
        const int ox = oxb + px;
        if (ox > Wo) break;
        uint2 hv = make_uint2(0u, 0u), lv = make_uint2(0u, 0u);   // pad row / column: zeros
        if (rowreal && ox < Wo) {
          const float nz = nw * nrow[px];
          float v0 = (a[px].x + nz) + bs.x, v1 = (a[px].y + nz) + bs.y;
          float v2 = (a[px].z + nz) + bs.z, v3 = (a[px].w + nz) + bs.w;
          v0 = fmaxf(v0, 0.2f * v0) * 1.4142135623730951f;        // leaky-ReLU(0.2) * sqrt(2)
          v1 = fmaxf(v1, 0.2f * v1) * 1.4142135623730951f;
          v2 = fmaxf(v2, 0.2f * v2) * 1.4142135623730951f;
          v3 = fmaxf(v3, 0.2f * v3) * 1.4142135623730951f;
          const float k0 = sc.x * v0, k1 = sc.y * v1, k2 = sc.z * v2, k3 = sc.w * v3;
          const __nv_bfloat162 h01 = __floats2bfloat162_rn(k0, k1), h23 = __floats2bfloat162_rn(k2, k3);
          const uint32_t u01 = *reinterpret_cast<const uint32_t*>(&h01);
          const uint32_t u23 = *reinterpret_cast<const uint32_t*>(&h23);
          // bf16 -> fp32 is a 16-bit shift: low half = first element
          const __nv_bfloat162 l01 = __floats2bfloat162_rn(k0 - __uint_as_float(u01 << 16),
                                                           k1 - __uint_as_float(u01 & 0xffff0000u));
          const __nv_bfloat162 l23 = __floats2bfloat162_rn(k2 - __uint_as_float(u23 << 16),
                                                           k3 - __uint_as_float(u23 & 0xffff0000u));
          hv = make_uint2(u01, u23);
          lv = make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
        }
        *reinterpret_cast<uint2*>(ph + static_cast<size_t>(px) * C) = hv;
        *reinterpret_cast<uint2*>(pl + static_cast<size_t>(px) * C) = lv;
      }
    }
    __syncthreads();                         // buffer `buf` is free for the prefetch of pass +1
    cur = nxt;
  }
}

// ---------------------------------------------------------------------------
// rgb_combine: out[b,c,y,x] = sum_nt part[nt][b][c][y][x] + bias[c] + Up2(prev)[b,c,y,x]
// (ToRGBF's `+ bias + skip` with the skip's UpsampleO = upfirdn2d(up=2, pad=(2,1)) inline;
//  models.py:435-447,639-655).  3-channel tensors: negligible traffic.
// ---------------------------------------------------------------------------
// grid (x quads, y, b*3+c), one thread = 4 consecutive x of one row (float4 partial loads / store);
// no integer division on the index path (the flat-index version spent its time in 64-bit div/mod).
__global__ void __launch_bounds__(256)
rgb_combine_kernel(const float* __restrict__ part, int nparts, long long part_stride, int H, int W,
                   const float* __restrict__ bias, const float* __restrict__ prev,
                   const float* __restrict__ k4, float* __restrict__ out,
                   uint8_t* __restrict__ out_u8) {
  const int xq = blockIdx.x * blockDim.x + threadIdx.x;          // quad index along x
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  const int bc = blockIdx.z;
  const int x0 = xq * 4;
  if (x0 >= W || y >= H) return;
  const size_t row = (static_cast<size_t>(bc) * H + y) * W + x0;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int n = 0; n < nparts; ++n) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(part + n * part_stride + row));
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  const float bv = __ldg(bias + bc % 3);
  acc.x += bv; acc.y += bv; acc.z += bv; acc.w += bv;
  if (prev) {
    // UpsampleO = upfirdn2d(up 2, pad (2,1)): out(y,x) = sum over taps with (y+ky-2), (x+kx-2)
    // even of prev[(y+ky)/2-1, (x+kx)/2-1] * k4[3-ky][3-kx]: 2 x 2 taps per output.  The four
    // outputs x0..x0+3 touch prev columns c-1..c+2 (c = x0/2) of two rows.
    const int h2 = H >> 1, w2 = W >> 1;
    const int c = x0 >> 1;
    const float* src = prev + static_cast<size_t>(bc) * h2 * w2;
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int ky = (y & 1) + 2 * j;
      const int iy = ((y + ky) >> 1) - 1;
      if (iy < 0 || iy >= h2) continue;
      const float* r = src + static_cast<size_t>(iy) * w2;
      const float pm = (c - 1 >= 0) ? __ldg(r + c - 1) : 0.f;
      const float p0 = __ldg(r + c);
      const float p1 = (c + 1 < w2) ? __ldg(r + c + 1) : 0.f;
      const float p2 = (c + 2 < w2) ? __ldg(r + c + 2) : 0.f;
      const float* kr = k4 + (3 - ky) * 4;
      const float w0 = __ldg(kr + 0), w1 = __ldg(kr + 1), w2k = __ldg(kr + 2), w3 = __ldg(kr + 3);
      // even x: kx = 0 -> column 3 of the kernel row, kx = 2 -> column 1; odd x: kx = 1 -> 2, 3 -> 0
      u.x = fmaf(pm, w3, fmaf(p0, w1, u.x));      // x0   : prev c-1 (kx 0), c   (kx 2)
      u.y = fmaf(p0, w2k, fmaf(p1, w0, u.y));     // x0+1 : prev c   (kx 1), c+1 (kx 3)
      u.z = fmaf(p0, w3, fmaf(p1, w1, u.z));      // x0+2 : prev c   (kx 0), c+1 (kx 2)
      u.w = fmaf(p1, w2k, fmaf(p2, w0, u.w));     // x0+3 : prev c+1 (kx 1), c+2 (kx 3)
    }
    acc.x += u.x; acc.y += u.y; acc.z += u.z; acc.w += u.w;
  }
  if (out) *reinterpret_cast<float4*>(out + row) = acc;
  if (out_u8) {
    // NHWC bytes of the final image: clamp(x * 127.5 + 127.5, 0, 255) truncated, i.e. exactly
    // (img * 127.5 + 127.5).clamp(0, 255).byte() (separate multiply and add: no fma contraction)
    const int b = bc / 3, c = bc - 3 * b;
    uint8_t* dst = out_u8 + ((static_cast<size_t>(b) * H + y) * W + x0) * 3 + c;
    const float v[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float s = fminf(fmaxf(__fadd_rn(__fmul_rn(v[i], 127.5f), 127.5f), 0.f), 255.f);
      dst[3 * i] = static_cast<uint8_t>(s);
    }
  }
}

// z * rsqrt(mean(z^2, dim=1) + 1e-8)   (PixelNormL, models.py:609-614); one warp per row
__global__ void pixel_norm_kernel(const float* __restrict__ z, int B, int K, float* __restrict__ out) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= B) return;
  const float* src = z + static_cast<size_t>(row) * K;
  float ss = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float v = __ldg(src + k);
    ss = fmaf(v, v, ss);
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
  const float r = rsqrtf(ss / static_cast<float>(K) + 1e-8f);
  for (int k = lane; k < K; k += 32) out[static_cast<size_t>(row) * K + k] = __ldg(src + k) * r;
}

// ---------------------------------------------------------------------------
// demod_multi: the demodulation factors of EVERY styled conv of the generator in one launch
// (they only depend on the styles), plus the ToRGB modulated 1x1 weights
//   kind 0: out[b,o]   = rsqrt(sum_i style[b,i]^2 * wsq[o,i] + eps)        one warp per (o, 8 samples)
//   kind 1: out[b,c,i] = (wscale * w[c,i]) * style[b,i]   (c < 3; `wsq` holds w) one warp per (b,c)
// ---------------------------------------------------------------------------
struct DemodJobs {
  const float* style[32];
  const float* wsq[32];
  float* out[32];
  int cout[32];
  int cin[32];
  int kind[32];
  float wscale[32];
  int first_block[33];
  int n;
};

__global__ void __launch_bounds__(256)
demod_multi_kernel(int B, float eps, const DemodJobs jobs) {
  int l = 0;
  const int blk = blockIdx.x;
  while (blk >= jobs.first_block[l + 1]) ++l;
  const int unit = (blk - jobs.first_block[l]) * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int Cout = jobs.cout[l], Cin = jobs.cin[l];
  if (jobs.kind[l] == 1) {                       // unit = (b, c): one modulated ToRGB weight row
    if (unit >= B * Cout) return;
    const int b = unit / Cout, o = unit - b * Cout;
    const float* s = jobs.style[l] + static_cast<size_t>(b) * Cin;
    const float* q = jobs.wsq[l] + static_cast<size_t>(o) * Cin;
    const float ws = jobs.wscale[l];
    float* dst = jobs.out[l] + static_cast<size_t>(unit) * Cin;
    for (int i = lane; i < Cin; i += 32) dst[i] = (ws * __ldg(q + i)) * __ldg(s + i);
    return;
  }
  // kind 0, unit = (output channel o, group of 8 samples): the wsq row is read once into
  // registers and reused for the group's samples.  (One warp per (b,o) re-read all of wsq B
  // times from L2: 48 us; one warp per o walking all B samples serially: 70 us.)
  const int nbg = (B + 7) >> 3;
  if (unit >= Cout * nbg) return;
  const int o = unit / nbg;
  const int b_lo = (unit - o * nbg) * 8;
  const int b_hi = min(B, b_lo + 8);
  const float* q = jobs.wsq[l] + static_cast<size_t>(o) * Cin;
  float* out = jobs.out[l];
  const int nk = (Cin + 31) >> 5;
  if (nk <= 16) {
    float qv[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int i = lane + 32 * j;
      qv[j] = (i < Cin) ? __ldg(q + i) : 0.f;
    }
#pragma unroll 2
    for (int b = b_lo; b < b_hi; ++b) {
      const float* s = jobs.style[l] + static_cast<size_t>(b) * Cin;
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int i = lane + 32 * j;
        if (i < Cin) {
          const float sv = __ldg(s + i);
          acc = fmaf(sv * sv, qv[j], acc);
        }
      }
#pragma unroll
      for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
      if (lane == 0) out[static_cast<size_t>(b) * Cout + o] = rsqrtf(acc + eps);
    }
  } else {
    for (int b = b_lo; b < b_hi; ++b) {
      const float* s = jobs.style[l] + static_cast<size_t>(b) * Cin;
      float acc = 0.f;
      for (int i = lane; i < Cin; i += 32) {
        const float sv = __ldg(s + i);
        acc = fmaf(sv * sv, __ldg(q + i), acc);
      }
#pragma unroll
      for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
      if (lane == 0) out[static_cast<size_t>(b) * Cout + o] = rsqrtf(acc + eps);
    }
  }
}

// ---------------------------------------------------------------------------
// small_gemm: out[b, o] = epi( sum_i f(A[b, i]) * W[o, i] ) for several (A, W, out) jobs in one
// launch — the latent-only linears of the generator at ANY batch size:
//   mode 0 (EqualLinear / modulation, models.py:487-533):  f = id,
//          out = act( acc * scale + bias[o] * bias_mul )           act = leaky-ReLU(0.2) * sqrt(2)
//   mode 1 (demodulation factor, models.py:320-328):       f = square,
//          out = rsqrt( acc + eps )                                (W = Wsq[o, i])
// Classic shared-memory tiling: 32 batch rows x 64 output channels per block, K chunks of 32,
// 2 x 4 outputs per thread.  The warp-per-channel kernels it replaces re-staged the whole
// latent batch per block (styles) or re-read every style row per output channel (demod): at the
// 250-row passes of the covariance collection they took 0.56 ms of a 3 ms pass.
// ---------------------------------------------------------------------------
struct GemmJobs {
  const float* a[32];       // [B, a_stride] rows (row b at a + b * a_stride)
  const float* w[32];       // [N, K]
  const float* bias[32];    // [N] or null
  float* out[32];           // [B, N]
  int n_out[32];
  int first_block[33];
  int n;
};

template <int MODE>
__global__ void __launch_bounds__(256)
small_gemm_kernel(int B, int K, long long a_stride, float scale, float bias_mul, int act, float eps,
                  const GemmJobs jobs) {
  __shared__ float As[32][33];
  __shared__ float Ws[64][33];
  int l = 0;
  const int blk = blockIdx.x;
  while (blk >= jobs.first_block[l + 1]) ++l;
  const int N = jobs.n_out[l];
  const int n0 = (blk - jobs.first_block[l]) * 64;
  const int b0 = blockIdx.y * 32;
  const float* A = jobs.a[l];
  const float* Wm = jobs.w[l];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;          // 16 x 16 threads: rows 2*ty.., cols 4*tx..
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  for (int k0 = 0; k0 < K; k0 += 32) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {                   // A tile: 32 rows x 32 k
      const int e = tid + 256 * i;
      const int r = e >> 5, c = e & 31;
      float v = 0.f;
      if (b0 + r < B && k0 + c < K) v = __ldg(A + static_cast<size_t>(b0 + r) * a_stride + k0 + c);
      As[r][c] = (MODE == 1) ? v * v : v;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {                   // W tile: 64 rows x 32 k
      const int e = tid + 256 * i;
      const int r = e >> 5, c = e & 31;
      float v = 0.f;
      if (n0 + r < N && k0 + c < K) v = __ldg(Wm + static_cast<size_t>(n0 + r) * K + k0 + c);
      Ws[r][c] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 32; ++kk) {
      const float a0 = As[2 * ty][kk], a1 = As[2 * ty + 1][kk];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float wv = Ws[4 * tx + c][kk];
        acc[0][c] = fmaf(a0, wv, acc[0][c]);
        acc[1][c] = fmaf(a1, wv, acc[1][c]);
      }
    }
    __syncthreads();
  }
  float* out = jobs.out[l];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int b = b0 + 2 * ty + r;
    if (b >= B) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int o = n0 + 4 * tx + c;
      if (o >= N) continue;
      float v;
      if (MODE == 1) {
        v = rsqrtf(acc[r][c] + eps);
      } else {
        v = acc[r][c] * scale;
        if (jobs.bias[l]) v += __ldg(jobs.bias[l] + o) * bias_mul;
        if (act) v = (v > 0.f ? v : 0.2f * v) * 1.4142135623730951f;
      }
      out[static_cast<size_t>(b) * N + o] = v;
    }
  }
}

// Same jobs for B <= 32 rows (the batch-32 generation step: 8 mapping layers, styles, demod):
// the tiled kernel above runs 8 CTAs of 16 dependent load-sync-compute rounds there (31 us per
// mapping layer, ncu).  Here one WARP owns one output column for all rows: lanes stride over K in
// float4, every load of the K loop is independent, the 32 per-row partial sums are reduced by
// recursive halving (31 shuffles) so that lane b ends with row b.  8 columns per block.
template <int MODE>
__global__ void __launch_bounds__(256)
skinny_gemm_kernel(int B, int K, long long a_stride, float scale, float bias_mul, int act, float eps,
                   const GemmJobs jobs) {
  int l = 0;
  const int blk = blockIdx.x;
  while (blk >= jobs.first_block[l + 1]) ++l;
  const int N = jobs.n_out[l];
  const int lane = threadIdx.x & 31;
  const int o = (blk - jobs.first_block[l]) * 8 + (threadIdx.x >> 5);
  if (o >= N) return;                               // whole warp; no block-level sync below
  const float* A = jobs.a[l];
  const float* wrow = jobs.w[l] + static_cast<size_t>(o) * K;
  float acc[32];
#pragma unroll
  for (int b = 0; b < 32; ++b) acc[b] = 0.f;
  for (int k0 = lane * 4; k0 < K; k0 += 128) {
    const float4 w4 = __ldg(reinterpret_cast<const float4*>(wrow + k0));
#pragma unroll
    for (int b = 0; b < 32; ++b) {
      if (b < B) {
        float4 a4 = __ldg(reinterpret_cast<const float4*>(A + static_cast<size_t>(b) * a_stride + k0));
        if (MODE == 1) { a4.x *= a4.x; a4.y *= a4.y; a4.z *= a4.z; a4.w *= a4.w; }
        acc[b] = fmaf(a4.w, w4.w, fmaf(a4.z, w4.z, fmaf(a4.y, w4.y, fmaf(a4.x, w4.x, acc[b]))));
      }
    }
  }
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {               // lane keeps the half whose row bit equals its own
    const bool upper = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < s; ++i) {
      const float keep = upper ? acc[i + s] : acc[i];
      const float send = upper ? acc[i] : acc[i + s];
      acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  if (lane < B) {
    float v;
    if (MODE == 1) {
      v = rsqrtf(acc[0] + eps);
    } else {
      v = acc[0] * scale;
      if (jobs.bias[l]) v += __ldg(jobs.bias[l] + o) * bias_mul;
      if (act) v = (v > 0.f ? v : 0.2f * v) * 1.4142135623730951f;
    }
    jobs.out[l][static_cast<size_t>(lane) * N + o] = v;
  }
}

// B <= 32 and float4-addressable rows: the skinny kernel; otherwise the tiled one
template <int MODE>
static int gemm_jobs_launch(GemmJobs& jobs, int B, int K, long long a_stride, float scale,
                            float bias_mul, int act, float eps, cudaStream_t stream) {
  bool skinny = B <= 32 && K % 4 == 0 && a_stride % 4 == 0;
  for (int i = 0; i < jobs.n && skinny; ++i)
    skinny = ((reinterpret_cast<uintptr_t>(jobs.a[i]) | reinterpret_cast<uintptr_t>(jobs.w[i])) & 15u) == 0;
  const int cols = skinny ? 8 : 64;
  int blocks = 0;
  for (int i = 0; i < jobs.n; ++i) {
    jobs.first_block[i] = blocks;
    blocks += (jobs.n_out[i] + cols - 1) / cols;
  }
  jobs.first_block[jobs.n] = blocks;
  if (skinny) {
    skinny_gemm_kernel<MODE><<<blocks, 256, 0, stream>>>(B, K, a_stride, scale, bias_mul, act, eps, jobs);
  } else {
    dim3 grid(blocks, (B + 31) / 32);
    small_gemm_kernel<MODE><<<grid, 256, 0, stream>>>(B, K, a_stride, scale, bias_mul, act, eps, jobs);
  }
  return check_cuda(cudaGetLastError(), MODE == 1 ? "demod gemm launch" : "styles launch");
}

// ---------------------------------------------------------------------------
// ProgGAN leaves (reference utils/proggan.py:128-141): PixelNormLayer
//   out[b,c,y,x] = x[b,c,y,x] / sqrt(mean_c x[b,:,y,x]^2 + 1e-8)
// optionally fused with the following DoubleResolutionLayer (nearest 2x): every normalised value
// is stored to its 2 x 2 output pixels.  One thread per input pixel, coalesced along x for every
// channel plane; two passes over the C values of the pixel (the second one hits L1/L2).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pixel_norm_nchw_kernel(const float* __restrict__ x, int B, int C, int H, int W, int up2,
                       float* __restrict__ out) {
  const long long hw = static_cast<long long>(H) * W;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long long>(B) * hw) return;
  const int b = static_cast<int>(idx / hw);
  const long long pix = idx - static_cast<long long>(b) * hw;
  const float* src = x + static_cast<long long>(b) * C * hw + pix;
  float ss = 0.f;
  for (int c = 0; c < C; ++c) {
    const float v = __ldg(src + c * hw);
    ss = fmaf(v, v, ss);
  }
  // x / sqrt(mean + eps): a true division like the reference (not x * rsqrt)
  const float den = sqrtf(ss / static_cast<float>(C) + 1e-8f);
  if (!up2) {
    float* dst = out + static_cast<long long>(b) * C * hw + pix;
    for (int c = 0; c < C; ++c) dst[c * hw] = __ldg(src + c * hw) / den;
  } else {
    const int y = static_cast<int>(pix / W), xx = static_cast<int>(pix - static_cast<long long>(y) * W);
    const long long hw2 = 4 * hw;
    float* dst = out + static_cast<long long>(b) * C * hw2 + (2LL * y) * (2 * W) + 2 * xx;
    for (int c = 0; c < C; ++c) {
      const float v = __ldg(src + c * hw) / den;
      float* d = dst + c * hw2;
      *reinterpret_cast<float2*>(d) = make_float2(v, v);
      *reinterpret_cast<float2*>(d + 2 * W) = make_float2(v, v);
    }
  }
}

// nearest-neighbour 2x of [planes, H, W] (DoubleResolutionLayer on its own)
__global__ void __launch_bounds__(256)
nearest_up2_kernel(const float* __restrict__ x, long long n_in, int H, int W,
                   float* __restrict__ out) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= n_in) return;
  const long long hw = static_cast<long long>(H) * W;
  const long long pl = idx / hw;
  const long long pix = idx - pl * hw;
  const int y = static_cast<int>(pix / W), xx = static_cast<int>(pix - static_cast<long long>(y) * W);
  const float v = __ldg(x + idx);
  float* d = out + pl * 4 * hw + (2LL * y) * (2 * W) + 2 * xx;
  *reinterpret_cast<float2*>(d) = make_float2(v, v);
  *reinterpret_cast<float2*>(d + 2 * W) = make_float2(v, v);
}

inline int grid_for(long long n, int threads, int cap = 148 * 16) {
  long long g = (n + threads - 1) / threads;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace

int prep_keys_launch(const float* x, const float* style, int B, int C, int H, int W, void* kp_hi,
                     void* kp_lo, float* k_out, cudaStream_t stream) {
  if (C % 32 != 0) {
    set_last_error("prep_keys: C=%d must be a multiple of 32", C);
    return RW_ERR_BAD_ARG;
  }
  const int img = (H + 1) * (W + 1);
  if (C % 64 == 0) {
    dim3 grid((img + 31) / 32, C / 64, B);
    prep_keys_kernel<64><<<grid, 256, 0, stream>>>(x, style, C, H, W,
                                                   static_cast<__nv_bfloat16*>(kp_hi),
                                                   static_cast<__nv_bfloat16*>(kp_lo), k_out);
  } else {
    dim3 grid((img + 31) / 32, C / 32, B);
    prep_keys_kernel<32><<<grid, 256, 0, stream>>>(x, style, C, H, W,
                                                   static_cast<__nv_bfloat16*>(kp_hi),
                                                   static_cast<__nv_bfloat16*>(kp_lo), k_out);
  }
  return check_cuda(cudaGetLastError(), "prep_keys launch");
}

int split_rows_launch(const float* a, long long n, void* hi, void* lo, cudaStream_t stream) {
  const int threads = 256;
  const long long n4 = (n + 3) / 4;
  const int blocks = static_cast<int>((n4 + threads - 1) / threads);
  split_rows_kernel<<<blocks, threads, 0, stream>>>(a, n, static_cast<__nv_bfloat16*>(hi),
                                                    static_cast<__nv_bfloat16*>(lo));
  return check_cuda(cudaGetLastError(), "split_rows launch");
}

int prep_weights_launch(const float* w, int Cout, int Cin, float scale, int transpose_io,
                        int flip_taps, void* wt_hi, void* wt_lo, float* wsq, cudaStream_t stream) {
  const int n = Cout * Cin;
  prep_weights_kernel<<<(n + 255) / 256, 256, 0, stream>>>(
      w, Cout, Cin, scale, transpose_io, flip_taps, static_cast<__nv_bfloat16*>(wt_hi),
      static_cast<__nv_bfloat16*>(wt_lo), wsq);
  return check_cuda(cudaGetLastError(), "prep_weights launch");
}

int demod_launch(const float* style, const float* wsq, int B, int Cout, int Cin, float eps,
                 float* demod, cudaStream_t stream) {
  const long long warps = static_cast<long long>(B) * Cout;
  const int threads = 256;
  const int blocks = static_cast<int>((warps * 32 + threads - 1) / threads);
  demod_kernel<<<blocks, threads, 0, stream>>>(style, wsq, B, Cout, Cin, eps, demod);
  return check_cuda(cudaGetLastError(), "demod launch");
}

int blur_up_act_launch(const float* t, int B, int C, int Hin, int Win, const float* kernel4x4,
                       const float* noise, long long noise_bstride, const float* noise_w,
                       const float* bias, int act, float* y, cudaStream_t stream) {
  const int Ht = 2 * Hin + 1, Wt = 2 * Win + 1;
  const int Ho = 2 * Hin, Wo = 2 * Win;
  if (static_cast<long long>(B) * C > 65535LL * 1) {
    // grid.z limit is 65535
    if (static_cast<long long>(B) * C > 65535) {
      set_last_error("blur_up_act: B*C=%lld exceeds grid.z", static_cast<long long>(B) * C);
      return RW_ERR_BAD_ARG;
    }
  }
  dim3 grid((Wo + 31) / 32, (Ho + 7) / 8, B * C);
  dim3 block(32, 8);
  blur_up_act_kernel<<<grid, block, 0, stream>>>(t, C, Ht, Wt, kernel4x4, noise, noise_bstride,
                                                 noise_w, bias, act, y);
  return check_cuda(cudaGetLastError(), "blur_up_act launch");
}

int upfirdn2d_launch(const float* in, const float* kernel, int major, int in_h, int in_w, int kh,
                     int kw, int up_x, int up_y, int down_x, int down_y, int px0, int px1, int py0,
                     int py1, float* out, int out_h, int out_w, cudaStream_t stream) {
  (void)px1;
  (void)py1;
  const long long total = static_cast<long long>(major) * out_h * out_w;
  if (total <= 0) return RW_OK;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  upfirdn2d_kernel<<<static_cast<unsigned>(blocks), threads, 0, stream>>>(
      in, kernel, in_h, in_w, kh, kw, up_x, up_y, down_x, down_y, px0, py0, out, out_h, out_w,
      total);
  return check_cuda(cudaGetLastError(), "upfirdn2d launch");
}

int bias_act_launch(const float* x, const float* bias, const float* ref, int act, int grad,
                    float alpha, float scale, long long n, int step_b, int size_b, float* y,
                    cudaStream_t stream) {
  if (n <= 0) return RW_OK;
  bias_act_kernel<<<grid_for(n, 256), 256, 0, stream>>>(x, bias, ref, act, grad, alpha, scale, n,
                                                        step_b > 0 ? step_b : 1,
                                                        size_b > 0 ? size_b : 1, y);
  return check_cuda(cudaGetLastError(), "bias_act launch");
}

int torgb_launch(const float* x, const float* style, const float* w, const float* bias,
                 const float* skip, int B, int C, int H, int W, float scale, float* out,
                 cudaStream_t stream) {
  const int HW = H * W;
  dim3 grid((HW + 255) / 256, B);
  torgb_kernel<<<grid, 256, 3 * C * sizeof(float), stream>>>(x, style, w, bias, skip, C, HW, scale,
                                                             out);
  return check_cuda(cudaGetLastError(), "torgb launch");
}

int add_noise_launch(const float* x, const float* noise, long long noise_bstride, const float* noise_w,
                     int B, int C, int HW, float* y, cudaStream_t stream) {
  const long long total = static_cast<long long>(B) * C * HW;
  if (total <= 0) return RW_OK;
  add_noise_kernel<<<grid_for(total, 256), 256, 0, stream>>>(x, noise, noise_bstride, noise_w, C,
                                                             HW, total, y);
  return check_cuda(cudaGetLastError(), "add_noise launch");
}

int blur_up_fused_launch(const float* t_cl, int B, int C, int Hin, int Win, const float* k4,
                         const float* noise, long long noise_bstride, const float* noise_w,
                         const float* bias, int act, const float* next_scale, void* next_hi,
                         void* next_lo, float* y_out, cudaStream_t stream) {
  if (C % 32 != 0) {
    set_last_error("blur_up_fused: C=%d must be a multiple of 32", C);
    return RW_ERR_BAD_ARG;
  }
  const int Ho = 2 * Hin, Wo = 2 * Win;
  const size_t smem = static_cast<size_t>(BF_PH) * BF_PW * 16 * sizeof(float4);
  static bool attr = false;
  if (!attr) {
    int rc = check_cuda(cudaFuncSetAttribute(blur_up_fused_kernel<16>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(smem)),
                        "blur_up_fused smem attr");
    if (rc) return rc;
    attr = true;
  }
  const int tiles_x = (Wo + 1 + BF_TX - 1) / BF_TX, tiles_y = (Ho + 1 + BF_TY - 1) / BF_TY;
  if (C % BF_C != 0) {
    // 32-channel multiples: half-width channel blocks on the generic kernel
    const long long gz32 = static_cast<long long>(B) * (C / 32);
    if (gz32 > 65535) {
      set_last_error("blur_up_fused: grid.z %lld too large", gz32);
      return RW_ERR_BAD_ARG;
    }
    dim3 grid(tiles_x, tiles_y, static_cast<unsigned>(gz32));
    blur_up_fused_kernel<8><<<grid, 128, smem / 2, stream>>>(
        t_cl, B, C, Hin, Win, k4, noise, noise_bstride, noise_w, bias, act, next_scale,
        static_cast<__nv_bfloat16*>(next_hi), static_cast<__nv_bfloat16*>(next_lo), y_out);
    return check_cuda(cudaGetLastError(), "blur_up_fused launch");
  }
  const long long gz = static_cast<long long>(B) * (C / BF_C);
  if (gz > 65535) {
    set_last_error("blur_up_fused: grid.z %lld too large", gz);
    return RW_ERR_BAD_ARG;
  }
  const long long ntiles = static_cast<long long>(tiles_x) * tiles_y * gz;
  const long long rows_in4 = 4LL * B * (Hin + 1) * (Win + 1);
  // the generation fast path's configuration runs the pipelined kernel; anything else (no noise,
  // no activation, fp32 NCHW output, huge index ranges) the generic one-tile-per-CTA kernel
  const bool fast = noise && noise_w && bias && act && next_scale && next_hi && next_lo && !y_out &&
                    ntiles < 0x7fffffffLL && rows_in4 < 0x7fffffffLL &&
                    ((reinterpret_cast<uintptr_t>(bias) | reinterpret_cast<uintptr_t>(next_scale)) & 15u) == 0;
  if (fast) {
    static bool attr2 = false;
    if (!attr2) {
      int rc = check_cuda(cudaFuncSetAttribute(blur_up_pipe_kernel,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(2 * smem)),
                          "blur_up_pipe smem attr");
      if (rc) return rc;
      attr2 = true;
    }
    long long g = 2LL * device_sm_count();
    if (g > ntiles) g = ntiles;
    blur_up_pipe_kernel<<<static_cast<unsigned>(g), 256, 2 * smem, stream>>>(
        t_cl, B, C, Hin, Win, k4, noise, noise_bstride, noise_w, bias, next_scale,
        static_cast<__nv_bfloat16*>(next_hi), static_cast<__nv_bfloat16*>(next_lo), tiles_x, tiles_y,
        static_cast<unsigned>(ntiles));
    return check_cuda(cudaGetLastError(), "blur_up_pipe launch");
  }
  dim3 grid(tiles_x, tiles_y, static_cast<unsigned>(gz));
  blur_up_fused_kernel<16><<<grid, 256, smem, stream>>>(
      t_cl, B, C, Hin, Win, k4, noise, noise_bstride, noise_w, bias, act, next_scale,
      static_cast<__nv_bfloat16*>(next_hi), static_cast<__nv_bfloat16*>(next_lo), y_out);
  return check_cuda(cudaGetLastError(), "blur_up_fused launch");
}

int rgb_combine_launch(const float* part, int nparts, int B, int H, int W, const float* bias,
                       const float* prev, const float* k4, float* out, unsigned char* out_u8,
                       cudaStream_t stream) {
  if ((W & 3) != 0 || (prev && ((H | W) & 1)) || static_cast<long long>(B) * 3 > 65535 ||
      (!out && !out_u8) ||
      (reinterpret_cast<uintptr_t>(part) & 15u) || (reinterpret_cast<uintptr_t>(out) & 15u)) {
    set_last_error("rgb_combine: W=%d must be a multiple of 4 (even H, W with a skip), B*3 <= 65535, "
                   "16-byte aligned buffers", W);
    return RW_ERR_BAD_ARG;
  }
  const int quads = W / 4;
  const int bx = quads >= 64 ? 64 : (quads >= 32 ? 32 : (quads >= 16 ? 16 : (quads >= 8 ? 8 : (quads >= 4 ? 4 : (quads >= 2 ? 2 : 1)))));
  const int by = 256 / bx > H ? H : 256 / bx;
  dim3 block(bx, by);
  dim3 grid((quads + bx - 1) / bx, (H + by - 1) / by, B * 3);
  const long long part_stride = static_cast<long long>(B) * 3 * H * W;
  rgb_combine_kernel<<<grid, block, 0, stream>>>(part, nparts, part_stride, H, W, bias, prev, k4,
                                                 out, out_u8);
  return check_cuda(cudaGetLastError(), "rgb_combine launch");
}

int styles_launch(const float* latent, int B, int n_latent, int K, float scale, float bias_mul,
                  int act, int n, const float* const* w, const float* const* bias,
                  float* const* out, const int* lat, const int* chans, cudaStream_t stream) {
  if (n < 1 || n > 32) {
    set_last_error("styles: %d layers (max 32)", n);
    return RW_ERR_BAD_ARG;
  }
  // NOTE the equalised-lr convention: out = x . (W * scale)^T + bias * bias_mul; the scale is
  // applied to the accumulated sum here (one rounding per output instead of one per weight)
  GemmJobs jobs;
  jobs.n = n;
  for (int i = 0; i < n; ++i) {
    jobs.a[i] = latent + static_cast<size_t>(lat[i]) * K;
    jobs.w[i] = w[i];
    jobs.bias[i] = bias[i];
    jobs.out[i] = out[i];
    jobs.n_out[i] = chans[i];
  }
  return gemm_jobs_launch<0>(jobs, B, K, static_cast<long long>(n_latent) * K, scale, bias_mul, act,
                             0.f, stream);
}

int pixel_norm_launch(const float* z, int B, int K, float* out, cudaStream_t stream) {
  const int blocks = (B * 32 + 255) / 256;
  pixel_norm_kernel<<<blocks, 256, 0, stream>>>(z, B, K, out);
  return check_cuda(cudaGetLastError(), "pixel_norm launch");
}

int pixel_norm_nchw_launch(const float* x, int B, int C, int H, int W, int up2, float* out,
                           cudaStream_t stream) {
  const long long n = static_cast<long long>(B) * H * W;
  if (n <= 0 || C < 1 || (up2 && (reinterpret_cast<uintptr_t>(out) & 7u))) {
    set_last_error("pixel_norm_nchw: bad shape / alignment");
    return RW_ERR_BAD_ARG;
  }
  const long long blocks = (n + 255) / 256;
  pixel_norm_nchw_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(x, B, C, H, W, up2, out);
  return check_cuda(cudaGetLastError(), "pixel_norm_nchw launch");
}

int nearest_up2_launch(const float* x, long long planes, int H, int W, float* out,
                       cudaStream_t stream) {
  const long long n = planes * H * W;
  if (n <= 0 || (reinterpret_cast<uintptr_t>(out) & 7u)) {
    set_last_error("nearest_up2: bad shape / alignment");
    return RW_ERR_BAD_ARG;
  }
  const long long blocks = (n + 255) / 256;
  nearest_up2_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(x, n, H, W, out);
  return check_cuda(cudaGetLastError(), "nearest_up2 launch");
}

int demod_multi_launch(int B, float eps, int n, const float* const* style,
                       const float* const* wsq, float* const* out, const int* cout,
                       const int* cin, const int* kind, const float* wscale,
                       cudaStream_t stream) {
  if (n < 1 || n > 32) {
    set_last_error("demod_multi: %d jobs (max 32)", n);
    return RW_ERR_BAD_ARG;
  }
  // kind 0 (demodulation factors): tiled GEMM over style^2, one launch per distinct Cin;
  // kind 1 (ToRGB modulated weights): the elementwise kernel
  for (int pass_cin = 0;;) {
    GemmJobs g;
    g.n = 0;
    int K = 0;                                      // K = smallest Cin above pass_cin
    for (int i = 0; i < n; ++i)
      if (kind[i] == 0 && cin[i] > pass_cin && (K == 0 || cin[i] < K)) K = cin[i];
    if (K == 0) break;
    for (int i = 0; i < n; ++i) {
      if (kind[i] != 0 || cin[i] != K) continue;
      g.a[g.n] = style[i];
      g.w[g.n] = wsq[i];
      g.bias[g.n] = nullptr;
      g.out[g.n] = out[i];
      g.n_out[g.n] = cout[i];
      ++g.n;
    }
    int rc = gemm_jobs_launch<1>(g, B, K, K, 1.f, 0.f, 0, eps, stream);
    if (rc) return rc;
    pass_cin = K;
  }
  DemodJobs jobs;
  jobs.n = 0;
  int blocks = 0;
  for (int i = 0; i < n; ++i) {
    if (kind[i] != 1) continue;
    const int j = jobs.n++;
    jobs.style[j] = style[i];
    jobs.wsq[j] = wsq[i];
    jobs.out[j] = out[i];
    jobs.cout[j] = cout[i];
    jobs.cin[j] = cin[i];
    jobs.kind[j] = 1;
    jobs.wscale[j] = wscale[i];
    jobs.first_block[j] = blocks;
    blocks += (B * cout[i] + 7) / 8;
  }
  if (jobs.n == 0) return RW_OK;
  jobs.first_block[jobs.n] = blocks;
  demod_multi_kernel<<<blocks, 256, 0, stream>>>(B, eps, jobs);
  return check_cuda(cudaGetLastError(), "demod_multi launch");
}

int prep_phase_keys_launch(const float* g, const float* scale_bc, int B, int C, int H, int W,
                           void* hi, void* lo, cudaStream_t stream) {
  if (C % 64 != 0) {
    set_last_error("prep_phase_keys: C=%d must be a multiple of 64", C);
    return RW_ERR_BAD_ARG;
  }
  const int img = (H + 1) * (W + 1);
  dim3 grid((img + 31) / 32, C / 64, B * 4);
  prep_phase_keys_kernel<<<grid, 256, 0, stream>>>(g, scale_bc, C, H, W,
                                                   static_cast<__nv_bfloat16*>(hi),
                                                   static_cast<__nv_bfloat16*>(lo));
  return check_cuda(cudaGetLastError(), "prep_phase_keys launch");
}

}  // namespace rw
