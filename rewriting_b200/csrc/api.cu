// api.cu — the extern "C" boundary declared in include/rewriting_b200.h plus the
// small host-side utilities shared by the kernel translation units.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "../../include/rewriting_b200.h"
#include "rw_common.cuh"
#include "rw_kernels.h"

namespace rw {

static thread_local char g_err[512] = "";

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return RW_OK;
  set_last_error("%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
  return RW_ERR_CUDA;
}

int device_sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

int make_tmap_2d_bf16(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer,
                      uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer,
                      uint32_t swizzle_bytes) {
  PFN_encodeTiled fn = get_encode_fn();
  if (!fn) {
    set_last_error("cuTensorMapEncodeTiled not available from the driver");
    return RW_ERR_NO_DRIVER_SYMBOL;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 0xF) != 0 || (row_stride_bytes & 0xF) != 0) {
    set_last_error("TMA operand must be 16-byte aligned (ptr=%p stride=%llu)", base,
                   (unsigned long long)row_stride_bytes);
    return RW_ERR_BAD_ARG;
  }
  if ((swizzle_bytes != 128 && swizzle_bytes != 64) || box_inner * 2 > swizzle_bytes) {
    set_last_error("TMA operand: box rows of %u B do not fit a %u B swizzle", box_inner * 2,
                   swizzle_bytes);
    return RW_ERR_BAD_ARG;
  }
  cuuint64_t gdim[2] = {inner, outer};
  cuuint64_t gstr[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw =
      swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed: CUresult %d (inner=%llu outer=%llu box=%ux%u)",
                   (int)r, (unsigned long long)inner, (unsigned long long)outer, box_inner,
                   box_outer);
    return RW_ERR_CUDA;
  }
  return RW_OK;
}

int make_tmap_4d_bf16(CUtensorMap* out, const void* base, const uint64_t dims[4],
                      const uint64_t strides_bytes[3], const uint32_t box[4]) {
  PFN_encodeTiled fn = get_encode_fn();
  if (!fn) {
    set_last_error("cuTensorMapEncodeTiled not available from the driver");
    return RW_ERR_NO_DRIVER_SYMBOL;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 0xF) != 0) {
    set_last_error("TMA operand must be 16-byte aligned (ptr=%p)", base);
    return RW_ERR_BAD_ARG;
  }
  cuuint64_t gdim[4] = {dims[0], dims[1], dims[2], dims[3]};
  cuuint64_t gstr[3] = {strides_bytes[0], strides_bytes[1], strides_bytes[2]};
  cuuint32_t bx[4] = {box[0], box[1], box[2], box[3]};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr, bx,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled(4d) failed: CUresult %d (dims %llu %llu %llu %llu box %u %u "
                   "%u %u)", (int)r, (unsigned long long)dims[0], (unsigned long long)dims[1],
                   (unsigned long long)dims[2], (unsigned long long)dims[3], box[0], box[1], box[2],
                   box[3]);
    return RW_ERR_CUDA;
  }
  return RW_OK;
}

// general form: rank <= 5, element strides (a stride s on dimension d loads every s-th element
// of the box extent box[d]), swizzle 0 = none, 1 = 32 B, 2 = 128 B
int make_tmap_nd_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box, const uint32_t* estrides,
                      int swizzle) {
  PFN_encodeTiled fn = get_encode_fn();
  if (!fn) {
    set_last_error("cuTensorMapEncodeTiled not available from the driver");
    return RW_ERR_NO_DRIVER_SYMBOL;
  }
  if (rank < 2 || rank > 5 || (reinterpret_cast<uintptr_t>(base) & 0xF) != 0) {
    set_last_error("TMA operand: rank %d, ptr %p (must be rank 2..5, 16-byte aligned)", rank, base);
    return RW_ERR_BAD_ARG;
  }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = estrides ? estrides[i] : 1u;
    if (i + 1 < rank) gstr[i] = strides_bytes[i];
  }
  const CUtensorMapSwizzle sw = swizzle == 2 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle == 1 ? CU_TENSOR_MAP_SWIZZLE_32B
                                               : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank),
                  const_cast<void*>(base), gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled(rank %d) failed: CUresult %d (dim0 %llu dim1 %llu box %u %u)",
                   rank, (int)r, (unsigned long long)dims[0], (unsigned long long)dims[1], box[0],
                   box[1]);
    return RW_ERR_CUDA;
  }
  return RW_OK;
}

// split heuristic shared by the workspace query and the launches
static int gram_splits(int tiles, long long rows, int ntaps) {
  const long long total_rb = (rows + 63) / 64;
  const int sms = 148;
  long long s = (sms + static_cast<long long>(tiles) * ntaps - 1) / (static_cast<long long>(tiles) * ntaps);
  if (s > total_rb) s = total_rb;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  (void)0;
  return static_cast<int>(s);
}

}  // namespace rw

using namespace rw;

extern "C" {

int rw_version(void) { return 100; }
const char* rw_last_error(void) { return g_err; }
int rw_set_device(int device) { return check_cuda(cudaSetDevice(device), "cudaSetDevice"); }
int rw_device_sm_count(void) { return device_sm_count(); }

int rw_prep_keys(const float* x, const float* style, int B, int C, int H, int W, void* kp_hi,
                 void* kp_lo, float* k_out, rw_stream_t stream) {
  if (!x || !kp_hi || !kp_lo || B < 1 || H < 1 || W < 1) {
    set_last_error("rw_prep_keys: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return prep_keys_launch(x, style, B, C, H, W, kp_hi, kp_lo, k_out, stream);
}

int rw_split_rows(const float* a, long long n, void* hi, void* lo, rw_stream_t stream) {
  if (n == 0) return RW_OK;
  if (!a || !hi || !lo || n < 0) {
    set_last_error("rw_split_rows: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return split_rows_launch(a, n, hi, lo, stream);
}

int rw_prep_weights(const float* w, int Cout, int Cin, float scale, int transpose_io,
                    int flip_taps, void* wt_hi, void* wt_lo, float* wsq, rw_stream_t stream) {
  if (!w || !wt_hi || !wt_lo || Cout < 1 || Cin < 1) {
    set_last_error("rw_prep_weights: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return prep_weights_launch(w, Cout, Cin, scale, transpose_io, flip_taps, wt_hi, wt_lo, wsq,
                             stream);
}

int rw_demod(const float* style, const float* wsq, int B, int Cout, int Cin, float eps,
             float* demod, rw_stream_t stream) {
  if (!style || !wsq || !demod) {
    set_last_error("rw_demod: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return demod_launch(style, wsq, B, Cout, Cin, eps, demod, stream);
}

int rw_modconv_fwd(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                   const float* scale_bo, const float* noise, long long noise_bstride,
                   const float* noise_w, const float* bias, int act, int B, int Cin, int Cout,
                   int H, int W, float* out, rw_stream_t stream) {
  if (!kp_hi || !kp_lo || !wt_hi || !wt_lo || !out || B < 1 || (noise && !noise_w)) {
    set_last_error("rw_modconv_fwd: bad argument");
    return RW_ERR_BAD_ARG;
  }
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  p.Hp = H + 1;
  p.Wp = W + 1;
  p.B = B;
  p.nphase = 1;
  p.ph_Hv[0] = H;
  p.ph_Wv[0] = W;
  const long long rows = static_cast<long long>(B) * p.Hp * p.Wp;
  if (rows > 0x7fffffffLL) {
    set_last_error("rw_modconv_fwd: too many rows");
    return RW_ERR_BAD_ARG;
  }
  p.rows = static_cast<int>(rows);
  p.Cin = Cin;
  p.Cout = Cout;
  p.ph_ntaps[0] = 9;
  for (int u = 0; u < 3; ++u)
    for (int v = 0; v < 3; ++v) {
      p.ph_shift[0][u * 3 + v] = (u - 1) * p.Wp + (v - 1);
      p.ph_kofs[0][u * 3 + v] = (u * 3 + v) * Cin;
    }
  p.scale_bo = scale_bo;
  p.bias = bias;
  p.noise = noise;
  p.noise_bstride = noise_bstride;
  p.noise_w = noise_w;
  p.act = act;
  p.out = out;
  p.out_sb = static_cast<long long>(Cout) * H * W;
  p.out_sc = static_cast<long long>(H) * W;
  p.out_sy = W;
  p.out_sx = 1;
  return conv_tc_launch(p, kp_hi, kp_lo, wt_hi, wt_lo, 9 * Cin, stream);
}

static int modconv_up_impl(const void* kp_hi, const void* kp_lo, const void* wt_hi,
                           const void* wt_lo, const float* scale_bo, int B, int Cin, int Cout,
                           int H, int W, float* t_out, int channels_last, rw_stream_t stream) {
  if (!kp_hi || !kp_lo || !wt_hi || !wt_lo || !t_out || B < 1) {
    set_last_error("rw_modconv_up_fwd: bad argument");
    return RW_ERR_BAD_ARG;
  }
  // conv_transpose2d(stride 2, pad 0, k 3): out[2m+a, 2n+b] gathers
  //   a == 0: (u=0, in row m), (u=2, in row m-1);  a == 1: (u=1, in row m)   (same along x)
  // over the padded-flat grid every phase is a row-GEMM with <= 4 shifted taps.
  const int Hp = H + 1, Wp = W + 1;
  const int Ht = 2 * H + 1, Wt = 2 * W + 1;
  const long long rows = static_cast<long long>(B) * Hp * Wp;
  if (rows > 0x7fffffffLL) {
    set_last_error("rw_modconv_up_fwd: too many rows");
    return RW_ERR_BAD_ARG;
  }
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  p.Hp = Hp;
  p.Wp = Wp;
  p.B = B;
  p.rows = static_cast<int>(rows);
  p.Cin = Cin;
  p.Cout = Cout;
  p.nphase = 4;
  p.scale_bo = scale_bo;
  p.out = t_out;
  p.out_sb = static_cast<long long>(Cout) * Ht * Wt;
  p.out_sc = static_cast<long long>(Ht) * Wt;
  p.out_sy = 2LL * Wt;
  p.out_sx = 2;
  p.out_mode = channels_last ? 1 : 0;
  // heaviest phase first within every (m, n) group: (0,0) has 4 taps, (1,1) has 1
  for (int a = 0; a < 2; ++a) {
    for (int b = 0; b < 2; ++b) {
      const int ph = a * 2 + b;
      p.ph_Hv[ph] = Hp - a;
      p.ph_Wv[ph] = Wp - b;
      p.ph_out_ofs[ph] = static_cast<long long>(a) * Wt + b;
      int us[2], dys[2], nu;
      int vs[2], dxs[2], nv;
      if (a == 0) { nu = 2; us[0] = 0; dys[0] = 0; us[1] = 2; dys[1] = -1; }
      else        { nu = 1; us[0] = 1; dys[0] = 0; }
      if (b == 0) { nv = 2; vs[0] = 0; dxs[0] = 0; vs[1] = 2; dxs[1] = -1; }
      else        { nv = 1; vs[0] = 1; dxs[0] = 0; }
      int n = 0;
      for (int iu = 0; iu < nu; ++iu)
        for (int iv = 0; iv < nv; ++iv) {
          p.ph_shift[ph][n] = dys[iu] * Wp + dxs[iv];
          p.ph_kofs[ph][n] = (us[iu] * 3 + vs[iv]) * Cin;
          ++n;
        }
      p.ph_ntaps[ph] = n;
    }
  }
  return conv_tc_launch(p, kp_hi, kp_lo, wt_hi, wt_lo, 9 * Cin, stream);
}

int rw_modconv_up_fwd(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                      const float* scale_bo, int B, int Cin, int Cout, int H, int W, float* t_out,
                      rw_stream_t stream) {
  return modconv_up_impl(kp_hi, kp_lo, wt_hi, wt_lo, scale_bo, B, Cin, Cout, H, W, t_out, 0, stream);
}

int rw_modconv_up_fwd_cl(const void* kp_hi, const void* kp_lo, const void* wt_hi,
                         const void* wt_lo, const float* scale_bo, int B, int Cin, int Cout, int H,
                         int W, float* t_cl, rw_stream_t stream) {
  return modconv_up_impl(kp_hi, kp_lo, wt_hi, wt_lo, scale_bo, B, Cin, Cout, H, W, t_cl, 1, stream);
}

static int fill_conv3x3(ConvTcParams& p, int B, int Cin, int Cout, int H, int W) {
  memset(&p, 0, sizeof(p));
  p.Hp = H + 1;
  p.Wp = W + 1;
  p.B = B;
  p.nphase = 1;
  p.ph_Hv[0] = H;
  p.ph_Wv[0] = W;
  const long long rows = static_cast<long long>(B) * p.Hp * p.Wp;
  if (rows > 0x7fffffffLL) {
    set_last_error("conv: too many rows");
    return RW_ERR_BAD_ARG;
  }
  p.rows = static_cast<int>(rows);
  p.Cin = Cin;
  p.Cout = Cout;
  p.ph_ntaps[0] = 9;
  for (int u = 0; u < 3; ++u)
    for (int v = 0; v < 3; ++v) {
      p.ph_shift[0][u * 3 + v] = (u - 1) * p.Wp + (v - 1);
      p.ph_kofs[0][u * 3 + v] = (u * 3 + v) * Cin;
    }
  p.out_sb = static_cast<long long>(Cout) * H * W;
  p.out_sc = static_cast<long long>(H) * W;
  p.out_sy = W;
  p.out_sx = 1;
  return RW_OK;
}

int rw_conv3x3_bias_act(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                        const float* bias, int act, float act_gain, int B, int Cin, int Cout, int H,
                        int W, float* out, rw_stream_t stream) {
  if (!kp_hi || !kp_lo || !wt_hi || !wt_lo || !out || B < 1) {
    set_last_error("rw_conv3x3_bias_act: bad argument");
    return RW_ERR_BAD_ARG;
  }
  ConvTcParams p;
  int rc = fill_conv3x3(p, B, Cin, Cout, H, W);
  if (rc) return rc;
  p.bias = bias;
  p.act = act;
  p.act_gain = act_gain;
  p.out = out;
  return conv_tc_launch(p, kp_hi, kp_lo, wt_hi, wt_lo, 9 * Cin, stream);
}

int rw_pixel_norm_nchw(const float* x, int B, int C, int H, int W, int up2, float* out,
                       rw_stream_t stream) {
  if (!x || !out) {
    set_last_error("rw_pixel_norm_nchw: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return pixel_norm_nchw_launch(x, B, C, H, W, up2, out, stream);
}

int rw_nearest_up2(const float* x, long long planes, int H, int W, float* out, rw_stream_t stream) {
  if (!x || !out) {
    set_last_error("rw_nearest_up2: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return nearest_up2_launch(x, planes, H, W, out, stream);
}

int rw_modconv_fwd_fused(const void* kp_hi, const void* kp_lo, const void* wt_hi,
                         const void* wt_lo, const float* scale_bo, const float* noise,
                         long long noise_bstride, const float* noise_w, const float* bias, int act,
                         int B, int Cin, int Cout, int H, int W, float* out,
                         const float* next_scale, void* next_hi, void* next_lo,
                         const float* rgb_w, float* rgb_part, rw_stream_t stream) {
  if (!kp_hi || !kp_lo || !wt_hi || !wt_lo || B < 1 || (noise && !noise_w) ||
      ((next_hi != nullptr) != (next_lo != nullptr)) || (next_hi && !next_scale) ||
      ((rgb_w != nullptr) != (rgb_part != nullptr)) || (!out && !next_hi && !rgb_part)) {
    set_last_error("rw_modconv_fwd_fused: bad argument");
    return RW_ERR_BAD_ARG;
  }
  ConvTcParams p;
  int rc = fill_conv3x3(p, B, Cin, Cout, H, W);
  if (rc) return rc;
  p.scale_bo = scale_bo;
  p.bias = bias;
  p.noise = noise;
  p.noise_bstride = noise_bstride;
  p.noise_w = noise_w;
  p.act = act;
  p.out = out;
  p.next_hi = next_hi;
  p.next_lo = next_lo;
  p.next_scale = next_scale;
  p.rgb_w = rgb_w;
  p.rgb_part = rgb_part;
  return conv_tc_launch(p, kp_hi, kp_lo, wt_hi, wt_lo, 9 * Cin, stream);
}

int rw_modconv_rgb_parts(int Cout) { return conv_tc_rgb_parts(Cout); }

int rw_modconv_up_fused(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                        const float* demod, const float* kernel4x4, const float* noise,
                        long long noise_bstride, const float* noise_w, const float* bias,
                        const float* next_scale, void* next_hi, void* next_lo, int B, int Cin,
                        int Cout, int H, int W, rw_stream_t stream) {
  if (!kp_hi || !kp_lo || !wt_hi || !wt_lo || !demod || !kernel4x4 || !noise || !noise_w || !bias ||
      !next_scale || !next_hi || !next_lo || (noise_bstride & 1)) {
    set_last_error("rw_modconv_up_fused: bad argument");
    return RW_ERR_BAD_ARG;
  }
  UpFusedParams p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.Cin = Cin; p.Cout = Cout; p.H = H; p.W = W;
  p.demod = demod; p.bias = bias; p.noise = noise; p.noise_bstride = noise_bstride;
  p.noise_w = noise_w; p.k4 = kernel4x4; p.next_scale = next_scale;
  p.next_hi = next_hi; p.next_lo = next_lo;
  return upconv_fused_launch(p, kp_hi, kp_lo, wt_hi, wt_lo, stream);
}

int rw_modconv_up_fused_y(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                          const float* demod, const float* kernel4x4, const float* noise,
                          long long noise_bstride, const float* noise_w, const float* bias, int act,
                          float* y, int B, int Cin, int Cout, int H, int W, rw_stream_t stream) {
  if (!kp_hi || !kp_lo || !wt_hi || !wt_lo || !kernel4x4 || !y || (noise && (noise_bstride & 3)) ||
      ((noise != nullptr) != (noise_w != nullptr))) {
    set_last_error("rw_modconv_up_fused_y: bad argument");
    return RW_ERR_BAD_ARG;
  }
  UpFusedParams p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.Cin = Cin; p.Cout = Cout; p.H = H; p.W = W;
  p.demod = demod; p.bias = bias; p.noise = noise; p.noise_bstride = noise_bstride;
  p.noise_w = noise_w; p.k4 = kernel4x4;
  p.y_out = y;
  p.act = act;
  return upconv_fused_launch(p, kp_hi, kp_lo, wt_hi, wt_lo, stream);
}

int rw_debug_upconv_taps(const void* kp_hi, const void* kp_lo, const void* wt_hi, const void* wt_lo,
                         const float* ones_bo, const float* kernel4x4, const float* noise,
                         long long noise_bstride, const float* noise_w, const float* bias,
                         void* next_hi, void* next_lo, int B, int Cin, int Cout, int H, int W,
                         float* taps_out, rw_stream_t stream) {
  UpFusedParams p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.Cin = Cin; p.Cout = Cout; p.H = H; p.W = W;
  p.demod = ones_bo; p.bias = bias; p.noise = noise; p.noise_bstride = noise_bstride;
  p.noise_w = noise_w; p.k4 = kernel4x4; p.next_scale = ones_bo;
  p.next_hi = next_hi; p.next_lo = next_lo;
  p.debug_p = taps_out;
  return upconv_fused_launch(p, kp_hi, kp_lo, wt_hi, wt_lo, stream);
}

int rw_debug_upconv_profile(const void* kp_hi, const void* kp_lo, const void* wt_hi,
                            const void* wt_lo, const float* demod, const float* kernel4x4,
                            const float* noise, long long noise_bstride, const float* noise_w,
                            const float* bias, const float* next_scale, void* next_hi, void* next_lo,
                            int B, int Cin, int Cout, int H, int W, long long* prof_out,
                            rw_stream_t stream) {
  UpFusedParams p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.Cin = Cin; p.Cout = Cout; p.H = H; p.W = W;
  p.demod = demod; p.bias = bias; p.noise = noise; p.noise_bstride = noise_bstride;
  p.noise_w = noise_w; p.k4 = kernel4x4; p.next_scale = next_scale;
  p.next_hi = next_hi; p.next_lo = next_lo;
  p.debug_prof = prof_out;
  p.debug_nostore = getenv("RW_UP_NOSTORE") != nullptr;
  return upconv_fused_launch(p, kp_hi, kp_lo, wt_hi, wt_lo, stream);
}

int rw_blur_up_fused(const float* t_cl, int B, int C, int Hin, int Win, const float* kernel4x4,
                     const float* noise, long long noise_bstride, const float* noise_w,
                     const float* bias, int act, const float* next_scale, void* next_hi,
                     void* next_lo, float* y_out, rw_stream_t stream) {
  if (!t_cl || !kernel4x4 || (noise && !noise_w) || ((next_hi != nullptr) != (next_lo != nullptr)) ||
      (!next_hi && !y_out)) {
    set_last_error("rw_blur_up_fused: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return blur_up_fused_launch(t_cl, B, C, Hin, Win, kernel4x4, noise, noise_bstride, noise_w, bias,
                              act, next_scale, next_hi, next_lo, y_out, stream);
}

int rw_styles(const float* latent, int B, int n_latent, int K, float scale, int n,
              const float* const* w, const float* const* bias, float* const* out, const int* lat,
              const int* chans, rw_stream_t stream) {
  if (!latent || !w || !bias || !out || !lat || !chans || B < 1) {
    set_last_error("rw_styles: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return styles_launch(latent, B, n_latent, K, scale, 1.f, 0, n, w, bias, out, lat, chans, stream);
}

int rw_equal_linear(const float* x, int B, int K, const float* w, const float* bias, int Cout,
                    float scale, float bias_mul, int act, float* out, rw_stream_t stream) {
  if (!x || !w || !bias || !out || B < 1 || K < 1 || Cout < 1) {
    set_last_error("rw_equal_linear: bad argument");
    return RW_ERR_BAD_ARG;
  }
  const int lat = 0;
  return styles_launch(x, B, 1, K, scale, bias_mul, act, 1, &w, &bias, &out, &lat, &Cout, stream);
}

int rw_pixel_norm(const float* z, int B, int K, float* out, rw_stream_t stream) {
  if (!z || !out || B < 1 || K < 1) {
    set_last_error("rw_pixel_norm: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return pixel_norm_launch(z, B, K, out, stream);
}

int rw_demod_multi(int B, float eps, int n, const float* const* style, const float* const* w,
                   float* const* out, const int* cout, const int* cin, const int* kind,
                   const float* wscale, rw_stream_t stream) {
  if (!style || !w || !out || !cout || !cin || !kind || !wscale || B < 1) {
    set_last_error("rw_demod_multi: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return demod_multi_launch(B, eps, n, style, w, out, cout, cin, kind, wscale, stream);
}

int rw_rgb_combine(const float* part, int nparts, int B, int H, int W, const float* bias,
                   const float* prev, const float* kernel4x4, float* out, rw_stream_t stream) {
  if (!part || nparts < 1 || !bias || !out || (prev && !kernel4x4)) {
    set_last_error("rw_rgb_combine: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return rgb_combine_launch(part, nparts, B, H, W, bias, prev, kernel4x4, out, nullptr, stream);
}

int rw_rgb_combine_u8(const float* part, int nparts, int B, int H, int W, const float* bias,
                      const float* prev, const float* kernel4x4, float* out,
                      unsigned char* out_u8_nhwc, rw_stream_t stream) {
  if (!part || nparts < 1 || !bias || (!out && !out_u8_nhwc) || (prev && !kernel4x4)) {
    set_last_error("rw_rgb_combine_u8: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return rgb_combine_launch(part, nparts, B, H, W, bias, prev, kernel4x4, out, out_u8_nhwc, stream);
}

int rw_blur_up_act(const float* t, int B, int C, int Hin, int Win, const float* kernel4x4,
                   const float* noise, long long noise_bstride, const float* noise_w,
                   const float* bias, int act, float* y, rw_stream_t stream) {
  if (!t || !kernel4x4 || !y || (noise && !noise_w)) {
    set_last_error("rw_blur_up_act: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return blur_up_act_launch(t, B, C, Hin, Win, kernel4x4, noise, noise_bstride, noise_w, bias, act,
                            y, stream);
}

int rw_add_noise(const float* x, const float* noise, long long noise_bstride,
                 const float* noise_w, int B, int C, int HW, float* y, rw_stream_t stream) {
  if (!x || !noise || !y || !noise_w) {
    set_last_error("rw_add_noise: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return add_noise_launch(x, noise, noise_bstride, noise_w, B, C, HW, y, stream);
}

int rw_torgb(const float* x, const float* style, const float* w, const float* bias,
             const float* skip, int B, int C, int H, int W, float scale, float* out,
             rw_stream_t stream) {
  if (!x || !style || !w || !bias || !out || C > 4096) {
    set_last_error("rw_torgb: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return torgb_launch(x, style, w, bias, skip, B, C, H, W, scale, out, stream);
}

int rw_fused_bias_act(const float* x, const float* bias, const float* ref, int act, int grad,
                      float alpha, float scale, long long n, int step_b, int size_b, float* y,
                      rw_stream_t stream) {
  if (n == 0) return RW_OK;
  if (!x || !y || n < 0) {
    set_last_error("rw_fused_bias_act: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return bias_act_launch(x, bias, ref, act, grad, alpha, scale, n, step_b, size_b, y, stream);
}

int rw_upfirdn2d(const float* in, const float* kernel, int major, int in_h, int in_w, int kh,
                 int kw, int up_x, int up_y, int down_x, int down_y, int pad_x0, int pad_x1,
                 int pad_y0, int pad_y1, float* out, int out_h, int out_w, rw_stream_t stream) {
  if (!in || !kernel || !out || up_x < 1 || up_y < 1 || down_x < 1 || down_y < 1) {
    set_last_error("rw_upfirdn2d: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return upfirdn2d_launch(in, kernel, major, in_h, in_w, kh, kw, up_x, up_y, down_x, down_y,
                          pad_x0, pad_x1, pad_y0, pad_y1, out, out_h, out_w, stream);
}

size_t rw_gram_workspace_bytes(int Cm, int Cn, long long rows, int ntaps) {
  if (Cm < 128 || Cn < 128 || ntaps < 1) return 0;
  const int mt = Cm / 128, nt = Cn / 128;
  const int tiles_full = mt * nt;
  // the symmetric path uses fewer tiles -> more splits; size for the larger of the two
  const int tiles_sym = (Cm == Cn) ? mt * (mt + 1) / 2 : tiles_full;
  const int s1 = gram_splits(tiles_full, rows, ntaps);
  const int s2 = gram_splits(tiles_sym, rows, ntaps);
  const int s = s1 > s2 ? s1 : s2;
  return static_cast<size_t>(s) * Cm * static_cast<size_t>(Cn) * ntaps * sizeof(float);
}

int rw_second_moment_accum(const void* hi, const void* lo, long long rows, int C, float* mom2,
                           void* workspace, size_t workspace_bytes, rw_stream_t stream) {
  if (rows == 0) return RW_OK;
  if (!hi || !lo || !mom2 || !workspace || rows < 0 || rows > 0x7fffffffLL || C % 128 != 0) {
    set_last_error("rw_second_moment_accum: bad argument (rows=%lld C=%d)", rows, C);
    return RW_ERR_BAD_ARG;
  }
  GramTcParams p;
  memset(&p, 0, sizeof(p));
  p.rows = static_cast<int>(rows);
  p.rows_a = p.rows_b = static_cast<int>(rows);
  p.Cm = p.Cn = C;
  p.ntaps = 1;
  p.upper_only = 1;
  const int mt = C / 128;
  p.splits = gram_splits(mt * (mt + 1) / 2, rows, 1);
  p.ldp = C;
  p.partial = static_cast<float*>(workspace);
  const size_t need = static_cast<size_t>(p.splits) * C * C * sizeof(float);
  if (workspace_bytes < need) {
    set_last_error("rw_second_moment_accum: workspace %zu < %zu bytes", workspace_bytes, need);
    return RW_ERR_BAD_ARG;
  }
  int rc = gram_tc_launch(p, hi, lo, hi, lo, stream);
  if (rc) return rc;
  return reduce_partials_launch(p.partial, p.splits, C, C, p.ldp, mom2, C, /*accumulate=*/1,
                                /*mirror_upper=*/1, stream);
}

int rw_conv_wgrad(const void* g_hi, const void* g_lo, const void* kp_hi, const void* kp_lo,
                  long long rows, int Cout, int Cin, int Wp, float* dw_toi, void* workspace,
                  size_t workspace_bytes, rw_stream_t stream) {
  if (!g_hi || !g_lo || !kp_hi || !kp_lo || !dw_toi || !workspace || rows <= 0 ||
      rows > 0x7fffffffLL) {
    set_last_error("rw_conv_wgrad: bad argument");
    return RW_ERR_BAD_ARG;
  }
  if (Cout < 128 || Cin < 128 || Cout % 128 != 0 || Cin % 128 != 0) {
    // the col-GEMM's 128 x 128 tiles: the 64- and 32-channel layers have no weight gradient
    set_last_error("rw_conv_wgrad: Cout=%d Cin=%d must be multiples of 128", Cout, Cin);
    return RW_ERR_BAD_ARG;
  }
  GramTcParams p;
  memset(&p, 0, sizeof(p));
  p.rows = static_cast<int>(rows);
  p.rows_a = p.rows_b = static_cast<int>(rows);
  p.Cm = Cout;
  p.Cn = Cin;
  p.ntaps = 9;
  for (int u = 0; u < 3; ++u)
    for (int v = 0; v < 3; ++v) {
      p.tap_shift_b[u * 3 + v] = (u - 1) * Wp + (v - 1);
      p.tap_col_ofs[u * 3 + v] = (u * 3 + v) * Cin;
    }
  p.upper_only = 0;
  p.splits = gram_splits((Cout / 128) * (Cin / 128), rows, 9);
  p.ldp = 9LL * Cin;
  p.partial = static_cast<float*>(workspace);
  const size_t need = static_cast<size_t>(p.splits) * Cout * 9 * Cin * sizeof(float);
  if (workspace_bytes < need) {
    set_last_error("rw_conv_wgrad: workspace %zu < %zu bytes", workspace_bytes, need);
    return RW_ERR_BAD_ARG;
  }
  int rc = gram_tc_launch(p, g_hi, g_lo, kp_hi, kp_lo, stream);
  if (rc) return rc;
  return reduce_partials_launch(p.partial, p.splits, Cout, 9 * Cin, p.ldp, dw_toi, 9LL * Cin,
                                /*accumulate=*/0, /*mirror_upper=*/0, stream);
}

int rw_prep_phase_keys(const float* g, const float* scale_bc, int B, int C, int H, int W,
                       void* hi, void* lo, rw_stream_t stream) {
  if (!g || !hi || !lo || B < 1) {
    set_last_error("rw_prep_phase_keys: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return prep_phase_keys_launch(g, scale_bc, B, C, H, W, hi, lo, stream);
}

// tap (u,v) of the stride-2 conv_transpose reads gradient phase (u&1, v&1) at row shift
// (u>>1)*(W+1) + (v>>1) of the INPUT-resolution padded grid.
int rw_modconv_up_dgrad(const void* gph_hi, const void* gph_lo, const void* wt_hi,
                        const void* wt_lo, const float* scale_bi, int B, int Cin, int Cout, int H,
                        int W, float* dk, rw_stream_t stream) {
  if (!gph_hi || !gph_lo || !wt_hi || !wt_lo || !dk || B < 1) {
    set_last_error("rw_modconv_up_dgrad: bad argument");
    return RW_ERR_BAD_ARG;
  }
  // GEMM: M = input pixels, K = 9 taps x Cout (gradient channels), N = Cin
  ConvTcParams p;
  int rc = fill_conv3x3(p, B, /*Cin(K)=*/Cout, /*Cout(N)=*/Cin, H, W);
  if (rc) return rc;
  p.a_cols = 4 * Cout;
  for (int u = 0; u < 3; ++u)
    for (int v = 0; v < 3; ++v) {
      const int t = u * 3 + v;
      p.ph_shift[0][t] = (u >> 1) * p.Wp + (v >> 1);
      p.ph_acol[0][t] = ((u & 1) * 2 + (v & 1)) * Cout;
      p.ph_kofs[0][t] = t * Cout;
    }
  p.scale_bo = scale_bi;
  p.out = dk;
  return conv_tc_launch(p, gph_hi, gph_lo, wt_hi, wt_lo, 9 * Cout, stream);
}

int rw_conv_up_wgrad(const void* gph_hi, const void* gph_lo, const void* kp_hi, const void* kp_lo,
                     long long rows, int Cout, int Cin, int Wp, float* dw_toi, void* workspace,
                     size_t workspace_bytes, rw_stream_t stream) {
  if (!gph_hi || !gph_lo || !kp_hi || !kp_lo || !dw_toi || !workspace || rows <= 0 ||
      rows > 0x7fffffffLL) {
    set_last_error("rw_conv_up_wgrad: bad argument");
    return RW_ERR_BAD_ARG;
  }
  if (Cout < 128 || Cin < 128 || Cout % 128 != 0 || Cin % 128 != 0) {
    // the col-GEMM's 128 x 128 tiles: the 64- and 32-channel layers have no weight gradient
    set_last_error("rw_conv_up_wgrad: Cout=%d Cin=%d must be multiples of 128", Cout, Cin);
    return RW_ERR_BAD_ARG;
  }
  GramTcParams p;
  memset(&p, 0, sizeof(p));
  p.rows = static_cast<int>(rows);
  p.rows_a = p.rows_b = static_cast<int>(rows);
  p.Cm = Cout;
  p.Cn = Cin;
  p.a_cols = 4 * Cout;
  p.ntaps = 9;
  for (int u = 0; u < 3; ++u)
    for (int v = 0; v < 3; ++v) {
      const int t = u * 3 + v;
      p.tap_shift_a[t] = (u >> 1) * Wp + (v >> 1);
      p.tap_acol[t] = ((u & 1) * 2 + (v & 1)) * Cout;
      p.tap_col_ofs[t] = t * Cin;
    }
  p.splits = gram_splits((Cout / 128) * (Cin / 128), rows, 9);
  p.ldp = 9LL * Cin;
  p.partial = static_cast<float*>(workspace);
  const size_t need = static_cast<size_t>(p.splits) * Cout * 9 * Cin * sizeof(float);
  if (workspace_bytes < need) {
    set_last_error("rw_conv_up_wgrad: workspace %zu < %zu bytes", workspace_bytes, need);
    return RW_ERR_BAD_ARG;
  }
  int rc = gram_tc_launch(p, gph_hi, gph_lo, kp_hi, kp_lo, stream);
  if (rc) return rc;
  return reduce_partials_launch(p.partial, p.splits, Cout, 9 * Cin, p.ldp, dw_toi, 9LL * Cin, 0, 0,
                                stream);
}

int rw_act_grad_reduce(const float* gy, const float* y, const float* noise,
                       long long noise_bstride, const float* noise_w, const float* bias, int act,
                       int B, int C, int HW, float* g_pre, float* s_sum, float* s_dot,
                       float* s_noise, rw_stream_t stream) {
  if (!gy || !y || !s_sum || !s_dot || !s_noise || B < 0 || C < 1 || HW < 0 ||
      (noise && !noise_w)) {
    set_last_error("rw_act_grad_reduce: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return act_grad_reduce_launch(gy, y, noise, noise_bstride, noise_w, bias, act, B, C, HW, g_pre,
                                s_sum, s_dot, s_noise, stream);
}

int rw_blur_adj_phase_keys(const float* g_pre, const float* scale_bc, const float* kernel4x4, int B,
                           int C, int H, int W, void* hi, void* lo, rw_stream_t stream) {
  if (!g_pre || !kernel4x4 || !hi || !lo || B < 1 || H < 1 || W < 1) {
    set_last_error("rw_blur_adj_phase_keys: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return blur_adj_phase_launch(g_pre, scale_bc, kernel4x4, B, C, H, W, hi, lo, stream);
}

int rw_dgrad_finish(float* dk, const float* x, const float* style, int B, int C, int HW,
                    float* gs_raw, rw_stream_t stream) {
  if (!dk || !x || !style || !gs_raw || B < 0 || C < 1 || HW < 0) {
    set_last_error("rw_dgrad_finish: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return dgrad_finish_launch(dk, x, style, B, C, HW, gs_raw, stream);
}

int rw_wgrad_finish(const float* dw_toi, const float* w, const float* s_dot, const float* demod,
                    const float* style, int B, int Cout, int Cin, float scale, float* gw,
                    rw_stream_t stream) {
  if (!dw_toi || !w || !gw || Cout < 1 || Cin < 1 || (s_dot && (!demod || !style || B < 1))) {
    set_last_error("rw_wgrad_finish: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return wgrad_finish_launch(dw_toi, w, s_dot, demod, style, B, Cout, Cin, scale, gw, stream);
}

int rw_style_grad_finish(const float* gs_raw, const float* style, const float* s_dot,
                         const float* demod, const float* wsq, int B, int Cout, int Cin,
                         float* g_style, rw_stream_t stream) {
  if (!style || !g_style || B < 1 || Cin < 1 || (s_dot && (!demod || !wsq || Cout < 1))) {
    set_last_error("rw_style_grad_finish: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return style_grad_finish_launch(gs_raw, style, s_dot, demod, wsq, B, Cout, Cin, g_style, stream);
}

int rw_project_rank(const float* w, const float* base, const float* d, int rank, int Cout,
                    int Cin, int taps, float sign, float* out, rw_stream_t stream) {
  if (!w || !d || !out) {
    set_last_error("rw_project_rank: bad argument");
    return RW_ERR_BAD_ARG;
  }
  return project_rank_launch_signed(w, base, d, rank, Cout, Cin, taps, sign, out, stream);
}

int rw_insert_loop(const rw_insert_args* a, rw_stream_t stream) {
  if (!a || !a->W || !a->m || !a->v || !a->d || !a->key_cl || (!a->style && !a->plain_conv) ||
      !a->target || !a->loss_out || (a->has_noise_act && !a->bias)) {
    set_last_error("rw_insert_loop: bad argument");
    return RW_ERR_BAD_ARG;
  }
  InsertLoopParams p;
  memset(&p, 0, sizeof(p));
  p.W = a->W; p.m = a->m; p.v = a->v; p.w_ortho = a->w_ortho; p.d = a->d; p.rank = a->rank;
  p.key = a->key_cl; p.style = a->style; p.target = a->target; p.noise = a->noise;
  p.noise_w = a->noise_w; p.bias = a->bias;
  p.B = a->B; p.Cin = a->Cin; p.Cout = a->Cout; p.h = a->h; p.w = a->w;
  p.has_noise_act = a->has_noise_act;
  p.lr = a->lr; p.beta1 = a->beta1; p.beta2 = a->beta2; p.eps = a->eps;
  p.it0 = a->it0; p.niter_total = a->niter_total; p.nsteps = a->nsteps;
  p.piter = a->piter > 0 ? a->piter : 1;
  p.project_gradient = a->project_gradient;
  p.loss_out = a->loss_out;
  p.plain_conv = a->plain_conv;
  p.one_minus_beta1 = a->one_minus_beta1 != 0.f ? a->one_minus_beta1 : 1.0f - a->beta1;
  p.one_minus_beta2 = a->one_minus_beta2 != 0.f ? a->one_minus_beta2 : 1.0f - a->beta2;
  p.beta1_exact = a->beta1_exact != 0.0 ? a->beta1_exact : static_cast<double>(a->beta1);
  p.beta2_exact = a->beta2_exact != 0.0 ? a->beta2_exact : static_cast<double>(a->beta2);
  return insert_loop_launch(p, stream);
}

int rw_debug_rowgemm(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo,
                     int rows, int K, int N, float* out, rw_stream_t stream) {
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  p.rows = rows; p.Cin = K; p.Cout = N; p.nphase = 1; p.ph_ntaps[0] = 1;
  p.Hp = 1; p.Wp = rows; p.ph_Hv[0] = 1; p.ph_Wv[0] = rows;   // one "image" = all rows
  p.out = out; p.out_sb = 0; p.out_sc = 1; p.out_sy = 0; p.out_sx = N;  // row-major [rows][N]
  return conv_tc_launch(p, a_hi, a_lo, w_hi, w_lo, K, stream);
}

int rw_rowgemm(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, int rows, int K,
               int N, float* out, rw_stream_t stream) {
  if (!a_hi || !a_lo || !w_hi || !w_lo || !out || rows < 1 || K % 64 != 0 || N % 128 != 0) {
    set_last_error("rw_rowgemm: bad argument (rows=%d K=%d N=%d)", rows, K, N);
    return RW_ERR_BAD_ARG;
  }
  return rw_debug_rowgemm(a_hi, a_lo, w_hi, w_lo, rows, K, N, out, stream);
}

int rw_debug_colgemm(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                     int rows, int Cm, int Cn, int lbo_bytes, int sbo_bytes, float* out,
                     void* workspace, size_t workspace_bytes, rw_stream_t stream) {
  GramTcParams p;
  memset(&p, 0, sizeof(p));
  p.rows = rows; p.rows_a = p.rows_b = rows; p.Cm = Cm; p.Cn = Cn; p.ntaps = 1;
  p.splits = gram_splits((Cm / 128) * (Cn / 128), rows, 1);
  p.ldp = Cn;
  p.partial = static_cast<float*>(workspace);
  const size_t need = static_cast<size_t>(p.splits) * Cm * Cn * sizeof(float);
  if (workspace_bytes < need) {
    set_last_error("rw_debug_colgemm: workspace %zu < %zu bytes", workspace_bytes, need);
    return RW_ERR_BAD_ARG;
  }
  if (lbo_bytes > 0 && sbo_bytes > 0) gram_tc_set_desc(lbo_bytes, sbo_bytes);
  int rc = gram_tc_launch(p, a_hi, a_lo, b_hi, b_lo, stream);
  if (rc) return rc;
  return reduce_partials_launch(p.partial, p.splits, Cm, Cn, p.ldp, out, Cn, 0, 0, stream);
}

}  // extern "C"
