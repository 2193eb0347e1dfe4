// C ABI of libmonoflex_b200.so (declared in include/monoflex_b200.h). Plain pointers and sizes only; the caller owns
// every buffer (torch's caching allocator in the Python host), kernels run on the caller's stream, no global state except
// the thread-local last-error string and the debug conv-implementation switch.
#include "mf_common.cuh"
#include "mf_kernels.h"
#include "mf_launch.h"
#include "../../include/monoflex_b200.h"
#include <cstdarg>
#include <cstdio>
#include <cstring>

namespace mf {

static thread_local char g_err[512] = "";
static int g_conv_impl = 0;  // 0 = tcgen05 implicit GEMM, 1 = CUDA-core cross-check

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  set_error("%s: %s", what, cudaGetErrorString(e));
  return -1;
}

// ---------------------------------------------------------------- weight repack: OIHW fp32 -> [n_pad, k_pad] fp16, k = tap*cin_pad + c
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, int Cout, int Cin, int taps, int cin_pad, int n_pad,
                                        int k_pad, __half* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(n_pad) * k_pad) return;
  const int k = static_cast<int>(i % k_pad), n = static_cast<int>(i / k_pad);
  const int tap = k / cin_pad, c = k - tap * cin_pad;
  float v = 0.f;
  if (n < Cout && tap < taps && c < Cin) v = w[(static_cast<long long>(n) * Cin + c) * taps + tap];
  out[i] = __float2half_rn(v);
}
int launch_pack_conv_weight(const float* w, int Cout, int Cin, int kh, int kw, int cin_pad, int n_pad, int k_pad,
                            __half* out, cudaStream_t st) {
  if (cin_pad < Cin || k_pad < kh * kw * cin_pad || n_pad < Cout) { set_error("pack_conv_weight: bad padding"); return -1; }
  const long long n = static_cast<long long>(n_pad) * k_pad;
  pack_conv_weight_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(w, Cout, Cin, kh * kw, cin_pad, n_pad,
                                                                                 k_pad, out);
  return check_cuda(cudaGetLastError(), "pack_conv_weight");
}

// data-gradient weights straight from the live OIHW parameter: the stride-1 dX conv is the forward kernel on dY with the taps
// rotated by 180 degrees and in / out channels transposed - out[n = ci][k = tap' * cout_pad + co] = w[co][ci][taps - 1 - tap']
// (one launch instead of flip + transpose + contiguous + zero-pad cat + pack)
__global__ void pack_conv_weight_dgrad_kernel(const float* __restrict__ w, int Cout, int Cin, int taps, int cout_pad, int n_pad,
                                              int k_pad, __half* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(n_pad) * k_pad) return;
  const int k = static_cast<int>(i % k_pad), n = static_cast<int>(i / k_pad);
  const int tap = k / cout_pad, co = k - tap * cout_pad;
  float v = 0.f;
  if (n < Cin && tap < taps && co < Cout) v = w[(static_cast<long long>(co) * Cin + n) * taps + (taps - 1 - tap)];
  out[i] = __float2half_rn(v);
}
int launch_pack_conv_weight_dgrad(const float* w, int Cout, int Cin, int kh, int kw, int cout_pad, int n_pad, int k_pad,
                                  __half* out, cudaStream_t st) {
  if (cout_pad < Cout || k_pad < kh * kw * cout_pad || n_pad < Cin) { set_error("pack_conv_weight_dgrad: bad padding"); return -1; }
  const long long n = static_cast<long long>(n_pad) * k_pad;
  pack_conv_weight_dgrad_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(w, Cout, Cin, kh * kw, cout_pad, n_pad,
                                                                                       k_pad, out);
  return check_cuda(cudaGetLastError(), "pack_conv_weight_dgrad");
}

// batched form for training plans: all weights of a plan are re-packed from their live fp32 parameters at the start of every
// run - one launch over a device table of descriptors instead of ~190 small ones. desc (5 x int64): w ptr, out ptr,
// Cout | Cin << 32, taps | cin_pad << 32, n_pad | k_pad << 32.
__global__ void pack_conv_weight_batched_kernel(const long long* __restrict__ descs, int n) {
  const int d = blockIdx.y;
  if (d >= n) return;
  const long long* q = descs + 5 * d;
  const float* w = reinterpret_cast<const float*>(q[0]);
  __half* out = reinterpret_cast<__half*>(q[1]);
  const int Cout = static_cast<int>(q[2] & 0xffffffffll), Cin = static_cast<int>(q[2] >> 32);
  const int taps = static_cast<int>(q[3] & 0xffffffffll), cin_pad = static_cast<int>(q[3] >> 32);
  const int n_pad = static_cast<int>(q[4] & 0xffffffffll), k_pad = static_cast<int>(q[4] >> 32);
  const long long total = static_cast<long long>(n_pad) * k_pad;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(i % k_pad), nn = static_cast<int>(i / k_pad);
    const int tap = k / cin_pad, c = k - tap * cin_pad;
    float v = 0.f;
    if (nn < Cout && tap < taps && c < Cin) v = w[(static_cast<long long>(nn) * Cin + c) * taps + tap];
    out[i] = __float2half_rn(v);
  }
}
int launch_pack_conv_weight_batched(const long long* descs, int n, cudaStream_t st) {
  if (n <= 0) return 0;
  pack_conv_weight_batched_kernel<<<dim3(64, n), 256, 0, st>>>(descs, n);
  return check_cuda(cudaGetLastError(), "pack_conv_weight_batched");
}

// boundary B (exact-fp32 `_ext.dcn_v2_forward/backward` on NCHW tensors): kernels and launchers live in mf_dcn_f32.cu

int igemm_block_n(int cout) {
  if (cout <= 16) return 16;
  if (cout <= 32) return 32;
  if (cout <= 64) return 64;
  return 128;
}

static int run_gemm(const IgemmParams& p, const void* wp, int n_pad, int k_pad, int mode, cudaStream_t st) {
  if (g_conv_impl == 1) return launch_simt_gemm(p, static_cast<const __half*>(wp), n_pad, k_pad, mode, st);
  return launch_igemm2(p, static_cast<const __half*>(wp), n_pad, k_pad, mode, st);
}

}  // namespace mf

using namespace mf;
#define MF_STREAM(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

const char* mf_last_error(void) { return g_err; }
int mf_version(void) { return 100; }
int mf_set_conv_impl(int impl) {
  if (impl != 0 && impl != 1) { set_error("mf_set_conv_impl: impl must be 0 or 1"); return -1; }
  g_conv_impl = impl;
  return 0;
}
int mf_conv_block_n(int cout) { return igemm_block_n(cout); }

int mf_pack_conv_weight(const float* w_oihw, int Cout, int Cin, int kh, int kw, int cin_pad, int n_pad, int k_pad,
                        void* out_f16, void* stream) {
  return launch_pack_conv_weight(w_oihw, Cout, Cin, kh, kw, cin_pad, n_pad, k_pad, static_cast<__half*>(out_f16),
                                 MF_STREAM(stream));
}

int mf_pack_conv_weight_dgrad(const float* w_oihw, int Cout, int Cin, int kh, int kw, int cout_pad, int n_pad, int k_pad,
                              void* out_f16, void* stream) {
  return launch_pack_conv_weight_dgrad(w_oihw, Cout, Cin, kh, kw, cout_pad, n_pad, k_pad, static_cast<__half*>(out_f16),
                                       MF_STREAM(stream));
}
int mf_pack_conv_weights_batched(const void* descs_dev, int n, void* stream) {
  return launch_pack_conv_weight_batched(static_cast<const long long*>(descs_dev), n, MF_STREAM(stream));
}

int mf_conv2d_nhwc_f16(const void* x, int x_ld, int B, int H, int W, int Cin, const void* w_packed, int n_pad, int k_pad,
                       int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift,
                       const void* res, int res_ld, int act, int out_mode, void* y, int y_ld, void* stream) {
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  p.x = static_cast<const __half*>(x); p.x_ld = x_ld; p.B = B; p.H = H; p.W = W; p.Cin = Cin;
  p.kh = kh; p.kw = kw; p.stride = stride; p.pad = pad;
  p.Ho = (H + 2 * pad - kh) / stride + 1;
  p.Wo = (W + 2 * pad - kw) / stride + 1;
  p.M = B * p.Ho * p.Wo;
  p.K_real = kh * kw * Cin;
  p.nkb = (p.K_real + 63) / 64;
  p.Cout = Cout; p.scale = scale; p.shift = shift;
  p.res = static_cast<const __half*>(res); p.res_ld = res_ld; p.act = act; p.out_mode = out_mode; p.y = y; p.y_ld = y_ld;
  if (p.Ho <= 0 || p.Wo <= 0 || Cout <= 0) { set_error("mf_conv2d_nhwc_f16: empty output"); return -1; }
  return run_gemm(p, w_packed, n_pad, k_pad, MODE_CONV, MF_STREAM(stream));
}

// strict-precision variants: operands / outputs are hi/lo fp16 pairs (mf_split.cu); K axis of a split-input GEMM = 3 x taps x Cin
int mf_pack_conv_weight_split(const float* w_oihw, int Cout, int Cin, int kh, int kw, int n_pad, int k_pad, void* out_f16,
                              void* stream) {
  return launch_pack_conv_weight_split(w_oihw, Cout, Cin, kh, kw, n_pad, k_pad, static_cast<__half*>(out_f16), MF_STREAM(stream));
}
int mf_conv2d_nhwc_f16x2(const void* x, int x_ld, int x_lo, int B, int H, int W, int Cin, const void* w_packed, int n_pad,
                         int k_pad, int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift,
                         const void* res, int res_ld, int res_lo, int act, int out_mode, void* y, int y_ld, int y_lo,
                         int split_in, int split_out, void* stream) {
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  p.x = static_cast<const __half*>(x); p.x_ld = x_ld; p.B = B; p.H = H; p.W = W; p.Cin = Cin;
  p.kh = kh; p.kw = kw; p.stride = stride; p.pad = pad;
  p.Ho = (H + 2 * pad - kh) / stride + 1;
  p.Wo = (W + 2 * pad - kw) / stride + 1;
  p.M = B * p.Ho * p.Wo;
  p.split_in = split_in ? 1 : 0; p.split_out = split_out ? 1 : 0;
  p.x_lo = x_lo; p.res_lo = res_lo; p.y_lo = y_lo;
  p.cw = Cin < 64 ? Cin : 64;
  p.K_real = (p.split_in ? 3 : 1) * kh * kw * Cin;
  p.nkb = (p.K_real + 63) / 64;
  p.Cout = Cout; p.scale = scale; p.shift = shift;
  p.res = static_cast<const __half*>(res); p.res_ld = res_ld; p.act = act; p.out_mode = out_mode; p.y = y; p.y_ld = y_ld;
  if (p.Ho <= 0 || p.Wo <= 0 || Cout <= 0) { set_error("mf_conv2d_nhwc_f16x2: empty output"); return -1; }
  if (g_conv_impl == 1) { set_error("mf_conv2d_nhwc_f16x2: no CUDA-core cross-check of the split path"); return -1; }
  return launch_igemm2(p, static_cast<const __half*>(w_packed), n_pad, k_pad, MODE_CONV, MF_STREAM(stream));
}
int mf_head_conv_f16x2(const void* x, int x_ld, int x_lo, int B, int H, int W, int Cin, const void* w_packed, int n_pad, int k_pad,
                       int nbranch, const float* scale, const float* shift, int act, const float* w2, float* part, int ntot,
                       const int* out_nch, const int* out_ch0, const int* hid_col, void* hid, int hid_ld, int hid_lo,
                       const unsigned char* hid_mask, void* stream) {
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  if (nbranch <= 0 || nbranch > 12) { set_error("mf_head_conv_f16x2: 1..12 branches"); return -1; }
  p.x = static_cast<const __half*>(x); p.x_ld = x_ld; p.B = B; p.H = H; p.W = W; p.Cin = Cin;
  p.kh = 3; p.kw = 3; p.stride = 1; p.pad = 1; p.Ho = H; p.Wo = W; p.M = B * H * W;
  p.split_in = 1; p.split_out = 0; p.x_lo = x_lo; p.cw = 64;
  p.K_real = 27 * Cin; p.nkb = (p.K_real + 63) / 64;
  p.Cout = nbranch * 256; p.scale = scale; p.shift = shift; p.act = act;
  p.out_mode = OUT_F32_NCHW;                     // no output tensor map: the epilogue writes partial planes + masked hidden rows
  p.y = hid; p.y_ld = hid_ld; p.y_lo = hid_lo;
  p.h2_w = w2; p.h2_part = part; p.h2_ntot = ntot; p.h2_mask = hid_mask;
  bool need_hid = false;
  for (int i = 0; i < nbranch; ++i) {
    if (out_nch[i] < 0 || out_nch[i] > 32 || out_ch0[i] < 0 || out_ch0[i] + out_nch[i] > ntot) {
      set_error("mf_head_conv_f16x2: branch %d has %d outputs at %d of %d", i, out_nch[i], out_ch0[i], ntot);
      return -1;
    }
    p.h2_nch[i] = out_nch[i]; p.h2_ch0[i] = out_ch0[i]; p.h2_hid_col[i] = hid_col[i];
    need_hid = need_hid || hid_col[i] >= 0;
  }
  if (need_hid && (hid == nullptr || hid_mask == nullptr || hid_ld % 8 != 0 || hid_lo % 8 != 0)) {
    set_error("mf_head_conv_f16x2: hidden rows requested without a buffer / mask (or unaligned strides)");
    return -1;
  }
  if (Cin % 64 != 0 || w2 == nullptr || part == nullptr) { set_error("mf_head_conv_f16x2: Cin %% 64, w2 and part are required"); return -1; }
  return launch_igemm2(p, static_cast<const __half*>(w_packed), n_pad, k_pad, MODE_CONV, MF_STREAM(stream));
}
int mf_head2_reduce(const float* part, const float* bias, float* cls, float* reg, int B, int ncls, int nreg, int HW, void* stream) {
  return launch_head2_reduce(part, bias, cls, reg, B, ncls, nreg, HW, MF_STREAM(stream));
}
int mf_dcn_nhwc_f16x2(const void* x, int x_ld, int x_lo, int B, int H, int W, int Cin, const float* offmask, int om_ld,
                      const void* w_packed, int n_pad, int k_pad, int Cout, const float* scale, const float* shift, int act,
                      void* y, int y_ld, int y_lo, void* stream) {
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  p.x = static_cast<const __half*>(x); p.x_ld = x_ld; p.B = B; p.H = H; p.W = W; p.Cin = Cin;
  p.kh = 3; p.kw = 3; p.stride = 1; p.pad = 1; p.Ho = H; p.Wo = W; p.M = B * H * W;
  p.split_in = 1; p.split_out = 1; p.x_lo = x_lo; p.y_lo = y_lo; p.cw = 64;
  p.K_real = 27 * Cin; p.nkb = (p.K_real + 63) / 64;
  p.offmask = offmask; p.om_ld = om_ld;
  p.Cout = Cout; p.scale = scale; p.shift = shift; p.act = act; p.out_mode = OUT_F16_NHWC; p.y = y; p.y_ld = y_ld;
  if (om_ld < 27) { set_error("mf_dcn_nhwc_f16x2: om_ld < 27"); return -1; }
  return launch_igemm2(p, static_cast<const __half*>(w_packed), n_pad, k_pad, MODE_DCN, MF_STREAM(stream));
}
int mf_pack_image_split(const float* x_nchw, void* y_rows16, int B, int C, int H, int W, void* stream) {
  return launch_pack_image_split(x_nchw, static_cast<__half*>(y_rows16), B, C, H, W, MF_STREAM(stream));
}
int mf_maxpool2_split(const void* x, int x_lo, void* y, int y_lo, int B, int H, int W, int C, int x_ld, int y_ld, void* stream) {
  return launch_maxpool2_split(static_cast<const __half*>(x), x_lo, static_cast<__half*>(y), y_lo, B, H, W, C, x_ld, y_ld,
                               MF_STREAM(stream));
}
int mf_upsample_add_split(const void* x, int x_lo, const float* w_taps, const void* skip, int skip_lo, void* y, int y_lo, int B,
                          int Hi, int Wi, int C, int f, int x_ld, int skip_ld, int y_ld, void* stream) {
  return launch_upsample_add_split(static_cast<const __half*>(x), x_lo, w_taps, static_cast<const __half*>(skip), skip_lo,
                                   static_cast<__half*>(y), y_lo, B, Hi, Wi, C, f, x_ld, skip_ld, y_ld, MF_STREAM(stream));
}
int mf_edge_gather_split(const void* feat, int feat_ld, int feat_lo, int ch_a, int ch_b, const long long* edge_idx, void* ea,
                         void* eb, int B, int H, int W, int K, int out_w, int out_h, void* stream) {
  return launch_edge_gather_split(static_cast<const __half*>(feat), feat_ld, feat_lo, ch_a, ch_b, edge_idx,
                                  static_cast<__half*>(ea), static_cast<__half*>(eb), B, H, W, K, out_w, out_h, MF_STREAM(stream));
}
int mf_edge_head_add_split(const void* t, int t_ld, int t_lo, const float* w, const float* bias, int n_out,
                           const long long* edge_idx, const long long* edge_len, float* out, int out_ctot, int out_ch0, int B,
                           int K, int H, int W, void* stream) {
  return launch_edge_head_add_split(static_cast<const __half*>(t), t_ld, t_lo, w, bias, n_out, edge_idx, edge_len, out, out_ctot,
                                    out_ch0, B, K, H, W, MF_STREAM(stream));
}
int mf_split_to_nchw_f32(const void* x, int x_ld, int x_lo, float* y, int B, int C, int HW, void* stream) {
  return launch_split_to_nchw(static_cast<const __half*>(x), x_ld, x_lo, y, B, C, HW, MF_STREAM(stream));
}

int mf_conv2d_rows_f16(const void* x, int B, int H, int W, int Cin, int in_npar, const void* w_packed, int n_pad, int k_pad,
                       int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift, int act,
                       int out_planar, int out_npar, void* y, int y_ld, void* stream) {
  return launch_rows_conv(static_cast<const __half*>(x), B, H, W, Cin, in_npar, static_cast<const __half*>(w_packed), n_pad,
                          k_pad, kh, kw, stride, pad, Cout, scale, shift, act, out_planar, out_npar, static_cast<__half*>(y),
                          y_ld, MF_STREAM(stream));
}

int mf_conv2d_rows_f16x2(const void* x, int B, int H, int W, int Cin, int in_npar, int in_mode, const void* w_packed, int n_pad,
                         int k_pad, int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift, int act,
                         int out_planar, int out_npar, void* y, int y_ld, int y_lo, void* stream) {
  return launch_rows_conv(static_cast<const __half*>(x), B, H, W, Cin, in_npar, static_cast<const __half*>(w_packed), n_pad,
                          k_pad, kh, kw, stride, pad, Cout, scale, shift, act, out_planar, out_npar, static_cast<__half*>(y),
                          y_ld, MF_STREAM(stream), in_mode, 1, y_lo);
}
int mf_pack_image_pair8(const float* x_nchw, void* y_nhwc8, int B, int C, int H, int W, void* stream) {
  return launch_pack_image_pair8(x_nchw, static_cast<__half*>(y_nhwc8), B, C, H, W, MF_STREAM(stream));
}

int mf_head_fused(const void* x, int x_ld, int B, int H, int W, int Cin, const void* w3_packed, const void* w2_packed,
                  const float* scale, const float* shift, const float* bias2, int nbranch, void* const* out_ptrs,
                  const int* out_ctot, const int* out_nch, const int* hid_col, void* hid, int hid_ld,
                  const unsigned char* hid_mask, void* stream) {
  return launch_head_fused(static_cast<const __half*>(x), x_ld, B, H, W, Cin, static_cast<const __half*>(w3_packed),
                           static_cast<const __half*>(w2_packed), scale, shift, bias2, nbranch,
                           reinterpret_cast<float* const*>(out_ptrs), out_ctot, out_nch, hid_col, static_cast<__half*>(hid),
                           hid_ld, hid_mask, MF_STREAM(stream));
}
int mf_edge_mask(const long long* edge_idx, unsigned char* mask, int B, int K, int H, int W, int out_w, int out_h,
                 void* stream) {
  return launch_edge_mask(edge_idx, mask, B, K, H, W, out_w, out_h, MF_STREAM(stream));
}

int mf_dcn_nhwc_f16(const void* x, int x_ld, int B, int H, int W, int Cin, const float* offmask, int om_ld,
                    const void* w_packed, int n_pad, int k_pad, int Cout, const float* scale, const float* shift, int act,
                    int out_mode, void* y, int y_ld, void* stream) {
  IgemmParams p;
  memset(&p, 0, sizeof(p));
  p.x = static_cast<const __half*>(x); p.x_ld = x_ld; p.B = B; p.H = H; p.W = W; p.Cin = Cin;
  p.kh = 3; p.kw = 3; p.stride = 1; p.pad = 1; p.Ho = H; p.Wo = W; p.M = B * H * W;
  p.K_real = 9 * Cin; p.nkb = (p.K_real + 63) / 64;
  p.offmask = offmask; p.om_ld = om_ld;
  p.Cout = Cout; p.scale = scale; p.shift = shift; p.act = act; p.out_mode = out_mode; p.y = y; p.y_ld = y_ld;
  if (om_ld < 27) { set_error("mf_dcn_nhwc_f16: om_ld < 27"); return -1; }
  return run_gemm(p, w_packed, n_pad, k_pad, MODE_DCN, MF_STREAM(stream));
}

int mf_pack_image(const float* x_nchw, void* y_nhwc8, int B, int C, int H, int W, void* stream) {
  return launch_pack_image(x_nchw, static_cast<__half*>(y_nhwc8), B, C, H, W, MF_STREAM(stream));
}
int mf_nchw_f32_to_nhwc_f16(const float* x, void* y, int B, int C, int HW, int y_ld, void* stream) {
  return launch_nchw_to_nhwc(x, static_cast<__half*>(y), B, C, HW, y_ld, MF_STREAM(stream));
}
int mf_nhwc_f16_to_nchw_f32(const void* x, float* y, int B, int C, int HW, int x_ld, void* stream) {
  return launch_nhwc_to_nchw(static_cast<const __half*>(x), y, B, C, HW, x_ld, MF_STREAM(stream));
}
int mf_pack_offmask(const float* offset, const float* mask, float* y, int B, int HW, void* stream) {
  return launch_pack_offmask(offset, mask, y, B, HW, MF_STREAM(stream));
}
int mf_maxpool2_nhwc_f16(const void* x, void* y, int B, int H, int W, int C, int x_ld, int y_ld, void* stream) {
  return launch_maxpool2(static_cast<const __half*>(x), static_cast<__half*>(y), B, H, W, C, x_ld, y_ld, MF_STREAM(stream));
}
int mf_upsample_add_nhwc_f16(const void* x, const float* w_taps, const void* skip, void* y, int B, int Hi, int Wi, int C,
                             int f, int x_ld, int skip_ld, int y_ld, void* stream) {
  return launch_upsample_add(static_cast<const __half*>(x), w_taps, static_cast<const __half*>(skip),
                             static_cast<__half*>(y), B, Hi, Wi, C, f, x_ld, skip_ld, y_ld, MF_STREAM(stream));
}
int mf_edge_gather(const void* feat, int feat_ld, int ch_a, int ch_b, const long long* edge_idx, void* ea, void* eb, int B,
                   int H, int W, int K, int out_w, int out_h, void* stream) {
  return launch_edge_gather(static_cast<const __half*>(feat), feat_ld, ch_a, ch_b, edge_idx, static_cast<__half*>(ea),
                            static_cast<__half*>(eb), B, H, W, K, out_w, out_h, MF_STREAM(stream));
}
int mf_edge_head_add(const void* t, const float* w, const float* bias, int n_out, const long long* edge_idx,
                     const long long* edge_len, float* out, int out_ctot, int out_ch0, int B, int K, int H, int W,
                     void* stream) {
  return launch_edge_head_add(static_cast<const __half*>(t), w, bias, n_out, edge_idx, edge_len, out, out_ctot, out_ch0, B,
                              K, H, W, MF_STREAM(stream));
}
int mf_sigmoid_clamp(float* x, long long n, void* stream) { return launch_sigmoid_clamp(x, n, MF_STREAM(stream)); }
int mf_focal_loss_forward(const float* pred, const float* target, long long n, float* out2, void* stream) {
  return launch_focal_loss(pred, target, n, out2, MF_STREAM(stream));
}
int mf_focal_loss_backward(const float* pred, const float* target, long long n, const float* scale, float* grad_pred,
                           void* stream) {
  return launch_focal_loss_backward(pred, target, n, scale, grad_pred, MF_STREAM(stream));
}
int mf_conv2d_wgrad_nhwc_f16(const void* x, int x_ld, int B, int H, int W, int Cin, const void* dy, int dy_ld, int Cout, int k,
                             int stride, int pad, float* dw, void* stream) {
  return launch_conv_wgrad(static_cast<const __half*>(x), x_ld, B, H, W, Cin, static_cast<const __half*>(dy), dy_ld, Cout, k, k,
                           stride, pad, pad, dw, MF_STREAM(stream));
}
int mf_conv2d_wgrad_rect_nhwc_f16(const void* x, int x_ld, int B, int H, int W, int Cin, const void* dy, int dy_ld, int Cout, int kh,
                                  int kw, int stride, int pad_h, int pad_w, float* dw, void* stream) {
  return launch_conv_wgrad(static_cast<const __half*>(x), x_ld, B, H, W, Cin, static_cast<const __half*>(dy), dy_ld, Cout, kh, kw,
                           stride, pad_h, pad_w, dw, MF_STREAM(stream));
}
int mf_maxpool2_bwd_nhwc_f16(const void* x, const void* dy, void* dx, int B, int H, int W, int C, int x_ld, int dy_ld, int dx_ld,
                             void* stream) {
  return launch_maxpool2_bwd(static_cast<const __half*>(x), static_cast<const __half*>(dy), static_cast<__half*>(dx), B, H, W, C,
                             x_ld, dy_ld, dx_ld, MF_STREAM(stream));
}
size_t mf_upsample_bwd_workspace(int B, int Hi, int Wi, int C, int f) { return sizeof(float) * upsample_bwd_workspace_floats(B, Hi, Wi, C, f); }
int mf_upsample_bwd_nhwc_f16(const void* x, const float* w_taps, const void* dy, void* dx, float* dw_taps, int B, int Hi, int Wi,
                             int C, int f, int x_ld, int dy_ld, int dx_ld, float* workspace, void* stream) {
  return launch_upsample_bwd(static_cast<const __half*>(x), w_taps, static_cast<const __half*>(dy), static_cast<__half*>(dx),
                             dw_taps, B, Hi, Wi, C, f, x_ld, dy_ld, dx_ld, workspace, MF_STREAM(stream));
}
int mf_sigmoid_clamp_bwd(const float* y, const float* dy, float* dx, long long n, void* stream) {
  return launch_sigmoid_clamp_bwd(y, dy, dx, n, MF_STREAM(stream));
}
size_t mf_column_sum_workspace(long long M, int C) { return sizeof(float) * column_sum_workspace_floats(M, C); }
int mf_column_sum_nhwc_f16(const void* x, int x_ld, long long M, int C, float* out, float* workspace, void* stream) {
  return launch_column_sum(static_cast<const __half*>(x), x_ld, M, C, out, workspace, MF_STREAM(stream));
}
int mf_edge_gather_bwd(const void* d_ea, const void* d_eb, int ch_a, int ch_b, const long long* edge_idx, void* d_feat, int feat_ld,
                       int B, int H, int W, int K, int out_w, int out_h, void* stream) {
  return launch_edge_gather_bwd(static_cast<const __half*>(d_ea), static_cast<const __half*>(d_eb), ch_a, ch_b, edge_idx,
                                static_cast<__half*>(d_feat), feat_ld, B, H, W, K, out_w, out_h, MF_STREAM(stream));
}
int mf_edge_head_add_bwd(const void* t, const float* w, int n_out, const long long* edge_idx, const long long* edge_len,
                         const float* d_out, int out_ctot, int out_ch0, void* d_t, float* dw, float* dbias, int B, int K, int H,
                         int W, void* stream) {
  return launch_edge_head_add_bwd(static_cast<const __half*>(t), w, n_out, edge_idx, edge_len, d_out, out_ctot, out_ch0,
                                  static_cast<__half*>(d_t), dw, dbias, B, K, H, W, MF_STREAM(stream));
}
int mf_add_rows_f16(void* dst, int dst_ld, const void* src, int src_ld, long long M, int C, void* stream) {
  return launch_add_rows(static_cast<__half*>(dst), dst_ld, static_cast<const __half*>(src), src_ld, M, C, MF_STREAM(stream));
}
int mf_interleave2x2_nhwc_f16(const void* p00, const void* p01, const void* p10, const void* p11, int part_ld, void* out, int out_ld,
                              int B, int Hh, int Wh, int C, void* stream) {
  return launch_interleave2x2(static_cast<const __half*>(p00), static_cast<const __half*>(p01), static_cast<const __half*>(p10),
                              static_cast<const __half*>(p11), part_ld, static_cast<__half*>(out), out_ld, B, Hh, Wh, C,
                              MF_STREAM(stream));
}
int mf_dcn_sample_cols_nhwc_f16(const void* x, int x_ld, const float* offmask, int om_ld, void* cols, int B, int H, int W, int C,
                                void* stream) {
  return launch_dcn_sample_cols(static_cast<const __half*>(x), x_ld, offmask, om_ld, static_cast<__half*>(cols), B, H, W, C,
                                MF_STREAM(stream));
}
int mf_dcn_col2im_nhwc_f16(const void* x, int x_ld, const float* offmask, int om_ld, const void* gcol, void* dx, int dx_ld,
                           float* d_offmask, int B, int H, int W, int C, void* stream) {
  return launch_dcn_col2im(static_cast<const __half*>(x), x_ld, offmask, om_ld, static_cast<const __half*>(gcol),
                           static_cast<__half*>(dx), dx_ld, d_offmask, B, H, W, C, MF_STREAM(stream));
}
size_t mf_bn_train_workspace(long long M, int C) { return sizeof(float) * bn_train_workspace_floats(M, C); }
int mf_bn_train_forward(const void* x, int x_ld, long long M, int C, const float* gamma, const float* beta, float eps,
                        float momentum, int abs_gamma, float* running_mean, float* running_var, const void* res, int res_ld,
                        int act, void* y, int y_ld, float* mean, float* rstd, float* scale, float* shift, float* workspace,
                        void* stream) {
  return launch_bn_train_forward(static_cast<const __half*>(x), x_ld, M, C, gamma, beta, eps, momentum, abs_gamma, running_mean,
                                 running_var, static_cast<const __half*>(res), res_ld, act, static_cast<__half*>(y), y_ld, mean,
                                 rstd, scale, shift, workspace, MF_STREAM(stream));
}
int mf_bn_train_backward(const void* x, int x_ld, const void* dy, int dy_ld, const void* y, int y_ld, long long M, int C,
                         const float* mean, const float* rstd, const float* scale, int act, void* dx, int dx_ld, void* dres,
                         int dres_ld, float* dgamma, float* dbeta, float* workspace, void* stream) {
  return launch_bn_train_backward(static_cast<const __half*>(x), x_ld, static_cast<const __half*>(dy), dy_ld,
                                  static_cast<const __half*>(y), y_ld, M, C, mean, rstd, scale, act, static_cast<__half*>(dx),
                                  dx_ld, static_cast<__half*>(dres), dres_ld, dgamma, dbeta, workspace, MF_STREAM(stream));
}
int mf_bn_sync_forward_stats(const void* x, int x_ld, long long M, int C, float* workspace, double* sums, void* stream) {
  return launch_bn_sync_forward_stats(static_cast<const __half*>(x), x_ld, M, C, workspace, sums, MF_STREAM(stream));
}
int mf_bn_sync_forward_apply(const void* x, int x_ld, long long M, int C, const double* sums, double count, const float* gamma,
                             const float* beta, float eps, float momentum, int abs_gamma, float* running_mean, float* running_var,
                             const void* res, int res_ld, int act, void* y, int y_ld, float* mean, float* rstd, float* scale,
                             float* shift, void* stream) {
  return launch_bn_sync_forward_apply(static_cast<const __half*>(x), x_ld, M, C, sums, count, gamma, beta, eps, momentum, abs_gamma,
                                      running_mean, running_var, static_cast<const __half*>(res), res_ld, act,
                                      static_cast<__half*>(y), y_ld, mean, rstd, scale, shift, MF_STREAM(stream));
}
int mf_bn_sync_backward_stats(const void* x, int x_ld, const void* dy, int dy_ld, const void* y, int y_ld, long long M, int C,
                              const float* mean, const float* rstd, int act, float* workspace, double* sums, float* dgamma,
                              float* dbeta, void* stream) {
  return launch_bn_sync_backward_stats(static_cast<const __half*>(x), x_ld, static_cast<const __half*>(dy), dy_ld,
                                       static_cast<const __half*>(y), y_ld, M, C, mean, rstd, act, workspace, sums, dgamma, dbeta,
                                       MF_STREAM(stream));
}
int mf_bn_sync_backward_apply(const void* x, int x_ld, const void* dy, int dy_ld, const void* y, int y_ld, long long M, int C,
                              const float* mean, const float* rstd, const float* scale, const double* sums, double count, int act,
                              void* dx, int dx_ld, void* dres, int dres_ld, float* workspace, void* stream) {
  return launch_bn_sync_backward_apply(static_cast<const __half*>(x), x_ld, static_cast<const __half*>(dy), dy_ld,
                                       static_cast<const __half*>(y), y_ld, M, C, mean, rstd, scale, sums, count, act,
                                       static_cast<__half*>(dx), dx_ld, static_cast<__half*>(dres), dres_ld, workspace,
                                       MF_STREAM(stream));
}
int mf_selftest_mn_major(const void* a_km, const void* b_kn, float* d_mn, void* stream) {
  return launch_mn_major_selftest(static_cast<const __half*>(a_km), static_cast<const __half*>(b_kn), d_mn, MF_STREAM(stream));
}
int mf_loss_obj_cols(void) { return MF_LOSS_OBJ_COLS; }
int mf_loss_forward(const float* pred_cls, const float* hm, const float* pred_reg, const float* obj, const float* img,
                    const float* weights11, const float* dim_mean9, int B, int ncls, int M, int H, int W, int C,
                    float* out48, float* ws64, void* stream) {
  return launch_loss_forward(pred_cls, hm, pred_reg, obj, img, weights11, dim_mean9, B, ncls, M, H, W, C, out48, ws64,
                             MF_STREAM(stream));
}
int mf_loss_backward(const float* pred_cls, const float* hm, const float* pred_reg, const float* obj, const float* img,
                     const float* weights11, const float* dim_mean9, int B, int ncls, int M, int H, int W, int C,
                     const float* ws64, const float* grad_losses11, float* grad_cls, float* grad_reg, void* stream) {
  return launch_loss_backward(pred_cls, hm, pred_reg, obj, img, weights11, dim_mean9, B, ncls, M, H, W, C, ws64,
                              grad_losses11, grad_cls, grad_reg, MF_STREAM(stream));
}
int mf_adamw_chunk(void) { return MF_ADAMW_CHUNK; }
int mf_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, const float* chunk_lr,
                  long long n_chunks, float beta1, float beta2, float eps, float weight_decay, long long step,
                  float grad_scale, float lr_scale, void* stream) {
  return launch_adamw_arena(params, grads, exp_avg, exp_avg_sq, chunk_lr, n_chunks, beta1, beta2, eps, weight_decay, step,
                            grad_scale, lr_scale, MF_STREAM(stream));
}
int mf_adamw_step_dyn(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, const float* chunk_lr,
                      long long n_chunks, float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                      float lr_scale, long long* state4, void* dyn16, int check_finite, void* stream) {
  return launch_adamw_arena_dyn(params, grads, exp_avg, exp_avg_sq, chunk_lr, n_chunks, beta1, beta2, eps, weight_decay,
                                grad_scale, lr_scale, state4, dyn16, check_finite, MF_STREAM(stream));
}
int mf_adamw_step_p2p(const unsigned long long* param_ptrs, const unsigned long long* grad_ptrs, int world, int rank,
                      unsigned long long mc_params, unsigned long long mc_grads, float* exp_avg, float* exp_avg_sq,
                      const float* chunk_lr, long long n_chunks, float beta1, float beta2, float eps, float weight_decay,
                      long long step, float lr_scale, void* stream) {
  return launch_adamw_p2p(param_ptrs, grad_ptrs, world, rank, mc_params, mc_grads, exp_avg, exp_avg_sq, chunk_lr, n_chunks,
                          beta1, beta2, eps, weight_decay, step, lr_scale, MF_STREAM(stream));
}
int mf_preprocess_images_u8(const void* const* src_ptrs, const int* hw4, const int* flip, int B, int H, int W,
                            const float* mean3, const float* std3, int to_bgr, float* out_nchw, void* stream) {
  return launch_preprocess_u8(reinterpret_cast<const unsigned char* const*>(src_ptrs), hw4, flip, B, H, W, mean3, std3, to_bgr,
                              out_nchw, MF_STREAM(stream));
}
int mf_draw_heatmaps(const int* obj6, int B, int max_objs, int ncls, int H, int W, float* hm, void* stream) {
  return launch_draw_heatmap(obj6, B, max_objs, ncls, H, W, hm, MF_STREAM(stream));
}
int mf_nms_hm(const float* heat, float* out, int planes, int H, int W, void* stream) {
  return launch_nms_hm(heat, out, planes, H, W, MF_STREAM(stream));
}
int mf_decode_detections(const float* heat, const float* reg, const float* calib, const float* pad, const float* size,
                         const float* dim_mean, int B, int C, int H, int W, int R, int K, float thresh, int apply_sigmoid,
                         float* ws_score, int* ws_idx, float* scores, long long* inds, float* clses, float* ys, float* xs,
                         float* pois, float* result, int* count, void* stream) {
  return launch_decode(heat, reg, calib, pad, size, dim_mean, B, C, H, W, R, K, thresh, apply_sigmoid, ws_score, ws_idx,
                       scores, inds, clses, ys, xs, pois, result, count, MF_STREAM(stream));
}

int mf_dcn_v2_forward(const float* x, const float* w, const float* bias, const float* offset, const float* mask, float* y,
                      int B, int Cin, int H, int W, int Cout, int kh, int kw, int sh, int sw, int ph, int pw, int dh,
                      int dw, int dg, void* workspace, size_t ws_bytes, void* stream) {
  (void)workspace; (void)ws_bytes;
  return launch_dcn_v2_forward_f32(x, w, bias, offset, mask, y, B, Cin, H, W, Cout, kh, kw, sh, sw, ph, pw, dh, dw, dg,
                                   MF_STREAM(stream));
}
size_t mf_dcn_v2_backward_workspace(int B, int Cin, int H, int W, int Cout, int kh, int kw, int sh, int sw, int ph, int pw,
                                    int dh, int dw, int dg) {
  return dcn_v2_backward_f32_workspace(B, Cin, H, W, Cout, kh, kw, sh, sw, ph, pw, dh, dw, dg);
}
int mf_dcn_v2_backward(const float* x, const float* w, const float* bias, const float* offset, const float* mask,
                       const float* grad_y, float* grad_x, float* grad_offset, float* grad_mask, float* grad_w,
                       float* grad_bias, int B, int Cin, int H, int W, int Cout, int kh, int kw, int sh, int sw, int ph,
                       int pw, int dh, int dw, int dg, void* workspace, size_t ws_bytes, void* stream) {
  (void)bias;
  return launch_dcn_v2_backward_f32(x, w, offset, mask, grad_y, grad_x, grad_offset, grad_mask, grad_w, grad_bias, B, Cin, H,
                                    W, Cout, kh, kw, sh, sw, ph, pw, dh, dw, dg, workspace, ws_bytes, MF_STREAM(stream));
}
int mf_dcn_v2_psroi_pooling_forward(void) {
  set_error("dcn_v2_psroi_pooling_forward: not built (dead code for MonoFlex, SURVEY 2.2 K6)");
  return -2;
}
int mf_dcn_v2_psroi_pooling_backward(void) {
  set_error("dcn_v2_psroi_pooling_backward: not built (dead code for MonoFlex, SURVEY 2.2 K6)");
  return -2;
}

}  // extern "C"
