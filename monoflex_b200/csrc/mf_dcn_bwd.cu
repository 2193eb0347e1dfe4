// Backward of the fused DCNv2 layer on the NHWC fp16 training path (row R5; reference _DCNv2.backward dcn_v2.py:35-51 ->
// dcn_v2_cuda_backward dcn_v2_cuda.cu:206-335). 3x3 / stride 1 / pad 1 / one deformable group, like the fused forward.
// The two GEMMs run on the existing tensor-core kernels; this file holds the two sampling kernels around them:
//   dcn_sample_cols   cols[p, tap*C + c] = mask * bilinear(x[., c], p, tap)   (fp16, the forward's A operand written out).
//                     dW = cols^T dY then is `mf_conv2d_wgrad_nhwc_f16` with k = 1 on a 9C-channel "image".
//   dcn_col2im        takes gcol[p, tap*C + c] = sum_co dY[p, co] W[co, c, tap] (a 1x1 forward conv of dY with W^T) and
//                     scatters gcol * mask * corner-weight into dX (half2 atomics; the reference's col2im also uses atomics),
//                     and reduces, over the channels of each (pixel, tap), the offset and mask gradients (the reference's
//                     col2im_coord). The mask gradient is multiplied by m (1 - m): the offset conv applies the sigmoid in its
//                     epilogue (ACT_OFFMASK), so its backward wants the pre-activation gradient. One row [32] fp32 per pixel:
//                     18 offset gradients (dy, dx interleaved per tap), 9 mask pre-activation gradients, 5 zeros.
#include "mf_common.cuh"
#include "mf_launch.h"

namespace mf {

struct DcnRec {
  float w[4];        // bilinear corner weights (0 where the corner is outside), WITHOUT the mask
  float dh[4], dw[4];
  int idx[4];        // clamped corner pixel indices (y * W + x)
  float mask;
  bool inside;
};
MF_DEVINL DcnRec dcn_rec(const float* __restrict__ om, int H, int W, int y, int x, int tap) {
  DcnRec r;
#pragma unroll
  for (int q = 0; q < 4; ++q) { r.w[q] = r.dh[q] = r.dw[q] = 0.f; r.idx[q] = 0; }
  const int ky = tap / 3, kx = tap - ky * 3;
  const float h_im = static_cast<float>(y - 1 + ky) + __ldg(om + 2 * tap);
  const float w_im = static_cast<float>(x - 1 + kx) + __ldg(om + 2 * tap + 1);
  r.mask = __ldg(om + 18 + tap);
  r.inside = h_im > -1.f && w_im > -1.f && h_im < static_cast<float>(H) && w_im < static_cast<float>(W);
  if (!r.inside) return r;
  const float hlf = floorf(h_im), wlf = floorf(w_im);
  const float lh = h_im - hlf, lw = w_im - wlf, hh = 1.f - lh, hw = 1.f - lw;
  const int hl = static_cast<int>(hlf), wl = static_cast<int>(wlf), hi = hl + 1, wi = wl + 1;
  const bool tp = hl >= 0, bt = hi <= H - 1, lf = wl >= 0, rt = wi <= W - 1;
  const int hlc = max(hl, 0), hic = min(hi, H - 1), wlc = max(wl, 0), wic = min(wi, W - 1);
  r.idx[0] = hlc * W + wlc; r.idx[1] = hlc * W + wic; r.idx[2] = hic * W + wlc; r.idx[3] = hic * W + wic;
  if (tp && lf) { r.w[0] = hh * hw; r.dh[0] = -hw; r.dw[0] = -hh; }
  if (tp && rt) { r.w[1] = hh * lw; r.dh[1] = -lw; r.dw[1] = hh; }
  if (bt && lf) { r.w[2] = lh * hw; r.dh[2] = hw; r.dw[2] = -lh; }
  if (bt && rt) { r.w[3] = lh * lw; r.dh[3] = lw; r.dw[3] = lh; }
  return r;
}
// red.global.add.noftz.v4.f16x2 (sm_90+): 8 fp16 additions to 16 contiguous, 16-byte aligned bytes as ONE L2 reduction request
MF_DEVINL void red_add_v4_f16x2(__half* addr, const __half2 (&v)[4]) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(v);
  asm volatile("red.global.add.noftz.v4.f16x2 [%0], {%1, %2, %3, %4};" ::"l"(addr), "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3])
               : "memory");
}
MF_DEVINL void dcn_unpack8(const uint4& v, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 t = __half22float2(h[e]);
    f[2 * e] = t.x; f[2 * e + 1] = t.y;
  }
}

// one thread per (pixel, tap, 8-channel chunk)
__global__ void __launch_bounds__(256) dcn_sample_cols_kernel(const __half* __restrict__ x, int x_ld, const float* __restrict__ om,
                                                              int om_ld, __half* __restrict__ cols, int B, int H, int W, int C) {
  const int CV = C / 8;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * H * W * 9 * CV) return;
  const int cv = static_cast<int>(i % CV);
  long long t = i / CV;
  const int tap = static_cast<int>(t % 9);
  const long long pix = t / 9;
  const int xx = static_cast<int>(pix % W);
  const long long t2 = pix / W;
  const int yy = static_cast<int>(t2 % H);
  const long long b = t2 / H;
  const DcnRec r = dcn_rec(om + pix * om_ld, H, W, yy, xx, tap);
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
  if (r.inside) {
    const __half* xb = x + b * H * W * x_ld + cv * 8;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float v[8];
      dcn_unpack8(__ldg(reinterpret_cast<const uint4*>(xb + static_cast<long long>(r.idx[q]) * x_ld)), v);
      const float wq = r.w[q] * r.mask;                       // same rounding points as the fused forward producer
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += wq * v[e];
    }
  }
  __half2 o[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) o[e] = __floats2half2_rn(acc[2 * e], acc[2 * e + 1]);
  *reinterpret_cast<uint4*>(cols + pix * (9LL * C) + tap * C + cv * 8) = *reinterpret_cast<uint4*>(o);
}

// L lanes (a power of two <= 32) cooperate on one (pixel, tap): lane l handles chunks l, l + L, ...
__global__ void __launch_bounds__(256) dcn_col2im_kernel(const __half* __restrict__ x, int x_ld, const float* __restrict__ om,
                                                         int om_ld, const __half* __restrict__ gcol, __half* __restrict__ dx,
                                                         int dx_ld, float* __restrict__ dom, int B, int H, int W, int C, int L) {
  const int CV = C / 8;
  const long long gid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long item = gid / L;
  const int l = static_cast<int>(gid % L);
  const long long nitems = static_cast<long long>(B) * H * W * 9;
  const bool ok = item < nitems;                                // no early return: every lane takes part in the shuffles below
  const int tap = ok ? static_cast<int>(item % 9) : 0;
  const long long pix = ok ? item / 9 : 0;
  const int xx = static_cast<int>(pix % W);
  const long long t2 = pix / W;
  const int yy = static_cast<int>(t2 % H);
  const long long b = t2 / H;
  const DcnRec r = dcn_rec(om + pix * om_ld, H, W, yy, xx, tap);
  float s_h = 0.f, s_w = 0.f, s_m = 0.f;
  if (ok && r.inside) {
    const __half* xb = x + b * H * W * x_ld;
    __half* dxb = dx + b * H * W * dx_ld;
    for (int cv = l; cv < CV; cv += L) {
      float g[8];
      dcn_unpack8(__ldg(reinterpret_cast<const uint4*>(gcol + pix * (9LL * C) + tap * C + cv * 8)), g);
      float val[8], vh[8], vw[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) val[e] = vh[e] = vw[e] = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float v[8];
        dcn_unpack8(__ldg(reinterpret_cast<const uint4*>(xb + static_cast<long long>(r.idx[q]) * x_ld + cv * 8)), v);
#pragma unroll
        for (int e = 0; e < 8; ++e) { val[e] += r.w[q] * v[e]; vh[e] += r.dh[q] * v[e]; vw[e] += r.dw[q] * v[e]; }
        if (r.w[q] != 0.f) {
          const float wq = r.w[q] * r.mask;
          // ONE 16-byte vector reduction per (corner, 8 channels) instead of four half2 atomics: the 2.6 G half2 atomics of a
          // B = 8 step ran AT the L2 atomic request rate (~220 G/s, 11.8 ms); the vector form is one L2 request
          __half2 hv[4];
#pragma unroll
          for (int h = 0; h < 4; ++h) hv[h] = __floats2half2_rn(g[2 * h] * wq, g[2 * h + 1] * wq);
          red_add_v4_f16x2(dxb + static_cast<long long>(r.idx[q]) * dx_ld + cv * 8, hv);
        }
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) { s_h += g[e] * vh[e]; s_w += g[e] * vw[e]; s_m += g[e] * val[e]; }
    }
  }
  for (int d = L >> 1; d > 0; d >>= 1) {                         // the L lanes of an item are consecutive lanes of one warp
    s_h += __shfl_xor_sync(0xffffffffu, s_h, d);
    s_w += __shfl_xor_sync(0xffffffffu, s_w, d);
    s_m += __shfl_xor_sync(0xffffffffu, s_m, d);
  }
  if (ok && l == 0) {
    float* o = dom + pix * 32;
    o[2 * tap] = s_h * r.mask;
    o[2 * tap + 1] = s_w * r.mask;
    o[18 + tap] = s_m * r.mask * (1.f - r.mask);                 // through the sigmoid of the offset conv's epilogue
    if (tap < 5) o[27 + tap] = 0.f;
  }
}

int launch_dcn_sample_cols(const __half* x, int x_ld, const float* om, int om_ld, __half* cols, int B, int H, int W, int C,
                           cudaStream_t st) {
  if (C % 8 || x_ld % 8 || om_ld < 27) { set_error("dcn_sample_cols: bad shape"); return -1; }
  const long long n = static_cast<long long>(B) * H * W * 9 * (C / 8);
  (void)launch_k(dcn_sample_cols_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, x_ld, om, om_ld, cols,
                 B, H, W, C);
  return check_cuda(cudaGetLastError(), "dcn_sample_cols");
}
int launch_dcn_col2im(const __half* x, int x_ld, const float* om, int om_ld, const __half* gcol, __half* dx, int dx_ld, float* dom,
                      int B, int H, int W, int C, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || dx_ld % 8 || om_ld < 27) { set_error("dcn_col2im: bad shape"); return -1; }
  const int CV = C / 8;
  int L = 1;
  while (L < CV && L < 32) L <<= 1;
  if (check_cuda(cudaMemsetAsync(dx, 0, sizeof(__half) * static_cast<size_t>(B) * H * W * dx_ld, st), "dcn_col2im memset")) return -1;
  const long long n = static_cast<long long>(B) * H * W * 9 * L;
  (void)launch_k(dcn_col2im_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, x_ld, om, om_ld, gcol, dx,
                 dx_ld, dom, B, H, W, C, L);
  return check_cuda(cudaGetLastError(), "dcn_col2im");
}

}  // namespace mf
