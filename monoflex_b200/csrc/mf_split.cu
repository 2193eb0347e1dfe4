// Strict-precision ("split") companions of the HBM-bound layout kernels (mf_elementwise.cu) and the split weight packer.
//
// Number format: an fp32-grade value v travels as TWO fp16 numbers, hi = fp16(v) and lo = fp16(v - hi) (22 significant
// bits, absolute floor 2^-25), stored in the same NHWC pixel row: the lo block starts `*_lo` elements after the hi block
// (engine.py gives every strict activation buffer the row layout [hi channels | lo channels]). The tensor-core kernels
// consume such operands as the K-concatenation A_hi W_hi + A_lo W_hi + A_hi W_lo (mf_igemm2.cu, `split_in`), which is what
// brings the end-to-end forward within 1e-3 of the fp32 reference (DESIGN.md §4 "Precision modes"); everything here is the
// plumbing between those GEMMs: image packing, max-pool, depth-wise up-sampling + add, the edge-fusion gather / final add.
#include "mf_common.cuh"
#include "mf_kernels.h"
#include "mf_launch.h"

namespace mf {

MF_DEVINL void ld8_split(const __half* p, int lo, float (&f)[8]) {
  const uint4 h = __ldg(reinterpret_cast<const uint4*>(p));
  const uint4 l = __ldg(reinterpret_cast<const uint4*>(p + lo));
  const __half2* hh = reinterpret_cast<const __half2*>(&h);
  const __half2* ll = reinterpret_cast<const __half2*>(&l);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 a = __half22float2(hh[e]), b = __half22float2(ll[e]);
    f[2 * e] = a.x + b.x;
    f[2 * e + 1] = a.y + b.y;
  }
}
MF_DEVINL void st8_split(__half* p, int lo, const float (&f)[8]) {
  __half2 h[4], l[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    h[e] = __floats2half2_rn(f[2 * e], f[2 * e + 1]);
    const float2 hf = __half22float2(h[e]);
    l[e] = __floats2half2_rn(f[2 * e] - hf.x, f[2 * e + 1] - hf.y);
  }
  *reinterpret_cast<uint4*>(p) = *reinterpret_cast<uint4*>(h);
  *reinterpret_cast<uint4*>(p + lo) = *reinterpret_cast<uint4*>(l);
}

// ---------------------------------------------------------------- split weight packer
// OIHW fp32 -> [n_pad, k_pad] fp16 in the virtual K order of `split_in` GEMMs:
//   k' = (((tap * nchunk + chunk) * 3 + which) * cw + c),  cw = min(Cin, 64), channel = chunk * cw + c,
//   which 0, 1 -> W_hi (multiplies A_hi, A_lo), which 2 -> W_lo = fp16(W - W_hi) (multiplies A_hi).
__global__ void pack_conv_weight_split_kernel(const float* __restrict__ w, int Cout, int Cin, int taps, int cw, int n_pad,
                                              int k_pad, __half* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(n_pad) * k_pad) return;
  const int k = static_cast<int>(i % k_pad), n = static_cast<int>(i / k_pad);
  const int unit = k / cw, c = k - unit * cw;
  const int tc = unit / 3, which = unit - tc * 3;
  const int nch = Cin / cw;
  const int tap = tc / nch, ci = (tc - tap * nch) * cw + c;
  __half r = __float2half_rn(0.f);
  if (n < Cout && tap < taps) {
    const float v = w[(static_cast<long long>(n) * Cin + ci) * taps + tap];
    const __half hi = __float2half_rn(v);
    r = which == 2 ? __float2half_rn(v - __half2float(hi)) : hi;
  }
  out[i] = r;
}
int launch_pack_conv_weight_split(const float* w, int Cout, int Cin, int kh, int kw, int n_pad, int k_pad, __half* out,
                                  cudaStream_t st) {
  const int cw = Cin < 64 ? Cin : 64;
  if (Cin % cw != 0 || 64 % cw != 0 || k_pad < 3 * kh * kw * Cin || n_pad < Cout) {
    set_error("pack_conv_weight_split: Cin=%d must be a multiple of 64 or one of 8/16/32; k_pad >= 3*taps*Cin", Cin);
    return -1;
  }
  const long long n = static_cast<long long>(n_pad) * k_pad;
  pack_conv_weight_split_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(w, Cout, Cin, kh * kw, cw, n_pad, k_pad, out);
  return check_cuda(cudaGetLastError(), "pack_conv_weight_split");
}

// ---------------------------------------------------------------- image: NCHW fp32 [B,3,H,W] -> [B*H*W, 16] fp16 rows
// channels [hi(3) | lo(3) | hi(3) | 0 x 7]: the 7x7 stem then is an ORDINARY 16-channel convolution whose per-tap weights are
// [W_hi | W_hi | W_lo | 0] (engine.py), i.e. the three split products in one pass over 16 instead of 3 x 8 channels.
__global__ void pack_image_split_kernel(const float* __restrict__ x, __half* __restrict__ y, int B, int C, long long HW) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= B * HW) return;
  const long long b = i / HW, pix = i - b * HW;
  __half o[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) o[c] = __float2half_rn(0.f);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (c < C) {
      const float v = __ldg(x + (b * C + c) * HW + pix);
      const __half hi = __float2half_rn(v);
      o[c] = hi;
      o[3 + c] = __float2half_rn(v - __half2float(hi));
      o[6 + c] = hi;
    }
  }
  uint4* dst = reinterpret_cast<uint4*>(y + i * 16);
  dst[0] = *reinterpret_cast<uint4*>(&o[0]);
  dst[1] = *reinterpret_cast<uint4*>(&o[8]);
}
int launch_pack_image_split(const float* x, __half* y, int B, int C, int H, int W, cudaStream_t st) {
  if (C > 3) { set_error("pack_image_split: C=%d > 3", C); return -1; }
  const long long n = static_cast<long long>(B) * H * W;
  (void)launch_k(pack_image_split_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, y, B, C,
                 static_cast<long long>(H) * W);
  return check_cuda(cudaGetLastError(), "pack_image_split");
}

// image -> ONE 16-byte-pixel plane [hi3 | lo3 | 0 0] for the row-segment stem kernel (mf_rows.cu, in_mode 1)
__global__ void pack_image_pair8_kernel(const float* __restrict__ x, __half* __restrict__ y, int B, int C, long long HW) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= B * HW) return;
  const long long b = i / HW, pix = i - b * HW;
  __half o[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) o[c] = __float2half_rn(0.f);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (c < C) {
      const float v = __ldg(x + (b * C + c) * HW + pix);
      const __half hi = __float2half_rn(v);
      o[c] = hi;
      o[3 + c] = __float2half_rn(v - __half2float(hi));
    }
  }
  *reinterpret_cast<uint4*>(y + i * 8) = *reinterpret_cast<uint4*>(&o[0]);
}
int launch_pack_image_pair8(const float* x, __half* y, int B, int C, int H, int W, cudaStream_t st) {
  if (C > 3) { set_error("pack_image_pair8: C=%d > 3", C); return -1; }
  const long long n = static_cast<long long>(B) * H * W;
  (void)launch_k(pack_image_pair8_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, y, B, C,
                 static_cast<long long>(H) * W);
  return check_cuda(cudaGetLastError(), "pack_image_pair8");
}

// ---------------------------------------------------------------- MaxPool2d(2) on hi/lo rows
__global__ void maxpool2_split_kernel(const __half* __restrict__ x, int x_lo, __half* __restrict__ y, int y_lo, int B, int H,
                                      int W, int C, int x_ld, int y_ld) {
  const int Ho = H / 2, Wo = W / 2, CV = C / 8;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * Ho * Wo * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long pix = i / CV;
  const int ox = static_cast<int>(pix % Wo);
  const long long t = pix / Wo;
  const int oy = static_cast<int>(t % Ho);
  const long long b = t / Ho;
  const __half* p = x + ((b * H + 2 * oy) * W + 2 * ox) * x_ld + cv * 8;
  float a[8], bq[8], c[8], d[8], o[8];
  ld8_split(p, x_lo, a);
  ld8_split(p + x_ld, x_lo, bq);
  ld8_split(p + static_cast<long long>(W) * x_ld, x_lo, c);
  ld8_split(p + static_cast<long long>(W + 1) * x_ld, x_lo, d);
#pragma unroll
  for (int e = 0; e < 8; ++e) o[e] = fmaxf(fmaxf(a[e], bq[e]), fmaxf(c[e], d[e]));
  st8_split(y + pix * y_ld + cv * 8, y_lo, o);       // hi + lo of one input is exactly representable again: lossless
}
int launch_maxpool2_split(const __half* x, int x_lo, __half* y, int y_lo, int B, int H, int W, int C, int x_ld, int y_ld,
                          cudaStream_t st) {
  if (C % 8 || x_ld % 8 || y_ld % 8 || x_lo % 8 || y_lo % 8 || H % 2 || W % 2) { set_error("maxpool2_split: bad shape"); return -1; }
  const long long n = static_cast<long long>(B) * (H / 2) * (W / 2) * (C / 8);
  (void)launch_k(maxpool2_split_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, x_lo, y, y_lo, B, H, W, C,
                 x_ld, y_ld);
  return check_cuda(cudaGetLastError(), "maxpool2_split");
}

// ---------------------------------------------------------------- depthwise ConvTranspose2d(k=2f, s=f, p=f/2) + skip add
__global__ void upsample_add_split_kernel(const __half* __restrict__ x, int x_lo, const float* __restrict__ w,
                                          const __half* __restrict__ skip, int skip_lo, __half* __restrict__ y, int y_lo, int B,
                                          int Hi, int Wi, int C, int f, int x_ld, int skip_ld, int y_ld) {
  const int Ho = Hi * f, Wo = Wi * f, CV = C / 8, k = 2 * f, pad = f / 2;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * Ho * Wo * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long pix = i / CV;
  const int ox = static_cast<int>(pix % Wo);
  const long long t = pix / Wo;
  const int oy = static_cast<int>(t % Ho);
  const long long b = t / Ho;
  // all (up to) ten 16-byte loads - skip hi/lo and the four contributing inputs' hi/lo - are issued before anything is
  // consumed: with the loads interleaved with the arithmetic the kernel was latency bound at ~2.5 TB/s
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  uint4 skh = zero4, skl = zero4;
  if (skip != nullptr) {
    skh = __ldg(reinterpret_cast<const uint4*>(skip + pix * skip_ld + cv * 8));
    skl = __ldg(reinterpret_cast<const uint4*>(skip + pix * skip_ld + cv * 8 + skip_lo));
  }
  const int iy_hi = (oy + pad) / f, ix_hi = (ox + pad) / f;
  uint4 xh[2][2], xl[2][2];
  int tap[2][2];
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int iy = iy_hi - dy, ky = oy + pad - iy * f, ix = ix_hi - dx, kx = ox + pad - ix * f;
      const bool ok = iy >= 0 && iy < Hi && ky < k && ix >= 0 && ix < Wi && kx < k;
      tap[dy][dx] = ok ? ky * k + kx : -1;
      const __half* src = x + ((b * Hi + (ok ? iy : 0)) * Wi + (ok ? ix : 0)) * x_ld + cv * 8;
      xh[dy][dx] = ok ? __ldg(reinterpret_cast<const uint4*>(src)) : zero4;
      xl[dy][dx] = ok ? __ldg(reinterpret_cast<const uint4*>(src + x_lo)) : zero4;
    }
  float acc[8], up[8];
  {
    const __half2* hh = reinterpret_cast<const __half2*>(&skh);
    const __half2* ll = reinterpret_cast<const __half2*>(&skl);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 a2 = __half22float2(hh[e]), b2 = __half22float2(ll[e]);
      acc[2 * e] = a2.x + b2.x;
      acc[2 * e + 1] = a2.y + b2.y;
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) up[e] = 0.f;
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      if (tap[dy][dx] < 0) continue;
      float v[8];
      const __half2* hh = reinterpret_cast<const __half2*>(&xh[dy][dx]);
      const __half2* ll = reinterpret_cast<const __half2*>(&xl[dy][dx]);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 a2 = __half22float2(hh[e]), b2 = __half22float2(ll[e]);
        v[2 * e] = a2.x + b2.x;
        v[2 * e + 1] = a2.y + b2.y;
      }
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(w + static_cast<long long>(tap[dy][dx]) * C + cv * 8));
      const float4 w1 = __ldg(reinterpret_cast<const float4*>(w + static_cast<long long>(tap[dy][dx]) * C + cv * 8 + 4));
      up[0] += v[0] * w0.x; up[1] += v[1] * w0.y; up[2] += v[2] * w0.z; up[3] += v[3] * w0.w;
      up[4] += v[4] * w1.x; up[5] += v[5] * w1.y; up[6] += v[6] * w1.z; up[7] += v[7] * w1.w;
    }
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] += up[e];
  st8_split(y + pix * y_ld + cv * 8, y_lo, acc);
}
int launch_upsample_add_split(const __half* x, int x_lo, const float* w, const __half* skip, int skip_lo, __half* y, int y_lo,
                              int B, int Hi, int Wi, int C, int f, int x_ld, int skip_ld, int y_ld, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || y_ld % 8 || (skip && skip_ld % 8) || x_lo % 8 || y_lo % 8 || (skip && skip_lo % 8) || f < 1) {
    set_error("upsample_add_split: bad shape");
    return -1;
  }
  const long long n = static_cast<long long>(B) * Hi * f * Wi * f * (C / 8);
  (void)launch_k(upsample_add_split_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, x_lo, w, skip, skip_lo,
                 y, y_lo, B, Hi, Wi, C, f, x_ld, skip_ld, y_ld);
  return check_cuda(cudaGetLastError(), "upsample_add_split");
}

// ---------------------------------------------------------------- edge fusion gather on hi/lo rows (see edge_gather_kernel)
// outputs ea / eb: [B, K+2, 512] rows = [hi 256 | lo 256]
__global__ void edge_gather_split_kernel(const __half* __restrict__ feat, int feat_ld, int feat_lo, int ch_a, int ch_b,
                                         const long long* __restrict__ edge_idx, __half* __restrict__ ea,
                                         __half* __restrict__ eb, int B, int H, int W, int K, int out_w, int out_h) {
  const int CV = 32;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * (K + 2) * CV * 2) return;
  const int cv = static_cast<int>(i % CV);
  long long t = i / CV;
  const int which = static_cast<int>(t & 1);
  t >>= 1;
  const int pos = static_cast<int>(t % (K + 2));
  const int b = static_cast<int>(t / (K + 2));
  int e = pos - 1;
  e = e < 0 ? 0 : (e > K - 1 ? K - 1 : e);
  const float ex = static_cast<float>(edge_idx[(static_cast<long long>(b) * K + e) * 2 + 0]);
  const float ey = static_cast<float>(edge_idx[(static_cast<long long>(b) * K + e) * 2 + 1]);
  const float gx = ex / static_cast<float>(out_w - 1) * 2.f - 1.f;
  const float gy = ey / static_cast<float>(out_h - 1) * 2.f - 1.f;
  const float ix = ((gx + 1.f) / 2.f) * static_cast<float>(W - 1);
  const float iy = ((gy + 1.f) / 2.f) * static_cast<float>(H - 1);
  const float x0f = floorf(ix), y0f = floorf(iy);
  const int x0 = static_cast<int>(x0f), y0 = static_cast<int>(y0f), x1 = x0 + 1, y1 = y0 + 1;
  const float wx1 = ix - x0f, wy1 = iy - y0f, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
  const int ch = (which ? ch_b : ch_a) + cv * 8;
  float acc[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = 0.f;
  const __half* fb = feat + static_cast<long long>(b) * H * W * feat_ld + ch;
  auto corner = [&](int yy, int xx, float wgt) {
    if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
      float v[8];
      ld8_split(fb + static_cast<long long>(yy * W + xx) * feat_ld, feat_lo, v);
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q] += v[q] * wgt;
    }
  };
  corner(y0, x0, wy0 * wx0);
  corner(y0, x1, wy0 * wx1);
  corner(y1, x0, wy1 * wx0);
  corner(y1, x1, wy1 * wx1);
  st8_split((which ? eb : ea) + (static_cast<long long>(b) * (K + 2) + pos) * 512 + cv * 8, 256, acc);
}
int launch_edge_gather_split(const __half* feat, int feat_ld, int feat_lo, int ch_a, int ch_b, const long long* edge_idx,
                             __half* ea, __half* eb, int B, int H, int W, int K, int out_w, int out_h, cudaStream_t st) {
  const long long n = static_cast<long long>(B) * (K + 2) * 32 * 2;
  (void)launch_k(edge_gather_split_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, feat, feat_ld, feat_lo, ch_a,
                 ch_b, edge_idx, ea, eb, B, H, W, K, out_w, out_h);
  return check_cuda(cudaGetLastError(), "edge_gather_split");
}

// final Conv1d(256 -> n_out, k=1) + indexed add, input rows [hi 256 | lo 256] with row stride t_ld (see edge_head_add_kernel)
__global__ void edge_head_add_split_kernel(const __half* __restrict__ t, int t_ld, int t_lo, const float* __restrict__ w,
                                           const float* __restrict__ bias, int n_out, const long long* __restrict__ edge_idx,
                                           const long long* __restrict__ edge_len, float* __restrict__ out, int out_ctot,
                                           int out_ch0, int B, int K, int H, int W) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B * K) return;
  const int b = warp / K, e = warp - b * K;
  if (e >= edge_len[b]) return;
  float v[8];
  ld8_split(t + static_cast<long long>(warp) * t_ld + lane * 8, t_lo, v);
  const long long ex = edge_idx[(static_cast<long long>(b) * K + e) * 2], ey = edge_idx[(static_cast<long long>(b) * K + e) * 2 + 1];
  for (int o = 0; o < n_out; ++o) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) s += v[q] * __ldg(w + o * 256 + lane * 8 + q);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) out[((static_cast<long long>(b) * out_ctot + out_ch0 + o) * H + ey) * W + ex] += s + bias[o];
  }
}
int launch_edge_head_add_split(const __half* t, int t_ld, int t_lo, const float* w, const float* bias, int n_out,
                               const long long* edge_idx, const long long* edge_len, float* out, int out_ctot, int out_ch0, int B,
                               int K, int H, int W, cudaStream_t st) {
  const long long threads = static_cast<long long>(B) * K * 32;
  (void)launch_k(edge_head_add_split_kernel, dim3(static_cast<unsigned>((threads + 255) / 256)), dim3(256), 0, st, t, t_ld, t_lo, w, bias,
                 n_out, edge_idx, edge_len, out, out_ctot, out_ch0, B, K, H, W);
  return check_cuda(cudaGetLastError(), "edge_head_add_split");
}

// hi/lo rows -> fp32 NCHW (tests / feature-map export): y = float(hi) + float(lo)
__global__ void split_to_nchw_kernel(const __half* __restrict__ x, int x_ld, int x_lo, float* __restrict__ y, int C, int HW) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int pp = p0 + i, c = c0 + threadIdx.x;
    float v = 0.f;
    if (pp < HW && c < C) {
      const __half* r = x + (static_cast<long long>(b) * HW + pp) * x_ld + c;
      v = __half2float(r[0]) + __half2float(r[x_lo]);
    }
    tile[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, pp = p0 + threadIdx.x;
    if (c < C && pp < HW) y[(static_cast<long long>(b) * C + c) * HW + pp] = tile[threadIdx.x][i];
  }
}
int launch_split_to_nchw(const __half* x, int x_ld, int x_lo, float* y, int B, int C, int HW, cudaStream_t st) {
  dim3 grid((HW + 31) / 32, (C + 31) / 32, B), block(32, 8);
  (void)launch_k(split_to_nchw_kernel, dim3(grid), dim3(block), 0, st, x, x_ld, x_lo, y, C, HW);
  return check_cuda(cudaGetLastError(), "split_to_nchw");
}

}  // namespace mf
