// HBM-bound layout / pooling / up-sampling / edge-fusion kernels: coalesced 16-byte vector accesses on NHWC fp16.
#include "mf_common.cuh"
#include "mf_kernels.h"
#include "mf_launch.h"

namespace mf {

MF_DEVINL void unpack8(const uint4& v, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 t = __half22float2(h[e]);
    f[2 * e] = t.x;
    f[2 * e + 1] = t.y;
  }
}
MF_DEVINL uint4 pack8(const float (&f)[8]) {
  __half2 o[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) o[e] = __floats2half2_rn(f[2 * e], f[2 * e + 1]);
  return *reinterpret_cast<uint4*>(o);
}

// ---------------------------------------------------------------- image: NCHW fp32 [B,3,H,W] -> NHWC fp16 [B,H,W,8]
__global__ void pack_image_kernel(const float* __restrict__ x, __half* __restrict__ y, int B, int C, long long HW) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= B * HW) return;
  const long long b = i / HW, pix = i - b * HW;
  float f[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) f[c] = c < C ? __ldg(x + (b * C + c) * HW + pix) : 0.f;
  *reinterpret_cast<uint4*>(y + i * 8) = pack8(f);
}
int launch_pack_image(const float* x, __half* y, int B, int C, int H, int W, cudaStream_t st) {
  if (C > 8) { set_error("pack_image: C=%d > 8", C); return -1; }
  const long long n = static_cast<long long>(B) * H * W;
  (void)launch_k(pack_image_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, y, B, C, static_cast<long long>(H) * W);
  return check_cuda(cudaGetLastError(), "pack_image");
}

// ---------------------------------------------------------------- generic NCHW fp32 <-> NHWC fp16 (tile transpose)
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ x, __half* __restrict__ y, int C, int HW, int y_ld) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, pp = p0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && pp < HW) ? x[(static_cast<long long>(b) * C + c) * HW + pp] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int pp = p0 + i, c = c0 + threadIdx.x;
    if (pp < HW && c < C) y[(static_cast<long long>(b) * HW + pp) * y_ld + c] = __float2half_rn(tile[threadIdx.x][i]);
  }
}
int launch_nchw_to_nhwc(const float* x, __half* y, int B, int C, int HW, int y_ld, cudaStream_t st) {
  dim3 grid((HW + 31) / 32, (C + 31) / 32, B), block(32, 8);
  (void)launch_k(nchw_to_nhwc_kernel, dim3(grid), dim3(block), 0, st, x, y, C, HW, y_ld);
  return check_cuda(cudaGetLastError(), "nchw_to_nhwc");
}
__global__ void nhwc_to_nchw_kernel(const __half* __restrict__ x, float* __restrict__ y, int C, int HW, int x_ld) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int pp = p0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (pp < HW && c < C) ? __half2float(x[(static_cast<long long>(b) * HW + pp) * x_ld + c]) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, pp = p0 + threadIdx.x;
    if (c < C && pp < HW) y[(static_cast<long long>(b) * C + c) * HW + pp] = tile[threadIdx.x][i];
  }
}
int launch_nhwc_to_nchw(const __half* x, float* y, int B, int C, int HW, int x_ld, cudaStream_t st) {
  dim3 grid((HW + 31) / 32, (C + 31) / 32, B), block(32, 8);
  (void)launch_k(nhwc_to_nchw_kernel, dim3(grid), dim3(block), 0, st, x, y, C, HW, x_ld);
  return check_cuda(cudaGetLastError(), "nhwc_to_nchw");
}

// offset [B,18,H,W] + mask [B,9,H,W] (fp32 NCHW, reference _ext layout) -> [B*H*W, 32] fp32 rows
__global__ void pack_offmask_kernel(const float* __restrict__ off, const float* __restrict__ mask, float* __restrict__ y,
                                    int B, int HW) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * HW * 32) return;
  const int ch = static_cast<int>(i & 31);
  const long long m = i >> 5;
  const long long b = m / HW, pix = m - b * HW;
  float v = 0.f;
  if (ch < 18) v = off[(b * 18 + ch) * HW + pix];
  else if (ch < 27) v = mask[(b * 9 + (ch - 18)) * HW + pix];
  y[i] = v;
}
int launch_pack_offmask(const float* off, const float* mask, float* y, int B, int HW, cudaStream_t st) {
  const long long n = static_cast<long long>(B) * HW * 32;
  (void)launch_k(pack_offmask_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, off, mask, y, B, HW);
  return check_cuda(cudaGetLastError(), "pack_offmask");
}

// ---------------------------------------------------------------- MaxPool2d(2) NHWC fp16 (dla_dcn.py:238)
__global__ void maxpool2_kernel(const __half* __restrict__ x, __half* __restrict__ y, int B, int H, int W, int C,
                                int x_ld, int y_ld) {
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
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
  const uint4 bq = __ldg(reinterpret_cast<const uint4*>(p + x_ld));
  const uint4 c = __ldg(reinterpret_cast<const uint4*>(p + static_cast<long long>(W) * x_ld));
  const uint4 d = __ldg(reinterpret_cast<const uint4*>(p + static_cast<long long>(W + 1) * x_ld));
  uint4 o;
  const __half2* ha = reinterpret_cast<const __half2*>(&a);
  const __half2* hb = reinterpret_cast<const __half2*>(&bq);
  const __half2* hc = reinterpret_cast<const __half2*>(&c);
  const __half2* hd = reinterpret_cast<const __half2*>(&d);
  __half2* ho = reinterpret_cast<__half2*>(&o);
#pragma unroll
  for (int e = 0; e < 4; ++e) ho[e] = __hmax2(__hmax2(ha[e], hb[e]), __hmax2(hc[e], hd[e]));
  *reinterpret_cast<uint4*>(y + pix * y_ld + cv * 8) = o;
}
int launch_maxpool2(const __half* x, __half* y, int B, int H, int W, int C, int x_ld, int y_ld, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || y_ld % 8 || H % 2 || W % 2) { set_error("maxpool2: bad shape"); return -1; }
  const long long n = static_cast<long long>(B) * (H / 2) * (W / 2) * (C / 8);
  (void)launch_k(maxpool2_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, y, B, H, W, C, x_ld, y_ld);
  return check_cuda(cudaGetLastError(), "maxpool2");
}

// ---------------------------------------------------------------- depthwise ConvTranspose2d(k=2f, s=f, p=f/2) + skip add
// (IDAUp.forward dla_dcn.py:419-425: layers[i] = up(proj(layers[i])); node(layers[i] + layers[i-1])).
// w: fp32 [k*k, C] (tap-major repack of the [C,1,k,k] parameter). Every output pixel has exactly 2x2 contributing inputs.
__global__ void upsample_add_kernel(const __half* __restrict__ x, const float* __restrict__ w,
                                    const __half* __restrict__ skip, __half* __restrict__ y, int B, int Hi, int Wi,
                                    int C, int f, int x_ld, int skip_ld, int y_ld) {
  const int Ho = Hi * f, Wo = Wi * f, CV = C / 8, k = 2 * f, pad = f / 2;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * Ho * Wo * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long pix = i / CV;
  const int ox = static_cast<int>(pix % Wo);
  const long long t = pix / Wo;
  const int oy = static_cast<int>(t % Ho);
  const long long b = t / Ho;
  // issue the skip load and the (up to) four tap loads together, then do the arithmetic (latency-bound otherwise)
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  const uint4 sk = skip != nullptr ? __ldg(reinterpret_cast<const uint4*>(skip + pix * skip_ld + cv * 8)) : zero4;
  const int iy_hi = (oy + pad) / f, ix_hi = (ox + pad) / f;
  uint4 xin[2][2];
  int tap[2][2];
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int iy = iy_hi - dy, ky = oy + pad - iy * f, ix = ix_hi - dx, kx = ox + pad - ix * f;
      const bool ok = iy >= 0 && iy < Hi && ky < k && ix >= 0 && ix < Wi && kx < k;
      tap[dy][dx] = ok ? ky * k + kx : -1;
      xin[dy][dx] = ok ? __ldg(reinterpret_cast<const uint4*>(x + ((b * Hi + iy) * Wi + ix) * x_ld + cv * 8)) : zero4;
    }
  float acc[8], up[8];
  unpack8(sk, acc);
#pragma unroll
  for (int e = 0; e < 8; ++e) up[e] = 0.f;
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      if (tap[dy][dx] < 0) continue;
      float v[8];
      unpack8(xin[dy][dx], v);
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(w + static_cast<long long>(tap[dy][dx]) * C + cv * 8));
      const float4 w1 = __ldg(reinterpret_cast<const float4*>(w + static_cast<long long>(tap[dy][dx]) * C + cv * 8 + 4));
      up[0] += v[0] * w0.x; up[1] += v[1] * w0.y; up[2] += v[2] * w0.z; up[3] += v[3] * w0.w;
      up[4] += v[4] * w1.x; up[5] += v[5] * w1.y; up[6] += v[6] * w1.z; up[7] += v[7] * w1.w;
    }
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] += up[e];
  *reinterpret_cast<uint4*>(y + pix * y_ld + cv * 8) = pack8(acc);
}
// f == 2 (k = 4, pad 1) specialisation: one thread produces the 2x2 output block {2a+1, 2a+2} x {2b+1, 2b+2}, which depends
// on exactly the four inputs (a..a+1, b..b+1): each input vector is loaded once instead of four times and every one of
// the 16 kernel taps is used exactly once.
__global__ void __launch_bounds__(256, 3)
upsample2_add_kernel(const __half* __restrict__ x, const float* __restrict__ w, const __half* __restrict__ skip,
                     __half* __restrict__ y, int B, int Hi, int Wi, int C, int x_ld, int skip_ld, int y_ld) {
  const int CV = C / 8, Ho = 2 * Hi, Wo = 2 * Wi;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * (Hi + 1) * (Wi + 1) * CV) return;
  const int cv = static_cast<int>(i % CV);
  long long t = i / CV;
  const int bb = static_cast<int>(t % (Wi + 1)) - 1;
  t /= (Wi + 1);
  const int a = static_cast<int>(t % (Hi + 1)) - 1;
  const long long b = t / (Hi + 1);
  // all 8 global loads (4 inputs, 4 skip vectors) are issued before anything is consumed: the kernel is latency bound
  // otherwise (measured 2 TB/s with the loads interleaved with the arithmetic at 2-3 resident blocks per SM)
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  uint4 xin[2][2], sk[2][2];
  long long opix[2][2];
#pragma unroll
  for (int iy = 0; iy < 2; ++iy)
#pragma unroll
    for (int ix = 0; ix < 2; ++ix) {
      const int yy = a + iy, xx = bb + ix;
      xin[iy][ix] = (yy >= 0 && yy < Hi && xx >= 0 && xx < Wi)
                        ? __ldg(reinterpret_cast<const uint4*>(x + ((b * Hi + yy) * Wi + xx) * x_ld + cv * 8)) : zero4;
      const int oy = 2 * a + 1 + iy, ox = 2 * bb + 1 + ix;             // (iy, ix) doubles as the output offset (dy, dx)
      const bool ok = oy >= 0 && oy < Ho && ox >= 0 && ox < Wo;
      opix[iy][ix] = ok ? (b * Ho + oy) * Wo + ox : -1;
      sk[iy][ix] = (ok && skip != nullptr) ? __ldg(reinterpret_cast<const uint4*>(skip + opix[iy][ix] * skip_ld + cv * 8)) : zero4;
    }
  float in[2][2][8];
#pragma unroll
  for (int iy = 0; iy < 2; ++iy)
#pragma unroll
    for (int ix = 0; ix < 2; ++ix) unpack8(xin[iy][ix], in[iy][ix]);
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      if (opix[dy][dx] < 0) continue;
      float acc[8], up[8];
      unpack8(sk[dy][dx], acc);
#pragma unroll
      for (int e = 0; e < 8; ++e) up[e] = 0.f;
      // same accumulation order as the generic kernel: input rows a+1 then a, columns b+1 then b
#pragma unroll
      for (int iy = 1; iy >= 0; --iy)
#pragma unroll
        for (int ix = 1; ix >= 0; --ix) {
          const int ky = dy + 2 * (1 - iy), kx = dx + 2 * (1 - ix);
          const float4 w0 = __ldg(reinterpret_cast<const float4*>(w + static_cast<long long>(ky * 4 + kx) * C + cv * 8));
          const float4 w1 = __ldg(reinterpret_cast<const float4*>(w + static_cast<long long>(ky * 4 + kx) * C + cv * 8 + 4));
          const float* v = in[iy][ix];
          up[0] += v[0] * w0.x; up[1] += v[1] * w0.y; up[2] += v[2] * w0.z; up[3] += v[3] * w0.w;
          up[4] += v[4] * w1.x; up[5] += v[5] * w1.y; up[6] += v[6] * w1.z; up[7] += v[7] * w1.w;
        }
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] += up[e];
      *reinterpret_cast<uint4*>(y + opix[dy][dx] * y_ld + cv * 8) = pack8(acc);
    }
  }
}
int launch_upsample_add(const __half* x, const float* w, const __half* skip, __half* y, int B, int Hi, int Wi, int C,
                        int f, int x_ld, int skip_ld, int y_ld, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || y_ld % 8 || (skip && skip_ld % 8) || f < 1) { set_error("upsample_add: bad shape"); return -1; }
  if (f == 2) {
    const long long n2 = static_cast<long long>(B) * (Hi + 1) * (Wi + 1) * (C / 8);
    (void)launch_k(upsample2_add_kernel, dim3(static_cast<unsigned>((n2 + 255) / 256)), dim3(256), 0, st, x, w, skip, y, B, Hi, Wi, C, x_ld, skip_ld,
                                                                                 y_ld);
    return check_cuda(cudaGetLastError(), "upsample2_add");
  }
  const long long n = static_cast<long long>(B) * Hi * f * Wi * f * (C / 8);
  (void)launch_k(upsample_add_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, w, skip, y, B, Hi, Wi, C, f, x_ld,
                                                                               skip_ld, y_ld);
  return check_cuda(cudaGetLastError(), "upsample_add");
}

// ---------------------------------------------------------------- edge fusion gather (detector_predictor.py:137-147)
// F.grid_sample(bilinear, zeros padding, align_corners=True) of two 256-channel slices of the head feature map at the
// border pixels, written as two replicate-padded Conv1d inputs [B, K+2, 256] (padding_mode='replicate', k=3).
__global__ void edge_gather_kernel(const __half* __restrict__ feat, int feat_ld, int ch_a, int ch_b,
                                   const long long* __restrict__ edge_idx, __half* __restrict__ ea,
                                   __half* __restrict__ eb, int B, int H, int W, int K, int out_w, int out_h) {
  const int CV = 32;  // 256 channels / 8
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
      unpack8(__ldg(reinterpret_cast<const uint4*>(fb + static_cast<long long>(yy * W + xx) * feat_ld)), v);
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q] += v[q] * wgt;
    }
  };
  corner(y0, x0, wy0 * wx0);
  corner(y0, x1, wy0 * wx1);
  corner(y1, x0, wy1 * wx0);
  corner(y1, x1, wy1 * wx1);
  __half* dst = (which ? eb : ea) + (static_cast<long long>(b) * (K + 2) + pos) * 256 + cv * 8;
  *reinterpret_cast<uint4*>(dst) = pack8(acc);
}
int launch_edge_gather(const __half* feat, int feat_ld, int ch_a, int ch_b, const long long* edge_idx, __half* ea,
                       __half* eb, int B, int H, int W, int K, int out_w, int out_h, cudaStream_t st) {
  const long long n = static_cast<long long>(B) * (K + 2) * 32 * 2;
  (void)launch_k(edge_gather_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, feat, feat_ld, ch_a, ch_b, edge_idx, ea, eb,
                                                                              B, H, W, K, out_w, out_h);
  return check_cuda(cudaGetLastError(), "edge_gather");
}

// byte mask [B*H*W] of the pixels edge_gather_kernel reads (the up-to-4 bilinear corners of every border position, computed
// with the same fp32 round trip), so that the fused head stores hidden activations for those pixels only.
__global__ void edge_mask_kernel(const long long* __restrict__ edge_idx, unsigned char* __restrict__ mask, int B, int H,
                                 int W, int K, int out_w, int out_h) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * K) return;
  const int b = i / K;
  const float ex = static_cast<float>(edge_idx[static_cast<long long>(i) * 2 + 0]);
  const float ey = static_cast<float>(edge_idx[static_cast<long long>(i) * 2 + 1]);
  const float gx = ex / static_cast<float>(out_w - 1) * 2.f - 1.f;
  const float gy = ey / static_cast<float>(out_h - 1) * 2.f - 1.f;
  const float ix = ((gx + 1.f) / 2.f) * static_cast<float>(W - 1);
  const float iy = ((gy + 1.f) / 2.f) * static_cast<float>(H - 1);
  const int x0 = static_cast<int>(floorf(ix)), y0 = static_cast<int>(floorf(iy));
  unsigned char* mb = mask + static_cast<long long>(b) * H * W;
  for (int dy = 0; dy < 2; ++dy)
    for (int dx = 0; dx < 2; ++dx) {
      const int yy = y0 + dy, xx = x0 + dx;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) mb[yy * W + xx] = 1;
    }
}
int launch_edge_mask(const long long* edge_idx, unsigned char* mask, int B, int K, int H, int W, int out_w, int out_h,
                     cudaStream_t st) {
  if (check_cuda(cudaMemsetAsync(mask, 0, static_cast<size_t>(B) * H * W, st), "edge_mask memset")) return -1;
  (void)launch_k(edge_mask_kernel, dim3((B * K + 255) / 256), dim3(256), 0, st, edge_idx, mask, B, H, W, K, out_w, out_h);
  return check_cuda(cudaGetLastError(), "edge_mask");
}

// final Conv1d(256 -> n_out, k=1) of one truncation branch + indexed add into an NCHW fp32 map
// (detector_predictor.py:155-158). One warp per (b, e); lanes split the 256 input channels.
__global__ void edge_head_add_kernel(const __half* __restrict__ t, const float* __restrict__ w,
                                     const float* __restrict__ bias, int n_out, const long long* __restrict__ edge_idx,
                                     const long long* __restrict__ edge_len, float* __restrict__ out, int out_ctot,
                                     int out_ch0, int B, int K, int H, int W) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B * K) return;
  const int b = warp / K, e = warp - b * K;
  if (e >= edge_len[b]) return;
  float v[8];
  unpack8(__ldg(reinterpret_cast<const uint4*>(t + static_cast<long long>(warp) * 256 + lane * 8)), v);
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
int launch_edge_head_add(const __half* t, const float* w, const float* bias, int n_out, const long long* edge_idx,
                         const long long* edge_len, float* out, int out_ctot, int out_ch0, int B, int K, int H, int W,
                         cudaStream_t st) {
  const long long threads = static_cast<long long>(B) * K * 32;
  (void)launch_k(edge_head_add_kernel, dim3(static_cast<unsigned>((threads + 255) / 256)), dim3(256), 0, st, t, w, bias, n_out, edge_idx, edge_len,
                                                                                     out, out_ctot, out_ch0, B, K, H, W);
  return check_cuda(cudaGetLastError(), "edge_head_add");
}

// sigmoid_hm (model/layers/utils.py:39-43): x = clamp(sigmoid(x), 1e-4, 1-1e-4), in place
__global__ void sigmoid_clamp_kernel(float* __restrict__ x, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = 1.f / (1.f + expf(-x[i]));
  x[i] = fminf(fmaxf(s, 1e-4f), 1.f - 1e-4f);
}
int launch_sigmoid_clamp(float* x, long long n, cudaStream_t st) {
  (void)launch_k(sigmoid_clamp_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, n);
  return check_cuda(cudaGetLastError(), "sigmoid_clamp");
}

// ---------------------------------------------------------------- penalty-reduced focal loss (layers/focal_loss.py:35-55)
// out[0] += -(sum_pos log(p)(1-p)^2 + sum_neg log(1-p) p^2 (1-t)^4), out[1] += #(t==1).  (alpha=2, beta=4)
__global__ void focal_loss_kernel(const float* __restrict__ pred, const float* __restrict__ tgt, long long n,
                                  float* __restrict__ out) {
  float loss = 0.f, npos = 0.f;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float p = __ldg(pred + i), t = __ldg(tgt + i);
    if (t == 1.f) {
      loss -= logf(p) * (1.f - p) * (1.f - p);
      npos += 1.f;
    } else if (t < 1.f && t >= 0.f) {
      const float omt = 1.f - t, omt2 = omt * omt;
      loss -= logf(1.f - p) * p * p * omt2 * omt2;
    }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    loss += __shfl_xor_sync(0xffffffffu, loss, d);
    npos += __shfl_xor_sync(0xffffffffu, npos, d);
  }
  __shared__ float sl[32], sn[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sl[warp] = loss; sn[warp] = npos; }
  __syncthreads();
  if (warp == 0) {
    loss = lane < (blockDim.x >> 5) ? sl[lane] : 0.f;
    npos = lane < (blockDim.x >> 5) ? sn[lane] : 0.f;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      loss += __shfl_xor_sync(0xffffffffu, loss, d);
      npos += __shfl_xor_sync(0xffffffffu, npos, d);
    }
    if (lane == 0) { atomicAdd(out, loss); atomicAdd(out + 1, npos); }
  }
}
int launch_focal_loss(const float* pred, const float* tgt, long long n, float* out2, cudaStream_t st) {
  if (check_cuda(cudaMemsetAsync(out2, 0, 2 * sizeof(float), st), "focal memset")) return -1;
  long long blocks = (n + 1023) / 1024;
  if (blocks > 148 * 8) blocks = 148 * 8;
  (void)launch_k(focal_loss_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, st, pred, tgt, n, out2);
  return check_cuda(cudaGetLastError(), "focal_loss");
}

}  // namespace mf
