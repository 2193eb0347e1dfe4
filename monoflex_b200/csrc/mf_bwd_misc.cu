// Backward of the HBM-bound layers (training path; forward twins in mf_elementwise.cu). All on NHWC fp16 rows with 16-byte
// vector accesses unless noted.
//   maxpool2_bwd        MaxPool2d(2) (dla_dcn.py:238): every input pixel belongs to exactly one window, the gradient goes to
//                       the first maximum in window scan order (torch's arg-max convention); dx is written completely.
//   upsample_bwd_dx     depth-wise ConvTranspose2d(k = 2f, s = f, p = f/2) (dla_dcn.py:408-412): dx = strided depth-wise
//                       correlation of dy with the k x k taps. (The skip input's gradient is dy itself.)
//   upsample_bwd_dw     dw[tap, c] = sum over input pixels of x * dy(shifted): per-CTA partials + fixed-order reduction.
//   sigmoid_clamp_bwd   sigmoid_hm (layers/utils.py:39-43): dx = dy * y (1 - y) where the clamp did not bind (fp32 NCHW).
//   column_sum          sum over rows of an [M, C] fp16 matrix (conv-bias gradients), deterministic two-level reduction.
//   edge_gather_bwd     transpose of edge_gather_kernel (detector_predictor.py:137-147): bilinear corner weights scatter the
//                       gradient of the two replicate-padded Conv1d inputs back onto the hidden feature rows (half2 atomics:
//                       border positions repeat).
//   interleave2x2       dX[b, 2i+py, 2j+px] = part[py][px][b, i, j]: recombines the four parity sub-convolutions of a
//                       stride-2 convolution's data gradient (monoflex_b200/backward.py::conv2d_dgrad_stride2).
#include "mf_common.cuh"
#include "mf_launch.h"

namespace mf {

MF_DEVINL void bm_unpack8(const uint4& v, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 t = __half22float2(h[e]);
    f[2 * e] = t.x; f[2 * e + 1] = t.y;
  }
}
MF_DEVINL uint4 bm_pack8(const float (&f)[8]) {
  __half2 o[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) o[e] = __floats2half2_rn(f[2 * e], f[2 * e + 1]);
  return *reinterpret_cast<uint4*>(o);
}

// ---------------------------------------------------------------- MaxPool2d(2) backward
__global__ void __launch_bounds__(256) maxpool2_bwd_kernel(const __half* __restrict__ x, const __half* __restrict__ dy,
                                                           __half* __restrict__ dx, int B, int H, int W, int C, int x_ld,
                                                           int dy_ld, int dx_ld) {
  const int Ho = H / 2, Wo = W / 2, CV = C / 8;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * Ho * Wo * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long pix = i / CV;
  const int ox = static_cast<int>(pix % Wo);
  const long long t = pix / Wo;
  const int oy = static_cast<int>(t % Ho);
  const long long b = t / Ho;
  const long long r00 = (b * H + 2 * oy) * W + 2 * ox;
  const long long rows[4] = {r00, r00 + 1, r00 + W, r00 + W + 1};           // window scan order
  float v[4][8], g[8], o[4][8];
#pragma unroll
  for (int q = 0; q < 4; ++q) bm_unpack8(__ldg(reinterpret_cast<const uint4*>(x + rows[q] * x_ld + cv * 8)), v[q]);
  bm_unpack8(__ldg(reinterpret_cast<const uint4*>(dy + pix * dy_ld + cv * 8)), g);
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    int arg = 0;
    float m = v[0][e];
#pragma unroll
    for (int q = 1; q < 4; ++q)
      if (v[q][e] > m) { m = v[q][e]; arg = q; }                              // strict: the first maximum keeps the gradient
#pragma unroll
    for (int q = 0; q < 4; ++q) o[q][e] = q == arg ? g[e] : 0.f;
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(dx + rows[q] * dx_ld + cv * 8) = bm_pack8(o[q]);
}
int launch_maxpool2_bwd(const __half* x, const __half* dy, __half* dx, int B, int H, int W, int C, int x_ld, int dy_ld,
                        int dx_ld, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || dy_ld % 8 || dx_ld % 8 || H % 2 || W % 2) { set_error("maxpool2_bwd: bad shape"); return -1; }
  const long long n = static_cast<long long>(B) * (H / 2) * (W / 2) * (C / 8);
  (void)launch_k(maxpool2_bwd_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, dy, dx, B, H, W, C, x_ld,
                 dy_ld, dx_ld);
  return check_cuda(cudaGetLastError(), "maxpool2_bwd");
}

// ---------------------------------------------------------------- depth-wise ConvTranspose2d backward: data
// forward: y[oy, ox] += x[iy, ix] * w[ky, kx] with ky = oy + pad - iy * f (0 <= ky < k), same for x
__global__ void __launch_bounds__(256) upsample_bwd_dx_kernel(const __half* __restrict__ dy, const float* __restrict__ w,
                                                              __half* __restrict__ dx, int B, int Hi, int Wi, int C, int f,
                                                              int dy_ld, int dx_ld) {
  const int CV = C / 8, k = 2 * f, pad = f / 2, Ho = Hi * f, Wo = Wi * f;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * Hi * Wi * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long pix = i / CV;
  const int ix = static_cast<int>(pix % Wi);
  const long long t = pix / Wi;
  const int iy = static_cast<int>(t % Hi);
  const long long b = t / Hi;
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
  for (int ky = 0; ky < k; ++ky) {
    const int oy = iy * f - pad + ky;
    if (oy < 0 || oy >= Ho) continue;
    for (int kx = 0; kx < k; ++kx) {
      const int ox = ix * f - pad + kx;
      if (ox < 0 || ox >= Wo) continue;
      float g[8];
      bm_unpack8(__ldg(reinterpret_cast<const uint4*>(dy + ((b * Ho + oy) * Wo + ox) * dy_ld + cv * 8)), g);
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(w + static_cast<long long>(ky * k + kx) * C + cv * 8));
      const float4 w1 = __ldg(reinterpret_cast<const float4*>(w + static_cast<long long>(ky * k + kx) * C + cv * 8 + 4));
      acc[0] += g[0] * w0.x; acc[1] += g[1] * w0.y; acc[2] += g[2] * w0.z; acc[3] += g[3] * w0.w;
      acc[4] += g[4] * w1.x; acc[5] += g[5] * w1.y; acc[6] += g[6] * w1.z; acc[7] += g[7] * w1.w;
    }
  }
  *reinterpret_cast<uint4*>(dx + pix * dx_ld + cv * 8) = bm_pack8(acc);
}
// weights: part[slab][tap][c] = sum over the slab's input pixels of x[pixel, c] * dy[shifted pixel, c].
// A warp owns one 8-channel group and 8 taps: its 32 lanes walk the slab's pixels (x loaded ONCE per pixel for the 8 taps, the
// 8 shifted dY loads issued together), accumulate in registers and are reduced by shuffles in a fixed order (deterministic).
// (Round-2 form: one thread per (tap, 8 channels) walking the slab serially - two dependent loads per iteration, x re-read per
// tap: 1.5 ms per training step for the 8 up-sampling layers.)
static constexpr int UPW_TAPS = 8;
__global__ void __launch_bounds__(256) upsample_bwd_dw_kernel(const __half* __restrict__ x, const __half* __restrict__ dy,
                                                              float* __restrict__ part, int B, int Hi, int Wi, int C, int f,
                                                              int x_ld, int dy_ld, long long pix_per_slab) {
  const int CV = C / 8, k = 2 * f, pad = f / 2, Ho = Hi * f, Wo = Wi * f, taps = k * k;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cv = blockIdx.x * 8 + warp;
  const int tap0 = blockIdx.z * UPW_TAPS;
  if (cv >= CV) return;
  const long long npix = static_cast<long long>(B) * Hi * Wi;
  const long long p0 = static_cast<long long>(blockIdx.y) * pix_per_slab;
  const long long p1 = p0 + pix_per_slab < npix ? p0 + pix_per_slab : npix;
  int kys[UPW_TAPS], kxs[UPW_TAPS];
#pragma unroll
  for (int t = 0; t < UPW_TAPS; ++t) {
    const int tap = tap0 + t;
    kys[t] = tap < taps ? tap / k : -100000;           // out-of-range tap: every pixel fails the bounds test below
    kxs[t] = tap < taps ? tap - (tap / k) * k : 0;
  }
  float acc[UPW_TAPS][8];
#pragma unroll
  for (int t = 0; t < UPW_TAPS; ++t)
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[t][e] = 0.f;
  for (long long pix = p0 + lane; pix < p1; pix += 32) {
    const int ix = static_cast<int>(pix % Wi);
    const long long tt = pix / Wi;
    const int iy = static_cast<int>(tt % Hi);
    const long long b = tt / Hi;
    const uint4 xr = __ldg(reinterpret_cast<const uint4*>(x + pix * x_ld + cv * 8));
    uint4 gr[UPW_TAPS];
#pragma unroll
    for (int t = 0; t < UPW_TAPS; ++t) {
      const int oy = iy * f - pad + kys[t], ox = ix * f - pad + kxs[t];
      const bool ok = oy >= 0 && oy < Ho && ox >= 0 && ox < Wo;
      gr[t] = ok ? __ldg(reinterpret_cast<const uint4*>(dy + ((b * Ho + oy) * Wo + ox) * dy_ld + cv * 8)) : make_uint4(0u, 0u, 0u, 0u);
    }
    float xv[8];
    bm_unpack8(xr, xv);
#pragma unroll
    for (int t = 0; t < UPW_TAPS; ++t) {
      float g[8];
      bm_unpack8(gr[t], g);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[t][e] += xv[e] * g[e];
    }
  }
#pragma unroll
  for (int t = 0; t < UPW_TAPS; ++t)
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float v = acc[t][e];
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
      acc[t][e] = v;
    }
  if (lane == 0) {
#pragma unroll
    for (int t = 0; t < UPW_TAPS; ++t) {
      if (tap0 + t < taps) {
        float* dst = part + (static_cast<long long>(blockIdx.y) * taps + tap0 + t) * C + cv * 8;
#pragma unroll
        for (int e = 0; e < 8; ++e) dst[e] = acc[t][e];
      }
    }
  }
}
__global__ void slab_reduce_kernel(const float* __restrict__ part, float* __restrict__ out, long long n, int nslab) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s = 0.0;
  for (int k = 0; k < nslab; ++k) s += part[static_cast<long long>(k) * n + i];      // fixed order
  out[i] = static_cast<float>(s);
}
static int upsample_slabs(long long npix, long long& per) {
  long long ns = (npix + 255) / 256;
  if (ns > 512) ns = 512;
  if (ns < 1) ns = 1;
  per = (npix + ns - 1) / ns;
  return static_cast<int>((npix + per - 1) / per);
}
size_t upsample_bwd_workspace_floats(int B, int Hi, int Wi, int C, int f) {
  long long per;
  const int ns = upsample_slabs(static_cast<long long>(B) * Hi * Wi, per);
  return static_cast<size_t>(ns) * 4 * f * f * C;
}
// w / dw: fp32 [k*k, C] tap-major (the layout mf_upsample_add_nhwc_f16 takes)
int launch_upsample_bwd(const __half* x, const float* w, const __half* dy, __half* dx, float* dw, int B, int Hi, int Wi, int C,
                        int f, int x_ld, int dy_ld, int dx_ld, float* workspace, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || dy_ld % 8 || dx_ld % 8 || f < 1 || f > 8) { set_error("upsample_bwd: bad shape"); return -1; }
  const long long npix = static_cast<long long>(B) * Hi * Wi;
  if (dx != nullptr) {
    const long long n = npix * (C / 8);
    (void)launch_k(upsample_bwd_dx_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, dy, w, dx, B, Hi, Wi, C,
                   f, dy_ld, dx_ld);
  }
  if (dw != nullptr) {
    long long per;
    const int ns = upsample_slabs(npix, per);
    const int taps = 4 * f * f, CV = C / 8;
    (void)launch_k(upsample_bwd_dw_kernel, dim3((CV + 7) / 8, ns, (taps + UPW_TAPS - 1) / UPW_TAPS), dim3(256), 0, st, x, dy,
                   workspace, B, Hi, Wi, C, f, x_ld, dy_ld, per);
    const long long n = static_cast<long long>(taps) * C;
    slab_reduce_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(workspace, dw, n, ns);
  }
  return check_cuda(cudaGetLastError(), "upsample_bwd");
}

// ---------------------------------------------------------------- sigmoid_hm backward (fp32, any layout)
__global__ void sigmoid_clamp_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dy, float* __restrict__ dx,
                                         long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = y[i];
  dx[i] = (s > 1e-4f && s < 1.f - 1e-4f) ? dy[i] * s * (1.f - s) : 0.f;      // where the clamp bound, the gradient is cut
}
int launch_sigmoid_clamp_bwd(const float* y, const float* dy, float* dx, long long n, cudaStream_t st) {
  (void)launch_k(sigmoid_clamp_bwd_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, y, dy, dx, n);
  return check_cuda(cudaGetLastError(), "sigmoid_clamp_bwd");
}

// ---------------------------------------------------------------- column sum of an [M, C] fp16 matrix
__global__ void __launch_bounds__(256) column_sum_partial_kernel(const __half* __restrict__ x, int x_ld, long long M, int C,
                                                                 long long rows_per_cta, float* __restrict__ part) {
  const int CV = C / 8;
  const int cv = threadIdx.x % CV, r = threadIdx.x / CV, RL = blockDim.x / CV;
  extern __shared__ float sm[];                                            // [RL][C]
  float a[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) a[e] = 0.f;
  const long long r0 = static_cast<long long>(blockIdx.x) * rows_per_cta;
  const long long r1 = r0 + rows_per_cta < M ? r0 + rows_per_cta : M;
  if (r < RL) {
    for (long long row = r0 + r; row < r1; row += RL) {
      float v[8];
      bm_unpack8(__ldg(reinterpret_cast<const uint4*>(x + row * x_ld + cv * 8)), v);
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] += v[e];
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) sm[r * C + cv * 8 + e] = a[e];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < RL; ++q) s += sm[q * C + i];
    part[static_cast<long long>(blockIdx.x) * C + i] = s;
  }
}
static int colsum_grid(long long M, long long& rpc) {
  long long n = (M + 63) / 64;                              // up to 8 CTAs per SM (see bn_grid in mf_bn_train.cu)
  if (n > 148 * 8) n = 148 * 8;
  if (n < 1) n = 1;
  rpc = (M + n - 1) / n;
  return static_cast<int>((M + rpc - 1) / rpc);
}
size_t column_sum_workspace_floats(long long M, int C) {
  long long rpc;
  return static_cast<size_t>(colsum_grid(M, rpc)) * C;
}
int launch_column_sum(const __half* x, int x_ld, long long M, int C, float* out, float* workspace, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || C > 2048 || M < 1) { set_error("column_sum: bad shape"); return -1; }
  long long rpc;
  const int ncta = colsum_grid(M, rpc);
  const int RL = 256 / (C / 8);
  if (RL < 1) { set_error("column_sum: C too wide"); return -1; }
  (void)launch_k(column_sum_partial_kernel, dim3(ncta), dim3(256), static_cast<size_t>(RL) * C * sizeof(float), st, x, x_ld, M, C,
                 rpc, workspace);
  slab_reduce_kernel<<<(C + 255) / 256, 256, 0, st>>>(workspace, out, C, ncta);
  return check_cuda(cudaGetLastError(), "column_sum");
}

// ---------------------------------------------------------------- edge-fusion gather backward
// d_ea / d_eb: [B, K+2, 256] fp16 gradients of the two replicate-padded Conv1d inputs; d_feat: [B*H*W, feat_ld] fp16, ADDED to
__global__ void edge_gather_bwd_kernel(const __half* __restrict__ d_ea, const __half* __restrict__ d_eb, int ch_a, int ch_b,
                                       const long long* __restrict__ edge_idx, __half* __restrict__ d_feat, int feat_ld, int B,
                                       int H, int W, int K, int out_w, int out_h) {
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
  const int x0 = static_cast<int>(x0f), y0 = static_cast<int>(y0f);
  const float wx1 = ix - x0f, wy1 = iy - y0f, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
  float g[8];
  bm_unpack8(__ldg(reinterpret_cast<const uint4*>((which ? d_eb : d_ea) + (static_cast<long long>(b) * (K + 2) + pos) * 256 + cv * 8)), g);
  __half* fb = d_feat + static_cast<long long>(b) * H * W * feat_ld + (which ? ch_b : ch_a) + cv * 8;
  const float wts[4] = {wy0 * wx0, wy0 * wx1, wy1 * wx0, wy1 * wx1};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int yy = y0 + (q >> 1), xx = x0 + (q & 1);
    if (yy < 0 || yy >= H || xx < 0 || xx >= W || wts[q] == 0.f) continue;
    __half2* dst = reinterpret_cast<__half2*>(fb + static_cast<long long>(yy * W + xx) * feat_ld);
#pragma unroll
    for (int h = 0; h < 4; ++h) atomicAdd(dst + h, __floats2half2_rn(g[2 * h] * wts[q], g[2 * h + 1] * wts[q]));
  }
}
int launch_edge_gather_bwd(const __half* d_ea, const __half* d_eb, int ch_a, int ch_b, const long long* edge_idx, __half* d_feat,
                           int feat_ld, int B, int H, int W, int K, int out_w, int out_h, cudaStream_t st) {
  const long long n = static_cast<long long>(B) * (K + 2) * 32 * 2;
  (void)launch_k(edge_gather_bwd_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, d_ea, d_eb, ch_a, ch_b,
                 edge_idx, d_feat, feat_ld, B, H, W, K, out_w, out_h);
  return check_cuda(cudaGetLastError(), "edge_gather_bwd");
}

// ---------------------------------------------------------------- edge_head_add backward (detector_predictor.py:155-158)
// forward: out[b, ch0 + o, ey, ex] += bias[o] + sum_c t[b, e, c] * w[o, c] for the first edge_len[b] border positions e.
// backward: d_t[b, e, c] = sum_o g[o] w[o, c] (0 past edge_len), dw[o, c] += g[o] t[b, e, c], dbias[o] += g[o], with
// g[o] = d_out[b, ch0 + o, ey, ex]. One warp per (b, e); dw / dbias by fp32 atomics (zeroed by the launcher).
template <int NO>
__global__ void __launch_bounds__(256) edge_head_add_bwd_kernel(const __half* __restrict__ t, const float* __restrict__ w, int n_out,
                                         const long long* __restrict__ edge_idx, const long long* __restrict__ edge_len,
                                         const float* __restrict__ d_out, int out_ctot, int out_ch0, __half* __restrict__ d_t,
                                         float* __restrict__ dw, float* __restrict__ dbias, int B, int K, int H, int W) {
  // 8 warps per CTA, each walking EDGE_PER_WARP consecutive (b, e) positions: the weight / bias gradients are summed in
  // registers, then across the CTA's warps in shared memory, and only one atomic per (o, c) per CTA reaches `dw` (the
  // first version issued one per position: ~6.6 k warps hammering the same 768 addresses, 0.9 ms per launch).
  constexpr int EDGE_PER_WARP = 8;
  __shared__ float red[8][NO][256 + 1];
  __shared__ float redb[8][NO];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float dwa[NO][8], dba[NO];
#pragma unroll
  for (int o = 0; o < NO; ++o) {
    dba[o] = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) dwa[o][q] = 0.f;
  }
  const int first = (blockIdx.x * 8 + wib) * EDGE_PER_WARP;
  for (int i = 0; i < EDGE_PER_WARP; ++i) {
    const int pos = first + i;
    if (pos >= B * K) break;
    const int b = pos / K, e = pos - b * K;
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.f;
    if (e < edge_len[b]) {
      float tv[8];
      bm_unpack8(__ldg(reinterpret_cast<const uint4*>(t + static_cast<long long>(pos) * 256 + lane * 8)), tv);
      const long long ex = edge_idx[(static_cast<long long>(b) * K + e) * 2], ey = edge_idx[(static_cast<long long>(b) * K + e) * 2 + 1];
#pragma unroll
      for (int o = 0; o < NO; ++o) {
        if (o < n_out) {
          const float g = __ldg(d_out + ((static_cast<long long>(b) * out_ctot + out_ch0 + o) * H + ey) * W + ex);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            acc[q] += g * __ldg(w + o * 256 + lane * 8 + q);
            dwa[o][q] += g * tv[q];
          }
          dba[o] += g;
        }
      }
    }
    *reinterpret_cast<uint4*>(d_t + static_cast<long long>(pos) * 256 + lane * 8) = bm_pack8(acc);
  }
#pragma unroll
  for (int o = 0; o < NO; ++o) {
#pragma unroll
    for (int q = 0; q < 8; ++q) red[wib][o][lane * 8 + q] = dwa[o][q];
    if (lane == 0) redb[wib][o] = dba[o];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n_out * 256; i += blockDim.x) {
    const int o = i >> 8, c = i & 255;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][o][c];
    if (s != 0.f) atomicAdd(dw + o * 256 + c, s);
  }
  if (threadIdx.x < n_out) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += redb[k][threadIdx.x];
    if (s != 0.f) atomicAdd(dbias + threadIdx.x, s);
  }
}
int launch_edge_head_add_bwd(const __half* t, const float* w, int n_out, const long long* edge_idx, const long long* edge_len,
                             const float* d_out, int out_ctot, int out_ch0, __half* d_t, float* dw, float* dbias, int B, int K,
                             int H, int W, cudaStream_t st) {
  if (check_cuda(cudaMemsetAsync(dw, 0, sizeof(float) * n_out * 256, st), "edge_head_add_bwd memset")) return -1;
  if (check_cuda(cudaMemsetAsync(dbias, 0, sizeof(float) * n_out, st), "edge_head_add_bwd memset")) return -1;
  if (n_out < 1 || n_out > 4) { set_error("edge_head_add_bwd: n_out %d (1..4 supported)", n_out); return -1; }
  const int blocks = (B * K + 63) / 64;                          // 8 warps x 8 positions per CTA
  (void)launch_k(edge_head_add_bwd_kernel<4>, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, st, t, w, n_out,
                 edge_idx, edge_len, d_out, out_ctot, out_ch0, d_t, dw, dbias, B, K, H, W);
  return check_cuda(cudaGetLastError(), "edge_head_add_bwd");
}

// ---------------------------------------------------------------- dst[r, 0:C] += src[r, 0:C] (gradient accumulation)
__global__ void __launch_bounds__(256) add_rows_kernel(__half* __restrict__ dst, int dst_ld, const __half* __restrict__ src,
                                                       int src_ld, long long M, int C) {
  const int CV = C / 8;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= M * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long row = i / CV;
  float a[8], b[8];
  bm_unpack8(*reinterpret_cast<const uint4*>(dst + row * dst_ld + cv * 8), a);
  bm_unpack8(__ldg(reinterpret_cast<const uint4*>(src + row * src_ld + cv * 8)), b);
#pragma unroll
  for (int e = 0; e < 8; ++e) a[e] += b[e];
  *reinterpret_cast<uint4*>(dst + row * dst_ld + cv * 8) = bm_pack8(a);
}
int launch_add_rows(__half* dst, int dst_ld, const __half* src, int src_ld, long long M, int C, cudaStream_t st) {
  if (C % 8 || dst_ld % 8 || src_ld % 8) { set_error("add_rows: bad shape"); return -1; }
  const long long n = M * (C / 8);
  (void)launch_k(add_rows_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, dst, dst_ld, src, src_ld, M, C);
  return check_cuda(cudaGetLastError(), "add_rows");
}

// ---------------------------------------------------------------- 2x2 parity interleave
// parts: 4 buffers [B*Hh*Wh, C] (order (py, px) = (0,0), (0,1), (1,0), (1,1)); out [B*(2Hh)*(2Wh), out_ld]
__global__ void __launch_bounds__(256) interleave2x2_kernel(const __half* __restrict__ p00, const __half* __restrict__ p01,
                                                            const __half* __restrict__ p10, const __half* __restrict__ p11,
                                                            int part_ld, __half* __restrict__ out, int out_ld, int B, int Hh,
                                                            int Wh, int C) {
  const int CV = C / 8;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * Hh * Wh * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long pix = i / CV;
  const int j = static_cast<int>(pix % Wh);
  const long long t = pix / Wh;
  const int ii = static_cast<int>(t % Hh);
  const long long b = t / Hh;
  const long long base = ((b * 2 * Hh + 2 * ii) * 2 * Wh + 2 * j);
  const long long src = pix * part_ld + cv * 8;
  *reinterpret_cast<uint4*>(out + base * out_ld + cv * 8) = __ldg(reinterpret_cast<const uint4*>(p00 + src));
  *reinterpret_cast<uint4*>(out + (base + 1) * out_ld + cv * 8) = __ldg(reinterpret_cast<const uint4*>(p01 + src));
  *reinterpret_cast<uint4*>(out + (base + 2 * Wh) * out_ld + cv * 8) = __ldg(reinterpret_cast<const uint4*>(p10 + src));
  *reinterpret_cast<uint4*>(out + (base + 2 * Wh + 1) * out_ld + cv * 8) = __ldg(reinterpret_cast<const uint4*>(p11 + src));
}
int launch_interleave2x2(const __half* p00, const __half* p01, const __half* p10, const __half* p11, int part_ld, __half* out,
                         int out_ld, int B, int Hh, int Wh, int C, cudaStream_t st) {
  if (C % 8 || part_ld % 8 || out_ld % 8) { set_error("interleave2x2: bad shape"); return -1; }
  const long long n = static_cast<long long>(B) * Hh * Wh * (C / 8);
  (void)launch_k(interleave2x2_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, p00, p01, p10, p11, part_ld,
                 out, out_ld, B, Hh, Wh, C);
  return check_cuda(cudaGetLastError(), "interleave2x2");
}

}  // namespace mf
