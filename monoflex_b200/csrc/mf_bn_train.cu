// Training-mode BatchNorm2d over NHWC fp16 rows (nn.BatchNorm2d(momentum=0.1) after every conv of the backbone,
// model/backbone/dla_dcn.py:76-79 etc.; eval mode is folded into the conv epilogue instead). HBM-bound kernels:
//   forward : bn_partial_kernel     per-CTA fp32 partial sums of x and x^2 per channel (deterministic: fixed row->CTA map)
//             bn_finalize_kernel    fixed-order double reduction -> mean, biased var, (scale, shift), running-stat update
//             bn_apply_kernel       y = act(x * scale + shift [+ residual])                     (one read, one write)
//   backward: bn_bwd_partial_kernel per-CTA partial sums of g and g * xhat, g = dy * act'(y)
//             bn_bwd_finalize_kernel dgamma, dbeta (fixed-order double reduction)
//             bn_bwd_apply_kernel   dx = scale * (g - mean(g) - xhat * mean(g * xhat))
// x is the raw conv output, y the activated output kept from the forward (its sign gives the ReLU / leaky mask).
#include "mf_common.cuh"
#include "mf_launch.h"

namespace mf {

MF_DEVINL void bn_unpack8(const uint4& v, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 t = __half22float2(h[e]);
    f[2 * e] = t.x; f[2 * e + 1] = t.y;
  }
}
MF_DEVINL uint4 bn_pack8(const float (&f)[8]) {
  __half2 o[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) o[e] = __floats2half2_rn(f[2 * e], f[2 * e + 1]);
  return *reinterpret_cast<uint4*>(o);
}
MF_DEVINL float bn_act_grad(float y, int act) {           // derivative of the activation, from the sign of its OUTPUT
  if (act == 1) return y > 0.f ? 1.f : 0.f;               // ReLU
  if (act == 2) return y > 0.f ? 1.f : 0.01f;             // leaky_relu(0.01) (InPlaceABN)
  return 1.f;
}

// thread (cv, r): channel chunk cv (8 channels), row lane r; the CTA walks rows r0 + r, r0 + r + RL, ... of ITS slab.
// part layout: [ncta][2][C] (sum a, sum b)
template <bool BWD>
__global__ void __launch_bounds__(256) bn_partial_kernel(const __half* __restrict__ x, int x_ld, const __half* __restrict__ dy,
                                                         int dy_ld, const __half* __restrict__ y, int y_ld,
                                                         const float* __restrict__ mean, const float* __restrict__ rstd,
                                                         long long M, int C, int act, long long rows_per_cta,
                                                         float* __restrict__ part) {
  extern __shared__ float sm[];                            // [RL][2][C]
  const int CV = C / 8, RL = blockDim.x / CV;
  const int cv = threadIdx.x % CV, r = threadIdx.x / CV;
  float a[8], b[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) a[e] = b[e] = 0.f;
  float mu[8], rs[8];
  if (BWD) {
#pragma unroll
    for (int e = 0; e < 8; ++e) { mu[e] = mean[cv * 8 + e]; rs[e] = rstd[cv * 8 + e]; }
  }
  const long long r0 = static_cast<long long>(blockIdx.x) * rows_per_cta;
  const long long r1 = r0 + rows_per_cta < M ? r0 + rows_per_cta : M;
  if (r < RL) {
    constexpr int U = 4;                                   // rows in flight per thread: all loads of a group are issued first
    for (long long row = r0 + r; row < r1; row += static_cast<long long>(U) * RL) {
      uint4 xq[U], gq[U], yq[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long rr = row + static_cast<long long>(u) * RL;
        const bool ok = rr < r1;
        const long long rc = ok ? rr : row;
        xq[u] = __ldg(reinterpret_cast<const uint4*>(x + rc * x_ld + cv * 8));
        if (BWD) {
          gq[u] = ok ? __ldg(reinterpret_cast<const uint4*>(dy + rc * dy_ld + cv * 8)) : make_uint4(0u, 0u, 0u, 0u);
          yq[u] = __ldg(reinterpret_cast<const uint4*>(y + rc * y_ld + cv * 8));
        } else if (!ok) {
          xq[u] = make_uint4(0u, 0u, 0u, 0u);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {                        // fixed accumulation order: row, row + RL, ...
        float xv[8];
        bn_unpack8(xq[u], xv);
        if (!BWD) {
#pragma unroll
          for (int e = 0; e < 8; ++e) { a[e] += xv[e]; b[e] += xv[e] * xv[e]; }
        } else {
          float gv[8], yv[8];
          bn_unpack8(gq[u], gv);
          bn_unpack8(yq[u], yv);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float g = gv[e] * bn_act_grad(yv[e], act);
            a[e] += g;
            b[e] += g * (xv[e] - mu[e]) * rs[e];
          }
        }
      }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) { sm[(r * 2 + 0) * C + cv * 8 + e] = a[e]; sm[(r * 2 + 1) * C + cv * 8 + e] = b[e]; }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {  // fixed order over the row lanes
    float s = 0.f;
    for (int q = 0; q < RL; ++q) s += sm[q * 2 * C + i];
    part[static_cast<long long>(blockIdx.x) * 2 * C + i] = s;
  }
}

// fixed-order double sum of part[k][which][c], k < ncta, by one warp: lane l takes k = l, l + 32, ... then a shuffle tree
MF_DEVINL double bn_warp_sum(const float* __restrict__ part, int ncta, int C, int which, int c, int lane) {
  double s = 0.0;
  for (int k = lane; k < ncta; k += 32) s += static_cast<double>(part[(static_cast<long long>(k) * 2 + which) * C + c]);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  return s;
}

// forward finalize: one WARP per channel (a single thread walking ~1000 partials was 22 us of pure latency per layer)
__global__ void bn_finalize_kernel(const float* __restrict__ part, int ncta, int C, long long M, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum, int abs_gamma,
                                   float* __restrict__ running_mean, float* __restrict__ running_var,
                                   float* __restrict__ mean_out, float* __restrict__ rstd_out, float* __restrict__ scale,
                                   float* __restrict__ shift) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  const double s = bn_warp_sum(part, ncta, C, 0, c, lane), ss = bn_warp_sum(part, ncta, C, 1, c, lane);
  if (lane != 0) return;
  const double mean = s / static_cast<double>(M);
  double var = ss / static_cast<double>(M) - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  float g = gamma[c];
  if (abs_gamma) g = fabsf(g) + eps;                       // InPlaceABN convention used by the head (see DESIGN §5)
  mean_out[c] = static_cast<float>(mean);
  rstd_out[c] = rstd;
  scale[c] = g * rstd;
  shift[c] = beta[c] - static_cast<float>(mean) * g * rstd;
  if (running_mean != nullptr) {                           // torch: running = (1 - m) running + m * batch (unbiased var)
    const double unb = M > 1 ? var * static_cast<double>(M) / static_cast<double>(M - 1) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(mean);
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unb);
  }
}

__global__ void __launch_bounds__(256) bn_apply_kernel(const __half* __restrict__ x, int x_ld, const float* __restrict__ scale,
                                                       const float* __restrict__ shift, const __half* __restrict__ res,
                                                       int res_ld, int act, __half* __restrict__ y, int y_ld, long long M, int C) {
  const int CV = C / 8;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= M * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long row = i / CV;
  float v[8], rv[8], sc[8], sh[8];
  const uint4 xq = __ldg(reinterpret_cast<const uint4*>(x + row * x_ld + cv * 8));
  const uint4 rq = res != nullptr ? __ldg(reinterpret_cast<const uint4*>(res + row * res_ld + cv * 8)) : make_uint4(0u, 0u, 0u, 0u);
  *reinterpret_cast<float4*>(&sc[0]) = __ldg(reinterpret_cast<const float4*>(scale + cv * 8));
  *reinterpret_cast<float4*>(&sc[4]) = __ldg(reinterpret_cast<const float4*>(scale + cv * 8 + 4));
  *reinterpret_cast<float4*>(&sh[0]) = __ldg(reinterpret_cast<const float4*>(shift + cv * 8));
  *reinterpret_cast<float4*>(&sh[4]) = __ldg(reinterpret_cast<const float4*>(shift + cv * 8 + 4));
  bn_unpack8(xq, v);
  bn_unpack8(rq, rv);
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    float t = v[e] * sc[e] + sh[e];
    if (res != nullptr) t += rv[e];
    if (act == 1) t = fmaxf(t, 0.f);
    else if (act == 2) t = fmaxf(t, 0.01f * t);
    v[e] = t;
  }
  *reinterpret_cast<uint4*>(y + row * y_ld + cv * 8) = bn_pack8(v);
}

__global__ void bn_bwd_finalize_kernel(const float* __restrict__ part, int ncta, int C, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta, float* __restrict__ sum_g, float* __restrict__ sum_gx) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  const double s = bn_warp_sum(part, ncta, C, 0, c, lane), sx = bn_warp_sum(part, ncta, C, 1, c, lane);
  if (lane != 0) return;
  dbeta[c] = static_cast<float>(s);
  dgamma[c] = static_cast<float>(sx);
  sum_g[c] = static_cast<float>(s);
  sum_gx[c] = static_cast<float>(sx);
}

// dx = scale * (g - sum_g / M - xhat * sum_gx / M); also returns g through `dres` when the layer had a residual input
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const __half* __restrict__ x, int x_ld, const __half* __restrict__ dy,
                                                           int dy_ld, const __half* __restrict__ y, int y_ld,
                                                           const float* __restrict__ mean, const float* __restrict__ rstd,
                                                           const float* __restrict__ scale, const float* __restrict__ sum_g,
                                                           const float* __restrict__ sum_gx, int act, __half* __restrict__ dx,
                                                           int dx_ld, __half* __restrict__ dres, int dres_ld, long long M, int C,
                                                           double count) {
  const int CV = C / 8;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= M * CV) return;
  const int cv = static_cast<int>(i % CV);
  const long long row = i / CV;
  float xv[8], gv[8], yv[8], o[8], gr[8], mu[8], rs[8], sc[8], sg[8], sgx[8];
  const uint4 xq = __ldg(reinterpret_cast<const uint4*>(x + row * x_ld + cv * 8));
  const uint4 gq = __ldg(reinterpret_cast<const uint4*>(dy + row * dy_ld + cv * 8));
  const uint4 yq = __ldg(reinterpret_cast<const uint4*>(y + row * y_ld + cv * 8));
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    *reinterpret_cast<float4*>(&mu[4 * h]) = __ldg(reinterpret_cast<const float4*>(mean + cv * 8 + 4 * h));
    *reinterpret_cast<float4*>(&rs[4 * h]) = __ldg(reinterpret_cast<const float4*>(rstd + cv * 8 + 4 * h));
    *reinterpret_cast<float4*>(&sc[4 * h]) = __ldg(reinterpret_cast<const float4*>(scale + cv * 8 + 4 * h));
    *reinterpret_cast<float4*>(&sg[4 * h]) = __ldg(reinterpret_cast<const float4*>(sum_g + cv * 8 + 4 * h));
    *reinterpret_cast<float4*>(&sgx[4 * h]) = __ldg(reinterpret_cast<const float4*>(sum_gx + cv * 8 + 4 * h));
  }
  bn_unpack8(xq, xv);
  bn_unpack8(gq, gv);
  bn_unpack8(yq, yv);
  const float inv_m = static_cast<float>(1.0 / count);          // global element count (== M unless SyncBatchNorm)
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float g = gv[e] * bn_act_grad(yv[e], act);
    const float xhat = (xv[e] - mu[e]) * rs[e];
    o[e] = sc[e] * (g - sg[e] * inv_m - xhat * sgx[e] * inv_m);
    gr[e] = g;
  }
  *reinterpret_cast<uint4*>(dx + row * dx_ld + cv * 8) = bn_pack8(o);
  if (dres != nullptr) *reinterpret_cast<uint4*>(dres + row * dres_ld + cv * 8) = bn_pack8(gr);
}

// ------------------------------------------------------------------------------------------------ SyncBatchNorm halves
// torch.nn.SyncBatchNorm (the reference converts every BatchNorm when MODEL.USE_SYNC_BN is set, tools/plain_train_net.py:131-132)
// normalises with statistics over the batches of ALL ranks. The kernels above are split around the exchange:
//   forward : bn_partial -> bn_reduce (per-channel local sums, double) | all-reduce of [2][C] doubles | bn_finalize_sums -> bn_apply
//   backward: bn_partial<BWD> -> bn_reduce (+ local dgamma / dbeta, which DDP averages like every other gradient) |
//             all-reduce of [2][C] doubles | bn_bwd_apply with the global sums and the global element count
// The collective itself is issued by the host between the two C-ABI calls (torch.distributed / NCCL on the same stream).
__global__ void bn_reduce_kernel(const float* __restrict__ part, int ncta, int C, double* __restrict__ sums) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  const double s0 = bn_warp_sum(part, ncta, C, 0, c, lane), s1 = bn_warp_sum(part, ncta, C, 1, c, lane);
  if (lane == 0) { sums[c] = s0; sums[C + c] = s1; }
}
__global__ void bn_finalize_sums_kernel(const double* __restrict__ sums, int C, double count, const float* __restrict__ gamma,
                                        const float* __restrict__ beta, float eps, float momentum, int abs_gamma,
                                        float* __restrict__ running_mean, float* __restrict__ running_var,
                                        float* __restrict__ mean_out, float* __restrict__ rstd_out, float* __restrict__ scale,
                                        float* __restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double mean = sums[c] / count;
  double var = sums[C + c] / count - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  float g = gamma[c];
  if (abs_gamma) g = fabsf(g) + eps;
  mean_out[c] = static_cast<float>(mean);
  rstd_out[c] = rstd;
  scale[c] = g * rstd;
  shift[c] = beta[c] - static_cast<float>(mean) * g * rstd;
  if (running_mean != nullptr) {
    const double unb = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(mean);
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unb);
  }
}
__global__ void bn_bwd_sums_kernel(const double* __restrict__ sums, int C, float* __restrict__ sum_g, float* __restrict__ sum_gx,
                                   float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float s = static_cast<float>(sums[c]), sx = static_cast<float>(sums[C + c]);
  if (sum_g != nullptr) { sum_g[c] = s; sum_gx[c] = sx; }
  if (dgamma != nullptr) { dbeta[c] = s; dgamma[c] = sx; }
}

// ------------------------------------------------------------------------------------------------ launchers
static int bn_grid(long long M, int C, long long& rows_per_cta, int& threads, size_t& smem) {
  const int CV = C / 8;
  threads = 256;
  if (CV > 256) return -1;
  const int RL = threads / CV;
  smem = static_cast<size_t>(RL) * 2 * C * sizeof(float);
  // Enough CTAs to keep every SM's memory pipe full: up to 8 per SM, each owning a whole number of 4 x RL row groups (the
  // kernel keeps 4 rows per thread in flight). The first version gave a CTA >= 1024 rows: 240 CTAs for the 245760-pixel maps
  // (1.6 per SM, ~26 KB in flight per SM) and 60 for level 3 - the statistics passes ran at ~1 TB/s.
  const long long group = 4ll * RL;
  long long ncta = (M + group - 1) / group;
  if (ncta > 148 * 8) ncta = 148 * 8;
  if (ncta < 1) ncta = 1;
  rows_per_cta = (M + ncta - 1) / ncta;
  rows_per_cta = (rows_per_cta + group - 1) / group * group;
  return static_cast<int>((M + rows_per_cta - 1) / rows_per_cta);
}
size_t bn_train_workspace_floats(long long M, int C) {
  long long rpc; int th; size_t sm;
  const int ncta = bn_grid(M, C, rpc, th, sm);
  return ncta < 0 ? 0 : static_cast<size_t>(ncta) * 2 * C + 2 * static_cast<size_t>(C);
}

int launch_bn_train_forward(const __half* x, int x_ld, long long M, int C, const float* gamma, const float* beta, float eps,
                            float momentum, int abs_gamma, float* running_mean, float* running_var, const __half* res,
                            int res_ld, int act, __half* y, int y_ld, float* mean, float* rstd, float* scale, float* shift,
                            float* workspace, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || y_ld % 8 || (res && res_ld % 8) || C > 2048 || M < 1) { set_error("bn_train_forward: bad shape (C=%d)", C); return -1; }
  long long rpc; int th; size_t sm;
  const int ncta = bn_grid(M, C, rpc, th, sm);
  if (ncta < 0) { set_error("bn_train_forward: C=%d too wide", C); return -1; }
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(bn_partial_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    cudaFuncSetAttribute(bn_partial_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    attr = true;
  }
  if (sm > 64 * 1024) { set_error("bn_train_forward: shared memory"); return -1; }
  (void)launch_k(bn_partial_kernel<false>, dim3(ncta), dim3(th), sm, st, x, x_ld, static_cast<const __half*>(nullptr), 0,
                 static_cast<const __half*>(nullptr), 0, static_cast<const float*>(nullptr), static_cast<const float*>(nullptr), M,
                 C, 0, rpc, workspace);
  bn_finalize_kernel<<<(C * 32 + 127) / 128, 128, 0, st>>>(workspace, ncta, C, M, gamma, beta, eps, momentum, abs_gamma, running_mean,
                                                      running_var, mean, rstd, scale, shift);
  const long long n = M * (C / 8);
  (void)launch_k(bn_apply_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, x_ld,
                 static_cast<const float*>(scale), static_cast<const float*>(shift), res, res_ld, act, y, y_ld, M, C);
  return check_cuda(cudaGetLastError(), "bn_train_forward");
}

int launch_bn_train_backward(const __half* x, int x_ld, const __half* dy, int dy_ld, const __half* y, int y_ld, long long M, int C,
                             const float* mean, const float* rstd, const float* scale, int act, __half* dx, int dx_ld,
                             __half* dres, int dres_ld, float* dgamma, float* dbeta, float* workspace, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || dy_ld % 8 || y_ld % 8 || dx_ld % 8 || (dres && dres_ld % 8) || C > 2048 || M < 1) {
    set_error("bn_train_backward: bad shape (C=%d)", C);
    return -1;
  }
  long long rpc; int th; size_t sm;
  const int ncta = bn_grid(M, C, rpc, th, sm);
  if (ncta < 0 || sm > 64 * 1024) { set_error("bn_train_backward: C=%d too wide", C); return -1; }
  float* sums = workspace + static_cast<size_t>(ncta) * 2 * C;        // [2][C] after the partials
  (void)launch_k(bn_partial_kernel<true>, dim3(ncta), dim3(th), sm, st, x, x_ld, dy, dy_ld, y, y_ld, mean, rstd, M, C, act, rpc,
                 workspace);
  bn_bwd_finalize_kernel<<<(C * 32 + 127) / 128, 128, 0, st>>>(workspace, ncta, C, dgamma, dbeta, sums, sums + C);
  const long long n = M * (C / 8);
  (void)launch_k(bn_bwd_apply_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, x_ld, dy, dy_ld, y, y_ld,
                 mean, rstd, scale, static_cast<const float*>(sums), static_cast<const float*>(sums + C), act, dx, dx_ld, dres,
                 dres_ld, M, C, static_cast<double>(M));
  return check_cuda(cudaGetLastError(), "bn_train_backward");
}

// ---- SyncBatchNorm halves (see above). sums: double [2][C] device buffer the host all-reduces between the two calls.
int launch_bn_sync_forward_stats(const __half* x, int x_ld, long long M, int C, float* workspace, double* sums, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || C > 2048 || M < 1) { set_error("bn_sync_forward_stats: bad shape (C=%d)", C); return -1; }
  long long rpc; int th; size_t sm;
  const int ncta = bn_grid(M, C, rpc, th, sm);
  if (ncta < 0 || sm > 64 * 1024) { set_error("bn_sync_forward_stats: C=%d too wide", C); return -1; }
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(bn_partial_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    cudaFuncSetAttribute(bn_partial_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    attr = true;
  }
  (void)launch_k(bn_partial_kernel<false>, dim3(ncta), dim3(th), sm, st, x, x_ld, static_cast<const __half*>(nullptr), 0,
                 static_cast<const __half*>(nullptr), 0, static_cast<const float*>(nullptr), static_cast<const float*>(nullptr), M,
                 C, 0, rpc, workspace);
  bn_reduce_kernel<<<(C * 32 + 127) / 128, 128, 0, st>>>(workspace, ncta, C, sums);
  return check_cuda(cudaGetLastError(), "bn_sync_forward_stats");
}
int launch_bn_sync_forward_apply(const __half* x, int x_ld, long long M, int C, const double* sums, double count, const float* gamma,
                                 const float* beta, float eps, float momentum, int abs_gamma, float* running_mean,
                                 float* running_var, const __half* res, int res_ld, int act, __half* y, int y_ld, float* mean,
                                 float* rstd, float* scale, float* shift, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || y_ld % 8 || (res && res_ld % 8) || count < 1.0) { set_error("bn_sync_forward_apply: bad shape"); return -1; }
  bn_finalize_sums_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, C, count, gamma, beta, eps, momentum, abs_gamma, running_mean,
                                                           running_var, mean, rstd, scale, shift);
  const long long n = M * (C / 8);
  (void)launch_k(bn_apply_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, x_ld,
                 static_cast<const float*>(scale), static_cast<const float*>(shift), res, res_ld, act, y, y_ld, M, C);
  return check_cuda(cudaGetLastError(), "bn_sync_forward_apply");
}
int launch_bn_sync_backward_stats(const __half* x, int x_ld, const __half* dy, int dy_ld, const __half* y, int y_ld, long long M,
                                  int C, const float* mean, const float* rstd, int act, float* workspace, double* sums,
                                  float* dgamma, float* dbeta, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || dy_ld % 8 || y_ld % 8 || C > 2048 || M < 1) { set_error("bn_sync_backward_stats: bad shape"); return -1; }
  long long rpc; int th; size_t sm;
  const int ncta = bn_grid(M, C, rpc, th, sm);
  if (ncta < 0 || sm > 64 * 1024) { set_error("bn_sync_backward_stats: C=%d too wide", C); return -1; }
  (void)launch_k(bn_partial_kernel<true>, dim3(ncta), dim3(th), sm, st, x, x_ld, dy, dy_ld, y, y_ld, mean, rstd, M, C, act, rpc,
                 workspace);
  bn_reduce_kernel<<<(C * 32 + 127) / 128, 128, 0, st>>>(workspace, ncta, C, sums);
  bn_bwd_sums_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, C, nullptr, nullptr, dgamma, dbeta);      // local parameter gradients
  return check_cuda(cudaGetLastError(), "bn_sync_backward_stats");
}
int launch_bn_sync_backward_apply(const __half* x, int x_ld, const __half* dy, int dy_ld, const __half* y, int y_ld, long long M,
                                  int C, const float* mean, const float* rstd, const float* scale, const double* sums, double count,
                                  int act, __half* dx, int dx_ld, __half* dres, int dres_ld, float* workspace, cudaStream_t st) {
  if (C % 8 || x_ld % 8 || dy_ld % 8 || y_ld % 8 || dx_ld % 8 || (dres && dres_ld % 8) || count < 1.0) {
    set_error("bn_sync_backward_apply: bad shape");
    return -1;
  }
  float* fs = workspace;                                            // [2][C] float copies of the global sums
  bn_bwd_sums_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, C, fs, fs + C, nullptr, nullptr);
  const long long n = M * (C / 8);
  (void)launch_k(bn_bwd_apply_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, x, x_ld, dy, dy_ld, y, y_ld,
                 mean, rstd, scale, static_cast<const float*>(fs), static_cast<const float*>(fs + C), act, dx, dx_ld, dres,
                 dres_ld, M, C, count);
  return check_cuda(cudaGetLastError(), "bn_sync_backward_apply");
}

}  // namespace mf
