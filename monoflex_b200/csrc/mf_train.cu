// Training-side HBM kernels (SURVEY §8 rows R11 backward, R13).
//
//  * adamw_arena_kernel: torch.optim.AdamW over ONE flat parameter / gradient / moment arena. The reference builds one
//    param group per tensor (solver/__init__.py:10-24, lr = BASE_LR or BASE_LR * BIAS_LR_FACTOR when "bias" is in the
//    name) => ~280 groups and ~1000 tiny kernels per step in eager torch; here each tensor is padded to a multiple of
//    ADAMW_CHUNK elements inside the arena and a per-chunk lr table selects the group's lr, so the whole step is one
//    launch that streams 28 B/parameter (read p, g, m, v; write p, m, v).
//  * focal_loss_backward_kernel: d/dpred of FocalLoss.forward (model/layers/focal_loss.py:35-55) scaled by a device
//    scalar (loss weight / clamp(num_pos, 1), detector_loss.py:276).
#include "mf_common.cuh"
#include "mf_launch.h"

namespace mf {

// ---------------------------------------------------------------- AdamW (torch/optim/adamw.py single-tensor semantics)
//   p   <- p * (1 - lr * wd)
//   m   <- m + (g - m) * (1 - beta1)                (torch: exp_avg.lerp_(grad, 1 - beta1))
//   v   <- v * beta2 + (1 - beta2) * g * g          (torch: exp_avg_sq.mul_(beta2).addcmul_(g, g, value = 1 - beta2))
//   p   <- p - (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
// g is first multiplied by grad_scale (1 / world_size when the arena holds an NCCL SUM; 1 otherwise).
struct AdamwConsts {
  float beta1, beta2, eps, wd, bc1, rsqrt_bc2, grad_scale, lr_scale;
};
__device__ __forceinline__ void adamw_update4(float4& pp, const float4& gg, float4& mm, float4& vv, float lr,
                                              const AdamwConsts& k) {
  const float omb1 = 1.f - k.beta1, omb2 = 1.f - k.beta2;
  const float decay = 1.f - lr * k.wd, step = lr / k.bc1;
  float* pe = reinterpret_cast<float*>(&pp);
  float* me = reinterpret_cast<float*>(&mm);
  float* ve = reinterpret_cast<float*>(&vv);
  const float* ge = reinterpret_cast<const float*>(&gg);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float gk = ge[e] * k.grad_scale;
    float pk = pe[e] * decay;
    const float mk = me[e] + (gk - me[e]) * omb1;
    const float vk = ve[e] * k.beta2 + omb2 * gk * gk;
    const float denom = sqrtf(vk) * k.rsqrt_bc2 + k.eps;
    pk -= step * (mk / denom);
    pe[e] = pk; me[e] = mk; ve[e] = vk;
  }
}

__global__ void __launch_bounds__(256) adamw_arena_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                          float* __restrict__ m, float* __restrict__ v,
                                                          const float* __restrict__ chunk_lr, long long n_chunks,
                                                          AdamwConsts k) {
  constexpr int VEC_PER_CHUNK = MF_ADAMW_CHUNK / 4;
  const long long n_vec = n_chunks * VEC_PER_CHUNK;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float lr = __ldg(chunk_lr + i / VEC_PER_CHUNK) * k.lr_scale;
    if (lr == 0.f) continue;                                   // padding-only chunk / frozen tensor
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = __ldcs(reinterpret_cast<const float4*>(g) + i);
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    adamw_update4(pp, gg, mm, vv, lr, k);
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
}

// ---------------------------------------------------------------- gradient exchange fused with the update (row R13, N > 1)
// DDP's allreduce + optimizer.step (tools/plain_train_net.py:100-104, engine/trainer.py:116-121) as ONE kernel over peer
// memory: every rank owns a contiguous 1/world shard of the arena's chunks. For its shard it
//   1. reduces the gradient of all ranks - either `multimem.ld_reduce` on the NVLS multicast address (the NVSwitch adds
//      the world copies in the fabric, one 16-byte request per float4) or a fixed-order sum of peer loads over NVLink;
//   2. applies AdamW with ITS shard of the moments (the optimizer state is only ever touched by the owner: ZeRO-1);
//   3. writes the new parameters into EVERY rank's parameter arena (`multimem.st` broadcast or peer stores).
// Per rank and step that is 1/world of (world x 4 + 12) bytes per parameter read and world x 4 + 8 written, against NCCL
// allreduce (2 x 4 x (world-1)/world over NVLink + 8 B HBM) followed by the 28 B/parameter update; the two system-scope
// barriers around the kernel are the only other synchronisation. Each element is produced by exactly one rank with a
// rank-independent summation order, so all replicas stay bit-identical.
struct PeerPtrs {
  float* p[MF_MAX_PEERS];
  const float* g[MF_MAX_PEERS];
};
__device__ __forceinline__ float4 multimem_ld_reduce_add(const float* addr) {
  float4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(addr) : "memory");
  return r;
}
__device__ __forceinline__ void multimem_st(float* addr, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};"
               :: "l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__global__ void __launch_bounds__(256) adamw_p2p_kernel(PeerPtrs peers, int world, int rank, float* mc_p, const float* mc_g,
                                                        float* __restrict__ m, float* __restrict__ v,
                                                        const float* __restrict__ chunk_lr, long long chunk_lo,
                                                        long long chunk_hi, AdamwConsts k) {
  constexpr int VEC_PER_CHUNK = MF_ADAMW_CHUNK / 4;
  const long long v_lo = chunk_lo * VEC_PER_CHUNK, v_hi = chunk_hi * VEC_PER_CHUNK;
  for (long long i = v_lo + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < v_hi;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float lr = __ldg(chunk_lr + i / VEC_PER_CHUNK) * k.lr_scale;
    if (lr == 0.f) continue;
    float4 gg;
    if (mc_g != nullptr) {
      gg = multimem_ld_reduce_add(mc_g + 4 * i);
    } else {
      gg = __ldcg(reinterpret_cast<const float4*>(peers.g[0]) + i);
      for (int r = 1; r < world; ++r) {
        const float4 t = __ldcg(reinterpret_cast<const float4*>(peers.g[r]) + i);
        gg.x += t.x; gg.y += t.y; gg.z += t.z; gg.w += t.w;
      }
    }
    float4 pp = reinterpret_cast<const float4*>(peers.p[rank])[i];
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    adamw_update4(pp, gg, mm, vv, lr, k);
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
    if (mc_p != nullptr) {
      multimem_st(mc_p + 4 * i, pp);
    } else {
      for (int r = 0; r < world; ++r) reinterpret_cast<float4*>(peers.p[r])[i] = pp;
    }
  }
}

static AdamwConsts adamw_consts(float beta1, float beta2, float eps, float wd, long long step, float grad_scale,
                                float lr_scale) {
  // bias corrections in double like torch's Python scalars
  const double bc1 = 1.0 - pow(static_cast<double>(beta1), static_cast<double>(step));
  const double bc2 = 1.0 - pow(static_cast<double>(beta2), static_cast<double>(step));
  AdamwConsts k;
  k.beta1 = beta1; k.beta2 = beta2; k.eps = eps; k.wd = wd;
  k.bc1 = static_cast<float>(bc1); k.rsqrt_bc2 = static_cast<float>(1.0 / sqrt(bc2));
  k.grad_scale = grad_scale; k.lr_scale = lr_scale;
  return k;
}

int launch_adamw_p2p(const unsigned long long* param_ptrs, const unsigned long long* grad_ptrs, int world, int rank,
                     unsigned long long mc_params, unsigned long long mc_grads, float* m, float* v, const float* chunk_lr,
                     long long n_chunks, float beta1, float beta2, float eps, float wd, long long step, float lr_scale,
                     cudaStream_t st) {
  if (world < 1 || world > MF_MAX_PEERS || rank < 0 || rank >= world) {
    set_error("adamw_p2p: world %d (max %d) / rank %d", world, MF_MAX_PEERS, rank);
    return -1;
  }
  if (step < 1) { set_error("adamw_p2p: step must be >= 1"); return -1; }
  if ((mc_params == 0) != (mc_grads == 0)) { set_error("adamw_p2p: give both multicast addresses or neither"); return -1; }
  PeerPtrs peers;
  for (int r = 0; r < MF_MAX_PEERS; ++r) {
    peers.p[r] = r < world ? reinterpret_cast<float*>(param_ptrs[r]) : nullptr;
    peers.g[r] = r < world ? reinterpret_cast<const float*>(grad_ptrs[r]) : nullptr;
  }
  const long long base = n_chunks / world, extra = n_chunks % world;      // parallel.shard_range semantics
  const long long lo = rank * base + (rank < extra ? rank : extra), hi = lo + base + (rank < extra ? 1 : 0);
  if (hi <= lo) return 0;
  const long long n_vec = (hi - lo) * (MF_ADAMW_CHUNK / 4);
  long long blocks = (n_vec + 255) / 256;
  const long long cap = 148LL * 8 * 4;
  if (blocks > cap) blocks = cap;
  const AdamwConsts k = adamw_consts(beta1, beta2, eps, wd, step, 1.f / static_cast<float>(world), lr_scale);
  adamw_p2p_kernel<<<dim3(static_cast<unsigned>(blocks)), dim3(256), 0, st>>>(
      peers, world, rank, reinterpret_cast<float*>(mc_params), reinterpret_cast<const float*>(mc_grads), m, v, chunk_lr, lo,
      hi, k);
  return check_cuda(cudaGetLastError(), "adamw_p2p");
}

int launch_adamw_arena(float* p, const float* g, float* m, float* v, const float* chunk_lr, long long n_chunks,
                       float beta1, float beta2, float eps, float wd, long long step, float grad_scale, float lr_scale,
                       cudaStream_t st) {
  if (n_chunks <= 0) return 0;
  if (step < 1) { set_error("adamw: step must be >= 1 (1-based count of the update being applied)"); return -1; }
  const long long n_vec = n_chunks * (MF_ADAMW_CHUNK / 4);
  long long blocks = (n_vec + 255) / 256;
  const long long cap = 148LL * 8 * 4;                          // a few waves; grid-stride for the rest
  if (blocks > cap) blocks = cap;
  (void)launch_k(adamw_arena_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, st, p, g, m, v, chunk_lr,
                 n_chunks, adamw_consts(beta1, beta2, eps, wd, step, grad_scale, lr_scale));
  return check_cuda(cudaGetLastError(), "adamw_arena");
}

// ---------------------------------------------------------------- CUDA-graph-safe AdamW step with a finite guard
// `mf_adamw_step` takes the step count (for the bias corrections) as a host scalar, which a captured graph would freeze.
// Here the count lives on the device and three launches make one optimiser step:
//   1. grad_finite_kernel : state[1] |= any non-finite element in the gradient arena (fp16 gradient flow under a loss
//                           scale can overflow; one inf written by AdamW poisons params, exp_avg and exp_avg_sq for good);
//   2. adamw_prepare_kernel (1 thread): if the flag is clean, step += 1 and the bias corrections of the new step are
//                           computed in double (torch computes them in Python doubles); else the step is skipped
//                           (state[2] += 1). Either way it publishes (bc1, rsqrt_bc2, skip) and clears the flag;
//   3. adamw_arena_dyn_kernel: the arena update, reading those three values from device memory.
// state = long long[4]: [0] step count, [1] found-non-finite flag of the current step, [2] skipped steps, [3] unused.
struct AdamwDyn { float bc1, rsqrt_bc2; int skip, pad; };

__global__ void __launch_bounds__(256) grad_finite_kernel(const float* __restrict__ g, long long n_vec, long long* state) {
  bool bad = false;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(g) + i);
    // x - x is 0 for finite x and NaN for inf / NaN
    const float t = (v.x - v.x) + (v.y - v.y) + (v.z - v.z) + (v.w - v.w);
    bad |= !(t == 0.f);
  }
  if (__syncthreads_or(bad ? 1 : 0) && threadIdx.x == 0) atomicExch(reinterpret_cast<unsigned long long*>(state + 1), 1ull);
}
__global__ void adamw_prepare_kernel(long long* state, AdamwDyn* dyn, float beta1, float beta2, int check) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const bool skip = check != 0 && state[1] != 0;
  if (skip) state[2] += 1; else state[0] += 1;
  state[1] = 0;
  const double step = static_cast<double>(state[0] < 1 ? 1 : state[0]);
  const double bc1 = 1.0 - pow(static_cast<double>(beta1), step);
  const double bc2 = 1.0 - pow(static_cast<double>(beta2), step);
  dyn->bc1 = static_cast<float>(bc1);
  dyn->rsqrt_bc2 = static_cast<float>(1.0 / sqrt(bc2));
  dyn->skip = skip ? 1 : 0;
}
__global__ void __launch_bounds__(256) adamw_arena_dyn_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                              float* __restrict__ m, float* __restrict__ v,
                                                              const float* __restrict__ chunk_lr, long long n_chunks,
                                                              AdamwConsts k, const AdamwDyn* __restrict__ dyn) {
  if (dyn->skip) return;
  k.bc1 = dyn->bc1;
  k.rsqrt_bc2 = dyn->rsqrt_bc2;
  constexpr int VEC_PER_CHUNK = MF_ADAMW_CHUNK / 4;
  const long long n_vec = n_chunks * VEC_PER_CHUNK;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float lr = __ldg(chunk_lr + i / VEC_PER_CHUNK) * k.lr_scale;
    if (lr == 0.f) continue;
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = __ldcs(reinterpret_cast<const float4*>(g) + i);
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    adamw_update4(pp, gg, mm, vv, lr, k);
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
}
int launch_adamw_arena_dyn(float* p, const float* g, float* m, float* v, const float* chunk_lr, long long n_chunks,
                           float beta1, float beta2, float eps, float wd, float grad_scale, float lr_scale, long long* state4,
                           void* dyn16, int check_finite, cudaStream_t st) {
  if (n_chunks <= 0) return 0;
  const long long n_vec = n_chunks * (MF_ADAMW_CHUNK / 4);
  long long blocks = (n_vec + 255) / 256;
  const long long cap = 148LL * 8 * 4;
  if (blocks > cap) blocks = cap;
  if (check_finite)
    (void)launch_k(grad_finite_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, st, g, n_vec, state4);
  (void)launch_k(adamw_prepare_kernel, dim3(1), dim3(32), 0, st, state4, static_cast<AdamwDyn*>(dyn16), beta1, beta2, check_finite);
  AdamwConsts k;
  k.beta1 = beta1; k.beta2 = beta2; k.eps = eps; k.wd = wd; k.bc1 = 1.f; k.rsqrt_bc2 = 1.f;
  k.grad_scale = grad_scale; k.lr_scale = lr_scale;
  (void)launch_k(adamw_arena_dyn_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, st, p, g, m, v, chunk_lr, n_chunks, k,
                 static_cast<const AdamwDyn*>(dyn16));
  return check_cuda(cudaGetLastError(), "adamw_arena_dyn");
}

// ---------------------------------------------------------------- focal loss backward (layers/focal_loss.py:35-55)
// L = -sum_{t==1} log(p)(1-p)^2 - sum_{0<=t<1} log(1-p) p^2 (1-t)^4
// dL/dp = -( (1-p)^2 / p - 2 (1-p) log p )                          at t == 1
//       = -(1-t)^4 ( 2 p log(1-p) - p^2 / (1-p) )                   at 0 <= t < 1,   0 elsewhere (ignored pixels, t = -1)
__global__ void focal_loss_backward_kernel(const float* __restrict__ pred, const float* __restrict__ tgt, long long n,
                                           const float* __restrict__ scale, float* __restrict__ grad) {
  const float s = __ldg(scale);
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float p = __ldg(pred + i), t = __ldg(tgt + i);
    float d = 0.f;
    if (t == 1.f) {
      const float q = 1.f - p;
      d = -(q * q / p - 2.f * q * logf(p));
    } else if (t < 1.f && t >= 0.f) {
      const float omt = 1.f - t, omt2 = omt * omt;
      d = -omt2 * omt2 * (2.f * p * logf(1.f - p) - p * p / (1.f - p));
    }
    grad[i] = d * s;
  }
}

int launch_focal_loss_backward(const float* pred, const float* tgt, long long n, const float* scale, float* grad,
                               cudaStream_t st) {
  if (n <= 0) return 0;
  long long blocks = (n + 1023) / 1024;
  if (blocks > 148 * 8) blocks = 148 * 8;
  (void)launch_k(focal_loss_backward_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, st, pred, tgt, n, scale,
                 grad);
  return check_cuda(cudaGetLastError(), "focal_loss_backward");
}

}  // namespace mf
