// Heat-map NMS + top-K + POI gather + keypoint->3D decode (model/layers/utils.py:45-145, model/head/detector_infer.py:77-237,
// model/anno_encoder.py:69-295). Integer outputs (indices, classes) are bit-exact against the oracle; the tie rule is
// (score desc, flat index asc) at both selection stages (torch.topk leaves ties unspecified, SURVEY H5).
//
// Stage 1: one CTA per (image, class). Each thread keeps its pixels' 47-bit keys (score bits << 15 | (32767-idx)) in
//          registers; an MSB-first 8-bit radix select with a shared-memory histogram finds the K-th largest key exactly
//          (keys are unique), the K survivors are compacted and bitonic-sorted. The 3x3 local-max test reads the logits'
//          neighbourhood straight from global memory (L1/L2 resident), so the heat map is read from HBM once.
// Stage 2: one CTA per image merges C*K candidates, gathers the 50 regression channels of each survivor and decodes.
#include "mf_common.cuh"
#include "mf_kernels.h"
#include "mf_launch.h"
#include <math_constants.h>

namespace mf {

#define MF_DECODE_SLABS 8
static constexpr int S1_THREADS = 1024;
static constexpr int S1_CAND = 2048;                   // candidate-list capacity of the rank-by-counting fast path (16 KB)

// hm: [B, C, H, W] fp32 (already sigmoid-ed when apply_sigmoid == 0). out_*: [B, C, K]
__global__ void __launch_bounds__(S1_THREADS)
nms_topk_stage1_kernel(const float* __restrict__ hm_all, int H, int W, int K, int apply_sigmoid, int slabs,
                       float* __restrict__ out_score, int* __restrict__ out_idx) {
  // blockIdx.x = plane * slabs + slab; a slab is a contiguous pixel range [lo, hi) of one (image, class) plane. The union
  // of the per-slab top-K sets contains the plane's top-K, so splitting only adds parallelism (148 SMs instead of B*C).
  const int HW = H * W;
  const int plane = blockIdx.x / slabs, slab = blockIdx.x - plane * slabs;
  const int chunk = (HW + slabs - 1) / slabs;
  const int lo = slab * chunk, hi = min(HW, lo + chunk);
  const float* hm = hm_all + static_cast<long long>(plane) * HW;
  __shared__ unsigned int hist[257];                  // bin 256 = "not a candidate" (keeps the warp converged)
  __shared__ unsigned long long sel[256];
  __shared__ unsigned long long s_prefix;
  __shared__ int s_remaining, s_count;
  // Fast path (round 2): after the 3x3 NMS only the local maxima are non-zero (~1/9 of the pixels), so the slab's non-zero keys are
  // compacted into `cand` and every candidate computes its RANK by counting the larger keys (keys are unique; all threads read
  // the same shared-memory word per iteration = broadcast, no barriers inside): O(n^2 / threads) comparisons instead of six
  // radix passes with three block-wide barriers each plus a 36-step bitonic sort. The exact radix path below remains the
  // fallback for degenerate maps (fewer non-zero maxima than K - zero-score pixels then enter by index order - or plateaus
  // with more than S1_CAND candidates).
  __shared__ unsigned long long cand[S1_CAND];
  __shared__ int s_ncand;
  if (threadIdx.x == 0) s_ncand = 0;
  __syncthreads();

  // per-thread score bits; the pixel index of item `it` is implicit (it*S1_THREADS + tid), the 47-bit key is rebuilt
  // on the fly: key = ((bits << 15) | (32767 - idx)) + 1   (0 = "no pixel")
  extern __shared__ unsigned int vbits_sm[];      // [S1_ITEMS][S1_THREADS] score bits (dynamic smem, <= 128 KB)
  unsigned int* vbits = vbits_sm + threadIdx.x;   // item `it` of this thread lives at vbits[it * S1_THREADS]
  const int n_items = (hi - lo + S1_THREADS - 1) / S1_THREADS;
  // The slab and its one-row halo are staged in shared memory first: coalesced, independent loads (6 per thread) instead of
  // 9 dependent neighbour loads per pixel from L2 (45 per thread, the bulk of this kernel's 26 us), same arithmetic per value.
  float* tile = reinterpret_cast<float*>(vbits_sm + static_cast<size_t>((chunk + S1_THREADS - 1) / S1_THREADS) * S1_THREADS);
  const int t_lo = max(0, lo - W - 1), t_hi = min(HW, hi + W + 1);
  for (int i = t_lo + static_cast<int>(threadIdx.x); i < t_hi; i += S1_THREADS) {
    float v = __ldg(hm + i);
    if (apply_sigmoid) {
      v = 1.f / (1.f + expf(-v));
      v = fminf(fmaxf(v, 1e-4f), 1.f - 1e-4f);
    }
    tile[i - t_lo] = v;
  }
  __syncthreads();
#define MF_KEY(it) (lo + (it) * S1_THREADS + static_cast<int>(threadIdx.x) < hi                                              \
                        ? ((static_cast<unsigned long long>(vbits[(it) * S1_THREADS]) << 15) |                                         \
                           static_cast<unsigned long long>(32767 - (lo + (it) * S1_THREADS + static_cast<int>(threadIdx.x)))) + 1ull \
                        : 0ull)
  int my_cnt = 0;
  for (int it = 0; it < n_items; ++it) {
    const int idx = lo + it * S1_THREADS + threadIdx.x;
    unsigned int key = 0u;
    if (idx < hi) {
      const int y = idx / W, x = idx - y * W;
      const float v = tile[idx - t_lo];
      float mx = v;                                   // max_pool2d 3x3 s1 p1 (-inf padding): nms_hm utils.py:45-58
#pragma unroll
      for (int dy = -1; dy <= 1; ++dy) {
        const int yy = y + dy;
        if (yy < 0 || yy >= H) continue;
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
          const int xx = x + dx;
          if (xx < 0 || xx >= W || (dx == 0 && dy == 0)) continue;
          mx = fmaxf(mx, tile[yy * W + xx - t_lo]);
        }
      }
      const float kept = (mx == v) ? v : 0.f;         // heat * (hmax == heat)
      key = __float_as_uint(kept);
    }
    vbits[it * S1_THREADS] = key;
    my_cnt += key != 0u ? 1 : 0;
  }
  // append the non-zero keys to the candidate list: ONE shared-memory atomic per warp (the per-item form issued 32 warps x 5
  // items = 160 serialised read-modify-writes on one address), then a second pass over the thread's own score bits
  {
    const int lane = threadIdx.x & 31;
    int incl = my_cnt;                                  // inclusive scan of the per-lane counts
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    const int warp_total = __shfl_sync(0xffffffffu, incl, 31);
    int base = 0;
    if (lane == 31 && warp_total > 0) base = atomicAdd(&s_ncand, warp_total);
    base = __shfl_sync(0xffffffffu, base, 31);
    int slot = base + incl - my_cnt;
    for (int it = 0; it < n_items; ++it) {
      const unsigned int key = vbits[it * S1_THREADS];
      if (key != 0u) {
        const int idx = lo + it * S1_THREADS + threadIdx.x;
        if (slot < S1_CAND) cand[slot] = ((static_cast<unsigned long long>(key) << 15) | static_cast<unsigned long long>(32767 - idx)) + 1ull;
        ++slot;
      }
    }
  }
  const int k_eff = min(K, hi - lo);                  // a slab narrower than K keeps everything it has
  __syncthreads();
  const int ncand = s_ncand;
  if (ncand >= k_eff && ncand <= S1_CAND) {           // block-uniform: the fast path
    for (int c = threadIdx.x; c < ncand; c += S1_THREADS) {
      const unsigned long long mine = cand[c];
      int rank = 0;
      for (int j = 0; j < ncand; ++j) rank += cand[j] > mine ? 1 : 0;
      if (rank < K) {
        const unsigned long long k = mine - 1ull;
        out_score[static_cast<long long>(blockIdx.x) * K + rank] = __uint_as_float(static_cast<unsigned int>(k >> 15));
        out_idx[static_cast<long long>(blockIdx.x) * K + rank] = 32767 - static_cast<int>(k & 32767ull);
      }
    }
    for (int r = k_eff + threadIdx.x; r < K; r += S1_THREADS) {      // a slab narrower than K: pad
      out_score[static_cast<long long>(blockIdx.x) * K + r] = 0.f;
      out_idx[static_cast<long long>(blockIdx.x) * K + r] = -1;
    }
    return;
  }
  if (threadIdx.x == 0) { s_prefix = 0ull; s_remaining = k_eff; }
  __syncthreads();

  // MSB-first radix select of the K-th largest key (48 significant bits -> 6 passes of 8 bits)
  for (int shift = 40; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 257; i += S1_THREADS) hist[i] = 0u;
    __syncthreads();
    const unsigned long long prefix = s_prefix;
    const unsigned long long himask = (shift + 8 >= 64) ? 0ull : (~0ull << (shift + 8));
    for (int it = 0; it < n_items; ++it) {
      const unsigned long long k = MF_KEY(it);
      const unsigned int digit = (k != 0ull && (k & himask) == prefix) ? static_cast<unsigned int>((k >> shift) & 255ull) : 256u;
      // warp-aggregated histogram: in the top passes every key of a warp has the same digit (same exponent bits), a plain
      // atomicAdd would serialise 32-fold on one shared-memory address
      const unsigned int peers = __match_any_sync(0xffffffffu, digit);
      if ((threadIdx.x & 31) == static_cast<unsigned int>(__ffs(peers) - 1)) atomicAdd(&hist[digit], __popc(peers));
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      // warp-parallel search of the digit holding the rem-th largest key: lane l owns bins [8l, 8l+8)
      const int lane = threadIdx.x;
      unsigned int c[8], tot = 0u;
#pragma unroll
      for (int i = 0; i < 8; ++i) { c[i] = hist[lane * 8 + i]; tot += c[i]; }
      unsigned int suf = tot;                       // inclusive suffix sum over lanes (higher lane = higher digit)
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const unsigned int t = __shfl_down_sync(0xffffffffu, suf, d);
        if (lane + d < 32) suf += t;
      }
      const unsigned int above = suf - tot;
      const unsigned int rem = static_cast<unsigned int>(s_remaining);
      __syncwarp();
      if (above < rem && suf >= rem) {              // exactly one lane
        unsigned int r = rem - above;
        int digit = lane * 8;
#pragma unroll
        for (int i = 7; i >= 0; --i) {
          if (c[i] >= r) { digit = lane * 8 + i; break; }
          r -= c[i];
        }
        s_remaining = static_cast<int>(r);
        s_prefix = prefix | (static_cast<unsigned long long>(digit) << shift);
      }
    }
    __syncthreads();
  }
  const unsigned long long kth = s_prefix;            // exact K-th largest key (keys unique)
  if (threadIdx.x == 0) s_count = 0;
  for (int i = threadIdx.x; i < 256; i += S1_THREADS) sel[i] = 0ull;
  __syncthreads();
  for (int it = 0; it < n_items; ++it) {
    const unsigned long long k = MF_KEY(it);
    if (k != 0ull && k >= kth) {
      const int slot = atomicAdd(&s_count, 1);
      if (slot < 256) sel[slot] = k;
    }
  }
  __syncthreads();
  // bitonic sort (descending) of 256 keys by the first 256 threads
  for (int size = 2; size <= 256; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      if (threadIdx.x < 256) {
        const int i = threadIdx.x, jn = i ^ stride;
        if (jn > i) {
          const unsigned long long a = sel[i], b = sel[jn];
          const bool desc = (i & size) == 0;
          if (desc ? (a < b) : (a > b)) { sel[i] = b; sel[jn] = a; }
        }
      }
      __syncthreads();
    }
  }
#undef MF_KEY
  if (threadIdx.x < K) {
    const bool have = threadIdx.x < k_eff;
    const unsigned long long k = have ? sel[threadIdx.x] - 1ull : 0ull;
    out_score[static_cast<long long>(blockIdx.x) * K + threadIdx.x] = have ? __uint_as_float(static_cast<unsigned int>(k >> 15)) : 0.f;
    out_idx[static_cast<long long>(blockIdx.x) * K + threadIdx.x] = have ? 32767 - static_cast<int>(k & 32767ull) : -1;
  }
}

// stand-alone nms_hm (model/layers/utils.py:45-58): out = heat * (maxpool3x3(heat) == heat)
__global__ void nms_hm_kernel(const float* __restrict__ hm, float* __restrict__ out, int H, int W, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int HW = H * W;
  const long long plane = i / HW;
  const int idx = static_cast<int>(i - plane * HW), y = idx / W, x = idx - y * W;
  const float* p = hm + plane * HW;
  const float v = p[idx];
  float mx = v;
  for (int dy = -1; dy <= 1; ++dy)
    for (int dx = -1; dx <= 1; ++dx) {
      const int yy = y + dy, xx = x + dx;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) mx = fmaxf(mx, p[yy * W + xx]);
    }
  out[i] = (mx == v) ? v : 0.f;
}
int launch_nms_hm(const float* hm, float* out, int planes, int H, int W, cudaStream_t st) {
  const long long n = static_cast<long long>(planes) * H * W;
  (void)launch_k(nms_hm_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, hm, out, H, W, n);
  return check_cuda(cudaGetLastError(), "nms_hm");
}

struct DecodeParams {
  const float* s1_score;  // [B, C, K]
  const int* s1_idx;      // [B, C, K]
  const float* reg;       // [B, R, H, W] fp32 NCHW
  const float* calib;     // [B, 6] f_u f_v c_u c_v b_x b_y
  const float* pad;       // [B, 2]
  const float* size;      // [B, 2] (W, H) of the padded image (ParamsList.size)
  const float* dim_mean;  // [C, 3]
  int B, C, K, R, H, W, S;
  float thresh;
  int down_ratio;
  // outputs
  float* scores;          // [B, K]
  long long* inds;        // [B, K]
  float* clses;           // [B, K]
  float* ys;              // [B, K]
  float* xs;              // [B, K]
  float* pois;            // [B, K, R]
  float* result;          // [B, K, 14]
  int* count;             // [B]
};

// channel map runs/monoflex.yaml:27-28: 2d_dim 0:4 | 3d_offset 4:6 | corner_offset 6:26 | corner_uncertainty 26:29 |
// 3d_dim 29:32 | ori_cls 32:40 | ori_offset 40:48 | depth 48 | depth_uncertainty 49
static constexpr int S2_THREADS = 1024;
static constexpr int S2_KEYS = 2048;

__global__ void __launch_bounds__(S2_THREADS) topk_decode_stage2_kernel(const DecodeParams p) {
  const int b = blockIdx.x;
  const int SK = p.S * p.K, CSK = p.C * SK;     // candidates per class / per image (<= 2048)
  __shared__ unsigned long long sel[S2_KEYS];
  __shared__ float s_poi[64 * 50];
  // key = score bits << 17 | (3 - class) << 15 | (32767 - pixel index): (score desc, class asc, index asc) is exactly the
  // order of the reference's two-stage top-k (per class, then over the concatenated [class][rank] list, utils.py:61-100)
  for (int i = threadIdx.x; i < S2_KEYS; i += S2_THREADS) {
    unsigned long long key = 0ull;
    if (i < CSK) {
      const int idx = p.s1_idx[static_cast<long long>(b) * CSK + i];
      if (idx >= 0) {
        const float sc = p.s1_score[static_cast<long long>(b) * CSK + i];
        const int c = i / SK;
        key = ((static_cast<unsigned long long>(__float_as_uint(sc)) << 17) | (static_cast<unsigned long long>(3 - c) << 15) |
               static_cast<unsigned long long>(32767 - idx)) + 1ull;
      }
    }
    sel[i] = key;
  }
  __syncthreads();
  // top-K of the C*S*K candidates by rank counting (unique keys; broadcast shared-memory reads, no barriers in the loops), in two
  // levels like the reference's two-stage top-k: (1) every candidate ranks itself among the S*K candidates of ITS class and the
  // K best of each class survive, (2) the C*K survivors rank themselves among each other. ~3x fewer comparisons than one flat
  // ranking; the 2048-key bitonic sort this replaces was 66 block-wide barrier steps.
  __shared__ unsigned long long cls_top[3 * 64];
  __shared__ unsigned long long top[64];
  for (int i = threadIdx.x; i < 3 * 64; i += S2_THREADS) cls_top[i] = 0ull;
  for (int i = threadIdx.x; i < 64; i += S2_THREADS) top[i] = 0ull;
  __syncthreads();
  for (int c = threadIdx.x; c < CSK; c += S2_THREADS) {
    const unsigned long long mine = sel[c];
    if (mine == 0ull) continue;
    const int cl = c / SK;
    const unsigned long long* grp = sel + cl * SK;
    int rank = 0;
    for (int j = 0; j < SK; ++j) rank += grp[j] > mine ? 1 : 0;
    if (rank < p.K) cls_top[cl * 64 + rank] = mine;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < p.C * 64; c += S2_THREADS) {
    const unsigned long long mine = cls_top[c];
    if (mine == 0ull) continue;
    int rank = 0;
    for (int j = 0; j < p.C * 64; ++j) rank += cls_top[j] > mine ? 1 : 0;
    if (rank < 64) top[rank] = mine;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 64; i += S2_THREADS) sel[i] = top[i];      // the code below reads the sorted prefix from sel[]
  __syncthreads();
  const int HW = p.H * p.W;
  // POI gather: K x R values straight from the NCHW map (no permute of the whole map: utils.py:120-145)
  for (int t = threadIdx.x; t < p.K * p.R; t += blockDim.x) {
    const int d = t / p.R, ch = t - d * p.R;
    const unsigned long long k = sel[d] - 1ull;
    const int idx = 32767 - static_cast<int>(k & 32767ull);
    const float v = __ldg(p.reg + (static_cast<long long>(b) * p.R + ch) * HW + idx);
    s_poi[d * p.R + ch] = v;
    p.pois[(static_cast<long long>(b) * p.K + d) * p.R + ch] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int n = 0;
    for (int d = 0; d < p.K; ++d) {
      const float sc = __uint_as_float(static_cast<unsigned int>((sel[d] - 1ull) >> 17));
      if (sc >= p.thresh) ++n;
    }
    p.count[b] = n;
  }
  const int d = threadIdx.x;
  if (d >= p.K) return;
  const unsigned long long k = sel[d] - 1ull;
  const float score = __uint_as_float(static_cast<unsigned int>(k >> 17));
  const int cls = 3 - static_cast<int>((k >> 15) & 3ull);
  const int idx = 32767 - static_cast<int>(k & 32767ull);
  const float yf = static_cast<float>(idx / p.W), xf = static_cast<float>(idx % p.W);
  const long long o = static_cast<long long>(b) * p.K + d;
  p.scores[o] = score; p.inds[o] = idx; p.clses[o] = static_cast<float>(cls); p.ys[o] = yf; p.xs[o] = xf;

  const float* q = s_poi + d * p.R;
  const float dr = static_cast<float>(p.down_ratio);
  const float padx = p.pad[b * 2], pady = p.pad[b * 2 + 1];
  const float f_u = p.calib[b * 6 + 0], f_v = p.calib[b * 6 + 1], c_u = p.calib[b * 6 + 2], c_v = p.calib[b * 6 + 3];
  const float b_x = p.calib[b * 6 + 4], b_y = p.calib[b * 6 + 5];
  // decode_box2d_fcos anno_encoder.py:69-86
  const float wmax = p.size[b * 2] - 1.f, hmax = p.size[b * 2 + 1] - 1.f;
  float x1 = (xf - fmaxf(q[0], 0.f)) * dr - padx, y1 = (yf - fmaxf(q[1], 0.f)) * dr - pady;
  float x2 = (xf + fmaxf(q[2], 0.f)) * dr - padx, y2 = (yf + fmaxf(q[3], 0.f)) * dr - pady;
  x1 = fminf(fmaxf(x1, 0.f), wmax); x2 = fminf(fmaxf(x2, 0.f), wmax);
  y1 = fminf(fmaxf(y1, 0.f), hmax); y2 = fminf(fmaxf(y2, 0.f), hmax);
  // decode_dimension :221-243 -> (l, h, w)
  const float dl = expf(q[29]) * p.dim_mean[cls * 3 + 0];
  const float dh = expf(q[30]) * p.dim_mean[cls * 3 + 1];
  const float dw = expf(q[31]) * p.dim_mean[cls * 3 + 2];
  // depths :124-140, :187-219
  float dep[4], sig[4];
  dep[0] = fminf(fmaxf(1.f / (1.f / (1.f + expf(-q[48]))) - 1.f, 0.1f), 100.f);
  sig[0] = expf(q[49]);
  const float* kp = q + 6;   // 10 x (x, y)
  const float ch_ = kp[8 * 2 + 1] - kp[9 * 2 + 1];
  dep[1] = f_u * dh / (fmaxf(ch_, 0.f) * dr + 1e-3f);
  const float a02 = f_u * dh / (fmaxf(kp[0 * 2 + 1] - kp[4 * 2 + 1], 0.f) * dr + 1e-3f);
  const float b02 = f_u * dh / (fmaxf(kp[2 * 2 + 1] - kp[6 * 2 + 1], 0.f) * dr + 1e-3f);
  dep[2] = (a02 + b02) / 2.f;
  const float a13 = f_u * dh / (fmaxf(kp[1 * 2 + 1] - kp[5 * 2 + 1], 0.f) * dr + 1e-3f);
  const float b13 = f_u * dh / (fmaxf(kp[3 * 2 + 1] - kp[7 * 2 + 1], 0.f) * dr + 1e-3f);
  dep[3] = (a13 + b13) / 2.f;
#pragma unroll
  for (int i = 1; i < 4; ++i) {
    dep[i] = fminf(fmaxf(dep[i], 0.1f), 100.f);
    sig[i] = expf(q[26 + i - 1]);
  }
  // soft ensemble detector_infer.py:176-198
  float wsum = 0.f, wts[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { wts[i] = 1.f / sig[i]; wsum += wts[i]; }
  float depth = 0.f, err = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float wn = wts[i] / wsum; depth += dep[i] * wn; err += wn * sig[i]; }
  // location :142-155 + kitti_utils.py:350-369
  const float u = (xf + q[4]) * dr - padx, v = (yf + q[5]) * dr - pady;
  const float lx = ((u - c_u) * depth) / f_u + b_x;
  float ly = ((v - c_v) * depth) / f_v + b_y;
  // multi-bin orientation :245-295: argmax over softmax(bin logits)[..., 1] (first max wins)
  int bi = 0; float best = -1.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float l0 = q[32 + 2 * i], l1 = q[32 + 2 * i + 1];
    const float mxl = fmaxf(l0, l1);
    const float e0 = expf(l0 - mxl), e1 = expf(l1 - mxl);
    const float pr = e1 / (e0 + e1);
    if (pr > best) { best = pr; bi = i; }
  }
  const float PI_F = 3.14159265358979323846f;
  const float centers[4] = {0.f, PI_F / 2.f, PI_F, -PI_F / 2.f};
  float alpha = atan2f(q[40 + 2 * bi], q[40 + 2 * bi + 1]) + centers[bi];
  const float ray = atan2f(lx, depth);
  float roty = alpha + ray;
  if (roty > PI_F) roty -= 2.f * PI_F;
  if (roty < -PI_F) roty += 2.f * PI_F;
  if (alpha > PI_F) alpha -= 2.f * PI_F;
  if (alpha < -PI_F) alpha += 2.f * PI_F;
  ly += dh / 2.f;
  const float conf = score * (1.f - fminf(fmaxf(err, 0.01f), 1.f));
  float* r = p.result + o * 14;
  r[0] = static_cast<float>(cls); r[1] = alpha; r[2] = x1; r[3] = y1; r[4] = x2; r[5] = y2;
  r[6] = dh; r[7] = dw; r[8] = dl; r[9] = lx; r[10] = ly; r[11] = depth; r[12] = roty; r[13] = conf;
}

int launch_decode(const float* heat, const float* reg, const float* calib, const float* pad, const float* size,
                  const float* dim_mean, int B, int C, int H, int W, int R, int K, float thresh, int apply_sigmoid,
                  float* s1_score, int* s1_idx, float* scores, long long* inds, float* clses, float* ys, float* xs,
                  float* pois, float* result, int* count, cudaStream_t st) {
  // slabs per (image, class) plane: more slabs = shorter per-CTA scans but more CTAs; one CTA of 1024 threads per SM, so a second
  // wave doubles the kernel (the fixed S = 8 of round 1 put 192 CTAs on 148 SMs at B = 8). Pick the S <= 8 that minimises
  // waves x (items per thread + the ~6 items' worth of radix-pass overhead).
  int S = 1, best = 1 << 30, nsm_dec = 148;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm_dec, cudaDevAttrMultiProcessorCount, dev);
    for (int s = 1; s <= MF_DECODE_SLABS; ++s) {
      if (C * s * K > S2_KEYS) break;
      const int waves = (B * C * s + nsm_dec - 1) / nsm_dec;
      const int items = ((H * W + s - 1) / s + S1_THREADS - 1) / S1_THREADS;
      const int cost = waves * (items + 6);
      if (cost < best) { best = cost; S = s; }
    }
  }
  if (H * W > 32768 || C > 3 || C * S * K > S2_KEYS || K > 64 || R != 50) {
    set_error("decode: unsupported shape H*W=%d C=%d K=%d R=%d", H * W, C, K, R);
    return -1;
  }
  const int n_items = ((H * W + S - 1) / S + S1_THREADS - 1) / S1_THREADS;
  // score bits of the slab's pixels + the staged slab with its one-row halo
  const int s1_smem = n_items * S1_THREADS * static_cast<int>(sizeof(unsigned int)) +
                      ((H * W + S - 1) / S + 2 * W + 2) * static_cast<int>(sizeof(float));
  static int s1_attr = 0;
  if (s1_smem > s1_attr) {
    if (check_cuda(cudaFuncSetAttribute(nms_topk_stage1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, s1_smem),
                   "stage1 smem attr"))
      return -1;
    s1_attr = s1_smem;
  }
  (void)launch_k(nms_topk_stage1_kernel, dim3(B * C * S), dim3(S1_THREADS), s1_smem, st, heat, H, W, K, apply_sigmoid, S, s1_score, s1_idx);
  if (check_cuda(cudaGetLastError(), "nms_topk_stage1")) return -1;
  DecodeParams p;
  p.s1_score = s1_score; p.s1_idx = s1_idx; p.reg = reg; p.calib = calib; p.pad = pad; p.size = size;
  p.dim_mean = dim_mean; p.B = B; p.C = C; p.K = K; p.R = R; p.H = H; p.W = W; p.S = S; p.thresh = thresh; p.down_ratio = 4;
  p.scores = scores; p.inds = inds; p.clses = clses; p.ys = ys; p.xs = xs; p.pois = pois; p.result = result;
  p.count = count;
  (void)launch_k(topk_decode_stage2_kernel, dim3(B), dim3(S2_THREADS), 0, st, p);
  return check_cuda(cudaGetLastError(), "topk_decode_stage2");
}

}  // namespace mf
