// Fused training loss (SURVEY §8 row R12): Loss_Computation.__call__ model/head/detector_loss.py:267-493 with
// prepare_predictions :116-265, Real_MultiBin_loss :495-517, IOULoss('giou') layers/iou_loss.py:12-49 and the Anno_Encoder
// decoders anno_encoder.py:88-295, for the runs/monoflex.yaml configuration (L1 regression, L1 depth + uncertainty, multi-bin
// orientation, soft_combine corner depth, 'log' truncation-offset loss, MODIFY_INVALID_KEYPOINT_DEPTH).
//
// The reference runs ~300 micro-kernels and 14+ .item() host syncs per step for O(objects) arithmetic. Here:
//   loss_forward_kernel  (1 CTA):   counts/normalisers -> per-object terms (one thread per object slot) -> deterministic
//                                   block reduction -> 11 losses + 12 logged metrics in one device buffer (no host sync);
//   loss_backward_kernel (1 thread per (object, regression channel)): the SAME templated per-object function evaluated on
//                                   forward-mode dual numbers seeded on that channel -> d(sum_k g_k loss_k)/d reg at the
//                                   object's centre pixel, atomically added into grad_reg (objects may share a pixel).
// Writing the gradient as a dual-number instantiation of the forward code keeps the two in lock-step: every clamp / relu /
// abs / detach carries torch's sub-gradient convention in one place (the Dual overloads below).
//
// The heat-map term is the focal-loss pair of mf_train.cu / mf_elementwise.cu; this file only scales it.
#include "mf_common.cuh"
#include "mf_launch.h"

namespace mf {

// ------------------------------------------------------------------------------------------------ dual numbers
struct Dual {
  float v, d;
};
__device__ __forceinline__ Dual mk(float v, float d = 0.f) { Dual r; r.v = v; r.d = d; return r; }
__device__ __forceinline__ Dual operator+(Dual a, Dual b) { return mk(a.v + b.v, a.d + b.d); }
__device__ __forceinline__ Dual operator-(Dual a, Dual b) { return mk(a.v - b.v, a.d - b.d); }
__device__ __forceinline__ Dual operator*(Dual a, Dual b) { return mk(a.v * b.v, a.d * b.v + a.v * b.d); }
__device__ __forceinline__ Dual operator/(Dual a, Dual b) {
  const float q = a.v / b.v;
  return mk(q, (a.d - q * b.d) / b.v);
}
__device__ __forceinline__ Dual operator+(Dual a, float b) { return mk(a.v + b, a.d); }
__device__ __forceinline__ Dual operator+(float a, Dual b) { return mk(a + b.v, b.d); }
__device__ __forceinline__ Dual operator-(Dual a, float b) { return mk(a.v - b, a.d); }
__device__ __forceinline__ Dual operator-(float a, Dual b) { return mk(a - b.v, -b.d); }
__device__ __forceinline__ Dual operator*(Dual a, float b) { return mk(a.v * b, a.d * b); }
__device__ __forceinline__ Dual operator*(float a, Dual b) { return mk(a * b.v, a * b.d); }
__device__ __forceinline__ Dual operator/(Dual a, float b) { return mk(a.v / b, a.d / b); }
__device__ __forceinline__ Dual operator/(float a, Dual b) {
  const float q = a / b.v;
  return mk(q, -q * b.d / b.v);
}
__device__ __forceinline__ Dual operator-(Dual a) { return mk(-a.v, -a.d); }

// elementary functions for both scalar types; sub-gradients follow torch.autograd (abs'(0) = 0, relu'(0) = 0,
// clamp passes the gradient on the closed interval, min/max send it to the selected operand)
__device__ __forceinline__ float val(float x) { return x; }
__device__ __forceinline__ float val(Dual x) { return x.v; }
__device__ __forceinline__ float detach(float x) { return x; }
__device__ __forceinline__ Dual detach(Dual x) { return mk(x.v, 0.f); }
__device__ __forceinline__ float f_exp(float x) { return expf(x); }
__device__ __forceinline__ Dual f_exp(Dual x) { const float e = expf(x.v); return mk(e, e * x.d); }
__device__ __forceinline__ float f_log(float x) { return logf(x); }
__device__ __forceinline__ Dual f_log(Dual x) { return mk(logf(x.v), x.d / x.v); }
__device__ __forceinline__ float f_sqrt(float x) { return sqrtf(x); }
__device__ __forceinline__ Dual f_sqrt(Dual x) { const float s = sqrtf(x.v); return mk(s, x.d / (2.f * s)); }
__device__ __forceinline__ float f_abs(float x) { return fabsf(x); }
__device__ __forceinline__ Dual f_abs(Dual x) { return mk(fabsf(x.v), x.v > 0.f ? x.d : (x.v < 0.f ? -x.d : 0.f)); }
__device__ __forceinline__ float f_relu(float x) { return x > 0.f ? x : 0.f; }
__device__ __forceinline__ Dual f_relu(Dual x) { return x.v > 0.f ? x : mk(0.f, 0.f); }
__device__ __forceinline__ float f_clamp(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }
__device__ __forceinline__ Dual f_clamp(Dual x, float lo, float hi) {
  return mk(fminf(fmaxf(x.v, lo), hi), (x.v >= lo && x.v <= hi) ? x.d : 0.f);
}
__device__ __forceinline__ float f_min(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ Dual f_min(Dual a, float b) { return a.v < b ? a : (a.v == b ? mk(b, 0.5f * a.d) : mk(b, 0.f)); }
__device__ __forceinline__ float f_max(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ Dual f_max(Dual a, float b) { return a.v > b ? a : (a.v == b ? mk(b, 0.5f * a.d) : mk(b, 0.f)); }
__device__ __forceinline__ float f_atan2(float y, float x) { return atan2f(y, x); }
__device__ __forceinline__ Dual f_atan2(Dual y, Dual x) {
  return mk(atan2f(y.v, x.v), (x.v * y.d - y.v * x.d) / (x.v * x.v + y.v * y.v));
}
__device__ __forceinline__ float f_sin(float x) { return sinf(x); }
__device__ __forceinline__ Dual f_sin(Dual x) { return mk(sinf(x.v), cosf(x.v) * x.d); }
__device__ __forceinline__ float f_cos(float x) { return cosf(x); }
__device__ __forceinline__ Dual f_cos(Dual x) { return mk(cosf(x.v), -sinf(x.v) * x.d); }
template <class T> __device__ __forceinline__ T cst(float x);
template <> __device__ __forceinline__ float cst<float>(float x) { return x; }
template <> __device__ __forceinline__ Dual cst<Dual>(float x) { return mk(x, 0.f); }

// ------------------------------------------------------------------------------------------------ layouts
// object table row (MF_LOSS_OBJ_COLS floats), one per (image, slot): packed by the host from the ParamsList fields
enum {
  O_CLS = 0, O_CX = 1, O_CY = 2, O_BOX = 3, O_REG = 7, O_TRUNC = 8, O_DIMS = 9, O_LOC = 12, O_ROTY = 15, O_OFF = 16,
  O_ORI = 18, O_KDM = 26, O_KP = 29 /* 10 x (x, y, visible) */
};
// internal terms (each = coef * sum over objects of a per-object value)
enum { T_BBOX = 0, T_DEPTH, T_OFF, T_TRUNC, T_ORI_CLS, T_ORI_REG, T_DIMS, T_CORNER, T_KP, T_KD_VALID, T_KD_INVALID, T_WAD, NTERM };
// loss index (LOSS_NAMES order of runs/monoflex.yaml:45) each internal term belongs to
__constant__ int kTermLoss[NTERM] = {1, 2, 3, 9, 4, 4, 5, 6, 7, 8, 8, 10};
enum { L_IOU = 0, L_DEPTH_L1, L_KD_VALID_L1, L_DEPTH_MAE, L_MAE_C, L_MAE_02, L_MAE_13, L_LOWER, L_HARD, L_SOFT, L_MEAN, NLOG };

struct LossCfg {
  float w[11];            // INIT_LOSS_WEIGHT in LOSS_NAMES order
  float dim_mean[9];      // DIMENSION_MEAN [cls][l,h,w]
  float unc_lo, unc_hi;   // UNCERTAINTY_RANGE
  float depth_lo, depth_hi;
  float down_ratio;
  int B, M, H, W, C;      // C = 50 regression channels
};

// ------------------------------------------------------------------------------------------------ per-object terms
// p: the 50 regression values at the object's centre; o: its target row; im: [f_u f_v c_u c_v b_x b_y pad_x pad_y] of ITS
// image; fu_kp: f_u used by decode_depth_from_keypoints_batch (anno_encoder.py:186 indexes calibs by rank, see below).
template <class T>
__device__ void object_terms(const T* p, const float* __restrict__ o, const float* __restrict__ im, float fu_kp,
                             const LossCfg& c, T* term, float* logs) {
  const float cx = o[O_CX], cy = o[O_CY];
  const float td = o[O_LOC + 2];
#pragma unroll
  for (int k = 0; k < NTERM; ++k) term[k] = cst<T>(0.f);
  // ---- 2D box: FCOS distances + GIoU (detector_loss.py:132-139, 158; iou_loss.py:12-49)
  const float bw = o[O_BOX + 2] - o[O_BOX], bh = o[O_BOX + 3] - o[O_BOX + 1];
  if (bh > 0.f && bw > 0.f) {
    const float tl = cx - o[O_BOX], tt = cy - o[O_BOX + 1], tr = o[O_BOX + 2] - cx, tb = o[O_BOX + 3] - cy;
    const T pl = f_relu(p[0]), pt = f_relu(p[1]), pr = f_relu(p[2]), pb = f_relu(p[3]);
    const float t_area = (tl + tr) * (tt + tb);
    const T p_area = (pl + pr) * (pt + pb);
    const T w_i = f_min(pl, tl) + f_min(pr, tr), g_w = f_max(pl, tl) + f_max(pr, tr);
    const T h_i = f_min(pb, tb) + f_min(pt, tt), g_h = f_max(pb, tb) + f_max(pt, tt);
    const T ac = g_w * g_h + 1e-7f;
    const T inter = w_i * h_i;
    const T uni = t_area + p_area - inter;
    const T iou = (inter + 1.0f) / (uni + 1.0f);
    term[T_BBOX] = 1.f - (iou - (ac - uni) / ac);
    if (logs) logs[L_IOU] = val(iou);
  }
  // ---- dimensions (decode_dimension anno_encoder.py:208-230: exp(offset) * class mean)
  const int cls = static_cast<int>(o[O_CLS]);
  T dims[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    dims[k] = f_exp(p[29 + k]) * c.dim_mean[cls * 3 + k];
    term[T_DIMS] = term[T_DIMS] + f_abs(dims[k] - o[O_DIMS + k]);          // DIMENSION_WEIGHT [1,1,1]
  }
  // ---- direct depth (decode_depth inv_sigmoid: 1/sigmoid(x) - 1 = exp(-x)) + uncertainty
  const T sig = 1.f / (1.f + f_exp(-p[48]));
  const T pd = f_clamp(1.f / sig - 1.f, c.depth_lo, c.depth_hi);
  const T du = f_clamp(p[49], c.unc_lo, c.unc_hi);
  const T d_l1 = f_abs(pd - td);
  term[T_DEPTH] = d_l1 * f_exp(-du) + du;                                  // x w_depth in coef (both summands carry it)
  // ---- 3D-centre offset: L1, 'log' variant for truncated objects (:305-320)
  const T ol = f_abs(p[4] - o[O_OFF]) + f_abs(p[5] - o[O_OFF + 1]);
  if (o[O_TRUNC] != 0.f) term[T_TRUNC] = f_log(1.f + ol);
  else term[T_OFF] = ol;
  // ---- multi-bin orientation (Real_MultiBin_loss :495-517); vector = [ori_cls 32:40 | ori_offset 40:48]
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const T a = p[32 + 2 * i], b = p[33 + 2 * i];
    const float m = fmaxf(val(a), val(b));
    const T lse = f_log(f_exp(a - m) + f_exp(b - m)) + m;
    const bool on = o[O_ORI + i] == 1.f;
    term[T_ORI_CLS] = term[T_ORI_CLS] + (lse - (on ? b : a));
    if (on) {
      const T x0 = p[40 + 2 * i], x1 = p[41 + 2 * i];
      const T nrm = f_sqrt(x0 * x0 + x1 * x1);
      const T den = val(nrm) > 1e-12f ? nrm : cst<T>(1e-12f);              // F.normalize eps
      const float ang = o[O_ORI + 4 + i];
      term[T_ORI_REG] = term[T_ORI_REG] + f_abs(x0 / den - sinf(ang)) + f_abs(x1 / den - cosf(ang));
    }
  }
  // ---- key points (:343-347) and the three key-point depths (decode_depth_from_keypoints_batch anno_encoder.py:174-206)
#pragma unroll
  for (int k = 0; k < 10; ++k)
    term[T_KP] = term[T_KP] + (f_abs(p[6 + 2 * k] - o[O_KP + 3 * k]) + f_abs(p[7 + 2 * k] - o[O_KP + 3 * k + 1])) * o[O_KP + 3 * k + 2];
  auto ky = [&](int k) { return p[7 + 2 * k]; };
  const T fh = fu_kp * dims[1];
  const float dr = c.down_ratio;
  T kd[3];
  kd[0] = fh / (f_relu(ky(8) - ky(9)) * dr + 1e-3f);
  kd[1] = (fh / (f_relu(ky(0) - ky(4)) * dr + 1e-3f) + fh / (f_relu(ky(2) - ky(6)) * dr + 1e-3f)) * 0.5f;
  kd[2] = (fh / (f_relu(ky(1) - ky(5)) * dr + 1e-3f) + fh / (f_relu(ky(3) - ky(7)) * dr + 1e-3f)) * 0.5f;
  T ku[3];
  float kmae[3];
#pragma unroll
  for (int g = 0; g < 3; ++g) {
    kd[g] = f_clamp(kd[g], c.depth_lo, c.depth_hi);
    ku[g] = f_clamp(p[26 + g], c.unc_lo, c.unc_hi);
    kmae[g] = fabsf(val(kd[g]) - td) / td;
    if (o[O_KDM + g] != 0.f) {                                             // valid group: loss * exp(-u) + u  (:349-377)
      const T l = f_abs(kd[g] - td);
      term[T_KD_VALID] = term[T_KD_VALID] + l * f_exp(-ku[g]) + ku[g];
      if (logs) logs[L_KD_VALID_L1] += val(l);
    } else {                                                               // invalid: depth detached, only u is trained
      term[T_KD_INVALID] = term[T_KD_INVALID] + f_abs(detach(kd[g]) - td) * f_exp(-ku[g]);
    }
  }
  // ---- soft combination of the four depths by 1/sigma (:241-248) -> weighted_avg_depth_loss (:419-421)
  const T iu0 = 1.f / f_exp(du), iu1 = 1.f / f_exp(ku[0]), iu2 = 1.f / f_exp(ku[1]), iu3 = 1.f / f_exp(ku[2]);
  const T isum = iu0 + iu1 + iu2 + iu3;
  const T soft = pd * (iu0 / isum) + kd[0] * (iu1 / isum) + kd[1] * (iu2 / isum) + kd[2] * (iu3 / isum);
  term[T_WAD] = f_abs(soft - td);
  // ---- 3D corners: predicted location / yaw / dims vs the label's (decode_location_flatten :142-155,
  //      decode_axes_orientation :245-295, encode_box3d :88-122)
  const float f_u = im[0], f_v = im[1], c_u = im[2], c_v = im[3], b_x = im[4], b_y = im[5], pad_x = im[6], pad_y = im[7];
  const T u = (cx + p[4]) * dr - pad_x, v = (cy + p[5]) * dr - pad_y;
  const T lx = ((u - c_u) * soft) / f_u + b_x, ly = ((v - c_v) * soft) / f_v + b_y, lz = soft;
  int best = 0;
  float bestp = -1.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {                                            // softmax(...)[..., 1], first arg-max
    const float a = val(p[32 + 2 * i]), b = val(p[33 + 2 * i]), m = fmaxf(a, b);
    const float ea = expf(a - m), eb = expf(b - m), pr1 = eb / (ea + eb);
    if (pr1 > bestp) { bestp = pr1; best = i; }
  }
  const float PI_F = 3.14159265358979323846f;
  const float centers[4] = {0.f, PI_F / 2, PI_F, -PI_F / 2};
  T roty = f_atan2(p[40 + 2 * best], p[41 + 2 * best]) + centers[best] + f_atan2(lx, lz);
  if (val(roty) > PI_F) roty = roty - 2.f * PI_F;
  if (val(roty) < -PI_F) roty = roty + 2.f * PI_F;
  // label box: location re-derived from the label's centre offset and depth (:147-148), not `locations` itself
  const float tu = (cx + o[O_OFF]) * dr - pad_x, tv = (cy + o[O_OFF + 1]) * dr - pad_y;
  const float tlx = ((tu - c_u) * td) / f_u + b_x, tly = ((tv - c_v) * td) / f_v + b_y;
  const float tcs = cosf(o[O_ROTY]), tsn = sinf(o[O_ROTY]);
  const T pcs = f_cos(roty), psn = f_sin(roty);
  const float sx[8] = {-1, -1, 1, 1, -1, -1, 1, 1}, sy[8] = {1, 1, 1, 1, -1, -1, -1, -1}, sz[8] = {-1, 1, 1, -1, -1, 1, 1, -1};
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const T X = dims[0] * (0.5f * sx[k]), Y = dims[1] * (0.5f * sy[k]), Z = dims[2] * (0.5f * sz[k]);
    const float tX = o[O_DIMS] * 0.5f * sx[k], tY = o[O_DIMS + 1] * 0.5f * sy[k], tZ = o[O_DIMS + 2] * 0.5f * sz[k];
    term[T_CORNER] = term[T_CORNER] + f_abs((pcs * X + psn * Z + lx) - (tcs * tX + tsn * tZ + tlx)) +
                     f_abs((Y + ly) - (tY + tly)) + f_abs((-psn * X + pcs * Z + lz) - (-tsn * tX + tcs * tZ + td));
  }
  if (logs) {                                                              // logged metrics (:296, :379-417)
    const float dmae = fabsf(val(pd) - td) / td;
    logs[L_DEPTH_L1] = val(d_l1);
    logs[L_DEPTH_MAE] = dmae;
    logs[L_MAE_C] = kmae[0]; logs[L_MAE_02] = kmae[1]; logs[L_MAE_13] = kmae[2];
    const float mae[4] = {dmae, kmae[0], kmae[1], kmae[2]};
    const float unc[4] = {expf(val(du)), expf(val(ku[0])), expf(val(ku[1])), expf(val(ku[2]))};
    float lo = mae[0];
    int am = 0;
#pragma unroll
    for (int k = 1; k < 4; ++k) { lo = fminf(lo, mae[k]); if (unc[k] < unc[am]) am = k; }
    logs[L_LOWER] = lo;
    logs[L_HARD] = mae[am];
    logs[L_SOFT] = fabsf(val(soft) - td) / td;
    logs[L_MEAN] = fabsf((val(pd) + val(kd[0]) + val(kd[1]) + val(kd[2])) * 0.25f - td) / td;
  }
}

// ------------------------------------------------------------------------------------------------ kernels
// ws layout (floats): [0..NTERM) coef (weight / normaliser) per internal term, [16] hm scale = w_hm / clamp(num_pos, 1),
// [17] hm scale * upstream grad (written by backward), [24..24+B) f_u used for the key-point depths of image b
#define WS_COEF 0
#define WS_HM 16
#define WS_HMG 17
#define WS_FUKP 24

template <int N>
__device__ void block_sum(float (&v)[N], float* sm /* [32*N] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int k = 0; k < N; ++k) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], d);
    if (lane == 0) sm[warp * N + k] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < N) {                                                   // fixed summation order: deterministic
    float s = 0.f;
    for (int w = 0; w < nw; ++w) s += sm[w * N + threadIdx.x];
    sm[threadIdx.x] = s;                                                   // nw*N >= N: slot 0..N-1 of warp 0 reused after sync below
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < N; ++k) v[k] = sm[k];
  __syncthreads();
}

__global__ void __launch_bounds__(256) loss_forward_kernel(const float* __restrict__ reg, const float* __restrict__ obj,
                                                           const float* __restrict__ img, const float* __restrict__ focal2,
                                                           LossCfg c, float* __restrict__ out, float* __restrict__ ws) {
  __shared__ float sm[32 * (NTERM + NLOG)];
  __shared__ float s_coef[NTERM];
  __shared__ float s_fukp[64];
  const int slots = c.B * c.M;
  // ---- phase 0: counts (they depend on the labels only)
  float cnt[7] = {0, 0, 0, 0, 0, 0, 0};                                    // n3, n2d, ntrunc, nkp, nkd_valid, ori_reg_cnt, -
  for (int s = threadIdx.x; s < slots; s += blockDim.x) {
    const float* o = obj + static_cast<long long>(s) * MF_LOSS_OBJ_COLS;
    if (o[O_REG] == 0.f) continue;
    cnt[0] += 1.f;
    if (o[O_BOX + 3] - o[O_BOX + 1] > 0.f && o[O_BOX + 2] - o[O_BOX] > 0.f) cnt[1] += 1.f;
    if (o[O_TRUNC] != 0.f) cnt[2] += 1.f;
    for (int k = 0; k < 10; ++k) cnt[3] += o[O_KP + 3 * k + 2];
    for (int g = 0; g < 3; ++g) cnt[4] += (o[O_KDM + g] != 0.f) ? 1.f : 0.f;
    for (int i = 0; i < 4; ++i) cnt[5] += (o[O_ORI + i] == 1.f) ? 1.f : 0.f;
  }
  block_sum<7>(cnt, sm);
  const float n3 = cnt[0], n2d = cnt[1], ntr = cnt[2], nkp = cnt[3], nkv = cnt[4], nor = cnt[5];
  if (threadIdx.x == 0) {
    const float* w = c.w;
    s_coef[T_BBOX] = n2d > 0.f ? w[1] / n2d : 0.f;                         // reference: NameError when no 2D box -> 0 here
    s_coef[T_DEPTH] = w[2] / n3;
    s_coef[T_OFF] = w[3] / (n3 - ntr);                                     // mean over an empty set is nan in the reference too
    s_coef[T_TRUNC] = w[9] / fmaxf(ntr, 1.f);
    s_coef[T_ORI_CLS] = w[4] / (4.f * n3);
    s_coef[T_ORI_REG] = nor > 0.f ? w[4] / nor : 0.f;
    s_coef[T_DIMS] = w[5] / n3;
    s_coef[T_CORNER] = w[6] / (8.f * n3);                                  // .sum(dim=2).mean() over [N, 8]
    s_coef[T_KP] = w[7] / fmaxf(nkp, 1.f);
    s_coef[T_KD_VALID] = w[8] / fmaxf(nkv, 1.f);
    s_coef[T_KD_INVALID] = w[8] / fmaxf(3.f * n3 - nkv, 1.f);
    s_coef[T_WAD] = w[10] / n3;
    if (n3 == 0.f)                                                         // no object in the whole batch (reference crashes)
      for (int k = 0; k < NTERM; ++k) s_coef[k] = 0.f;
    // anno_encoder.py:186: `calib = calibs[idx]` with idx = rank of the image among the images that own objects
    int rank = 0;
    for (int b = 0; b < c.B && b < 64; ++b) {
      bool any = false;
      for (int m = 0; m < c.M; ++m) any |= obj[(static_cast<long long>(b) * c.M + m) * MF_LOSS_OBJ_COLS + O_REG] != 0.f;
      s_fukp[b] = img[(c.B == 1 ? 0 : rank) * 8];
      if (any) ++rank;
    }
    for (int k = 0; k < NTERM; ++k) ws[WS_COEF + k] = s_coef[k];
    for (int b = 0; b < c.B && b < 64; ++b) ws[WS_FUKP + b] = s_fukp[b];
    ws[WS_HM] = c.w[0] / fmaxf(focal2[1], 1.f);
  }
  __syncthreads();
  // ---- phase 1: per-object terms
  float acc[NTERM + NLOG];
#pragma unroll
  for (int k = 0; k < NTERM + NLOG; ++k) acc[k] = 0.f;
  const long long HW = static_cast<long long>(c.H) * c.W;
  for (int s = threadIdx.x; s < slots; s += blockDim.x) {
    const float* o = obj + static_cast<long long>(s) * MF_LOSS_OBJ_COLS;
    if (o[O_REG] == 0.f) continue;
    const int b = s / c.M;
    const long long pix = static_cast<long long>(o[O_CY]) * c.W + static_cast<long long>(o[O_CX]);
    float p[50];
    for (int ch = 0; ch < 50; ++ch) p[ch] = __ldg(reg + (static_cast<long long>(b) * c.C + ch) * HW + pix);
    float term[NTERM], logs[NLOG];
    for (int k = 0; k < NLOG; ++k) logs[k] = 0.f;
    object_terms<float>(p, o, img + b * 8, s_fukp[b], c, term, logs);
#pragma unroll
    for (int k = 0; k < NTERM; ++k) acc[k] += term[k];
#pragma unroll
    for (int k = 0; k < NLOG; ++k) acc[NTERM + k] += logs[k];
  }
  block_sum<NTERM + NLOG>(acc, sm);
  if (threadIdx.x == 0) {
    float L[11];
    for (int k = 0; k < 11; ++k) L[k] = 0.f;
    L[0] = focal2[0] * ws[WS_HM];
    for (int k = 0; k < NTERM; ++k) L[kTermLoss[k]] += s_coef[k] * acc[k];
    for (int k = 0; k < 11; ++k) out[k] = L[k];
    const float* lg = acc + NTERM;
    const float i3 = n3 > 0.f ? 1.f / n3 : 0.f;
    out[16 + 0] = n2d > 0.f ? lg[L_IOU] / n2d : 0.f;                       // 2D_IoU
    out[16 + 1] = c.w[2] * lg[L_DEPTH_L1] * i3;                            // log depth_loss (without uncertainty)
    out[16 + 2] = nkv > 0.f ? c.w[8] * lg[L_KD_VALID_L1] / nkv : nanf(""); // log keypoint_depth_loss (mean over valid)
    out[16 + 3] = lg[L_DEPTH_MAE] * i3;
    out[16 + 4] = lg[L_MAE_C] * i3; out[16 + 5] = lg[L_MAE_02] * i3; out[16 + 6] = lg[L_MAE_13] * i3;
    out[16 + 7] = lg[L_LOWER] * i3; out[16 + 8] = lg[L_HARD] * i3; out[16 + 9] = lg[L_SOFT] * i3; out[16 + 10] = lg[L_MEAN] * i3;
    out[32] = n3; out[33] = n2d; out[34] = ntr; out[35] = nkp; out[36] = nkv; out[37] = nor; out[38] = focal2[1];
  }
}

// one thread per (object slot, regression channel): d/d reg[ch] of sum_k gw[k] * loss_k restricted to this object
__global__ void __launch_bounds__(128) loss_backward_kernel(const float* __restrict__ reg, const float* __restrict__ obj,
                                                            const float* __restrict__ img, const float* __restrict__ ws,
                                                            const float* __restrict__ gw, LossCfg c,
                                                            float* __restrict__ grad_reg) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int slots = c.B * c.M;
  if (t >= slots * 50) return;
  const int s = t / 50, ch = t - s * 50;
  const float* o = obj + static_cast<long long>(s) * MF_LOSS_OBJ_COLS;
  if (o[O_REG] == 0.f) return;
  const int b = s / c.M;
  const long long HW = static_cast<long long>(c.H) * c.W;
  const long long pix = static_cast<long long>(o[O_CY]) * c.W + static_cast<long long>(o[O_CX]);
  Dual p[50];
  for (int k = 0; k < 50; ++k) p[k] = mk(__ldg(reg + (static_cast<long long>(b) * c.C + k) * HW + pix), k == ch ? 1.f : 0.f);
  Dual term[NTERM];
  object_terms<Dual>(p, o, img + b * 8, ws[WS_FUKP + b], c, term, nullptr);
  float g = 0.f;
#pragma unroll
  for (int k = 0; k < NTERM; ++k) {
    const float coef = ws[WS_COEF + k] * __ldg(gw + kTermLoss[k]);
    if (coef != 0.f && term[k].d != 0.f) g += coef * term[k].d;           // (skips 0 * inf of an empty normaliser)
  }
  if (g != 0.f) atomicAdd(grad_reg + (static_cast<long long>(b) * c.C + ch) * HW + pix, g);
}

__global__ void loss_hm_scale_kernel(float* ws, const float* gw) { ws[WS_HMG] = ws[WS_HM] * gw[0]; }

// ------------------------------------------------------------------------------------------------ launchers
static int fill_cfg(LossCfg& c, const float* weights11, const float* dim_mean9, int B, int M, int H, int W, int C) {
  if (C != 50) { set_error("loss: the regression map must have the 50 channels of runs/monoflex.yaml:27-28 (got %d)", C); return -1; }
  if (B < 1 || B > 64 || M < 1) { set_error("loss: batch %d (1..64) / max objects %d not supported", B, M); return -1; }
  for (int k = 0; k < 11; ++k) c.w[k] = weights11[k];
  for (int k = 0; k < 9; ++k) c.dim_mean[k] = dim_mean9[k];
  c.unc_lo = -10.f; c.unc_hi = 10.f;                                       // config/defaults.py:162
  c.depth_lo = 0.1f; c.depth_hi = 100.f;                                   // config/defaults.py:175
  c.down_ratio = 4.f;
  c.B = B; c.M = M; c.H = H; c.W = W; c.C = C;
  return 0;
}

int launch_loss_forward(const float* pred_cls, const float* hm, const float* pred_reg, const float* obj, const float* img,
                        const float* weights11, const float* dim_mean9, int B, int ncls, int M, int H, int W, int C,
                        float* out48, float* ws64, cudaStream_t st) {
  LossCfg c;
  if (fill_cfg(c, weights11, dim_mean9, B, M, H, W, C)) return -1;
  float* focal2 = ws64 + 20;                                               // [20] loss sum, [21] num_pos
  if (launch_focal_loss(pred_cls, hm, static_cast<long long>(B) * ncls * H * W, focal2, st)) return -1;
  (void)launch_k(loss_forward_kernel, dim3(1), dim3(256), 0, st, pred_reg, obj, img, static_cast<const float*>(focal2), c,
                 out48, ws64);
  return check_cuda(cudaGetLastError(), "loss_forward");
}

int launch_loss_backward(const float* pred_cls, const float* hm, const float* pred_reg, const float* obj, const float* img,
                         const float* weights11, const float* dim_mean9, int B, int ncls, int M, int H, int W, int C,
                         const float* ws64, const float* grad_losses11, float* grad_cls, float* grad_reg, cudaStream_t st) {
  LossCfg c;
  if (fill_cfg(c, weights11, dim_mean9, B, M, H, W, C)) return -1;
  const long long n_reg = static_cast<long long>(B) * C * H * W, n_cls = static_cast<long long>(B) * ncls * H * W;
  if (grad_reg) {
    if (check_cuda(cudaMemsetAsync(grad_reg, 0, n_reg * sizeof(float), st), "loss_backward memset")) return -1;
    const int threads = B * M * 50;
    (void)launch_k(loss_backward_kernel, dim3((threads + 127) / 128), dim3(128), 0, st, pred_reg, obj, img, ws64,
                   grad_losses11, c, grad_reg);
    if (check_cuda(cudaGetLastError(), "loss_backward")) return -1;
  }
  if (grad_cls) {
    float* wsm = const_cast<float*>(ws64);
    (void)launch_k(loss_hm_scale_kernel, dim3(1), dim3(1), 0, st, wsm, grad_losses11);
    if (launch_focal_loss_backward(pred_cls, hm, n_cls, ws64 + WS_HMG, grad_cls, st)) return -1;
  }
  return 0;
}

}  // namespace mf
