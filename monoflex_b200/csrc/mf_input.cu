// GPU input pipeline (SURVEY §8f N4): what KITTIDataset.__getitem__ + the transforms do on the host per image
// (data/datasets/kitti.py:218-228 pad_image, data/transforms/transforms.py:14-30 ToTensor + Normalize) and the heat-map half of
// the target encoding (model/heatmap_coder.py:83-124 draw_umich_gaussian / draw_umich_gaussian_2D), as two HBM-bound kernels.
//
//   preprocess_u8_kernel : uint8 HWC images of individual sizes (<= HxW) -> centred zero padding (pad = (H - h) / 2, (W - w) / 2,
//                          padding is done on the uint8 image, i.e. padded pixels become (0 - mean) / std) -> x / 255 ->
//                          (x - mean) / std with IEEE divisions (bit-identical to torch's fp32 ops) -> optional horizontal flip
//                          of the un-padded image (training augmentation) -> optional RGB->BGR -> fp32 NCHW [B,3,H,W],
//                          the detector's input boundary. 3 B read + 12 B written per pixel.
//   draw_heatmap_kernel  : per (image, class) plane the element-wise maximum of the objects' Gaussians, window |dx| <= rx,
//                          |dy| <= ry, sigma = (2 r + 1) / 6 per axis, evaluated in double and rounded to fp32 like numpy's
//                          float64 -> float32 store. One thread per heat-map element, <= 40 objects per image.
#include "mf_common.cuh"
#include "mf_launch.h"

namespace mf {

struct NormConsts { float mean[3], stdv[3]; int to_bgr; };

// hw: int32 [B][4] = (h, w, pad_x, pad_y); flip: int32 [B] (nullable)
__global__ void __launch_bounds__(256) preprocess_u8_kernel(const unsigned char* const* __restrict__ src,
                                                            const int* __restrict__ hw, const int* __restrict__ flip, int B,
                                                            int H, int W, NormConsts k, float* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long HW = static_cast<long long>(H) * W;
  if (i >= B * HW) return;
  const int b = static_cast<int>(i / HW);
  const int pix = static_cast<int>(i - b * HW);
  const int y = pix / W, x = pix - y * W;
  const int h = hw[4 * b], w = hw[4 * b + 1], px = hw[4 * b + 2], py = hw[4 * b + 3];
  const int sy = y - py;
  int sx = x - px;
  float v[3] = {0.f, 0.f, 0.f};
  if (sy >= 0 && sy < h && sx >= 0 && sx < w) {
    if (flip != nullptr && flip[b]) sx = w - 1 - sx;
    const unsigned char* p = src[b] + (static_cast<long long>(sy) * w + sx) * 3;
    v[0] = static_cast<float>(p[0]); v[1] = static_cast<float>(p[1]); v[2] = static_cast<float>(p[2]);
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float t = __fdiv_rn(__fsub_rn(__fdiv_rn(v[c], 255.f), k.mean[c]), k.stdv[c]);   // to_tensor, then normalize
    const int oc = k.to_bgr ? 2 - c : c;
    out[(static_cast<long long>(b) * 3 + oc) * HW + pix] = t;
  }
}
int launch_preprocess_u8(const unsigned char* const* src, const int* hw, const int* flip, int B, int H, int W,
                         const float* mean3, const float* std3, int to_bgr, float* out, cudaStream_t st) {
  NormConsts k;
  for (int c = 0; c < 3; ++c) { k.mean[c] = mean3[c]; k.stdv[c] = std3[c]; }
  k.to_bgr = to_bgr;
  const long long n = static_cast<long long>(B) * H * W;
  (void)launch_k(preprocess_u8_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, src, hw, flip, B, H, W, k, out);
  return check_cuda(cudaGetLastError(), "preprocess_u8");
}

// obj: int32 [B][max_objs][6] = (valid, cls, cx, cy, rx, ry); hm: fp32 [B][ncls][H][W]
__global__ void __launch_bounds__(256) draw_heatmap_kernel(const int* __restrict__ obj, int B, int max_objs, int ncls, int H,
                                                           int W, float* __restrict__ hm) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long plane = static_cast<long long>(H) * W;
  if (i >= B * ncls * plane) return;
  const int b = static_cast<int>(i / (ncls * plane));
  const long long r = i - static_cast<long long>(b) * ncls * plane;
  const int cls = static_cast<int>(r / plane);
  const int pix = static_cast<int>(r - cls * plane);
  const int y = pix / W, x = pix - y * W;
  float best = 0.f;
  const int* ob = obj + static_cast<long long>(b) * max_objs * 6;
  for (int j = 0; j < max_objs; ++j) {
    const int* o = ob + 6 * j;
    if (__ldg(o) == 0 || __ldg(o + 1) != cls) continue;
    const int dx = x - __ldg(o + 2), dy = y - __ldg(o + 3), rx = __ldg(o + 4), ry = __ldg(o + 5);
    if (dx < -rx || dx > rx || dy < -ry || dy > ry) continue;
    const double sx = (2 * rx + 1) / 6.0, sy = (2 * ry + 1) / 6.0;
    double g;
    if (rx == ry) g = exp(-static_cast<double>(dx * dx + dy * dy) / (2.0 * sx * sx));                      // gaussian2D :56-64
    else g = exp(-static_cast<double>(dx * dx) / (2.0 * sx * sx) - static_cast<double>(dy * dy) / (2.0 * sy * sy));  // ellip_gaussian2D :126-134
    best = fmaxf(best, static_cast<float>(g));
  }
  hm[i] = best;
}
int launch_draw_heatmap(const int* obj, int B, int max_objs, int ncls, int H, int W, float* hm, cudaStream_t st) {
  const long long n = static_cast<long long>(B) * ncls * H * W;
  (void)launch_k(draw_heatmap_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st, obj, B, max_objs, ncls, H, W, hm);
  return check_cuda(cudaGetLastError(), "draw_heatmap");
}

}  // namespace mf
