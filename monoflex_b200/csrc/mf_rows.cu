// "Row-segment" convolution for the full-resolution stem (base_layer 7x7 3->16, level0 3x3 16->16, level1 3x3/2 16->32,
// dla_dcn.py:268-282): tensors whose pixels are 16 bytes (8 fp16 channels) are kept as planes [B][H][G][Wg][8]
// (G = channel-planes x column-parities), and the implicit-GEMM A operand is never materialised:
//
//   * per output tile (128 consecutive pixels of one output row) the TMA warp loads each needed input row segment ONCE
//     (144 pixels x 16 B, two tiled cp.async.bulk.tensor boxes of 8-byte elements per (row, plane, parity), zero fill outside
//     the image);
//   * the MMA warp reads the im2col matrix *through descriptors*: with the no-swizzle K-major layout a core matrix is
//     8 rows x 16 B with rows 16 B apart, which is exactly "8 consecutive pixels" of a segment, so
//       A[r, tap kx] = segment[(r + kx) * 16 B]      -> start address + kx*16, SBO = 128 (8 pixels)
//     and the second 16-byte K chunk of an MMA (the next tap for Cin = 8, the second channel plane for Cin = 16) is
//     reached through LBO. A 7x7 conv is 28 MMAs per tile, a 3x3 one 9 - no 49x / 9x copies through L1/L2 (the
//     cp.async gather this replaces ran at 0.57 ms for the 7x7 layer; its unique HBM traffic is 0.03 ms);
//   * stride 2 works on column-parity planes (pixel 2*ox + kx - 1 = parity (kx+1)&1, index ox + (kx-1)>>1);
//   * the whole packed weight matrix stays resident in smem (<= 14 KB), accumulators are double-buffered in TMEM, the
//     epilogue (scale/shift + ReLU) writes either the planar layout of the next stem layer or plain NHWC rows.
#include "mf_common.cuh"
#include "mf_kernels.h"
#include <cstring>

namespace mf {

static constexpr int RBM = 128;
static constexpr int SEG_PIX = 144;                // 128 + 2 x 4 halo, rounded so that half a segment is a multiple of 128 B
static constexpr int SEG_BYTES = SEG_PIX * 16;     // 2304 = 18 * 128
static constexpr int R_STAGES = 6;
static constexpr int MAX_SEG = 24;          // strict stride-2 layer: 3 rows x 4 planes (hi0 hi1 lo0 lo1) x 2 column parities
static constexpr int MAX_MMA = 56;          // strict precision: 2 x 28 (image pair plane) or 3 x 9 (pair planes) products

struct RowsParams {
  int B, H, Gin, Wg_in;          // input planes [B][H][Gin][Wg_in][8]
  int Ho, Wo, stride, pad;
  int nseg, nmma, nkb;           // nkb = k_pad / 64 weight K blocks
  int nstages;                   // row-segment ring depth (<= R_STAGES), sized on the host so that two CTAs fit one SM
  int seg_g[MAX_SEG], seg_dy[MAX_SEG], seg_dx[MAX_SEG];      // group, input row = oy*stride + dy, start index = ox0 + dx
  int mma_a[MAX_MMA], mma_lbo[MAX_MMA], mma_b[MAX_MMA];      // byte offsets: A start within the stage, LBO, B start
  int Cout;
  const float* scale;
  const float* shift;
  int act;
  int out_planar;                // 1: y = [B][Ho][Cout/8 * out_npar][Wo/out_npar][8]; 0: NHWC rows with y_ld
  int out_npar;
  __half* y;
  int y_ld;
  int split_out;                 // strict precision: output = fp16 pair (hi planes then lo planes / lo block y_lo after hi)
  int y_lo;
};

template <int BLOCK_N>
__global__ void __launch_bounds__(192, 2)
rows_conv_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                 const __grid_constant__ RowsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stage_bytes = p.nseg * SEG_BYTES;                 // multiple of 128
  const int stage_stride = (stage_bytes + 1023) & ~1023;
  uint8_t* b_smem = smem;                                     // [nkb][BLOCK_N][128 B] swizzled weight blocks
  uint8_t* a_smem = smem + ((p.nkb * BLOCK_N * 128 + 1023) & ~1023);
  const int NST = p.nstages;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(a_smem + NST * stage_stride);
  uint64_t* empty_bar = full_bar + R_STAGES;
  uint64_t* acc_full = empty_bar + R_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint64_t* w_bar = acc_empty + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(w_bar + 1);
  uint64_t* desc_tab = w_bar + 2;                              // [2 * MAX_MMA]

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;      // warp-uniform for the compiler
  const int tiles_x = (p.Wo + RBM - 1) / RBM;
  const int ntiles = p.B * p.Ho * tiles_x;
  constexpr int ACC_COLS = 32;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_x);
    tma_prefetch_desc(&tmap_w);
    for (int s = 0; s < NST; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 128); }
    mbar_init(w_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr_smem, 2 * ACC_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ================================================================ TMA: resident weights, then row segments per tile
    // (all lanes walk the loop, one elected lane issues)
    {
      if (elect_one()) {
        mbar_arrive_expect_tx(w_bar, p.nkb * BLOCK_N * 128);
        for (int kb = 0; kb < p.nkb; ++kb)
          tma_load_2d(smem_u32(b_smem + kb * BLOCK_N * 128), &tmap_w, w_bar, kb * 64, 0);
      }
      __syncwarp();
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int tx = t % tiles_x, row = t / tiles_x;
        const int oy = row % p.Ho, b = row / p.Ho;
        const int ox0 = tx * RBM;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        const uint32_t dst = smem_u32(a_smem + stage * stage_stride);
        if (elect_one()) {
          mbar_arrive_expect_tx(&full_bar[stage], stage_bytes);
          for (int sgi = 0; sgi < p.nseg; ++sgi) {             // a segment = two boxes of 144 eight-byte elements (see host)
            const int xe = 2 * (ox0 + p.seg_dx[sgi]), yy = oy * p.stride + p.seg_dy[sgi];
            tma_load_4d(dst + sgi * SEG_BYTES, &tmap_x, &full_bar[stage], xe, p.seg_g[sgi], yy, b);
            tma_load_4d(dst + sgi * SEG_BYTES + SEG_BYTES / 2, &tmap_x, &full_bar[stage], xe + SEG_PIX, p.seg_g[sgi], yy, b);
          }
        }
        __syncwarp();
        if (++stage == NST) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ================================================================ MMA issuer (all lanes walk the loop, one issues)
    {
      constexpr uint32_t idesc = umma_idesc_f16(RBM, BLOCK_N);
      mbar_wait(w_bar, 0);
      tc_fence_after();
      const uint32_t a0 = smem_u32(a_smem), b0 = smem_u32(b_smem);
      // descriptor tables in smem (stage 0 addresses): the issue loop is ld.shared + 64-bit add per MMA
      for (int i = lane; i < p.nmma; i += 32) {
        desc_tab[2 * i] = umma_desc_kmajor(a0 + p.mma_a[i], p.mma_lbo[i], 128, 0);
        desc_tab[2 * i + 1] = umma_desc_sw128(b0 + p.mma_b[i]);
      }
      __syncwarp();
      const int nmma = p.nmma;
      int stage = 0, ti = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++ti) {
        const int acc = ti & 1;
        mbar_wait(&acc_empty[acc], ((ti >> 1) & 1) ^ 1);
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * ACC_COLS;
        const uint64_t a_off = static_cast<uint64_t>((stage * stage_stride) >> 4);
        if (elect_one()) {
#pragma unroll 7
          for (int i = 0; i < nmma; ++i)
            umma_f16(d_tmem, desc_tab[2 * i] + a_off, desc_tab[2 * i + 1], idesc, i != 0 ? 1u : 0u);
          umma_commit(&empty_bar[stage]);
          umma_commit(&acc_full[acc]);
        }
        __syncwarp();
        if (++stage == NST) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ================================================================ epilogue (warps 2..5)
    const int quad = warp & 3;
    const int r = quad * 32 + lane;
    float sc[BLOCK_N], sh[BLOCK_N];                     // tile-invariant affine: registers, not per-tile loads
#pragma unroll
    for (int i = 0; i < BLOCK_N; ++i) { sc[i] = __ldg(p.scale + i); sh[i] = __ldg(p.shift + i); }
    const bool relu = p.act == ACT_RELU;
    int ti = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++ti) {
      const int acc = ti & 1;
      const int tx = t % tiles_x, row = t / tiles_x;
      const int oy = row % p.Ho, b = row / p.Ho;
      const int ox = tx * RBM + r;
      mbar_wait(&acc_full[acc], (ti >> 1) & 1);
      tc_fence_after();
      uint32_t v[BLOCK_N];
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * ACC_COLS;
      if constexpr (BLOCK_N == 32) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&acc_empty[acc]);
      if (ox >= p.Wo) continue;
      __half2 o[BLOCK_N / 2], ol[BLOCK_N / 2];
#pragma unroll
      for (int i = 0; i < BLOCK_N; i += 2) {
        float f0 = __uint_as_float(v[i]) * sc[i] + sh[i];
        float f1 = __uint_as_float(v[i + 1]) * sc[i + 1] + sh[i + 1];
        if (relu) { f0 = fmaxf(f0, 0.f); f1 = fmaxf(f1, 0.f); }
        o[i / 2] = __floats2half2_rn(f0, f1);
        const float2 hf = __half22float2(o[i / 2]);
        ol[i / 2] = __floats2half2_rn(f0 - hf.x, f1 - hf.y);          // lo half of the pair (dead code unless split_out)
      }
      if (p.out_planar) {
        const int npar = p.out_npar, Wg = p.Wo / npar;
        const int par = npar == 2 ? (ox & 1) : 0, xi = npar == 2 ? (ox >> 1) : ox;
        const int Ghalf = (p.Cout / 8) * npar, G = p.split_out ? 2 * Ghalf : Ghalf;
#pragma unroll
        for (int pl = 0; pl < BLOCK_N / 8; ++pl) {
          if (pl * 8 < p.Cout) {
            __half* dst = p.y + ((static_cast<long long>(b * p.Ho + oy) * G + (pl * npar + par)) * Wg + xi) * 8;
            *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(&o[pl * 4]);
            if (p.split_out)
              *reinterpret_cast<uint4*>(dst + static_cast<long long>(Ghalf) * Wg * 8) = *reinterpret_cast<const uint4*>(&ol[pl * 4]);
          }
        }
      } else {
        __half* dst = p.y + (static_cast<long long>(b * p.Ho + oy) * p.Wo + ox) * p.y_ld;
#pragma unroll
        for (int pl = 0; pl < BLOCK_N / 8; ++pl)
          if (pl * 8 < p.Cout) {
            *reinterpret_cast<uint4*>(dst + pl * 8) = *reinterpret_cast<const uint4*>(&o[pl * 4]);
            if (p.split_out) *reinterpret_cast<uint4*>(dst + p.y_lo + pl * 8) = *reinterpret_cast<const uint4*>(&ol[pl * 4]);
          }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 2 * ACC_COLS);
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiledR)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiledR rows_encode_fn() {
  static PFN_encodeTiledR fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess || ptr == nullptr) {
      set_error("cuTensorMapEncodeTiled entry point unavailable");
      return nullptr;
    }
    fn = reinterpret_cast<PFN_encodeTiledR>(ptr);
  }
  return fn;
}

// x: planes [B][H][Gin][Wg_in][8] fp16 with Gin = (Cin/8) * in_npar; wp: packed weights [n_pad, k_pad] fp16 whose K order is
// (ky, kx, c) with c over Cin (Cin = 16) or (ky, kx over kw_pad = 8, c over 8) (Cin = 8).
// in_mode 0: plain fp16 planes. Strict precision (fp16 pairs):
//   in_mode 1 (Cin = 8): the image pair plane [hi3 | lo3 | 0 0]; weights packed as TWO tap sets stacked along ky,
//              [W_hi | W_hi | 0 0] (A_hi W_hi + A_lo W_hi in one K = 8 slot) and [W_lo | 0 ...] (A_hi W_lo);
//   in_mode 2 (Cin = 16): pair planes [hi0 hi1 lo0 lo1]; weights packed as THREE tap sets stacked along ky:
//              W_hi (x hi planes), W_hi (x lo planes), W_lo (x hi planes).
// The extra products are extra entries of the MMA table over the SAME resident row segments - no extra loads for in_mode 1.
int launch_rows_conv(const __half* x, int B, int H, int W, int Cin, int in_npar, const __half* wp, int n_pad, int k_pad,
                     int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift, int act,
                     int out_planar, int out_npar, __half* y, int y_ld, cudaStream_t st, int in_mode, int split_out,
                     int y_lo) {
  PFN_encodeTiledR enc = rows_encode_fn();
  if (!enc) return -1;
  RowsParams p;
  memset(&p, 0, sizeof(p));
  const int P = Cin / 8;
  const int nsets = in_mode == 1 ? 2 : (in_mode == 2 ? 3 : 1);
  const int Ptot = in_mode == 2 ? 2 * P : P;             // planes in memory (hi planes, then lo planes)
  if (in_mode < 0 || in_mode > 2 || (in_mode == 1 && Cin != 8) || (in_mode == 2 && Cin != 16) ||
      (split_out && !out_planar && y_lo % 8 != 0)) {
    set_error("rows_conv: unsupported strict-precision configuration (in_mode %d, Cin %d, stride %d)", in_mode, Cin, stride);
    return -1;
  }
  if ((Cin != 8 && Cin != 16) || (stride != 1 && stride != 2) || (stride == 2 && (in_npar != 2 || kw != 3 || pad != 1)) ||
      (stride == 1 && in_npar != 1) || (n_pad != 16 && n_pad != 32) || k_pad % 64 != 0 || W % in_npar != 0 ||
      (Cin == 8 && kw > 8) || pad > 3 || kw - 1 - pad > 4) {
    set_error("rows_conv: unsupported configuration Cin=%d stride=%d in_npar=%d kw=%d pad=%d n_pad=%d", Cin, stride, in_npar,
              kw, pad, n_pad);
    return -1;
  }
  p.B = B; p.H = H; p.Gin = Ptot * in_npar; p.Wg_in = W / in_npar;
  p.split_out = split_out; p.y_lo = y_lo;
  p.Ho = (H + 2 * pad - kh) / stride + 1;
  p.Wo = (W + 2 * pad - kw) / stride + 1;
  p.stride = stride; p.pad = pad; p.nkb = k_pad / 64;
  p.Cout = Cout; p.scale = scale; p.shift = shift; p.act = act;
  p.out_planar = out_planar; p.out_npar = out_npar; p.y = y; p.y_ld = y_ld;
  if (out_planar && (Cout % 8 != 0 || p.Wo % out_npar != 0)) { set_error("rows_conv: planar output needs Cout %% 8 == 0"); return -1; }
  // ---- segments and MMA table
  int nseg = 0, nmma = 0;
  auto seg_index = [&](int ky, int plane, int par) { return (ky * Ptot + plane) * (stride == 2 ? 2 : 1) + par; };
  for (int ky = 0; ky < kh; ++ky)
    for (int plane = 0; plane < Ptot; ++plane)
      for (int par = 0; par < (stride == 2 ? 2 : 1); ++par) {
        if (nseg >= MAX_SEG) { set_error("rows_conv: too many segments"); return -1; }
        p.seg_g[nseg] = plane * in_npar + par;
        p.seg_dy[nseg] = ky - pad;
        p.seg_dx[nseg] = stride == 2 ? -1 : -pad;
        ++nseg;
      }
  const int kw_pad = Cin == 8 ? 8 : kw;
  if (k_pad < nsets * kh * kw_pad * Cin) { set_error("rows_conv: k_pad too small"); return -1; }
  for (int set = 0; set < nsets; ++set)
  for (int ky = 0; ky < kh; ++ky) {
    const int kyw = set * kh + ky;                      // row of the stacked weight tap sets
    if (Cin == 8) {
      for (int q = 0; q < kw_pad / 2; ++q) {            // two taps per MMA, second tap through LBO = one pixel
        if (nmma >= MAX_MMA) { set_error("rows_conv: too many MMAs"); return -1; }
        p.mma_a[nmma] = seg_index(ky, 0, 0) * SEG_BYTES + (2 * q) * 16;
        p.mma_lbo[nmma] = 16;
        const int koff = (kyw * kw_pad + 2 * q) * 8;
        p.mma_b[nmma] = (koff / 64) * n_pad * 128 + ((koff % 64) / 16) * 32;
        ++nmma;
      }
    } else {
      const int pl0 = (in_mode == 2 && set == 1) ? P : 0;   // second set reads the lo planes
      for (int kx = 0; kx < kw; ++kx) {                 // one tap per MMA, second channel plane through LBO
        if (nmma >= MAX_MMA) { set_error("rows_conv: too many MMAs"); return -1; }
        int par = 0, shift_px = kx;
        if (stride == 2) { par = (kx == 1) ? 0 : 1; shift_px = (kx == 0) ? 0 : 1; }
        p.mma_a[nmma] = seg_index(ky, pl0, par) * SEG_BYTES + shift_px * 16;
        p.mma_lbo[nmma] = (seg_index(ky, pl0 + 1, par) - seg_index(ky, pl0, par)) * SEG_BYTES;
        const int koff = (kyw * kw + kx) * 16;
        p.mma_b[nmma] = (koff / 64) * n_pad * 128 + ((koff % 64) / 16) * 32;
        ++nmma;
      }
    }
  }
  p.nseg = nseg; p.nmma = nmma;
  // ---- tensor maps
  CUtensorMap tx, tw;
  {
    // A plane row is contiguous (Wg pixels x 16 B). Described with its natural {8 ch, Wg, ..} dimensions the TMA unit issues
    // one 16-byte request per pixel and a tile's 7-12 segments cost ~1000-1600 requests (the kernel was request-bound:
    // 2.5 us per 128-pixel tile). As 8-byte elements a row is ONE dimension of 2*Wg elements; a box holds <= 256 elements,
    // so a 144-pixel segment is two boxes of 144 elements (1152 B each, TMA needs 128-byte aligned smem destinations).
    // Out-of-range elements are zero-filled as before.
    cuuint64_t gdim[4] = {static_cast<cuuint64_t>(p.Wg_in) * 2, static_cast<cuuint64_t>(p.Gin), static_cast<cuuint64_t>(H),
                          static_cast<cuuint64_t>(B)};
    cuuint64_t gstr[3] = {static_cast<cuuint64_t>(p.Wg_in) * 16, static_cast<cuuint64_t>(p.Wg_in) * 16 * p.Gin,
                          static_cast<cuuint64_t>(p.Wg_in) * 16 * p.Gin * H};
    cuuint32_t box[4] = {SEG_PIX, 1, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&tx, CU_TENSOR_MAP_DATA_TYPE_UINT64, 4, const_cast<__half*>(x), gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("rows_conv: cuTensorMapEncodeTiled(x) failed (%d)", static_cast<int>(r)); return -1; }
  }
  {
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(k_pad), static_cast<cuuint64_t>(n_pad)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(k_pad) * 2};
    cuuint32_t box[2] = {64, static_cast<cuuint32_t>(n_pad)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&tw, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(wp), gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("rows_conv: cuTensorMapEncodeTiled(w) failed (%d)", static_cast<int>(r)); return -1; }
  }
  const int stage_stride = (nseg * SEG_BYTES + 1023) & ~1023;
  const int w_bytes = (p.nkb * n_pad * 128 + 1023) & ~1023;
  int nst = (113 * 1024 - w_bytes - 3072) / stage_stride;            // two CTAs per SM whenever >= 2 stages fit
  if (nst < 2) nst = (226 * 1024 - w_bytes - 3072) / stage_stride;
  if (nst > R_STAGES) nst = R_STAGES;
  if (nst < 2) { set_error("rows_conv: row segments do not fit in shared memory"); return -1; }
  p.nstages = nst;
  const int smem = w_bytes + nst * stage_stride + 1024 + 2048;
  const int tiles = B * p.Ho * ((p.Wo + RBM - 1) / RBM);
  int dev = 0, nsm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  const int grid = tiles < 2 * nsm ? tiles : 2 * nsm;    // two CTAs per SM (<= 110 KB of smem each)
  if (n_pad == 16) {
    static int attr = 0;
    if (smem > attr) {
      if (check_cuda(cudaFuncSetAttribute(rows_conv_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), "rows smem")) return -1;
      attr = smem;
    }
    if (check_cuda(launch_k(rows_conv_kernel<16>, dim3(grid), dim3(192), smem, st, tx, tw, p), "rows_conv launch")) return -1;
  } else {
    static int attr = 0;
    if (smem > attr) {
      if (check_cuda(cudaFuncSetAttribute(rows_conv_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), "rows smem")) return -1;
      attr = smem;
    }
    if (check_cuda(launch_k(rows_conv_kernel<32>, dim3(grid), dim3(192), smem, st, tx, tw, p), "rows_conv launch")) return -1;
  }
  return check_cuda(cudaGetLastError(), "rows_conv launch");
}

}  // namespace mf
