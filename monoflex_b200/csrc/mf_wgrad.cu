// Convolution weight gradient on tensor cores (training rows: backward of R2/R3/R6 convs).
//   dW[co, ci, ky, kx] = sum over (b, oy, ox) of  dY[b, oy, ox, co] * X[b, oy*s - p + ky, ox*s - p + kx, ci]
// As a GEMM per tap: D[(tap, ci), co] = A^T B with A = im2col(X; tap) [pixels x ci] and B = dY [pixels x co]: the
// reduction index (output pixels) is the ROW index of both NHWC operands in memory, so both are consumed as MN-major
// tcgen05 operands (instruction-descriptor bits 15/16; smem descriptor LBO = stride between 64-channel blocks, SBO = 1024 B
// between 8-pixel groups - validated by mf_selftest.cu) straight from SWIZZLE_128B TMA boxes:
//   A stage = two 64-channel "slots" (slot = (tap, 64-channel block)), each ONE im2col-mode TMA box of 64 output pixels
//             (zero padding / stride / row and image wrap-around done by the TMA unit, as in the forward kernel);
//   B stage = BLOCK_N/64 tiled-TMA boxes [64 pixels x 64 output channels] of dY.
// Persistent, warp specialised (TMA warp, MMA thread, 4 epilogue warps); the long reduction (B*Ho*Wo pixels) is split over
// the CTAs (split-K work items), each finishing with fp32 atomic adds (RED) into the OIHW fp32 gradient - the summation
// order across splits is therefore not fixed (like cuDNN's non-deterministic wgrad algorithms).
#include "mf_common.cuh"
#include "mf_kernels.h"
#include <cstring>

namespace mf {

static constexpr int WG_BK = 64;                        // pixels per k block
static constexpr int WG_STAGES = 6;
// Narrow layers (Cin or Cout = 16 / 32: level0 / level1 of DLA-34) use narrower boxes: an A slot is AW = min(Cin, 64)
// channels wide (128 / AW slots per M tile), a B box BW = min(Cout, 64); the TMA swizzle and the descriptor layout type
// follow the box width (128B / 64B / 32B), LBO = box bytes, SBO = 8 rows of the box.
MF_DEVINL constexpr uint32_t wg_layout(int width) { return width == 64 ? 2u : (width == 32 ? 4u : 6u); }

struct WgradParams {
  int B, H, W, Cin, Ho, Wo, Cout, kh, kw, stride, pad_h, pad_w;
  int nslots;            // taps * Cin / AW
  int ntm, ntn;          // M tiles (slot pairs), N tiles
  int nkb;               // ceil(B*Ho*Wo / 64)
  int splits;            // K splits per tile
  float* dw;             // [Cout, Cin, k, k] fp32, zero-initialised by the launcher
};

template <int BLOCK_N, int AW, int BW>
__global__ void __launch_bounds__(192, 1)
wgrad_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_dy, const WgradParams p) {
  constexpr int SPT = 128 / AW;                            // A slots per M tile
  constexpr int A_BOX = WG_BK * AW * 2, B_BOX = WG_BK * BW * 2;
  constexpr int A_STAGE = SPT * A_BOX;                     // = 16 KB
  constexpr int NB = BLOCK_N / BW;
  constexpr int B_STAGE = NB * B_BOX < 1024 ? 1024 : NB * B_BOX;
  constexpr int TCOLS = BLOCK_N < 32 ? 32 : BLOCK_N;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_smem = smem;
  uint8_t* b_smem = a_smem + WG_STAGES * A_STAGE;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(b_smem + WG_STAGES * B_STAGE);
  uint64_t* empty_bar = full_bar + WG_STAGES;
  uint64_t* acc_full = empty_bar + WG_STAGES;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(acc_empty + 1);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  const int nitems = p.ntm * p.ntn * p.splits;
  const int HoWo = p.Ho * p.Wo, cblocks = p.Cin / AW;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tmap_x); tma_prefetch_desc(&tmap_dy);
    for (int s = 0; s < WG_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(acc_full, 1); mbar_init(acc_empty, 128);
    fence_mbar_init();
  }
  if (warp == 5) tmem_alloc(tmem_ptr_smem, TCOLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // item -> (m tile, n tile, k range)
  auto decode = [&](int item, int& mt, int& nt, int& kb_lo, int& kb_hi) {
    const int sp = item % p.splits;
    const int t = item / p.splits;
    nt = t % p.ntn;
    mt = t / p.ntn;
    const int base = p.nkb / p.splits, extra = p.nkb % p.splits;
    kb_lo = sp * base + (sp < extra ? sp : extra);
    kb_hi = kb_lo + base + (sp < extra ? 1 : 0);
  };

  if (warp == 4) {
    // ================================================================ TMA producer (all lanes walk the loops, one issues)
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        int mt, nt, kb_lo, kb_hi;
        decode(item, mt, nt, kb_lo, kb_hi);
        int s_tap[SPT], s_c0[SPT];
#pragma unroll
        for (int h = 0; h < SPT; ++h) {
          int slot = SPT * mt + h;
          if (slot >= p.nslots) slot = p.nslots - 1;             // dummy slot (its rows are discarded by the epilogue)
          s_tap[h] = slot / cblocks;
          s_c0[h] = (slot - s_tap[h] * cblocks) * AW;
        }
        for (int kb = kb_lo; kb < kb_hi; ++kb) {
          const int p0 = kb * WG_BK;                              // first output pixel of the block
          const int n = p0 / HoWo, rem = p0 - n * HoWo;
          const int oy = rem / p.Wo, ox = rem - oy * p.Wo;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&full_bar[stage], A_STAGE + NB * B_BOX);
#pragma unroll
            for (int h = 0; h < SPT; ++h) {
              const int ky = s_tap[h] / p.kw, kx = s_tap[h] - ky * p.kw;
              tma_load_im2col_4d(smem_u32(a_smem + stage * A_STAGE + h * A_BOX), &tmap_x, &full_bar[stage], s_c0[h],
                                 ox * p.stride - p.pad_w, oy * p.stride - p.pad_h, n, static_cast<uint16_t>(kx),
                                 static_cast<uint16_t>(ky));
            }
#pragma unroll
            for (int j = 0; j < NB; ++j)
              tma_load_2d(smem_u32(b_smem + stage * B_STAGE + j * B_BOX), &tmap_dy, &full_bar[stage], nt * BLOCK_N + j * BW, p0);
          }
          __syncwarp();
          if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 5) {
    // ================================================================ MMA issuer (all lanes walk the loops, one issues)
    {
      constexpr uint32_t idesc = umma_idesc_f16(128, BLOCK_N) | (1u << 15) | (1u << 16);      // A and B MN-major
      const uint64_t a_d0 = umma_desc_kmajor(smem_u32(a_smem), A_BOX, 16 * AW, wg_layout(AW));
      const uint64_t b_d0 = umma_desc_kmajor(smem_u32(b_smem), B_BOX, 16 * BW, wg_layout(BW));
      int stage = 0, it = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
        int mt, nt, kb_lo, kb_hi;
        decode(item, mt, nt, kb_lo, kb_hi);
        mbar_wait(acc_empty, (it & 1) ^ 1);
        tc_fence_after();
        for (int kb = kb_lo; kb < kb_hi; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t a_off = static_cast<uint64_t>((stage * A_STAGE) >> 4), b_off = static_cast<uint64_t>((stage * B_STAGE) >> 4);
          if (elect_one()) {
#pragma unroll
            for (int k4 = 0; k4 < WG_BK / 16; ++k4)               // 16 pixels = two 8-row groups (2 * SBO) per MMA
              umma_f16(tmem_base, a_d0 + a_off + static_cast<uint64_t>(k4 * ((2 * 16 * AW) >> 4)),
                       b_d0 + b_off + static_cast<uint64_t>(k4 * ((2 * 16 * BW) >> 4)), idesc, (kb > kb_lo || k4 != 0) ? 1u : 0u);
            umma_commit(&empty_bar[stage]);
            if (kb == kb_hi - 1) umma_commit(acc_full);
          }
          __syncwarp();
          if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
        }
        if (kb_hi <= kb_lo) {                                     // empty K range (host never asks for more splits than blocks)
          if (elect_one()) umma_commit(acc_full);
          __syncwarp();
        }
      }
    }
  } else {
    // ================================================================ epilogue: TMEM -> fp32 atomics into OIHW dW
    const int row = warp * 32 + lane;                              // M index inside the tile
    const int taps = p.kh * p.kw;
    int it = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
      int mt, nt, kb_lo, kb_hi;
      decode(item, mt, nt, kb_lo, kb_hi);
      const int slot = SPT * mt + row / AW;
      const bool valid = slot < p.nslots && kb_hi > kb_lo;
      const int tap = valid ? slot / cblocks : 0;
      const int ci = valid ? (slot - tap * cblocks) * AW + (row % AW) : 0;
      mbar_wait(acc_full, it & 1);
      tc_fence_after();
      constexpr int CH = BLOCK_N >= 32 ? 32 : 16;
#pragma unroll
      for (int c = 0; c < BLOCK_N; c += CH) {
        uint32_t r[CH];
        if constexpr (CH == 32) tmem_ld32(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + c, r);
        else tmem_ld16(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + c, r);
        tmem_ld_wait();
        if (valid) {
#pragma unroll
          for (int j = 0; j < CH; ++j) {
            const int co = nt * BLOCK_N + c + j;
            if (co < p.Cout) atomicAdd(p.dw + (static_cast<long long>(co) * p.Cin + ci) * taps + tap, __uint_as_float(r[j]));
          }
        }
      }
      tc_fence_before();
      mbar_arrive(acc_empty);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem_base, TCOLS);
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encTiledW)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_encIm2colW)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static void* wg_driver_fn(const char* name) {
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint(name, &ptr, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess)
    return nullptr;
  return ptr;
}

template <int BLOCK_N, int AW, int BW>
static int launch_wgrad_cfg(const CUtensorMap& tx, const CUtensorMap& tdy, const WgradParams& p, int grid, cudaStream_t st) {
  constexpr int B_ST = (BLOCK_N / BW) * WG_BK * BW * 2 < 1024 ? 1024 : (BLOCK_N / BW) * WG_BK * BW * 2;
  constexpr int SMEM = WG_STAGES * (WG_BK * 128 * 2 + B_ST) + 1024 + 1024;
  static bool attr = false;
  if (!attr) {
    if (check_cuda(cudaFuncSetAttribute(wgrad_kernel<BLOCK_N, AW, BW>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM), "wgrad smem")) return -1;
    attr = true;
  }
  wgrad_kernel<BLOCK_N, AW, BW><<<grid, 192, SMEM, st>>>(tx, tdy, p);
  return check_cuda(cudaGetLastError(), "conv wgrad launch");
}
template <int AW>
static int launch_wgrad_n(int bn, const CUtensorMap& tx, const CUtensorMap& tdy, const WgradParams& p, int grid, cudaStream_t st) {
  if (bn == 128) return launch_wgrad_cfg<128, AW, 64>(tx, tdy, p, grid, st);
  if (bn == 64) return launch_wgrad_cfg<64, AW, 64>(tx, tdy, p, grid, st);
  if (bn == 32) return launch_wgrad_cfg<32, AW, 32>(tx, tdy, p, grid, st);
  return launch_wgrad_cfg<16, AW, 16>(tx, tdy, p, grid, st);
}

// x: [B*H*W, x_ld] fp16 NHWC rows; dy: [B*Ho*Wo, dy_ld] fp16 rows; dw: [Cout, Cin, kh, kw] fp32 (overwritten)
int launch_conv_wgrad(const __half* x, int x_ld, int B, int H, int W, int Cin, const __half* dy, int dy_ld, int Cout, int kh,
                      int kw, int stride, int pad_h, int pad_w, float* dw, cudaStream_t st) {
  static PFN_encTiledW enc = reinterpret_cast<PFN_encTiledW>(wg_driver_fn("cuTensorMapEncodeTiled"));
  static PFN_encIm2colW enc2 = reinterpret_cast<PFN_encIm2colW>(wg_driver_fn("cuTensorMapEncodeIm2col"));
  if (!enc || !enc2) { set_error("conv wgrad: tensor-map driver entry points unavailable"); return -1; }
  const bool cin_ok = Cin == 16 || Cin == 32 || (Cin > 0 && Cin % 64 == 0);
  const bool cout_ok = Cout == 16 || Cout == 32 || (Cout > 0 && Cout % 64 == 0);
  if (!cin_ok || !cout_ok || x_ld % 8 != 0 || dy_ld % 8 != 0 || kh < 1 || kh > 7 || kw < 1 || kw > 7 || stride < 1 || stride > 8 ||
      (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(dy) & 15)) {
    set_error("conv wgrad: needs Cin, Cout in {16, 32, multiples of 64} and 16-byte aligned rows (Cin=%d Cout=%d k=%dx%d s=%d)", Cin,
              Cout, kh, kw, stride);
    return -1;
  }
  // full-resolution stem layers: all reduction, no tile (mf_wgrad_narrow.cu)
  if (Cin == 16 && Cout == 16 && stride == 1 && kh == kw && (kh == 3 || kh == 7) && pad_h == kh / 2 && pad_w == kh / 2)
    return launch_conv_wgrad_narrow(x, x_ld, B, H, W, dy, dy_ld, kh, dw, st);
  const int aw = Cin < 64 ? Cin : 64, bw = Cout < 64 ? Cout : 64;
  WgradParams p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.H = H; p.W = W; p.Cin = Cin; p.Cout = Cout; p.kh = kh; p.kw = kw; p.stride = stride; p.pad_h = pad_h; p.pad_w = pad_w;
  p.Ho = (H + 2 * pad_h - kh) / stride + 1;
  p.Wo = (W + 2 * pad_w - kw) / stride + 1;
  if (p.Ho < 1 || p.Wo < 1) { set_error("conv wgrad: empty output"); return -1; }
  const long long Mout = static_cast<long long>(B) * p.Ho * p.Wo;
  const int bn = Cout < 64 ? Cout : (Cout % 128 == 0 ? 128 : 64);
  const int spt = 128 / aw;
  p.nslots = kh * kw * (Cin / aw);
  p.ntm = (p.nslots + spt - 1) / spt;
  p.ntn = Cout / bn;
  p.nkb = static_cast<int>((Mout + WG_BK - 1) / WG_BK);
  p.dw = dw;
  int dev = 0, nsm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  const int tiles = p.ntm * p.ntn;
  int splits = (2 * nsm + tiles - 1) / tiles;                   // ~2 work items per SM
  if (splits > p.nkb) splits = p.nkb;
  if (splits < 1) splits = 1;
  p.splits = splits;
  CUtensorMap tx, tdy;
  {
    cuuint64_t gdim[4] = {static_cast<cuuint64_t>(Cin), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(B)};
    cuuint64_t gstr[3] = {static_cast<cuuint64_t>(x_ld) * 2, static_cast<cuuint64_t>(x_ld) * 2 * W, static_cast<cuuint64_t>(x_ld) * 2 * W * H};
    int lower[2] = {-pad_w, -pad_h}, upper[2] = {pad_w - (kw - 1), pad_h - (kh - 1)};
    cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(stride), static_cast<cuuint32_t>(stride), 1};
    const CUtensorMapSwizzle swa = aw == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : aw == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    if (enc2(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(x), gdim, gstr, lower, upper, static_cast<cuuint32_t>(aw),
             WG_BK, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swa, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) { set_error("conv wgrad: im2col map failed"); return -1; }
  }
  {
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(Cout), static_cast<cuuint64_t>(Mout)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(dy_ld) * 2};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(bw), WG_BK};
    cuuint32_t estr[2] = {1, 1};
    const CUtensorMapSwizzle swb = bw == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : bw == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    if (enc(&tdy, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(dy), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            swb, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
      set_error("conv wgrad: dY map failed");
      return -1;
    }
  }
  if (check_cuda(cudaMemsetAsync(dw, 0, sizeof(float) * Cout * Cin * kh * kw, st), "conv wgrad memset")) return -1;
  const int nitems = tiles * splits;
  const int grid = nitems < nsm ? nitems : nsm;
  if (aw == 64) return launch_wgrad_n<64>(bn, tx, tdy, p, grid, st);
  if (aw == 32) return launch_wgrad_n<32>(bn, tx, tdy, p, grid, st);
  return launch_wgrad_n<16>(bn, tx, tdy, p, grid, st);
}

}  // namespace mf
