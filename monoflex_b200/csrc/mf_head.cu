// Fused predictor head (detector_predictor.py:121-135): the nine shared-input 3x3 convs (64 -> 9 x 256) + InPlaceABN +
// the 1x1 output convs (256 -> {3,4,2,20,3,3,16,1,1}) in ONE persistent kernel. The 2304-channel hidden map (1.13 GB at
// B = 8) is never written to HBM except for the two branches the edge-fusion gather needs.
//
// Per CTA (one per SM): for every 128-pixel m-tile, for every 128-channel n-tile nt (branch b = nt/2, half h = nt%2):
//   main GEMM   TMA warp: im2col-mode TMA A boxes + weight boxes -> 4-stage ring; MMA thread: tcgen05.mma into one of two
//               128-column TMEM accumulators (exactly the MODE_CONV_TMA pipeline of mf_igemm2.cu)
//   epilogue    8 warps: tcgen05.ld -> |gamma| BN affine -> leaky 0.01 -> fp16 -> 128B-swizzled smem staging. The staged
//               128 x 128 tile IS a canonical K-major UMMA A operand (two 64-channel sub-tiles), so ...
//   stage 2     ... the MMA thread contracts it with the branch's 1x1 weights (32 x 256, TMA-loaded per branch into a
//               2-deep ring) into a 32-column TMEM accumulator D2, accumulating over the branch's two n-tiles. It is
//               issued one tile late (after the next tile's main MMAs) so it never stalls the main pipeline.
//   epilogue 2  4 warps read D2, add the 1x1 bias and write the fp32 NCHW `cls` / `reg` channels of that branch.
#include "mf_common.cuh"
#include "mf_kernels.h"
#include <cstring>

namespace mf {

static constexpr int HBM = 128, HBN = 128, HBK = 64;
static constexpr int H_STAGES = 4;
static constexpr int H_ASTAGE = HBM * HBK * 2;          // 16 KB
static constexpr int H_BSTAGE = HBN * HBK * 2;          // 16 KB
static constexpr int H_OUT = 2 * H_ASTAGE;              // staged 128 x 128 fp16 tile
static constexpr int H_W2 = 4 * 32 * 128;               // 1x1 weights of one branch: 4 K blocks x [32 rows x 128 B]
static constexpr int H_MAXBR = 16;
static constexpr int H_SMEM = H_STAGES * (H_ASTAGE + H_BSTAGE) + H_OUT + 2 * H_W2 + 2048 + 1024;
static constexpr int H_TMEM_D2 = 256;                   // D2 accumulators live at TMEM columns [256, 320)

struct HeadParams {
  int B, H, W, Cin;              // feature map [B,H,W,Cin] fp16 rows, x_ld given to the tensor map
  int M, nkb, nbranch;           // M = B*H*W, nkb = 9*Cin/64
  const float* scale;            // [nbranch*256] folded |gamma| BN
  const float* shift;
  const float* bias2;            // [nbranch*32]
  float* out[H_MAXBR];           // per branch: fp32 NCHW base pointer already offset to its first channel
  int out_ctot[H_MAXBR];         // channels of the tensor it points into (batch stride = out_ctot*H*W)
  int out_nch[H_MAXBR];          // real output channels of the branch (<= 32)
  int hid_col[H_MAXBR];          // >= 0: hidden activations of this branch are stored at this column of `hid`
  __half* hid;                   // [M, hid_ld]
  int hid_ld;
  const unsigned char* hid_mask; // [M] or null. Non-null: only flagged pixels are stored (the ~830 border pixels per image
};                               // the edge fusion gathers), by per-thread stores instead of a TMA store of every tile

__global__ void __launch_bounds__(320, 1)
head_fused_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                  const __grid_constant__ CUtensorMap tmap_w2, const __grid_constant__ CUtensorMap tmap_hid,
                  const __grid_constant__ HeadParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_smem = smem;
  uint8_t* b_smem = a_smem + H_STAGES * H_ASTAGE;
  uint8_t* o_smem = b_smem + H_STAGES * H_BSTAGE;
  uint8_t* w2_smem = o_smem + H_OUT;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(w2_smem + 2 * H_W2);
  uint64_t* empty_bar = full_bar + H_STAGES;
  uint64_t* acc_full = empty_bar + H_STAGES;    // [2]
  uint64_t* acc_empty = acc_full + 2;           // [2]
  uint64_t* w2_full = acc_empty + 2;            // [2]
  uint64_t* w2_empty = w2_full + 2;             // [2]
  uint64_t* d2_full = w2_empty + 2;             // [2]
  uint64_t* d2_empty = d2_full + 2;             // [2]
  uint64_t* s2_full = d2_empty + 2;             // staging written  (epilogue -> MMA)
  uint64_t* s2_done = s2_full + 1;              // staging consumed (MMA -> epilogue)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(s2_done + 1);
  float* sc_s = reinterpret_cast<float*>(w2_smem + 2 * H_W2 + 1024);
  float* sh_s = sc_s + HBN;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  const int ntn = p.nbranch * 2;
  const int ntm = (p.M + HBM - 1) / HBM;
  const int HW = p.H * p.W;
  const int nkb = p.nkb;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tmap_x); tma_prefetch_desc(&tmap_w); tma_prefetch_desc(&tmap_w2); tma_prefetch_desc(&tmap_hid);
    for (int s = 0; s < H_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 256);
      mbar_init(&w2_full[a], 1); mbar_init(&w2_empty[a], 1);
      mbar_init(&d2_full[a], 1); mbar_init(&d2_empty[a], 128);
    }
    mbar_init(s2_full, 1); mbar_init(s2_done, 1);
    fence_mbar_init();
  }
  if (warp == 5) tmem_alloc(tmem_ptr_smem, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 4) {
    // ================================================================ TMA producer (all lanes walk the loops, one issues)
    {
      int stage = 0, bc = 0;
      uint32_t phase = 0;
      for (int mt = blockIdx.x; mt < ntm; mt += gridDim.x) {
        const int m0 = mt * HBM;
        const int cn = m0 / HW, rem = m0 - cn * HW;
        const int cw = rem % p.W - 1, chh = rem / p.W - 1;          // 3x3, stride 1, pad 1
        for (int nt = 0; nt < ntn; ++nt) {
          if ((nt & 1) == 0) {                                       // 1x1 weights of branch nt/2 -> w2 ring
            const int buf = bc & 1;
            mbar_wait(&w2_empty[buf], ((bc >> 1) & 1) ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(&w2_full[buf], H_W2);
              for (int kk = 0; kk < 4; ++kk)
                tma_load_2d(smem_u32(w2_smem + buf * H_W2 + kk * 32 * 128), &tmap_w2, &w2_full[buf], kk * 64, (nt >> 1) * 32);
            }
            __syncwarp();
            ++bc;
          }
          int tap = 0, c0 = 0, kx = 0, ky = 0;
          for (int kb = 0; kb < nkb; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(&full_bar[stage], H_ASTAGE + H_BSTAGE);
              tma_load_im2col_4d(smem_u32(a_smem + stage * H_ASTAGE), &tmap_x, &full_bar[stage], c0, cw, chh, cn,
                                 static_cast<uint16_t>(kx), static_cast<uint16_t>(ky));
              tma_load_2d(smem_u32(b_smem + stage * H_BSTAGE), &tmap_w, &full_bar[stage], kb * HBK, nt * HBN);
            }
            __syncwarp();
            c0 += HBK;
            if (c0 >= p.Cin) { c0 = 0; ++tap; if (++kx == 3) { kx = 0; ++ky; } }
            if (++stage == H_STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 5) {
    // ================================================================ MMA issuer (main GEMM + deferred stage 2): every lane
    // walks the loops and waits, one elected lane issues (see elect_one in mf_common.cuh)
    {
      constexpr uint32_t idesc = umma_idesc_f16(HBM, HBN);
      constexpr uint32_t idesc2 = umma_idesc_f16(HBM, 32);
      const uint64_t a_d0 = umma_desc_sw128(smem_u32(a_smem)), b_d0 = umma_desc_sw128(smem_u32(b_smem));
      const uint64_t o_d0 = umma_desc_sw128(smem_u32(o_smem)), w2_d0 = umma_desc_sw128(smem_u32(w2_smem));
      int stage = 0, ti = 0;
      uint32_t phase = 0;
      auto stage2 = [&](int tj) {                                  // 1x1 contraction of the staged tile of global tile tj
        const int h = tj & 1, bcj = tj >> 1, buf = bcj & 1;        // ntn is even: tile parity == branch half
        if (h == 0) {
          mbar_wait(&d2_empty[buf], ((bcj >> 1) & 1) ^ 1);         // epilogue 2 has drained this D2 buffer
          mbar_wait(&w2_full[buf], (bcj >> 1) & 1);
        }
        mbar_wait(s2_full, tj & 1);
        tc_fence_after();
        const uint32_t d2 = tmem_base + H_TMEM_D2 + buf * 32;
        if (elect_one()) {
#pragma unroll
          for (int s = 0; s < 2; ++s)
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)
              umma_f16(d2, o_d0 + ((s * H_ASTAGE) >> 4) + 2 * k4,
                       w2_d0 + ((buf * H_W2 + (2 * h + s) * 32 * 128) >> 4) + 2 * k4, idesc2, (h | s | k4) != 0 ? 1u : 0u);
          umma_commit(s2_done);
          if (h == 1) { umma_commit(&d2_full[buf]); umma_commit(&w2_empty[buf]); }
        }
        __syncwarp();
      };
      for (int mt = blockIdx.x; mt < ntm; mt += gridDim.x) {
        for (int nt = 0; nt < ntn; ++nt, ++ti) {
          const int acc = ti & 1;
          mbar_wait(&acc_empty[acc], ((ti >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * HBN;
          for (int kb = 0; kb < nkb; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint64_t a_off = static_cast<uint64_t>((stage * H_ASTAGE) >> 4);
            const uint64_t b_off = static_cast<uint64_t>((stage * H_BSTAGE) >> 4);
            if (elect_one()) {
#pragma unroll
              for (int k4 = 0; k4 < HBK / 16; ++k4)
                umma_f16(d_tmem, a_d0 + a_off + 2 * k4, b_d0 + b_off + 2 * k4, idesc, (kb | k4) != 0 ? 1u : 0u);
              umma_commit(&empty_bar[stage]);
              if (kb == nkb - 1) umma_commit(&acc_full[acc]);
            }
            __syncwarp();
            if (++stage == H_STAGES) { stage = 0; phase ^= 1; }
          }
          if (ti >= 1) stage2(ti - 1);
        }
      }
      if (ti >= 1) stage2(ti - 1);
    }
  } else {
    // ================================================================ epilogue: warps 6-9 = group 0, warps 0-3 = group 1
    const int group = warp < 4 ? 1 : 0;
    const int et = group * 128 + (warp & 3) * 32 + lane;   // group 0 covers et 0..127 (its warp & 3 spans 2,3,0,1)
    const int quad = warp & 3, row = quad * 32 + lane;
    const uint32_t sc_u = smem_u32(sc_s), sh_u = smem_u32(sh_s), o_u = smem_u32(o_smem);
    bool store_pending = false;
    int ti = 0;
    auto epilogue2 = [&](int tj, int mtj) {                // 1x1 outputs of the branch whose second half was tile tj
      if (group != 0) return;
      const int bcj = tj >> 1, buf = bcj & 1, br = (tj % ntn) >> 1;
      mbar_wait(&d2_full[buf], (bcj >> 1) & 1);
      tc_fence_after();
      uint32_t r[32];
      tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + H_TMEM_D2 + buf * 32, r);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&d2_empty[buf]);
      const int m = mtj * HBM + row;
      if (m < p.M) {
        const int img = m / HW, pix = m - img * HW;
        float* yp = p.out[br] + static_cast<long long>(img) * p.out_ctot[br] * HW + pix;
        const int nch = p.out_nch[br];
#pragma unroll
        for (int n = 0; n < 32; ++n)
          if (n < nch) yp[static_cast<long long>(n) * HW] = __uint_as_float(r[n]) + __ldg(p.bias2 + br * 32 + n);
      }
    };
    int prev_mt = 0;
    for (int mt = blockIdx.x; mt < ntm; mt += gridDim.x) {
      for (int nt = 0; nt < ntn; ++nt, ++ti) {
        const int acc = ti & 1, br = nt >> 1, n0 = nt * HBN;
        if (store_pending && et == 0) bulk_wait_read0();
        if (et < HBN) {
          sts32f(sc_u + et * 4, __ldg(p.scale + n0 + et));
          sts32f(sh_u + et * 4, __ldg(p.shift + n0 + et));
        }
        bar_sync_named(1, 256);
        mbar_wait(&acc_full[acc], (ti >> 1) & 1);
        tc_fence_after();
        // this group converts two of the four 32-column chunks: group 0 -> chunks 0, 2; group 1 -> chunks 1, 3
        float v[2][32];
#pragma unroll
        for (int c2 = 0; c2 < 2; ++c2) {
          const int ch = c2 * 2 + group;
          uint32_t r[32];
          tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * HBN + ch * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 s4 = lds128f(sc_u + (ch * 32 + i) * 4), h4 = lds128f(sh_u + (ch * 32 + i) * 4);
            float t0 = __uint_as_float(r[i]) * s4.x + h4.x, t1 = __uint_as_float(r[i + 1]) * s4.y + h4.y;
            float t2 = __uint_as_float(r[i + 2]) * s4.z + h4.z, t3 = __uint_as_float(r[i + 3]) * s4.w + h4.w;
            v[c2][i] = fmaxf(t0, 0.01f * t0); v[c2][i + 1] = fmaxf(t1, 0.01f * t1);     // leaky_relu(0.01)
            v[c2][i + 2] = fmaxf(t2, 0.01f * t2); v[c2][i + 3] = fmaxf(t3, 0.01f * t3);
          }
        }
        tc_fence_before();
        mbar_arrive(&acc_empty[acc]);                          // accumulator is in registers: hand it back
        if (ti >= 1) mbar_wait(s2_done, (ti - 1) & 1);         // stage 2 of the previous tile no longer reads the staging
        __half* hid_row = nullptr;                             // this thread's pixel is one the edge fusion will gather
        if (p.hid_mask != nullptr && p.hid_col[br] >= 0) {
          const int m = mt * HBM + row;
          if (m < p.M && __ldg(p.hid_mask + m))
            hid_row = p.hid + static_cast<long long>(m) * p.hid_ld + p.hid_col[br] + (nt & 1) * HBN;
        }
#pragma unroll
        for (int c2 = 0; c2 < 2; ++c2) {
          const int ch = c2 * 2 + group;
          const uint32_t sub = o_u + (ch >> 1) * H_ASTAGE;
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            __half2 o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) o[e] = __floats2half2_rn(v[c2][i + 2 * e], v[c2][i + 2 * e + 1]);
            sts128(sub + sw128_off(row, (ch & 1) * 4 + (i >> 3)), *reinterpret_cast<uint4*>(o));
            if (hid_row != nullptr) *reinterpret_cast<uint4*>(hid_row + ch * 32 + i) = *reinterpret_cast<uint4*>(o);
          }
        }
        fence_proxy_async();
        bar_sync_named(1, 256);
        if (et == 0) {
          store_pending = false;
          if (p.hid_col[br] >= 0 && p.hid_mask == nullptr) {   // unmasked: store the whole tile of hidden activations
            const int col = p.hid_col[br] + (nt & 1) * HBN;
            tma_store_2d(&tmap_hid, o_u, col, mt * HBM);
            tma_store_2d(&tmap_hid, o_u + H_ASTAGE, col + 64, mt * HBM);
            bulk_commit();
            store_pending = true;
          }
          mbar_arrive(s2_full);
        }
        // the previous tile closed a branch: its 1x1 result is complete once stage2(ti-1) (issued after this tile's main
        // MMAs) has run - it has, or is about to: wait on d2_full
        if (ti >= 1 && ((ti - 1) & 1) == 1) epilogue2(ti - 1, (nt == 0) ? prev_mt : mt);
      }
      prev_mt = mt;
    }
    if (ti >= 1) epilogue2(ti - 1, prev_mt);
    if (store_pending && et == 0) bulk_wait0();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encTiledH)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_encIm2colH)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static void* driver_fn(const char* name) {
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint(name, &ptr, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess)
    return nullptr;
  return ptr;
}

// x: features [B*H*W, x_ld] fp16 (Cin channels used); w3: packed 3x3 weights [nbranch*256, 9*Cin]; w2: packed 1x1 weights
// [nbranch*32, 256]; hid: [M, hid_ld] fp16 buffer receiving the hidden activations of the branches with hid_col >= 0.
int launch_head_fused(const __half* x, int x_ld, int B, int H, int W, int Cin, const __half* w3, const __half* w2,
                      const float* scale, const float* shift, const float* bias2, int nbranch, float* const* out,
                      const int* out_ctot, const int* out_nch, const int* hid_col, __half* hid, int hid_ld,
                      const unsigned char* hid_mask, cudaStream_t st) {
  static PFN_encTiledH enc = reinterpret_cast<PFN_encTiledH>(driver_fn("cuTensorMapEncodeTiled"));
  static PFN_encIm2colH enc2 = reinterpret_cast<PFN_encIm2colH>(driver_fn("cuTensorMapEncodeIm2col"));
  if (!enc || !enc2) { set_error("head_fused: tensor-map driver entry points unavailable"); return -1; }
  if (Cin % 64 != 0 || nbranch < 1 || nbranch > H_MAXBR || x_ld % 8 != 0 || hid_ld % 8 != 0) {
    set_error("head_fused: unsupported shape Cin=%d nbranch=%d", Cin, nbranch);
    return -1;
  }
  HeadParams p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.H = H; p.W = W; p.Cin = Cin; p.M = B * H * W; p.nkb = 9 * Cin / 64; p.nbranch = nbranch;
  p.scale = scale; p.shift = shift; p.bias2 = bias2;
  p.hid = hid; p.hid_ld = hid_ld; p.hid_mask = hid_mask;
  for (int i = 0; i < nbranch; ++i) {
    p.out[i] = out[i]; p.out_ctot[i] = out_ctot[i]; p.out_nch[i] = out_nch[i]; p.hid_col[i] = hid_col[i];
    if (out_nch[i] > 32) { set_error("head_fused: branch %d has %d > 32 output channels", i, out_nch[i]); return -1; }
  }
  CUtensorMap tx, tw, tw2, th;
  {
    cuuint64_t gdim[4] = {static_cast<cuuint64_t>(Cin), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(B)};
    cuuint64_t gstr[3] = {static_cast<cuuint64_t>(x_ld) * 2, static_cast<cuuint64_t>(x_ld) * 2 * W, static_cast<cuuint64_t>(x_ld) * 2 * W * H};
    int lower[2] = {-1, -1}, upper[2] = {-1, -1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if (enc2(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(x), gdim, gstr, lower, upper, 64, HBM, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) { set_error("head_fused: im2col map failed"); return -1; }
  }
  auto tiled2d = [&](CUtensorMap* m, const void* ptr, int inner, int rows, int ld_elems, int box_inner, int box_rows) {
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(inner), static_cast<cuuint64_t>(rows)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld_elems) * 2};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(box_inner), static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  };
  const int K3 = 9 * Cin;
  if (!tiled2d(&tw, w3, K3, nbranch * 256, K3, 64, HBN) || !tiled2d(&tw2, w2, 256, nbranch * 32, 256, 64, 32) ||
      !tiled2d(&th, hid, hid_ld, p.M, hid_ld, 64, HBM)) { set_error("head_fused: tiled tensor map failed"); return -1; }
  static bool attr = false;
  if (!attr) {
    if (check_cuda(cudaFuncSetAttribute(head_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, H_SMEM), "head smem")) return -1;
    attr = true;
  }
  int dev = 0, nsm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  const int ntm = (p.M + HBM - 1) / HBM;
  const int grid = ntm < nsm ? ntm : nsm;
  return check_cuda(launch_k(head_fused_kernel, dim3(grid), dim3(320), H_SMEM, st, tx, tw, tw2, th, p), "head_fused launch");
}

}  // namespace mf
