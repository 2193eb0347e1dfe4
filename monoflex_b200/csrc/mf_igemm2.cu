// Persistent, warp-specialised implicit-GEMM convolution / fused DCNv2 for sm_100a (second generation of mf_igemm.cu).
//
//   D[m, n] = sum_k A[m, k] * Wp[n, k]      m = output pixel, n = output channel, k = (tap, cin) cin fastest
//
// One CTA per SM (two for the narrow-N stem tiles) loops over 128 x BLOCK_N output tiles, n fastest:
//   warps [0, NPW)        A producers. MODE_CONV: 16-byte cp.async gathers of the zero-padded taps into the 128B-swizzled
//                         K-major stage (Cin < 64 layers). MODE_DCN: per (pixel, tap) 4 neighbour NHWC vectors, fp32
//                         bilinear blend * mask, fp16, st.shared; a tile is an 8x16 pixel block so its neighbourhood
//                         stays L1-resident. MODE_CONV_TMA (Cin % 64 == 0): no producer warps at all - the TMA warp
//                         fetches each (tap, 64-channel) A block with ONE im2col-mode cp.async.bulk.tensor.4d (zero
//                         padding, strides and row/image wrap-around done by the TMA unit) and these warps become a
//                         second epilogue group.
//   warp NPW              weight tiles by TMA (cp.async.bulk.tensor.2d, SWIZZLE_128B), same mbarrier ring as A
//   warp NPW+1            single-thread tcgen05.mma (kind::f16) into one of TWO TMEM accumulators
//   warps [NPW+2, NPW+6)  epilogue: tcgen05.ld -> scale/shift (+residual) -> activation -> fp16 -> swizzled smem staging
//                         -> one TMA store per 64-channel sub-tile (fp32 NHWC / NCHW outputs: direct stores)
// The accumulator double buffer lets the epilogue of tile i overlap the main loop of tile i+1; the smem ring and the
// barriers persist across tiles, so the per-tile cost is the MMA time, not a pipeline fill + drain.
#include "mf_common.cuh"
#include "mf_kernels.h"

namespace mf {

static constexpr int BM = 128;
static constexpr int BK = 64;
static constexpr int A_STAGE = BM * BK * 2;   // 16 KB

// SPLIT: the fp16 NHWC output is a hi/lo pair (strict-precision mode): two staging tiles per 64-channel sub-tile, paid for
// with one pipeline stage (the K loop of a split layer is 3x longer, so the shallower ring costs nothing measurable).
// EPI (see igemm2_kernel): 1 = SPLIT doubles the staging, 2 = HEAD2 has no output staging at all.
template <int BLOCK_N, int MODE, int EPI = 0>
struct Cfg2 {
  static constexpr bool SPLIT = EPI == 1;
  static constexpr int STAGES0 = MODE == MODE_DCN ? 4 : (BLOCK_N >= 128 ? 5 : (BLOCK_N >= 64 ? 6 : (BLOCK_N >= 32 ? 5 : 6)));
  static constexpr int STAGES = (SPLIT && BLOCK_N >= 64) ? ((MODE == MODE_DCN && BLOCK_N < 128) ? STAGES0 : STAGES0 - 1) : STAGES0;
  static constexpr int A_REGION = STAGES * A_STAGE;
  static constexpr int LAG = BLOCK_N >= 64 ? 3 : (BLOCK_N >= 32 ? 3 : 4);   // cp.async groups in flight per producer thread
  static constexpr int CTAS_PER_SM = BLOCK_N >= 64 ? 1 : 2;
  static constexpr int B_STAGE = BLOCK_N * BK * 2;
  static constexpr int OUT_HALF = BLOCK_N >= 64 ? (BLOCK_N / 64) * A_STAGE : 0;     // staging of one fp16 tile
  static constexpr int OUT_STAGE = EPI == 2 ? 0 : (SPLIT ? 2 * OUT_HALF : OUT_HALF);
  static constexpr int BAR_BYTES = 384;                         // barriers + tmem ptr
  static constexpr int PRM_BYTES = MODE == MODE_DCN ? 9 * BM * 32 : 0;   // DCN sampling records
  static constexpr int SMEM = A_REGION + STAGES * B_STAGE + OUT_STAGE + BAR_BYTES + 2 * BLOCK_N * 4 + PRM_BYTES + 1024;
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
  static constexpr int ACC_COLS = BLOCK_N < 32 ? 32 : BLOCK_N;  // columns per accumulator
  static constexpr int TMEM_COLS = 2 * ACC_COLS;                // power of two >= 32 for every BLOCK_N used
};

template <int N>
MF_DEVINL void act_chunk(float (&v)[N], int act, int nb) {
  if (act == ACT_RELU) {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = fmaxf(v[i], 0.f);
  } else if (act == ACT_LEAKY) {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = fmaxf(v[i], 0.01f * v[i]);      // == v > 0 ? v : 0.01 v
  } else if (act == ACT_OFFMASK) {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = (nb + i >= 18) ? 1.f / (1.f + __expf(-v[i])) : v[i];
  }
}

// EPI: 0 = plain epilogue, 1 = SPLIT (staged hi/lo output tiles), 2 = HEAD2 (1x1 head contraction in the epilogue, see IgemmParams)
template <int BLOCK_N, int MODE, int NPW, int EPI>
__global__ void __launch_bounds__((NPW + 6) * 32, Cfg2<BLOCK_N, MODE, EPI>::CTAS_PER_SM)
igemm2_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_y,
              const __grid_constant__ CUtensorMap tmap_x, const IgemmParams p, const int use_tma_store) {
  constexpr bool PTILE = (MODE == MODE_DCN);            // m-tile = 16 x 8 patch of one image
  constexpr bool A_TMA = (MODE == MODE_CONV_TMA);
  constexpr int EPI_THREADS = A_TMA ? 128 + NPW * 32 : 128;
  constexpr bool SPLIT = EPI == 1;
  constexpr bool HEAD2 = EPI == 2;
  using C = Cfg2<BLOCK_N, MODE, EPI>;
  constexpr int STAGES = C::STAGES;
  constexpr int LAG = C::LAG;
  const bool split_out = SPLIT || p.split_out != 0;      // SPLIT == staged hi/lo tiles; narrow tiles store both halves directly
  constexpr int B_STAGE = C::B_STAGE;
  constexpr int NPT = NPW * 32;
  constexpr int RPP = NPT / 8;
  constexpr int PASSES = BM / RPP;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + C::A_REGION;
  uint8_t* o_smem = b_smem + STAGES * B_STAGE;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(o_smem + C::OUT_STAGE);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* acc_full = empty_bar + STAGES;     // [2]
  uint64_t* acc_empty = acc_full + 2;          // [2]
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* sc_s = reinterpret_cast<float*>(o_smem + C::OUT_STAGE + C::BAR_BYTES);
  float* sh_s = sc_s + BLOCK_N;
  uint8_t* prm_smem = reinterpret_cast<uint8_t*>(sh_s + BLOCK_N);      // MODE_DCN only: 9*128 sampling records (36 KB)

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);      // warp-uniform for the compiler as well
  const int lane = threadIdx.x & 31;
  const int ntn = (p.Cout + BLOCK_N - 1) / BLOCK_N;
  const int tiles_x = (p.W + 15) >> 4, tiles_y = (p.H + 7) >> 3;
  const int ntm = PTILE ? p.B * tiles_x * tiles_y : (p.M + BM - 1) / BM;
  const int ntiles = ntn * ntm;
  const int nkb = p.nkb;
  const int HoWo = p.Ho * p.Wo;

  if (warp == NPW && lane == 0) {
    tma_prefetch_desc(&tmap_w);
    if (use_tma_store) tma_prefetch_desc(&tmap_y);
    if (A_TMA) tma_prefetch_desc(&tmap_x);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], A_TMA ? 1 : NPT + 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&acc_full[a], 1);
      mbar_init(&acc_empty[a], EPI_THREADS);
    }
    fence_mbar_init();
  }
  if (warp == NPW + 1) tmem_alloc(tmem_ptr_smem, C::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // ================================================================ epilogue body (run by 1 or 2 warp groups)
  auto run_epilogue = [&](const int group, const int et) {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    constexpr int CHUNK = BLOCK_N >= 32 ? 32 : 16;
    constexpr int NCHUNK = BLOCK_N / CHUNK;
    constexpr int NGROUPS = EPI_THREADS / 128;
    const bool staged = use_tma_store != 0;             // host guarantees OUT_F16_NHWC && BLOCK_N >= 64
    const uint32_t sc_u = smem_u32(sc_s), sh_u = smem_u32(sh_s), o_u = smem_u32(o_smem);
    int ti = -1;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      ++ti;
      const int acc = ti & 1;
      const int n0 = (t % ntn) * BLOCK_N;
      const int m_tile = t / ntn;
      int m = m_tile * BM + row;
      bool mvalid = m < p.M;
      int tile_b = 0, tile_y0 = 0, tile_x0 = 0;
      if (PTILE) {
        tile_b = m_tile / (tiles_x * tiles_y);
        const int tile_t = m_tile - tile_b * (tiles_x * tiles_y);
        tile_y0 = (tile_t / tiles_x) << 3;
        tile_x0 = (tile_t % tiles_x) << 4;
        const int yy = tile_y0 + (row >> 4), xx = tile_x0 + (row & 15);
        mvalid = yy < p.H && xx < p.W;
        m = (tile_b * p.H + yy) * p.W + xx;
      }
      if (staged && et == 0) bulk_wait_read0();         // previous tile's TMA store has finished reading the staging
      if (et < BLOCK_N) {
        sts32f(sc_u + et * 4, __ldg(p.scale + n0 + et));
        sts32f(sh_u + et * 4, __ldg(p.shift + n0 + et));
      }
      bar_sync_named(1, EPI_THREADS);
      mbar_wait(&acc_full[acc], (ti >> 1) & 1);
      tc_fence_after();
      if (group >= NCHUNK) {                                        // nothing to read: hand the accumulator back
        tc_fence_before();
        mbar_arrive(&acc_empty[acc]);
      }
#pragma unroll
      for (int ch0 = 0; ch0 < NCHUNK; ch0 += NGROUPS) {
        const int ch = ch0 + group;
        if (ch >= NCHUNK) break;
        uint32_t r[CHUNK];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + acc * C::ACC_COLS + ch * CHUNK;
        if constexpr (CHUNK == 32) tmem_ld32(taddr, r); else tmem_ld16(taddr, r);
        tmem_ld_wait();
        if (ch + NGROUPS >= NCHUNK) {                    // last chunk of this thread: accumulator fully read
          tc_fence_before();
          mbar_arrive(&acc_empty[acc]);
        }
        const int nb = n0 + ch * CHUNK;
        float v[CHUNK];
#pragma unroll
        for (int i = 0; i < CHUNK; i += 4) {
          const float4 s4 = lds128f(sc_u + (ch * CHUNK + i) * 4);
          const float4 h4 = lds128f(sh_u + (ch * CHUNK + i) * 4);
          v[i] = __uint_as_float(r[i]) * s4.x + h4.x;
          v[i + 1] = __uint_as_float(r[i + 1]) * s4.y + h4.y;
          v[i + 2] = __uint_as_float(r[i + 2]) * s4.z + h4.z;
          v[i + 3] = __uint_as_float(r[i + 3]) * s4.w + h4.w;
        }
        if (p.res != nullptr && mvalid) {
          const __half* rp = p.res + static_cast<long long>(m) * p.res_ld + nb;
#pragma unroll
          for (int i = 0; i < CHUNK; i += 8) {
            if (nb + i < p.Cout) {
              const uint4 rv = __ldg(reinterpret_cast<const uint4*>(rp + i));
              const __half2* rh = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float2 f = __half22float2(rh[e]);
                v[i + 2 * e] += f.x;
                v[i + 2 * e + 1] += f.y;
              }
              if (split_out) {                                   // residual = hi + lo
                const uint4 rl = __ldg(reinterpret_cast<const uint4*>(rp + p.res_lo + i));
                const __half2* rlh = reinterpret_cast<const __half2*>(&rl);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 f = __half22float2(rlh[e]);
                  v[i + 2 * e] += f.x;
                  v[i + 2 * e + 1] += f.y;
                }
              }
            }
          }
        }
        act_chunk<CHUNK>(v, p.act, nb);
        if constexpr (HEAD2) {
          // ---- 1x1 heads of this branch on the fp32 hidden values of this thread's pixel (32 of the branch's 256 channels)
          const int branch = n0 >> 8, cin0 = (n0 & 255) + ch * CHUNK;            // 256 hidden channels per branch
          const int nout = p.h2_nch[branch];
          const int plane = cin0 >> 5;
          if (mvalid) {
            const int bimg = m / HoWo, pix = m - bimg * HoWo;
            float* dst = p.h2_part + ((static_cast<long long>(plane) * p.B + bimg) * p.h2_ntot + p.h2_ch0[branch]) * HoWo + pix;
            const float* wb = p.h2_w + static_cast<long long>(branch) * 32 * 256 + cin0;
            // two outputs per pass (the second row of an odd tail re-reads the first and is not stored): 16 independent
            // 16-byte weight loads in flight and four independent FMA chains per thread - the epilogue, not the tensor pipe,
            // is what the accumulator hand-over waits on once the MMA issue is tight
            for (int o = 0; o < nout; o += 2) {
              const float* wr0 = wb + o * 256;
              const float* wr1 = (o + 1 < nout) ? wr0 + 256 : wr0;
              float4 wa[CHUNK / 4], wc[CHUNK / 4];
#pragma unroll
              for (int i = 0; i < CHUNK / 4; ++i) {
                wa[i] = __ldg(reinterpret_cast<const float4*>(wr0) + i);
                wc[i] = __ldg(reinterpret_cast<const float4*>(wr1) + i);
              }
              float a0 = 0.f, a1 = 0.f, c0 = 0.f, c1 = 0.f;
#pragma unroll
              for (int i = 0; i < CHUNK / 4; i += 2) {
                a0 += v[4 * i] * wa[i].x + v[4 * i + 1] * wa[i].y + v[4 * i + 2] * wa[i].z + v[4 * i + 3] * wa[i].w;
                a1 += v[4 * i + 4] * wa[i + 1].x + v[4 * i + 5] * wa[i + 1].y + v[4 * i + 6] * wa[i + 1].z + v[4 * i + 7] * wa[i + 1].w;
                c0 += v[4 * i] * wc[i].x + v[4 * i + 1] * wc[i].y + v[4 * i + 2] * wc[i].z + v[4 * i + 3] * wc[i].w;
                c1 += v[4 * i + 4] * wc[i + 1].x + v[4 * i + 5] * wc[i + 1].y + v[4 * i + 6] * wc[i + 1].z + v[4 * i + 7] * wc[i + 1].w;
              }
              dst[static_cast<long long>(o) * HoWo] = a0 + a1;
              if (o + 1 < nout) dst[static_cast<long long>(o + 1) * HoWo] = c0 + c1;
            }
            // hidden pair rows for the edge fusion: two branches only, border pixels only
            const int hc = p.h2_hid_col[branch];
            if (hc >= 0 && p.h2_mask[m] != 0) {
              __half* yp = reinterpret_cast<__half*>(p.y) + static_cast<long long>(m) * p.y_ld + hc + cin0;
#pragma unroll
              for (int i = 0; i < CHUNK; i += 8) {
                __half2 o[4], l[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  o[e] = __floats2half2_rn(v[i + 2 * e], v[i + 2 * e + 1]);
                  const float2 h = __half22float2(o[e]);
                  l[e] = __floats2half2_rn(v[i + 2 * e] - h.x, v[i + 2 * e + 1] - h.y);
                }
                *reinterpret_cast<uint4*>(yp + i) = *reinterpret_cast<uint4*>(o);
                *reinterpret_cast<uint4*>(yp + p.y_lo + i) = *reinterpret_cast<uint4*>(l);
              }
            }
          }
        } else
        if (p.out_mode == OUT_F16_NHWC) {
          if (staged) {
            if constexpr (BLOCK_N >= 64) {
              const uint32_t sub = o_u + (ch >> 1) * A_STAGE;
#pragma unroll
              for (int i = 0; i < CHUNK; i += 8) {
                __half2 o[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) o[e] = __floats2half2_rn(v[i + 2 * e], v[i + 2 * e + 1]);
                sts128(sub + sw128_off(row, (ch & 1) * 4 + (i >> 3)), *reinterpret_cast<uint4*>(o));
                if constexpr (SPLIT) {
                  __half2 l[4];
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float2 h = __half22float2(o[e]);
                    l[e] = __floats2half2_rn(v[i + 2 * e] - h.x, v[i + 2 * e + 1] - h.y);
                  }
                  sts128(sub + C::OUT_HALF + sw128_off(row, (ch & 1) * 4 + (i >> 3)), *reinterpret_cast<uint4*>(l));
                }
              }
            }
          } else if (mvalid) {
            __half* yp = reinterpret_cast<__half*>(p.y) + static_cast<long long>(m) * p.y_ld + nb;
#pragma unroll
            for (int i = 0; i < CHUNK; i += 8) {
              if (nb + i < p.Cout) {
                __half2 o[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) o[e] = __floats2half2_rn(v[i + 2 * e], v[i + 2 * e + 1]);
                *reinterpret_cast<uint4*>(yp + i) = *reinterpret_cast<uint4*>(o);
                if (split_out) {
                  __half2 l[4];
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float2 h = __half22float2(o[e]);
                    l[e] = __floats2half2_rn(v[i + 2 * e] - h.x, v[i + 2 * e + 1] - h.y);
                  }
                  *reinterpret_cast<uint4*>(yp + p.y_lo + i) = *reinterpret_cast<uint4*>(l);
                }
              }
            }
          }
        } else if (mvalid) {
          if (p.out_mode == OUT_F32_NHWC) {
            float* yp = reinterpret_cast<float*>(p.y) + static_cast<long long>(m) * p.y_ld + nb;
#pragma unroll
            for (int i = 0; i < CHUNK; i += 4) {
              if (nb + i < p.y_ld) *reinterpret_cast<float4*>(yp + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            }
          } else {
            const int b = m / HoWo, pix = m - b * HoWo;
            float* yp = reinterpret_cast<float*>(p.y) + (static_cast<long long>(b) * p.y_ld + nb) * HoWo + pix;
#pragma unroll
            for (int i = 0; i < CHUNK; ++i) {
              if (nb + i < p.Cout) yp[static_cast<long long>(i) * HoWo] = v[i];
            }
          }
        }
      }
      if (staged) {
        fence_proxy_async();
        bar_sync_named(1, EPI_THREADS);
        if (et == 0) {
          if constexpr (BLOCK_N >= 64) {
#pragma unroll
            for (int sidx = 0; sidx < BLOCK_N / 64; ++sidx) {
              if (n0 + sidx * 64 < p.Cout) {
#pragma unroll
                for (int hl = 0; hl < (SPLIT ? 2 : 1); ++hl) {
                  const uint32_t src = smem_u32(o_smem + hl * C::OUT_HALF + sidx * A_STAGE);
                  const int col = n0 + sidx * 64 + hl * p.y_lo;
                  if (PTILE)
                    tma_store_4d(&tmap_y, src, col, tile_x0, tile_y0, tile_b);
                  else
                    tma_store_2d(&tmap_y, src, col, m_tile * BM);
                }
              }
            }
          }
          bulk_commit();
        }
      } else {
        bar_sync_named(1, EPI_THREADS);       // sc_s / sh_s are rewritten by the next tile
      }
    }
    if (staged && et == 0) bulk_wait0();                 // all stores complete before the CTA exits
  };

  if (warp < NPW && A_TMA) {
    run_epilogue(1, 128 + threadIdx.x);                   // second epilogue group (odd 32-column chunks)
  } else if (warp < NPW) {
    // ================================================================ A producers
    const int tid = threadIdx.x;
    const int j = tid & 7;
    const int rsub = tid >> 3;
    int it = 0;                       // running K-block counter (stage = it % STAGES)
    if (MODE == MODE_CONV) {
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int m0 = (t / ntn) * BM;
        int iy0[PASSES], ix0[PASSES];
        long long base[PASSES];
#pragma unroll
        for (int q = 0; q < PASSES; ++q) {
          const int m = m0 + q * RPP + rsub;
          if (m < p.M) {
            const int b = m / HoWo, rem = m - b * HoWo;
            const int oy = rem / p.Wo, ox = rem - oy * p.Wo;
            iy0[q] = oy * p.stride - p.pad;
            ix0[q] = ox * p.stride - p.pad;
            base[q] = (static_cast<long long>(b * p.H + iy0[q]) * p.W + ix0[q]) * p.x_ld;
          } else {
            iy0[q] = -100000; ix0[q] = -100000; base[q] = 0;
          }
        }
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(&empty_bar[s], ((it / STAGES) & 1) ^ 1);
          const int k = kb * BK + j * 8;
          int tap, c0;
          if (p.split_in) {                 // virtual K order: ((tap, chunk), which in {hi.Whi, lo.Whi, hi.Wlo}, channel)
            const int unit = k / p.cw, c = k - unit * p.cw;
            const int tc = unit / 3, which = unit - tc * 3;
            const int nch = p.Cin / p.cw;
            tap = tc / nch;
            c0 = (tc - tap * nch) * p.cw + c + (which == 1 ? p.x_lo : 0);
          } else {
            tap = k / p.Cin;
            c0 = k - tap * p.Cin;
          }
          const int ky = tap / p.kw, kx = tap - ky * p.kw;
          const bool kvalid = k < p.K_real;
          const long long koff = static_cast<long long>(ky * p.W + kx) * p.x_ld + c0;
          const uint32_t a_stage = smem_u32(a_smem + s * A_STAGE);
#pragma unroll
          for (int q = 0; q < PASSES; ++q) {
            const int r = q * RPP + rsub;
            const int iy = iy0[q] + ky, ix = ix0[q] + kx;
            const bool ok = kvalid && iy >= 0 && iy < p.H && ix >= 0 && ix < p.W;
            const __half* src = ok ? p.x + base[q] + koff : p.x;
            cp_async16_ca(a_stage + sw128_off(r, j), src, ok ? 16u : 0u);
          }
          cp_async_commit();
          if (it >= LAG) {
            cp_async_wait<LAG>();
            fence_proxy_async();
            mbar_arrive(&full_bar[(it - LAG) % STAGES]);
          }
        }
      }
      cp_async_wait<0>();
      fence_proxy_async();
      for (int i = (it > LAG ? it - LAG : 0); i < it; ++i) mbar_arrive(&full_bar[i % STAGES]);
    } else {
      // ---------------------------------------------------------- DCNv2 (3x3, stride 1, pad 1, dil 1, dg 1)
      // Phase P, once per tile: every (pixel, tap) gets its sampling record - 4 bilinear weights already multiplied by
      // the modulation mask (0 for corners / samples outside the image, dcn_v2_im2col_cuda.cu:37-48,180) and the 4
      // corner pixel indices (clamped, so the gather needs no predication). The reference recomputes this per channel;
      // the first version of this kernel per 8-channel chunk. Phase G then is pure load / blend / store.
      const uint32_t prm_w = smem_u32(prm_smem);                    // [9*128] float4 weights
      const uint32_t prm_o = prm_w + 9 * BM * 16;                    // [9*128] int4 corner pixel indices
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int m_tile = t / ntn;
        const int tile_b = m_tile / (tiles_x * tiles_y);
        const int tile_t = m_tile - tile_b * (tiles_x * tiles_y);
        const int tile_y0 = (tile_t / tiles_x) << 3, tile_x0 = (tile_t % tiles_x) << 4;
        bar_sync_named(2, NPT);                              // previous tile's gather no longer reads the records
        for (int item = tid; item < 9 * BM; item += NPT) {
          const int tap = item >> 7, r = item & (BM - 1);
          const int yy = tile_y0 + (r >> 4), xx = tile_x0 + (r & 15);
          float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
          int4 o = make_int4(0, 0, 0, 0);
          if (yy < p.H && xx < p.W) {
            const float* om = p.offmask + (static_cast<long long>(tile_b * p.H + yy) * p.W + xx) * p.om_ld;
            const int ky = tap / 3, kx = tap - ky * 3;
            const float h_im = static_cast<float>(yy - 1 + ky) + __ldg(om + 2 * tap);
            const float w_im = static_cast<float>(xx - 1 + kx) + __ldg(om + 2 * tap + 1);
            if (h_im > -1.f && w_im > -1.f && h_im < static_cast<float>(p.H) && w_im < static_cast<float>(p.W)) {
              const float mk = __ldg(om + 18 + tap);
              const float hlf = floorf(h_im), wlf = floorf(w_im);
              const float lh = h_im - hlf, lw = w_im - wlf, hh = 1.f - lh, hw = 1.f - lw;
              const int hl = static_cast<int>(hlf), wl = static_cast<int>(wlf), hi = hl + 1, wi = wl + 1;
              const bool tp = hl >= 0, bt = hi <= p.H - 1, lf = wl >= 0, rt = wi <= p.W - 1;
              w.x = (tp && lf) ? hh * hw * mk : 0.f;
              w.y = (tp && rt) ? hh * lw * mk : 0.f;
              w.z = (bt && lf) ? lh * hw * mk : 0.f;
              w.w = (bt && rt) ? lh * lw * mk : 0.f;
              const int hlc = max(hl, 0), hic = min(hi, p.H - 1), wlc = max(wl, 0), wic = min(wi, p.W - 1);
              const int pb = p.x_ld * 2;                      // bytes per pixel: records hold 32-bit BYTE offsets
              o = make_int4((hlc * p.W + wlc) * pb, (hlc * p.W + wic) * pb, (hic * p.W + wlc) * pb, (hic * p.W + wic) * pb);
            }
          }
          sts128f(prm_w + item * 16, w);
          sts128(prm_o + item * 16, make_uint4(o.x, o.y, o.z, o.w));
        }
        bar_sync_named(2, NPT);
        const char* x_img = reinterpret_cast<const char*>(p.x + static_cast<long long>(tile_b) * p.H * p.W * p.x_ld + j * 8);
        int tap = 0, c0 = 0;
        uint32_t dst_off[PASSES];
#pragma unroll
        for (int q = 0; q < PASSES; ++q) dst_off[q] = sw128_off(q * RPP + rsub, j);
        if constexpr (SPLIT) {
          // strict precision: hi and lo halves of the four corners are blended in fp32 ONCE per (tap, 64-channel chunk) and
          // fill the two stages of the pair schedule (see IgemmParams::pair): hi, then lo.
          const int lo_bytes = p.x_lo * 2;
          for (int kb = 0; kb < nkb; kb += 2) {
            const char* xb = x_img + c0 * 2;
            const uint32_t rec = (tap * BM + rsub) * 16;
            uint4 hi4[PASSES], lo4[PASSES];
#pragma unroll
            for (int q = 0; q < PASSES; ++q) {
              const float4 wq = lds128f(prm_w + rec + q * RPP * 16);
              const uint4 o = lds128(prm_o + rec + q * RPP * 16);
              uint4 vh[4], vl[4];
              vh[0] = __ldg(reinterpret_cast<const uint4*>(xb + o.x));
              vh[1] = __ldg(reinterpret_cast<const uint4*>(xb + o.y));
              vh[2] = __ldg(reinterpret_cast<const uint4*>(xb + o.z));
              vh[3] = __ldg(reinterpret_cast<const uint4*>(xb + o.w));
              vl[0] = __ldg(reinterpret_cast<const uint4*>(xb + o.x + lo_bytes));
              vl[1] = __ldg(reinterpret_cast<const uint4*>(xb + o.y + lo_bytes));
              vl[2] = __ldg(reinterpret_cast<const uint4*>(xb + o.z + lo_bytes));
              vl[3] = __ldg(reinterpret_cast<const uint4*>(xb + o.w + lo_bytes));
              const float wv[4] = {wq.x, wq.y, wq.z, wq.w};
              // the lo halves are 2^-11 of the value: their blend needs 11 bits only and runs in packed fp16 (HFMA2, no
              // conversions, error 2^-22 of the value); the hi halves are blended in fp32 with the fp32 weights
              __half2 wh2[4];
#pragma unroll
              for (int cn = 0; cn < 4; ++cn) wh2[cn] = __float2half2_rn(wv[cn]);
              __half2* oh = reinterpret_cast<__half2*>(&hi4[q]);
              __half2* ol = reinterpret_cast<__half2*>(&lo4[q]);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                unsigned long long acc = f2_pack(0.f, 0.f);
                __half2 lacc = __hmul2(wh2[0], reinterpret_cast<const __half2*>(&vl[0])[e]);
#pragma unroll
                for (int cn = 0; cn < 4; ++cn) {
                  const float2 fh = __half22float2(reinterpret_cast<const __half2*>(&vh[cn])[e]);
                  const unsigned long long w2 = f2_pack(wv[cn], wv[cn]);
                  acc = f2_fma(w2, f2_pack(fh.x, fh.y), acc);
                  if (cn > 0) lacc = __hfma2(wh2[cn], reinterpret_cast<const __half2*>(&vl[cn])[e], lacc);
                }
                float2 r2 = f2_unpack(acc);
                const float2 lf = __half22float2(lacc);
                r2.x += lf.x;
                r2.y += lf.y;
                oh[e] = __floats2half2_rn(r2.x, r2.y);
                const float2 hf = __half22float2(oh[e]);
                ol[e] = __floats2half2_rn(r2.x - hf.x, r2.y - hf.y);
              }
            }
#pragma unroll
            for (int which = 0; which < 2; ++which) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              const uint32_t a_stage = smem_u32(a_smem + stage * A_STAGE);
#pragma unroll
              for (int q = 0; q < PASSES; ++q) sts128(a_stage + dst_off[q], which == 1 ? lo4[q] : hi4[q]);
              fence_proxy_async();
              mbar_arrive(&full_bar[stage]);
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            c0 += BK;
            if (c0 >= p.Cin) { c0 = 0; ++tap; }
          }
        } else
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          const uint32_t a_stage = smem_u32(a_smem + stage * A_STAGE);
          uint4 v[PASSES][4];
          float4 wq[PASSES];
          const char* xb = x_img + c0 * 2;
          const uint32_t rec = (tap * BM + rsub) * 16;
#pragma unroll
          for (int q = 0; q < PASSES; ++q) {               // all loads of the K block first (memory-level parallelism)
            wq[q] = lds128f(prm_w + rec + q * RPP * 16);
            const uint4 o = lds128(prm_o + rec + q * RPP * 16);
            v[q][0] = __ldg(reinterpret_cast<const uint4*>(xb + o.x));
            v[q][1] = __ldg(reinterpret_cast<const uint4*>(xb + o.y));
            v[q][2] = __ldg(reinterpret_cast<const uint4*>(xb + o.z));
            v[q][3] = __ldg(reinterpret_cast<const uint4*>(xb + o.w));
          }
#pragma unroll
          for (int q = 0; q < PASSES; ++q) {
            const __half2* h1 = reinterpret_cast<const __half2*>(&v[q][0]);
            const __half2* h2 = reinterpret_cast<const __half2*>(&v[q][1]);
            const __half2* h3 = reinterpret_cast<const __half2*>(&v[q][2]);
            const __half2* h4 = reinterpret_cast<const __half2*>(&v[q][3]);
            const unsigned long long w1 = f2_pack(wq[q].x, wq[q].x), w2 = f2_pack(wq[q].y, wq[q].y);
            const unsigned long long w3 = f2_pack(wq[q].z, wq[q].z), w4 = f2_pack(wq[q].w, wq[q].w);
            __half2 o2[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {                  // two channels per FFMA2 (packed fp32 math of sm_100)
              const float2 f1 = __half22float2(h1[e]), f2 = __half22float2(h2[e]);
              const float2 f3 = __half22float2(h3[e]), f4 = __half22float2(h4[e]);
              unsigned long long acc = f2_mul(w1, f2_pack(f1.x, f1.y));
              acc = f2_fma(w2, f2_pack(f2.x, f2.y), acc);
              acc = f2_fma(w3, f2_pack(f3.x, f3.y), acc);
              acc = f2_fma(w4, f2_pack(f4.x, f4.y), acc);
              const float2 r2 = f2_unpack(acc);
              o2[e] = __floats2half2_rn(r2.x, r2.y);
            }
            sts128(a_stage + dst_off[q], *reinterpret_cast<uint4*>(o2));
          }
          fence_proxy_async();
          mbar_arrive(&full_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
          c0 += BK;
          if (c0 >= p.Cin) { c0 = 0; ++tap; }
        }
      }
    }
  } else if (warp == NPW) {
    // ================================================================ weight tiles (and MODE_CONV_TMA A boxes) by TMA (all
    // lanes walk, one issues)
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int n0 = (t % ntn) * BLOCK_N;
        int cw = 0, chh = 0, cn = 0;
        if (A_TMA) {                                    // coordinates of the tile's first output pixel in input space (incl. -pad)
          const int m0 = (t / ntn) * BM;
          cn = m0 / HoWo;
          const int rem = m0 - cn * HoWo;
          const int oy = rem / p.Wo, ox = rem - oy * p.Wo;
          cw = ox * p.stride - p.pad;
          chh = oy * p.stride - p.pad;
        }
        int c0 = 0, kx = 0, ky = 0;                     // running (tap, channel) cursor: no divisions in the K loop
        int which = 0;                                  // split_in: 0 = A_hi box, 1 = A_lo box of the same (tap, chunk)
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          const bool issuer = elect_one();
          if (issuer) mbar_arrive_expect_tx(&full_bar[stage], A_TMA ? A_STAGE + B_STAGE : B_STAGE);
          if (A_TMA) {
            if (issuer)
              tma_load_im2col_4d(smem_u32(a_smem + stage * A_STAGE), &tmap_x, &full_bar[stage], c0 + (which == 1 ? p.x_lo : 0),
                                 cw, chh, cn, static_cast<uint16_t>(kx), static_cast<uint16_t>(ky));
            if (!p.split_in || ++which == 2) {
              which = 0;
              c0 += BK;
              if (c0 >= p.Cin) {
                c0 = 0;
                if (++kx == p.kw) { kx = 0; ++ky; }
              }
            }
          }
          // weight K coordinate: plain / K-concatenation = K block kb; pair schedule = block 3*(kb/2) (W_hi) for the hi stage
          // and 3*(kb/2)+2 (W_lo) for the lo stage of the same (tap, chunk)
          const int wk = p.pair ? (3 * (kb >> 1) + ((kb & 1) << 1)) : kb;
          if (issuer) tma_load_2d(smem_u32(b_smem + stage * B_STAGE), &tmap_w, &full_bar[stage], wk * BK, n0);
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == NPW + 1) {
    // ================================================================ MMA issuer: every lane walks the loops and waits on
    // the barriers (warp-uniform control flow, descriptors in uniform registers), one elected lane issues (see elect_one)
    {
      constexpr uint32_t idesc = umma_idesc_f16(BM, BLOCK_N);
      // Descriptors are "base + small delta": everything except the 14-bit start-address field is loop invariant, and
      // the field is linear in the byte address, so the hot loop only does 64-bit adds.
      uint64_t a_d0[BK / 16];
      const uint32_t a0 = smem_u32(a_smem), b0 = smem_u32(b_smem);
#pragma unroll
      for (int k4 = 0; k4 < BK / 16; ++k4) a_d0[k4] = umma_desc_sw128(a0 + k4 * 32);
      const uint64_t b_d0 = umma_desc_sw128(b0);
      int stage = 0, ti = -1;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        ++ti;
        const int acc = ti & 1;
        mbar_wait(&acc_empty[acc], ((ti >> 1) & 1) ^ 1);          // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * C::ACC_COLS;
        if (p.pair) {
          // pair schedule: stage s0 = (A_hi, W_hi), stage s1 = (A_lo, W_lo) of one (tap, 64-channel chunk); three products
          for (int kb = 0; kb < nkb; kb += 2) {
            const int s0 = stage;
            mbar_wait(&full_bar[s0], phase);
            tc_fence_after();
            const uint64_t a0 = static_cast<uint64_t>((s0 * A_STAGE) >> 4), b0s = static_cast<uint64_t>((s0 * B_STAGE) >> 4);
            if (elect_one()) {
#pragma unroll
              for (int k4 = 0; k4 < BK / 16; ++k4)                                   // A_hi W_hi
                umma_f16(d_tmem, a_d0[k4] + a0, b_d0 + b0s + 2 * k4, idesc, (kb | k4) != 0 ? 1u : 0u);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
            const int s1 = stage;
            mbar_wait(&full_bar[s1], phase);
            tc_fence_after();
            const uint64_t a1 = static_cast<uint64_t>((s1 * A_STAGE) >> 4), b1s = static_cast<uint64_t>((s1 * B_STAGE) >> 4);
            if (elect_one()) {
#pragma unroll
              for (int k4 = 0; k4 < BK / 16; ++k4)                                   // A_lo W_hi
                umma_f16(d_tmem, a_d0[k4] + a1, b_d0 + b0s + 2 * k4, idesc, 1u);
#pragma unroll
              for (int k4 = 0; k4 < BK / 16; ++k4)                                   // A_hi W_lo
                umma_f16(d_tmem, a_d0[k4] + a0, b_d0 + b1s + 2 * k4, idesc, 1u);
              umma_commit(&empty_bar[s0]);
              umma_commit(&empty_bar[s1]);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        } else
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t a_off = static_cast<uint64_t>((stage * A_STAGE) >> 4);
          const uint64_t b_off = static_cast<uint64_t>((stage * B_STAGE) >> 4);
          if (elect_one()) {
#pragma unroll
            for (int k4 = 0; k4 < BK / 16; ++k4) {
              umma_f16(d_tmem, a_d0[k4] + a_off, b_d0 + b_off + 2 * k4, idesc, (kb | k4) != 0 ? 1u : 0u);
            }
            umma_commit(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) umma_commit(&acc_full[acc]);
        __syncwarp();
      }
    }
  } else {
    run_epilogue(0, (warp - (NPW + 2)) * 32 + lane);      // first epilogue group (even chunks, or all of them)
  }

  tc_fence_before();
  __syncthreads();
  if (warp == NPW + 1) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled2 encode_fn() {
  static PFN_encodeTiled2 fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess || ptr == nullptr) {
      set_error("cuTensorMapEncodeTiled entry point unavailable");
      return nullptr;
    }
    fn = reinterpret_cast<PFN_encodeTiled2>(ptr);
  }
  return fn;
}

typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                     CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                     CUtensorMapFloatOOBfill);

static PFN_encodeIm2col encode_im2col_fn() {
  static PFN_encodeIm2col fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess || ptr == nullptr) {
      set_error("cuTensorMapEncodeIm2col entry point unavailable");
      return nullptr;
    }
    fn = reinterpret_cast<PFN_encodeIm2col>(ptr);
  }
  return fn;
}

static int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int BLOCK_N, int MODE, int NPW, int EPI = 0>
static int launch2_cfg(const CUtensorMap& tw, const CUtensorMap& ty, const CUtensorMap& tx, const IgemmParams& p,
                       int use_tma_store, cudaStream_t st) {
  using C = Cfg2<BLOCK_N, MODE, EPI>;
  auto kern = igemm2_kernel<BLOCK_N, MODE, NPW, EPI>;
  static bool attr_set = false;
  if (!attr_set) {
    if (check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM), "smem attr")) return -1;
    attr_set = true;
  }
  const int ntn = (p.Cout + BLOCK_N - 1) / BLOCK_N;
  const int ntm = MODE == MODE_DCN ? p.B * ((p.H + 7) / 8) * ((p.W + 15) / 16) : (p.M + BM - 1) / BM;
  int grid = num_sms() * C::CTAS_PER_SM;
  if (grid > ntn * ntm) grid = ntn * ntm;
  return check_cuda(launch_k(kern, dim3(grid), dim3((NPW + 6) * 32), C::SMEM, st, tw, ty, tx, p, use_tma_store), "igemm2 launch");
}

// out[b, ch, pix] = bias[ch] + sum over the eight partial planes (fixed order: deterministic), ch < ncls -> cls, else reg
__global__ void head2_reduce_kernel(const float* __restrict__ part, const float* __restrict__ bias, float* __restrict__ cls,
                                    float* __restrict__ reg, int B, int ncls, int nreg, int HW) {
  const int ntot = ncls + nreg;
  const long long plane = static_cast<long long>(B) * ntot * HW;
  const long long i = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i >= plane) return;
  float4 s = __ldg(reinterpret_cast<const float4*>(part + i));
#pragma unroll
  for (int q = 1; q < 8; ++q) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(part + q * plane + i));
    s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
  }
  const long long row = i / HW;                       // HW % 4 == 0 is checked by the launcher: 4 elements share (b, ch)
  const int ch = static_cast<int>(row % ntot), b = static_cast<int>(row / ntot);
  const int pix = static_cast<int>(i - row * HW);
  const float bv = __ldg(bias + ch);
  s.x += bv; s.y += bv; s.z += bv; s.w += bv;
  float* dst = ch < ncls ? cls + (static_cast<long long>(b) * ncls + ch) * HW + pix
                         : reg + (static_cast<long long>(b) * nreg + (ch - ncls)) * HW + pix;
  *reinterpret_cast<float4*>(dst) = s;
}
int launch_head2_reduce(const float* part, const float* bias, float* cls, float* reg, int B, int ncls, int nreg, int HW,
                        cudaStream_t st) {
  if (HW % 4 != 0) { set_error("head2_reduce: H*W must be a multiple of 4"); return -1; }
  const long long n4 = static_cast<long long>(B) * (ncls + nreg) * HW / 4;
  (void)launch_k(head2_reduce_kernel, dim3(static_cast<unsigned>((n4 + 255) / 256)), dim3(256), 0, st, part, bias, cls, reg, B, ncls,
                 nreg, HW);
  return check_cuda(cudaGetLastError(), "head2_reduce");
}

int launch_igemm2(const IgemmParams& p, const __half* wp, int n_pad, int k_pad, int mode, cudaStream_t st) {
  PFN_encodeTiled2 enc = encode_fn();
  if (!enc) return -1;
  // HEAD2 tiles: 128 columns (1.39 ms at B = 8; 256-column tiles measured 1.56 ms)
  const int bn = p.h2_w != nullptr ? 128 : igemm_block_n(p.Cout);
  const bool store_ok = p.out_mode == OUT_F16_NHWC && bn >= 64 && (reinterpret_cast<uintptr_t>(p.y) & 15) == 0 && p.y_ld % 8 == 0;
  if (n_pad % bn != 0 || k_pad % BK != 0 || k_pad < p.nkb * BK) {
    set_error("igemm: packed weight shape [%d,%d] incompatible with block_n=%d nkb=%d", n_pad, k_pad, bn, p.nkb);
    return -1;
  }
  if (mode == MODE_DCN && (p.Cin % 64 != 0 || p.kh != 3 || p.kw != 3 || p.stride != 1 || p.pad != 1)) {
    set_error("dcn igemm: only 3x3 s1 p1 with Cin %% 64 == 0 is built (got Cin=%d)", p.Cin);
    return -1;
  }
  if (mode == MODE_DCN && (p.split_in != p.split_out || (p.split_in && p.out_mode != OUT_F16_NHWC))) {
    set_error("dcn igemm: strict precision needs split input AND split fp16 output");
    return -1;
  }
  if (p.split_in && (p.cw <= 0 || p.Cin % p.cw != 0 || (p.cw != 64 && 64 % p.cw != 0) || p.x_lo % 8 != 0)) {
    set_error("igemm: split input needs Cin %% 64 == 0 or Cin in {8,16,32} and an 8-aligned lo offset (Cin=%d cw=%d)", p.Cin, p.cw);
    return -1;
  }
  if (p.split_out && (p.out_mode != OUT_F16_NHWC || p.y_lo % 8 != 0 || (p.res != nullptr && p.res_lo % 8 != 0))) {
    set_error("igemm: split output needs fp16 NHWC rows and 8-aligned lo offsets");
    return -1;
  }
  if (mode == MODE_CONV && (p.Cin % 8 != 0 || p.x_ld % 8 != 0)) {
    set_error("conv igemm: Cin and pixel stride must be multiples of 8 (got %d, %d)", p.Cin, p.x_ld);
    return -1;
  }
  CUtensorMap tw, ty;
  {
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(k_pad), static_cast<cuuint64_t>(n_pad)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(k_pad) * 2};
    cuuint32_t box[2] = {BK, static_cast<cuuint32_t>(bn)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&tw, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(wp), gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(weights) failed (%d)", static_cast<int>(r)); return -1; }
  }
  int use_tma_store = 0;
  ty = tw;
  if (store_ok) {
    CUresult r;
    if (mode == MODE_DCN) {
      cuuint64_t gdim[4] = {static_cast<cuuint64_t>(p.Cout + (p.split_out ? p.y_lo : 0)), static_cast<cuuint64_t>(p.W),
                            static_cast<cuuint64_t>(p.H), static_cast<cuuint64_t>(p.B)};
      cuuint64_t gstr[3] = {static_cast<cuuint64_t>(p.y_ld) * 2, static_cast<cuuint64_t>(p.y_ld) * 2 * p.W,
                            static_cast<cuuint64_t>(p.y_ld) * 2 * p.W * p.H};
      cuuint32_t box[4] = {64, 16, 8, 1};
      cuuint32_t estr[4] = {1, 1, 1, 1};
      r = enc(&ty, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, p.y, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
      cuuint64_t gdim[2] = {static_cast<cuuint64_t>(p.Cout + (p.split_out ? p.y_lo : 0)), static_cast<cuuint64_t>(p.M)};
      cuuint64_t gstr[1] = {static_cast<cuuint64_t>(p.y_ld) * 2};
      cuuint32_t box[2] = {64, BM};
      cuuint32_t estr[2] = {1, 1};
      r = enc(&ty, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, p.y, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(output) failed (%d)", static_cast<int>(r)); return -1; }
    use_tma_store = 1;
  }
  // A operand by im2col-mode TMA whenever a K block is one (tap, 64-channel) box. Narrower boxes (Cin 8 / 16 / 32) are
  // request-bound inside the TMA unit (measured: the 7x7 stem 1.8x slower than the cp.async gather), so those layers stay on
  // the gather producers.
  CUtensorMap tx = tw;
  bool a_tma = false;
  IgemmParams pp = p;
  if (mode == MODE_CONV && p.Cin % 64 == 0 && (reinterpret_cast<uintptr_t>(p.x) & 15) == 0 && p.kw <= 16 && p.kh <= 16 &&
      p.stride <= 8) {
    PFN_encodeIm2col enc2 = encode_im2col_fn();
    if (!enc2) return -1;
    cuuint64_t gdim[4] = {static_cast<cuuint64_t>(p.Cin + (p.split_in ? p.x_lo : 0)), static_cast<cuuint64_t>(p.W),
                          static_cast<cuuint64_t>(p.H), static_cast<cuuint64_t>(p.B)};
    cuuint64_t gstr[3] = {static_cast<cuuint64_t>(p.x_ld) * 2, static_cast<cuuint64_t>(p.x_ld) * 2 * p.W,
                          static_cast<cuuint64_t>(p.x_ld) * 2 * p.W * p.H};
    int lower[2] = {-p.pad, -p.pad};
    int upper[2] = {p.pad - (p.kw - 1), p.pad - (p.kh - 1)};
    cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(p.stride), static_cast<cuuint32_t>(p.stride), 1};
    CUresult r = enc2(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(p.x), gdim, gstr, lower, upper, BK, BM, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeIm2col failed (%d)", static_cast<int>(r)); return -1; }
    a_tma = true;
  }
  if (p.split_in && (mode == MODE_DCN || a_tma)) {
    pp.pair = 1;                                                   // see IgemmParams::pair
    pp.nkb = 2 * p.kh * p.kw * (p.Cin / 64);
  }
  if (p.h2_w != nullptr) {                     // HEAD2 epilogue: the strict-precision predictor GEMM (see IgemmParams)
    if (!(a_tma && pp.pair && p.Cout % 256 == 0 && p.h2_part != nullptr && p.Cout / 256 <= 12)) {
      set_error("igemm2 HEAD2: needs the pair-schedule TMA path and Cout a multiple of 256");
      return -1;
    }
    return launch2_cfg<128, MODE_CONV_TMA, 4, 2>(tw, ty, tx, pp, 0, st);
  }
  if (p.split_out && use_tma_store) {          // staged hi/lo tiles: the SPLIT instantiations (N tiles of 64 / 128 only)
    if (mode == MODE_DCN && bn == 64) return launch2_cfg<64, MODE_DCN, 16, 1>(tw, ty, tx, pp, use_tma_store, st);
    if (mode == MODE_DCN && bn == 128) return launch2_cfg<128, MODE_DCN, 16, 1>(tw, ty, tx, pp, use_tma_store, st);
    if (a_tma && bn == 64) return launch2_cfg<64, MODE_CONV_TMA, 4, 1>(tw, ty, tx, pp, use_tma_store, st);
    if (a_tma && bn == 128) return launch2_cfg<128, MODE_CONV_TMA, 4, 1>(tw, ty, tx, pp, use_tma_store, st);
    if (bn == 64) return launch2_cfg<64, MODE_CONV, 4, 1>(tw, ty, tx, pp, use_tma_store, st);
    if (bn == 128) return launch2_cfg<128, MODE_CONV, 4, 1>(tw, ty, tx, pp, use_tma_store, st);
  }
  if (mode == MODE_DCN && p.split_in) { set_error("dcn igemm: strict precision needs the staged TMA-store epilogue"); return -1; }
  if (mode == MODE_DCN) {                      // 16 gather warps for 64 / 128-column tiles, 8 for Cout <= 32
    if (bn == 16) return launch2_cfg<16, MODE_DCN, 8>(tw, ty, tx, pp, use_tma_store, st);
    if (bn == 32) return launch2_cfg<32, MODE_DCN, 8>(tw, ty, tx, pp, use_tma_store, st);
    if (bn == 64) return launch2_cfg<64, MODE_DCN, 16>(tw, ty, tx, pp, use_tma_store, st);
    if (bn == 128) return launch2_cfg<128, MODE_DCN, 16>(tw, ty, tx, pp, use_tma_store, st);
  }
#define MF_DISPATCH2(BN)                                                                          \
  if (bn == BN) {                                                                                 \
    if (a_tma) return launch2_cfg<BN, MODE_CONV_TMA, 4>(tw, ty, tx, pp, use_tma_store, st);        \
    return launch2_cfg<BN, MODE_CONV, 4>(tw, ty, tx, pp, use_tma_store, st);                       \
  }
  MF_DISPATCH2(16)
  MF_DISPATCH2(32)
  MF_DISPATCH2(64)
  MF_DISPATCH2(128)
#undef MF_DISPATCH2
  set_error("igemm2: unsupported block_n %d", bn);
  return -1;
}

}  // namespace mf
