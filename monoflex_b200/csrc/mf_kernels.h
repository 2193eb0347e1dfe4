// Internal launcher declarations shared by the .cu files of libmonoflex_b200.so (not part of the public C ABI).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace mf {

enum { MODE_CONV = 0, MODE_DCN = 1, MODE_CONV_TMA = 2 };
enum { ACT_NONE = 0, ACT_RELU = 1, ACT_LEAKY = 2, ACT_OFFMASK = 3 };
enum { OUT_F16_NHWC = 0, OUT_F32_NHWC = 1, OUT_F32_NCHW = 2 };

struct IgemmParams {
  // A operand: NHWC fp16 activations, `x_ld` elements between consecutive pixels (>= Cin: channel-slice views)
  const __half* x;
  int x_ld;
  int B, H, W, Cin;
  int Ho, Wo, kh, kw, stride, pad;
  int M;        // B*Ho*Wo
  int K_real;   // kh*kw*Cin
  int nkb;      // ceil(K_real / 64)
  // DCN: per output pixel 18 offsets (dy,dx per tap) + 9 masks (already sigmoid-ed), fp32, row stride om_ld
  const float* offmask;
  int om_ld;
  // epilogue: y = act(acc*scale[n] + shift[n] (+ res[m,n]))
  int Cout;
  const float* scale;
  const float* shift;
  const __half* res;
  int res_ld;
  int act;
  int out_mode;
  void* y;
  int y_ld;
  // strict-precision ("split") operands: an fp32-grade value v is stored as two fp16 numbers hi = fp16(v), lo = fp16(v - hi)
  // in the same pixel row, the lo block `*_lo` elements after the hi block. split_in: A and the packed weights are split and
  // the K axis is the concatenation, per (tap, 64-channel chunk), of the three products A_hi W_hi, A_lo W_hi, A_hi W_lo
  // (K_real / nkb already count that tripling). split_out: the fp16 NHWC output (and the residual) are hi/lo pairs.
  int split_in, split_out;
  int x_lo, res_lo, y_lo;
  int cw;       // split_in: channels per chunk = min(Cin, 64)
  // pair schedule (set by launch_igemm2 for split_in on the im2col-TMA and DCN paths): per (tap, chunk) only TWO stages are filled,
  // (A_hi, W_hi) and (A_lo, W_lo), and the MMA warp issues the three products A_hi W_hi, A_lo W_hi, A_hi W_lo across them -
  // one third less operand traffic into shared memory than the K-concatenation (which loads A_hi and W_hi twice).
  // nkb then counts stage fills = 2 * taps * Cin / 64.
  int pair;
  // HEAD2 epilogue (strict-precision predictor, EPI == 2 instantiation): this GEMM is the nine 3x3 head branches (N = nbranch x 256,
  // 128-column tiles, IABN + leaky folded into scale / shift / act). Instead of storing the hidden tile, every epilogue thread
  // contracts its 32 fp32 hidden values with the branch's 1x1 head weights (fp32, <= 32 outputs) and writes the partial dot
  // products to plane (n_tile_in_branch * 4 + chunk) of `h2_part` [8][B][h2_ntot][Ho*Wo]; mf_head2_reduce sums the eight planes
  // in a fixed order (+ bias) into the fp32 NCHW cls / reg maps. The hidden pair rows are stored only for the branches the edge
  // fusion gathers (h2_hid_col >= 0) and only at the pixels flagged in h2_mask.
  const float* h2_w;             // [nbranch][32][256] fp32, rows >= h2_nch[b] unused
  float* h2_part;
  int h2_ntot;                   // channels of the combined output (cls + reg = 53)
  int h2_nch[12], h2_ch0[12], h2_hid_col[12];
  const unsigned char* h2_mask;
};

int igemm_block_n(int cout);
int launch_conv_wgrad_narrow(const __half* x, int x_ld, int B, int H, int W, const __half* dy, int dy_ld, int k, float* dw,
                             cudaStream_t st);
int launch_head2_reduce(const float* part, const float* bias, float* cls, float* reg, int B, int ncls, int nreg, int HW,
                        cudaStream_t st);
int launch_igemm2(const IgemmParams& p, const __half* wp, int n_pad, int k_pad, int mode, cudaStream_t st);
int launch_rows_conv(const __half* x, int B, int H, int W, int Cin, int in_npar, const __half* wp, int n_pad, int k_pad,
                     int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift, int act,
                     int out_planar, int out_npar, __half* y, int y_ld, cudaStream_t st, int in_mode = 0, int split_out = 0,
                     int y_lo = 0);
int launch_head_fused(const __half* x, int x_ld, int B, int H, int W, int Cin, const __half* w3, const __half* w2,
                      const float* scale, const float* shift, const float* bias2, int nbranch, float* const* out,
                      const int* out_ctot, const int* out_nch, const int* hid_col, __half* hid, int hid_ld,
                      const unsigned char* hid_mask, cudaStream_t st);
int launch_conv_wgrad(const __half* x, int x_ld, int B, int H, int W, int Cin, const __half* dy, int dy_ld, int Cout, int kh,
                      int kw, int stride, int pad_h, int pad_w, float* dw, cudaStream_t st);
int launch_simt_gemm(const IgemmParams& p, const __half* wp, int n_pad, int k_pad, int mode, cudaStream_t st);

}  // namespace mf
