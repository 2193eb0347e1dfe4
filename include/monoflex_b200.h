/* libmonoflex_b200.so — C ABI of the B200-native MonoFlex hot path.
 *
 * Conventions (all entry points):
 *   - plain device pointers and sizes; no torch / ATen types. Every buffer (inputs, outputs, workspaces) is allocated
 *     and owned by the caller; the library never calls cudaMalloc on the hot path and keeps no global device state.
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that stream.
 *   - return value 0 = success, negative = error; mf_last_error() returns the thread-local message
 *     (the Python host raises RuntimeError, mirroring AT_ASSERTM/AT_ERROR -> RuntimeError in the reference,
 *     /root/reference/model/backbone/DCNv2/src/dcn_v2.h:25-45).
 *   - internal activation layout is NHWC fp16 ("pixel rows"): `*_ld` is the element stride between consecutive pixels,
 *     so a tensor may be a channel slice of a wider buffer (used to write Root/concat inputs in place).
 *
 * Each entry point names the reference interface it replaces.
 */
#ifndef MONOFLEX_B200_H
#define MONOFLEX_B200_H
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library state ------------------------------------------------------------------------------------------ */
const char* mf_last_error(void);
int mf_version(void);
/* 0 = tcgen05 tensor-core implicit GEMM (default, the product), 1 = CUDA-core cross-check kernels (diagnostics). */
int mf_set_conv_impl(int impl);
/* N tile (16/32/64/128) the conv kernels use for `cout`; packed weights / scale / shift are padded to a multiple. */
int mf_conv_block_n(int cout);

/* ---- activation codes / output modes ------------------------------------------------------------------------ */
#define MF_ACT_NONE 0
#define MF_ACT_RELU 1
#define MF_ACT_LEAKY 2   /* leaky_relu 0.01 (InPlaceABN, detector_predictor.py:50,74) */
#define MF_ACT_OFFMASK 3 /* channels >= 18 -> sigmoid (DCN.forward dcn_v2.py:119-122) */
#define MF_OUT_F16_NHWC 0
#define MF_OUT_F32_NHWC 1
#define MF_OUT_F32_NCHW 2

/* OIHW fp32 conv weight -> [n_pad, k_pad] fp16, k = (ky*kw + kx)*cin_pad + c, zero padded
 * (replaces the cuDNN/THC weight layouts behind nn.Conv2d and _ext, dla_dcn.py:70-98, dcn_v2.py:69-73). */
int mf_pack_conv_weight(const float* w_oihw, int Cout, int Cin, int kh, int kw, int cin_pad, int n_pad, int k_pad,
                        void* out_f16, void* stream);

/* Packed weights of the stride-1 DATA-GRADIENT convolution of a layer (torch autograd's conv backward w.r.t. the input,
 * what `losses.backward()` of engine/trainer.py:112 runs through cuDNN), straight from the layer's OIHW fp32 parameter:
 * dX = conv(dY, W^T rotated by 180 degrees, padding k-1-p); out[ci][tap' * cout_pad + co] = w[co][ci][taps-1-tap']. */
int mf_pack_conv_weight_dgrad(const float* w_oihw, int Cout, int Cin, int kh, int kw, int cout_pad, int n_pad, int k_pad,
                              void* out_f16, void* stream);

/* mf_pack_conv_weight for MANY tensors in one launch (training plans re-pack every weight from its live fp32 parameter at the
 * start of each step). descs_dev: DEVICE array of n descriptors of 5 int64 each: OIHW fp32 source pointer, fp16 destination
 * pointer, Cout | Cin << 32, (kh*kw) | cin_pad << 32, n_pad | k_pad << 32. */
int mf_pack_conv_weights_batched(const void* descs_dev, int n, void* stream);

/* Conv2d + per-channel affine (folded BatchNorm / bias) + optional residual + activation as one tcgen05 implicit GEMM.
 * Replaces nn.Conv2d -> BatchNorm2d -> (+=residual) -> ReLU chains: dla_dcn.py:84-98 (BasicBlock), :195-203 (Root),
 * :268-322 (base layers), DCN.conv_offset_mask dcn_v2.py:106-122 (MF_ACT_OFFMASK, MF_OUT_F32_NHWC, y_ld = 32),
 * head 3x3 + InPlaceABN detector_predictor.py:47-75 (MF_ACT_LEAKY), head 1x1 :52,:83 (MF_OUT_F32_NCHW).
 * y[m, n] = act(scale[n] * sum_k x[...] w[n, k] + shift[n] (+ res[m, n])); scale/shift have n_pad entries. */
int mf_conv2d_nhwc_f16(const void* x, int x_ld, int B, int H, int W, int Cin, const void* w_packed, int n_pad, int k_pad,
                       int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift,
                       const void* res, int res_ld, int act, int out_mode, void* y, int y_ld, void* stream);

/* Full-resolution stem convolutions (DLA base_layer 7x7 3->16, level0 3x3 16->16, level1 3x3/2 16->32,
 * dla_dcn.py:268-282) on "planar" tensors [B][H][G][W/npar][8] fp16 (G = Cin/8 channel planes x npar column parities):
 * every input row segment is loaded once by TMA and the taps are read through shifted no-swizzle UMMA descriptors, no
 * im2col copies. Cin in {8, 16}; stride 1 (in_npar 1) or 2 (in_npar 2, 3x3, pad 1). Cin = 8 weights are packed with kw
 * padded to 8. Output: planar for the next stem layer (out_planar = 1, out_npar 1 or 2) or NHWC rows (y_ld). */
int mf_conv2d_rows_f16(const void* x, int B, int H, int W, int Cin, int in_npar, const void* w_packed, int n_pad, int k_pad,
                       int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift, int act,
                       int out_planar, int out_npar, void* y, int y_ld, void* stream);

/* ---- Strict-precision ("split") operators: the reference computes in fp32 (dcn_v2_cuda.cu:58 `scalar_t = float`, cuDNN fp32
 * convs); one fp16 tensor-core pass per layer leaves 2-4e-3 end to end, above the 1e-3 parity contract. In strict mode every
 * activation / weight is an fp16 PAIR hi = fp16(v), lo = fp16(v - hi) (lo block `*_lo` elements after the hi block in the same
 * NHWC row) and a GEMM accumulates A_hi W_hi + A_lo W_hi + A_hi W_lo in fp32 (K axis tripled, weights packed by
 * mf_pack_conv_weight_split: k' = ((tap*nchunk + chunk)*3 + which)*cw + c, cw = min(Cin, 64)).
 * split_in: x (and w_packed) are pairs; split_out: the fp16 NHWC output and the residual are pairs (fp32 outputs are plain). */
int mf_pack_conv_weight_split(const float* w_oihw, int Cout, int Cin, int kh, int kw, int n_pad, int k_pad, void* out_f16,
                              void* stream);
int mf_conv2d_nhwc_f16x2(const void* x, int x_ld, int x_lo, int B, int H, int W, int Cin, const void* w_packed, int n_pad,
                         int k_pad, int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift,
                         const void* res, int res_ld, int res_lo, int act, int out_mode, void* y, int y_ld, int y_lo,
                         int split_in, int split_out, void* stream);
/* fused DCNv2 (mf_dcn_nhwc_f16) on pairs: corners of both halves are blended in fp32 once per (pixel, tap, 8 channels) */
int mf_dcn_nhwc_f16x2(const void* x, int x_ld, int x_lo, int B, int H, int W, int Cin, const float* offmask, int om_ld,
                      const void* w_packed, int n_pad, int k_pad, int Cout, const float* scale, const float* shift, int act,
                      void* y, int y_ld, int y_lo, void* stream);
/* Strict-precision predictor (detector_predictor.py:62-132 class head + regression heads): the nbranch 3x3 convs (Cin -> 256 each,
 * IABN + leaky folded into scale / shift / act) run as ONE pair GEMM with N = nbranch*256, and the 1x1 heads are contracted in
 * its epilogue from the fp32 accumulators (w2 [nbranch][32][256] fp32, branch b owns out_nch[b] <= 32 channels starting at
 * out_ch0[b] of the ntot = num_classes + num_reg combined maps). The epilogue writes partial sums to part [8][B][ntot][H*W] fp32
 * (8 = 256 hidden channels / 32 per epilogue thread); mf_head2_reduce adds the planes in a fixed order plus the bias into the
 * NCHW cls / reg maps, so results are run-to-run identical. Hidden pair rows reach HBM only for branches with hid_col[b] >= 0
 * (hi block at that column of `hid`, lo block hid_lo further) and only at pixels flagged in hid_mask (mf_edge_mask). */
int mf_head_conv_f16x2(const void* x, int x_ld, int x_lo, int B, int H, int W, int Cin, const void* w_packed, int n_pad, int k_pad,
                       int nbranch, const float* scale, const float* shift, int act, const float* w2, float* part, int ntot,
                       const int* out_nch, const int* out_ch0, const int* hid_col, void* hid, int hid_ld, int hid_lo,
                       const unsigned char* hid_mask, void* stream);
int mf_head2_reduce(const float* part, const float* bias, float* cls, float* reg, int B, int ncls, int nreg, int HW, void* stream);
/* Row-segment stem kernel (mf_conv2d_rows_f16) on pairs. in_mode 1 (Cin = 8): x is the image pair plane [hi3 | lo3 | 0 0]
 * (mf_pack_image_pair8) and w_packed holds TWO tap sets stacked along ky ([W_hi | W_hi | 0 0] then [W_lo | 0 ...], kw padded
 * to 8); in_mode 2 (Cin = 16, stride 1): x = pair planes [hi0 hi1 lo0 lo1], w_packed = THREE stacked tap sets (W_hi, W_hi,
 * W_lo). Output always a pair: planar (hi planes then lo planes) or NHWC rows with the lo block y_lo elements after hi. */
int mf_conv2d_rows_f16x2(const void* x, int B, int H, int W, int Cin, int in_npar, int in_mode, const void* w_packed, int n_pad,
                         int k_pad, int kh, int kw, int stride, int pad, int Cout, const float* scale, const float* shift, int act,
                         int out_planar, int out_npar, void* y, int y_ld, int y_lo, void* stream);
int mf_pack_image_pair8(const float* x_nchw, void* y_nhwc8, int B, int C, int H, int W, void* stream);
/* image [B,3,H,W] fp32 -> [B*H*W, 16] fp16 rows [hi3 | lo3 | hi3 | 0 x 7] (the stem then is a plain 16-channel conv with
 * per-tap weights [W_hi | W_hi | W_lo | 0]) */
int mf_pack_image_split(const float* x_nchw, void* y_rows16, int B, int C, int H, int W, void* stream);
int mf_maxpool2_split(const void* x, int x_lo, void* y, int y_lo, int B, int H, int W, int C, int x_ld, int y_ld, void* stream);
int mf_upsample_add_split(const void* x, int x_lo, const float* w_taps, const void* skip, int skip_lo, void* y, int y_lo, int B,
                          int Hi, int Wi, int C, int f, int x_ld, int skip_ld, int y_ld, void* stream);
/* edge fusion on pairs: ea / eb are [B, K+2, 512] rows = [hi 256 | lo 256] */
int mf_edge_gather_split(const void* feat, int feat_ld, int feat_lo, int ch_a, int ch_b, const long long* edge_idx, void* ea,
                         void* eb, int B, int H, int W, int K, int out_w, int out_h, void* stream);
int mf_edge_head_add_split(const void* t, int t_ld, int t_lo, const float* w, const float* bias, int n_out,
                           const long long* edge_idx, const long long* edge_len, float* out, int out_ctot, int out_ch0, int B,
                           int K, int H, int W, void* stream);
/* pair rows -> fp32 NCHW (hi + lo): feature-map export */
int mf_split_to_nchw_f32(const void* x, int x_ld, int x_lo, float* y, int B, int C, int HW, void* stream);

/* Fused predictor head (detector_predictor.py:121-135): `nbranch` shared-input 3x3 convs (Cin -> 256 each) + InPlaceABN
 * (scale/shift, leaky 0.01) + the 1x1 output convs of every branch in one persistent kernel; the 256-channel hidden
 * activations stay on chip (staged in smem as the A operand of a second tcgen05.mma) except for branches with
 * hid_col[i] >= 0, which are also stored to `hid` [B*H*W, hid_ld] at that column (edge fusion reads them).
 * w3_packed [nbranch*256, 9*Cin] fp16 (k = tap*Cin + c); w2_packed [nbranch*32, 256] fp16 (rows >= out_nch[i] zero);
 * bias2 [nbranch*32]; out_ptrs[i] = fp32 NCHW base pointer of branch i's first output channel (host array of device
 * pointers), out_ctot[i] = channel count of the tensor it points into, out_nch[i] <= 32 real channels.
 * hid_mask (nullable) [B*H*W] bytes: when given only pixels with a non-zero flag are stored to `hid` (mf_edge_mask marks the
 * border pixels the edge fusion gathers: ~830 of 30 720 per image, 245 MB less DRAM traffic per B = 8 forward). */
int mf_head_fused(const void* x, int x_ld, int B, int H, int W, int Cin, const void* w3_packed, const void* w2_packed,
                  const float* scale, const float* shift, const float* bias2, int nbranch, void* const* out_ptrs,
                  const int* out_ctot, const int* out_nch, const int* hid_col, void* hid, int hid_ld,
                  const unsigned char* hid_mask, void* stream);
/* mask[b, y, x] = 1 for every pixel mf_edge_gather reads for edge_idx [B, K, 2] (x, y), 0 elsewhere */
int mf_edge_mask(const long long* edge_idx, unsigned char* mask, int B, int K, int H, int W, int out_w, int out_h,
                 void* stream);

/* Fused DCNv2 (3x3, stride 1, pad 1, dilation 1, deformable_groups 1): bilinear gather of the modulated columns straight
 * into the MMA operand tile, contraction with the packed weights, affine (+bias, BN) and activation epilogue.
 * Replaces _ext.dcn_v2_forward + BatchNorm2d + ReLU of DeformConv (dla_dcn.py:384-396; src/cuda/dcn_v2_cuda.cu:42-172,
 * src/cuda/dcn_v2_im2col_cuda.cu:125-195) without the [B, 9C, HW] columns buffer.
 * offmask: [B*H*W, om_ld] fp32 rows = 18 offsets (dy,dx per tap) + 9 sigmoid-ed masks. */
int mf_dcn_nhwc_f16(const void* x, int x_ld, int B, int H, int W, int Cin, const float* offmask, int om_ld,
                    const void* w_packed, int n_pad, int k_pad, int Cout, const float* scale, const float* shift, int act,
                    int out_mode, void* y, int y_ld, void* stream);

/* ---- layout / HBM-bound kernels ----------------------------------------------------------------------------- */
/* images [B,C<=8,H,W] fp32 NCHW (engine/trainer.py:106, engine/inference.py:29) -> NHWC fp16 with 8 channels */
int mf_pack_image(const float* x_nchw, void* y_nhwc8, int B, int C, int H, int W, void* stream);
int mf_nchw_f32_to_nhwc_f16(const float* x, void* y, int B, int C, int HW, int y_ld, void* stream);
int mf_nhwc_f16_to_nchw_f32(const void* x, float* y, int B, int C, int HW, int x_ld, void* stream);
/* offset [B,18,H,W] + mask [B,9,H,W] (reference _ext layout) -> [B*HW, 32] fp32 rows */
int mf_pack_offmask(const float* offset, const float* mask, float* y, int B, int HW, void* stream);
/* nn.MaxPool2d(2) of Tree.downsample (dla_dcn.py:238) */
int mf_maxpool2_nhwc_f16(const void* x, void* y, int B, int H, int W, int C, int x_ld, int y_ld, void* stream);
/* depthwise ConvTranspose2d(k=2f, stride f, pad f/2) + skip add (IDAUp.forward dla_dcn.py:419-425).
 * w_taps: fp32 [k*k, C] */
int mf_upsample_add_nhwc_f16(const void* x, const float* w_taps, const void* skip, void* y, int B, int Hi, int Wi, int C,
                             int f, int x_ld, int skip_ld, int y_ld, void* stream);
/* edge fusion (detector_predictor.py:137-158): grid_sample of two 256-ch slices at the border pixels into two
 * replicate-padded Conv1d inputs [B, K+2, 256]; final Conv1d(256->n_out,k=1) + indexed add into an NCHW fp32 map. */
int mf_edge_gather(const void* feat, int feat_ld, int ch_a, int ch_b, const long long* edge_idx, void* ea, void* eb, int B,
                   int H, int W, int K, int out_w, int out_h, void* stream);
int mf_edge_head_add(const void* t, const float* w, const float* bias, int n_out, const long long* edge_idx,
                     const long long* edge_len, float* out, int out_ctot, int out_ch0, int B, int K, int H, int W,
                     void* stream);
/* sigmoid_hm (model/layers/utils.py:39-43), in place */
int mf_sigmoid_clamp(float* x, long long n, void* stream);
/* FocalLoss.forward (model/layers/focal_loss.py:35-55): out2[0] = loss sum, out2[1] = num_pos */
int mf_focal_loss_forward(const float* pred, const float* target, long long n, float* out2, void* stream);
/* autograd of the above: grad_pred[i] = scale[0] * dLoss/dpred[i]; scale is a DEVICE scalar
 * (loss weight / clamp(num_pos, 1), model/head/detector_loss.py:276) so the step needs no host sync */
int mf_focal_loss_backward(const float* pred, const float* target, long long n, const float* scale, float* grad_pred,
                           void* stream);

/* Convolution weight gradient (backward of `nn.Conv2d` in BasicBlock / Root / IDA nodes, model/backbone/dla_dcn.py:69-203):
 *   dw[co, ci, ky, kx] = sum_{b, oy, ox} dy[b, oy, ox, co] * x[b, oy*stride - pad + ky, ox*stride - pad + kx, ci]
 * x [B*H*W, x_ld], dy [B*Ho*Wo, dy_ld] fp16 NHWC rows; dw fp32 OIHW, overwritten. Cin, Cout multiples of 64, square kernel.
 * tcgen05 GEMM with MN-major operands fed by im2col / tiled TMA, split-K with fp32 atomics (summation order not fixed). */
int mf_conv2d_wgrad_nhwc_f16(const void* x, int x_ld, int B, int H, int W, int Cin, const void* dy, int dy_ld, int Cout, int k,
                             int stride, int pad, float* dw, void* stream);
/* same with a rectangular kernel / padding (the edge fusion's Conv1d(256, 256, 3) is a 1 x 3 convolution over [B, 1, K+2, 256]) */
int mf_conv2d_wgrad_rect_nhwc_f16(const void* x, int x_ld, int B, int H, int W, int Cin, const void* dy, int dy_ld, int Cout, int kh,
                                  int kw, int stride, int pad_h, int pad_w, float* dw, void* stream);

/* Backward twins of the HBM-bound layers (csrc/mf_bwd_misc.cu), NHWC fp16 rows unless noted:
 *  maxpool2_bwd: MaxPool2d(2) (dla_dcn.py:238); gradient to the first maximum of each window (torch arg-max order).
 *  upsample_bwd: depth-wise ConvTranspose2d(k = 2f, s = f, p = f/2) (dla_dcn.py:408-412): dx (nullable) and dw_taps [k*k, C]
 *                fp32 (nullable; needs mf_upsample_bwd_workspace bytes of scratch); the skip input's gradient is dy itself.
 *  sigmoid_clamp_bwd: sigmoid_hm (layers/utils.py:39-43), fp32: dx = dy * y (1 - y) where the clamp did not bind.
 *  column_sum: out[c] = sum over rows (conv-bias gradients); scratch mf_column_sum_workspace bytes.
 *  edge_gather_bwd: transpose of mf_edge_gather: ADDS the gradients of the two [B, K+2, 256] Conv1d inputs onto d_feat rows.
 *  interleave2x2: out[b, 2i+py, 2j+px] = p{py}{px}[b, i, j] (recombines the parity sub-convolutions of a stride-2 dgrad). */
int mf_maxpool2_bwd_nhwc_f16(const void* x, const void* dy, void* dx, int B, int H, int W, int C, int x_ld, int dy_ld, int dx_ld,
                             void* stream);
size_t mf_upsample_bwd_workspace(int B, int Hi, int Wi, int C, int f);
int mf_upsample_bwd_nhwc_f16(const void* x, const float* w_taps, const void* dy, void* dx, float* dw_taps, int B, int Hi, int Wi,
                             int C, int f, int x_ld, int dy_ld, int dx_ld, float* workspace, void* stream);
int mf_sigmoid_clamp_bwd(const float* y, const float* dy, float* dx, long long n, void* stream);
size_t mf_column_sum_workspace(long long M, int C);
int mf_column_sum_nhwc_f16(const void* x, int x_ld, long long M, int C, float* out, float* workspace, void* stream);
int mf_edge_gather_bwd(const void* d_ea, const void* d_eb, int ch_a, int ch_b, const long long* edge_idx, void* d_feat, int feat_ld,
                       int B, int H, int W, int K, int out_w, int out_h, void* stream);
/* backward of mf_edge_head_add: d_t [B, K, 256] fp16 (0 past edge_len), dw [n_out, 256] and dbias [n_out] fp32 (overwritten;
 * fp32 atomics), from d_out = gradient of the fp32 NCHW map the forward added into */
int mf_edge_head_add_bwd(const void* t, const float* w, int n_out, const long long* edge_idx, const long long* edge_len,
                         const float* d_out, int out_ctot, int out_ch0, void* d_t, float* dw, float* dbias, int B, int K, int H,
                         int W, void* stream);
/* dst[r, 0:C] += src[r, 0:C] on fp16 rows (gradient accumulation of activations with several consumers) */
int mf_add_rows_f16(void* dst, int dst_ld, const void* src, int src_ld, long long M, int C, void* stream);
int mf_interleave2x2_nhwc_f16(const void* p00, const void* p01, const void* p10, const void* p11, int part_ld, void* out, int out_ld,
                              int B, int Hh, int Wh, int C, void* stream);

/* Backward of the fused DCNv2 layer on the NHWC fp16 path (_DCNv2.backward dcn_v2.py:35-51; 3x3, stride 1, pad 1, one group).
 * The two GEMMs are existing kernels: gcol = 1x1 conv of dY with W^T (mf_conv2d_nhwc_f16), dW = mf_conv2d_wgrad_nhwc_f16
 * with k = 1 on `cols`. offmask: the forward's [M, om_ld >= 27] fp32 rows (18 offsets, 9 sigmoid-ed masks).
 *  sample_cols: cols[p, tap*C + c] = mask * bilinear sample (fp16 [M, 9C]) - the forward's operand tiles written out.
 *  col2im: dx (zeroed, then half2 atomics) and d_offmask [M, 32] fp32 = gradients of the offset conv's PRE-activation
 *          outputs (offsets; masks through m (1 - m)); gcol fp16 [M, 9C] (k = tap*C + c). */
int mf_dcn_sample_cols_nhwc_f16(const void* x, int x_ld, const float* offmask, int om_ld, void* cols, int B, int H, int W, int C,
                                void* stream);
int mf_dcn_col2im_nhwc_f16(const void* x, int x_ld, const float* offmask, int om_ld, const void* gcol, void* dx, int dx_ld,
                           float* d_offmask, int B, int H, int W, int C, void* stream);

/* Training-mode nn.BatchNorm2d(momentum 0.1) / InPlaceABN over NHWC fp16 rows (dla_dcn.py:76-79, detector_predictor.py:50,74;
 * eval mode is folded into the conv epilogues instead). x = raw conv output [M, x_ld], C channels (multiple of 8).
 * forward: batch mean / biased variance (deterministic two-level reduction), running-stat update like torch (unbiased
 *   variance, skipped when running_mean is NULL), y = act(x * scale + shift [+ res]); act 0 none / 1 ReLU / 2 leaky 0.01;
 *   abs_gamma = 1 uses |gamma| + eps (InPlaceABN). Outputs mean, rstd, scale, shift [C] are kept for the backward call.
 * backward: g = dy * act'(y); dgamma = sum g * xhat, dbeta = sum g; dx = scale * (g - mean(g) - xhat * mean(g * xhat));
 *   dres (nullable) receives g (gradient of the residual input).
 * workspace: mf_bn_train_workspace(M, C) bytes of device scratch. */
size_t mf_bn_train_workspace(long long M, int C);
int mf_bn_train_forward(const void* x, int x_ld, long long M, int C, const float* gamma, const float* beta, float eps,
                        float momentum, int abs_gamma, float* running_mean, float* running_var, const void* res, int res_ld,
                        int act, void* y, int y_ld, float* mean, float* rstd, float* scale, float* shift, float* workspace,
                        void* stream);
int mf_bn_train_backward(const void* x, int x_ld, const void* dy, int dy_ld, const void* y, int y_ld, long long M, int C,
                         const float* mean, const float* rstd, const float* scale, int act, void* dx, int dx_ld, void* dres,
                         int dres_ld, float* dgamma, float* dbeta, float* workspace, void* stream);

/* SyncBatchNorm (torch.nn.SyncBatchNorm after the reference's `convert_sync_batchnorm`, tools/plain_train_net.py:131-132): the
 * train-mode BatchNorm kernels split around the exchange. `sums` is a DEVICE double [2][C] buffer: *_stats writes the local
 * per-channel sums (forward: sum x, sum x^2; backward: sum g, sum g*xhat, plus the LOCAL dgamma / dbeta that DDP averages like any
 * gradient), the host all-reduces it (SUM, NCCL, same stream), *_apply normalises with `count` = the global number of elements per
 * channel. workspace: mf_bn_train_workspace(M, C) bytes. With one rank the pair equals mf_bn_train_forward / _backward. */
int mf_bn_sync_forward_stats(const void* x, int x_ld, long long M, int C, float* workspace, double* sums, void* stream);
int mf_bn_sync_forward_apply(const void* x, int x_ld, long long M, int C, const double* sums, double count, const float* gamma,
                             const float* beta, float eps, float momentum, int abs_gamma, float* running_mean, float* running_var,
                             const void* res, int res_ld, int act, void* y, int y_ld, float* mean, float* rstd, float* scale,
                             float* shift, void* stream);
int mf_bn_sync_backward_stats(const void* x, int x_ld, const void* dy, int dy_ld, const void* y, int y_ld, long long M, int C,
                              const float* mean, const float* rstd, int act, float* workspace, double* sums, float* dgamma,
                              float* dbeta, void* stream);
int mf_bn_sync_backward_apply(const void* x, int x_ld, const void* dy, int dy_ld, const void* y, int y_ld, long long M, int C,
                              const float* mean, const float* rstd, const float* scale, const double* sums, double count, int act,
                              void* dx, int dx_ld, void* dres, int dres_ld, float* workspace, void* stream);

/* diagnostics: D[128,128] = A^T B with A [64,128] and B [64,128] fp16 row-major (reduction index = rows), computed with
 * MN-major tcgen05 operand descriptors - the operand form the weight-gradient GEMM of the training path needs */
int mf_selftest_mn_major(const void* a_km, const void* b_kn, float* d_mn, void* stream);

/* Loss_Computation.__call__ (model/head/detector_loss.py:267-493, prepare_predictions :116-265, Real_MultiBin_loss
 * :495-517, IOULoss layers/iou_loss.py:12-49, decoders model/anno_encoder.py:88-295) for the runs/monoflex.yaml losses.
 *   pred_cls [B,ncls,H,W] sigmoid-ed heat map, hm [B,ncls,H,W] label heat map, pred_reg [B,50,H,W]       (device, fp32)
 *   obj [B*M, mf_loss_obj_cols()] packed per-object labels (device): 0 cls_id | 1-2 target_centers x,y | 3-6 2d_bboxes |
 *       7 reg_mask | 8 trunc_mask | 9-11 dimensions | 12-14 locations | 15 rotys | 16-17 offset_3D | 18-25 orientations |
 *       26-28 keypoints_depth_mask | 29-58 keypoints 10 x (x, y, visible)        (data/datasets/kitti.py:496-521)
 *   img [B,8] (device): f_u f_v c_u c_v b_x b_y pad_x pad_y;  weights11 / dim_mean9: HOST arrays (INIT_LOSS_WEIGHT in
 *       LOSS_NAMES order runs/monoflex.yaml:45-47, DIMENSION_MEAN config/defaults.py:206-208)
 *   out48 (device): [0..10] the 11 losses in LOSS_NAMES order; [16..26] 2D_IoU, depth_loss(log), keypoint_depth_loss(log),
 *       depth_MAE, center_MAE, 02_MAE, 13_MAE, lower_MAE, hard_MAE, soft_MAE, mean_MAE; [32..38] counts
 *   ws64 (device): normalisers kept for the backward call.  No host synchronisation in either call.
 * mf_loss_backward: grad_losses11 (device) = upstream gradient of each loss (ones for the trainer's plain sum,
 * engine/trainer.py:109-110); writes grad_reg [B,50,H,W] (zero except at object centres) and grad_cls [B,ncls,H,W];
 * either may be NULL. */
int mf_loss_obj_cols(void);
int mf_loss_forward(const float* pred_cls, const float* hm, const float* pred_reg, const float* obj, const float* img,
                    const float* weights11, const float* dim_mean9, int B, int ncls, int M, int H, int W, int C,
                    float* out48, float* ws64, void* stream);
int mf_loss_backward(const float* pred_cls, const float* hm, const float* pred_reg, const float* obj, const float* img,
                     const float* weights11, const float* dim_mean9, int B, int ncls, int M, int H, int W, int C,
                     const float* ws64, const float* grad_losses11, float* grad_cls, float* grad_reg, void* stream);

/* torch.optim.AdamW as configured by solver/__init__.py:10-37 (one param group per tensor, lr x BIAS_LR_FACTOR for
 * "bias" tensors, betas (0.9, 0.99), weight decay 1e-5) over ONE flat fp32 arena: every tensor starts at a multiple of
 * mf_adamw_chunk() elements and chunk_lr[n_chunks] (device) holds its group's lr (0 = padding / frozen). step is the
 * 1-based update count; grads are multiplied by grad_scale first (1/world_size after an NCCL SUM of the arena);
 * lr_scale is the scheduler's multiplier (solver/__init__.py:64-92). One launch, 28 B per parameter. */
int mf_adamw_chunk(void);
/* CUDA-graph-safe AdamW step with a finite guard (the reference's optimizer.step(), engine/trainer.py:121, for a training
 * step captured in one graph): the 1-based step count lives in device memory (state4[0]) instead of being a host scalar;
 * with check_finite the gradient arena is scanned first and a non-finite gradient SKIPS the update (state4[2] counts the
 * skipped steps) instead of being written into params / exp_avg / exp_avg_sq. state4: long long[4] zero-initialised by the
 * caller; dyn16: 16 bytes of device scratch. Three launches: scan, 1-thread prepare (bias corrections in double), update. */
int mf_adamw_step_dyn(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, const float* chunk_lr,
                      long long n_chunks, float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                      float lr_scale, long long* state4, void* dyn16, int check_finite, void* stream);

/* DDP gradient all-reduce (tools/plain_train_net.py:100-104) FUSED with the AdamW step for world > 1: one kernel over
 * peer-mapped memory. param_ptrs / grad_ptrs: HOST arrays [world] of device addresses of every rank's parameter / gradient
 * arena as mapped into THIS process (symmetric memory / CUDA IPC); mc_params / mc_grads: NVLS multicast addresses of the
 * same arenas (both 0 = plain NVLink peer loads/stores). Rank r reduces the gradients of its 1/world shard of chunks
 * (multimem.ld_reduce or a fixed-order peer sum), scales by 1/world, updates with ITS shard of exp_avg / exp_avg_sq, and
 * writes the new parameters into all world arenas. The caller brackets the call with two cross-rank barriers (gradients
 * complete everywhere before, parameters visible everywhere after). */
int mf_adamw_step_p2p(const unsigned long long* param_ptrs, const unsigned long long* grad_ptrs, int world, int rank,
                      unsigned long long mc_params, unsigned long long mc_grads, float* exp_avg, float* exp_avg_sq,
                      const float* chunk_lr, long long n_chunks, float beta1, float beta2, float eps, float weight_decay,
                      long long step, float lr_scale, void* stream);
int mf_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, const float* chunk_lr,
                  long long n_chunks, float beta1, float beta2, float eps, float weight_decay, long long step,
                  float grad_scale, float lr_scale, void* stream);

/* ---- GPU input pipeline (SURVEY 8f N4). mf_preprocess_images_u8: B uint8 HWC RGB images of individual sizes h x w <= H x W
 * (src_ptrs: DEVICE array of B device pointers; hw4: DEVICE int32 [B][4] = h, w, pad_x, pad_y with pad = (W - w) / 2, (H - h) / 2
 * as in KITTIDataset.pad_image, data/datasets/kitti.py:218-228; flip: DEVICE int32 [B] or NULL, horizontal flip of the un-padded
 * image) -> zero padding on the uint8 image, x / 255 (ToTensor), (x - mean) / std (Normalize, data/transforms/transforms.py:14-30,
 * IEEE divisions: bit-identical to torch), optional RGB->BGR -> fp32 NCHW [B,3,H,W] = the detector's input. mean3 / std3: HOST.
 * mf_draw_heatmaps: obj6 DEVICE int32 [B][max_objs][6] = valid, class, cx, cy, rx, ry -> hm fp32 [B][ncls][H][W], element-wise
 * max of the objects' Gaussians (model/heatmap_coder.py:56-64, 83-124: rx == ry draw_umich_gaussian, else the one-sided
 * draw_umich_gaussian_2D), sigma = (2 r + 1) / 6, double arithmetic rounded to fp32 like numpy. */
int mf_preprocess_images_u8(const void* const* src_ptrs, const int* hw4, const int* flip, int B, int H, int W,
                            const float* mean3, const float* std3, int to_bgr, float* out_nchw, void* stream);
int mf_draw_heatmaps(const int* obj6, int B, int max_objs, int ncls, int H, int W, float* hm, void* stream);

/* nms_hm alone (model/layers/utils.py:45-58): out = heat * (maxpool3x3(heat) == heat), planes = B*C */
int mf_nms_hm(const float* heat, float* out, int planes, int H, int W, void* stream);

/* nms_hm + select_topk + select_point_of_interest + PostProcessor decode (model/layers/utils.py:45-145,
 * model/head/detector_infer.py:77-237, model/anno_encoder.py:69-295) for a whole batch.
 * heat [B,C,H,W] fp32 (apply_sigmoid=1: raw logits), reg [B,R=50,H,W] fp32, calib [B,6] = f_u,f_v,c_u,c_v,b_x,b_y,
 * pad [B,2], size [B,2] = (W,H) of the padded image, dim_mean [C,3]. Workspaces ws_score/ws_idx: [B*C*K*8]
 * (stage 1 runs 8 CTAs per (image, class) plane; stage 2 merges their candidates).
 * Outputs: scores/clses/ys/xs [B,K] fp32, inds [B,K] int64, pois [B,K,R], result [B,K,14], count [B] = #(score>=thresh). */
int mf_decode_detections(const float* heat, const float* reg, const float* calib, const float* pad, const float* size,
                         const float* dim_mean, int B, int C, int H, int W, int R, int K, float thresh, int apply_sigmoid,
                         float* ws_score, int* ws_idx, float* scores, long long* inds, float* clses, float* ys, float* xs,
                         float* pois, float* result, int* count, void* stream);

/* ---- boundary B: the reference's native operator ABI (_ext, src/vision.cpp:4-9, src/dcn_v2.h:9-59) ------------ */
/* at::Tensor dcn_v2_forward(input, weight, bias, offset, mask, kh,kw,sh,sw,ph,pw,dh,dw,deformable_group): fp32 NCHW,
 * exact fp32 arithmetic (passes testcuda.py:check_zero_offset at 1e-10). y is caller-allocated [B,Cout,Ho,Wo]. */
int mf_dcn_v2_forward(const float* x, const float* w, const float* bias, const float* offset, const float* mask, float* y,
                      int B, int Cin, int H, int W, int Cout, int kh, int kw, int sh, int sw, int ph, int pw, int dh,
                      int dw, int dg, void* workspace, size_t ws_bytes, void* stream);
/* std::vector<at::Tensor>{dX,dOffset,dMask,dW,dB} dcn_v2_backward(input, weight, bias, offset, mask, grad_output, ...)
 * (src/dcn_v2.h:48-59, dcn_v2_cuda.cu:206-335): fp32 NCHW, caller-allocated gradients (they are overwritten, not
 * accumulated into). dX uses atomicAdd like the reference's col2im kernel (summation order not fixed); dOffset, dMask, dW
 * and dB are deterministic. workspace: caller-owned device scratch of at least mf_dcn_v2_backward_workspace(...) bytes
 * (the grad-columns buffer [B, Cin*kh*kw, Ho*Wo] + the split-K partials of dW).
 * Exact-fp32 operator path for `_DCNv2.backward` (autograd / gradcheck); smem-tiled CUDA-core GEMMs (mf_dcn_f32.cu). */
size_t mf_dcn_v2_backward_workspace(int B, int Cin, int H, int W, int Cout, int kh, int kw, int sh, int sw, int ph, int pw,
                                    int dh, int dw, int dg);
int mf_dcn_v2_backward(const float* x, const float* w, const float* bias, const float* offset, const float* mask,
                       const float* grad_y, float* grad_x, float* grad_offset, float* grad_mask, float* grad_w,
                       float* grad_bias, int B, int Cin, int H, int W, int Cout, int kh, int kw, int sh, int sw, int ph,
                       int pw, int dh, int dw, int dg, void* workspace, size_t ws_bytes, void* stream);
/* dcn_v2_psroi_pooling_forward/backward (src/dcn_v2.h:94-153): never instantiated by MonoFlex -> stubs returning -2 */
int mf_dcn_v2_psroi_pooling_forward(void);
int mf_dcn_v2_psroi_pooling_backward(void);

#ifdef __cplusplus
}
#endif
#endif /* MONOFLEX_B200_H */
