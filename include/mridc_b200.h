/*
 * mridc_b200 -- C-ABI of the B200-native (sm_100a) unrolled-MRI-reconstruction hot path.
 *
 * The reference (wdika/mridc) is pure Python/PyTorch: it has no FFI seam of its own.  The entry points
 * below are what a maintainer would bind (ctypes stub in INTEGRATION.md) behind the reference's Python
 * API for this path.  Each entry cites the reference interface it replaces (paths relative to the
 * upstream repo root, `mridc/collections/` abbreviated `mc/`).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is DEVICE memory owned by the caller (PyTorch),
 *     contiguous, fp32 unless stated; complex tensors are interleaved (re,im) = "complex-last-2".
 *   - every pointer is 16-byte aligned (the tensor-core kernels read and write through TMA and bulk copies, which
 *     require it; PyTorch's allocator hands out 512-byte aligned blocks).
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden synchronisation,
 *     graph-capturable after one eager warm-up call (twiddle tables are created on first use per device
 *     and FFT length, owned by the library, immutable afterwards).
 *   - return 0 on success, negative MRB_E* otherwise; `mrb_last_error()` gives a thread-local message.
 *   - norm:  0 = "backward"/"none", 1 = "ortho", 2 = "forward"   (mc/common/parts/fft.py:77-81,155-159)
 *   - centered != 0: fftshift(F(ifftshift(x))) on both transforms (fft.py:74-84,152-162), any length.
 *   - mask descriptor: `mask` points to [mask_b, mask_h, W] values of dtype `mask_dtype`
 *     (0 = uint8/bool bytes, 1 = float32); mask_b in {1,B}, mask_h in {1,H} (broadcast when 1).
 */
#ifndef MRIDC_B200_H
#define MRIDC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRB_OK 0
#define MRB_EINVAL (-1)   /* bad argument (shape, enum, null pointer) */
#define MRB_EUNSUPPORTED (-2) /* valid but outside what the kernels cover (e.g. FFT length too large for smem) */
#define MRB_ECUDA (-3)    /* CUDA runtime error; message holds cudaGetErrorString */

#define MRB_NORM_BACKWARD 0
#define MRB_NORM_ORTHO 1
#define MRB_NORM_FORWARD 2

#define MRB_MASK_U8 0
#define MRB_MASK_F32 1

#define MRB_PAD_ZERO 0
#define MRB_PAD_REPLICATE 1

#define MRB_ACT_NONE 0
#define MRB_ACT_RELU 1
#define MRB_ACT_LEAKY 2 /* slope passed separately */

const char* mrb_last_error(void);
int mrb_version(void);
/* Number of kernel launches issued by this library on the calling thread since the last reset
 * (bench.py's "gpu_launches"). */
long long mrb_launch_count(void);
void mrb_reset_launch_count(void);
/* account for kernel launches replayed from a CUDA graph (captured launches are counted once, at capture time) */
void mrb_add_launch_count(long long n);

/* ---------------------------------------------------------------------------------------------------
 * L1 primitives -- mc/common/parts/fft.py, utils.py
 * ------------------------------------------------------------------------------------------------- */

/* 1-D complex FFT along the middle axis of a contiguous [outer, n, inner] complex64 tensor.
 * Building block of fft2/ifft2 for arbitrary `spatial_dims` (fft.py:13-88, 91-166).
 * in == out allowed. scale is applied to the output. in_rot/out_rot implement the centered variant:
 * logical input index j is read from storage (j + in_rot) % n, logical output k is written to storage
 * (k + out_rot) % n (in_rot = out_rot = n/2 for centered; see DESIGN.md). */
int mrb_fft1d_c2c(const void* in, void* out, long long outer, int n, long long inner, int inverse,
                  int in_rot, int out_rot, float scale, void* stream);

/* fft2 / ifft2 over the last two axes of [batch, H, W] complex64 (fft.py:13-88 / 91-166). */
int mrb_fft2_c2c(const void* in, void* out, long long batch, int H, int W, int inverse, int centered,
                 int norm, void* stream);

/* roll along one axis of a contiguous [outer, n, inner] tensor of `elem_bytes`-byte elements
 * (fft.py:169-202 roll_one_dim; bit-exact, any dtype incl. int64). out != in. */
int mrb_roll(const void* in, void* out, long long outer, long long n, long long inner, int elem_bytes,
             long long shift, void* stream);

/* Strided element-wise complex ops with broadcasting (utils.py:96-118 complex_mul, conj_y != 0 multiplies by
 * conj(y) as in utils.py:248).  ndim <= 6; strides in complex elements, 0 = broadcast; out contiguous. */
int mrb_complex_mul(const void* x, const void* y, void* out, int ndim, const long long* shape,
                    const long long* xstride, const long long* ystride, int conj_y, void* stream);
/* utils.py:121-139 */
int mrb_complex_conj(const void* x, void* out, long long n, void* stream);
/* utils.py:142-157 (squared == 0) and :160-175 (squared != 0): [n,2] -> [n] */
int mrb_complex_abs(const void* x, void* out, long long n, int squared, void* stream);
/* utils.py:194-209 rss on a real view: x [outer, C, inner] fp32 -> out [outer, inner] = sqrt(sum_c x^2) */
int mrb_rss(const void* x, void* out, long long outer, int C, long long inner, void* stream);
/* utils.py:212-227 rss_complex: x [outer, C, inner] complex -> out [outer, inner] real */
int mrb_rss_complex(const void* x, void* out, long long outer, int C, long long inner, void* stream);
/* utils.py:230-248 sense(): sum_c x * conj(S): x,S [outer, C, inner] complex -> [outer, inner] complex */
int mrb_sense_combine(const void* x, const void* S, void* out, long long outer, int C, long long inner,
                      void* stream);
/* BaseSensitivityModel.divide_root_sum_of_squares (reconstruction/models/base.py:826-840):
 * x [outer, C, inner] complex64 -> out = x / sqrt(sum_c |x_c|^2) (same shape, distinct buffer) */
int mrb_divide_rss(const void* x, void* out, long long outer, int C, long long inner, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Fused data-consistency operator
 * ------------------------------------------------------------------------------------------------- */

/* Workspace bytes for the DC entry points below at (B, C, H, W): two complex64 [B,C,H,W] scratch images. */
size_t mrb_dc_workspace_bytes(int B, int C, int H, int W);

/* RIM log-likelihood gradient -- mc/reconstruction/models/rim/rim_utils.py:11-67.
 *   eta [B,H,W,2], y,S [B,C,H,W,2], out [B,4,H,W] = (eta_re, eta_im, g_re, g_im)  (the reference layout, :67),
 *   or [B,H,W,4] when out_nhwc != 0 (channels-last feed of the tensor-core regulariser);
 *   g = sum_c conj(S) * ifft2(mask * (fft2(S*eta) - y)) * inv_sigma2  (mask VALUE multiplies: :54). */
int mrb_dc_rim_grad(const void* eta, const void* y, const void* S, const void* mask, int mask_dtype,
                    int mask_b, int mask_h, float inv_sigma2, void* out, int out_nhwc, int B, int C, int H,
                    int W, int centered, int norm, void* ws, size_t ws_bytes, void* stream);

/* Hybrid-space form of the same gradient for 1-D (column) masks, mask [mask_b, 1, W].  When the mask does not depend
 * on k_h the H-direction transforms of fft2 / ifft2 in rim_utils.py:50-58 cancel:
 *     ifft2(M * (fft2(x) - y)) = bs*H * V_W[ M * (fs * U_W x - yh) ],   yh = (1/H) * V_H y   (U/V: centred DFTs)
 * mrb_dc_hybrid_prepare computes yh once per slice batch (y is constant over the unrolled network): [B,C,H,W,2] buffer
 * whose rows hold the sampled columns packed at the front; ws as for mrb_sens_reduce (one [B,C,H,W] complex image).
 * mrb_dc_rim_grad_hybrid is then one kernel of row transforms per evaluation (same outputs as mrb_dc_rim_grad).
 * out_nhwc == 2 (W == 320, C <= 16 only): `out` is a G8 buffer (mrb_g8_bytes, zero-initialised once) and the kernel
 * writes the regulariser's conv input directly -- 4 bf16 hi + 4 bf16 lo per position, replicate border included. */
int mrb_dc_hybrid_prepare(const void* y, const void* mask, int mask_dtype, int mask_b, void* yh, int B, int C,
                          int H, int W, int centered, void* ws, size_t ws_bytes, void* stream);
int mrb_dc_rim_grad_hybrid(const void* eta, const void* yh, const void* S, const void* mask, int mask_dtype,
                           int mask_b, float inv_sigma2, void* out, int out_nhwc, int B, int C, int H, int W,
                           int centered, int norm, void* stream);

/* sum_c ifft2(x) * conj(S) -- mc/reconstruction/models/varnet/vn_block.py:71-87 sens_reduce, also the
 * zero-filled SENSE init of rim_block.py:195-211, zf.py:90-97, vn.py:131-139, unet.py:108-117.
 *   x,S [B,C,H,W,2] -> out [B,H,W,2] */
int mrb_sens_reduce(const void* x, const void* S, void* out, int B, int C, int H, int W, int centered,
                    int norm, void* ws, size_t ws_bytes, void* stream);

/* Soft data consistency -- vn_block.py:51-69 (sens_expand) + :109-119, and rim_block.py:256-267.
 *   img [B,H,W,2]; S,base,pred,y,out [B,C,H,W,2];
 *   E = fft2(S*img);  out = no_dc ? E : base - (mask != 0 ? pred - y : 0) * dc_weight - E
 *   (mask TRUTHINESS selects: `torch.where(mask.bool(), ...)`, vn_block.py:110).
 *   VarNet passes base = pred (:117); the RIM no_dc=False branch passes base = y (rim_block.py:258).
 *   dc_weight: DEVICE pointer to one float (the learnable parameter; no host sync needed).
 *   base/pred/y/mask/dc_weight may be null if no_dc. */
int mrb_sens_expand_softdc(const void* img, const void* S, const void* base, const void* pred, const void* y,
                           const void* mask, int mask_dtype, int mask_b, int mask_h, const void* dc_weight,
                           int no_dc, void* out, int B, int C, int H, int W, int centered, int norm,
                           void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Convolutional / recurrent regulariser kernels (NCHW fp32)
 * ------------------------------------------------------------------------------------------------- */

/* "same" 2-D convolution, odd kernel k, dilation dil, padding dil*(k-1)/2 of kind pad_mode.
 *   ConvNonlinear (rim/conv_layers.py:36-123: replicate pad, bias, ReLU/LeakyReLU/none),
 *   ConvGRU/MGU/IndRNN ih/hh convs (rim/rnn_cells.py:23-38: zero pad), U-Net 3x3 / 1x1 convs
 *   (unet_base/unet_block.py:250-259,:185).
 *   x [N,Cin,H,W] with batch stride x_bstride floats; w [Cout,Cin,k,k]; bias [Cout] or null;
 *   out [N,Cout,H,W] with batch stride out_bstride floats.
 *   Epilogue: v = acc + bias;  if (add) v += add_scale[co] * add[n,co,h,w]  (IndRNN: rnn_cells.py:391);
 *             v = act(v) (leaky slope `slope`);
 *   out_nhwc_residual != 0: out is [N,H,W,Cout] and v is ADDED to residual [N,H,W,Cout]
 *   (rim_block.py:241-248: eta + grad.permute(0,2,3,1)). */
int mrb_conv2d(const void* x, long long x_bstride, const void* w, const void* bias, void* out,
               long long out_bstride, int N, int Cin, int Cout, int H, int W, int k, int dil, int pad_mode,
               int act, float slope, const void* add, const void* add_scale, const void* residual,
               int out_nhwc_residual, void* stream);

/* Fused ConvGRU cell for kernel_size 1 (rim/rnn_cells.py:93-127; every shipped config uses k=1):
 *   x [N,Cx,H,W], h [N,Ch,H,W] -> h_out [N,Ch,H,W]; w_ih [3Ch,Cx], b_ih [3Ch] or null, w_hh [3Ch,Ch]. */
int mrb_gru_cell_1x1(const void* x, const void* h, const void* w_ih, const void* b_ih, const void* w_hh,
                     void* h_out, int N, int Cx, int Ch, long long HW, void* stream);

/* Gate arithmetic of ConvGRUCell (rnn_cells.py:121-125) on precomputed ih,hh [N,3Ch,HW]. */
int mrb_gru_gates(const void* ih, const void* hh, const void* h, void* h_out, int N, int Ch, long long HW,
                  void* stream);
/* Gate arithmetic of ConvMGUCell (rnn_cells.py:257-261) on precomputed ih,hh [N,2Ch,HW]. */
int mrb_mgu_gates(const void* ih, const void* hh, const void* h, void* h_out, int N, int Ch, long long HW,
                  void* stream);

/* Per-(n,c) InstanceNorm2d(affine=False, eps, biased var) followed by LeakyReLU(slope)
 * (unet_block.py:251-253,:256-258,:294-295).  x [N,C,HW] batch stride x_bstride; out batch stride
 * out_bstride (lets the caller write straight into a concat buffer, unet_block.py:223).
 * stats: workspace of 2*N*C doubles. */
int mrb_instnorm_lrelu(const void* x, long long x_bstride, void* out, long long out_bstride, int N, int C,
                       long long HW, float eps, float slope, void* stats, void* stream);

/* avg_pool2d(kernel 2, stride 2) (unet_block.py:204): x [NC,H,W] (plane stride via bstride/C) */
int mrb_avgpool2(const void* x, long long x_bstride, void* out, long long out_bstride, int N, int C, int H,
                 int W, void* stream);

/* Conv2d(kernel 1) with bias (the last layer of the U-Net, unet_block.py:185): x [N,Cin,HW] -> out [N,Cout,HW], batch
 * strides in floats; w [Cout,Cin]; bias [Cout] or null.  HW and the strides must be multiples of 4 (16-byte loads). */
int mrb_conv1x1(const void* x, long long x_bstride, const void* w, const void* bias, void* out, long long out_bstride, int N,
                int Cin, int Cout, long long HW, void* stream);

/* ConvTranspose2d(kernel 2, stride 2, bias False) (unet_block.py:293): x [N,Cin,H,W], w [Cin,Cout,2,2]
 * -> out [N,Cout,2H,2W] */
int mrb_conv_transpose2x2(const void* x, long long x_bstride, const void* w, void* out,
                          long long out_bstride, int N, int Cin, int Cout, int H, int W, void* stream);

/* Generic 2-D pad/crop copy: out[n,c,y,x] = in[n,c,map(y-off_y),map(x-off_x)], mode 0 zero fill outside,
 * 1 replicate, 2 reflect (unet_block.py:93-111 pad/unpad, :216-222 reflect). */
int mrb_pad2d(const void* x, long long x_bstride, void* out, long long out_bstride, int N, int C, int Hin,
              int Win, int Hout, int Wout, int off_y, int off_x, int mode, void* stream);

/* NormUnet.norm + complex_to_chan_dim (unet_block.py:55-60,:71-85): x [B,C,H,W,2] -> out [B,2C,H,W]
 * normalised per (b, re/im group) with mean and UNBIASED std; mean_std out: [B,2,2] floats (mean,std);
 * normalize == 0 only permutes.  stats: workspace of 4*B doubles. */
int mrb_normunet_in(const void* x, void* out, void* mean_std, int B, int C, long long HW, int normalize,
                    void* stats, void* stream);
/* NormUnet.unnorm + chan_complex_to_last_dim (unet_block.py:62-69,:87-91): x [B,2C,HW] -> [B,C,HW,2] */
int mrb_normunet_out(const void* x, const void* mean_std, void* out, int B, int C, long long HW,
                     int normalize, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Tensor-core (tcgen05 / TMEM, error-compensated bf16 hi/lo split, fp32 accumulation) RIM regulariser, used by RIMBlock's
 * time loop (rim_block.py:217-249) when the layer geometry matches (64 channels, cell kernel size 1).  Same arithmetic as
 * mrb_conv2d / mrb_gru_cell_1x1 to ~3e-6 relative per operator (products are evaluated as a_hi*b_hi + a_hi*b_lo +
 * a_lo*b_hi with 16-17 significant bits per operand).
 * Weights are packed once per parameter version into the UMMA shared-memory layout (bf16 hi/lo split).
 * (The profiling hooks of these kernels live in the tools-only build, tools/libmridc_b200_tools.so.)
 * ------------------------------------------------------------------------------------------------- */
/* size of the packed weights in 4-byte units: kind 0 = conv k x k (cin 64); any other kind: 0 */
size_t mrb_tc_packed_floats(int kind, int cout, int cin, int k);
/* w [cout, 64, k, k] (conv_layers.py:78-85) */
int mrb_tc_pack_conv(const void* w, void* dst, int cout, int cin, int k, void* stream);
/* ---------------------------------------------------------------------------------------------------
 * Second-generation tensor-core engine: split-bf16 ("BH") activations, TMA + shared-memory operands.
 * BH layout: [B][H+4][W+4][hi 64 bf16 | lo 64 bf16] (x ~= hi + lo; 256 B per pixel; replicate border of 2 pixels, which
 * is ConvNonlinear's ReplicationPad2d, conv_layers.py:72-76, materialised once by the producer).
 * ------------------------------------------------------------------------------------------------- */
/* bytes of a BH tensor for B images of H x W pixels (64 channels) */
size_t mrb_bh_bytes(int B, int H, int W);
/* fp32 channels-last [B,H,W,64] -> BH (split + replicate border) and back (interior, hi + lo) */
int mrb_bh_from_nhwc(const void* x, void* bh, int B, int H, int W, void* stream);
int mrb_bh_to_nhwc(const void* bh, void* x, int B, int H, int W, void* stream);
/* packed ConvGRUCell weights for mrb_tc2_gru: w_ih, w_hh [192, 64] (rnn_cells.py:23-38) */
size_t mrb_tc2_gru_packed_bytes(void);
int mrb_tc2_pack_gru(const void* w_ih, const void* w_hh, void* dst, int ch, int cx, void* stream);
/* ConvNonlinear on BH tensors (conv_layers.py:36-123): k x k (dilation dil, dil*(k-1)/2 <= 2) BH -> BH, bias, optional
 * ReLU; wpack from mrb_tc_pack_conv; cout == 64.  x_bh needs a valid replicate border; the border of the output is not a
 * replicate copy. */
int mrb_tc_conv_bh(const void* x_bh, const void* wpack, const void* bias, void* out_bh, int B, int H, int W, int cout, int k,
                   int dil, int relu, void* stream);
/* First RIM conv fed by bulk copies.  "G8" input layout: the conv input [eta.re, eta.im, grad.re, grad.im] of a position as
 * 4 hi + 4 lo bf16 (16 bytes), positions in the padded BH geometry [B][H+4][W+4] with a replicate border, plus guard
 * positions before and after.  mrb_g8_bytes: allocation size (the caller zero-initialises the buffer ONCE; the guards are
 * only ever read); mrb_g8_from_nhwc4: fp32 channels-last [B,H,W,4] (the output of mrb_dc_rim_grad with nhwc) -> G8;
 * mrb_tc2_conv5x5x4: ConvNonlinear(4 -> 64, k = 5, replicate padding, optional ReLU; conv_layers.py:36-123) G8 -> BH with
 * w [64,4,5,5] fp32 (split into bf16 hi/lo on the fly), bias [64] or null.  Every position of out_bh is written; its
 * border is not a replicate copy. */
size_t mrb_g8_bytes(int B, int H, int W);
int mrb_g8_from_nhwc4(const void* x, void* g8, int B, int H, int W, void* stream);
int mrb_tc2_conv5x5x4(const void* g8, const void* w, const void* bias, void* out_bh, int B, int H, int W, int relu,
                      void* stream);
/* final RIM conv (rim_block.py:239-248) on a BH source with a valid border: out [B,H,W,2] = eta + conv3x3(x) (+ bias) */
int mrb_conv_c2_bh_residual(const void* x_bh, const void* w, const void* bias, const void* eta, void* out, int B, int H,
                            int W, void* stream);
/* U-Net 3x3 convolution (unet_base/unet_block.py:250-259: Conv2d(kernel 3, padding 1, bias False)) as an implicit GEMM on
 * tcgen05 with error-compensated fp16-split operands (x = hi + lo to 2^-22, three products per MAC, fp32 accumulation:
 * ~5e-7 relative per operator; operands must be O(1), i.e. instance-normalised activations -- values below 2^-14 lose
 * relative accuracy).  x [N,Cin,H,W] / out [N,Cout,H,W] NCHW fp32
 * with batch strides in floats (skip connections are read / written in place inside the concat buffers); wpack from
 * mrb_tc2_unet_pack (mrb_tc2_unet_packed_bytes bytes); Cin <= 64. */
size_t mrb_tc2_unet_packed_bytes(int Cin, int Cout);
/* w [Cout,Cin,3,3] fp32 -> the kernel's weight image (fp16 hi / lo rows per tap and group of 8 input channels); once per
 * parameter version */
int mrb_tc2_unet_pack(const void* w, void* dst, int Cin, int Cout, void* stream);
int mrb_tc2_unet_conv3x3(const void* x, long long x_bstride, const void* wpack, void* out, long long out_bstride, int N,
                         int Cin, int Cout, int H, int W, void* stream);
/* the same final conv (rim_block.py:239-248, conv_layers.py:72-123) on the tensor core: the channel contraction runs once
 * per position as a tap GEMM (T[pos][tap, o] = sum_c h[pos][c] w[o][c][tap], split-bf16 tcgen05), the nine taps are gathered
 * in shared memory with their coordinates clamped to the image (= ReplicationPad2d(1)); the BH border of x_bh is never
 * read, so a pointwise producer needs no mrb_bh_fix_border before this call */
int mrb_tc2_final_conv(const void* x_bh, const void* w, const void* bias, const void* eta, void* out, int B, int H, int W,
                       void* stream);
/* edge pixels -> replicate border of a BH tensor (after a pointwise producer, before a spatial consumer) */
int mrb_bh_fix_border(void* bh, int B, int H, int W, void* stream);
/* ConvGRUCell, kernel size 1, 64 -> 64 (rnn_cells.py:93-127): x, h, out in BH layout; b_ih [192] or null; out must not
 * alias x or h.  Pointwise over all (H+4)(W+4) positions: the interior of out is the cell output, its border is NOT a
 * replicate copy (follow with mrb_bh_fix_border before a spatial consumer); the border of x and h is never read for an
 * interior result. */
int mrb_tc2_gru(const void* x_bh, const void* h_bh, const void* wpack, const void* b_ih, void* out_bh, int B, int H, int W,
                void* stream);
/* IndRNNCell, kernel size 1, 64 -> 64 (rnn_cells.py:264-391, the cell base_cirim_run.yaml ships) on BH tensors:
 * out = ReLU(W_ih x + b_ih + hh * h); wpack = mrb_tc_pack_conv(ih.weight, 64, 64, 1); b_ih [64] or null; hh [64]; out must
 * not alias x or h.  Pointwise over all positions like mrb_tc2_gru. */
int mrb_tc2_indrnn(const void* x_bh, const void* h_bh, const void* wpack, const void* b_ih, const void* hh, void* out_bh, int B,
                   int H, int W, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Quantitative MRI (qRIM / qCIRIM, BASELINE.json configs[4]): pointwise kernels around the fused DC operator.
 * The data-consistency part of analytical_log_likelihood_gradient
 * (mridc/collections/quantitative/models/qrim/utils.py:166-295) is mrb_dc_rim_grad with the echoes folded into the
 * batch: eta = mrb_megre_signal(maps), then mrb_megre_grad turns its per-echo output into the map gradient.
 * maps are [B, HW] fp32; gamma4 (host pointer, may be null = ones) multiplies (R2*, S0, B0, phi) first
 * (qrim_block.py:196-199); tes: n_echoes echo times (host doubles); scaling: SignalForwardModel.scaling (1e-3).
 * ------------------------------------------------------------------------------------------------- */
/* SignalForwardModel.__call__ (qrim/utils.py:36-155): -> out [B, E, HW] complex64 (NaN -> 0); no_phase != 0 selects
 * MEGRENoPhaseSignalModel (b0 / phi unused). */
int mrb_megre_signal(const void* r2star, const void* s0, const void* b0, const void* phi, const float* gamma4,
                     const double* tes, int n_echoes, double scaling, int B, long long HW, int no_phase, void* out,
                     void* stream);
/* qrim/utils.py:236-295: d [B*E, 4, HW] = mrb_dc_rim_grad output for the B*E signal images (channels 2,3 = the
 * coil-combined residual) -> out[b, 0..3, HW] = (R2*_re, S0_re, R2*_im, S0_im) gradient, mean over echoes, divided by
 * `divisor` (qrim_block.py:222: 100), NaN -> 0 when zero_nan (:223); out has out_channels (>= 4) channels per sample. */
int mrb_megre_grad(const void* d, const void* r2star, const void* s0, const void* b0, const void* phi,
                   const float* gamma4, const double* tes, int n_echoes, double scaling, int B, long long HW,
                   float divisor, int zero_nan, void* out, int out_channels, void* stream);
/* qrim_block.py:232-236: eta <- eta + delta with channel 0 (R2*) clamped at >= 0; eta = channels
 * [eta_offset, eta_offset + 4) of a [B, eta_channels, HW] buffer (updated in place), delta / out [B, 4, HW]. */
int mrb_qrim_eta_update(void* eta, int eta_channels, int eta_offset, const void* delta, void* out, int B,
                        long long HW, void* stream);
/* RescaleByMax.reverse (qrim/utils.py:25-28): out[b] = x[b] * scales[b], or |x[b]| * scales[b] when take_abs
 * (qcirim.py:287-289 applies it to torch.abs(pred)); the reference indexes its 4 regularisation factors by BATCH
 * index (four in every shipped config), so one call takes B <= 4; longer batches are chunked by the caller.  scales:
 * host pointer, B floats. */
int mrb_scale_batch(const void* x, void* out, int B, long long per_batch, const float* scales, int take_abs,
                    void* stream);

/* ---------------------------------------------------------------------------------------------------
 * On-device evaluation (SURVEY 8f rank 3): what test_step computes on the host after .cpu()
 * (mridc/collections/reconstruction/models/base.py:415-436, common/metrics/reconstruction_metrics.py:11-41).
 * ------------------------------------------------------------------------------------------------- */
/* bytes of the device workspace both calls below take (B = slices) */
size_t mrb_metrics_workspace_bytes(int B);
/* base.py:415-420: out[i] = |x[i]| / max_j |x[j]|; x: n complex64 (is_complex) or fp32 values, out: n fp32 */
int mrb_abs_max_normalize(const void* x, long long n, int is_complex, void* out, void* ws, void* stream);
/* gt, pred [B,H,W] fp32 -> res (device, 5 doubles) = mse, nmse, psnr, ssim, data range used.  maxval_mode 0: max(gt)
 * (reconstruction_metrics.py:23,35), 1: max(pred) - min(pred) (base.py:431,434), 2: `maxval`.  SSIM = skimage
 * structural_similarity defaults (7x7 uniform window, sample covariance, K1 0.01, K2 0.03, 3-px border crop, float64),
 * averaged over slices; PSNR = 10 log10(R^2 / mse).  maxval_mode + 4 skips the SSIM kernels (res[3] = NaN; any H, W >= 1):
 * the reference's mse / nmse / psnr accept images smaller than the SSIM window. */
int mrb_recon_metrics(const void* gt, const void* pred, int B, int H, int W, int maxval_mode, double maxval, void* res,
                      void* ws, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MRIDC_B200_H */
