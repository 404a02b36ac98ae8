/*
 * mridc_b200 PICS -- C-ABI of the l1-wavelet SENSE reconstruction (libmridc_b200_pics.so).
 *
 * Per slice, min_x 1/2 |M (.) F(S x) - y|^2 + lambda |Psi x|_1 by FISTA (DESIGN.md section 4.8).  The Python wrapper
 * (mridc_b200/pics.py) chains, per iteration:
 *   mrb_dc_rim_grad[_hybrid]  (libmridc_b200.so) the data-term gradient at z_k, channels 2-3 of its [B,4,H,W] output
 *   mrbp_fista_step           x_{k+1} = prox_{alpha lambda |Psi.|_1}(z_k - alpha grad),
 *                             z_{k+1} = x_{k+1} + beta (x_{k+1} - x_k)
 * with alpha from mrbp_step_size once per call.
 *
 * Psi: orthonormal 2-D Daubechies-4 wavelet (8 taps, pywt `db4`), periodic boundary, separable, `levels` levels in the
 * Mallat layout of an [H, W] array: at level l the band [0, h) x [0, w) (h = H / 2^(l-1), w = W / 2^(l-1)) becomes
 * LL in [0, h/2) x [0, w/2), LH (low along H, high along W) in [0, h/2) x [w/2, w), HL in [h/2, h) x [0, w/2) and HH in
 * [h/2, h) x [w/2, w).  One level along a line of n samples: a[k] = sum_j h[j] v[(2k + j) mod n],
 * d[k] = sum_j g[j] v[(2k + j) mod n], g[j] = (-1)^j h[7 - j]; the inverse is the transpose.  Real and imaginary parts
 * are transformed alike.
 *
 * Conventions (as include/mridc_b200.h)
 *   - plain pointers and sizes only; every pointer is DEVICE memory owned by the caller, contiguous, 16-byte aligned;
 *     complex images are interleaved (re,im) [B, H, W, 2] fp32.
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden synchronisation, no allocation,
 *     graph-capturable.  `ws` is scratch: its contents on entry are never read.
 *   - return 0 on success, negative MRBP_E* otherwise; `mrbp_last_error()` gives a thread-local message.  Arguments
 *     are checked before any CUDA call.
 */
#ifndef MRIDC_B200_PICS_H
#define MRIDC_B200_PICS_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRBP_OK 0
#define MRBP_EINVAL (-1)       /* bad argument (shape, null pointer, levels, workspace too small) */
#define MRBP_EUNSUPPORTED (-2) /* valid but outside what the kernels cover: B > 65535 or H * W > 2^30 */
#define MRBP_ECUDA (-3)        /* CUDA runtime error; message holds cudaGetErrorString */

const char* mrbp_last_error(void);
int mrbp_version(void);

/* Host only.  The number of wavelet levels PICS uses at H x W: the largest l <= floor(log2(min(H, W) / 7)) with 2^l
 * dividing H and W (320 x 320 -> 5, 640 x 320 -> 5, 232 x 288 -> 3, 14 x 14 -> 1).  0 when there is none (odd H or W,
 * min(H, W) < 14); MRBP_EINVAL when H or W < 1. */
int mrbp_levels(int H, int W);

/* Bytes of `ws` that mrbp_dwt and mrbp_fista_step take at (B, H, W): 12 * B * H * W (one coefficient array and two
 * half-size coarse bands, complex64). */
size_t mrbp_workspace_bytes(int B, int H, int W);

/* Step size.  S [B, C, H, W, 2] fp32 maps; mask [mask_b, mask_h, W] in the canonical form of the DC entry points
 * (mask_dtype 0: uint8, 1: fp32; mask_b in {1, B}, mask_h in {1, H}).  Writes
 *   alpha[b] = 1 / (max_r sum_c |S_bc(r)|^2 * max |M_b|)      (0 where that product is 0)
 * fp32, one value per slice, by a fixed-order reduction (bit-identical run to run and for any batch). */
int mrbp_step_size(const void* S, const void* mask, int mask_dtype, int mask_b, int mask_h, int B, int C, int H, int W,
                   void* alpha, void* stream);

/* Plain transform.  inverse == 0: out = Psi in (Mallat layout), else out = Psi^H in.  in, out [B, H, W, 2] fp32, distinct
 * buffers; 1 <= levels, 2^levels divides H and W (coarse bands shorter than the filter wrap around). */
int mrbp_dwt(const void* in, void* out, int inverse, int B, int H, int W, int levels, void* ws, size_t ws_bytes,
             void* stream);

/* One FISTA step.  grad [B, 4, H, W] fp32: the output of mrb_dc_rim_grad / mrb_dc_rim_grad_hybrid at eta = z (channels
 * 2-3 are read, 0-1 never); alpha [B] fp32 device (mrbp_step_size); lamda >= 0, beta host scalars.
 *   x <- x_{k+1} = Psi^H soft(Psi (z - alpha grad), alpha lamda),  z <- x_{k+1} + beta (x_{k+1} - x_k)
 * soft(c, t) = c * max(0, 1 - t / |c|) on every coefficient, the coarse band included.  z, x [B, H, W, 2] fp32, updated
 * in place.  2 * levels launches; level 1 reads z and grad once and writes x and z once. */
int mrbp_fista_step(void* z, const void* grad, const void* alpha, float lamda, float beta, void* x, int B, int H, int W,
                    int levels, void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif

#endif
