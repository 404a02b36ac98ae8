/*
 * mridc_b200 ESPIRiT -- C-ABI of the coil-sensitivity estimator (libmridc_b200_espirit.so).
 *
 * One ESPIRiT map set from the calibration (ACS) region of multi-coil k-space, with the semantics of sigpy's
 * `EspiritCalib` (the maps upstream mridc obtains offline from BART `ecalib`).  The Python wrapper
 * (mridc_b200/espirit.py) chains, per slice:
 *   mrbe_calib_gram   A^H A of the calibration matrix, fp64
 *   (eigendecomposition of A^H A, fp64; torch.linalg.eigh)
 *   mrbe_kernel_taps  the kernel-subspace projector as zero-padded autocorrelation taps per coil pair
 *   mrb_fft2_c2c      (libmridc_b200.so) taps -> per-pixel matrix G(r), inverse transform, norm "forward"
 *   mrbe_power_maps   the dominant eigenvector of every G(r) by a fixed number of power iterations
 *
 * Conventions (as include/mridc_b200.h)
 *   - plain pointers and sizes only; every pointer is DEVICE memory owned by the caller, contiguous, 16-byte aligned;
 *     complex tensors are interleaved (re,im).  Entry points take no workspace: every buffer they write is an output.
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden synchronisation, no allocation,
 *     graph-capturable.
 *   - return 0 on success, negative MRBE_E* otherwise; `mrbe_last_error()` gives a thread-local message.  Arguments
 *     are checked before any CUDA call.
 *   - centered != 0: k-space with DC at (H/2, W/2) (integer division).  centered == 0: DC at (0, 0); the result is
 *     then ifftshift(espirit(fftshift(y))) over (H, W), done by index rotation inside the kernels.
 *
 * Definitions (N = C*kw*kw calibration columns, P = C*(C+1)/2 coil pairs c <= d, pair index of (c,d) =
 * c*C - c*(c-1)/2 + (d - c)):
 *   ACS       rows H/2 - cw/2 ... + cw - 1, columns W/2 - cw/2 ... + cw - 1 of the centred k-space;
 *   A         one row per kw x kw window of the ACS (stride 1, (cw-kw+1)^2 rows), columns (c, p, q) row-major;
 *   kernels   v_i: the eigenvectors of A^H A with sigma_i = sqrt(max(eig_i, 0)) > threshold * sigma_max;
 *   G(r)      (1/kw^2) F_r conj(P) F_r^H, P = sum_i v_i v_i^H, F_r[c, (c,p,q)] = exp(+2 pi i (p n_y/H + q n_x/W)),
 *             n = r - (H/2, W/2) (centred coordinates).
 */
#ifndef MRIDC_B200_ESPIRIT_H
#define MRIDC_B200_ESPIRIT_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRBE_OK 0
#define MRBE_EINVAL (-1)       /* bad argument (shape, null pointer) */
#define MRBE_EUNSUPPORTED (-2) /* valid but outside what the kernels cover (see the limits below) */
#define MRBE_ECUDA (-3)        /* CUDA runtime error; message holds cudaGetErrorString */

#define MRBE_MAX_COILS 32
#define MRBE_MAX_CALIB_WIDTH 112 /* two coils' ACS blocks (complex64) in one CTA's shared memory */
#define MRBE_MAX_CALIB_COLS 2048 /* N = C * kw * kw */

const char* mrbe_last_error(void);
int mrbe_version(void);

/* Calibration Gram matrix.  y [B, C, H, W, 2] fp32 k-space -> gram [B, N, N, 2] fp64 = A^H A (both triangles,
 * exactly Hermitian), accumulated in fp64 in a fixed order.  1 <= kw <= cw <= min(H, W), C <= MRBE_MAX_COILS. */
int mrbe_calib_gram(const void* y, void* gram, int B, int C, int H, int W, int cw, int kw, int centered,
                    void* stream);

/* Kernel-subspace taps.  vecs [B, N, N, 2] fp64: row j of slice b is eigenvector j of A^H A, eigenvalues ascending
 * (the layout of torch.linalg.eigh(...).eigenvectors.mT); rank [B] int32: the kernel count K of each slice (0..N), the
 * last K rows are used.  taps [B, P, H, W, 2] fp32: for every coil pair c <= d the autocorrelation
 *   T_cd(dy, dx) = (1/kw^2) sum_i sum_{p-p'=dy, q-q'=dx} conj(v_i[c,p,q]) v_i[d,p',q'],  |dy|, |dx| < kw,
 * summed in fp64, placed at ((dy + H/2) mod H, (dx + W/2) mod W) (centered) or (dy mod H, dx mod W) (not centered),
 * lags that alias to one position added, every other position zero.  The inverse fft2 of each plane (norm "forward",
 * same `centered`) is G(r)[c, d] at the output pixels.  Every element of taps is written. */
int mrbe_kernel_taps(const void* vecs, const int* rank, void* taps, int B, int C, int H, int W, int kw, int centered,
                     void* stream);

/* Per-pixel power method.  g [B, P, H, W, 2] fp32: G(r)[c, d] for c <= d (G is Hermitian).  Per pixel, from x = 1:
 * max_iter times y = G x, lambda = |y|_2, x = y / lambda (x = 0, lambda = 0 when y = 0); then
 * x <- x * conj(x_0) / |x_0| where x_0 != 0, and maps = lambda > crop ? x : 0.
 * maps [B, C, H, W, 2] fp32, lambda [B, H, W] fp32; every element written.  max_iter >= 1. */
int mrbe_power_maps(const void* g, void* maps, void* lambda, int B, int C, int H, int W, int max_iter, float crop,
                    void* stream);

#ifdef __cplusplus
}
#endif

#endif
