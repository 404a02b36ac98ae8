"""ESPIRiT coil sensitivity maps estimated on the GPU from the calibration region of multi-coil k-space.

The SENSE models of this package (CIRIM, E2EVN without ``use_sens_net``, ZF-SENSE, qCIRIM) take coil sensitivity maps as
an input; upstream mridc obtains them offline from BART ``ecalib``.  ``espirit_maps`` computes one map set with the
semantics of sigpy's ``EspiritCalib`` from k-space alone.  The arithmetic is hand-written CUDA behind the C-ABI of
``include/mridc_b200_espirit.h`` (``libmridc_b200_espirit.so``) plus the FFT of ``libmridc_b200.so``; the one
eigendecomposition per slice is ``torch.linalg.eigh`` in float64.  No CPU fallback.
"""
import ctypes
import os
import threading

import torch

from . import _lib

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libmridc_b200_espirit.so")

_vp, _i, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_float

# name -> (restype, argtypes); must list every symbol of include/mridc_b200_espirit.h (tests/test_gpu_espirit.py checks)
SIGNATURES = {
    "mrbe_last_error": (ctypes.c_char_p, []),
    "mrbe_version": (_i, []),
    "mrbe_calib_gram": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mrbe_kernel_taps": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "mrbe_power_maps": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
}
MAX_COILS = 32
# per-chunk bytes of the per-pixel matrices G(r): C(C+1)/2 complex64 planes per slice (432 MB at 32 coils x 320 x 320)
G_CHUNK_BYTES = 1 << 30

_lib_handle = None
_lock = threading.Lock()


def load():
    """Load libmridc_b200_espirit.so (once). Raises RuntimeError if it has not been built."""
    global _lib_handle
    if _lib_handle is not None:
        return _lib_handle
    with _lock:
        if _lib_handle is not None:
            return _lib_handle
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("mridc_b200: CUDA library %s is missing. Build it with `python -m mridc_b200.build` "
                               "(there is no CPU fallback)." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib_handle = lib
    return _lib_handle


def check(rc):
    if rc != 0:
        msg = load().mrbe_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError("mridc_b200.espirit: " + msg)
        if rc == -2:
            raise NotImplementedError("mridc_b200.espirit: " + msg)
        raise RuntimeError("mridc_b200.espirit (code %d): %s" % (rc, msg))


def _validate(y, calib_width, kernel_width, threshold, crop, max_iter):
    _lib.require_cuda(y, "y", torch.float32)
    if y.dim() != 5 or y.shape[-1] != 2:
        raise ValueError("mridc_b200.espirit: y must be [B, C, H, W, 2] (got %s)" % (tuple(y.shape),))
    B, C, H, W, _ = y.shape
    if not 1 <= C <= MAX_COILS:
        raise ValueError("mridc_b200.espirit: %d coils; 1 to %d are supported" % (C, MAX_COILS))
    for name, v in (("calib_width", calib_width), ("kernel_width", kernel_width), ("max_iter", max_iter)):
        if int(v) != v or v < 1:
            raise ValueError("mridc_b200.espirit: %s must be a positive integer (got %r)" % (name, v))
    if not kernel_width <= calib_width <= min(H, W):
        raise ValueError("mridc_b200.espirit: need kernel_width <= calib_width <= min(H, W) (got %d, %d, %dx%d)" % (
            kernel_width, calib_width, H, W))
    if not threshold >= 0 or not crop == crop:
        raise ValueError("mridc_b200.espirit: threshold must be >= 0 and crop a number")


def calibrate(y, calib_width=24, kernel_width=6, threshold=0.02, fft_centered=True):
    """Steps 1-3: -> (vecs [B, N, N] complex128, row j = eigenvector j of A^H A in ascending eigenvalue order;
    rank [B] int32, the number of kernels K = #{sigma_i > threshold * sigma_max} of each slice; the last K rows span the
    kernel subspace).  N = C * kernel_width**2."""
    _validate(y, calib_width, kernel_width, threshold, 0.0, 1)
    lib = load()
    B, C, H, W, _ = y.shape
    N = C * kernel_width * kernel_width
    y = y.contiguous()
    gram = torch.empty(B, N, N, 2, dtype=torch.float64, device=y.device)
    check(lib.mrbe_calib_gram(_lib.ptr(y), _lib.ptr(gram), B, C, H, W, calib_width, kernel_width, int(fft_centered),
                              _lib.stream_ptr()))
    gram = torch.view_as_complex(gram)
    vecs = torch.empty(B, N, N, dtype=torch.complex128, device=y.device)
    rank = torch.empty(B, dtype=torch.int32, device=y.device)
    for b in range(B):  # one slice per call: the eigenvectors of a slice do not depend on the rest of the batch
        ev, V = torch.linalg.eigh(gram[b])
        s = ev.clamp_min(0).sqrt()
        rank[b] = (s > threshold * s[-1]).sum()
        vecs[b] = V.mT
    return vecs, rank


def espirit_maps(y, calib_width=24, kernel_width=6, threshold=0.02, crop=0.95, max_iter=100, fft_centered=True,
                 return_eigenvalues=False):
    """ESPIRiT coil sensitivity maps (sigpy ``EspiritCalib`` semantics, one map set) of k-space ``y`` [B, C, H, W, 2]
    (CUDA float32, C <= 32).  The calibration region is the centred ``calib_width`` square of k-space (DC at (H//2,
    W//2) when ``fft_centered``, at (0, 0) otherwise).  Returns maps [B, C, H, W, 2] float32, zero where the dominant
    eigenvalue is not above ``crop``, and with ``return_eigenvalues`` also that eigenvalue [B, H, W]."""
    _validate(y, calib_width, kernel_width, threshold, crop, max_iter)
    vecs, rank = calibrate(y, calib_width, kernel_width, threshold, fft_centered)
    lib, base = load(), _lib.load()
    B, C, H, W, _ = y.shape
    P = C * (C + 1) // 2
    maps = torch.empty(B, C, H, W, 2, dtype=torch.float32, device=y.device)
    lam = torch.empty(B, H, W, dtype=torch.float32, device=y.device)
    chunk = max(1, min(B, G_CHUNK_BYTES // (P * H * W * 8)))
    g = torch.empty(chunk, P, H, W, 2, dtype=torch.float32, device=y.device)
    st = _lib.stream_ptr()
    for b0 in range(0, B, chunk):
        n = min(chunk, B - b0)
        check(lib.mrbe_kernel_taps(_lib.ptr(vecs[b0]), _lib.ptr(rank[b0:]), _lib.ptr(g), n, C, H, W, kernel_width,
                                   int(fft_centered), st))
        _lib.check(base.mrb_fft2_c2c(_lib.ptr(g), _lib.ptr(g), n * P, H, W, 1, int(fft_centered), 2, st))
        check(lib.mrbe_power_maps(_lib.ptr(g), _lib.ptr(maps[b0]), _lib.ptr(lam[b0]), n, C, H, W, int(max_iter),
                                  float(crop), st))
    return (maps, lam) if return_eigenvalues else maps
