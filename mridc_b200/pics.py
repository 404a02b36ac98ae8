"""PICS: l1-wavelet compressed-sensing SENSE reconstruction on the GPU.

Upstream mridc's ``PICS`` model hands k-space and coil maps to BART ``pics`` with an l1-wavelet regulariser.  Here, per
slice, ``min_x 1/2 |M (.) F(S x) - y|^2 + lamda |Psi x|_1`` is solved by FISTA with the contract of DESIGN.md section 4.8:
Psi the orthonormal periodic 2-D Daubechies-4 wavelet, step 1 / (max_r sum_c |S_c(r)|^2 * max |M|) per slice, x_0 = 0,
exactly ``max_iter`` iterations, no random shifts and no data scaling.  Each iteration is one data-term gradient of
``libmridc_b200.so`` (the fused DC operator, hybrid row form for 1-D masks) and one fused proximal step of
``libmridc_b200_pics.so`` (C-ABI ``include/mridc_b200_pics.h``).  No CPU fallback.
"""
import ctypes
import math
import os
import threading

import torch

from . import _lib, _ops

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libmridc_b200_pics.so")

_vp, _i, _f, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol of include/mridc_b200_pics.h (tests/test_pics_cpu.py checks)
SIGNATURES = {
    "mrbp_last_error": (ctypes.c_char_p, []),
    "mrbp_version": (_i, []),
    "mrbp_levels": (_i, [_i, _i]),
    "mrbp_workspace_bytes": (_sz, [_i, _i, _i]),
    "mrbp_step_size": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "mrbp_dwt": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "mrbp_fista_step": (_i, [_vp, _vp, _vp, _f, _f, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
}
# pywt `db4` low-pass analysis taps (extremal phase); csrc/pics.cu holds the same values
DB4_LO = (0.2303778133088964, 0.7148465705529154, 0.6308807679298587, -0.0279837694168599, -0.1870348117190931,
          0.0308413818355607, 0.0328830116668852, -0.0105974017850690)

_lib_handle = None
_lock = threading.Lock()


def load():
    """Load libmridc_b200_pics.so (once). Raises RuntimeError if it has not been built."""
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
        msg = load().mrbp_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError("mridc_b200.pics: " + msg)
        if rc == -2:
            raise NotImplementedError("mridc_b200.pics: " + msg)
        raise RuntimeError("mridc_b200.pics (code %d): %s" % (rc, msg))


def wavelet_levels(H, W):
    """Levels of Psi at H x W (``mrbp_levels``); ValueError when no level fits (odd H or W, min(H, W) < 14)."""
    L = load().mrbp_levels(int(H), int(W))
    if L < 0:
        check(L)
    if L == 0:
        raise ValueError("mridc_b200.pics: no wavelet level fits %d x %d (H and W must be even and at least 14)" % (H, W))
    return L


def _workspace(B, H, W, device):
    n = load().mrbp_workspace_bytes(B, H, W)
    return torch.empty(n // 4, dtype=torch.float32, device=device), n


def _check_image(x, name):
    _lib.require_cuda(x, name, torch.float32)
    if x.dim() != 4 or x.shape[-1] != 2:
        raise ValueError("mridc_b200.pics: %s must be [B, H, W, 2] (got %s)" % (name, tuple(x.shape)))
    return x.contiguous()


def dwt(x, inverse=False, levels=None):
    """Psi x (Mallat layout, see include/mridc_b200_pics.h) of complex images x [B, H, W, 2], or Psi^H x with
    ``inverse``.  ``levels`` defaults to ``wavelet_levels(H, W)``."""
    x = _check_image(x, "x")
    B, H, W, _ = x.shape
    levels = wavelet_levels(H, W) if levels is None else int(levels)
    out = torch.empty_like(x)
    ws, n = _workspace(B, H, W, x.device)
    check(load().mrbp_dwt(_lib.ptr(x), _lib.ptr(out), int(bool(inverse)), B, H, W, levels, _lib.ptr(ws), n,
                          _lib.stream_ptr()))
    return out


def step_size(sensitivity_maps, mask):
    """alpha [B] fp32 = 1 / (max_r sum_c |S_c(r)|^2 * max |M|) per slice (0 where that is 0)."""
    S = _ops._check5(sensitivity_maps, "sensitivity_maps")
    B, C, H, W, _ = S.shape
    m, code, mb, mh = _ops.canonical_mask(mask, B, H, W)
    alpha = torch.empty(B, dtype=torch.float32, device=S.device)
    check(load().mrbp_step_size(_lib.ptr(S), _lib.ptr(m), code, mb, mh, B, C, H, W, _lib.ptr(alpha),
                                _lib.stream_ptr()))
    return alpha


def _validate(y, sensitivity_maps, lamda, max_iter, fft_normalization):
    y = _ops._check5(y, "y")
    S = _ops._check5(sensitivity_maps, "sensitivity_maps")
    if S.shape != y.shape:
        raise ValueError("mridc_b200.pics: shape mismatch: y %s, sensitivity_maps %s" % (tuple(y.shape), tuple(S.shape)))
    if isinstance(lamda, torch.Tensor) or not (isinstance(lamda, (int, float)) and math.isfinite(lamda) and lamda >= 0):
        raise ValueError("mridc_b200.pics: lamda must be a finite number >= 0 (got %r)" % (lamda,))
    if isinstance(max_iter, bool) or int(max_iter) != max_iter or max_iter < 1:
        raise ValueError("mridc_b200.pics: max_iter must be a positive integer (got %r)" % (max_iter,))
    _ops.norm_code(fft_normalization)
    return y, S


def fista_iterates(y, sensitivity_maps, mask, lamda, max_iter=100, fft_centered=True, fft_normalization="ortho"):
    """The FISTA iteration of ``l1_wavelet_recon``: yields (x_k, z_k, grad) for k = 1 .. max_iter, grad being the
    [B, 4, H, W] data-term gradient at z_{k-1} that step k used.  The tensors are the solver's own buffers, updated in
    place by the next step.  No host synchronisation after the argument checks."""
    y, S = _validate(y, sensitivity_maps, lamda, max_iter, fft_normalization)
    B, C, H, W, _ = y.shape
    levels = wavelet_levels(H, W)
    lib = load()
    m = _ops.canonical_mask(mask, B, H, W)[0]  # canonical [mb, mh, W]: passed through unchanged by the DC wrappers
    alpha = step_size(S, m)
    yh = _ops.dc_hybrid_prepare(y, m, fft_centered)
    dc_ws = _ops._ws(B, C, H, W, y.device) if yh is None else None
    x = torch.zeros(B, H, W, 2, dtype=torch.float32, device=y.device)
    z = torch.zeros_like(x)
    g = torch.empty(B, 4, H, W, dtype=torch.float32, device=y.device)
    ws, n = _workspace(B, H, W, y.device)
    t = 1.0
    for _ in range(int(max_iter)):
        _ops.dc_rim_grad(z, y, S, m, 1.0, fft_centered, fft_normalization, out=g, ws=dc_ws, y_hybrid=yh)
        t_next = (1.0 + math.sqrt(1.0 + 4.0 * t * t)) / 2.0
        beta = (t - 1.0) / t_next
        check(lib.mrbp_fista_step(_lib.ptr(z), _lib.ptr(g), _lib.ptr(alpha), float(lamda), beta, _lib.ptr(x), B, H, W,
                                  levels, _lib.ptr(ws), n, _lib.stream_ptr()))
        t = t_next
        yield x, z, g


def l1_wavelet_recon(y, sensitivity_maps, mask, lamda, max_iter=100, fft_centered=True, fft_normalization="ortho"):
    """l1-wavelet SENSE reconstruction of masked multi-coil k-space ``y`` [B, C, H, W, 2] with coil maps
    ``sensitivity_maps`` of the same shape and a ``mask`` broadcastable as for the DC operator (uint8, bool or float;
    1-D column or 2-D, shared or per slice), all CUDA: ``max_iter`` FISTA iterations on
    1/2 |M (.) F(S x) - y|^2 + lamda |Psi x|_1 (DESIGN.md section 4.8), F = fft2 under ``fft_centered`` /
    ``fft_normalization``.  Returns x [B, H, W, 2] float32.  H and W must be even and at least 14."""
    x = None
    for x, _, _ in fista_iterates(y, sensitivity_maps, mask, lamda, max_iter, fft_centered, fft_normalization):
        pass
    return x
