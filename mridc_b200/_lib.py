"""ctypes binding of libmridc_b200.so (the C-ABI declared in include/mridc_b200.h).

There is NO CPU fallback: if the CUDA library is missing, cannot be loaded, or a tensor is not a CUDA
tensor, the call raises.
"""
import ctypes
import os
import threading

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libmridc_b200.so")

_vp, _ll, _i, _f, _sz = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_float, ctypes.c_size_t
_llp = ctypes.POINTER(ctypes.c_longlong)
_fp, _dp, _d = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double), ctypes.c_double

# name -> (restype, argtypes); must list every symbol of include/mridc_b200.h (tests/test_abi.py checks)
SIGNATURES = {
    "mrb_last_error": (ctypes.c_char_p, []),
    "mrb_version": (_i, []),
    "mrb_launch_count": (_ll, []),
    "mrb_reset_launch_count": (None, []),
    "mrb_add_launch_count": (None, [_ll]),
    "mrb_fft1d_c2c": (_i, [_vp, _vp, _ll, _i, _ll, _i, _i, _i, _f, _vp]),
    "mrb_fft2_c2c": (_i, [_vp, _vp, _ll, _i, _i, _i, _i, _i, _vp]),
    "mrb_roll": (_i, [_vp, _vp, _ll, _ll, _ll, _i, _ll, _vp]),
    "mrb_complex_mul": (_i, [_vp, _vp, _vp, _i, _llp, _llp, _llp, _i, _vp]),
    "mrb_complex_conj": (_i, [_vp, _vp, _ll, _vp]),
    "mrb_complex_abs": (_i, [_vp, _vp, _ll, _i, _vp]),
    "mrb_rss": (_i, [_vp, _vp, _ll, _i, _ll, _vp]),
    "mrb_rss_complex": (_i, [_vp, _vp, _ll, _i, _ll, _vp]),
    "mrb_sense_combine": (_i, [_vp, _vp, _vp, _ll, _i, _ll, _vp]),
    "mrb_divide_rss": (_i, [_vp, _vp, _ll, _i, _ll, _vp]),
    "mrb_dc_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mrb_dc_rim_grad": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "mrb_dc_hybrid_prepare": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "mrb_dc_rim_grad_hybrid": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mrb_sens_reduce": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "mrb_sens_expand_softdc": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _i,
                                    _vp, _sz, _vp]),
    "mrb_conv2d": (_i, [_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp, _i,
                        _vp]),
    "mrb_gru_cell_1x1": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _ll, _vp]),
    "mrb_gru_gates": (_i, [_vp, _vp, _vp, _vp, _i, _i, _ll, _vp]),
    "mrb_mgu_gates": (_i, [_vp, _vp, _vp, _vp, _i, _i, _ll, _vp]),
    "mrb_instnorm_lrelu": (_i, [_vp, _ll, _vp, _ll, _i, _i, _ll, _f, _f, _vp, _vp]),
    "mrb_conv1x1": (_i, [_vp, _ll, _vp, _vp, _vp, _ll, _i, _i, _i, _ll, _vp]),
    "mrb_avgpool2": (_i, [_vp, _ll, _vp, _ll, _i, _i, _i, _i, _vp]),
    "mrb_conv_transpose2x2": (_i, [_vp, _ll, _vp, _vp, _ll, _i, _i, _i, _i, _i, _vp]),
    "mrb_pad2d": (_i, [_vp, _ll, _vp, _ll, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mrb_normunet_in": (_i, [_vp, _vp, _vp, _i, _i, _ll, _i, _vp, _vp]),
    "mrb_normunet_out": (_i, [_vp, _vp, _vp, _i, _i, _ll, _i, _vp]),
    "mrb_tc_packed_floats": (_sz, [_i, _i, _i, _i]),
    "mrb_tc_pack_conv": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "mrb_bh_bytes": (_sz, [_i, _i, _i]),
    "mrb_bh_from_nhwc": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "mrb_bh_to_nhwc": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "mrb_tc_conv_bh": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "mrb_conv_c2_bh_residual": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "mrb_bh_fix_border": (_i, [_vp, _i, _i, _i, _vp]),
    "mrb_tc2_final_conv": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "mrb_tc2_unet_packed_bytes": (_sz, [_i, _i]),
    "mrb_tc2_unet_pack": (_i, [_vp, _vp, _i, _i, _vp]),
    "mrb_tc2_unet_conv3x3": (_i, [_vp, _ll, _vp, _vp, _ll, _i, _i, _i, _i, _i, _vp]),
    "mrb_g8_bytes": (_sz, [_i, _i, _i]),
    "mrb_g8_from_nhwc4": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "mrb_tc2_conv5x5x4": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "mrb_tc2_gru_packed_bytes": (_sz, []),
    "mrb_tc2_pack_gru": (_i, [_vp, _vp, _vp, _i, _i, _vp]),
    "mrb_tc2_gru": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "mrb_tc2_indrnn": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "mrb_metrics_workspace_bytes": (_sz, [_i]),
    "mrb_abs_max_normalize": (_i, [_vp, _ll, _i, _vp, _vp, _vp]),
    "mrb_recon_metrics": (_i, [_vp, _vp, _i, _i, _i, _i, _d, _vp, _vp, _vp]),
    "mrb_megre_signal": (_i, [_vp, _vp, _vp, _vp, _fp, _dp, _i, _d, _i, _ll, _i, _vp, _vp]),
    "mrb_megre_grad": (_i, [_vp, _vp, _vp, _vp, _vp, _fp, _dp, _i, _d, _i, _ll, _f, _i, _vp, _i, _vp]),
    "mrb_qrim_eta_update": (_i, [_vp, _i, _i, _vp, _vp, _i, _ll, _vp]),
    "mrb_scale_batch": (_i, [_vp, _vp, _i, _ll, _fp, _i, _vp]),
}

_lib = None
_lock = threading.Lock()


def load():
    """Load the shared library (once). Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "mridc_b200: CUDA library %s is missing. Build it with `python -m mridc_b200.build` "
                "(there is no CPU fallback)." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        msg = load().mrb_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError("mridc_b200: " + msg)
        if rc == -2:
            raise NotImplementedError("mridc_b200: " + msg)
        raise RuntimeError("mridc_b200 (code %d): %s" % (rc, msg))


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def require_cuda(t, name="tensor", dtype=torch.float32):
    """No CPU fallback: anything that is not a CUDA tensor of the expected dtype raises."""
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError(
            "mridc_b200: %s is on %s; this package only runs on CUDA (sm_100a) -- there is no CPU fallback" % (name, t.device))
    if dtype is not None and t.dtype != dtype:
        raise TypeError("mridc_b200: %s must be %s (got %s)" % (name, dtype, t.dtype))
    if t.device.index != torch.cuda.current_device():
        # kernels launch on the current device's stream with raw pointers: a tensor of another GPU would be an illegal
        # address (or, with peer access, silent remote execution)
        raise RuntimeError("mridc_b200: %s lives on %s but the current CUDA device is cuda:%d; wrap the call in "
                           "`with torch.cuda.device(t.device)` (one process per GPU is the supported layout)"
                           % (name, t.device, torch.cuda.current_device()))
    return t


def launch_count():
    return int(load().mrb_launch_count())


def reset_launch_count():
    load().mrb_reset_launch_count()
