"""ctypes loader of tools/libmridc_b200_tools.so: the tensor-core kernels compiled with -DMRB_TC_PROF (per-role cycle
counters, role switches) and the tcgen05 issue micro-benchmark.  Tools only -- the package never loads this library."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mridc_b200 import _lib, build as _build

_vp, _i = ctypes.c_void_p, ctypes.c_int


def load():
    if not os.path.exists(_build.TOOLS_LIB_PATH):
        _build.build_tools()
    lib = ctypes.CDLL(os.path.abspath(_build.TOOLS_LIB_PATH))
    for name in ("mrb_tc_packed_floats", "mrb_tc_pack_conv", "mrb_last_error", "mrb_tc_conv_bh", "mrb_conv_c2_bh_residual",
                 "mrb_bh_fix_border",
                 "mrb_bh_bytes", "mrb_bh_from_nhwc", "mrb_bh_to_nhwc", "mrb_tc2_gru_packed_bytes", "mrb_tc2_pack_gru", "mrb_tc2_gru", "mrb_tc2_unet_conv3x3"):
        res, args = _lib.SIGNATURES[name]
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    lib.mrb_tc_set_debug.restype, lib.mrb_tc_set_debug.argtypes = None, [_i]
    lib.mrb_tc_set_prof.restype, lib.mrb_tc_set_prof.argtypes = None, [_vp]
    lib.mrb_tc2_set_debug.restype, lib.mrb_tc2_set_debug.argtypes = None, [_i]
    lib.mrb_tc2_set_prof.restype, lib.mrb_tc2_set_prof.argtypes = None, [_vp]
    lib.mrb_tc_microbench.restype, lib.mrb_tc_microbench.argtypes = _i, [_i, _i, _i, _i, _vp, _vp]
    return lib
