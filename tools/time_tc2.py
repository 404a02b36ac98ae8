"""Timing of the second-generation kernels (BH activations) at the bench geometry."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mridc_b200 import _lib
lib = _lib.load(); st = _lib.stream_ptr()
B = int(sys.argv[1]) if len(sys.argv) > 1 else 4
H = W = 320
dev = "cuda"
def t(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3
nb = lib.mrb_bh_bytes(B, H, W)
x = torch.randn(B, H, W, 64, device=dev); h = torch.randn(B, H, W, 64, device=dev)
xb = torch.empty(nb, dtype=torch.uint8, device=dev); hb = torch.empty_like(xb); ob = torch.empty_like(xb)
lib.mrb_bh_from_nhwc(_lib.ptr(x), _lib.ptr(xb), B, H, W, st); lib.mrb_bh_from_nhwc(_lib.ptr(h), _lib.ptr(hb), B, H, W, st)
wih = torch.randn(192, 64, device=dev) * 0.1; whh = torch.randn(192, 64, device=dev) * 0.1; b = torch.randn(192, device=dev)
pk = torch.empty(lib.mrb_tc2_gru_packed_bytes(), dtype=torch.uint8, device=dev)
_lib.check(lib.mrb_tc2_pack_gru(_lib.ptr(wih), _lib.ptr(whh), _lib.ptr(pk), 64, 64, st))
us = t(lambda: _lib.check(lib.mrb_tc2_gru(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pk), _lib.ptr(b), _lib.ptr(ob), B, H, W, st)))
px = B * H * W
print("tc2 gru B=%d: %.1f us  (%.0f GB/s at 768 B/px, %.1f TFLOP/s algorithmic)" % (B, us, px * 768 / us / 1e3, px * 2 * 128 * 192 / us / 1e6))
# final conv: CUDA-core kernel (+ the border fix it needs) vs the tensor-core tap GEMM, each right after a GRU wrote its input
w3 = torch.randn(2, 64, 3, 3, device=dev) * 0.05
eta = torch.randn(B, H, W, 2, device=dev); o2 = torch.empty_like(eta)
gru = lambda: lib.mrb_tc2_gru(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pk), _lib.ptr(b), _lib.ptr(ob), B, H, W, st)
def after_gru(fn, n=20):
    for _ in range(3): gru(); fn()
    torch.cuda.synchronize(); tot = 0.0
    for _ in range(n):
        gru()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / n * 1e3
def old():
    _lib.check(lib.mrb_bh_fix_border(_lib.ptr(ob), B, H, W, st))
    _lib.check(lib.mrb_conv_c2_bh_residual(_lib.ptr(ob), _lib.ptr(w3), None, _lib.ptr(eta), _lib.ptr(o2), B, H, W, st))
new = lambda: _lib.check(lib.mrb_tc2_final_conv(_lib.ptr(ob), _lib.ptr(w3), None, _lib.ptr(eta), _lib.ptr(o2), B, H, W, st))
u0, u1 = after_gru(old), after_gru(new)
print("final conv B=%d: fp32 CUDA-core + border fix %.1f us, tensor-core tap GEMM %.1f us (%.0f GB/s at 272 B/px)" %
      (B, u0, u1, px * 272 / u1 / 1e3))
# first conv: the bulk-copy-fed G8 kernel and its fp32 -> G8 converter
from mridc_b200.rim_tc import RimTcEngine
import mridc_b200 as mb
from mridc_b200 import synth
blk = mb.CIRIM(synth.cirim_cfg("GRU")).cuda().eval().cirim[0]
eng = RimTcEngine(blk); packs = eng.packs()
c0 = blk.layers[0].convs; c1 = blk.layers[1].convs
g4 = torch.randn(B, H, W, 4, device=dev)
g8 = torch.zeros(lib.mrb_g8_bytes(B, H, W), dtype=torch.uint8, device=dev)
u_cv = t(lambda: _lib.check(lib.mrb_g8_from_nhwc4(_lib.ptr(g4), _lib.ptr(g8), B, H, W, st)))
u_new = t(lambda: _lib.check(lib.mrb_tc2_conv5x5x4(_lib.ptr(g8), _lib.ptr(c0.conv_layer.weight), _lib.ptr(c0.conv_layer.bias), _lib.ptr(ob), B, H, W, 1, st)))
print("conv5x5 B=%d: G8 converter %.1f us + bulk-copy kernel %.1f us (%.0f GB/s at 272 B/px)" % (B, u_cv, u_new, px * 272 / u_new / 1e3))
u3 = t(lambda: _lib.check(lib.mrb_tc_conv_bh(_lib.ptr(hb), _lib.ptr(packs[1][0]), _lib.ptr(c1.conv_layer.bias), _lib.ptr(ob), B, H, W, 64, 3, 2, 1, st)))
print("conv3x3 d2 B=%d: %.1f us (%.1f TFLOP/s algorithmic)" % (B, u3, px * 2 * 64 * 64 * 9 / u3 / 1e6))
# IndRNN cell on BH activations
wi = torch.randn(64, 64, 1, 1, device=dev) * 0.1
pki = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, 1), device=dev)
_lib.check(lib.mrb_tc_pack_conv(_lib.ptr(wi), _lib.ptr(pki), 64, 64, 1, st))
bi = torch.randn(64, device=dev); hhv = torch.randn(64, device=dev)
ui = t(lambda: _lib.check(lib.mrb_tc2_indrnn(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pki), _lib.ptr(bi), _lib.ptr(hhv), _lib.ptr(ob), B, H, W, st)))
print("tc2 indrnn B=%d: %.1f us  (%.0f GB/s at 768 B/px)" % (B, ui, px * 768 / ui / 1e3))
