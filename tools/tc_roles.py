"""Per-role cycle counters of tc_kernel (the BH k x k conv of conv_tc.cu) at the dilated 3x3 of the CIRIM time step."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import mridc_b200 as mb
from mridc_b200 import _lib, synth
from mridc_b200.rim_tc import RimTcEngine
import _toolslib
lib = _toolslib.load(); st = _lib.stream_ptr()   # profiling build of the same kernels (weights packed by the product library)
B, H, W = int(sys.argv[1]) if len(sys.argv) > 1 else 1, 320, 320
dev = torch.device("cuda")
model = mb.CIRIM(synth.cirim_cfg("GRU")).cuda().eval()
blk = model.cirim[0]; eng = RimTcEngine(blk); packs = eng.packs()
x = torch.randn(B, H, W, 64, device=dev)
c1 = blk.layers[1].convs
def t(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3
nb = lib.mrb_bh_bytes(B, H, W)
xb = torch.empty(nb, dtype=torch.uint8, device=dev); ob = torch.empty(nb, dtype=torch.uint8, device=dev)
lib.mrb_bh_from_nhwc(_lib.ptr(x), _lib.ptr(xb), B, H, W, st)
ops = {
 "conv3x3d2_bh": lambda: lib.mrb_tc_conv_bh(_lib.ptr(xb), _lib.ptr(packs[1][0]), _lib.ptr(c1.conv_layer.bias), _lib.ptr(ob), B, H, W, 64, 3, 2, 1, st),
}
for flags, name in ((0, "full"),):
    lib.mrb_tc_set_debug(flags)
    print("%-18s" % name, "  ".join("%s %7.1f us" % (k, t(f)) for k, f in ops.items()), flush=True)
lib.mrb_tc_set_debug(0)
prof = torch.zeros(148 * 16, dtype=torch.int64, device=dev)
lib.mrb_tc_set_prof(_lib.ptr(prof))
for dbg in (0,):
  lib.mrb_tc_set_debug(dbg)
  print("debug flags", dbg)
  for k, f in ops.items():
    prof.zero_(); f(); torch.cuda.synchronize()
    p = prof.view(148, 16).double().mean(0).tolist()
    print("%-12s loader: total %7.0f wait_empty %7.0f store %7.0f (st-wait+arrive %7.0f) issue %7.0f | mma: total %7.0f wait_full %7.0f wait_acc %7.0f issue %7.0f commit %7.0f wait_b %7.0f seg-top..issue %7.0f | epi: total %7.0f wait %7.0f (cycles, mean over CTAs)" % (
        k, p[0], p[1], p[2], p[13], p[3], p[4], p[5], p[6], p[7], p[10], p[11], p[12], p[8], p[9]))
lib.mrb_tc_set_debug(0); lib.mrb_tc_set_prof(None)
lib.mrb_tc_set_prof(_lib.ptr(prof))
for k, f in ops.items():
    prof.zero_(); f(); torch.cuda.synchronize()
    pv = prof.view(148, 16).double()
    tot = pv[:, 8]  # epilogue total per CTA (runs to the end of the kernel)
    print("%-12s per-CTA epilogue-total cycles: min %.0f mean %.0f max %.0f  (max/mean %.2f)" % (k, tot.min(), tot.mean(), tot.max(), tot.max() / tot.mean()))
lib.mrb_tc_set_prof(None)
