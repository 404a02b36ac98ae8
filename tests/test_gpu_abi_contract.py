"""Every launching entry point of include/mridc_b200.h held to its buffer and stream contract.

test_gpu_kernel_paths.py checks *what* each kernel computes.  This file checks *where* it writes, *what memory* it reads
and *which stream* it runs on -- what the header promises every caller ("every pointer is DEVICE memory owned by the
caller", workspaces are scratch, "all work is enqueued on `stream`; no hidden synchronisation, graph-capturable after one
eager warm-up call", and the per-entry claims about BH borders, G8 guards and partially written outputs).  A parity test
sees none of these: an out-of-bounds write lands in another allocation, an unwritten element keeps the right value from
the previous identical run, a kernel that needs a zeroed workspace passes because the wrappers allocate fresh ones, and
work sent to the wrong stream passes in single-stream tests.

A row declares its buffers with a role (``in``, ``out``, ``inout``, ``ws`` = contents undefined on entry, ``g8`` = zero
guard positions by contract), the call with raw pointers, an fp64 reference (the ones of test_gpu_kernel_paths.py and the
oracle package) and, per output, the region the header says is written.  Each buffer is a view inside an allocation with
64 KiB on each side (more than one BH tile of 128 positions x 256 B; offsets stay multiples of 256 B).  Each check runs once:

  eager, set A     input guards NaN, outputs and their guards a byte sentinel, workspaces zero: the guards and every byte
                   outside the declared written region are unchanged, no sentinel is left inside it, the result is finite
                   and matches fp64 within the per-slice contract (2e-6 fp32, 1e-5 split-bf16, 2e-6 uconv3, exact ops
                   bit-exact);
  poisoned, set A  workspaces 0xFF (NaN), outputs NaN, BH borders NaN where the header says they are never read: the same
                   bits as the first run;
  graph, set B     the call captured with torch.cuda.graph on a side stream (global capture mode: a hidden sync, a
                   cudaMalloc or legacy-stream work fails the capture), set B copied into the same inputs, outputs and
                   workspaces re-poisoned, replayed: the same bits as an eager run of set B into separate buffers, guards
                   intact.  Work on any other stream is not replayed, host state baked into the graph shows as a wrong
                   result.  Host-pointer arguments (tes, gamma4, scales, maxval, complex_mul's shape) stay fixed, because a
                   graph legitimately bakes them.

The second-device rows run the entry points that raise the dynamic shared-memory limit of their kernel on cuda:0 and then
on cuda:1 in one process (function attributes belong to a device's context) and compare the bits.

This file stands in for the compute-sanitizer memcheck / initcheck passes of profiles/r02_sanitizer, which predate the
current tc_kernel and plane_stats_kernel and cannot be rerun where the suite runs.
"""
import ctypes
import gc

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_bench_shapes import check_slices
from test_gpu_kernel_paths import _dc_inputs, _fft_ref, _gen, _instnorm_ref, _lib, _mask, _norm

GUARD = 64 * 1024
SENTINEL = 0xA5
ROLES = ("in", "out", "inout", "ws", "g8")

# symbols of _lib.SIGNATURES that enqueue no work, with the reason they have no contract row
NON_LAUNCHING = {
    "mrb_last_error": "host-side error message",
    "mrb_version": "host-side constant",
    "mrb_launch_count": "host-side counter",
    "mrb_reset_launch_count": "host-side counter",
    "mrb_add_launch_count": "host-side counter",
    "mrb_dc_workspace_bytes": "size query",
    "mrb_tc_packed_floats": "size query",
    "mrb_bh_bytes": "size query",
    "mrb_tc2_unet_packed_bytes": "size query",
    "mrb_g8_bytes": "size query",
    "mrb_tc2_gru_packed_bytes": "size query",
    "mrb_metrics_workspace_bytes": "size query",
}


# ---------------------------------------------------------------------------------------------- harness
class Buf:
    """One buffer of a row.  written / defined / unread: bool masks over the buffer's elements (None = all / all / none).
    written: the elements the call must write; defined: those whose value the contract fixes (compared bit for bit across
    runs); unread: input elements the header says are never read (NaN in the poisoned runs).  rtol: compare across runs
    to this relative tolerance instead of bit for bit, for values the kernel reduces with floating-point atomics (their
    order, so their last bits, change from run to run); NaN must still meet NaN."""

    def __init__(self, role, numel, dtype=torch.float32, written=None, defined=None, unread=None, finite=True, rtol=None):
        assert role in ROLES, role
        self.role, self.numel, self.dtype = role, int(numel), dtype
        self.written, self.unread, self.finite, self.rtol = written, unread, finite, rtol
        self.defined = written if defined is None else defined


class Row:
    """bufs: name -> Buf; make(seed) -> dict of the in / inout contents (keys starting with "_" carry reference data);
    call(V, stream) launches on the typed 1-D views V; check(V, X) compares the outputs of set X with fp64."""

    def __init__(self, bufs, make, call, check):
        self.bufs, self.make, self.call, self.check = bufs, make, call, check


def _elsize(dtype):
    return torch.empty((), dtype=dtype).element_size()


def _fill_nan(t):
    if t.dtype.is_floating_point:
        t.fill_(float("nan"))
    else:
        t.view(torch.uint8).fill_(0xFF)


class Slot:
    """A buffer placed GUARD bytes into its own allocation."""

    def __init__(self, name, buf, device):
        self.name, self.buf = name, buf
        self.el = _elsize(buf.dtype)
        self.word = 4 if self.el == 1 else self.el  # byte buffers are checked in 4-byte words
        self.nbytes = buf.numel * self.el
        assert self.nbytes % self.word == 0, (name, self.nbytes)
        assert self.el > 1 or (buf.written is None and buf.unread is None), "byte buffers take whole-buffer regions"
        span = -(-self.nbytes // 256) * 256
        self.base = torch.empty(GUARD + span + GUARD, dtype=torch.uint8, device=device)
        self.bytes = self.base[GUARD:GUARD + self.nbytes]
        self.view = self.bytes.view(buf.dtype)
        self.mask = {k: (None if getattr(buf, k) is None else getattr(buf, k).reshape(-1).to(device))
                     for k in ("written", "defined", "unread")}
        for k, m in self.mask.items():
            assert m is None or m.numel() == buf.numel, (name, k)
        self.pre = None

    def guards(self):
        return self.base[:GUARD], self.base[GUARD + self.nbytes:]

    def byte_mask(self, key):
        m = self.mask[key]
        return None if m is None else m.repeat_interleave(self.el)

    def words(self, b=None):
        return (self.bytes if b is None else b).view(-1, self.word)


def alloc(bufs, device):
    return {name: Slot(name, b, device) for name, b in bufs.items()}


def prime(slots, X, poison):
    """Fill guards, inputs, outputs and workspaces for one run (see the module docstring)."""
    for s in slots.values():
        role = s.buf.role
        if role in ("in", "inout"):
            for g in s.guards():
                _fill_nan(g.view(s.buf.dtype))
            src = X[s.name].reshape(-1)
            assert src.numel() == s.buf.numel and src.dtype == s.buf.dtype, (s.name, src.shape, src.dtype)
            s.view.copy_(src)
            if poison and s.mask["unread"] is not None:
                s.view[s.mask["unread"]] = float("nan")
        elif role == "out":
            s.base.fill_(SENTINEL)
            if poison:
                _fill_nan(s.view)
        elif role == "g8":
            s.base.fill_(SENTINEL)
            s.view.zero_()
            bm = s.byte_mask("written")
            if poison:
                nan = torch.empty_like(s.view)
                _fill_nan(nan)
                s.view.copy_(torch.where(s.mask["written"], nan, s.view) if bm is not None else nan)
            elif bm is None:
                s.bytes.fill_(SENTINEL)
            else:
                s.bytes[bm] = SENTINEL
        else:  # ws
            s.base.fill_(SENTINEL)
            s.bytes.fill_(0xFF if poison else 0)
        s.pre = s.base.clone()


def _where(s, off):
    if off < 0:
        return "in the guard before the buffer"
    if off >= s.nbytes:
        return "in the guard after the buffer (%d bytes long)" % s.nbytes
    return "inside the buffer, outside the region the call writes"


def verify(slots, tag, ref=None):
    """Guards and unowned bytes unchanged; with ref (name -> bytes of a reference run) the defined region equal to ref bit
    for bit, without ref no sentinel left in the written region and no non-finite value in the defined region."""
    for s in slots.values():
        role, el = s.buf.role, s.el
        allowed = torch.zeros_like(s.base, dtype=torch.bool)
        if role in ("out", "inout", "g8"):
            bm = s.byte_mask("written")
            allowed[GUARD:GUARD + s.nbytes] = True if bm is None else bm
        elif role == "ws":
            allowed[GUARD:GUARD + s.nbytes] = True
        bad = (s.base != s.pre) & ~allowed
        if bool(bad.any()):
            off = int(bad.nonzero()[0, 0]) - GUARD
            raise AssertionError("%s: %s buffer %r modified at byte offset %d, %s (%d bytes changed)" % (
                tag, role, s.name, off, _where(s, off), int(bad.sum())))
        if role not in ("out", "inout", "g8"):
            continue
        wm, dm = s.mask["written"], s.mask["defined"]
        if ref is None:
            left = (s.words() == SENTINEL).all(1)
            if wm is not None:
                left &= wm
            if bool(left.any()):
                i = int(left.nonzero()[0, 0])
                raise AssertionError("%s: %s buffer %r: byte offset %d (element %d) not written (sentinel left; %d elements)" % (
                    tag, role, s.name, i * s.word, i * s.word // el, int(left.sum())))
            if s.buf.finite and s.buf.dtype.is_floating_point:
                nf = ~torch.isfinite(s.view)
                if dm is not None:
                    nf &= dm
                if bool(nf.any()):
                    i = int(nf.nonzero()[0, 0])
                    raise AssertionError("%s: %s buffer %r: non-finite value at byte offset %d (element %d; %d elements) -- "
                                         "a read outside an input or of unwritten memory" % (
                                             tag, role, s.name, i * el, i, int(nf.sum())))
        else:
            diff = (s.words() != s.words(ref[s.name])).any(1)
            if s.buf.rtol is not None:
                a, b = s.view, ref[s.name].view(s.buf.dtype)
                diff &= ~((a - b).abs() <= s.buf.rtol * b.abs()) & ~(torch.isnan(a) & torch.isnan(b))
            if dm is not None:
                diff &= dm
            if bool(diff.any()):
                i = int(diff.nonzero()[0, 0])
                raise AssertionError("%s: %s buffer %r differs from the reference run at byte offset %d (element %d; %d "
                                     "elements)" % (tag, role, s.name, i * s.word, i * s.word // el, int(diff.sum())))


def outputs(slots):
    return {n: s.bytes.clone() for n, s in slots.items() if s.buf.role in ("out", "inout", "g8")}


def views(slots):
    return {n: s.view for n, s in slots.items()}


def _sync(device):
    if torch.device(device).type == "cuda":
        torch.cuda.synchronize()


def _stream(device):
    if torch.device(device).type != "cuda":
        return None
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def eager(row, X, device, poison=False, tag="eager"):
    slots = alloc(row.bufs, device)
    prime(slots, X, poison)
    row.call(views(slots), _stream(device))
    _sync(device)
    verify(slots, tag)
    return slots


def run_contract(row, device="cuda", graph=True):
    """The checks of the module docstring, each run once."""
    A = row.make(1)
    slots = eager(row, A, device, tag="eager set A")
    row.check(views(slots), A)
    resA = outputs(slots)
    prime(slots, A, True)
    row.call(views(slots), _stream(device))
    _sync(device)
    verify(slots, "poisoned eager set A", resA)
    if not graph:
        return
    Bx = row.make(2)
    resB = outputs(eager(row, Bx, device, tag="eager set B"))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        row.call(views(slots), _stream(device))
    prime(slots, Bx, True)
    g.replay()
    torch.cuda.synchronize()
    verify(slots, "graph replay of set B", resB)
    del g


# ---------------------------------------------------------------------------------------------- row helpers
ROWS = {}        # row name -> (symbols it calls, factory)
ATTR_ROWS = []   # one row per entry point that raises its kernel's dynamic shared-memory limit


def row(name, *symbols, attr=False):
    def deco(fn):
        assert name not in ROWS, name
        ROWS[name] = (symbols, fn)
        if attr:
            ATTR_ROWS.append(name)
        return fn
    return deco


def _rn(g, *shape, scale=1.0, dtype=torch.float32):
    return torch.randn(shape, device="cuda", generator=g, dtype=dtype) * scale


def _bh_numel(B, H, W):
    return _lib()[1].mrb_bh_bytes(B, H, W) // 2


def _bh_border(B, H, W, per=128):
    """bool over the bf16 elements of a BH-geometry tensor: True on the 2-pixel border."""
    m = torch.ones((B, H + 4, W + 4), dtype=torch.bool)
    m[:, 2:H + 2, 2:W + 2] = False
    return m[..., None].expand(B, H + 4, W + 4, per).reshape(-1)


def _to_bh(x, B, H, W):
    L, lib, st = _lib()
    buf = torch.empty(_bh_numel(B, H, W), dtype=torch.bfloat16, device="cuda")
    L.check(lib.mrb_bh_from_nhwc(L.ptr(x), L.ptr(buf), B, H, W, st))
    return buf


def _split(v, B, H, W, per):
    """[B, H+4, W+4, hi per | lo per] bf16 -> fp64 hi + lo, [B, H+4, W+4, per]."""
    t = v.reshape(B, H + 4, W + 4, 2, per).double()
    return t[..., 0, :] + t[..., 1, :]


def _replicated(t, H, W):
    """t [B, H+4, W+4, ...] -> the same tensor with its 2-pixel border replaced by copies of the nearest interior pixel."""
    iy = ((torch.arange(H + 4) - 2).clamp(0, H - 1) + 2).to(t.device)
    ix = ((torch.arange(W + 4) - 2).clamp(0, W - 1) + 2).to(t.device)
    return t[:, iy][:, :, ix]


def _interior_nchw(t, H, W):
    return t[:, 2:H + 2, 2:W + 2].permute(0, 3, 1, 2)


def _nchw(x):
    return x.permute(0, 3, 1, 2).double()


# ---------------------------------------------------------------------------------------------- FFT, roll, complex ops
def _fft1d_row(outer, n, inner, inverse, in_rot, out_rot, scale):
    N = outer * n * inner * 2

    def make(seed):
        return {"x": _rn(_gen(seed), N)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_fft1d_c2c(L.ptr(V["x"]), L.ptr(V["out"]), outer, n, inner, inverse, in_rot, out_rot, scale, st))

    def check(V, X):
        x = torch.view_as_complex(X["x"].double().reshape(outer, n, inner, 2))
        ref = torch.view_as_real(_fft_ref(x, inverse, in_rot, out_rot, scale))
        check_slices("fft1d n=%d [%d,%d,%d]" % (n, outer, n, inner), V["out"].reshape(outer, n, inner, 2), ref, 2e-6)

    return Row({"x": Buf("in", N), "out": Buf("out", N)}, make, call, check)


row("fft1d_n1", "mrb_fft1d_c2c")(lambda: _fft1d_row(3, 1, 5, 0, 0, 0, 0.5))
row("fft1d_prime_331", "mrb_fft1d_c2c")(lambda: _fft1d_row(2, 331, 3, 1, 165, 165, 1.0 / 331))
row("fft1d_320", "mrb_fft1d_c2c")(lambda: _fft1d_row(5, 320, 1, 0, 160, 160, 1.0))
row("fft1d_640", "mrb_fft1d_c2c")(lambda: _fft1d_row(2, 640, 3, 1, 320, 320, 1.0 / 640))


@row("fft2_33x320_centred", "mrb_fft2_c2c")
def _fft2_row():
    B, H, W = 2, 33, 320
    N = B * H * W * 2

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_fft2_c2c(L.ptr(V["x"]), L.ptr(V["out"]), B, H, W, 1, 1, 1, st))

    def check(V, X):
        z = torch.fft.ifftshift(torch.view_as_complex(X["x"].double().reshape(B, H, W, 2)), dim=(-2, -1))
        ref = torch.fft.fftshift(torch.fft.ifft2(z, norm="ortho"), dim=(-2, -1))
        check_slices("fft2 inverse centred [2, 33, 320]", V["out"].reshape(B, H, W, 2), torch.view_as_real(ref), 2e-6)

    return Row({"x": Buf("in", N), "out": Buf("out", N)}, lambda s: {"x": _rn(_gen(s), N)}, call, check)


@row("roll", "mrb_roll")
def _roll_row():
    shape = (3, 7, 5)

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_roll(L.ptr(V["x"]), L.ptr(V["out"]), 3, 7, 5, 4, 3, st))

    def check(V, X):
        assert torch.equal(V["out"].reshape(shape), torch.roll(X["x"].reshape(shape), 3, 1))

    return Row({"x": Buf("in", 105), "out": Buf("out", 105)}, lambda s: {"x": _rn(_gen(s), 105)}, call, check)


@row("complex_mul_broadcast_conj", "mrb_complex_mul")
def _cmul_row():
    xs, ys = (2, 5, 9, 11), (1, 5, 1, 11)
    shape = (ctypes.c_longlong * 4)(*xs)
    xst = (ctypes.c_longlong * 4)(495, 99, 11, 1)
    yst = (ctypes.c_longlong * 4)(0, 11, 0, 1)
    nx, ny = 990 * 2, 55 * 2

    def make(seed):
        g = _gen(seed)
        return {"x": _rn(g, nx), "y": _rn(g, ny)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_complex_mul(L.ptr(V["x"]), L.ptr(V["y"]), L.ptr(V["out"]), 4, shape, xst, yst, 1, st))

    def check(V, X):
        xc = torch.view_as_complex(X["x"].double().reshape(*xs, 2))
        yc = torch.view_as_complex(X["y"].double().reshape(*ys, 2))
        check_slices("complex_mul conj_y broadcast", V["out"].reshape(*xs, 2), torch.view_as_real(xc * yc.conj()), 2e-6)

    return Row({"x": Buf("in", nx), "y": Buf("in", ny), "out": Buf("out", nx)}, make, call, check)


def _pointwise_row(symbol, n_out, args, ref):
    """complex_conj / complex_abs on n = 999 complex values."""
    n = 999

    def call(V, st):
        L, lib, _ = _lib()
        L.check(getattr(lib, symbol)(L.ptr(V["x"]), L.ptr(V["out"]), n, *args, st))

    def check(V, X):
        ref(V["out"], torch.view_as_complex(X["x"].double().reshape(n, 2)), X["x"].reshape(n, 2))

    return Row({"x": Buf("in", 2 * n), "out": Buf("out", n_out * n)}, lambda s: {"x": _rn(_gen(s), 2 * n)}, call, check)


row("complex_conj", "mrb_complex_conj")(lambda: _pointwise_row(
    "mrb_complex_conj", 2, (), lambda o, xc, x: _assert_equal(o.reshape(-1, 2), torch.stack((x[:, 0], -x[:, 1]), -1))))
row("complex_abs", "mrb_complex_abs")(lambda: _pointwise_row(
    "mrb_complex_abs", 1, (0,), lambda o, xc, x: check_slices("complex_abs", o[None], xc.abs()[None], 2e-6)))


def _assert_equal(a, b):
    assert torch.equal(a, b)


def _coil_row(symbol, complex_in, complex_out, ref):
    """rss / rss_complex / sense_combine / divide_rss on [outer 2, C 5, inner 99] (inner odd: no vector path)."""
    outer, C, inner = 2, 5, 99
    k = 2 if complex_in else 1
    nin = outer * C * inner * k
    nout = nin if symbol == "mrb_divide_rss" else outer * inner * (2 if complex_out else 1)
    two = symbol == "mrb_sense_combine"
    bufs = {"x": Buf("in", nin), "out": Buf("out", nout)}
    if two:
        bufs["S"] = Buf("in", nin)

    def make(seed):
        g = _gen(seed)
        return {"x": _rn(g, nin), "S": _rn(g, nin)} if two else {"x": _rn(g, nin)}

    def call(V, st):
        L, lib, _ = _lib()
        fn = getattr(lib, symbol)
        if two:
            L.check(fn(L.ptr(V["x"]), L.ptr(V["S"]), L.ptr(V["out"]), outer, C, inner, st))
        else:
            L.check(fn(L.ptr(V["x"]), L.ptr(V["out"]), outer, C, inner, st))

    def check(V, X):
        x = X["x"].double().reshape(outer, C, inner, k)
        x = torch.view_as_complex(x) if complex_in else x[..., 0]
        S = torch.view_as_complex(X["S"].double().reshape(outer, C, inner, 2)) if two else None
        r = ref(x, S)
        r = torch.view_as_real(r) if r.is_complex() else r
        check_slices(symbol, V["out"].reshape(r.shape), r, 2e-6)

    return Row(bufs, make, call, check)


row("rss", "mrb_rss")(lambda: _coil_row("mrb_rss", False, False, lambda x, S: x.pow(2).sum(1).sqrt()))
row("rss_complex", "mrb_rss_complex")(lambda: _coil_row("mrb_rss_complex", True, False,
                                                        lambda x, S: x.abs().pow(2).sum(1).sqrt()))
row("sense_combine", "mrb_sense_combine")(lambda: _coil_row("mrb_sense_combine", True, True,
                                                            lambda x, S: (x * S.conj()).sum(1)))
row("divide_rss", "mrb_divide_rss")(lambda: _coil_row("mrb_divide_rss", True, True,
                                                      lambda x, S: x / x.abs().pow(2).sum(1, keepdim=True).sqrt()))


# ---------------------------------------------------------------------------------------------- data consistency
def _canon(m, B, H, W):
    from mridc_b200 import _ops

    mc, code, mb, mh = _ops.canonical_mask(m, B, H, W)
    return mc, code, mb, mh


def _dc_set(B, C, H, W, kind, two_d, seed):
    """y, S, eta from the seed; the mask is the same for every seed (the packed hybrid rows depend on it)."""
    y, S, eta, _ = _dc_inputs(B, C, H, W, seed)
    m = _mask(kind, B, H, W, _gen(777), two_d=two_d)
    return y, S, eta, m


def _mask_buf(mc):
    return Buf("in", mc.numel(), mc.dtype)


def _dc_grad_ref(X, centered):
    from oracle import nets as onets

    return onets.log_likelihood_gradient(X["_eta"].double(), X["_y"].double(), X["_S"].double(), X["_m"].double(), 1.3,
                                         centered, _norm(centered), [-2, -1], 1)


def _check_grad(tag, out, X, B, H, W, nhwc, centered):
    out = out.reshape(B, H, W, 4).permute(0, 3, 1, 2) if nhwc else out.reshape(B, 4, H, W)
    assert torch.equal(out[:, :2], X["_eta"].permute(0, 3, 1, 2)), tag + ": eta channels"
    check_slices(tag, out[:, 2:], _dc_grad_ref(X, centered)[:, 2:], 2e-6)


def _dc3_row(B, C, H, W, kind, centered, nhwc):
    """mrb_dc_rim_grad (general three-pass form) with a 2-D mask."""
    L, lib, _ = _lib()
    mc = _canon(_dc_set(B, 1, H, W, kind, True, 0)[3], B, H, W)
    code, mb, mh = mc[1:]
    N = B * C * H * W * 2
    wsb = lib.mrb_dc_workspace_bytes(B, C, H, W)
    bufs = {"eta": Buf("in", B * H * W * 2), "y": Buf("in", N), "S": Buf("in", N), "mask": _mask_buf(mc[0]),
            "out": Buf("out", B * 4 * H * W), "ws": Buf("ws", wsb // 4)}

    def make(seed):
        y, S, eta, m = _dc_set(B, C, H, W, kind, True, seed)
        return {"eta": eta, "y": y, "S": S, "mask": _canon(m, B, H, W)[0], "_eta": eta, "_y": y, "_S": S, "_m": m}

    def call(V, st):
        L.check(lib.mrb_dc_rim_grad(L.ptr(V["eta"]), L.ptr(V["y"]), L.ptr(V["S"]), L.ptr(V["mask"]), code, mb, mh,
                                    1.0 / 1.3 ** 2, L.ptr(V["out"]), nhwc, B, C, H, W, int(centered),
                                    _lib_norm(centered), L.ptr(V["ws"]), wsb, st))

    def check(V, X):
        _check_grad("dc_rim_grad %dx%dx%dx%d 2-D mask" % (B, C, H, W), V["out"], X, B, H, W, nhwc, centered)

    return Row(bufs, make, call, check)


def _lib_norm(centered):
    return 1 if centered else 0  # _norm(): ortho when centred, backward otherwise


row("dc_rim_grad_w96_2d", "mrb_dc_rim_grad")(lambda: _dc3_row(2, 4, 40, 96, "u8-per-slice", True, 0))
row("dc_rim_grad_320_c15_2d", "mrb_dc_rim_grad")(lambda: _dc3_row(1, 15, 320, 320, "f32-shared", True, 1))
row("dc_rim_grad_320_c20_2d", "mrb_dc_rim_grad")(lambda: _dc3_row(1, 20, 320, 320, "u8-shared", False, 0))


def _packed_written(mc, B, C, H, W):
    """mrb_dc_hybrid_prepare writes, per (b, c, row), the first ns_b complex values (ns_b = sampled columns of slice b)."""
    ns = (mc.reshape(mc.shape[0], W) != 0).sum(1).cpu()
    ns = ns.expand(B) if ns.numel() == 1 else ns
    cols = torch.arange(W)[None, :] < ns[:, None]                       # [B, W]
    return cols[:, None, None, :, None].expand(B, C, H, W, 2).reshape(-1)


def _dch_prepare_row(B, C, H, W, kind, centered):
    from mridc_b200 import _ops

    L, lib, _ = _lib()
    mc, code, mb, _ = _canon(_dc_set(B, 1, H, W, kind, False, 0)[3], B, H, W)
    N = B * C * H * W * 2
    bufs = {"y": Buf("in", N), "mask": _mask_buf(mc), "yh": Buf("out", N, written=_packed_written(mc, B, C, H, W)),
            "ws": Buf("ws", N)}

    def make(seed):
        y, S, eta, m = _dc_set(B, C, H, W, kind, False, seed)
        return {"y": y, "mask": _canon(m, B, H, W)[0], "_eta": eta, "_y": y, "_S": S, "_m": m}

    def call(V, st):
        L.check(lib.mrb_dc_hybrid_prepare(L.ptr(V["y"]), L.ptr(V["mask"]), code, mb, L.ptr(V["yh"]), B, C, H, W,
                                          int(centered), L.ptr(V["ws"]), N * 4, st))

    def check(V, X):
        # the hybrid k-space has no plain reference of its own: the gradient computed from it is compared with fp64
        yh = V["yh"].reshape(B, C, H, W, 2)
        g = _ops.dc_rim_grad(X["_eta"], X["_y"], X["_S"], mc, 1.3, centered, _norm(centered), y_hybrid=yh)
        _check_grad("dc_hybrid_prepare %dx%dx%dx%d -> gradient" % (B, C, H, W), g, X, B, H, W, False, centered)

    return Row(bufs, make, call, check)


row("dc_hybrid_prepare_w96", "mrb_dc_hybrid_prepare")(lambda: _dch_prepare_row(2, 4, 40, 96, "u8-per-slice", True))
row("dc_hybrid_prepare_320_c15", "mrb_dc_hybrid_prepare")(lambda: _dch_prepare_row(2, 15, 36, 320, "f32-shared", False))


def _g8_layout(B, H, W):
    """-> (bf16 elements of a G8 buffer, bool mask of its position region); guard positions: 2(W+4)+2 before."""
    L, lib, _ = _lib()
    n = lib.mrb_g8_bytes(B, H, W) // 2
    lo, Q = 2 * (W + 4) + 2, B * (H + 4) * (W + 4)
    m = torch.zeros(n, dtype=torch.bool)
    m[lo * 8:(lo + Q) * 8] = True
    return n, m, lo, Q


def _g8_positions(v, lo, Q, B, H, W):
    return v[lo * 8:(lo + Q) * 8].reshape(B, H + 4, W + 4, 8)


def _dch_grad_row(B, C, H, W, kind, centered, nhwc):
    """mrb_dc_rim_grad_hybrid: nhwc 0 / 1 (fp32 outputs), 2 (G8 output: W = 320, C <= 16)."""
    from mridc_b200 import _ops

    L, lib, _ = _lib()
    mc, code, mb, _ = _canon(_dc_set(B, 1, H, W, kind, False, 0)[3], B, H, W)
    N = B * C * H * W * 2
    if nhwc == 2:
        n8, w8, lo, Q = _g8_layout(B, H, W)
        out = Buf("g8", n8, torch.bfloat16, written=w8)
    else:
        out = Buf("out", B * 4 * H * W)
    bufs = {"eta": Buf("in", B * H * W * 2), "yh": Buf("in", N), "S": Buf("in", N), "mask": _mask_buf(mc), "out": out}

    def make(seed):
        y, S, eta, m = _dc_set(B, C, H, W, kind, False, seed)
        mcs = _canon(m, B, H, W)[0]
        yh = _ops.dc_hybrid_prepare(y, mcs, centered)
        # the tail of each packed row is not part of the hybrid k-space: fixed bytes, the same in both sets
        yh.view(-1)[~_packed_written(mcs, B, C, H, W).cuda()] = 0.0
        return {"eta": eta, "yh": yh, "S": S, "mask": mcs, "_eta": eta, "_y": y, "_S": S, "_m": m, "_mc": mcs, "_yh": yh}

    def call(V, st):
        L.check(lib.mrb_dc_rim_grad_hybrid(L.ptr(V["eta"]), L.ptr(V["yh"]), L.ptr(V["S"]), L.ptr(V["mask"]), code, mb,
                                           1.0 / 1.3 ** 2, L.ptr(V["out"]), nhwc, B, C, H, W, int(centered),
                                           _lib_norm(centered), st))

    def check(V, X):
        tag = "dc_rim_grad_hybrid %dx%dx%dx%d nhwc=%d" % (B, C, H, W, nhwc)
        if nhwc != 2:
            _check_grad(tag, V["out"], X, B, H, W, nhwc, centered)
            return
        # G8: the fp32 channels-last gradient (vs fp64) through mrb_g8_from_nhwc4, byte for byte
        g4 = _ops.dc_rim_grad(X["_eta"], X["_y"], X["_S"], X["_mc"], 1.3, centered, _norm(centered), nhwc=True,
                              y_hybrid=X["_yh"])
        _check_grad(tag + " (fp32 form)", g4, X, B, H, W, True, centered)
        ref = torch.zeros(n8, dtype=torch.bfloat16, device="cuda")
        L.check(lib.mrb_g8_from_nhwc4(L.ptr(g4), L.ptr(ref), B, H, W, _lib()[2]))
        assert torch.equal(V["out"].view(torch.int16), ref.view(torch.int16)), tag

    return Row(bufs, make, call, check)


row("dc_grad_hybrid_320_c15_g8", "mrb_dc_rim_grad_hybrid")(lambda: _dch_grad_row(2, 15, 36, 320, "u8-shared", False, 2))
row("dc_grad_hybrid_320_c20", "mrb_dc_rim_grad_hybrid")(lambda: _dch_grad_row(2, 20, 36, 320, "f32-per-slice", True, 0))
row("dc_grad_hybrid_w96", "mrb_dc_rim_grad_hybrid")(lambda: _dch_grad_row(2, 4, 40, 96, "u8-per-slice", True, 1))


def _sens_reduce_row(B, C, H, W, centered):
    from oracle import nets as onets

    L, lib, _ = _lib()
    N = B * C * H * W * 2
    bufs = {"x": Buf("in", N), "S": Buf("in", N), "out": Buf("out", B * H * W * 2), "ws": Buf("ws", N)}

    def make(seed):
        y, S, _, _ = _dc_inputs(B, C, H, W, seed)
        return {"x": y, "S": S}

    def call(V, st):
        L.check(lib.mrb_sens_reduce(L.ptr(V["x"]), L.ptr(V["S"]), L.ptr(V["out"]), B, C, H, W, int(centered),
                                    _lib_norm(centered), L.ptr(V["ws"]), N * 4, st))

    def check(V, X):
        x, S = (X[k].double().reshape(B, C, H, W, 2) for k in ("x", "S"))
        ref = onets.sens_reduce(x, S, centered, _norm(centered), [-2, -1], 1)[:, 0]
        check_slices("sens_reduce %dx%dx%dx%d" % (B, C, H, W), V["out"].reshape(B, H, W, 2), ref, 2e-6)

    return Row(bufs, make, call, check)


def _sens_expand_row(B, C, H, W, centered, kind):
    from oracle import nets as onets

    L, lib, _ = _lib()
    N = B * C * H * W * 2
    mc, code, mb, mh = _canon(_mask(kind, B, H, W, _gen(777)), B, H, W)
    bufs = {"img": Buf("in", B * H * W * 2), "S": Buf("in", N), "base": Buf("in", N), "pred": Buf("in", N),
            "y": Buf("in", N), "mask": _mask_buf(mc), "dcw": Buf("in", 1), "out": Buf("out", N), "ws": Buf("ws", N)}

    def make(seed):
        y, S, _, g = _dc_inputs(B, C, H, W, seed)
        return {"img": _rn(g, B * H * W * 2), "S": S, "base": _rn(g, N), "pred": _rn(g, N), "y": y, "mask": mc,
                "dcw": torch.rand(1, device="cuda", generator=g) + 0.5}

    def call(V, st):
        L.check(lib.mrb_sens_expand_softdc(L.ptr(V["img"]), L.ptr(V["S"]), L.ptr(V["base"]), L.ptr(V["pred"]),
                                           L.ptr(V["y"]), L.ptr(V["mask"]), code, mb, mh, L.ptr(V["dcw"]), 0,
                                           L.ptr(V["out"]), B, C, H, W, int(centered), _lib_norm(centered),
                                           L.ptr(V["ws"]), N * 4, st))

    def check(V, X):
        S, base, pred, y = (X[k].double().reshape(B, C, H, W, 2) for k in ("S", "base", "pred", "y"))
        E = onets.sens_expand(X["img"].double().reshape(B, 1, H, W, 2), S, centered, _norm(centered), [-2, -1])
        m = mc.reshape(mb, 1, mh, W, 1).bool()
        ref = base - torch.where(m, pred - y, torch.zeros((), dtype=torch.float64, device="cuda")) * X["dcw"].double() - E
        check_slices("sens_expand_softdc %dx%dx%dx%d" % (B, C, H, W), V["out"].reshape(B, C, H, W, 2), ref, 2e-6)

    return Row(bufs, make, call, check)


row("sens_reduce_640x320", "mrb_sens_reduce")(lambda: _sens_reduce_row(1, 4, 640, 320, True))
row("sens_reduce_w96", "mrb_sens_reduce")(lambda: _sens_reduce_row(2, 3, 40, 96, False))
row("sens_expand_softdc_640x320", "mrb_sens_expand_softdc")(lambda: _sens_expand_row(1, 3, 640, 320, True, "f32-per-slice"))
row("sens_expand_softdc_w96", "mrb_sens_expand_softdc")(lambda: _sens_expand_row(2, 3, 40, 96, False, "u8-shared"))


# ---------------------------------------------------------------------------------------------- fp32 regulariser kernels
def _batch_rows(N, row_len, used):
    """bool over [N, row_len]: the first `used` values of each batch row (an output inside a concat buffer)."""
    m = torch.zeros((N, row_len), dtype=torch.bool)
    m[:, :used] = True
    return m.reshape(-1)


@row("conv2d_concat_odd", "mrb_conv2d")
def _conv2d_concat_row():
    """3x3 replicate conv, ReLU, odd 19 x 37 (partial 4 x 32 tiles), written at a batch stride inside a concat buffer
    (two channels of each sample belong to another producer)."""
    from mridc_b200 import _ops

    N, Cin, Cout, H, W = 2, 5, 16, 19, 37
    HW = H * W
    xbs, obs = Cin * HW + 13, (Cout + 2) * HW
    bufs = {"x": Buf("in", N * xbs), "w": Buf("in", Cout * Cin * 9), "b": Buf("in", Cout),
            "out": Buf("out", N * obs, written=_batch_rows(N, obs, Cout * HW))}

    def make(seed):
        g = _gen(seed)
        return {"x": _rn(g, N * xbs), "w": _rn(g, Cout * Cin * 9, scale=(Cin * 9) ** -0.5), "b": _rn(g, Cout)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_conv2d(L.ptr(V["x"]), xbs, L.ptr(V["w"]), L.ptr(V["b"]), L.ptr(V["out"]), obs, N, Cin, Cout, H, W,
                               3, 1, _ops.PAD_REPLICATE, _ops.ACT_RELU, 0.0, None, None, None, 0, st))

    def check(V, X):
        x = X["x"].reshape(N, xbs)[:, :Cin * HW].reshape(N, Cin, H, W).double()
        ref = F.relu(F.conv2d(F.pad(x, (1, 1, 1, 1), mode="replicate"), X["w"].double().reshape(Cout, Cin, 3, 3),
                              X["b"].double()))
        check_slices("conv2d concat 19x37", V["out"].reshape(N, obs)[:, :Cout * HW].reshape(N, Cout, H, W), ref, 2e-6)

    return Row(bufs, make, call, check)


@row("conv2d_add_residual_nhwc", "mrb_conv2d")
def _conv2d_residual_row():
    """5x5 zero-padded conv with the IndRNN add * add_scale term and leaky ReLU, ADDED to a channels-last residual."""
    from mridc_b200 import _ops

    N, Cin, Cout, H, W = 2, 3, 8, 17, 33
    HW = H * W
    bufs = {"x": Buf("in", N * Cin * HW), "w": Buf("in", Cout * Cin * 25), "b": Buf("in", Cout),
            "add": Buf("in", N * Cout * HW), "scale": Buf("in", Cout), "res": Buf("in", N * HW * Cout),
            "out": Buf("out", N * HW * Cout)}

    def make(seed):
        g = _gen(seed)
        return {"x": _rn(g, N * Cin * HW), "w": _rn(g, Cout * Cin * 25, scale=(Cin * 25) ** -0.5), "b": _rn(g, Cout),
                "add": _rn(g, N * Cout * HW), "scale": _rn(g, Cout), "res": _rn(g, N * HW * Cout)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_conv2d(L.ptr(V["x"]), Cin * HW, L.ptr(V["w"]), L.ptr(V["b"]), L.ptr(V["out"]), Cout * HW, N, Cin,
                               Cout, H, W, 5, 1, _ops.PAD_ZERO, _ops.ACT_LEAKY, 0.2, L.ptr(V["add"]), L.ptr(V["scale"]),
                               L.ptr(V["res"]), 1, st))

    def check(V, X):
        x = X["x"].reshape(N, Cin, H, W).double()
        ref = F.conv2d(x, X["w"].double().reshape(Cout, Cin, 5, 5), X["b"].double(), padding=2)
        ref = F.leaky_relu(ref + X["scale"].double()[:, None, None] * X["add"].double().reshape(N, Cout, H, W), 0.2)
        ref = X["res"].double().reshape(N, H, W, Cout) + ref.permute(0, 2, 3, 1)
        check_slices("conv2d add + residual", V["out"].reshape(N, H, W, Cout), ref, 2e-6)

    return Row(bufs, make, call, check)


def _cell_row(symbol):
    from oracle import nets as onets

    N, Cx, Ch, H, W = 2, 12, 20, 9, 17
    HW = H * W
    gates = {"mrb_gru_cell_1x1": 0, "mrb_gru_gates": 3, "mrb_mgu_gates": 2}[symbol]
    if gates == 0:
        bufs = {"x": Buf("in", N * Cx * HW), "h": Buf("in", N * Ch * HW), "wih": Buf("in", 3 * Ch * Cx),
                "bih": Buf("in", 3 * Ch), "whh": Buf("in", 3 * Ch * Ch), "out": Buf("out", N * Ch * HW)}
    else:
        bufs = {"ih": Buf("in", N * gates * Ch * HW), "hh": Buf("in", N * gates * Ch * HW), "h": Buf("in", N * Ch * HW),
                "out": Buf("out", N * Ch * HW)}

    def make(seed):
        g = _gen(seed)
        return {k: _rn(g, b.numel, scale=0.3 if k in ("wih", "whh") else 1.0) for k, b in bufs.items() if b.role == "in"}

    def call(V, st):
        L, lib, _ = _lib()
        if gates == 0:
            L.check(lib.mrb_gru_cell_1x1(L.ptr(V["x"]), L.ptr(V["h"]), L.ptr(V["wih"]), L.ptr(V["bih"]), L.ptr(V["whh"]),
                                         L.ptr(V["out"]), N, Cx, Ch, HW, st))
        else:
            L.check(getattr(lib, symbol)(L.ptr(V["ih"]), L.ptr(V["hh"]), L.ptr(V["h"]), L.ptr(V["out"]), N, Ch, HW, st))

    def check(V, X):
        h = X["h"].double().reshape(N, Ch, H, W)
        if gates == 0:
            ref = onets.conv_gru_cell(X["x"].double().reshape(N, Cx, H, W), h, X["wih"].double().reshape(3 * Ch, Cx, 1, 1),
                                      X["bih"].double(), X["whh"].double().reshape(3 * Ch, Ch, 1, 1), 1, 1)
        else:
            a = X["ih"].double().reshape(N, gates * Ch, H, W).chunk(gates, 1)
            b = X["hh"].double().reshape(N, gates * Ch, H, W).chunk(gates, 1)
            if gates == 3:
                r, z = torch.sigmoid(a[0] + b[0]), torch.sigmoid(a[1] + b[1])
                ref = torch.tanh(a[2] + r * b[2]) * (1 - z) + z * h
            else:
                f = torch.sigmoid(a[0] + b[0])
                c = torch.tanh(a[1] + f * b[1])
                ref = c + f * (h - c)
        check_slices(symbol, V["out"].reshape(N, Ch, H, W), ref, 2e-6)

    return Row(bufs, make, call, check)


for _s in ("mrb_gru_cell_1x1", "mrb_gru_gates", "mrb_mgu_gates"):
    row(_s[4:], _s)(lambda _s=_s: _cell_row(_s))


def _instnorm_row(N, C, HW, out_extra):
    """x [N, C, HW] -> out at batch stride (C + out_extra) * HW (the extra channels belong to another producer)."""
    obs = (C + out_extra) * HW
    bufs = {"x": Buf("in", N * C * HW), "out": Buf("out", N * obs, written=_batch_rows(N, obs, C * HW)),
            "stats": Buf("ws", 2 * N * C, torch.float64)}

    def make(seed):
        return {"x": _rn(_gen(seed), N * C * HW, scale=1.5) + 0.3}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_instnorm_lrelu(L.ptr(V["x"]), C * HW, L.ptr(V["out"]), obs, N, C, HW, 1e-5, 0.2, L.ptr(V["stats"]),
                                       st))

    def check(V, X):
        check_slices("instnorm HW=%d" % HW, V["out"].reshape(N, obs)[:, :C * HW].reshape(N, C, HW),
                     _instnorm_ref(X["x"], N, C, HW), 2e-6)

    return Row(bufs, make, call, check)


row("instnorm_cluster_concat", "mrb_instnorm_lrelu", attr=True)(lambda: _instnorm_row(2, 3, 4099, 2))
row("instnorm_two_pass_720x720", "mrb_instnorm_lrelu")(lambda: _instnorm_row(1, 2, 720 * 720, 1))


@row("conv1x1_strided", "mrb_conv1x1")
def _conv1x1_row():
    N, Cin, Cout, HW = 2, 6, 5, 13 * 20
    xbs, obs = Cin * HW + 4, Cout * HW + 8
    bufs = {"x": Buf("in", N * xbs), "w": Buf("in", Cout * Cin), "b": Buf("in", Cout),
            "out": Buf("out", N * obs, written=_batch_rows(N, obs, Cout * HW))}

    def make(seed):
        g = _gen(seed)
        return {"x": _rn(g, N * xbs), "w": _rn(g, Cout * Cin), "b": _rn(g, Cout)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_conv1x1(L.ptr(V["x"]), xbs, L.ptr(V["w"]), L.ptr(V["b"]), L.ptr(V["out"]), obs, N, Cin, Cout, HW, st))

    def check(V, X):
        x = X["x"].reshape(N, xbs)[:, :Cin * HW].reshape(N, Cin, HW).double()
        ref = torch.einsum("oc,nch->noh", X["w"].double().reshape(Cout, Cin), x) + X["b"].double()[:, None]
        check_slices("conv1x1", V["out"].reshape(N, obs)[:, :Cout * HW].reshape(N, Cout, HW), ref, 2e-6)

    return Row(bufs, make, call, check)


@row("avgpool2_odd", "mrb_avgpool2")
def _avgpool_row():
    N, C, H, W = 2, 3, 13, 21

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_avgpool2(L.ptr(V["x"]), C * H * W, L.ptr(V["out"]), C * 6 * 10, N, C, H, W, st))

    def check(V, X):
        check_slices("avgpool2 13x21", V["out"].reshape(N, C, 6, 10), F.avg_pool2d(X["x"].double().reshape(N, C, H, W), 2),
                     2e-6)

    return Row({"x": Buf("in", N * C * H * W), "out": Buf("out", N * C * 60)}, lambda s: {"x": _rn(_gen(s), N * C * H * W)},
               call, check)


@row("conv_transpose2x2", "mrb_conv_transpose2x2")
def _convt_row():
    N, Cin, Cout, H, W = 2, 6, 5, 13, 19

    def make(seed):
        g = _gen(seed)
        return {"x": _rn(g, N * Cin * H * W), "w": _rn(g, Cin * Cout * 4)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_conv_transpose2x2(L.ptr(V["x"]), Cin * H * W, L.ptr(V["w"]), L.ptr(V["out"]), Cout * 4 * H * W, N,
                                          Cin, Cout, H, W, st))

    def check(V, X):
        ref = F.conv_transpose2d(X["x"].double().reshape(N, Cin, H, W), X["w"].double().reshape(Cin, Cout, 2, 2), stride=2)
        check_slices("conv_transpose2x2", V["out"].reshape(N, Cout, 2 * H, 2 * W), ref, 2e-6)

    return Row({"x": Buf("in", N * Cin * H * W), "w": Buf("in", Cin * Cout * 4), "out": Buf("out", N * Cout * 4 * H * W)},
               make, call, check)


def _pad_row(mode, Ho, Wo, oy, ox):
    N, C, H, W = 2, 3, 13, 20
    modes = {0: "constant", 1: "replicate", 2: "reflect"}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_pad2d(L.ptr(V["x"]), C * H * W, L.ptr(V["out"]), C * Ho * Wo, N, C, H, W, Ho, Wo, oy, ox, mode, st))

    def check(V, X):
        x = X["x"].reshape(N, C, H, W)
        if oy >= 0:
            ref = F.pad(x, (ox, Wo - W - ox, oy, Ho - H - oy), mode=modes[mode])
        else:
            ref = x[:, :, -oy:-oy + Ho, -ox:-ox + Wo]
        assert torch.equal(V["out"].reshape(N, C, Ho, Wo), ref)

    return Row({"x": Buf("in", N * C * H * W), "out": Buf("out", N * C * Ho * Wo)}, lambda s: {"x": _rn(_gen(s), N * C * H * W)},
               call, check)


row("pad2d_reflect", "mrb_pad2d")(lambda: _pad_row(2, 18, 26, 2, 3))
row("pad2d_crop", "mrb_pad2d")(lambda: _pad_row(1, 9, 14, -2, -3))


@row("normunet_in", "mrb_normunet_in")
def _normunet_in_row():
    B, C, HW = 2, 3, 37 * 29
    bufs = {"x": Buf("in", B * C * HW * 2), "out": Buf("out", B * 2 * C * HW), "ms": Buf("out", B * 4),
            "stats": Buf("ws", 4 * B, torch.float64)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_normunet_in(L.ptr(V["x"]), L.ptr(V["out"]), L.ptr(V["ms"]), B, C, HW, 1, L.ptr(V["stats"]), st))

    def check(V, X):
        planes = X["x"].double().reshape(B, C * HW, 2).permute(0, 2, 1)
        mean, std = planes.mean(-1, keepdim=True), planes.std(-1, keepdim=True)
        check_slices("normunet_in mean/std", V["ms"].reshape(B, 2, 2), torch.cat((mean, std), -1), 2e-6)
        check_slices("normunet_in", V["out"].reshape(B, -1), ((planes - mean) / std).reshape(B, -1), 2e-6)

    return Row(bufs, lambda s: {"x": _rn(_gen(s), B * C * HW * 2, scale=2.0) + 0.5}, call, check)


@row("normunet_out", "mrb_normunet_out")
def _normunet_out_row():
    B, C, HW = 2, 3, 37 * 29

    def make(seed):
        g = _gen(seed)
        ms = torch.stack((_rn(g, B, 2), torch.rand((B, 2), device="cuda", generator=g) + 0.5), -1)
        return {"x": _rn(g, B * 2 * C * HW), "ms": ms.reshape(-1)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_normunet_out(L.ptr(V["x"]), L.ptr(V["ms"]), L.ptr(V["out"]), B, C, HW, 1, st))

    def check(V, X):
        ms = X["ms"].double().reshape(B, 2, 2)
        pl = X["x"].double().reshape(B, 2, C * HW) * ms[:, :, 1:] + ms[:, :, :1]
        check_slices("normunet_out", V["out"].reshape(B, -1), pl.permute(0, 2, 1).reshape(B, -1), 2e-6)

    return Row({"x": Buf("in", B * 2 * C * HW), "ms": Buf("in", B * 4), "out": Buf("out", B * C * HW * 2)}, make, call, check)


# ---------------------------------------------------------------------------------------------- tensor-core engine (BH, G8)
# B = 1, H = 9, W = 28 (the narrowest width the engine covers): Q = B (H+4)(W+4) = 416 positions, 3.25 BH tiles of 128
BH_B, BH_H, BH_W = 1, 9, 28


def _pack_conv(w, k):
    L, lib, st = _lib()
    pk = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, k), device="cuda")
    L.check(lib.mrb_tc_pack_conv(L.ptr(w), L.ptr(pk), 64, 64, k, st))
    return pk


def _tc_conv_ref(xb, w, b, B, H, W, k, dil, relu):
    from oracle import nets as onets

    x = _interior_nchw(_split(xb, B, H, W, 64), H, W)
    return onets.conv_nonlinear(x, w.double().reshape(64, 64, k, k), None if b is None else b.double(), k, dil,
                                "relu" if relu else None)


def _bh_out(B, H, W):
    """A BH output written at every position whose border is not a replicate copy: only the interior is defined."""
    return Buf("out", _bh_numel(B, H, W), torch.bfloat16, defined=~_bh_border(B, H, W))


def _check_bh(tag, v, ref, B, H, W):
    check_slices(tag, _interior_nchw(_split(v, B, H, W, 64), H, W), ref, 1e-5)


@row("tc_pack_conv", "mrb_tc_pack_conv")
def _tc_pack_row():
    L, lib, _ = _lib()
    B, H, W, k = BH_B, BH_H, BH_W, 3
    bufs = {"w": Buf("in", 64 * 64 * 9), "dst": Buf("out", lib.mrb_tc_packed_floats(0, 64, 64, k))}

    def make(seed):
        g = _gen(seed)
        x = _rn(g, B, H, W, 64)
        return {"w": _rn(g, 64 * 64 * 9, scale=(64 * 9) ** -0.5), "_xb": _to_bh(x, B, H, W)}

    def call(V, st):
        L.check(lib.mrb_tc_pack_conv(L.ptr(V["w"]), L.ptr(V["dst"]), 64, 64, k, st))

    def check(V, X):
        # the packed image has no plain reference: the conv that consumes it is compared with fp64
        ob = torch.empty(_bh_numel(B, H, W), dtype=torch.bfloat16, device="cuda")
        L.check(lib.mrb_tc_conv_bh(L.ptr(X["_xb"]), L.ptr(V["dst"]), None, L.ptr(ob), B, H, W, 64, k, 2, 0, _lib()[2]))
        _check_bh("tc_pack_conv -> tc_conv_bh", ob, _tc_conv_ref(X["_xb"], X["w"], None, B, H, W, k, 2, False), B, H, W)

    return Row(bufs, make, call, check)


@row("bh_from_nhwc", "mrb_bh_from_nhwc")
def _bh_from_row(B=2, H=5, W=29):

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_bh_from_nhwc(L.ptr(V["x"]), L.ptr(V["out"]), B, H, W, st))

    def check(V, X):
        v = V["out"].reshape(B, H + 4, W + 4, 128)
        assert torch.equal(v.view(torch.int16), _replicated(v, H, W).view(torch.int16)), "BH border is not a replicate copy"
        check_slices("bh_from_nhwc hi + lo", _interior_nchw(_split(v, B, H, W, 64), H, W), _nchw(X["x"].reshape(B, H, W, 64)),
                     1e-5)

    n = B * H * W * 64
    return Row({"x": Buf("in", n), "out": Buf("out", _bh_numel(B, H, W), torch.bfloat16)}, lambda s: {"x": _rn(_gen(s), n)},
               call, check)


@row("bh_to_nhwc", "mrb_bh_to_nhwc")
def _bh_to_row(B=2, H=5, W=29):
    n = B * H * W * 64

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_bh_to_nhwc(L.ptr(V["x"]), L.ptr(V["out"]), B, H, W, st))

    def check(V, X):
        t = X["x"].reshape(B, H + 4, W + 4, 2, 64)[:, 2:H + 2, 2:W + 2].float()
        assert torch.equal(V["out"].reshape(B, H, W, 64), t[..., 0, :] + t[..., 1, :])  # hi + lo is exact in fp32

    bufs = {"x": Buf("in", _bh_numel(B, H, W), torch.bfloat16, unread=_bh_border(B, H, W)), "out": Buf("out", n)}
    return Row(bufs, lambda s: {"x": _to_bh(_rn(_gen(s), n), B, H, W)}, call, check)


@row("bh_fix_border", "mrb_bh_fix_border")
def _bh_fix_row(B=2, H=5, W=29):
    border = _bh_border(B, H, W)
    n = B * H * W * 64

    def make(seed):
        ref = _to_bh(_rn(_gen(seed), n), B, H, W)
        bh = ref.clone()
        bh.view(torch.uint8).view(-1, 2)[border.cuda()] = SENTINEL  # what the producer left there
        return {"bh": bh, "_ref": ref}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_bh_fix_border(L.ptr(V["bh"]), B, H, W, st))

    def check(V, X):
        assert torch.equal(V["bh"].view(torch.int16), X["_ref"].view(torch.int16))

    return Row({"bh": Buf("inout", _bh_numel(B, H, W), torch.bfloat16, written=border, unread=border)}, make, call, check)


@row("tc_conv_bh_w28", "mrb_tc_conv_bh", attr=True)
def _tc_conv_row(B=BH_B, H=BH_H, W=BH_W, k=3, dil=2):
    L, lib, _ = _lib()
    npk = lib.mrb_tc_packed_floats(0, 64, 64, k)
    bufs = {"x": Buf("in", _bh_numel(B, H, W), torch.bfloat16), "wp": Buf("in", npk), "b": Buf("in", 64),
            "out": _bh_out(B, H, W)}

    def make(seed):
        g = _gen(seed)
        w = _rn(g, 64 * 64 * k * k, scale=(64 * k * k) ** -0.5)
        return {"x": _to_bh(_rn(g, B * H * W * 64), B, H, W), "wp": _pack_conv(w, k), "b": _rn(g, 64), "_w": w}

    def call(V, st):
        L.check(lib.mrb_tc_conv_bh(L.ptr(V["x"]), L.ptr(V["wp"]), L.ptr(V["b"]), L.ptr(V["out"]), B, H, W, 64, k, dil, 1, st))

    def check(V, X):
        _check_bh("tc_conv_bh %dx%d d%d %dx%dx%d" % (k, k, dil, B, H, W), V["out"],
                  _tc_conv_ref(X["x"], X["_w"], X["b"], B, H, W, k, dil, True), B, H, W)

    return Row(bufs, make, call, check)


def _final_conv_row(symbol, B, H, W):
    """eta + conv3x3(x) (+ bias): mrb_conv_c2_bh_residual reads the replicate border, mrb_tc2_final_conv never does."""
    from oracle import nets as onets

    L, lib, _ = _lib()
    tc = symbol == "mrb_tc2_final_conv"
    nb = _bh_numel(B, H, W)
    bufs = {"x": Buf("in", nb, torch.bfloat16, unread=_bh_border(B, H, W) if tc else None), "w": Buf("in", 2 * 64 * 9),
            "b": Buf("in", 2), "eta": Buf("in", B * H * W * 2), "out": Buf("out", B * H * W * 2)}

    def make(seed):
        g = _gen(seed)
        return {"x": _to_bh(_rn(g, B * H * W * 64), B, H, W), "w": _rn(g, 2 * 64 * 9, scale=0.05), "b": _rn(g, 2),
                "eta": _rn(g, B * H * W * 2)}

    def call(V, st):
        L.check(getattr(lib, symbol)(L.ptr(V["x"]), L.ptr(V["w"]), L.ptr(V["b"]), L.ptr(V["eta"]), L.ptr(V["out"]), B, H,
                                     W, st))

    def check(V, X):
        x = _interior_nchw(_split(X["x"], B, H, W, 64), H, W)
        conv = onets.conv_nonlinear(x, X["w"].double().reshape(2, 64, 3, 3), X["b"].double(), 3, 1, None)
        eta = X["eta"].double().reshape(B, H, W, 2)
        ref = eta + conv.permute(0, 2, 3, 1)
        mag = onets.conv_nonlinear(x.abs(), X["w"].double().abs().reshape(2, 64, 3, 3), X["b"].double().abs(), 3, 1, None)
        # split-bf16 tap GEMM 1e-5; the CUDA-core kernel is exact fp32 arithmetic on x = hi + lo
        check_slices("%s %dx%dx%d (B(H+4) = %d)" % (symbol, B, H, W, B * (H + 4)), V["out"].reshape(B, H, W, 2), ref,
                     1e-5 if tc else 5e-6, scale=eta.abs() + mag.permute(0, 2, 3, 1))

    return Row(bufs, make, call, check)


row("conv_c2_bh_residual_15_rows", "mrb_conv_c2_bh_residual", attr=True)(
    lambda: _final_conv_row("mrb_conv_c2_bh_residual", 1, 11, BH_W))
row("tc2_final_conv_16_rows", "mrb_tc2_final_conv", attr=True)(lambda: _final_conv_row("mrb_tc2_final_conv", 1, 12, BH_W))
row("tc2_final_conv_17_rows", "mrb_tc2_final_conv")(lambda: _final_conv_row("mrb_tc2_final_conv", 1, 13, BH_W))
row("tc2_final_conv_26_rows", "mrb_tc2_final_conv")(lambda: _final_conv_row("mrb_tc2_final_conv", 2, 9, 30))


@row("g8_from_nhwc4", "mrb_g8_from_nhwc4")
def _g8_row(B=BH_B, H=BH_H, W=BH_W):
    n8, w8, lo, Q = _g8_layout(B, H, W)

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_g8_from_nhwc4(L.ptr(V["x"]), L.ptr(V["g8"]), B, H, W, st))

    def check(V, X):
        v = _g8_positions(V["g8"], lo, Q, B, H, W)
        assert torch.equal(v.view(torch.int16), _replicated(v, H, W).view(torch.int16)), "G8 border is not a replicate copy"
        x = _split(v, B, H, W, 4)[:, 2:H + 2, 2:W + 2]
        check_slices("g8_from_nhwc4 hi + lo", x, X["x"].double().reshape(B, H, W, 4), 1e-5)

    return Row({"x": Buf("in", B * H * W * 4), "g8": Buf("g8", n8, torch.bfloat16, written=w8)},
               lambda s: {"x": _rn(_gen(s), B * H * W * 4)}, call, check)


@row("tc2_conv5x5x4_w28", "mrb_tc2_conv5x5x4", attr=True)
def _conv5_row(B=BH_B, H=BH_H, W=BH_W):
    from oracle import nets as onets

    L, lib, _ = _lib()
    n8 = _g8_layout(B, H, W)[0]
    bufs = {"g8": Buf("in", n8, torch.bfloat16), "w": Buf("in", 64 * 4 * 25), "b": Buf("in", 64), "out": _bh_out(B, H, W)}

    def make(seed):
        g = _gen(seed)
        x4 = _rn(g, B * H * W * 4)
        g8 = torch.zeros(n8, dtype=torch.bfloat16, device="cuda")
        L.check(lib.mrb_g8_from_nhwc4(L.ptr(x4), L.ptr(g8), B, H, W, _lib()[2]))
        return {"g8": g8, "w": _rn(g, 64 * 4 * 25, scale=0.2), "b": _rn(g, 64), "_x4": x4}

    def call(V, st):
        L.check(lib.mrb_tc2_conv5x5x4(L.ptr(V["g8"]), L.ptr(V["w"]), L.ptr(V["b"]), L.ptr(V["out"]), B, H, W, 1, st))

    def check(V, X):
        ref = onets.conv_nonlinear(_nchw(X["_x4"].reshape(B, H, W, 4)), X["w"].double().reshape(64, 4, 5, 5),
                                   X["b"].double(), 5, 1, "relu")
        _check_bh("tc2_conv5x5x4 %dx%dx%d" % (B, H, W), V["out"], ref, B, H, W)

    return Row(bufs, make, call, check)


def _gru_weights(g):
    return _rn(g, 192 * 64, scale=0.1), _rn(g, 192 * 64, scale=0.1)


@row("tc2_pack_gru", "mrb_tc2_pack_gru")
def _pack_gru_row():
    from oracle import nets as onets

    L, lib, _ = _lib()
    B, H, W = BH_B, BH_H, BH_W
    bufs = {"wih": Buf("in", 192 * 64), "whh": Buf("in", 192 * 64), "dst": Buf("out", lib.mrb_tc2_gru_packed_bytes(), torch.uint8)}

    def make(seed):
        g = _gen(seed)
        wih, whh = _gru_weights(g)
        return {"wih": wih, "whh": whh, "_x": _rn(g, B, H, W, 64), "_h": _rn(g, B, H, W, 64)}

    def call(V, st):
        L.check(lib.mrb_tc2_pack_gru(L.ptr(V["wih"]), L.ptr(V["whh"]), L.ptr(V["dst"]), 64, 64, st))

    def check(V, X):
        # the packed image has no plain reference: the cell that consumes it is compared with fp64
        ob = torch.empty(_bh_numel(B, H, W), dtype=torch.bfloat16, device="cuda")
        xb, hb = _to_bh(X["_x"], B, H, W), _to_bh(X["_h"], B, H, W)
        L.check(lib.mrb_tc2_gru(L.ptr(xb), L.ptr(hb), L.ptr(V["dst"]), None, L.ptr(ob), B, H, W, _lib()[2]))
        ref = onets.conv_gru_cell(_nchw(X["_x"]), _nchw(X["_h"]), X["wih"].double().reshape(192, 64, 1, 1), None,
                                  X["whh"].double().reshape(192, 64, 1, 1), 1, 1)
        _check_bh("tc2_pack_gru -> tc2_gru", ob, ref, B, H, W)

    return Row(bufs, make, call, check)


def _cell_bh_row(symbol, B=BH_B, H=BH_H, W=BH_W):
    """ConvGRU / IndRNN on BH tensors: the border of x and h is never read for an interior result (NaN there in the
    poisoned runs); every position of the output is written, its border is not a replicate copy."""
    from oracle import nets as onets

    L, lib, _ = _lib()
    gru = symbol == "mrb_tc2_gru"
    nb = _bh_numel(B, H, W)
    border = _bh_border(B, H, W)
    bufs = {"x": Buf("in", nb, torch.bfloat16, unread=border), "h": Buf("in", nb, torch.bfloat16, unread=border),
            "wp": Buf("in", lib.mrb_tc2_gru_packed_bytes() // 4 if gru else lib.mrb_tc_packed_floats(0, 64, 64, 1)),
            "b": Buf("in", 192 if gru else 64), "out": _bh_out(B, H, W)}
    if not gru:
        bufs["hh"] = Buf("in", 64)

    def make(seed):
        g = _gen(seed)
        x, h = _rn(g, B, H, W, 64), _rn(g, B, H, W, 64)
        X = {"x": _to_bh(x, B, H, W), "h": _to_bh(h, B, H, W)}
        if gru:
            wih, whh = _gru_weights(g)
            pk = torch.empty(bufs["wp"].numel, device="cuda")
            L.check(lib.mrb_tc2_pack_gru(L.ptr(wih), L.ptr(whh), L.ptr(pk), 64, 64, _lib()[2]))
            X.update(wp=pk, b=_rn(g, 192, scale=0.1), _wih=wih, _whh=whh)
        else:
            wi = _rn(g, 64 * 64, scale=0.1)
            X.update(wp=_pack_conv(wi, 1), b=_rn(g, 64, scale=0.1), hh=_rn(g, 64, scale=0.5), _wi=wi)
        return X

    def call(V, st):
        if gru:
            L.check(lib.mrb_tc2_gru(L.ptr(V["x"]), L.ptr(V["h"]), L.ptr(V["wp"]), L.ptr(V["b"]), L.ptr(V["out"]), B, H, W, st))
        else:
            L.check(lib.mrb_tc2_indrnn(L.ptr(V["x"]), L.ptr(V["h"]), L.ptr(V["wp"]), L.ptr(V["b"]), L.ptr(V["hh"]),
                                       L.ptr(V["out"]), B, H, W, st))

    def check(V, X):
        x, h = (_interior_nchw(_split(X[k], B, H, W, 64), H, W) for k in ("x", "h"))
        if gru:
            ref = onets.conv_gru_cell(x, h, X["_wih"].double().reshape(192, 64, 1, 1), X["b"].double(),
                                      X["_whh"].double().reshape(192, 64, 1, 1), 1, 1)
        else:
            ref = onets.indrnn_cell(x, h, X["_wi"].double().reshape(64, 64, 1, 1), X["b"].double(),
                                    X["hh"].double().reshape(1, 64, 1, 1), 1, 1)
        _check_bh("%s %dx%dx%d" % (symbol, B, H, W), V["out"], ref, B, H, W)

    return Row(bufs, make, call, check)


row("tc2_gru_w28", "mrb_tc2_gru", attr=True)(lambda: _cell_bh_row("mrb_tc2_gru"))
row("tc2_indrnn_w28", "mrb_tc2_indrnn", attr=True)(lambda: _cell_bh_row("mrb_tc2_indrnn"))


# U-Net 3x3: H (W + 1) = 23 * 42 = 966 positions per image, not a multiple of 128; strided input and concat output
UC_N, UC_CIN, UC_COUT, UC_H, UC_W = 2, 20, 24, 23, 41


def _uconv_pack(w):
    L, lib, st = _lib()
    pk = torch.empty(lib.mrb_tc2_unet_packed_bytes(UC_CIN, UC_COUT), dtype=torch.uint8, device="cuda")
    L.check(lib.mrb_tc2_unet_pack(L.ptr(w), L.ptr(pk), UC_CIN, UC_COUT, st))
    return pk


def _uconv_ref(x, w):
    N, Cin, Cout, H, W = UC_N, UC_CIN, UC_COUT, UC_H, UC_W
    xbs = Cin * H * W + 4
    return F.conv2d(x.reshape(N, xbs)[:, :Cin * H * W].reshape(N, Cin, H, W).double(), w.double().reshape(Cout, Cin, 3, 3),
                    padding=1)


def _uconv_x(g):
    return _rn(g, UC_N * (UC_CIN * UC_H * UC_W + 4))


def _uconv_w(g):
    return _rn(g, UC_COUT * UC_CIN * 9, scale=(9 * UC_CIN) ** -0.5)


@row("tc2_unet_pack", "mrb_tc2_unet_pack")
def _uconv_pack_row():
    L, lib, _ = _lib()
    N, Cin, Cout, H, W = UC_N, UC_CIN, UC_COUT, UC_H, UC_W
    HW = H * W
    bufs = {"w": Buf("in", Cout * Cin * 9), "dst": Buf("out", lib.mrb_tc2_unet_packed_bytes(Cin, Cout), torch.uint8)}

    def make(seed):
        g = _gen(seed)
        return {"w": _uconv_w(g), "_x": _uconv_x(g)}

    def call(V, st):
        L.check(lib.mrb_tc2_unet_pack(L.ptr(V["w"]), L.ptr(V["dst"]), Cin, Cout, st))

    def check(V, X):
        out = torch.empty((N, Cout, H, W), device="cuda")
        L.check(lib.mrb_tc2_unet_conv3x3(L.ptr(X["_x"]), Cin * HW + 4, L.ptr(V["dst"]), L.ptr(out), Cout * HW, N, Cin, Cout,
                                         H, W, _lib()[2]))
        check_slices("tc2_unet_pack -> uconv3", out, _uconv_ref(X["_x"], X["w"]), 2e-6)

    return Row(bufs, make, call, check)


@row("tc2_unet_conv3x3_concat", "mrb_tc2_unet_conv3x3", attr=True)
def _uconv_row():
    L, lib, _ = _lib()
    N, Cin, Cout, H, W = UC_N, UC_CIN, UC_COUT, UC_H, UC_W
    HW = H * W
    xbs, obs = Cin * HW + 4, (Cout + 8) * HW
    bufs = {"x": Buf("in", N * xbs), "wp": Buf("in", lib.mrb_tc2_unet_packed_bytes(Cin, Cout), torch.uint8),
            "out": Buf("out", N * obs, written=_batch_rows(N, obs, Cout * HW))}

    def make(seed):
        g = _gen(seed)
        w = _uconv_w(g)
        return {"x": _uconv_x(g), "wp": _uconv_pack(w), "_w": w}

    def call(V, st):
        L.check(lib.mrb_tc2_unet_conv3x3(L.ptr(V["x"]), xbs, L.ptr(V["wp"]), L.ptr(V["out"]), obs, N, Cin, Cout, H, W, st))

    def check(V, X):
        check_slices("uconv3 concat 23x41", V["out"].reshape(N, obs)[:, :Cout * HW].reshape(N, Cout, H, W),
                     _uconv_ref(X["x"], X["_w"]), 2e-6)

    return Row(bufs, make, call, check)


# ---------------------------------------------------------------------------------------------- metrics, qMRI
@row("abs_max_normalize", "mrb_abs_max_normalize")
def _absmax_row():
    L, lib, _ = _lib()
    n = 2 * 19 * 23
    bufs = {"x": Buf("in", 2 * n), "out": Buf("out", n), "ws": Buf("ws", lib.mrb_metrics_workspace_bytes(1) // 8,
                                                                    torch.float64)}

    def call(V, st):
        L.check(lib.mrb_abs_max_normalize(L.ptr(V["x"]), n, 1, L.ptr(V["out"]), L.ptr(V["ws"]), st))

    def check(V, X):
        mag = torch.view_as_complex(X["x"].double().reshape(n, 2)).abs()
        check_slices("abs_max_normalize", V["out"][None], (mag / mag.max())[None], 2e-6)

    return Row(bufs, lambda s: {"x": _rn(_gen(s), 2 * n)}, call, check)


def _metrics_row(B, H, W, mode, maxval):
    """res = mse, nmse, psnr, ssim, data range (mode 0: max(gt), 1: max(pred) - min(pred), 2: maxval; + 4: no SSIM).
    metric_sums_kernel and ssim_sum_kernel add their fp64 block partials with atomicAdd, so across runs res agrees to
    rounding (1e-10 relative), not bit for bit."""
    from oracle import metrics as om

    L, lib, _ = _lib()
    n = B * H * W
    ssim = not mode & 4
    bufs = {"gt": Buf("in", n), "pred": Buf("in", n), "res": Buf("out", 5, torch.float64, finite=ssim, rtol=1e-10),
            "ws": Buf("ws", lib.mrb_metrics_workspace_bytes(B) // 8, torch.float64)}

    def make(seed):
        g = _gen(seed)
        gt = torch.rand(n, device="cuda", generator=g)
        return {"gt": gt, "pred": gt + 0.05 * _rn(g, n)}

    def call(V, st):
        L.check(lib.mrb_recon_metrics(L.ptr(V["gt"]), L.ptr(V["pred"]), B, H, W, mode, maxval, L.ptr(V["res"]),
                                      L.ptr(V["ws"]), st))

    def check(V, X):
        a, b = (X[k].reshape(B, H, W).double().cpu().numpy() for k in ("gt", "pred"))
        R = {0: float(np.max(a)), 1: float(X["pred"].max() - X["pred"].min()), 2: maxval}[mode & 3]
        v = V["res"].cpu().tolist()
        ref = [om.mse(a, b), om.nmse(a, b), om.psnr(a, b, R), om.ssim(a, b, R) if ssim else float("nan"), R]
        print("[abi contract] metrics %dx%dx%d mode %d: CUDA %s | fp64 %s" % (B, H, W, mode, v, ref))
        assert abs(v[0] - ref[0]) <= 2e-6 * ref[0] and abs(v[1] - ref[1]) <= 2e-6 * ref[1], (v, ref)
        assert abs(v[2] - ref[2]) <= 1e-5 and v[4] == R, (v, ref)
        assert abs(v[3] - ref[3]) <= 1e-7 if ssim else np.isnan(v[3]), (v, ref)

    return Row(bufs, make, call, check)


row("recon_metrics_7x7", "mrb_recon_metrics")(lambda: _metrics_row(1, 7, 7, 0, 0.0))
row("recon_metrics_3x33x45_maxval", "mrb_recon_metrics")(lambda: _metrics_row(3, 33, 45, 2, 1.25))
row("recon_metrics_no_ssim", "mrb_recon_metrics")(lambda: _metrics_row(2, 5, 6, 1 + 4, 0.0))


QM_B, QM_E, QM_C, QM_H, QM_W = 2, 4, 3, 17, 13
QM_TES = [3.0, 11.5, 20.0, 28.5]


@row("megre_signal", "mrb_megre_signal")
def _megre_signal_row():
    from oracle import qnets as oq

    L, lib, _ = _lib()
    B, E, HW = QM_B, QM_E, QM_H * QM_W
    gamma = (ctypes.c_float * 4)(1.5, 0.75, 1.25, 0.5)
    tes = (ctypes.c_double * E)(*QM_TES)
    bufs = {k: Buf("in", B * HW) for k in ("r2", "s0", "b0", "ph")}
    bufs["out"] = Buf("out", B * E * HW * 2)

    def make(seed):
        g = _gen(seed)
        return {"r2": torch.rand(B * HW, device="cuda", generator=g) * 90 + 5, "s0": _rn(g, B * HW),
                "b0": _rn(g, B * HW, scale=40.0), "ph": _rn(g, B * HW)}

    def call(V, st):
        L.check(lib.mrb_megre_signal(L.ptr(V["r2"]), L.ptr(V["s0"]), L.ptr(V["b0"]), L.ptr(V["ph"]), gamma, tes, E, 1e-3, B,
                                     HW, 0, L.ptr(V["out"]), st))

    def check(V, X):
        maps = [X[k].double().reshape(B, 1, HW) * gamma[i] for i, k in enumerate(("r2", "s0", "b0", "ph"))]
        ref = oq.megre_signal(*maps, QM_TES, 1e-3).reshape(B, E, HW, 2)
        check_slices("megre_signal", V["out"].reshape(B, E, HW, 2), ref, 5e-6)

    return Row(bufs, make, call, check)


@row("megre_grad_4_of_8_channels", "mrb_megre_grad")
def _megre_grad_row():
    """d = the DC gradient of the echo-folded MEGRE signal (as qrim._qmri_gradient builds it); out [B, 8, HW] of which the
    call writes channels 0..3."""
    from mridc_b200 import _ops
    from oracle import qnets as oq
    from oracle.make_golden import qmri_inputs

    L, lib, _ = _lib()
    B, E, C, H, W = QM_B, QM_E, QM_C, QM_H, QM_W
    HW = H * W
    tes = (ctypes.c_double * E)(*QM_TES)
    written = torch.zeros((B, 8, HW), dtype=torch.bool)
    written[:, :4] = True
    bufs = {"d": Buf("in", B * E * 4 * HW), **{k: Buf("in", B * HW) for k in ("r2", "s0", "b0", "ph")},
            "out": Buf("out", B * 8 * HW, written=written)}

    def make(seed):
        r2, s0, b0, ph, tes_l, y, S, m = qmri_inputs(B, E, C, H, W, 55 + seed, "2db")
        maps = [t.cuda().reshape(B, HW).contiguous() for t in (r2, s0, b0, ph)]
        eta = torch.empty((B, E, HW, 2), device="cuda")
        L.check(lib.mrb_megre_signal(*(L.ptr(t) for t in maps), None, tes, E, 1e-3, B, HW, 0, L.ptr(eta), _lib()[2]))
        Se = S.cuda()[:, None].expand(B, E, C, H, W, 2).reshape(B * E, C, H, W, 2)
        me = m.cuda()[:, None].expand(B, E, 1, H, W, 1).reshape(B * E, 1, H, W, 1)
        d = _ops.dc_rim_grad(eta.reshape(B * E, H, W, 2), y.cuda().reshape(B * E, C, H, W, 2), Se, me, 1.0, False,
                             "backward")
        X = dict(zip(("r2", "s0", "b0", "ph"), maps))
        X.update(d=d, _in=(r2, s0, b0, ph, y, S, m))
        return X

    def call(V, st):
        L.check(lib.mrb_megre_grad(L.ptr(V["d"]), L.ptr(V["r2"]), L.ptr(V["s0"]), L.ptr(V["b0"]), L.ptr(V["ph"]), None, tes,
                                   E, 1e-3, B, HW, 100.0, 1, L.ptr(V["out"]), 8, st))

    def check(V, X):
        r2, s0, b0, ph, y, S, m = X["_in"]
        ref = torch.stack([oq.analytical_log_likelihood_gradient(r2[b].double(), s0[b].double(), b0[b].double(),
                                                                 ph[b].double(), QM_TES, S[b].double(), y[b].double(), m[b],
                                                                 False, "backward", [-2, -1], 2) / 100 for b in range(B)])
        check_slices("megre_grad", V["out"].reshape(B, 8, H, W)[:, :4].cpu(), ref, 5e-6)

    return Row(bufs, make, call, check)


@row("qrim_eta_update_channels_4_to_7", "mrb_qrim_eta_update")
def _eta_update_row():
    B, HW = 2, 17 * 13
    written = torch.zeros((B, 8, HW), dtype=torch.bool)
    written[:, 4:] = True
    bufs = {"eta": Buf("inout", B * 8 * HW, written=written), "delta": Buf("in", B * 4 * HW), "out": Buf("out", B * 4 * HW)}

    def make(seed):
        g = _gen(seed)
        return {"eta": _rn(g, B * 8 * HW), "delta": _rn(g, B * 4 * HW)}

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_qrim_eta_update(L.ptr(V["eta"]), 8, 4, L.ptr(V["delta"]), L.ptr(V["out"]), B, HW, st))

    def check(V, X):
        upd = X["eta"].reshape(B, 8, HW)[:, 4:] + X["delta"].reshape(B, 4, HW)
        upd[:, 0] = upd[:, 0].clamp_min(0)
        assert torch.equal(V["eta"].reshape(B, 8, HW)[:, 4:], upd) and torch.equal(V["out"].reshape(B, 4, HW), upd)

    return Row(bufs, make, call, check)


@row("scale_batch_abs", "mrb_scale_batch")
def _scale_row():
    B, per = 3, 4 * 5 * 6
    scales = (ctypes.c_float * B)(2.0, 3.0, 0.625)

    def call(V, st):
        L, lib, _ = _lib()
        L.check(lib.mrb_scale_batch(L.ptr(V["x"]), L.ptr(V["out"]), B, per, scales, 1, st))

    def check(V, X):
        s = torch.tensor(list(scales), device="cuda")[:, None]
        assert torch.equal(V["out"].reshape(B, per), X["x"].reshape(B, per).abs() * s)

    return Row({"x": Buf("in", B * per), "out": Buf("out", B * per)}, lambda s: {"x": _rn(_gen(s), B * per)}, call, check)


# ---------------------------------------------------------------------------------------------- CPU: inventory and self-tests
def test_every_launching_entry_point_has_a_contract_row():
    """Every symbol of _lib.SIGNATURES has a contract row or is listed in NON_LAUNCHING with its reason."""
    from mridc_b200 import _lib as L

    rows = {s for syms, _ in ROWS.values() for s in syms}
    assert all(NON_LAUNCHING.values()), "every exclusion needs a reason"
    assert not rows & set(NON_LAUNCHING), sorted(rows & set(NON_LAUNCHING))
    missing = sorted(set(L.SIGNATURES) - rows - set(NON_LAUNCHING))
    assert not missing, "entry points without a row in tests/test_gpu_abi_contract.py: %s" % missing
    stale = sorted((rows | set(NON_LAUNCHING)) - set(L.SIGNATURES))
    assert not stale, "rows or exclusions name symbols _lib.SIGNATURES does not have: %s" % stale
    print("[abi contract] %d launching entry points, %d rows, %d excluded" % (len(rows), len(ROWS), len(NON_LAUNCHING)))


def _fake_row(kernel):
    """A CPU "kernel" on 64 fp32 values: out = 2 x, with an 8-value workspace."""
    bufs = {"x": Buf("in", 64), "out": Buf("out", 64), "ws": Buf("ws", 8)}

    def make(seed):
        return {"x": torch.randn(64, generator=torch.Generator().manual_seed(seed))}

    def check(V, X):
        assert torch.equal(V["out"], 2 * X["x"])

    return Row(bufs, make, lambda V, st: kernel(V), check)


def _past(t, offset, n=1):
    """n elements of t's storage starting `offset` elements from t's first element (may lie outside t)."""
    return torch.as_strided(t, (n,), (1,), t.storage_offset() + offset)


def test_harness_passes_a_correct_kernel():
    run_contract(_fake_row(lambda V: V["out"].copy_(2 * V["x"])), "cpu", graph=False)


def test_harness_catches_a_write_past_the_end():
    def k(V):
        V["out"].copy_(2 * V["x"])
        _past(V["out"], 64).fill_(1.0)

    with pytest.raises(AssertionError, match=r"out buffer 'out' modified at byte offset 256, in the guard after the buffer"):
        run_contract(_fake_row(k), "cpu", graph=False)


def test_harness_catches_an_unwritten_element():
    def k(V):
        V["out"][:17] = 2 * V["x"][:17]
        V["out"][18:] = 2 * V["x"][18:]

    with pytest.raises(AssertionError, match=r"buffer 'out': byte offset 68 \(element 17\) not written"):
        run_contract(_fake_row(k), "cpu", graph=False)


def test_harness_catches_a_read_of_the_workspace():
    def k(V):
        V["out"].copy_(2 * V["x"] + V["ws"][3])

    with pytest.raises(AssertionError, match=r"poisoned eager set A: out buffer 'out' differs from the reference run at "
                                             r"byte offset 0 \(element 0; 64 elements\)"):
        run_contract(_fake_row(k), "cpu", graph=False)


def test_harness_catches_a_read_before_the_input():
    def k(V):
        V["out"].copy_(2 * V["x"])
        V["out"][5] = 2 * _past(V["x"], -1)[0]

    with pytest.raises(AssertionError, match=r"buffer 'out': non-finite value at byte offset 20 \(element 5"):
        run_contract(_fake_row(k), "cpu", graph=False)


def test_harness_tolerance_still_catches_a_workspace_read():
    """A buffer compared to a relative tolerance (atomic reductions) still fails when the result depends on the workspace."""
    r = _fake_row(lambda V: V["out"].copy_(2 * V["x"] + V["ws"][3]))
    r.bufs["out"].rtol = 1e-10
    with pytest.raises(AssertionError, match=r"poisoned eager set A: out buffer 'out' differs"):
        run_contract(r, "cpu", graph=False)


def test_harness_catches_a_write_into_an_input():
    def k(V):
        V["out"].copy_(2 * V["x"])
        V["x"][9] = 0.0

    with pytest.raises(AssertionError, match=r"in buffer 'x' modified at byte offset 36, inside the buffer"):
        run_contract(_fake_row(k), "cpu", graph=False)


# ---------------------------------------------------------------------------------------------- GPU rows
@pytest.fixture(autouse=True)
def _release_gpu_memory():
    yield
    gc.collect()
    if torch.cuda.is_available() and torch.cuda.is_initialized():
        torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ROWS))
def test_contract(name):
    run_contract(ROWS[name][1]())


@pytest.mark.gpu
def test_entry_points_on_a_second_device():
    """The entry points that raise a kernel's dynamic shared-memory limit, first on cuda:0, then on cuda:1 in the same
    process: the same bits on both devices (the limit is an attribute of the device's context)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    assert len(ATTR_ROWS) == 8, ATTR_ROWS
    res = {}
    for d in (0, 1):
        with torch.cuda.device(d):
            for name in ATTR_ROWS:
                r = ROWS[name][1]()
                res[name, d] = {k: v.cpu() for k, v in outputs(eager(r, r.make(1), "cuda:%d" % d,
                                                                     tag="%s on cuda:%d" % (name, d))).items()}
    for name in ATTR_ROWS:
        for k in res[name, 0]:
            assert torch.equal(res[name, 0][k], res[name, 1][k]), "%s: %r differs between cuda:0 and cuda:1" % (name, k)
