"""Every compiled kernel instantiation reached from its inputs, proved launched with the profiler, and checked against fp64.

Each entry point of libmridc_b200.so picks its kernel from the input: the length and the axis of a transform, the coil
count, the mask (1-D or 2-D), the image width, the output channel count, the presence of a bias, a plane size.  A test
that only checks the result cannot tell which of those kernels produced it, so a variant can be compiled, reachable and
never run.  Every row here has four parts:

  inputs     chosen so that the dispatch takes one branch, with no environment switch set;
  kernels    the demangled instantiations the call must launch (and, where a branch replaces another, the ones it must
             not launch), recorded with torch.profiler (CUPTI) around the call;
  reference  the same operation in plain torch on CUDA float64 tensors (the oracle package or torch.fft / F.conv2d / ...);
             float64 never takes a TF32 path, so no global torch flag is touched;
  tolerance  the existing per-slice contract of test_gpu_bench_shapes.py: 2e-6 for fp32 operators, 1e-5 for split-bf16
             tensor-core operators, 2e-6 for uconv3, 3e-5 per RIM block, 1e-4 per model; exact operations are bit-exact.

EXPECTED below is the union the CPU inventory test compares with the instantiations listed in the built library: a new
kernel or template instantiation without a row fails the CPU suite.  Each GPU row asserts only its own entry, so ``-k``
selects rows freely.
"""
import gc
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_bench_shapes import check_slices

# When set (tools/kernel_coverage.py installs a set here), launched() adds every kernel it records: torch.profiler
# sessions do not nest, so the rows of this file report their kernels themselves.
KERNEL_SINK = None


def _k(*names):
    return frozenset(names)


R320, TC2 = "mrb::r320::", "mrb::tc2::"
CONV_KD = [(5, 1), (3, 2), (3, 1), (1, 1), (7, 1)]  # (k, dil); k = 7 takes the runtime-k instantiation <TN, 0, 0>
CONV_COUT = [8, 16, 32, 64]                           # TN = 1, 2, 4, 8


def _conv_name(cout, k, dil):
    tn = 8 if cout > 32 else 4 if cout > 16 else 2 if cout > 8 else 1
    kk, dd = (k, dil) if (k, dil) in ((5, 1), (3, 2), (3, 1)) else (1, 1) if k == 1 else (0, 0)
    return "mrb::conv2d_kernel<%d, %d, %d>" % (tn, kk, dd)


ROW_DC = {(m, keep): "mrb::row_dc_kernel<%d, %s>" % (m, "true" if keep else "false") for m in (1, 2) for keep in (0, 1)}
THREE_PASS = _k("void mrb::expand_rowfft_kernel<true>", "mrb::col_dc_kernel", "mrb::rowifft_reduce_kernel<1, true>",
                "mrb::rowifft_reduce_kernel<2, true>")
FFT_GENERIC = _k("mrb::fft1d_rows_kernel<false>", "mrb::fft1d_rows_kernel<true>", "mrb::fft1d_cols_kernel<false>",
                 "mrb::fft1d_cols_kernel<true>")

# row -> (kernels it must launch, kernels it must not launch); names without "void " and without the argument list
EXPECTED = {
    "fft320": (_k(*("%sfft320_kernel<%s, %s>" % (R320, a, b) for a in ("false", "true") for b in ("false", "true"))), _k()),
    "fft640_cols": (_k(R320 + "fft640_cols_kernel<false>", R320 + "fft640_cols_kernel<true>"), _k()),
    "fft640_rows": (_k("mrb::fft1d_rows_kernel<false>", "mrb::fft1d_rows_kernel<true>"), _k()),
    "fft_other_rotations": (FFT_GENERIC, _k(*("%sfft320_kernel<%s, %s>" % (R320, a, b) for a in ("false", "true")
                                               for b in ("false", "true")), R320 + "fft640_cols_kernel<false>",
                                             R320 + "fft640_cols_kernel<true>")),
    "fft_long": (FFT_GENERIC, _k()),
    "fft2_primes": (FFT_GENERIC, _k()),
    "roll": (_k("mrb::roll_kernel<unsigned char>", "mrb::roll_kernel<unsigned short>", "mrb::roll_kernel<unsigned int>",
                "mrb::roll_kernel<unsigned long>", "mrb::roll_kernel<uint4>"), _k()),
    "row_dc_keep": (_k(ROW_DC[1, 1], ROW_DC[2, 1], "mrb::compact_hybrid_kernel"), _k(ROW_DC[1, 0], ROW_DC[2, 0])),
    "row_dc_nokeep": (_k(ROW_DC[1, 0], ROW_DC[2, 0], "mrb::compact_hybrid_kernel"), _k(ROW_DC[1, 1], ROW_DC[2, 1])),
    "dc_wide": (_k(ROW_DC[1, 0], ROW_DC[2, 0], "mrb::compact_hybrid_kernel") | THREE_PASS, _k(ROW_DC[1, 1], ROW_DC[2, 1])),
    "dc_c20_320_1d": (_k(ROW_DC[1, 1], ROW_DC[2, 1]), _k(*("%srow_dc320_kernel<%d>" % (R320, i) for i in (1, 2, 3)))),
    "dc_c20_320_2d": (THREE_PASS, _k(R320 + "expand_row320_kernel", R320 + "col_dc320_kernel",
                                     R320 + "reduce_row320_kernel<1>", R320 + "reduce_row320_kernel<2>")),
    "dc_2d_640": (THREE_PASS, _k(R320 + "col_dc320_kernel")),
    "dc_full_columns": (_k("mrb::compact_hybrid_kernel", ROW_DC[1, 1]), _k()),
    "sens_c20": (_k("mrb::rowifft_reduce_kernel<0, false>", "void mrb::expand_rowfft_kernel<false>",
                    "mrb::col_softdc_kernel", R320 + "fft320_kernel<true, true>", R320 + "fft640_cols_kernel<true>"),
                 _k(R320 + "reduce_row320_kernel<0>", R320 + "expand_row320_kernel", R320 + "col_softdc320_kernel",
                    R320 + "col_softdc640_kernel")),
    "sens_row320_other_h": (_k(R320 + "expand_row320_kernel", "mrb::col_softdc_kernel", R320 + "reduce_row320_kernel<0>"),
                            _k("void mrb::expand_rowfft_kernel<false>")),
    "dc320": (_k(*("%srow_dc320_kernel<%d>" % (R320, i) for i in (1, 2, 3)), R320 + "expand_row320_kernel",
                 R320 + "col_dc320_kernel", R320 + "reduce_row320_kernel<1>", R320 + "reduce_row320_kernel<2>",
                 TC2 + "g8_from_nhwc4_kernel"), _k()),
    "sens320": (_k(R320 + "reduce_row320_kernel<0>", R320 + "expand_row320_kernel", R320 + "col_softdc320_kernel",
                   R320 + "col_softdc640_kernel"), _k("mrb::col_softdc_kernel")),
    "conv2d": (_k(*(_conv_name(co, k, d) for co in CONV_COUT for k, d in CONV_KD)), _k()),
    "final_conv_cuda_core": (_k("mrb::conv_c2_k3_kernel<4, 16>", TC2 + "bh_fix_border_kernel"), _k(TC2 + "fin2_kernel")),
    "final_conv_tc": (_k(TC2 + "fin2_kernel"), _k("mrb::conv_c2_k3_kernel<4, 16>")),
    "tc_conv_bh": (_k("mrb::tc::tc_kernel", "mrb::tc::pack_weights_kernel", TC2 + "bh_from_nhwc_kernel",
                      TC2 + "bh_to_nhwc_kernel"), _k()),
    "tc2_ops": (_k(TC2 + "gru2_kernel", TC2 + "ind2_kernel", TC2 + "conv5g_kernel", TC2 + "fin2_kernel",
                   TC2 + "bh_fix_border_kernel", TC2 + "g8_from_nhwc4_kernel"), _k()),
    **{"uconv3_%d" % i: (_k(TC2 + "uconv3_kernel<%d>" % i, TC2 + "uconv3_pack_kernel"),
                         _k(*(TC2 + "uconv3_kernel<%d>" % j for j in (1, 2, 4) if j != i))) for i in (1, 2, 4)},
    "rim_block_k5_nobias": (_k("mrb::tc::tc_kernel", TC2 + "conv5g_kernel", TC2 + "gru2_kernel"), _k()),
    "cirim_c20": (_k(TC2 + "g8_from_nhwc4_kernel", ROW_DC[2, 1], "mrb::tc::tc_kernel"),
                  _k(R320 + "row_dc320_kernel<3>")),
    "rim_block_w27": (_k(_conv_name(64, 5, 1), "mrb::gru_cell_1x1_kernel"), _k("mrb::tc::tc_kernel")),
    "rim_cells_fp32": (_k("mrb::gru_cell_1x1_kernel", "mrb::gru_gates_kernel", "mrb::mgu_gates_kernel"), _k()),
    "instnorm_cluster": (_k("mrb::instnorm_cluster_kernel"), _k("mrb::plane_stats_kernel")),
    "instnorm_two_pass": (_k("mrb::plane_stats_kernel", "mrb::instnorm_apply_kernel"), _k("mrb::instnorm_cluster_kernel")),
    "unet_final_conv1x1": (_k("mrb::conv1x1_kernel"), _k(_conv_name(2, 1, 1))),
    "unet_final_conv2d": (_k(_conv_name(2, 1, 1)), _k("mrb::conv1x1_kernel")),
    "unet_small_ops": (_k("mrb::conv1x1_kernel", "mrb::avgpool2_kernel", "mrb::conv_transpose2x2_kernel",
                          "mrb::pad2d_kernel"), _k()),
    "normunet_1": (_k("mrb::normunet_stats_kernel", "mrb::normunet_finalize_kernel", "mrb::normunet_in_kernel",
                      "mrb::normunet_out_kernel"), _k()),
    "normunet_0": (_k("mrb::normunet_in_kernel", "mrb::normunet_out_kernel"),
                   _k("mrb::normunet_stats_kernel", "mrb::normunet_finalize_kernel")),
    "complex_ops": (_k("mrb::complex_mul_kernel", "mrb::complex_conj_kernel", "mrb::complex_abs_kernel",
                       "mrb::coil_reduce_kernel<0>", "mrb::coil_reduce_kernel<1>", "mrb::coil_reduce_kernel<2>",
                       "mrb::divide_rss_kernel"), _k()),
    "metrics": (_k("mrb::abs_max_kernel", "mrb::abs_normalize_kernel", "mrb::metric_sums_kernel",
                   "mrb::metrics_finish_kernel", "mrb::ssim_sum_kernel", "mrb::ssim_finish_kernel"), _k()),
    "qmri": (_k("mrb::megre_signal_kernel", "mrb::megre_grad_kernel", "mrb::qrim_eta_update_kernel",
                "mrb::scale_batch_kernel"), _k()),
}
# instantiations no row launches, with the reason (none today)
EXCLUDED = {}


# ---------------------------------------------------------------------------------------------- helpers
def kernel_name(name):
    """Demangled kernel name without "void " and without the argument list: "mrb::conv2d_kernel<8, 5, 1>"."""
    if name.startswith("void "):
        name = name[5:]
    depth = 0
    for i, ch in enumerate(name):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            return name[:i]
    return name


def launched(fn):
    """-> (fn(), set of the library's kernel names launched while it ran), recorded with torch.profiler (CUPTI)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {kernel_name(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    ours = {n for n in names if n.startswith("mrb::")}
    assert ours, "the profiler recorded no kernel of the library around a call that launches (recorded: %s)" % sorted(names)
    if KERNEL_SINK is not None:
        KERNEL_SINK.update(ours)
    return out, ours


class Path:
    """Collects the kernels a row's calls launched and checks them against EXPECTED[row] at the end."""

    def __init__(self, row):
        self.row, self.seen = row, set()

    def __call__(self, fn):
        out, names = launched(fn)
        self.seen |= names
        return out

    def check(self):
        want, forbid = EXPECTED[self.row]
        # names written with a "void " prefix in the table (template functions whose demangled name keeps it) compare bare
        want = {kernel_name(n) for n in want}
        forbid = {kernel_name(n) for n in forbid}
        print("[kernel paths] %-22s launched: %s" % (self.row, ", ".join(sorted(self.seen))))
        missing, wrong = sorted(want - self.seen), sorted(forbid & self.seen)
        assert not missing, "%s: expected kernels not launched: %s" % (self.row, missing)
        assert not wrong, "%s: kernels of another branch launched: %s" % (self.row, wrong)


@pytest.fixture(autouse=True)
def _release_gpu_memory():
    """The B200 machines are shared: hand the cached blocks of each test back to the driver."""
    yield
    gc.collect()
    if torch.cuda.is_available() and torch.cuda.is_initialized():
        torch.cuda.empty_cache()


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _lib():
    from mridc_b200 import _lib

    return _lib, _lib.load(), _lib.stream_ptr()


# ---------------------------------------------------------------------------------------------- inventory (CPU)
def library_instantiations(path=None):
    """Every kernel instantiation in the built library: the .text.<mangled> sections of `cuobjdump -elf`, demangled with
    GNU c++filt (the format the profiler reports)."""
    from mridc_b200 import _lib

    path = path or _lib.LIB_PATH
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    cxxfilt = shutil.which("c++filt")
    assert os.path.exists(path), "build the library first (python -m mridc_b200.build)"
    assert os.path.exists(cuobjdump) and cxxfilt, "the inventory needs cuobjdump (CUDA toolkit) and GNU c++filt (binutils)"
    elf = subprocess.run([cuobjdump, "-elf", path], check=True, capture_output=True, text=True).stdout
    mangled = sorted(set(re.findall(r"\.text\.([A-Za-z0-9_$]+)", elf)))
    assert mangled, "no kernel sections found in %s" % path
    out = subprocess.run([cxxfilt], input="\n".join(mangled), check=True, capture_output=True, text=True).stdout
    return sorted({kernel_name(line.strip()) for line in out.splitlines() if line.strip()})


def test_every_kernel_instantiation_has_a_row():
    """The built library's instantiations == the union of the rows' expected kernels + EXCLUDED (each with a reason)."""
    inv = set(library_instantiations())
    rows = set()
    for want, forbid in EXPECTED.values():
        rows |= {kernel_name(n) for n in want}
        assert {kernel_name(n) for n in forbid} <= inv, "a row forbids a kernel the library does not have: %s" % (
            sorted({kernel_name(n) for n in forbid} - inv))
    assert all(EXCLUDED.values()), "every exclusion needs a reason"
    print("[kernel paths] %d instantiations in the library, %d reached by rows, %d excluded" % (
        len(inv), len(rows & inv), len(EXCLUDED)))
    untested = sorted(inv - rows - set(EXCLUDED))
    assert not untested, "kernel instantiations without a row in tests/test_gpu_kernel_paths.py: %s" % untested
    stale = sorted((rows | set(EXCLUDED)) - inv)
    assert not stale, "rows name kernels the library does not contain: %s" % stale


def test_kernel_name_normalisation():
    assert kernel_name("void mrb::conv2d_kernel<8, 5, 1>(mrb::ConvParams)") == "mrb::conv2d_kernel<8, 5, 1>"
    assert kernel_name("mrb::tc::tc_kernel(CUtensorMap_st, mrb::tc::Params)") == "mrb::tc::tc_kernel"
    assert kernel_name("void mrb::roll_kernel<unsigned long>(unsigned long const*, unsigned long*)") == \
        "mrb::roll_kernel<unsigned long>"


# ---------------------------------------------------------------------------------------------- self-tests
def test_tolerance_check_fails_a_perturbed_output():
    """A copy of an fp64 reference with one 64-value run of one slice off by 1e-4 relative fails the 2e-6 operator check."""
    g = torch.Generator().manual_seed(1)
    ref = torch.randn(4, 2, 64, 64, generator=g, dtype=torch.float64)
    out = ref.clone()
    out[3].view(-1)[100:164] *= 1 + 1e-4
    check_slices("self-test: exact copy", ref.clone(), ref, 2e-6)
    with pytest.raises(AssertionError, match=r"\[\(3, "):
        check_slices("self-test: perturbed slice 3", out, ref, 2e-6)


@pytest.mark.gpu
def test_path_check_fails_when_a_switch_moves_the_call(monkeypatch):
    """With MRIDC_B200_DC_STOCKHAM=1 the sens operators at W = 320 leave the 320-point kernels: every result still matches
    fp64, and the path assertion of the row fails naming the missing kernels."""
    monkeypatch.setenv("MRIDC_B200_DC_STOCKHAM", "1")
    with pytest.raises(AssertionError, match=r"sens320: expected kernels not launched: .*reduce_row320_kernel<0>"):
        _sens320_rows()


# ---------------------------------------------------------------------------------------------- FFT (fft.cu)
def _fft_ref(x, inverse, in_rot, out_rot, scale):
    """x: complex128 [outer, n, inner]; the semantics of mrb_fft1d_c2c (input index j read from (j + in_rot) % n, output
    index k written to (k + out_rot) % n, unnormalised transforms times scale)."""
    n = x.shape[1]
    xr = torch.roll(x, -in_rot, 1)
    X = torch.fft.ifft(xr, dim=1) * n if inverse else torch.fft.fft(xr, dim=1)
    return torch.roll(X, out_rot, 1) * scale


def _fft1d(path, x, inverse, in_rot, out_rot, scale=1.0):
    """x: complex64 [outer, n, inner] -> mrb_fft1d_c2c into a new tensor."""
    L, lib, st = _lib()
    outer, n, inner = x.shape
    out = torch.empty_like(x)
    path(lambda: L.check(lib.mrb_fft1d_c2c(L.ptr(x), L.ptr(out), outer, n, inner, int(inverse), in_rot, out_rot, scale, st)))
    return out


def _fft_case(path, tag, outer, n, inner, seed, cases, tol=2e-6):
    x = torch.randn((outer, n, inner), dtype=torch.complex64, device="cuda", generator=_gen(seed))
    errs = []
    for inverse, in_rot, out_rot, scale in cases:
        out = _fft1d(path, x, inverse, in_rot, out_rot, scale)
        ref = _fft_ref(x.to(torch.complex128), inverse, in_rot, out_rot, scale)
        errs.append(check_slices("%s n=%d [%d,%d,%d] inv=%d rot=(%d,%d)" % (tag, n, outer, n, inner, inverse, in_rot, out_rot),
                                 out, ref, tol).max().item())
    return max(errs)


@pytest.mark.gpu
def test_fft320_variants():
    """The register-resident 320-point transform, forward / inverse, along the contiguous axis (ROWS) and a strided one
    (COLS), centred and not (its rotations become sign flips)."""
    p = Path("fft320")
    for outer, inner in ((37, 1), (3, 45)):
        _fft_case(p, "fft320", outer, 320, inner, 1, [(0, 0, 0, 1.0), (1, 160, 160, 1 / 320), (0, 160, 0, 0.5),
                                                      (1, 0, 160, 1.0)])
    p.check()


@pytest.mark.gpu
def test_fft640_strided_and_contiguous():
    """640 points along a strided axis (fft640_cols) and along the contiguous axis ([B, 320, 640]: fft1d_rows_kernel with
    the fixed 10 x 8 x 8 plan, which no other test runs)."""
    p = Path("fft640_cols")
    _fft_case(p, "fft640 cols", 2, 640, 21, 2, [(0, 0, 0, 1.0), (1, 320, 320, 1 / 640), (0, 320, 0, 1.0), (1, 0, 320, 1.0)])
    p.check()
    p = Path("fft640_rows")
    _fft_case(p, "fft640 rows", 2 * 320, 640, 1, 3, [(0, 0, 0, 1.0), (1, 320, 320, 1 / 640), (0, 7, 0, 1.0)])
    p.check()
    from mridc_b200 import fft as mfft

    x = torch.randn((2, 320, 640, 2), device="cuda", generator=_gen(4))
    for centered in (False, True):
        out = p(lambda: mfft.fft2(x, centered, "ortho"))
        xc = torch.view_as_complex(x.double())
        if centered:
            xc = torch.fft.ifftshift(xc, dim=(-2, -1))
        ref = torch.fft.fft2(xc, norm="ortho")
        if centered:
            ref = torch.fft.fftshift(ref, dim=(-2, -1))
        check_slices("fft2 [2, 320, 640] centred=%d" % centered, out, torch.view_as_real(ref), 2e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [320, 640])
def test_fft_rotations_outside_the_fast_paths(n):
    """Rotations other than 0 and n/2 (mrb_fft1d_c2c's general index rotation) take the generic kernels at 320 and 640."""
    p = Path("fft_other_rotations")
    _fft_case(p, "rot rows", 5, n, 1, 5, [(0, 7, 100, 1.0), (1, n - 1, 3, 1.0 / n)])
    _fft_case(p, "rot cols", 2, n, 9, 6, [(0, 11, 0, 1.0), (1, 0, 1, 1.0)])
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1024, 2048, 4096, 6144, 8192, 4093, 8191])
def test_fft_long_lengths(n):
    """Lengths past the tested 1000, up to kMaxFftLen = 8192 (one line per CTA: ~196 KB of shared memory), on the rows
    and on the cols kernel; 4093 and 8191 are primes, one O(p^2) generic stage."""
    p = Path("fft_long")
    e = _fft_case(p, "long rows", 3, n, 1, n, [(0, 0, 0, 1.0), (1, n // 2, n // 2, 1.0 / n)])
    e = max(e, _fft_case(p, "long cols", 2, n, 5, n + 1, [(0, 0, 0, 1.0), (1, n // 2, n // 2, 1.0 / n)]))
    print("[kernel paths] fft n=%d worst rel-L2 vs fp64 %.2e" % (n, e))
    p.check()


@pytest.mark.gpu
def test_fft2_over_two_prime_axes():
    """A 2-D transform whose both axes are large primes (4093 x 8191): two generic O(p^2) stages in a row, vs fp64."""
    from mridc_b200 import fft as mfft

    p = Path("fft2_primes")
    x = torch.randn((1, 4093, 8191, 2), device="cuda", generator=_gen(8191))
    xc = torch.view_as_complex(x.double())
    for inverse, centered, norm in ((False, False, "backward"), (True, True, "ortho")):
        out = p(lambda: (mfft.ifft2 if inverse else mfft.fft2)(x, centered, norm))
        z = torch.fft.ifftshift(xc, dim=(-2, -1)) if centered else xc
        z = (torch.fft.ifft2 if inverse else torch.fft.fft2)(z, norm=norm)
        z = torch.fft.fftshift(z, dim=(-2, -1)) if centered else z
        e = check_slices("fft2 4093 x 8191 inverse=%d centred=%d" % (inverse, centered), out, torch.view_as_real(z), 2e-6)
        print("[kernel paths] fft2 4093 x 8191 inverse=%d rel-L2 vs fp64 %.2e" % (inverse, float(e.max())))
        del out, z
    p.check()


@pytest.mark.gpu
def test_fft_length_8193_is_refused():
    x = torch.zeros((1, 8193, 1), dtype=torch.complex64, device="cuda")
    for inner in (1, 2):
        with pytest.raises(NotImplementedError, match="8193"):
            _fft1d(lambda f: f(), x.reshape(1, 8193, 1).expand(1, 8193, inner).contiguous(), 0, 0, 0)


@pytest.mark.gpu
def test_roll_every_element_size():
    """mrb_roll moves 1, 2, 4, 8 and 16-byte elements, bit-exact."""
    from mridc_b200 import fft as mfft

    p = Path("roll")
    g = torch.Generator().manual_seed(9)
    base = torch.randint(-2 ** 31, 2 ** 31 - 1, (3, 7, 5), generator=g, dtype=torch.int64)
    for dt in (torch.uint8, torch.int16, torch.float32, torch.int64, torch.complex128):
        x = (base.to(torch.float64) / 3).to(dt) if dt.is_floating_point or dt.is_complex else base.to(dt)
        x = x.cuda()
        for dim, shift in ((1, 3), (0, -1), (2, 9)):
            out = p(lambda: mfft.roll_one_dim(x, shift, dim))
            assert torch.equal(out, torch.roll(x, shift, dim)), (dt, dim, shift)
    p.check()


# ---------------------------------------------------------------------------------------------- DC (dc.cu)
MASKS = ["u8-shared", "f32-shared", "u8-per-slice", "f32-per-slice"]


def _dc_inputs(B, C, H, W, seed):
    g = _gen(seed)
    y = torch.randn((B, C, H, W, 2), device="cuda", generator=g)
    S = torch.randn((B, C, H, W, 2), device="cuda", generator=g) * 0.5
    eta = torch.randn((B, H, W, 2), device="cuda", generator=g)
    return y, S, eta, g


def _mask(kind, B, H, W, g, two_d=False, density=0.3):
    dtype, scope = kind.split("-", 1)
    shape = ((B if scope == "per-slice" else 1), 1, H if two_d else 1, W, 1)
    m = torch.rand(shape, device="cuda", generator=g) < density
    m[..., W // 2 - 2:W // 2 + 2, :] = True  # a sampled centre
    if dtype == "u8":
        return m.to(torch.uint8)
    return m.float() * (0.5 + torch.rand(shape, device="cuda", generator=g))  # the mask value multiplies


def _norm(centered):
    return "ortho" if centered else "backward"


def _dc_check(path, tag, y, S, eta, m, centered, hybrid, nhwc_modes=(False, True), tol=2e-6):
    """dc_rim_grad (hybrid row form or general three-pass) vs the oracle in fp64, per slice; eta channels bit-exact."""
    from mridc_b200 import _ops
    from oracle import nets as onets

    B, C, H, W, _ = y.shape
    nrm = _norm(centered)
    yh = None
    if hybrid:
        mcan = _ops.canonical_mask(m, B, H, W)[0]
        yh = path(lambda: _ops.dc_hybrid_prepare(y, mcan, centered))
        assert yh is not None
    ref = onets.log_likelihood_gradient(eta.double(), y.double(), S.double(), m.double(), 1.3, centered, nrm, [-2, -1], 1)
    for nhwc in nhwc_modes:
        out = path(lambda: _ops.dc_rim_grad(eta, y, S, m, 1.3, centered, nrm, nhwc=nhwc, y_hybrid=yh))
        if nhwc:
            out = out.permute(0, 3, 1, 2)
        assert torch.equal(out[:, :2], eta.permute(0, 3, 1, 2))
        check_slices("%s %s %dx%dx%dx%d cen=%d nhwc=%d" % (tag, "hybrid" if hybrid else "3-pass", B, C, H, W, centered, nhwc),
                     out[:, 2:], ref[:, 2:], tol)


@pytest.mark.gpu
@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("centered", [False, True])
def test_row_dc_kernel_register_resident_coils(centered, mask):
    """row_dc_kernel<1|2, true>: every column on its own thread (W <= 1024) and at most 8 coils per chunk keep the coil
    images in registers (W = 256, C = 8)."""
    p = Path("row_dc_keep")
    y, S, eta, g = _dc_inputs(2, 8, 24, 256, 11)
    _dc_check(p, "row_dc keep", y, S, eta, _mask(mask, 2, 24, 256, g), centered, True)
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("centered", [False, True])
def test_row_dc_kernel_streamed_coils(centered, mask):
    """row_dc_kernel<1|2, false>: 20 coils of a narrow image fit one chunk (> 8 coils: re-read from shared memory)."""
    p = Path("row_dc_nokeep")
    y, S, eta, g = _dc_inputs(2, 20, 16, 64, 12)
    _dc_check(p, "row_dc stream", y, S, eta, _mask(mask, 2, 16, 64, g), centered, True)
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("W", [1025, 2048, 4096])
@pytest.mark.parametrize("mask", ["u8-shared", "f32-per-slice"])
@pytest.mark.parametrize("centered", [False, True])
def test_dc_rows_wider_than_1024(W, centered, mask):
    """W > 1024: the row kernels give each thread up to kMaxOwn = 4 columns (hybrid row form and the three-pass form with
    the same column mask)."""
    p = Path("dc_wide")
    y, S, eta, g = _dc_inputs(2, 3, 8, W, W)
    m = _mask(mask, 2, 8, W, g)
    _dc_check(p, "dc W=%d" % W, y, S, eta, m, centered, True)
    _dc_check(p, "dc W=%d" % W, y, S, eta, m, centered, False)
    p.check()


@pytest.mark.gpu
def test_dc_width_4097_is_refused():
    from mridc_b200 import _ops

    y, S, eta, g = _dc_inputs(1, 1, 4, 4097, 1)
    m = torch.ones((1, 1, 1, 4097, 1), dtype=torch.uint8, device="cuda")
    yh = _ops.dc_hybrid_prepare(y, m, False)
    with pytest.raises(NotImplementedError, match="4097"):
        _ops.dc_rim_grad(eta, y, S, m, 1.0, False, "backward", y_hybrid=yh)
    with pytest.raises(NotImplementedError, match="4097"):
        _ops.dc_rim_grad(eta, y, S, m, 1.0, False, "backward")
    with pytest.raises(NotImplementedError, match="4097"):
        _ops.sens_reduce(y, S, False, "backward")


@pytest.mark.gpu
@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("centered", [False, True])
def test_dc_twenty_coils_at_320(centered, mask):
    """C = 20 > 16 at 320 x 320 leaves the 320-point kernels: the generic hybrid row kernel for a column mask, the
    generic three-pass kernels for a 2-D mask."""
    p = Path("dc_c20_320_1d")
    y, S, eta, g = _dc_inputs(2, 20, 320, 320, 20)
    _dc_check(p, "dc C=20", y, S, eta, _mask(mask, 2, 320, 320, g), centered, True)
    p.check()
    p = Path("dc_c20_320_2d")
    _dc_check(p, "dc C=20 2-D mask", y, S, eta, _mask(mask, 2, 320, 320, g, two_d=True), centered, False)
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("HW", [(640, 320), (320, 640)])
@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("centered", [False, True])
def test_dc_2d_masks_off_320x320(HW, centered, mask):
    """2-D masks at 640 x 320 (generic column kernel on the 640 plan) and 320 x 640 (640-point rows)."""
    H, W = HW
    p = Path("dc_2d_640")
    y, S, eta, g = _dc_inputs(2, 4, H, W, 21)
    _dc_check(p, "dc 2-D mask", y, S, eta, _mask(mask, 2, H, W, g, two_d=True), centered, False)
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("centered", [False, True])
def test_dc_fully_sampled_columns(centered):
    """Every column sampled: compact_hybrid_kernel packs all W columns."""
    p = Path("dc_full_columns")
    y, S, eta, g = _dc_inputs(2, 4, 40, 96, 22)
    m = torch.ones((1, 1, 1, 96, 1), dtype=torch.uint8, device="cuda")
    _dc_check(p, "dc all columns", y, S, eta, m, centered, True, nhwc_modes=(False,))
    p.check()


def _sens_check(path, tag, B, C, H, W, centered, mask, seed):
    from mridc_b200 import _ops
    from oracle import nets as onets

    y, S, _, g = _dc_inputs(B, C, H, W, seed)
    y64, S64, nrm = y.double(), S.double(), _norm(centered)
    red = path(lambda: _ops.sens_reduce(y, S, centered, nrm))
    check_slices("sens_reduce %s %dx%dx%dx%d cen=%d" % (tag, B, C, H, W, centered), red,
                 onets.sens_reduce(y64, S64, centered, nrm, [-2, -1], 1)[:, 0], 2e-6)
    img = torch.randn((B, H, W, 2), device="cuda", generator=g)
    E = onets.sens_expand(img.double().unsqueeze(1), S64, centered, nrm, [-2, -1])
    out = path(lambda: _ops.sens_expand_softdc(img, S, None, None, None, None, None, True, centered, nrm))
    check_slices("sens_expand %s %dx%dx%dx%d cen=%d" % (tag, B, C, H, W, centered), out, E, 2e-6)
    m = _mask(mask, B, H, W, g)
    pred = torch.randn(y.shape, device="cuda", generator=g) * E.std().item()
    dcw = torch.tensor([0.8], device="cuda")
    out = path(lambda: _ops.sens_expand_softdc(img, S, pred, pred, y, m, dcw, False, centered, nrm))
    p64 = pred.double()
    ref = p64 - torch.where(m.bool(), p64 - y64, torch.zeros((), dtype=torch.float64, device="cuda")) * 0.8 - E
    check_slices("sens_expand_softdc %s %dx%dx%dx%d cen=%d" % (tag, B, C, H, W, centered), out, ref, 2e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("mask", ["u8-shared", "f32-per-slice"])
@pytest.mark.parametrize("centered", [False, True])
def test_sens_operators_twenty_coils(centered, mask):
    """sens_reduce / sens_expand_softdc at C = 20 for H = 320 and 640 (W = 320): the generic row and column kernels."""
    p = Path("sens_c20")
    for H in (320, 640):
        _sens_check(p, "C=20", 2, 20, H, 320, centered, mask, H)
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("centered", [False, True])
def test_sens_operators_320_rows_other_heights(centered):
    """W = 320, C <= 16, H neither 320 nor 640: the 320-point row kernels feed the generic soft-DC column kernel, which then
    must not rotate along W a second time (the ``row320 ? 0 : rw`` argument)."""
    p = Path("sens_row320_other_h")
    _sens_check(p, "H=200", 2, 4, 200, 320, centered, "u8-per-slice", 23)
    p.check()


def _dc320_rows():
    """The 320-point DC kernels on 2 slices of 15 x 320 x 320: the hybrid row kernel in all three output modes (the G8 mode
    == the fp32 output through mrb_g8_from_nhwc4, byte for byte) and the three-pass kernels for a 2-D mask."""
    from mridc_b200 import _ops

    L, lib, st = _lib()
    p = Path("dc320")
    y, S, eta, g = _dc_inputs(2, 15, 320, 320, 24)
    _dc_check(p, "dc320", y, S, eta, _mask("u8-per-slice", 2, 320, 320, g), False, True)
    _dc_check(p, "dc320 2-D mask", y, S, eta, _mask("f32-shared", 2, 320, 320, g, two_d=True), True, False)
    m = _mask("u8-shared", 2, 320, 320, g)
    mcan = _ops.canonical_mask(m, 2, 320, 320)[0]
    yh = _ops.dc_hybrid_prepare(y, mcan, False)
    g4 = _ops.dc_rim_grad(eta, y, S, mcan, 1.0, False, "backward", nhwc=True, y_hybrid=yh)
    ga = torch.zeros(lib.mrb_g8_bytes(2, 320, 320), dtype=torch.uint8, device="cuda")
    p(lambda: L.check(lib.mrb_g8_from_nhwc4(L.ptr(g4), L.ptr(ga), 2, 320, 320, st)))
    gb = torch.zeros_like(ga)
    p(lambda: _ops.dc_rim_grad(eta, y, S, mcan, 1.0, False, "backward", out=gb, nhwc=2, y_hybrid=yh))
    assert torch.equal(ga, gb)
    p.check()


@pytest.mark.gpu
def test_dc_320_point_kernels():
    _dc320_rows()


@pytest.mark.gpu
def test_sens_320_point_kernels():
    _sens320_rows()


def _sens320_rows():
    """reduce_row320<0>, expand_row320, col_softdc320 (H = 320, C = 15) and col_softdc640 (H = 640, C = 16)."""
    p = Path("sens320")
    _sens_check(p, "320", 2, 15, 320, 320, False, "u8-shared", 25)
    _sens_check(p, "640", 1, 16, 640, 320, True, "f32-per-slice", 26)
    p.check()


# ---------------------------------------------------------------------------------------------- convolutions
@pytest.mark.gpu
def test_conv2d_every_instantiation():
    """All 20 conv2d_kernel<TN, K, DIL>: Cout 8 / 16 / 32 / 64 (TN 1 / 2 / 4 / 8) x (k, dil) (5,1) (3,2) (3,1) (1,1) and
    (7,1) (runtime k).  The epilogues rotate over the rows: zero / replicate padding, none / ReLU / leaky activation, the
    IndRNN add * add_scale term, the channels-last residual output, batch strides wider than the tensor."""
    from mridc_b200 import _ops

    p = Path("conv2d")
    g = _gen(30)
    i = 0
    for cout in CONV_COUT:
        for k, dil in CONV_KD:
            N, Cin, H, W = 2, 5, 19, 37
            pad_mode = _ops.PAD_REPLICATE if i % 2 else _ops.PAD_ZERO
            act, slope = [(_ops.ACT_NONE, 0.0), (_ops.ACT_RELU, 0.0), (_ops.ACT_LEAKY, 0.2)][i % 3]
            use_add, use_res, wide = i % 4 == 1, i % 5 == 2, i % 3 == 0
            xbs, obs = Cin * H * W + (13 if wide else 0), cout * H * W + (7 if wide else 0)
            xbuf = torch.randn((N, xbs), device="cuda", generator=g)
            x = xbuf[:, :Cin * H * W].reshape(N, Cin, H, W)
            w = torch.randn((cout, Cin, k, k), device="cuda", generator=g) / (Cin * k * k) ** 0.5
            b = torch.randn((cout,), device="cuda", generator=g)
            add = torch.randn((N, cout, H, W), device="cuda", generator=g) if use_add else None
            add_scale = torch.randn((cout,), device="cuda", generator=g) if use_add else None
            res = torch.randn((N, H, W, cout), device="cuda", generator=g) if use_res else None
            out = torch.full((N, obs), float("nan"), device="cuda") if not use_res else None
            r = p(lambda: _ops.conv2d(xbuf, w, b, k, dil, pad_mode, act, slope, add, add_scale, res, out=out,
                                      x_bstride=xbs, out_bstride=obs, N=N, Cin=Cin, H=H, W=W))
            pd = dil * (k - 1) // 2
            x64 = F.pad(x.double(), (pd, pd, pd, pd), mode="replicate" if pad_mode == _ops.PAD_REPLICATE else "constant")
            ref = F.conv2d(x64, w.double(), b.double(), dilation=dil)
            if use_add:
                ref = ref + add_scale.double()[:, None, None] * add.double()
            ref = F.relu(ref) if act == _ops.ACT_RELU else F.leaky_relu(ref, slope) if act == _ops.ACT_LEAKY else ref
            tag = "conv2d Cout=%d k=%d dil=%d pad=%d act=%d add=%d res=%d wide=%d" % (cout, k, dil, pad_mode, act, use_add,
                                                                                 use_res, wide)
            if use_res:
                check_slices(tag, r, res.double() + ref.permute(0, 2, 3, 1), 2e-6)
            else:
                check_slices(tag, r[:, :cout * H * W].reshape(N, cout, H, W), ref, 2e-6)
                assert torch.isnan(r[:, cout * H * W:]).all()
            i += 1
    p.check()


def _bh(lib, L, t, B, H, W, st):
    buf = torch.empty(lib.mrb_bh_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    L.check(lib.mrb_bh_from_nhwc(L.ptr(t), L.ptr(buf), B, H, W, st))
    return buf


def _from_bh(lib, L, buf, B, H, W, st):
    out = torch.empty((B, H, W, 64), device="cuda")
    L.check(lib.mrb_bh_to_nhwc(L.ptr(buf), L.ptr(out), B, H, W, st))
    return out.permute(0, 3, 1, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [11, 12])
def test_final_conv_on_both_sides_of_16_padded_rows(H):
    """A RIM block on one 11 x 40 image (B * (H + 4) = 15) runs its final conv on the CUDA-core conv_c2_k3 kernel after a
    border fix-up, on a 12 x 40 image (16 padded rows, the height of the tap GEMM's TMA box) on the tensor-core fin2 kernel:
    the engine's own dispatch; every time step vs the fp64 oracle (3e-5 per RIM block)."""
    from mridc_b200 import synth
    from oracle import nets as onets

    cfg = synth.cirim_cfg("GRU", centered=True, normalization="ortho")
    blk = _rim_block(cfg, 8)
    with torch.no_grad():
        for st in blk.layers:
            st.convs.conv_layer.bias.normal_(0, 0.1)
            st.rnn.ih.bias.normal_(0, 0.1)
    sd64 = {k: v.detach().cuda().double() for k, v in blk.state_dict().items()}
    batch = synth.make_batch(1, 3, H, 40, centered=True, normalization="ortho")
    y, S, m = (batch[k].cuda() for k in ("y", "sensitivity_maps", "mask"))
    blk = blk.cuda()
    p = Path("final_conv_tc" if H + 4 >= 16 else "final_conv_cuda_core")
    etas, _ = p(lambda: blk(y, y, S, m, None, None, 1.0, False))
    assert blk._tc_engine and blk._tc_engine.covers(40)
    with torch.no_grad():
        ref, _ = onets.rim_block(sd64, dict(cfg), y.double(), y.double(), S.double(), m, None, None, 1.0, False)
    for t, (a_, b_) in enumerate(zip(etas, ref)):
        check_slices("RIM block 1x%dx40 step %d" % (H, t), a_, b_, 3e-5)
    p.check()




@pytest.mark.gpu
@pytest.mark.parametrize("k,dil,bias", [(5, 1, False), (1, 1, True), (1, 1, False), (3, 1, False)])
def test_tc_conv_bh_kernel_sizes_and_null_bias(k, dil, bias):
    """mrb_tc_conv_bh (tc_kernel) at the kernel sizes RimTcEngine.supported() accepts besides the shipped 3x3 d2: 5x5 and
    1x1, and with a null bias; split-bf16 tolerance 1e-5."""
    from oracle import nets as onets

    L, lib, st = _lib()
    p = Path("tc_conv_bh")
    B, H, W = 2, 30, 45
    g = _gen(50 + k)
    x = torch.randn((B, H, W, 64), device="cuda", generator=g)
    xb = p(lambda: _bh(lib, L, x, B, H, W, st))
    w = torch.randn((64, 64, k, k), device="cuda", generator=g) * (1.0 / (64 * k * k)) ** 0.5
    b = torch.randn(64, device="cuda", generator=g) if bias else None
    pk = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, k), device="cuda")
    p(lambda: L.check(lib.mrb_tc_pack_conv(L.ptr(w), L.ptr(pk), 64, 64, k, st)))
    ob = torch.full((lib.mrb_bh_bytes(B, H, W),), 0x7F, dtype=torch.uint8, device="cuda")
    p(lambda: L.check(lib.mrb_tc_conv_bh(L.ptr(xb), L.ptr(pk), L.ptr(b), L.ptr(ob), B, H, W, 64, k, dil, 1, st)))
    ref = onets.conv_nonlinear(x.permute(0, 3, 1, 2).double(), w.double(), b.double() if bias else None, k, dil, "relu")
    check_slices("tc_conv_bh k=%d dil=%d bias=%d" % (k, dil, bias), p(lambda: _from_bh(lib, L, ob, B, H, W, st)), ref, 1e-5)
    p.check()


@pytest.mark.gpu
def test_tc2_kernels_with_null_biases():
    """conv5x5x4 (G8 -> BH), ConvGRU with b_ih = null (the config's recurrent_bias False), IndRNN, final conv and the border
    fix-up, each vs fp64 (split-bf16: 1e-5)."""
    from oracle import nets as onets

    L, lib, st = _lib()
    p = Path("tc2_ops")
    B, H, W = 2, 20, 36
    g = _gen(60)
    x4 = torch.randn((B, H, W, 4), device="cuda", generator=g)
    w1 = torch.randn((64, 4, 5, 5), device="cuda", generator=g) * 0.2
    g8 = torch.zeros(lib.mrb_g8_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    p(lambda: L.check(lib.mrb_g8_from_nhwc4(L.ptr(x4), L.ptr(g8), B, H, W, st)))
    ob = torch.empty(lib.mrb_bh_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    p(lambda: L.check(lib.mrb_tc2_conv5x5x4(L.ptr(g8), L.ptr(w1), None, L.ptr(ob), B, H, W, 1, st)))
    ref = onets.conv_nonlinear(x4.permute(0, 3, 1, 2).double(), w1.double(), None, 5, 1, "relu")
    check_slices("tc2_conv5x5x4 null bias", _from_bh(lib, L, ob, B, H, W, st), ref, 1e-5)
    x, h = torch.randn((B, H, W, 64), device="cuda", generator=g), torch.randn((B, H, W, 64), device="cuda", generator=g)
    xb, hb = _bh(lib, L, x, B, H, W, st), _bh(lib, L, h, B, H, W, st)
    x64, h64 = x.permute(0, 3, 1, 2).double(), h.permute(0, 3, 1, 2).double()
    wih, whh = torch.randn((192, 64, 1, 1), device="cuda", generator=g) * 0.1, torch.randn((192, 64, 1, 1), device="cuda",
                                                                                          generator=g) * 0.1
    pk = torch.empty(lib.mrb_tc2_gru_packed_bytes(), dtype=torch.uint8, device="cuda")
    L.check(lib.mrb_tc2_pack_gru(L.ptr(wih), L.ptr(whh), L.ptr(pk), 64, 64, st))
    p(lambda: L.check(lib.mrb_tc2_gru(L.ptr(xb), L.ptr(hb), L.ptr(pk), None, L.ptr(ob), B, H, W, st)))
    check_slices("tc2_gru null b_ih", _from_bh(lib, L, ob, B, H, W, st),
                 onets.conv_gru_cell(x64, h64, wih.double(), None, whh.double(), 1, 1), 1e-5)
    wi, hh = torch.randn((64, 64, 1, 1), device="cuda", generator=g) * 0.1, torch.randn((1, 64, 1, 1), device="cuda",
                                                                                       generator=g) * 0.5
    pi = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, 1), device="cuda")
    L.check(lib.mrb_tc_pack_conv(L.ptr(wi), L.ptr(pi), 64, 64, 1, st))
    hhd = hh.reshape(-1).contiguous()
    p(lambda: L.check(lib.mrb_tc2_indrnn(L.ptr(xb), L.ptr(hb), L.ptr(pi), None, L.ptr(hhd), L.ptr(ob), B, H, W, st)))
    check_slices("tc2_indrnn null b_ih", _from_bh(lib, L, ob, B, H, W, st),
                 onets.indrnn_cell(x64, h64, wi.double(), None, hh.double(), 1, 1), 1e-5)
    # the border fix-up: a BH tensor whose 2-pixel border is poisoned gets back, byte for byte, the replicate border
    # mrb_bh_from_nhwc writes
    ref_bh = _bh(lib, L, x, B, H, W, st)
    v = xb.view(B, H + 4, W + 4, 256)
    v[:, :2] = 0x7F
    v[:, -2:] = 0x7F
    v[:, :, :2] = 0x7F
    v[:, :, -2:] = 0x7F
    assert not torch.equal(xb, ref_bh)
    p(lambda: L.check(lib.mrb_bh_fix_border(L.ptr(xb), B, H, W, st)))
    assert torch.equal(xb, ref_bh)
    w3, eta = torch.randn((2, 64, 3, 3), device="cuda", generator=g) * 0.05, torch.randn((B, H, W, 2), device="cuda", generator=g)
    o = torch.empty((B, H, W, 2), device="cuda")
    p(lambda: L.check(lib.mrb_tc2_final_conv(L.ptr(xb), L.ptr(w3), None, L.ptr(eta), L.ptr(o), B, H, W, st)))
    ref = eta.double() + onets.conv_nonlinear(x64, w3.double(), None, 3, 1, None).permute(0, 2, 3, 1)
    check_slices("tc2_final_conv null bias", o, ref, 1e-5)
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("Cin", [16, 32, 64, 3, 20])
def test_uconv3_instantiations(Cin):
    """uconv3_kernel<1> for Cin <= 16, <2> for Cin <= 32, <4> above (channel groups of 8, padded); O(1) inputs (what the
    U-Net's instance norm hands it), uconv3 tolerance 2e-6."""
    L, lib, st = _lib()
    inst = 1 if Cin <= 16 else 2 if Cin <= 32 else 4
    p = Path("uconv3_%d" % inst)
    N, H, W, Cout = 2, 23, 41, 24
    g = _gen(70 + Cin)
    xbs = Cin * H * W + 4
    x = torch.randn((N, xbs), device="cuda", generator=g)
    w = torch.randn((Cout, Cin, 3, 3), device="cuda", generator=g) / (9 * Cin) ** 0.5
    pk = torch.empty(lib.mrb_tc2_unet_packed_bytes(Cin, Cout), dtype=torch.uint8, device="cuda")
    p(lambda: L.check(lib.mrb_tc2_unet_pack(L.ptr(w), L.ptr(pk), Cin, Cout, st)))
    out = torch.empty((N, Cout, H, W), device="cuda")
    p(lambda: L.check(lib.mrb_tc2_unet_conv3x3(L.ptr(x), xbs, L.ptr(pk), L.ptr(out), Cout * H * W, N, Cin, Cout, H, W, st)))
    ref = F.conv2d(x[:, :Cin * H * W].reshape(N, Cin, H, W).double(), w.double(), padding=1)
    check_slices("uconv3 Cin=%d" % Cin, out, ref, 2e-6)
    p.check()


# ---------------------------------------------------------------------------------------------- model level
def _rim_block(cfg, seed):
    from mridc_b200.rim import RIMBlock

    kw = {k: cfg[k] for k in ("recurrent_layer", "conv_filters", "conv_kernels", "conv_dilations", "conv_bias",
                              "recurrent_filters", "recurrent_kernels", "recurrent_dilations", "recurrent_bias",
                              "depth", "time_steps", "conv_dim", "no_dc", "fft_centered", "fft_normalization",
                              "spatial_dims", "coil_dim", "dimensionality")}
    torch.manual_seed(seed)
    return RIMBlock(**kw).eval()


def _k5_cfg():
    from mridc_b200 import synth

    cfg = synth.cirim_cfg("GRU", centered=True, normalization="ortho")
    cfg.update(conv_kernels=[5, 5, 3], conv_dilations=[1, 1, 1], conv_bias=[False, False, False],
               recurrent_bias=[False, False, False])
    return cfg


@pytest.mark.gpu
@pytest.mark.parametrize("W", [40, 28, 27])
def test_rim_block_5x5_second_conv_no_biases(W):
    """A RIM block with conv_kernels [5, 5, 3], dilations 1 and every conv and recurrent bias off: the engine runs it at
    W >= 28 (tc_kernel with k = 5, null biases), the exact-fp32 loop at W = 27; every time step vs the fp64 oracle (3e-5)."""
    from mridc_b200 import synth
    from oracle import nets as onets

    cfg = _k5_cfg()
    blk = _rim_block(cfg, 6)
    assert all(st.convs.conv_layer.bias is None for st in blk.layers) and all(st.rnn.ih.bias is None for st in blk.layers)
    sd64 = {k: v.detach().cuda().double() for k, v in blk.state_dict().items()}
    batch = synth.make_batch(2, 4, 36, W, centered=True, normalization="ortho")
    y, S, m = (batch[k].cuda() for k in ("y", "sensitivity_maps", "mask"))
    blk = blk.cuda()
    (etas, hx), names = launched(lambda: blk(y, y, S, m, None, None, 1.0, False))
    with torch.no_grad():
        ref, _ = onets.rim_block(sd64, dict(cfg), y.double(), y.double(), S.double(), m, None, None, 1.0, False)
    p = Path("rim_block_k5_nobias" if W >= 28 else "rim_block_w27")
    p.seen = names
    assert bool(blk._tc_engine) and blk._tc_engine.covers(W) == (W >= 28)
    for t, (a, b) in enumerate(zip(etas, ref)):
        check_slices("RIM block k5 no-bias W=%d step %d" % (W, t), a, b, 3e-5)
    p.check()


@pytest.mark.gpu
def test_cirim_twenty_coils_at_320():
    """One CIRIM cascade at (1, 20, 320, 320): C > 16 turns off the DC kernel's direct G8 write, so the engine takes the
    fp32 g4 gradient through mrb_g8_from_nhwc4; every estimate vs the fp64 oracle (1e-4)."""
    import mridc_b200 as mb
    from mridc_b200 import synth
    from oracle import models as omodels

    cfg = synth.cirim_cfg("GRU", num_cascades=1)
    batch = synth.make_batch(1, 20, 320, 320)
    torch.manual_seed(7)
    model = mb.CIRIM(cfg).eval()
    sd64 = {k: v.detach().cuda().double() for k, v in model.state_dict().items()}
    y, S, m, tgt = (batch[k].cuda() for k in ("y", "sensitivity_maps", "mask", "target"))
    model = model.cuda()
    out, names = launched(lambda: [list(c) for c in next(model(y, S, m, None, tgt))])
    p = Path("cirim_c20")
    p.seen = names
    assert model.cirim[0]._tc_engine
    with torch.no_grad():
        ref = omodels.cirim_forward(sd64, cfg, y.double(), S.double(), m, None, tgt)
    for t, (a, b) in enumerate(zip(out[0], ref[0])):
        check_slices("CIRIM 1x20x320x320 step %d" % t, a, b, 1e-4)
    p.check()


@pytest.mark.gpu
def test_rim_cells_on_cuda_cores():
    """The exact-fp32 cells: the fused 1x1 ConvGRU cell, and the GRU / MGU gate kernels on precomputed ih, hh (the k > 1
    cells), each vs the oracle's gate arithmetic in fp64 (2e-6)."""
    L, lib, st = _lib()
    from oracle import nets as onets

    p = Path("rim_cells_fp32")
    g = _gen(80)
    N, Cx, Ch, H, W = 2, 12, 20, 9, 17
    HW = H * W
    x, h = torch.randn((N, Cx, H, W), device="cuda", generator=g), torch.randn((N, Ch, H, W), device="cuda", generator=g)
    wih, whh = torch.randn((3 * Ch, Cx, 1, 1), device="cuda", generator=g) * 0.3, torch.randn((3 * Ch, Ch, 1, 1), device="cuda",
                                                                                             generator=g) * 0.3
    bih = torch.randn(3 * Ch, device="cuda", generator=g)
    out = torch.empty_like(h)
    p(lambda: L.check(lib.mrb_gru_cell_1x1(L.ptr(x), L.ptr(h), L.ptr(wih), L.ptr(bih), L.ptr(whh), L.ptr(out), N, Cx, Ch, HW, st)))
    check_slices("gru_cell_1x1", out, onets.conv_gru_cell(x.double(), h.double(), wih.double(), bih.double(), whh.double(),
                                                          1, 1), 2e-6)
    for gates, fn in ((3, lib.mrb_gru_gates), (2, lib.mrb_mgu_gates)):
        ih = torch.randn((N, gates * Ch, H, W), device="cuda", generator=g)
        hh = torch.randn((N, gates * Ch, H, W), device="cuda", generator=g)
        o = torch.empty_like(h)
        p(lambda: L.check(fn(L.ptr(ih), L.ptr(hh), L.ptr(h), L.ptr(o), N, Ch, HW, st)))
        a, b, h64 = ih.double().chunk(gates, 1), hh.double().chunk(gates, 1), h.double()
        if gates == 3:
            r, z = torch.sigmoid(a[0] + b[0]), torch.sigmoid(a[1] + b[1])
            n = torch.tanh(a[2] + r * b[2])
            ref = n * (1 - z) + z * h64
        else:
            f = torch.sigmoid(a[0] + b[0])
            c = torch.tanh(a[1] + f * b[1])
            ref = c + f * (h64 - c)
        check_slices("%s gates" % ("gru" if gates == 3 else "mgu"), o, ref, 2e-6)
    p.check()


# ---------------------------------------------------------------------------------------------- U-Net (unet.cu)
def _instnorm_ref(x, N, C, HW):
    return F.leaky_relu(F.instance_norm(x.reshape(N, C, HW).double(), eps=1e-5), 0.2)


def _instnorm(path, x, x_bs, out, out_bs, N, C, HW, stats=None):
    L, lib, st = _lib()
    stats = torch.empty((2 * N * C,), dtype=torch.float64, device="cuda") if stats is None else stats
    path(lambda: L.check(lib.mrb_instnorm_lrelu(L.ptr(x), x_bs, L.ptr(out), out_bs, N, C, HW, 1e-5, 0.2, L.ptr(stats), st)))
    return stats


@pytest.mark.gpu
@pytest.mark.parametrize("HW", [16384, 16385, 32768, 32769, 65536, 65537, 131072, 131073, 409600, 4099])
def test_instnorm_cluster_sizes(HW):
    """instnorm_cluster_kernel at cluster sizes 1, 2, 4 and 8: HW on both sides of each 64 KB step (16384, 32768, 65536,
    131072 floats), odd HW (scalar path), the largest single-pass plane (409,600), into a strided concat buffer, with a
    misaligned batch stride (the scalar path for odd slices) and in place."""
    p = Path("instnorm_cluster")
    N, C = 2, 2
    g = _gen(HW)
    for x_bs in (C * HW, C * HW + 1):
        x = torch.randn((N, x_bs), device="cuda", generator=g) * 1.5 + 0.3
        ref = _instnorm_ref(x[:, :C * HW], N, C, HW)
        out = torch.full((N, C * HW + 8), float("nan"), device="cuda")
        _instnorm(p, x, x_bs, out, C * HW + 8, N, C, HW)
        check_slices("instnorm HW=%d x_bs=%d" % (HW, x_bs), out[:, :C * HW].reshape(N, C, HW), ref, 2e-6)
        assert torch.isnan(out[:, C * HW:]).all()
        _instnorm(p, x, x_bs, x, x_bs, N, C, HW)  # in place
        check_slices("instnorm HW=%d x_bs=%d in place" % (HW, x_bs), x[:, :C * HW].reshape(N, C, HW), ref, 2e-6)
    p.check()


@pytest.mark.gpu
def test_instnorm_two_pass_parity_and_determinism():
    """Planes above 409,600 values (720 x 720) take the two-kernel form.  fp64 parity; the statistics and the output are the
    same bits over two runs and for plane (0, c) whether the launch holds N = 1 or N = 2 planes per channel."""
    p = Path("instnorm_two_pass")
    N, C, HW = 2, 2, 720 * 720
    x = torch.randn((N, C * HW), device="cuda", generator=_gen(90)) * 1.5 + 0.3
    out = torch.empty_like(x)
    s1 = _instnorm(p, x, C * HW, out, C * HW, N, C, HW).clone()
    check_slices("instnorm 2-pass 720x720", out.reshape(N, C, HW), _instnorm_ref(x, N, C, HW), 2e-6)
    out2 = torch.empty_like(x)
    s2 = _instnorm(p, x, C * HW, out2, C * HW, N, C, HW)
    one = torch.empty((1, C * HW), device="cuda")
    s3 = _instnorm(p, x[:1].contiguous(), C * HW, one, C * HW, 1, C, HW)
    same_runs, same_batch = torch.equal(s1, s2) and torch.equal(out, out2), torch.equal(s1[:2 * C], s3) and torch.equal(out[:1], one)
    print("[kernel paths] instnorm two-pass: two runs bit-identical %s, N=1 vs N=2 bit-identical %s" % (same_runs, same_batch))
    assert same_runs and same_batch
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("HW", [(16, 20), (13, 15)])
def test_unet_final_conv_and_its_fallback(HW):
    """The U-Net's last 1x1 conv: mrb_conv1x1 when H * W is a multiple of 4, conv2d with k = 1 otherwise (13 x 15, which
    also takes the reflect pad of odd skip sizes); the whole U-Net vs the fp64 oracle (1e-5)."""
    from mridc_b200.unet import Unet
    from oracle import nets as onets

    H, W = HW
    torch.manual_seed(9)
    net = Unet(2, 2, chans=8, num_pool_layers=2).eval()
    sd64 = {k: v.detach().cuda().double() for k, v in net.state_dict().items()}
    x = torch.randn((2, 2, H, W), device="cuda", generator=_gen(100 + H))
    net = net.cuda()
    p = Path("unet_final_conv1x1" if (H * W) % 4 == 0 else "unet_final_conv2d")
    out = p(lambda: net(x))
    with torch.no_grad():
        ref = onets.unet(x.double(), sd64, 2)
    check_slices("U-Net 2x2x%dx%d" % (H, W), out, ref, 1e-5)
    p.check()


@pytest.mark.gpu
def test_unet_small_ops():
    """conv1x1 (strided batches), avgpool2 on odd sizes, conv_transpose2x2, pad2d in its three modes with positive and
    negative offsets (a crop), each vs fp64 (2e-6) or bit-exact (pad / crop)."""
    L, lib, st = _lib()
    p = Path("unet_small_ops")
    g = _gen(95)
    N, Cin, Cout, H, W = 2, 6, 5, 13, 20
    HW = H * W
    xbs, obs = Cin * HW + 4, Cout * HW + 8
    x = torch.randn((N, xbs), device="cuda", generator=g)
    w = torch.randn((Cout, Cin), device="cuda", generator=g)
    b = torch.randn(Cout, device="cuda", generator=g)
    out = torch.full((N, obs), float("nan"), device="cuda")
    p(lambda: L.check(lib.mrb_conv1x1(L.ptr(x), xbs, L.ptr(w), L.ptr(b), L.ptr(out), obs, N, Cin, Cout, HW, st)))
    ref = torch.einsum("oc,nch->noh", w.double(), x[:, :Cin * HW].reshape(N, Cin, HW).double()) + b.double()[:, None]
    check_slices("conv1x1", out[:, :Cout * HW].reshape(N, Cout, HW), ref, 2e-6)
    assert torch.isnan(out[:, Cout * HW:]).all()
    with pytest.raises(NotImplementedError):  # H * W % 4 != 0: the U-Net takes conv2d with k = 1 instead
        L.check(lib.mrb_conv1x1(L.ptr(x), xbs, L.ptr(w), L.ptr(b), L.ptr(out), obs, N, Cin, Cout, 13 * 19, st))
    for Hp, Wp in ((13, 21), (14, 20), (3, 2)):
        xp = torch.randn((N, Cin, Hp, Wp), device="cuda", generator=g)
        op = torch.empty((N, Cin, Hp // 2, Wp // 2), device="cuda")
        p(lambda: L.check(lib.mrb_avgpool2(L.ptr(xp), Cin * Hp * Wp, L.ptr(op), Cin * (Hp // 2) * (Wp // 2), N, Cin, Hp, Wp, st)))
        check_slices("avgpool2 %dx%d" % (Hp, Wp), op, F.avg_pool2d(xp.double(), 2), 2e-6)
    wt = torch.randn((Cin, Cout, 2, 2), device="cuda", generator=g)
    xt = torch.randn((N, Cin, H, W), device="cuda", generator=g)
    ot = torch.empty((N, Cout, 2 * H, 2 * W), device="cuda")
    p(lambda: L.check(lib.mrb_conv_transpose2x2(L.ptr(xt), Cin * HW, L.ptr(wt), L.ptr(ot), Cout * 4 * HW, N, Cin, Cout, H, W, st)))
    check_slices("conv_transpose2x2", ot, F.conv_transpose2d(xt.double(), wt.double(), stride=2), 2e-6)
    modes = {0: "constant", 1: "replicate", 2: "reflect"}
    for mode in (0, 1, 2):
        for (Ho, Wo, oy, ox) in ((H + 5, W + 6, 2, 3), (H - 4, W - 6, -2, -3)):
            o = torch.empty((N, Cin, Ho, Wo), device="cuda")
            p(lambda: L.check(lib.mrb_pad2d(L.ptr(xt), Cin * HW, L.ptr(o), Cin * Ho * Wo, N, Cin, H, W, Ho, Wo, oy, ox, mode, st)))
            if oy >= 0:
                ref = F.pad(xt, (ox, Wo - W - ox, oy, Ho - H - oy), mode=modes[mode])
            else:
                ref = xt[:, :, -oy:-oy + Ho, -ox:-ox + Wo]
            assert torch.equal(o, ref), (mode, Ho, Wo, oy, ox)
    p.check()


@pytest.mark.gpu
@pytest.mark.parametrize("normalize", [0, 1])
def test_normunet_prologue_epilogue(normalize):
    L, lib, st = _lib()
    p = Path("normunet_%d" % normalize)
    B, C, HW = 2, 3, 37 * 29
    g = _gen(96)
    x = torch.randn((B, C * HW * 2), device="cuda", generator=g) * 2 + 0.5
    out = torch.empty((B, 2 * C * HW), device="cuda")
    ms = torch.empty((B, 2, 2), device="cuda")
    stats = torch.empty((4 * B,), dtype=torch.float64, device="cuda")
    p(lambda: L.check(lib.mrb_normunet_in(L.ptr(x), L.ptr(out), L.ptr(ms), B, C, HW, normalize, L.ptr(stats), st)))
    planes = x.double().reshape(B, C * HW, 2).permute(0, 2, 1)
    mean, std = planes.mean(-1, keepdim=True), planes.std(-1, keepdim=True)
    if normalize:
        check_slices("normunet_in mean/std", ms, torch.cat((mean, std), -1), 2e-6)
        planes = (planes - mean) / std
    check_slices("normunet_in normalize=%d" % normalize, out, planes.reshape(B, -1), 2e-6)
    y = torch.randn((B, 2 * C * HW), device="cuda", generator=g)
    ms = torch.stack((torch.randn((B, 2), device="cuda", generator=g), torch.rand((B, 2), device="cuda", generator=g) + 0.5),
                     -1).contiguous()
    o = torch.empty((B, C * HW * 2), device="cuda")
    p(lambda: L.check(lib.mrb_normunet_out(L.ptr(y), L.ptr(ms), L.ptr(o), B, C, HW, normalize, st)))
    pl = y.double().reshape(B, 2, C * HW)
    if normalize:
        pl = pl * ms[:, :, 1:].double() + ms[:, :, :1].double()
    check_slices("normunet_out normalize=%d" % normalize, o, pl.permute(0, 2, 1).reshape(B, -1), 2e-6)
    p.check()


# ---------------------------------------------------------------------------------------------- core, metrics, qMRI
@pytest.mark.gpu
def test_complex_and_coil_ops():
    """complex_mul with broadcast strides and conj(y), conj, |x| and |x|^2, rss / rss_complex / sense (coil_reduce<0|1|2>)
    and divide_rss, vs fp64 (2e-6)."""
    import mridc_b200 as mb

    L, lib, st = _lib()
    p = Path("complex_ops")
    g = _gen(97)
    x = torch.randn((2, 5, 9, 11, 2), device="cuda", generator=g)
    yb = torch.randn((1, 5, 1, 11, 2), device="cuda", generator=g)
    xc, yc = torch.view_as_complex(x.double()), torch.view_as_complex(yb.double())
    check_slices("complex_mul broadcast", p(lambda: mb.complex_mul(x, yb)), torch.view_as_real(xc * yc), 2e-6)
    check_slices("complex_mul conj_y", p(lambda: mb.complex_mul(x, yb, True)), torch.view_as_real(xc * yc.conj()), 2e-6)
    assert torch.equal(p(lambda: mb.complex_conj(x)), torch.stack((x[..., 0], -x[..., 1]), -1))
    check_slices("complex_abs", p(lambda: mb.complex_abs(x)), xc.abs(), 2e-6)
    check_slices("complex_abs_sq", p(lambda: mb.complex_abs_sq(x)), xc.abs() ** 2, 2e-6)
    check_slices("rss dim 1", p(lambda: mb.rss(x, 1)), x.double().pow(2).sum(1).sqrt(), 2e-6)
    check_slices("rss_complex dim 1", p(lambda: mb.rss_complex(x, 1)), xc.abs().pow(2).sum(1).sqrt(), 2e-6)
    S = torch.randn_like(x)
    Sc = torch.view_as_complex(S.double())
    check_slices("sense dim 1", p(lambda: mb.sense(x, S, 1)), torch.view_as_real((xc * Sc.conj()).sum(1)), 2e-6)
    out = torch.empty_like(x)
    p(lambda: L.check(lib.mrb_divide_rss(L.ptr(x), L.ptr(out), 2, 5, 9 * 11, st)))
    check_slices("divide_rss", out, torch.view_as_real(xc / xc.abs().pow(2).sum(1, keepdim=True).sqrt()), 2e-6)
    p.check()


@pytest.mark.gpu
def test_metric_kernels():
    """mse / nmse / psnr / ssim and the magnitude normalisation against the numpy fp64 oracle."""
    import mridc_b200 as mb
    from oracle import metrics as om

    p = Path("metrics")
    g = _gen(98)
    G = torch.rand((3, 40, 37), device="cuda", generator=g)
    P = G + 0.05 * torch.randn((3, 40, 37), device="cuda", generator=g)
    a, b = G.double().cpu().numpy(), P.double().cpu().numpy()
    v = p(lambda: (mb.metrics.mse(G, P), mb.metrics.nmse(G, P), mb.metrics.psnr(G, P), mb.metrics.ssim(G, P)))
    ref = (om.mse(a, b), om.nmse(a, b), om.psnr(a, b), om.ssim(a, b))
    print("[kernel paths] metrics CUDA %s | fp64 %s" % (["%.10g" % t for t in v], ["%.10g" % t for t in ref]))
    assert abs(v[0] - ref[0]) <= 2e-6 * ref[0] and abs(v[1] - ref[1]) <= 2e-6 * ref[1]
    assert abs(v[2] - ref[2]) <= 1e-5 and abs(v[3] - ref[3]) <= 1e-7
    xc = torch.randn((2, 19, 23, 2), device="cuda", generator=g)
    nm = p(lambda: mb.metrics.normalized_magnitude(torch.view_as_complex(xc)))
    mag = torch.view_as_complex(xc.double()).abs()
    check_slices("normalized_magnitude", nm, mag / mag.max(), 2e-6)
    p.check()


@pytest.mark.gpu
def test_qmri_kernels():
    """The MEGRE signal model and the qRIM map gradient (echoes folded into the DC batch) vs the per-sample oracle in fp64;
    the eta update with its R2* clamp and RescaleByMax.reverse, bit-exact."""
    import mridc_b200 as mb
    from mridc_b200 import qrim
    from oracle import qnets as oq
    from oracle.make_golden import qmri_inputs

    L, lib, st = _lib()
    p = Path("qmri")
    B, E, C, H, W = 2, 4, 3, 17, 13
    r2, s0, b0, ph, tes, y, S, m = qmri_inputs(B, E, C, H, W, 56, "2db")
    ref = torch.stack([oq.analytical_log_likelihood_gradient(r2[b].double(), s0[b].double(), b0[b].double(), ph[b].double(),
                                                             tes, S[b].double(), y[b].double(), m[b], False, "backward",
                                                             [-2, -1], 2) / 100 for b in range(B)])
    out = torch.full((B, 8, H, W), 7.0, device="cuda")
    maps = [t.cuda() for t in (r2, s0, b0, ph)]
    p(lambda: qrim._qmri_gradient(qrim.SignalForwardModel("MEGRE"), maps, None, tes, S.cuda(), y.cuda(), m.cuda(), False,
                                  "backward", 1e-3, 100.0, True, out, 8))
    check_slices("qMRI map gradient (MEGRE signal + DC + grad)", out[:, :4].cpu(), ref, 5e-6)
    assert (out[:, 4:] == 7.0).all()
    g = _gen(99)
    eta = torch.randn((B, 8, H * W), device="cuda", generator=g)
    delta = torch.randn((B, 4, H * W), device="cuda", generator=g)
    e0 = eta.clone()
    o = torch.empty_like(delta)
    p(lambda: L.check(lib.mrb_qrim_eta_update(L.ptr(eta), 8, 4, L.ptr(delta), L.ptr(o), B, H * W, st)))
    upd = e0[:, 4:8] + delta
    upd[:, 0] = upd[:, 0].clamp_min(0)
    assert torch.equal(eta[:, 4:8], upd) and torch.equal(o, upd) and torch.equal(eta[:, :4], e0[:, :4])
    x = torch.randn((3, 4, 5, 6), device="cuda", generator=g)
    gam = torch.tensor([2.0, 3.0, 5.0])
    r = p(lambda: mb.RescaleByMax.reverse(x, gam))
    assert torch.equal(r, x * gam.cuda().view(3, 1, 1, 1))
    p.check()
