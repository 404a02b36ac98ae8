"""PICS (mridc_b200.pics.l1_wavelet_recon, mridc_b200.PICS, libmridc_b200_pics.so) against the fp64 reference of
tests/test_pics_cpu.py, run in float64 torch on the GPU.

Tolerances.
- Per operator (mrbp_dwt, mrbp_step_size): 2e-6 rel-L2 per slice.  One analysis level is two 8-tap fp32 sums per
  coefficient (about 8 u |c| each, u = 2^-24 = 6e-8, with the fp32 taps themselves off by u); after five levels and back,
  that is a few 1e-7.  The step size is one C-term sum of squares and one division: a few u.
- One step fed from the library's own fp32 state (x_k, z_k) and its own gradient and alpha: 2e-6 per slice for x_{k+1}
  and z_{k+1}.  The step is Psi, a soft-threshold and Psi^H, each 1-Lipschitz up to the fp32 rounding of the transform,
  so the bound is the per-operator one and does not grow with k.
- Free-running solve, 100 iterations: 1e-4 rel-L2 per slice (the package's model contract) and 1e-5 relative objective
  difference.  The fp32 gradient (2e-6 per evaluation, DESIGN section 4.2) and the fp32 step enter every iteration; FISTA
  carries them forward but, on these well-posed problems, does not amplify them by more than the iteration count.  The
  error at k = 1, 10, 30 and 100 is printed so the drift is visible.
- Optimality after 1000 iterations: the library result's fp64 fixed-point residual is at most twice the fp64 solver's
  at the same k, plus 1e-6 (the fp32 floor of a residual relative to |x|).
"""
import ctypes
import gc
import math

import pytest
import torch

from test_gpu_abi_contract import Buf, Row, run_contract
from test_gpu_bench_shapes import check_slices
from test_gpu_kernel_paths import kernel_name, library_instantiations
from test_pics_cpu import Problem, psi, psi_h

OP_TOL = 2e-6
SOLVE_TOL = 1e-4
OBJ_TOL = 1e-5
P_ = "mrb::pics::"
# path -> the kernels it launches; the CPU inventory test compares the union with the instantiations of the library.
# Each path is checked against fp64 here: step_size by test_step_size_against_fp64, dwt by the mrbp_dwt tests,
# fista_step (levels >= 2) by the solves and fista_step_one_level by the contract row fista_step_1_level.
EXPECTED = {
    "step_size": {P_ + "step_size_kernel"},
    "dwt": {P_ + "analysis_kernel<false, false>", P_ + "synthesis_kernel<false>"},
    "fista_step_one_level": {P_ + "analysis_kernel<true, true>", P_ + "synthesis_kernel<true>"},
    "fista_step": {P_ + "analysis_kernel<true, true>", P_ + "analysis_kernel<false, true>",
                   P_ + "synthesis_kernel<false>", P_ + "synthesis_kernel<true>"},
}
SHAPES = [(320, 320), (640, 320), (232, 288), (14, 14), (18, 16)]


@pytest.fixture(autouse=True)
def _release_gpu_memory():
    """The B200 machines are shared: hand the cached blocks of each test back to the driver."""
    yield
    gc.collect()
    if torch.cuda.is_available() and torch.cuda.is_initialized():
        torch.cuda.empty_cache()


def _c(t):
    """[..., 2] real -> complex128."""
    return torch.view_as_complex(t.double().contiguous())


def _r(t):
    """complex -> [..., 2] float32."""
    return torch.view_as_real(t.to(torch.complex64)).contiguous()


def _betas(n):
    t, out = 1.0, []
    for _ in range(n):
        tn = (1 + math.sqrt(1 + 4 * t * t)) / 2
        out.append((t - 1) / tn)
        t = tn
    return out


def _canon(mask, B, H, W):
    from mridc_b200 import _ops

    return _ops.canonical_mask(mask, B, H, W)[0].double()


def _problem(y, S, mask, lamda, centered=True, norm="ortho"):
    B, C, H, W, _ = y.shape
    return Problem(_c(y), _c(S), _canon(mask, B, H, W), lamda, centered, norm)


def _lam_max(y, S, mask, centered=True, norm="ortho"):
    """max |Psi E^H y| per slice: the smallest lamda whose minimiser is 0."""
    P = _problem(y, S, mask, 0.0, centered, norm)
    return psi(-P.grad(torch.zeros_like(P.y[:, 0])), P.levels).abs().amax((-2, -1))


def _batch(B, C, H, W, acc=4, centered=True, norm="ortho", mask_dtype="uint8", first=0):
    from mridc_b200 import synth

    b = synth.make_batch(B, C, H, W, mask_func=synth.Equispaced1DMask([0.08 * 4 / acc], [acc]), centered=centered,
                         normalization=norm, mask_dtype=mask_dtype, first_slice=first)
    return b["y"].cuda(), b["sensitivity_maps"].cuda(), b["mask"].cuda()


def _gaussian_2d_masks(B, H, W, acc, seed=0):
    """Per-slice 2-D variable-density masks [B, 1, H, W, 1] float32 with a fully sampled 16 x 16 centre."""
    g = torch.Generator().manual_seed(seed)
    ky = torch.linspace(-1, 1, H)[:, None]
    kx = torch.linspace(-1, 1, W)[None, :]
    dens = torch.exp(-(ky ** 2 + kx ** 2) / (2 * 0.3 ** 2))
    dens = dens / dens.mean() / acc
    m = (torch.rand(B, H, W, generator=g) < dens).float()
    m[:, H // 2 - 8:H // 2 + 8, W // 2 - 8:W // 2 + 8] = 1
    return m[:, None, :, :, None].cuda()


# ---------------------------------------------------------------------------------------------- per operator
@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 16])
@pytest.mark.parametrize("H,W", SHAPES)
def test_dwt_per_level_against_fp64(H, W, B):
    from mridc_b200 import pics

    g = torch.Generator(device="cuda").manual_seed(H * W + B)
    x = torch.randn(B, H, W, 2, device="cuda", generator=g)
    for levels in range(1, pics.wavelet_levels(H, W) + 1):
        c = pics.dwt(x, levels=levels)
        check_slices("mrbp_dwt %dx%d L=%d" % (H, W, levels), c, _r(psi(_c(x), levels)), OP_TOL)
        back = pics.dwt(c, inverse=True, levels=levels)
        check_slices("mrbp_dwt inverse %dx%d L=%d" % (H, W, levels), back, _r(psi_h(_c(c), levels)), OP_TOL)
        check_slices("mrbp_dwt round trip %dx%d L=%d" % (H, W, levels), back, x, OP_TOL)


@pytest.mark.gpu
def test_dwt_bands_shorter_than_the_filter():
    """16 x 16 at 4 levels: the last bands hold 2 samples and wrap the 8 taps four times."""
    from mridc_b200 import pics

    x = torch.randn(3, 16, 16, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
    for levels in (3, 4):
        c = pics.dwt(x, levels=levels)
        check_slices("mrbp_dwt 16x16 L=%d" % levels, c, _r(psi(_c(x), levels)), OP_TOL)
        check_slices("mrbp_dwt inverse 16x16 L=%d" % levels, pics.dwt(c, True, levels), x, OP_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 16])
@pytest.mark.parametrize("H,W", SHAPES)
def test_step_size_against_fp64(H, W, B):
    from mridc_b200 import pics

    g = torch.Generator(device="cuda").manual_seed(H + W + B)
    S = torch.randn(B, 6, H, W, 2, device="cuda", generator=g) * torch.rand(B, 1, 1, 1, 1, device="cuda", generator=g)
    for mask in (torch.rand(B, 1, H, W, 1, device="cuda", generator=g) * 2,       # per slice, 2-D, float values
                 (torch.rand(1, 1, 1, W, 1, device="cuda", generator=g) < 0.3).to(torch.uint8),
                 torch.ones(1, 1, 1, W, 1, dtype=torch.bool, device="cuda")):
        a = pics.step_size(S, mask)
        ref = _problem(torch.zeros_like(S), S, mask, 0.0).alpha
        check_slices("mrbp_step_size %dx%d B=%d %s" % (H, W, B, mask.dtype), a[:, None], ref[:, None], OP_TOL)


# ---------------------------------------------------------------------------------------------- one step
@pytest.mark.gpu
def test_one_step_from_the_library_state():
    """At the steps producing x_k, k in {1, 10, 50, 100}, of a 15 x 320 x 320 solve: the fp64 step applied to the
    library's (x_{k-1}, z_{k-1}), its gradient and its alpha gives its (x_k, z_k) to 2e-6 per slice."""
    from mridc_b200 import pics

    y, S, mask = _batch(2, 15, 320, 320)
    lam = 0.02 * float(_lam_max(y, S, mask).min())
    P = _problem(y, S, mask, lam)
    alpha = pics.step_size(S, mask).double()
    betas = _betas(100)
    prev = (torch.zeros(2, 320, 320, dtype=torch.complex128, device="cuda"),) * 2
    for k, (x, z, g) in enumerate(pics.fista_iterates(y, S, mask, lam, 100), start=1):
        if k in (1, 10, 50, 100):
            grad = torch.complex(g[:, 2].double(), g[:, 3].double())
            xr, zr = P.step(prev[0], prev[1], betas[k - 1], g=grad, alpha=alpha)
            check_slices("one step k=%d x" % k, x, _r(xr).double(), OP_TOL)
            check_slices("one step k=%d z" % k, z, _r(zr).double(), OP_TOL)
        prev = (_c(x), _c(z))


# ---------------------------------------------------------------------------------------------- free-running solve
def _solve_and_compare(name, y, S, mask, lam_frac=0.02, centered=True, norm="ortho", iters=100):
    """Library vs fp64 FISTA per slice; prints the error at k = 1, 10, 30, 100.  Returns (x_lib, problem)."""
    from mridc_b200 import pics

    lam = lam_frac * float(_lam_max(y, S, mask, centered, norm).min())
    P = _problem(y, S, mask, lam, centered, norm)
    marks = [k for k in (1, 10, 30, 100) if k <= iters] + ([iters] if iters not in (1, 10, 30, 100) else [])
    xr, seen = P.solve(iters, record=marks)
    errs = {}
    for k, (x, _, _) in enumerate(pics.fista_iterates(y, S, mask, lam, iters, centered, norm), start=1):
        if k in marks:
            d = (_c(x) - seen[k]).abs().square().sum((-2, -1)).sqrt()
            errs[k] = (d / seen[k].abs().square().sum((-2, -1)).sqrt()).tolist()
    print("[pics] %-34s rel-L2 per slice at k: %s" % (name, "; ".join(
        "%d: %s" % (k, " ".join("%.1e" % e for e in v)) for k, v in errs.items())))
    check_slices("pics " + name, x, _r(xr).double(), SOLVE_TOL)
    fo, fr = P.objective(_c(x)), P.objective(xr)
    # relative to the minimum, or with lamda = 0 and noiseless data (minimum 0) to the objective at x = 0
    den = fr.abs() if lam > 0 else P.objective(torch.zeros_like(xr))
    rel = ((fo - fr).abs() / den).max().item()
    print("[pics] %-34s relative objective difference %.2e" % (name, rel))
    assert rel <= OBJ_TOL, (name, rel)
    return x, P


SOLVES = {
    "equispaced4x": dict(),
    "equispaced8x": dict(acc=8),
    "gaussian2d_per_slice": dict(mask="gaussian2d"),
    "equispaced4x_uncentred": dict(centered=False),
    "equispaced4x_backward": dict(norm="backward"),
    "equispaced4x_forward": dict(norm="forward"),
    "equispaced4x_none": dict(norm="none"),
    "equispaced4x_bool": dict(mask_dtype="bool"),
    "equispaced4x_float": dict(mask_dtype="float"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(SOLVES))
def test_solve_against_fp64(case):
    o = dict(SOLVES[case])
    centered, norm = o.get("centered", True), o.get("norm", "ortho")
    y, S, mask = _batch(4, 15, 320, 320, o.get("acc", 4), centered, norm, o.get("mask_dtype", "uint8"))
    if o.get("mask") == "gaussian2d":  # the same slices sampled by a different 2-D mask each
        from mridc_b200 import synth
        from test_pics_cpu import fft2

        mask = _gaussian_2d_masks(4, 320, 320, 4)
        x = torch.stack([torch.from_numpy(synth.phantom(320, 320, b)) for b in range(4)]).cuda()
        y = _r(fft2(_c(S) * x[:, None], centered, norm) * mask[..., 0].double())
    _solve_and_compare(case, y, S, mask, centered=centered, norm=norm)


@pytest.mark.gpu
def test_optimality_after_1000_iterations():
    from mridc_b200 import pics

    y, S, mask = _batch(2, 8, 64, 64)
    lam = 0.02 * float(_lam_max(y, S, mask).min())
    P = _problem(y, S, mask, lam)
    xr, _ = P.solve(1000)
    x = pics.l1_wavelet_recon(y, S, mask, lam, 1000)
    rl, rr = P.residual(_c(x)), P.residual(xr)
    print("[pics] fixed-point residual after 1000 iterations: library %s, fp64 %s" % (rl.tolist(), rr.tolist()))
    assert bool((rl <= 2 * rr + 1e-6).all())


# ---------------------------------------------------------------------------------------------- exact cases
@pytest.mark.gpu
def test_above_lambda_max_every_iterate_is_zero():
    from mridc_b200 import pics

    y, S, mask = _batch(2, 15, 320, 320)
    lam = 1.01 * float(_lam_max(y, S, mask).max())
    for x, z, _ in pics.fista_iterates(y, S, mask, lam, 20):
        assert torch.equal(x, torch.zeros_like(x)) and torch.equal(z, torch.zeros_like(z))


@pytest.mark.gpu
def test_zero_maps_or_empty_mask_give_zero():
    from mridc_b200 import pics

    y, S, mask = _batch(2, 8, 64, 64)
    for yy, SS, mm in ((y, torch.zeros_like(S), mask), (torch.zeros_like(y), S, torch.zeros_like(mask))):
        assert bool((pics.step_size(SS, mm) == 0).all())
        x = pics.l1_wavelet_recon(yy, SS, mm, 0.01, 10)
        assert torch.equal(x, torch.zeros_like(x))


@pytest.mark.gpu
def test_lambda_zero_is_least_squares_fista():
    y, S, mask = _batch(4, 15, 320, 320)
    _solve_and_compare("lambda0", y, S, mask, lam_frac=0.0)


# ---------------------------------------------------------------------------------------------- determinism, use
@pytest.mark.gpu
@pytest.mark.parametrize("two_d", [False, True])
def test_deterministic_and_batch_invariant(two_d):
    """Each slice gives the same bits run to run and inside two different batches of 16 (hybrid and three-pass
    gradient)."""
    from mridc_b200 import pics

    y, S, mask = _batch(24, 8, 128, 96)
    if two_d:
        mask = _gaussian_2d_masks(24, 128, 96, 4, seed=1)
        y = (y * mask).contiguous()
    a = pics.l1_wavelet_recon(y[:16], S[:16], mask[:16] if two_d else mask, 0.01, 30)
    b = pics.l1_wavelet_recon(y[:16], S[:16], mask[:16] if two_d else mask, 0.01, 30)
    assert torch.equal(a, b)
    c = pics.l1_wavelet_recon(y[8:], S[8:], mask[8:] if two_d else mask, 0.01, 30)
    assert torch.equal(a[8:], c[:8])


@pytest.mark.gpu
def test_pics_beats_zero_filled_sense_on_noisy_8x_data():
    """synth.make_batch at 8x (equispaced columns, 4 % centre), 15 coils, complex Gaussian noise at 10 % of the rms of
    the sampled k-space.  The truth is the SENSE image of the fully sampled k-space in the units of y.  NMSE: ZF-SENSE
    (mridc_b200.ZF), PICS at lamda = 0 and at the test's lamda, which must beat both."""
    import mridc_b200 as mb
    from mridc_b200 import synth
    from test_pics_cpu import fft2

    b = synth.make_batch(2, 15, 320, 320, mask_func=synth.Equispaced1DMask([0.04], [8]), centered=True,
                         normalization="ortho")
    y, S, mask = _c(b["y"].cuda()), _c(b["sensitivity_maps"].cuda()), b["mask"].cuda()
    k = _c(b["kspace"].cuda())
    M = mask[..., 0].double()
    scale = (M * y.conj() * k).sum((1, 2, 3)).real / (M * y.abs() ** 2).sum((1, 2, 3))  # y = k / scale where sampled
    truth = (S.conj() * fft2(k, True, "ortho", inverse=True)).sum(1) / (S.abs() ** 2).sum(1) / scale[:, None, None]
    g = torch.Generator(device="cuda").manual_seed(3)
    sig = 0.1 * ((M * y.abs() ** 2).sum() / (M.sum() * 15 * 320 * 2)).sqrt()
    noise = torch.complex(torch.randn(y.shape, device="cuda", dtype=torch.float64, generator=g),
                          torch.randn(y.shape, device="cuda", dtype=torch.float64, generator=g)) / math.sqrt(2)
    y = _r(M * (y + sig * noise))
    S = _r(S)

    def nmse(a):
        a = torch.view_as_complex(a.double()) if not a.is_complex() else a.to(torch.complex128)
        return ((a - truth).abs().square().sum() / truth.abs().square().sum()).item()

    lam = LAMBDA_USE * float(_lam_max(y, S, mask).max())
    zf = nmse(mb.ZF(synth.zf_cfg(centered=True, normalization="ortho"))(y, S, mask, truth))
    e0 = nmse(mb.l1_wavelet_recon(y, S, mask, 0.0, 100))
    e = nmse(mb.l1_wavelet_recon(y, S, mask, lam, 100))
    print("[pics] NMSE at 8x with noise: ZF-SENSE %.4f, lambda = 0 %.4f, lambda = %g lambda_max %.4f" % (
        zf, e0, LAMBDA_USE, e))
    assert e < zf and e < e0


LAMBDA_USE = 0.001


# ---------------------------------------------------------------------------------------------- kernels and C-ABI
def test_every_kernel_instantiation_has_a_row():
    from mridc_b200 import pics

    inv = set(library_instantiations(pics.LIB_PATH))
    rows = {kernel_name(n) for want in EXPECTED.values() for n in want}
    print("[pics] instantiations: %s" % sorted(inv))
    assert inv == rows, "library %s, rows %s" % (sorted(inv - rows), sorted(rows - inv))


def _lib():
    from mridc_b200 import _lib as L, pics

    return pics, pics.load(), L


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _dwt_row(B, H, W, levels, inverse):
    n = B * H * W * 2

    def make(seed):
        return {"x": torch.randn(n, device="cuda", generator=_gen(seed))}

    def call(V, st):
        P, lib, L = _lib()
        P.check(lib.mrbp_dwt(L.ptr(V["x"]), L.ptr(V["out"]), inverse, B, H, W, levels, L.ptr(V["ws"]),
                             V["ws"].numel(), st))

    def check(V, X):
        x = _c(X["x"].reshape(B, H, W, 2))
        ref = psi_h(x, levels) if inverse else psi(x, levels)
        check_slices("mrbp_dwt contract", V["out"].reshape(B, H, W, 2), _r(ref).double(), OP_TOL)

    ws = 12 * B * H * W
    return Row({"x": Buf("in", n), "out": Buf("out", n), "ws": Buf("ws", ws, torch.uint8)}, make, call, check)


def _step_row(B, C, H, W, mask_shape, mask_dtype):
    ns = B * C * H * W * 2
    mb_, mh = mask_shape
    nm = mb_ * mh * W

    def make(seed):
        g = _gen(seed)
        m = torch.rand(nm, device="cuda", generator=g) * 3
        m = m.round().to(torch.uint8) if mask_dtype == 0 else m
        return {"S": torch.randn(ns, device="cuda", generator=g), "mask": m}

    def call(V, st):
        P, lib, L = _lib()
        P.check(lib.mrbp_step_size(L.ptr(V["S"]), L.ptr(V["mask"]), mask_dtype, mb_, mh, B, C, H, W, L.ptr(V["alpha"]),
                                   st))

    def check(V, X):
        S = _c(X["S"].reshape(B, C, H, W, 2))
        M = X["mask"].double().reshape(mb_, mh, W)
        ref = Problem(torch.zeros_like(S), S, M, 0.0).alpha
        check_slices("mrbp_step_size contract", V["alpha"][:, None], ref[:, None], OP_TOL)

    bufs = {"S": Buf("in", ns), "mask": Buf("in", nm, torch.uint8 if mask_dtype == 0 else torch.float32),
            "alpha": Buf("out", B)}
    return Row(bufs, make, call, check)


def _fista_row(B, H, W, levels, lamda, beta):
    n = B * H * W * 2
    ng = B * 4 * H * W
    unread = torch.zeros(B, 4, H, W, dtype=torch.bool)
    unread[:, :2] = True  # channels 0-1 of the DC output are never read

    def make(seed):
        g = _gen(seed)
        return {"z": torch.randn(n, device="cuda", generator=g), "x": torch.randn(n, device="cuda", generator=g),
                "grad": torch.randn(ng, device="cuda", generator=g),
                "alpha": torch.rand(B, device="cuda", generator=g) + 0.5}

    def call(V, st):
        P, lib, L = _lib()
        P.check(lib.mrbp_fista_step(L.ptr(V["z"]), L.ptr(V["grad"]), L.ptr(V["alpha"]), lamda, beta, L.ptr(V["x"]), B,
                                    H, W, levels, L.ptr(V["ws"]), V["ws"].numel(), st))

    def check(V, X):
        z, x = _c(X["z"].reshape(B, H, W, 2)), _c(X["x"].reshape(B, H, W, 2))
        gr = X["grad"].reshape(B, 4, H, W).double()
        a = X["alpha"].double()[:, None, None]
        c = psi(z - a * torch.complex(gr[:, 2], gr[:, 3]), levels)
        xn = psi_h(torch.where(c.abs() > a * lamda, c * (1 - a * lamda / c.abs().clamp_min(1e-300)), 0 * c), levels)
        zn = xn + beta * (xn - x)
        check_slices("mrbp_fista_step contract x", V["x"].reshape(B, H, W, 2), _r(xn).double(), OP_TOL)
        check_slices("mrbp_fista_step contract z", V["z"].reshape(B, H, W, 2), _r(zn).double(), OP_TOL)

    bufs = {"z": Buf("inout", n), "x": Buf("inout", n), "grad": Buf("in", ng, unread=unread), "alpha": Buf("in", B),
            "ws": Buf("ws", 12 * B * H * W, torch.uint8)}
    return Row(bufs, make, call, check)


ROWS = {
    "dwt_forward": (("mrbp_dwt",), lambda: _dwt_row(2, 48, 40, 3, 0)),
    "dwt_inverse_wrapping": (("mrbp_dwt",), lambda: _dwt_row(2, 16, 24, 3, 1)),
    "step_size_uint8_1d": (("mrbp_step_size",), lambda: _step_row(3, 5, 20, 36, (1, 1), 0)),
    "step_size_float_2d_per_slice": (("mrbp_step_size",), lambda: _step_row(3, 5, 20, 36, (3, 20), 1)),
    "fista_step_3_levels": (("mrbp_fista_step",), lambda: _fista_row(2, 64, 48, 3, 0.3, 0.6)),
    "fista_step_1_level": (("mrbp_fista_step",), lambda: _fista_row(3, 14, 18, 1, 0.5, 0.0)),
}


def test_header_symbols_have_contract_rows():
    from test_pics_cpu import declared

    rows = {s for syms, _ in ROWS.values() for s in syms}
    host = {"mrbp_last_error", "mrbp_version", "mrbp_levels", "mrbp_workspace_bytes"}
    assert sorted(rows | host) == declared()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ROWS))
def test_contract(name):
    run_contract(ROWS[name][1]())


# ---------------------------------------------------------------------------------------------- the model
@pytest.mark.gpu
def test_model_forward_equals_the_solver_and_never_synchronises():
    import mridc_b200 as mb
    from mridc_b200 import pics, synth

    b = synth.make_batch(2, 8, 96, 80, centered=True, normalization="ortho")
    y, S, mask = b["y"].cuda(), b["sensitivity_maps"].cuda(), b["mask"].cuda()
    target = b["target"][:, 8:-8, 4:-4].cuda()
    cfg = dict(reg_wt=0.005, num_iters=25, fft_centered=True, fft_normalization="ortho", spatial_dims=[-2, -1],
               coil_dim=1)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        x = pics.l1_wavelet_recon(y, S, mask, 0.005, 25)
        out = mb.PICS(cfg)(y, S, mask, None, target)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert out.shape == target.shape and out.dtype == torch.complex64
    assert torch.equal(torch.view_as_real(out), x[:, 8:-8, 4:-4])
