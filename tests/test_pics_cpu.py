"""PICS (mridc_b200.pics) without a GPU: the db4 taps, the level rule, the fp64 reference of Psi and of FISTA that
tests/test_gpu_pics.py holds the library to, and the C-ABI table.

The reference runs in float64 torch on whatever device its inputs live on.  Psi is built from 1-D periodised analysis
matrices (a[k] = sum_j h[j] v[(2k + j) mod n]) applied along H and W level by level in the Mallat layout of
include/mridc_b200_pics.h; Psi^H applies their transposes.  A dense matrix assembled from the periodised filters (the
aliases h[i - 2k + m n] summed) checks it independently.
"""
import ctypes
import math
import os
import re

import pytest
import torch

from conftest import ROOT

NORM_SCALE = {"backward": lambda n: math.sqrt(n), "none": lambda n: math.sqrt(n), "ortho": lambda n: 1.0,
              "forward": lambda n: 1.0 / math.sqrt(n)}


# ---------------------------------------------------------------------------------------------- fp64 reference
def db4(device="cpu"):
    from mridc_b200 import pics

    h = torch.tensor(pics.DB4_LO, dtype=torch.float64, device=device)
    g = torch.tensor([(-1) ** j for j in range(8)], dtype=torch.float64, device=device) * h.flip(0)
    return h, g


def analysis_matrices(n, device="cpu"):
    """(lo, hi) [n/2, n]: one periodic level along a line of n samples."""
    h, g = db4(device)
    k = torch.arange(n // 2, device=device)
    lo = torch.zeros(n // 2, n, dtype=torch.float64, device=device)
    hi = torch.zeros_like(lo)
    for j in range(8):
        lo.index_put_((k, (2 * k + j) % n), h[j].expand(n // 2), accumulate=True)
        hi.index_put_((k, (2 * k + j) % n), g[j].expand(n // 2), accumulate=True)
    return lo, hi


def psi(x, levels):
    """Psi x for complex x [..., H, W] (Mallat layout)."""
    out = x.clone()
    band = x
    H, W = x.shape[-2:]
    for l in range(levels):
        h, w = H >> l, W >> l
        lo_h, hi_h = (m.to(x.dtype) for m in analysis_matrices(h, x.device))
        lo_w, hi_w = (m.to(x.dtype) for m in analysis_matrices(w, x.device))
        Lx, Hx = band @ lo_w.T, band @ hi_w.T
        h2, w2 = h // 2, w // 2
        out[..., :h2, w2:w] = lo_h @ Hx
        out[..., h2:h, :w2] = hi_h @ Lx
        out[..., h2:h, w2:w] = hi_h @ Hx
        band = lo_h @ Lx
        out[..., :h2, :w2] = band
    return out


def psi_h(c, levels):
    """Psi^H c (the inverse of psi: Psi is orthonormal)."""
    H, W = c.shape[-2:]
    band = c[..., :H >> levels, :W >> levels]
    for l in range(levels - 1, -1, -1):
        h, w = H >> l, W >> l
        h2, w2 = h // 2, w // 2
        lo_h, hi_h = (m.to(c.dtype) for m in analysis_matrices(h, c.device))
        lo_w, hi_w = (m.to(c.dtype) for m in analysis_matrices(w, c.device))
        Lx = lo_h.T @ band + hi_h.T @ c[..., h2:h, :w2]
        Hx = lo_h.T @ c[..., :h2, w2:w] + hi_h.T @ c[..., h2:h, w2:w]
        band = Lx @ lo_w + Hx @ hi_w
    return band


def soft(c, t):
    """c * max(0, 1 - t / |c|); t broadcast against c."""
    a = c.abs()
    return torch.where(a > t, c * ((a - t) / a.clamp_min(1e-300)), torch.zeros_like(c))


def fft2(x, centered, norm, inverse=False):
    nm = "backward" if norm in ("backward", "none") else norm
    if centered:
        x = torch.fft.ifftshift(x, dim=(-2, -1))
    x = (torch.fft.ifft2 if inverse else torch.fft.fft2)(x, norm=nm)
    if centered:
        x = torch.fft.fftshift(x, dim=(-2, -1))
    return x


class Problem:
    """One batch of PICS problems in fp64: y, S [B, C, H, W] complex128, M [B|1, H|1, W] float64 (the mask value
    multiplies, as in the DC operator)."""

    def __init__(self, y, S, M, lamda, centered=True, norm="ortho"):
        self.y, self.S, self.M, self.lamda, self.centered, self.norm = y, S, M, float(lamda), centered, norm
        self.levels = wavelet_levels(*y.shape[-2:])
        s2 = (S.abs() ** 2).sum(1).amax((-2, -1))
        bound = s2 * M.abs().amax((-2, -1)).expand(s2.shape)
        self.alpha = torch.where(bound > 0, 1.0 / bound.clamp_min(1e-300), torch.zeros_like(bound))

    def grad(self, x):
        r = self.M[:, None] * (fft2(self.S * x[:, None], self.centered, self.norm) - self.y)
        return (self.S.conj() * fft2(r, self.centered, self.norm, inverse=True)).sum(1)

    def prox(self, v, alpha=None):
        a = (self.alpha if alpha is None else alpha)[:, None, None]
        return psi_h(soft(psi(v, self.levels), a * self.lamda), self.levels)

    def step(self, x, z, beta, g=None, alpha=None):
        """One FISTA step from (x_k, z_k) -> (x_{k+1}, z_{k+1}); g defaults to the fp64 gradient at z."""
        a = (self.alpha if alpha is None else alpha)[:, None, None]
        xn = self.prox(z - a * (self.grad(z) if g is None else g), alpha)
        return xn, xn + beta * (xn - x)

    def objective(self, x):
        """Per slice: 1/2 sum M |U(S x) - y / s|^2 + lamda |Psi x|_1, U the unitary DFT, fft2 = s U."""
        H, W = x.shape[-2:]
        s = NORM_SCALE[self.norm](H * W)
        r = fft2(self.S * x[:, None], self.centered, self.norm) - self.y
        data = 0.5 * (self.M[:, None] * r.abs() ** 2).sum((1, 2, 3)) / s ** 2
        return data + self.lamda * psi(x, self.levels).abs().sum((-2, -1))

    def residual(self, x):
        """Fixed-point residual |x - prox(x - alpha grad f(x))| / |x| per slice."""
        d = x - self.prox(x - self.alpha[:, None, None] * self.grad(x))
        return d.abs().square().sum((-2, -1)).sqrt() / x.abs().square().sum((-2, -1)).sqrt()

    def solve(self, iters, record=()):
        """FISTA from zero -> (x_iters, {k: x_k for k in record})."""
        x = torch.zeros_like(self.y[:, 0])
        z, t, seen = x, 1.0, {}
        for k in range(1, iters + 1):
            tn = (1 + math.sqrt(1 + 4 * t * t)) / 2
            x, z = self.step(x, z, (t - 1) / tn)
            t = tn
            if k in record:
                seen[k] = x.clone()
        return x, seen


def wavelet_levels(H, W):
    from mridc_b200 import pics

    return pics.wavelet_levels(H, W)


# ---------------------------------------------------------------------------------------------- taps and levels
def test_db4_taps():
    h, g = db4()
    assert abs(h.sum().item() - math.sqrt(2)) < 1e-15
    assert abs(h.square().sum().item() - 1) < 1e-15
    for m in (1, 2, 3):
        assert abs((h[:8 - 2 * m] * h[2 * m:]).sum().item()) < 1e-15, m
    j = torch.arange(8, dtype=torch.float64)
    for p in range(4):
        assert abs((g * j ** p).sum().item()) < 1e-13, p
    assert abs(g.square().sum().item() - 1) < 1e-15 and abs((h * g).sum().item()) < 1e-15


def test_library_holds_the_same_taps():
    from mridc_b200 import pics

    src = open(os.path.join(ROOT, "mridc_b200", "csrc", "pics.cu")).read()
    taps = [float(v) for v in re.findall(r"#define DB4_H\d (\S+)", src)]
    assert taps == list(pics.DB4_LO)


@pytest.mark.parametrize("H,W,L", [(320, 320, 5), (640, 320, 5), (232, 288, 3), (14, 14, 1), (18, 16, 1),
                                   (16, 16, 1), (28, 28, 2), (448, 448, 6)])
def test_levels(H, W, L):
    assert wavelet_levels(H, W) == L


@pytest.mark.parametrize("H,W", [(321, 320), (320, 321), (13, 14), (12, 12), (14, 13), (1, 1)])
def test_no_level_raises(H, W):
    with pytest.raises(ValueError):
        wavelet_levels(H, W)


# ---------------------------------------------------------------------------------------------- the reference Psi
@pytest.mark.parametrize("H,W", [(320, 320), (640, 320), (232, 288), (14, 14), (18, 16)])
def test_psi_is_orthonormal(H, W):
    g = torch.Generator().manual_seed(H + W)
    x = torch.randn(2, H, W, dtype=torch.complex128, generator=g)
    L = wavelet_levels(H, W)
    c = psi(x, L)
    back = psi_h(c, L)
    err = ((back - x).abs().norm() / x.abs().norm()).item()
    par = abs(c.abs().norm().item() / x.abs().norm().item() - 1)
    print("%dx%d L=%d: reconstruction %.1e, Parseval %.1e" % (H, W, L, err, par))
    assert err < 1e-13 and par < 1e-13


def dense_psi(H, W, levels):
    """Psi as an explicit [HW, HW] matrix from the periodised filters (aliases h[i - 2k + m n] summed)."""
    h, g = db4()

    def per(f, n):
        A = torch.zeros(n // 2, n, dtype=torch.float64)
        for k in range(n // 2):
            for i in range(n):
                A[k, i] = sum(f[d].item() for d in range(8) if (d - (i - 2 * k)) % n == 0)
        return A

    M = torch.eye(H * W, dtype=torch.float64)
    for l in range(levels):
        hb, wb = H >> l, W >> l
        Ah = torch.cat([per(h, hb), per(g, hb)])  # rows: low then high along H
        Aw = torch.cat([per(h, wb), per(g, wb)])
        step = torch.eye(H * W, dtype=torch.float64)
        idx = torch.tensor([r * W + c for r in range(hb) for c in range(wb)])
        step[idx[:, None], idx[None, :]] = torch.kron(Ah, Aw)
        M = step @ M
    return M


@pytest.mark.parametrize("levels", [1, 2, 3, 4])
def test_psi_against_a_dense_matrix(levels):
    """16 x 16: from level 3 the bands (4 and 2 samples) are shorter than the filter and wrap more than once."""
    H = W = 16
    D = dense_psi(H, W, levels)
    assert (D @ D.T - torch.eye(H * W, dtype=torch.float64)).abs().max() < 1e-13
    g = torch.Generator().manual_seed(levels)
    x = torch.randn(H, W, dtype=torch.complex128, generator=g)
    ref = (D.to(x.dtype) @ x.reshape(-1)).reshape(H, W)
    assert (psi(x, levels) - ref).abs().max() < 1e-13
    assert (psi_h(ref, levels) - x).abs().max() < 1e-13


# ---------------------------------------------------------------------------------------------- the reference FISTA
def tiny_problem(lamda_frac=0.05, C=4, H=32, W=32, seed=0):
    from mridc_b200 import synth

    S = torch.from_numpy(synth.coil_maps(C, H, W))[None]
    x = torch.from_numpy(synth.phantom(H, W, 1))[None]
    g = torch.Generator().manual_seed(seed)
    M = torch.zeros(1, 1, W, dtype=torch.float64)
    M[..., ::2] = 1
    M[..., W // 2 - 2:W // 2 + 2] = 1
    y = M[:, None] * (fft2(S * x[:, None], True, "ortho")
                      + 0.01 * torch.randn(1, C, H, W, dtype=torch.complex128, generator=g))
    P = Problem(y, S, M, 0.0)
    lam_max = psi(-P.grad(torch.zeros_like(x)), P.levels).abs().max().item()
    return Problem(y, S, M, lamda_frac * lam_max), x


def test_reference_fista_reaches_a_fixed_point():
    """4 coils, 32 x 32, a 2x column mask with noise: 100 iterations drive the fixed-point residual below 1e-8 (1e-12
    measured), and the objective does not rise from iteration 50 on."""
    P, _ = tiny_problem()
    x, seen = P.solve(100, record=(10, 50))
    res = P.residual(x).item()
    objs = [P.objective(seen[k]).item() for k in (10, 50)] + [P.objective(x).item()]
    print("fixed-point residual after 100 iterations: %.2e; objective at 10, 50, 100: %s" % (res, objs))
    assert res < 1e-8
    assert objs[2] <= objs[1] * (1 + 1e-14) and objs[1] <= objs[0]


def test_reference_exact_cases():
    """Above lamda_max = max |Psi E^H y| the minimiser is 0 and FISTA never leaves it; lamda = 0 is least squares."""
    P, _ = tiny_problem()
    lam_max = P.lamda / 0.05
    Z = Problem(P.y, P.S, P.M, 1.01 * lam_max)
    x, _ = Z.solve(20)
    assert torch.equal(x, torch.zeros_like(x))
    Q = Problem(P.y, P.S, P.M, 0.0)
    x, _ = Q.solve(400)
    assert (Q.grad(x).abs().norm() / Q.grad(torch.zeros_like(x)).abs().norm()).item() < 1e-3


def test_objective_gradient_agree_for_every_normalization():
    """The objective's derivative along a random direction is Re <grad, d> under every normalization."""
    P, _ = tiny_problem()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, 32, 32, dtype=torch.complex128, generator=g)
    d = torch.randn(1, 32, 32, dtype=torch.complex128, generator=g)
    for norm in ("ortho", "backward", "forward", "none"):
        s = NORM_SCALE[norm](32 * 32)
        Q = Problem(P.y * s, P.S, P.M, 0.0, norm=norm)
        eps = 1e-6
        num = (Q.objective(x + eps * d) - Q.objective(x - eps * d)).item() / (2 * eps)
        ana = (Q.grad(x).conj() * d).real.sum().item()
        assert abs(num - ana) < 1e-6 * abs(ana), (norm, num, ana)


# ---------------------------------------------------------------------------------------------- the C-ABI table
def declared():
    src = open(os.path.join(ROOT, "include", "mridc_b200_pics.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mrbp_[a-z0-9_]+)\s*\(", src)))


def test_signatures_match_the_header():
    from mridc_b200 import pics

    names = declared()
    lib = ctypes.CDLL(pics.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "symbol %s declared in the header but not exported" % n
    assert sorted(pics.SIGNATURES) == names
    assert pics.load().mrbp_version() >= 100
    assert pics.load().mrbp_workspace_bytes(2, 320, 320) == 12 * 2 * 320 * 320


def test_argument_errors_before_any_cuda_call():
    from mridc_b200 import pics

    lib = pics.load()
    p = ctypes.c_void_p(16)  # never dereferenced: every call below fails its argument check first
    n = lib.mrbp_workspace_bytes(1, 64, 64)
    cases = [
        (lambda: lib.mrbp_dwt(None, p, 0, 1, 64, 64, 2, p, n, None), -1, b"null"),
        (lambda: lib.mrbp_dwt(p, p, 0, 1, 64, 64, 2, p, n, None), -1, b"distinct"),
        (lambda: lib.mrbp_dwt(p, ctypes.c_void_p(32), 0, 1, 64, 64, 7, p, n, None), -1, b"7 levels"),
        (lambda: lib.mrbp_dwt(p, ctypes.c_void_p(32), 0, 1, 64, 64, 0, p, n, None), -1, b"0 levels"),
        (lambda: lib.mrbp_dwt(p, ctypes.c_void_p(32), 0, 1, 64, 64, 2, p, n - 1, None), -1, b"workspace"),
        (lambda: lib.mrbp_fista_step(p, p, p, -1.0, 0.0, p, 1, 64, 64, 2, p, n, None), -1, b"lamda"),
        (lambda: lib.mrbp_fista_step(p, p, p, 1.0, 0.0, p, 0, 64, 64, 2, p, n, None), -1, b"bad shape"),
        (lambda: lib.mrbp_fista_step(p, p, p, 1.0, 0.0, p, 70000, 64, 64, 2, p, 1 << 62, None), -2, b"batch"),
        (lambda: lib.mrbp_step_size(p, p, 2, 1, 1, 1, 4, 64, 64, p, None), -1, b"mask_dtype"),
        (lambda: lib.mrbp_step_size(p, p, 0, 3, 1, 2, 4, 64, 64, p, None), -1, b"broadcast"),
        (lambda: lib.mrbp_levels(0, 64), -1, b"bad size"),
    ]
    for call, want, msg in cases:
        rc = call()
        err = lib.mrbp_last_error() if rc < 0 else b""
        assert rc == want and msg in err, (rc, want, err)


def test_python_validation_without_a_gpu():
    import mridc_b200 as mb

    y = torch.zeros(1, 4, 32, 32, 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mb.l1_wavelet_recon(y, y, torch.ones(1, 1, 1, 32, 1), 0.1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mb.PICS(dict(reg_wt=0.1, num_iters=10, fft_centered=True, fft_normalization="ortho", spatial_dims=[-2, -1],
                     coil_dim=1))(y, y, torch.ones(1, 1, 1, 32, 1), None, None)
