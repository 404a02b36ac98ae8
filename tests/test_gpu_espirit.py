"""ESPIRiT coil sensitivity maps (mridc_b200.espirit_maps, libmridc_b200_espirit.so) against an fp64 reference.

The reference below restates the eight steps of sigpy's EspiritCalib (one map set) in float64 torch: the calibration
matrix A of the kw x kw windows of the centred cw x cw ACS block, its SVD, K = #{sigma_i > threshold * sigma_max}, the
kernels w_i = conj(v_i) (the rows of V^H), G(r) = (1/kw^2) sum_i a_i a_i^H with a_i(r)_c = sum_{p,q} w_i[c,p,q]
exp(+2 pi i (p n_y/H + q n_x/W)), n = r - (H//2, W//2), and max_iter power iterations from x = 1 with the phase of
coil 0 removed and the maps cropped where lambda <= crop.  G is evaluated through the autocorrelation taps of the w_i
placed on the zero-padded grid the library uses and one inverse transform; a CPU test checks that route against a
direct evaluation of a_i.  The conventions (the conj of step 3, the sign of the DFT) are pinned by the correlation of
the maps with the true maps of synth.coil_maps: 0.999 with the right ones, far less with either flipped.

Tolerance of the GPU comparison.  The library computes A^H A and the taps in fp64 (like the reference) and the rest in
fp32: the taps are rounded once to fp32 (u = 2^-24 = 6e-8 relative), the inverse 2-D transform adds the 2e-6 per-operator
contract of the FFT (measured 1e-7 to 4e-7 rms at these lengths), and each power iteration rounds a C-term dot product
(~u * sqrt(C) <= 3.4e-7 at 32 coils).  Errors along the dominant eigenvector are normalised away; those across it are
damped by lambda_2 / lambda_1 per iteration, so they settle at about (|dG| + u sqrt(C)) / (1 - lambda_2 / lambda_1).  On
the support lambda_1 >= 0.99 and lambda_2 <= 0.32 (eigengap >= 0.67), which gives 1e-6 to 3e-6; pixels outside the object
with a smaller gap carry more.  The maps and lambda are held to TOL = 2e-5 rel-L2 per slice, over the pixels whose crop
decision is fixed (|lambda_ref - crop| > 1e-4) and, for the maps, whose coil-0 magnitude |x_0| >= 1e-3 (the phase
normalisation divides by it).  The projector x x^H, free of that phase, is compared over every pixel of fixed crop
decision to the same tolerance.
"""
import ctypes
import gc
import os
import re

import numpy as np
import pytest
import torch

from test_gpu_abi_contract import Buf, Row, run_contract
from test_gpu_bench_shapes import check_slices
from test_gpu_kernel_paths import kernel_name, launched, library_instantiations

from conftest import ROOT, rel_l2

TOL = 2e-5
CROP_BAND = 1e-4
X0_MIN = 1e-3
ESP = "mrb::espirit::"
# row -> kernels it must launch (the CPU inventory test compares the union with the instantiations of the library)
EXPECTED = {
    "pipeline_c16": {ESP + "calib_gram_kernel", ESP + "kernel_taps_kernel", ESP + "power_maps_kernel<16>"},
    "pipeline_c32": {ESP + "calib_gram_kernel", ESP + "kernel_taps_kernel", ESP + "power_maps_kernel<32>"},
}


@pytest.fixture(autouse=True)
def _release_gpu_memory():
    """The B200 machines are shared: hand the cached blocks of each test back to the driver."""
    yield
    gc.collect()
    if torch.cuda.is_available() and torch.cuda.is_initialized():
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- fp64 reference
def _complex(y):
    """[..., 2] real -> complex128."""
    return torch.view_as_complex(y.double().contiguous())


def calib_matrix(yc, cw, kw):
    """yc [C, H, W] complex, centred -> A [(cw-kw+1)^2, C*kw*kw], columns (c, p, q) row-major."""
    C, H, W = yc.shape
    y0, x0 = H // 2 - cw // 2, W // 2 - cw // 2
    acs = yc[:, y0:y0 + cw, x0:x0 + cw]
    n = cw - kw + 1
    win = acs.unfold(1, kw, 1).unfold(2, kw, 1)  # [C, n, n, kw, kw]
    return win.permute(1, 2, 0, 3, 4).reshape(n * n, C * kw * kw)


def kernels(yc, cw, kw, threshold, conj=True):
    """-> (w [K, C, kw, kw] complex128, K, sigma).  w_i = conj(v_i), the rows of V^H (conj=False: v_i)."""
    C = yc.shape[0]
    _, s, vh = torch.linalg.svd(calib_matrix(yc, cw, kw), full_matrices=False)
    K = int((s > threshold * s[0]).sum())
    w = vh[:K] if conj else vh[:K].conj().resolve_conj()
    return w.reshape(K, C, kw, kw), K, s


def taps(w):
    """T [C, C, L, L] (L = 2kw-1): T_cd(dy, dx) = (1/kw^2) sum_i sum_{p-p'=dy, q-q'=dx} w_i[c,p,q] conj(w_i[d,p',q']),
    lag dy at index dy mod L (a zero-padded cross-correlation, exact at this length)."""
    K, C, kw, _ = w.shape
    L = 2 * kw - 1
    if K == 0:
        return torch.zeros(C, C, L, L, dtype=w.dtype, device=w.device)
    wp = torch.zeros(K, C, L, L, dtype=w.dtype, device=w.device)
    wp[..., :kw, :kw] = w
    f = torch.fft.fft2(wp)
    return torch.fft.ifft2(torch.einsum("icab,idab->cdab", f, f.conj())) / kw ** 2


def G_from_taps(w, H, W, sign=1):
    """G [H, W, C, C] at the centred pixels: the taps placed at ((dy + H//2) mod H, (dx + W//2) mod W) (the library's
    centred layout, lags that alias added), G = H*W * fftshift(ifft2(ifftshift(grid))).  sign=-1 flips the DFT sign."""
    T = taps(w)
    C, L, kw = T.shape[0], T.shape[-1], w.shape[-1]
    lag = torch.arange(L, device=w.device)
    lag = torch.where(lag < kw, lag, lag - L) * sign
    iy, ix = (lag + H // 2) % H, (lag + W // 2) % W
    grid = torch.zeros(C, C, H, W, dtype=T.dtype, device=T.device)
    grid.permute(2, 3, 0, 1).index_put_((iy[:, None].expand(L, L), ix[None, :].expand(L, L)), T.permute(2, 3, 0, 1),
                                        accumulate=True)
    G = torch.fft.fftshift(torch.fft.ifft2(torch.fft.ifftshift(grid, dim=(-2, -1))), dim=(-2, -1)) * (H * W)
    return G.permute(2, 3, 0, 1)


def G_brute(w, H, W):
    """Step 4 and 5 evaluated directly: a_i(r)_c = sum_{p,q} w_i[c,p,q] exp(+2 pi i (p n_y/H + q n_x/W))."""
    K, C, kw, _ = w.shape
    ny = torch.arange(H, dtype=torch.float64, device=w.device) - H // 2
    nx = torch.arange(W, dtype=torch.float64, device=w.device) - W // 2
    p = torch.arange(kw, dtype=torch.float64, device=w.device)
    ey = torch.exp(2j * np.pi * ny[:, None] * p[None] / H)
    ex = torch.exp(2j * np.pi * nx[:, None] * p[None] / W)
    a = torch.einsum("yp,xq,icpq->yxic", ey, ex, w)  # [H, W, K, C]
    return torch.einsum("yxic,yxid->yxcd", a, a.conj()) / kw ** 2


def power(G, max_iter, crop):
    """Steps 6-8 on G [H, W, C, C] -> (maps [C, H, W], lam [H, W])."""
    H, W, C, _ = G.shape
    x = torch.ones(H, W, C, 1, dtype=G.dtype, device=G.device)
    lam = torch.zeros(H, W, dtype=torch.float64, device=G.device)
    for _ in range(max_iter):
        yv = G @ x
        lam = yv.abs().square().sum((-2, -1)).sqrt()
        x = torch.where(lam[..., None, None] > 0, yv / lam.clamp_min(1e-300)[..., None, None], torch.zeros_like(yv))
    x = x[..., 0]
    x0 = x[..., :1]
    ph = torch.where(x0.abs() > 0, x0.conj() / x0.abs().clamp_min(1e-300), torch.ones_like(x0))
    x = x * ph
    x = torch.where((lam > crop)[..., None], x, torch.zeros_like(x))
    return x.permute(2, 0, 1), lam


def espirit_ref(y, cw=24, kw=6, threshold=0.02, crop=0.95, max_iter=100, centered=True, conj=True, sign=1):
    """One slice y [C, H, W, 2] (any device) -> dict(maps [C, H, W] complex128, lam [H, W], K, sigma), in fp64."""
    yc = _complex(y)
    C, H, W = yc.shape
    if not centered:
        yc = torch.fft.fftshift(yc, dim=(-2, -1))
    w, K, s = kernels(yc, cw, kw, threshold, conj)
    maps, lam = power(G_from_taps(w, H, W, sign), max_iter, crop)
    if not centered:
        maps, lam = torch.fft.ifftshift(maps, dim=(-2, -1)), torch.fft.ifftshift(lam, dim=(-2, -1))
    return {"maps": maps, "lam": lam, "K": K, "sigma": s}


def support(H, W):
    from mridc_b200 import synth

    img = np.abs(synth.phantom(H, W, 0))
    return torch.from_numpy(img > 0.1 * img.max())


def true_correlation(maps, C, H, W):
    """|<s_est, s_true>| per pixel against synth.coil_maps (unit-norm over coils)."""
    from mridc_b200 import synth

    S = torch.from_numpy(synth.coil_maps(C, H, W)).to(maps.device)
    return (maps.conj() * S).sum(0).abs()


# ---------------------------------------------------------------------------------------------- CPU: the reference
@pytest.mark.parametrize("C,H,W,cw,kw", [(3, 12, 10, 8, 3), (2, 5, 7, 5, 4)])
def test_tap_route_equals_direct_evaluation(C, H, W, cw, kw):
    """The tap placement (centred grid, aliasing lags added when 2kw-1 > H or W) and one inverse transform give the G(r)
    of the direct evaluation of step 4; a misplaced tap, a wrong centring or a flipped sign breaks the equality."""
    g = torch.Generator().manual_seed(C * H)
    yc = torch.randn(C, H, W, dtype=torch.complex128, generator=g)
    w, K, _ = kernels(yc, cw, kw, 0.3)  # a threshold that keeps part of the subspace (all of it gives G = I)
    ref = G_brute(w, H, W)
    assert 0 < K < C * kw * kw
    assert rel_l2(G_from_taps(w, H, W), ref) < 1e-12
    assert rel_l2(G_from_taps(w, H, W, sign=-1), ref) > 1e-2
    # G is Hermitian, PSD, with eigenvalues <= 1 (w_i orthonormal)
    assert rel_l2(ref, ref.mH.resolve_conj()) < 1e-14
    ev = torch.linalg.eigvalsh(ref)
    assert ev.min() > -1e-12 and ev.max() < 1 + 1e-12


def test_conventions_against_the_true_maps():
    """8 coils, 96 x 80, fully sampled: K = 43, |<s_est, s_true>| >= 0.999 on the phantom support with the right
    conventions, well below without the conj of step 3 or with the DFT sign flipped."""
    from mridc_b200 import synth

    C, H, W = 8, 96, 80
    k = synth.make_batch(1, C, H, W, centered=True, normalization="ortho")["kspace"][0]
    sup = support(H, W)
    r = espirit_ref(k)
    corr = true_correlation(r["maps"], C, H, W)[sup]
    s = r["sigma"] / r["sigma"][0]
    print("K = %d, sigma_K/sigma_1 = %.4f, sigma_K+1/sigma_1 = %.4f; |<s,s_true>| min %.5f median %.5f; lambda on support "
          "%.4f..%.4f" % (r["K"], s[r["K"] - 1], s[r["K"]], corr.min(), corr.median(), r["lam"][sup].min(),
                           r["lam"][sup].max()))
    assert r["K"] == 43
    assert corr.min() >= 0.999 and corr.median() > 0.9999
    assert r["lam"][sup].min() > 0.99
    for tag, kw in (("no conj", dict(conj=False)), ("flipped sign", dict(sign=-1))):
        bad = true_correlation(espirit_ref(k, **kw)["maps"], C, H, W)[sup]
        print("%s: |<s,s_true>| min %.4f median %.4f" % (tag, bad.min(), bad.median()))
        assert bad.min() < 0.97, tag


# ---------------------------------------------------------------------------------------------- CPU: the library
def _declared():
    src = open(os.path.join(ROOT, "include", "mridc_b200_espirit.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mrbe_[a-z0-9_]+)\s*\(", src)))


NON_LAUNCHING = {"mrbe_last_error": "host-side error message", "mrbe_version": "host-side constant"}


def test_header_ctypes_table_and_contract_rows_agree():
    from mridc_b200 import espirit

    names = _declared()
    lib = ctypes.CDLL(espirit.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "symbol %s declared in the header but not exported" % n
    assert sorted(espirit.SIGNATURES) == names, "ctypes signature table out of sync with the header"
    rows = {s for syms, _ in ROWS.values() for s in syms}
    assert not rows & set(NON_LAUNCHING)
    assert sorted(rows | set(NON_LAUNCHING)) == names, "entry points without a contract row: %s" % sorted(
        set(names) - rows - set(NON_LAUNCHING))
    assert espirit.load().mrbe_version() >= 100


def test_every_kernel_instantiation_has_a_row():
    from mridc_b200 import espirit

    inv = set(library_instantiations(espirit.LIB_PATH))
    rows = {kernel_name(n) for want in EXPECTED.values() for n in want}
    print("[espirit] instantiations: %s" % sorted(inv))
    assert inv == rows, "library %s, rows %s" % (sorted(inv - rows), sorted(rows - inv))


def test_argument_errors_before_any_cuda_call():
    from mridc_b200 import espirit

    lib = espirit.load()
    p = ctypes.c_void_p(16)  # never dereferenced: every call below fails its argument check first
    cases = [
        (lambda: lib.mrbe_calib_gram(None, p, 1, 8, 64, 64, 24, 6, 1, None), -1, b"null"),
        (lambda: lib.mrbe_calib_gram(p, p, 1, 33, 64, 64, 24, 6, 1, None), -2, b"33 coils"),
        (lambda: lib.mrbe_calib_gram(p, p, 1, 8, 64, 64, 5, 6, 1, None), -1, b"calibration width 5"),
        (lambda: lib.mrbe_calib_gram(p, p, 1, 8, 64, 20, 24, 6, 1, None), -1, b"calibration width 24"),
        (lambda: lib.mrbe_calib_gram(p, p, 1, 8, 200, 200, 120, 6, 1, None), -2, b"calibration width 120"),
        (lambda: lib.mrbe_calib_gram(p, p, 1, 32, 64, 64, 24, 9, 1, None), -2, b"C*kw*kw"),
        (lambda: lib.mrbe_calib_gram(p, p, 0, 8, 64, 64, 24, 6, 1, None), -1, b"bad shape"),
        (lambda: lib.mrbe_kernel_taps(p, None, p, 1, 8, 64, 64, 6, 1, None), -1, b"null"),
        (lambda: lib.mrbe_kernel_taps(p, p, p, 1, 8, 64, 64, 0, 1, None), -1, b"kernel width 0"),
        (lambda: lib.mrbe_power_maps(p, p, None, 1, 8, 64, 64, 100, 0.95, None), -1, b"null"),
        (lambda: lib.mrbe_power_maps(p, p, p, 1, 8, 64, 64, 0, 0.95, None), -1, b"max_iter 0"),
        (lambda: lib.mrbe_power_maps(p, p, p, 1, 40, 64, 64, 10, 0.95, None), -2, b"40 coils"),
    ]
    for call, want, msg in cases:
        rc = call()
        err = lib.mrbe_last_error() if rc else b""
        assert rc == want and msg in err, (rc, want, err)
    with pytest.raises(NotImplementedError, match=r"C\*kw\*kw"):
        espirit.check(lib.mrbe_calib_gram(p, p, 1, 32, 64, 64, 24, 9, 1, None))


def test_python_validation_without_a_gpu():
    import mridc_b200 as mb

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mb.espirit_maps(torch.zeros(1, 4, 32, 32, 2))


# ---------------------------------------------------------------------------------------------- GPU: end to end
def _kspace(B, C, H, W, centered=True, masked=False):
    from mridc_b200 import synth

    if masked:
        b = synth.make_batch(B, C, H, W, mask_func=synth.Equispaced1DMask([0.08], [4]), centered=centered,
                             normalization="ortho")
        return b["y"]
    return synth.make_batch(B, C, H, W, centered=centered, normalization="ortho")["kspace"]


def _compare(name, y, maps, lam, centered=True, cw=24, kw=6):
    """Per slice against espirit_ref; returns the reference maps [B, C, H, W] complex128 (on the GPU)."""
    from mridc_b200 import espirit

    B, C, H, W, _ = y.shape
    vecs, rank = espirit.calibrate(y, cw, kw, 0.02, centered)
    refs = []
    rm, rl, om, ol, pm, po = [], [], [], [], [], []
    for b in range(B):
        r = espirit_ref(y[b], cw, kw, centered=centered)
        assert int(rank[b]) == r["K"], "%s slice %d: K = %d, reference %d" % (name, b, int(rank[b]), r["K"])
        lr, lo = r["lam"], lam[b].double()
        fixed = (lr - 0.95).abs() > CROP_BAND
        assert torch.equal((lo > 0.95)[fixed], (lr > 0.95)[fixed]), "%s slice %d: crop decisions differ at %d pixels" % (
            name, b, int(((lo > 0.95) != (lr > 0.95))[fixed].sum()))
        mo = _complex(maps[b])
        keep = fixed & (r["maps"][0].abs() >= X0_MIN)
        rm.append(r["maps"] * keep)
        om.append(mo * keep)
        rl.append(lr * fixed)
        ol.append(lo * fixed)
        # phase-free projector x x^H: || a a^H - b b^H ||_F^2 = |a|^4 + |b|^4 - 2 |a^H b|^2 per pixel
        a2, b2 = mo.abs().square().sum(0), r["maps"].abs().square().sum(0)
        d2 = (a2.square() + b2.square() - 2 * (mo.conj() * r["maps"]).sum(0).abs().square()).clamp_min(0)
        pm.append((d2 * fixed).sum().sqrt()[None])
        po.append((b2.square() * fixed).sum().sqrt()[None])
        refs.append(r["maps"])
        print("[espirit] %-28s slice %d: K = %d, %d pixels in the crop band, %d with |x0| < 1e-3" % (
            name, b, r["K"], int((~fixed).sum()), int((fixed & (r["maps"][0].abs() < X0_MIN) & (lr > 0.95)).sum())))
    check_slices(name + " maps", torch.stack(om), torch.stack(rm), TOL)
    check_slices(name + " lambda", torch.stack(ol), torch.stack(rl), TOL)
    proj = torch.cat(pm) / torch.cat(po)
    print("[espirit] %-28s projector rel-L2 worst %.2e (tol %.0e)" % (name, proj.max(), TOL))
    assert bool((proj <= TOL).all()), "%s projector: %s" % (name, proj.tolist())
    return torch.stack(refs)


GEOMETRIES = {
    "15x320x320_b4": dict(B=4, C=15, H=320, W=320),
    "16x640x320": dict(B=1, C=16, H=640, W=320),
    "32x232x288": dict(B=1, C=32, H=232, W=288),
    "8x97x81_odd": dict(B=2, C=8, H=97, W=81),
    "8x96x80_uncentred": dict(B=1, C=8, H=96, W=80, centered=False),
    "16x320x320_equispaced4x": dict(B=1, C=16, H=320, W=320, masked=True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("geom", sorted(GEOMETRIES))
def test_maps_against_fp64(geom):
    import mridc_b200 as mb

    g = dict(GEOMETRIES[geom])
    centered = g.pop("centered", True)
    y = _kspace(g["B"], g["C"], g["H"], g["W"], centered, g.pop("masked", False)).cuda()
    maps, lam = mb.espirit_maps(y, fft_centered=centered, return_eigenvalues=True)
    assert maps.shape == y.shape and lam.shape == (g["B"], g["H"], g["W"])
    _compare(geom, y, maps, lam, centered)
    if geom == "15x320x320_b4":  # the bench geometry: the estimate is the true map set
        sup = support(g["H"], g["W"]).cuda()
        corr = true_correlation(_complex(maps[0]), g["C"], g["H"], g["W"])[sup]
        frac = float((corr >= 0.999).double().mean())
        print("[espirit] |<s_est, s_true>| on the support: min %.5f median %.6f, %.4f of the pixels >= 0.999" % (
            corr.min(), corr.median(), frac))
        # measured on a B200: min 0.99865 (the fp64 reference agrees to 1e-7), median 0.999985
        assert corr.median() >= 0.9999 and corr.min() >= 0.998 and frac >= 0.99


@pytest.mark.gpu
def test_deterministic_and_batch_invariant(monkeypatch):
    """Two runs give the same bits; each slice alone, and in a batch processed in chunks of 2, gives the bits it has in
    the whole batch (both power-iteration instantiations)."""
    import mridc_b200 as mb
    from mridc_b200 import espirit

    for C in (12, 20):
        y = _kspace(3, C, 128, 96).cuda()
        y[1] *= 0.5
        y[2] = torch.flip(y[2], (-2,))
        m1, l1 = mb.espirit_maps(y, return_eigenvalues=True)
        m2, l2 = mb.espirit_maps(y, return_eigenvalues=True)
        assert torch.equal(m1, m2) and torch.equal(l1, l2)
        for b in range(3):
            mb_, lb = mb.espirit_maps(y[b:b + 1].clone(), return_eigenvalues=True)
            assert torch.equal(mb_[0], m1[b]) and torch.equal(lb[0], l1[b]), (C, b)
        P = C * (C + 1) // 2
        monkeypatch.setattr(espirit, "G_CHUNK_BYTES", 2 * P * 128 * 96 * 8)
        m3, l3 = mb.espirit_maps(y, return_eigenvalues=True)
        monkeypatch.undo()
        assert torch.equal(m3, m1) and torch.equal(l3, l1)


@pytest.mark.gpu
@pytest.mark.parametrize("row,C", [("pipeline_c16", 16), ("pipeline_c32", 20)])
def test_every_instantiation_is_launched_by_its_row(row, C):
    import mridc_b200 as mb

    y = _kspace(1, C, 64, 48).cuda()
    _, seen = launched(lambda: mb.espirit_maps(y))
    want = {kernel_name(n) for n in EXPECTED[row]}
    print("[espirit] %s launched: %s" % (row, ", ".join(sorted(seen))))
    assert want <= seen, sorted(want - seen)
    other = {n for r, ns in EXPECTED.items() if r != row for n in ns} - want
    assert not other & seen, sorted(other & seen)


@pytest.mark.gpu
def test_sense_models_on_estimated_maps():
    """ZF-SENSE and a CIRIM on the estimated maps meet the 1e-4 model contract against the oracle given the same maps."""
    import mridc_b200 as mb
    from mridc_b200 import synth
    from oracle import models as omodels

    batch = synth.make_batch(2, 8, 96, 320, centered=True, normalization="ortho")
    maps = mb.espirit_maps(batch["y"].cuda())
    assert bool(torch.isfinite(maps).all()) and float(maps.abs().amax()) > 0
    S = maps.cpu()
    zcfg = synth.zf_cfg(centered=True, normalization="ortho")
    zo = mb.ZF(zcfg)(batch["y"].cuda(), maps, batch["mask"].cuda(), batch["target"].cuda())
    zr = omodels.zf_forward(zcfg, batch["y"], S, batch["mask"], batch["target"])
    e_zf = rel_l2(zo, zr)
    torch.manual_seed(1)
    cfg = synth.cirim_cfg("GRU", num_cascades=2, centered=True, normalization="ortho")
    model = mb.CIRIM(cfg).eval()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    out = next(model.cuda()(batch["y"].cuda(), maps, batch["mask"].cuda(), None, batch["target"].cuda()))
    with torch.no_grad():
        ref = omodels.cirim_forward(sd, cfg, batch["y"], S, batch["mask"], None, batch["target"])
    e_cirim = rel_l2(out[-1][-1], ref[-1][-1])
    print("[espirit] on estimated maps: ZF rel-L2 %.2e, CIRIM 2x8 GRU rel-L2 %.2e" % (e_zf, e_cirim))
    assert e_zf <= 1e-4 and e_cirim <= 1e-4


# ---------------------------------------------------------------------------------------------- GPU: ABI contract
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _esp():
    from mridc_b200 import _lib, espirit

    return espirit, espirit.load(), _lib


def _gram_row(B, C, H, W, cw, kw, centered):
    N = C * kw * kw
    ny = B * C * H * W * 2

    def make(seed):
        return {"y": torch.randn(ny, device="cuda", generator=_gen(seed))}

    def call(V, st):
        E, lib, L = _esp()
        E.check(lib.mrbe_calib_gram(L.ptr(V["y"]), L.ptr(V["gram"]), B, C, H, W, cw, kw, centered, st))

    def check(V, X):
        y = _complex(X["y"].reshape(B, C, H, W, 2))
        if not centered:
            y = torch.fft.fftshift(y, dim=(-2, -1))
        ref = torch.stack([(lambda A: A.conj().T @ A)(calib_matrix(y[b], cw, kw)) for b in range(B)])
        check_slices("mrbe_calib_gram", V["gram"].reshape(B, N, N, 2), torch.view_as_real(ref), 1e-13)

    return Row({"y": Buf("in", ny), "gram": Buf("out", B * N * N * 2, torch.float64)}, make, call, check)


def _taps_ref(vecs, K, C, H, W, kw, centered):
    """vecs [N, N] complex128 (rows = eigenvectors), the last K used -> taps grid [P, H, W] complex128."""
    N = C * kw * kw
    w = vecs[N - K:].conj().reshape(K, C, kw, kw)  # w_i = conj(v_i)
    T = taps(w)
    L = 2 * kw - 1
    lag = torch.arange(L, device=vecs.device)
    lag = torch.where(lag < kw, lag, lag - L)
    iy, ix = ((lag + H // 2) % H, (lag + W // 2) % W) if centered else (lag % H, lag % W)
    grid = torch.zeros(H, W, C, C, dtype=T.dtype, device=T.device)
    grid.index_put_((iy[:, None].expand(L, L), ix[None, :].expand(L, L)), T.permute(2, 3, 0, 1), accumulate=True)
    iu = torch.triu_indices(C, C)
    return grid[:, :, iu[0], iu[1]].permute(2, 0, 1)


def _taps_row(B, C, H, W, kw, centered, ranks):
    N, P = C * kw * kw, C * (C + 1) // 2

    def make(seed):
        g = _gen(seed)
        v = torch.linalg.qr(torch.randn(B, N, N, dtype=torch.complex128, device="cuda", generator=g))[0].mT
        return {"vecs": torch.view_as_real(v.contiguous()).reshape(-1).clone(),
                "rank": torch.tensor(ranks, dtype=torch.int32, device="cuda")}

    def call(V, st):
        E, lib, L = _esp()
        E.check(lib.mrbe_kernel_taps(L.ptr(V["vecs"]), L.ptr(V["rank"]), L.ptr(V["taps"]), B, C, H, W, kw, centered, st))

    def check(V, X):
        v = _complex(X["vecs"].reshape(B, N, N, 2))
        ref = torch.stack([_taps_ref(v[b], ranks[b], C, H, W, kw, centered) for b in range(B)])
        out = V["taps"].reshape(B, P, H, W, 2)
        check_slices("mrbe_kernel_taps", out, torch.view_as_real(ref), 1e-6)
        assert bool((out.reshape(B, P, -1, 2)[..., 0] != 0).any()) or sum(ranks) == 0

    bufs = {"vecs": Buf("in", B * N * N * 2, torch.float64), "rank": Buf("in", B, torch.int32),
            "taps": Buf("out", B * P * H * W * 2)}
    return Row(bufs, make, call, check)


def _power_row(B, C, H, W, max_iter, crop):
    P, HW = C * (C + 1) // 2, H * W
    iu = torch.triu_indices(C, C)

    def make(seed):
        g = _gen(seed)
        # G = a u u^H + (1/C) R R^H per pixel, a spread around the crop; one pixel with G = 0
        u = torch.randn(B, HW, C, 1, dtype=torch.complex128, device="cuda", generator=g)
        u = u / u.norm(dim=-2, keepdim=True)
        R = torch.randn(B, HW, C, C, dtype=torch.complex128, device="cuda", generator=g) * 0.15 / C ** 0.5
        a = 0.7 + 0.5 * torch.rand(B, HW, 1, 1, dtype=torch.float64, device="cuda", generator=g)
        G = a * u @ u.mH + R @ R.mH
        G[:, 3] = 0
        planes = G[:, :, iu[0], iu[1]].permute(0, 2, 1)  # [B, P, HW]
        return {"g": torch.view_as_real(planes.to(torch.complex64).contiguous()).reshape(-1).clone()}

    def call(V, st):
        E, lib, L = _esp()
        E.check(lib.mrbe_power_maps(L.ptr(V["g"]), L.ptr(V["maps"]), L.ptr(V["lam"]), B, C, H, W, max_iter, crop, st))

    def check(V, X):
        planes = _complex(X["g"].reshape(B, P, HW, 2))
        G = torch.zeros(B, HW, C, C, dtype=torch.complex128, device="cuda")
        G[:, :, iu[0], iu[1]] = planes.permute(0, 2, 1)
        G = G + torch.triu(G, 1).mH
        maps, lams = [], []
        for b in range(B):
            m, l = power(G[b].reshape(H, W, C, C), max_iter, crop)
            maps.append(torch.view_as_real(m))
            lams.append(l)
        lam_out = V["lam"].reshape(B, H, W)
        assert bool((lam_out.reshape(B, -1)[:, 3] == 0).all()) and bool((V["maps"].reshape(B, C, HW, 2)[:, :, 3] == 0).all())
        check_slices("mrbe_power_maps lambda", lam_out, torch.stack(lams), 1e-5)
        check_slices("mrbe_power_maps maps", V["maps"].reshape(B, C, H, W, 2), torch.stack(maps), 1e-5)

    bufs = {"g": Buf("in", B * P * HW * 2), "maps": Buf("out", B * C * HW * 2), "lam": Buf("out", B * HW)}
    return Row(bufs, make, call, check)


ROWS = {
    "gram_centred": (("mrbe_calib_gram",), lambda: _gram_row(2, 3, 30, 27, 12, 4, 1)),
    "gram_uncentred_odd": (("mrbe_calib_gram",), lambda: _gram_row(1, 5, 31, 33, 15, 5, 0)),
    "taps_centred": (("mrbe_kernel_taps",), lambda: _taps_row(2, 3, 20, 17, 4, 1, [20, 7])),
    "taps_uncentred_aliased": (("mrbe_kernel_taps",), lambda: _taps_row(2, 2, 5, 6, 4, 0, [32, 0])),
    "power_c5": (("mrbe_power_maps",), lambda: _power_row(2, 5, 7, 9, 60, 0.95)),
    "power_c20": (("mrbe_power_maps",), lambda: _power_row(2, 20, 5, 7, 60, 0.95)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(ROWS))
def test_contract(name):
    run_contract(ROWS[name][1]())
