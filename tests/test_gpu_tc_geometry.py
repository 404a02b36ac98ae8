"""Every geometry the tensor-core entry points of the CIRIM time step accept, checked against fp64 on raw pointers.

The C entry points take any B, H, W >= 1; RimTcEngine calls them on a narrower set (RimTcEngine.covers, and the final
conv routed by RimTcEngine.final_conv_symbol).  Every kernel tiles a flat position space, and its edges are where a
kernel goes wrong:
  tc_kernel, gru2, ind2, conv5g   128-position tiles over the B (H+4)(W+4) positions of the BH grid; tc_kernel loads
                                  TMA boxes of 136 positions, conv5g five bulk copies per tile, W+4 positions apart,
                                  reaching into the G8 guard positions
  fin2                            16 x 16 3-D TMA boxes over the [B (H+4)] x (W+4) grid and 14 x 14 output patches: a box
                                  can be wider than W+4 or taller than B (H+4), a patch can cross two slices, H mod 14 and
                                  W mod 14 set the phase of the last patch
  uconv3                          an [H][W+1] grid in 128-position tiles, three loader groups, at most 32 output channels
                                  per launch, channel groups of 8 padded to 2, 4 or 8
GEOMS lists shapes on each of those edges with the boundary they sit on; a CPU test derives the quantities from the list
and fails when a class has no shape.

Each call goes through the buffer harness of test_gpu_abi_contract.py with fresh seeded inputs: inputs inside NaN guard
bands, outputs pre-filled with a byte sentinel (every position the header says is written must be), and a second run
with the BH borders the header says are never read set to NaN and the outputs NaN, which must give the same bits.
Results are compared per slice with an fp64 evaluation of oracle/nets.py on the GPU: 1e-5 for the split-bf16 kernels,
5e-6 for the CUDA-core final conv, 2e-6 for uconv3; a slice of fewer than SMALL_SLICE values (a final conv on one pixel
has two) is measured against the magnitudes of the terms it sums, since its own values can cancel to any smallness
(check_slices' ``scale``), and those rows are repeated over 16 seeds.  The rule of every row: status 0 and within tolerance, or
MRB_EUNSUPPORTED with a message naming a limit include/mridc_b200.h states (LIMITS below).  Status 0 with a wrong result
fails, and so does a refusal the header does not state.
"""
import gc

import pytest
import torch
import torch.nn.functional as F

import test_gpu_abi_contract as abi
from test_gpu_bench_shapes import SMALL_SLICE, check_slices
from test_gpu_kernel_paths import _gen, _lib

TILE, BOX, PATCH, OUT = 128, 136, 16, 14

# (B, H, W): the boundary each shape sits on.  Q = B (H+4)(W+4) flat positions, "rows" = B (H+4) padded rows.
GEOMS = [
    (1, 1, 1),     # Q = 25: the smallest tensor, one partial tile; W + 4 = 5 < 16; H, W = 1 mod 14
    (2, 1, 1),     # Q = 50 < 128, two slices in one partial tile; fin2 patch of slice 0 runs into slice 1
    (1, 2, 5),     # Q = 54 < 128; W = 5
    (3, 1, 2),     # Q = 90 < 128; rows 15 (B = 3, H = 1); W = 2; fin2 patches straddle slices
    (1, 4, 12),    # Q = 128: exactly one tile, below one 136-position box; W + 4 = 16 = the fin2 box width
    (1, 5, 11),    # Q = 135: one tile + 7, still below one box; W + 4 = 15
    (1, 13, 8),    # rows 17 (B = 1, H = 13); H = 13 mod 14; W = 8
    (2, 4, 12),    # Q = 256 = 2 tiles; rows 16 (B = 2, H = 4); fin2 patch of slice 0 runs into slice 1
    (1, 11, 13),   # Q = 255 = 2 tiles - 1; rows 15 (B = 1, H = 11); W = 13 mod 14
    (1, 12, 20),   # Q = 384 = 3 tiles; rows 16 (B = 1, H = 12); W = 20
    (1, 1, 73),    # Q = 385 = 3 tiles + 1: the last tile holds one position
    (1, 3, 69),    # Q = 511 = 4 tiles - 1
    (1, 15, 23),   # Q = 513 = 4 tiles + 1; H = 1 mod 14
    (2, 15, 13),   # two patch rows per slice, the second crosses into slice 1; W = 13 mod 14
    (1, 27, 1),    # H = 13 mod 14 over two patch rows; W = 1
    (4, 2, 27),    # W = 27, one under the engine's width, W = 13 mod 14; patches of slices 0-2 straddle
    (1, 14, 27),   # H = 0 mod 14; W = 27
    (2, 4, 28),    # Q = 512 = 4 tiles; rows 16; W = 28 = 0 mod 14, the narrowest width the engine covers
    (1, 9, 28),    # the contract rows' geometry: Q = 416 = 3.25 tiles
    (1, 28, 28),   # Q = 1024 = 8 tiles; H, W = 0 mod 14
    (2, 14, 29),   # W = 29 = 1 mod 14; H = 0 mod 14, B = 2
    (3, 17, 29),   # 17 tiles: tc_kernel tile pairs across slices; fin2 patches straddle
]

# The limits include/mridc_b200.h states for the entry points below: symbol -> (refused(B, H, W), text of the message).
# Empty: every entry point of the time step serves every B, H, W >= 1.  A refusal the C side adds without an entry here
# fails the GPU rows (an unstated refusal); the entry makes the routing test below hold the engine to it.
LIMITS = {}


def padded_rows(B, H):
    return B * (H + 4)


def positions(B, H, W):
    return B * (H + 4) * (W + 4)


def fin2_straddles(B, H):
    """The last 16-row box of a slice reaches past its padded rows into the next slice."""
    py = -(-H // OUT)
    return B >= 2 and OUT * (py - 1) + PATCH > H + 3


def refused(symbol, B, H, W):
    lim = LIMITS.get(symbol)
    return lim is not None and lim[0](B, H, W)


# ---------------------------------------------------------------------------------------------- CPU: the list itself
def test_geometry_list_reaches_every_class():
    Q = [positions(B, H, W) for B, H, W in GEOMS]
    assert len(set(GEOMS)) == len(GEOMS)
    classes = {
        "1x1x1 (25 positions)": (1, 1, 1) in GEOMS,
        "below one tile": any(q < TILE for q in Q),
        "one tile or more, below one box": any(TILE <= q < BOX for q in Q),
        "a multiple of 128": any(q % TILE == 0 for q in Q),
        "one under a multiple of 128": any(q % TILE == TILE - 1 for q in Q),
        "one over a multiple of 128": any(q % TILE == 1 and q > TILE for q in Q),
        "fin2 patch across slices": any(fin2_straddles(B, H) for B, H, _ in GEOMS),
    }
    for w in (1, 2, 5, 8, 11, 12, 13, 20, 27, 28, 29):
        classes["W = %d" % w] = any(W == w for _, _, W in GEOMS)
    for bh in ((1, 11), (1, 12), (1, 13), (3, 1), (2, 4)):
        classes["(B, H) = %s, rows %d" % (bh, padded_rows(*bh))] = any((B, H) == bh for B, H, _ in GEOMS)
    for r in (0, 1, 13):
        classes["H mod 14 = %d" % r] = any(H % OUT == r for _, H, _ in GEOMS)
        classes["W mod 14 = %d" % r] = any(W % OUT == r for _, _, W in GEOMS)
    for wp in ("<", "=", ">"):
        classes["W + 4 %s 16" % wp] = any({"<": W + 4 < PATCH, "=": W + 4 == PATCH, ">": W + 4 > PATCH}[wp]
                                          for _, _, W in GEOMS)
    missing = sorted(k for k, v in classes.items() if not v)
    assert not missing, "geometry classes without a shape in GEOMS: %s" % missing


class _Recorder:
    """Stands in for the loaded library: records the entry points called, returns status 0."""

    def __init__(self):
        self.calls = set()

    def __getattr__(self, name):
        def call(*args):
            self.calls.add(name)
            return 0
        return call


def _rim_block(layer):
    from mridc_b200 import synth
    from mridc_b200.rim import RIMBlock

    cfg = synth.cirim_cfg(layer)
    kw = {k: cfg[k] for k in ("recurrent_layer", "conv_filters", "conv_kernels", "conv_dilations", "conv_bias",
                              "recurrent_filters", "recurrent_kernels", "recurrent_dilations", "recurrent_bias",
                              "depth", "time_steps", "conv_dim", "no_dc", "fft_centered", "fft_normalization",
                              "spatial_dims", "coil_dim", "dimensionality")}
    return RIMBlock(**kw)


def test_engine_routes_only_geometries_its_entry_points_accept(monkeypatch):
    """Every geometry RimTcEngine.covers takes reaches only entry points whose stated limits (LIMITS) accept it.  The
    entry points are those RimTcEngine.conv_stack_bh calls, recorded on the CPU with the library replaced by a recorder.
    While LIMITS is empty this can only fail on the recording itself; it holds the engine to the first limit added."""
    from mridc_b200 import _lib as L
    from mridc_b200.rim_tc import RimTcEngine

    rec = _Recorder()
    monkeypatch.setattr(L, "load", lambda: rec)
    monkeypatch.setattr(L, "stream_ptr", lambda: None)
    t = torch.zeros(1)
    shapes = set(GEOMS) | {(B, H, W) for B in (1, 2, 3, 4, 16) for H in range(1, 41) for W in (1, 13, 27, 28, 29, 45, 320)}
    routed = 0
    for layer in ("GRU", "IndRNN"):
        eng = RimTcEngine(_rim_block(layer))
        assert RimTcEngine.supported(eng.block)
        for B, H, W in sorted(shapes):
            if not eng.covers(W):
                continue
            routed += 1
            for g4 in (t, None) if W == 320 else (t,):  # None: the W = 320 DC kernel has written G8 itself
                rec.calls = set()
                eng.conv_stack_bh(g4, [t, t], [t, t], t, torch.zeros(B, H, W, 2), [(t, t), (t, t)], B, H, W, t)
                assert "mrb_tc2_conv5x5x4" in rec.calls and ("mrb_g8_from_nhwc4" in rec.calls) == (g4 is not None)
                assert RimTcEngine.final_conv_symbol(B, H) in rec.calls
                bad = sorted(c for c in rec.calls if refused(c, B, H, W))
                assert not bad, "RimTcEngine routes %dx%dx%d to entry points that refuse it: %s" % (B, H, W, bad)
    assert routed > 0


# ---------------------------------------------------------------------------------------------- CPU: the check bites
def _bh_cpu(x):
    """fp64 [B, 64, H, W] -> BH bf16 [B, H+4, W+4, 128] (hi | lo, replicate border) on the CPU."""
    B, _, H, W = x.shape
    t = F.pad(x.float(), (2, 2, 2, 2), mode="replicate").permute(0, 2, 3, 1)
    hi = t.to(torch.bfloat16)
    lo = (t - hi.float()).to(torch.bfloat16)
    return torch.cat([hi, lo], -1).contiguous()


def _smallest(n, pred):
    return sorted((g for g in GEOMS if pred(*g)), key=lambda g: positions(*g))[:n]


def _last_tile_interior(B, H, W):
    """-> (interior positions in the last 128-position tile, interior positions of the last slice)."""
    Q = positions(B, H, W)
    interior = torch.zeros((B, H + 4, W + 4), dtype=torch.bool)
    interior[:, 2:H + 2, 2:W + 2] = True
    return int(interior.reshape(-1)[(Q - 1) // TILE * TILE:].sum()), H * W


def test_check_fails_when_the_last_partial_tile_is_zero():
    """A BH output whose last, partial 128-position tile was never computed (zero) fails the per-slice check that the
    GPU rows apply where that tile holds only some rows of a slice of several tiles; the exact output passes."""
    geoms = _smallest(4, lambda B, H, W: positions(B, H, W) > TILE and positions(B, H, W) % TILE != 0
                      and 0 < _last_tile_interior(B, H, W)[0] < _last_tile_interior(B, H, W)[1])
    assert len(geoms) == 4
    for B, H, W in geoms:
        g = torch.Generator().manual_seed(B * 1000 + H * 31 + W)
        ref = torch.randn((B, 64, H, W), generator=g, dtype=torch.float64)
        bh = _bh_cpu(ref)
        abi._check_bh("self-test exact %dx%dx%d" % (B, H, W), bh.reshape(-1), ref, B, H, W)
        Q = positions(B, H, W)
        bh.view(Q, 128)[(Q - 1) // TILE * TILE:] = 0
        with pytest.raises(AssertionError, match=r"slices over the rel-L2 tolerance 1e-05: \[\(%d, " % (B - 1)):
            abi._check_bh("self-test last tile zero %dx%dx%d" % (B, H, W), bh.reshape(-1), ref, B, H, W)


def _final_conv_ref(B, H, W, seed):
    """fp64 eta + conv3x3(h) (+ bias) on the CPU, with the term magnitudes |eta| + |b| + sum |w| |h| of every output."""
    from oracle import nets as onets

    g = torch.Generator().manual_seed(seed)
    h = torch.randn((B, 64, H, W), generator=g, dtype=torch.float64)
    w = torch.randn((2, 64, 3, 3), generator=g, dtype=torch.float64) * 0.05
    b = torch.randn(2, generator=g, dtype=torch.float64)
    eta = torch.randn((B, H, W, 2), generator=g, dtype=torch.float64)
    conv = onets.conv_nonlinear(h, w, b, 3, 1, None).permute(0, 2, 3, 1)
    mag = onets.conv_nonlinear(h.abs(), w.abs(), b.abs(), 3, 1, None).permute(0, 2, 3, 1)
    return h, w, b, eta, eta + conv, eta.abs() + mag


def test_check_fails_when_a_fin2_patch_row_is_shifted():
    """A final-conv output with one row of its last patch shifted by one column fails the per-slice check the GPU rows
    apply (the term-magnitude scale included); the fp32 rounding of the fp64 reference passes it."""
    geoms = _smallest(4, lambda B, H, W: W >= 2) + [(2, 15, 13), (1, 28, 28)]
    for B, H, W in geoms:
        _, _, _, _, ref, mag = _final_conv_ref(B, H, W, B * 1000 + H * 31 + W)
        out = ref.float()
        check_slices("self-test exact %dx%dx%d" % (B, H, W), out, ref, 1e-5, scale=mag)
        py, px = -(-H // OUT), -(-W // OUT)
        y, x0 = OUT * (py - 1), OUT * (px - 1)
        row = out[B - 1, y, x0:x0 + OUT]
        row.copy_(torch.roll(row.clone(), 1, 0))
        with pytest.raises(AssertionError, match=r"slices over the rel-L2 tolerance 1e-05: \[\(%d, " % (B - 1)):
            check_slices("self-test shifted patch row %dx%dx%d" % (B, H, W), out, ref, 1e-5, scale=mag)


def test_small_slices_are_measured_against_their_terms():
    """A one-pixel final conv whose eta cancels the conv: an error of 2^-20 of its terms (rounding) is a large rel-L2 of
    the two cancelled values but passes against the term magnitudes; a conv with one tap's weights dropped still fails."""
    from oracle import nets as onets

    h, w, b, eta, ref, mag = _final_conv_ref(1, 1, 1, 5)
    conv, terms = ref - eta, mag - eta.abs()
    eta = -conv * (1 - 1e-6)  # eta + conv = 1e-6 of the conv
    ref, mag = eta + conv, eta.abs() + terms
    out = ref + mag * 2.0 ** -20
    with pytest.raises(AssertionError, match="slices over the rel-L2 tolerance"):
        check_slices("self-test cancelled, own norm", out, ref, 1e-5)
    check_slices("self-test cancelled, term magnitudes", out, ref, 1e-5, scale=mag)
    w1 = w.clone()
    w1[:, :, 0, 0] = 0
    wrong = eta + onets.conv_nonlinear(h, w1, b, 3, 1, None).permute(0, 2, 3, 1)
    with pytest.raises(AssertionError, match="slices over the rel-L2 tolerance"):
        check_slices("self-test one tap dropped", wrong, ref, 1e-5, scale=mag)


# ---------------------------------------------------------------------------------------------- GPU rows
@pytest.fixture(autouse=True)
def _release_gpu_memory():
    yield
    gc.collect()
    if torch.cuda.is_available() and torch.cuda.is_initialized():
        torch.cuda.empty_cache()


def _steps(B, H, W):
    """(symbol, tag, row factory) of every entry point of the time step, in the order the engine calls them."""
    return [
        ("mrb_bh_from_nhwc", "bh_from_nhwc", lambda: abi._bh_from_row(B, H, W)),
        ("mrb_bh_to_nhwc", "bh_to_nhwc", lambda: abi._bh_to_row(B, H, W)),
        ("mrb_g8_from_nhwc4", "g8_from_nhwc4", lambda: abi._g8_row(B, H, W)),
        ("mrb_tc2_conv5x5x4", "tc2_conv5x5x4", lambda: abi._conv5_row(B, H, W)),
        ("mrb_tc2_gru", "tc2_gru", lambda: abi._cell_bh_row("mrb_tc2_gru", B, H, W)),
        ("mrb_tc2_indrnn", "tc2_indrnn", lambda: abi._cell_bh_row("mrb_tc2_indrnn", B, H, W)),
        ("mrb_bh_fix_border", "bh_fix_border", lambda: abi._bh_fix_row(B, H, W)),
        ("mrb_tc_conv_bh", "tc_conv_bh k3 d2", lambda: abi._tc_conv_row(B, H, W, 3, 2)),
        ("mrb_tc_conv_bh", "tc_conv_bh k5 d1", lambda: abi._tc_conv_row(B, H, W, 5, 1)),
        ("mrb_tc_conv_bh", "tc_conv_bh k1 d1", lambda: abi._tc_conv_row(B, H, W, 1, 1)),
        ("mrb_tc2_final_conv", "tc2_final_conv", lambda: abi._final_conv_row("mrb_tc2_final_conv", B, H, W)),
        ("mrb_conv_c2_bh_residual", "conv_c2_bh_residual", lambda: abi._final_conv_row("mrb_conv_c2_bh_residual", B, H, W)),
    ]


def _run_row(symbol, tag, factory, B, H, W, run):
    """Status 0 and the row's checks pass, or MRB_EUNSUPPORTED (NotImplementedError) where LIMITS states it."""
    try:
        run(factory())
    except NotImplementedError as e:
        lim = LIMITS.get(symbol)
        assert refused(symbol, B, H, W) and lim[1] in str(e), (
            "%s %dx%dx%d: refused (%s) outside the limits the header states" % (tag, B, H, W, e))
        print("[tc geometry] %-50s refused: %s" % ("%s %dx%dx%d" % (tag, B, H, W), e))
        return
    assert not refused(symbol, B, H, W), "%s %dx%dx%d: accepted although the header refuses it" % (tag, B, H, W)


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W", GEOMS, ids=["%dx%dx%d" % g for g in GEOMS])
def test_time_step_entry_points(B, H, W):
    """Every entry point of the time step at one geometry (each with fresh inputs); all failures are reported."""
    bad = []
    for symbol, tag, factory in _steps(B, H, W):
        try:
            _run_row(symbol, tag, factory, B, H, W, lambda r: abi.run_contract(r, graph=False))
        except (AssertionError, RuntimeError, ValueError) as e:
            bad.append("%s: %s" % (tag, str(e).splitlines()[0][:400]))
    assert not bad, "%dx%dx%d:\n  %s" % (B, H, W, "\n  ".join(bad))


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 16])
@pytest.mark.parametrize("H", [1, 2, 3, 17])
def test_dc_direct_g8_output_at_small_heights(H, C):
    """The W = 320 row-form DC kernel writing the G8 conv input itself (edge rows write the replicate border, H = 1 all
    five rows of a slice): byte for byte the converter of its fp32 output, which is compared per slice with fp64."""
    abi.run_contract(abi._dch_grad_row(2, C, H, 320, "u8-shared", H % 2 == 1, 2), graph=False)


# ---------------------------------------------------------------------------------------------- U-Net 3x3 conv
# (H, W): H (W + 1) positions per image in 128-position tiles
UC_SHAPES = [(1, 1), (2, 1), (1, 2), (3, 3), (5, 7),
             (1, 126),                    # 127 positions: one under a tile
             (2, 63), (4, 31), (64, 1),   # 128: exactly one tile (W = 1: every other position is the dummy column)
             (1, 128), (3, 42), (43, 2)]  # 129: one position in the second tile
UC_CIN = [1, 7, 8, 9, 15, 16, 17, 33, 63, 64]   # uconv3_kernel<1> (<= 16), <2> (<= 32), <4>, with padded groups of 8
UC_COUT = [1, 31, 32, 33, 65]                    # launches of <= 32 output channels, padded to 16


def _uconv_sweep_row(N, Cin, Cout, H, W):
    """x: channels [3, 3 + Cin) of a concat buffer, out: channels [2, 2 + Cout) of another; nothing else is written."""
    L, lib, _ = _lib()
    HW = H * W
    xbs, obs = (Cin + 3) * HW, (Cout + 3) * HW
    written = torch.zeros((N, obs), dtype=torch.bool)
    written[:, 2 * HW:(2 + Cout) * HW] = True
    nw = lib.mrb_tc2_unet_packed_bytes(Cin, Cout)
    bufs = {"x": abi.Buf("in", N * xbs), "wp": abi.Buf("in", nw, torch.uint8), "out": abi.Buf("out", N * obs, written=written)}

    def make(seed):
        g = _gen(seed)
        w = abi._rn(g, Cout * Cin * 9, scale=(9 * Cin) ** -0.5)
        pk = torch.empty(nw, dtype=torch.uint8, device="cuda")
        L.check(lib.mrb_tc2_unet_pack(L.ptr(w), L.ptr(pk), Cin, Cout, _lib()[2]))
        return {"x": abi._rn(g, N * xbs), "wp": pk, "_w": w}

    def call(V, st):
        L.check(lib.mrb_tc2_unet_conv3x3(L.ptr(V["x"][3 * HW:]), xbs, L.ptr(V["wp"]), L.ptr(V["out"][2 * HW:]), obs, N, Cin,
                                         Cout, H, W, st))

    def check(V, X):
        x = X["x"].reshape(N, xbs)[:, 3 * HW:].reshape(N, Cin, H, W).double()
        w = X["_w"].double().reshape(Cout, Cin, 3, 3)
        ref = F.conv2d(x, w, padding=1)
        out = V["out"].reshape(N, obs)[:, 2 * HW:(2 + Cout) * HW].reshape(N, Cout, H, W)
        check_slices("uconv3 %dx%dx%d Cin %d Cout %d" % (N, H, W, Cin, Cout), out, ref, 2e-6,
                     scale=F.conv2d(x.abs(), w.abs(), padding=1))

    return abi.Row(bufs, make, call, check)


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", UC_SHAPES, ids=["%dx%d" % s for s in UC_SHAPES])
def test_uconv3_channel_sweep(H, W):
    """Every (Cin, Cout) of the sweep at one image size, N alternating 1 and 3 (each pair sees both over the shapes)."""
    bad = []
    for i, (Cin, Cout) in enumerate((ci, co) for ci in UC_CIN for co in UC_COUT):
        N = 1 if (i + H + W) % 2 else 3
        r = _uconv_sweep_row(N, Cin, Cout, H, W)

        def run(row):
            X = row.make(1)
            row.check(abi.views(abi.eager(row, X, "cuda")), X)

        try:
            _run_row("mrb_tc2_unet_conv3x3", "uconv3 N %d Cin %d Cout %d" % (N, Cin, Cout), lambda: r, N, H, W, run)
        except (AssertionError, RuntimeError, ValueError) as e:
            bad.append("N %d Cin %d Cout %d: %s" % (N, Cin, Cout, str(e).splitlines()[0][:300]))
    assert not bad, "uconv3 %dx%d:\n  %s" % (H, W, "\n  ".join(bad))


def _eager_check(row, seed):
    X = row.make(seed)
    row.check(abi.views(abi.eager(row, X, "cuda", tag="eager seed %d" % seed)), X)


SEEDS = range(2, 18)


@pytest.mark.gpu
def test_small_slices_over_seeds():
    """The rows whose slices hold fewer than SMALL_SLICE values (final conv on one to 27 pixels, uconv3 on one or two
    pixels with one or 31 output channels), each over 16 further seeds: measured against the term magnitudes, none of
    them passes by the luck of one draw."""
    bad = []
    for B, H, W in (g for g in GEOMS if 2 * g[1] * g[2] < SMALL_SLICE):
        for symbol, tag, factory in _steps(B, H, W):
            row = factory()
            for seed in SEEDS:
                try:
                    _eager_check(row, seed)
                except AssertionError as e:
                    bad.append("%s %dx%dx%d seed %d: %s" % (tag, B, H, W, seed, str(e).splitlines()[0][:300]))
    for H, W in ((1, 1), (2, 1), (1, 2)):
        for Cin in UC_CIN:
            for Cout in (1, 31):
                row = _uconv_sweep_row(1 + 2 * (Cin % 2), Cin, Cout, H, W)
                for seed in SEEDS:
                    try:
                        _eager_check(row, seed)
                    except AssertionError as e:
                        bad.append("uconv3 %dx%d Cin %d Cout %d seed %d: %s" % (H, W, Cin, Cout, seed,
                                                                              str(e).splitlines()[0][:300]))
    assert not bad, "\n  ".join(bad)
