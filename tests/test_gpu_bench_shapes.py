"""The hot path at the batch sizes bench.py reports, checked slice by slice against an fp64 run of the oracle on the GPU,
and the batch invariance of the bench workloads.

Why per slice: a whole-batch rel-L2 dilutes an error confined to one slice by sqrt(B).  One 128-position tile of one
slice of 16, wrong by 1e-3, is 3.5e-5 of that slice but 8.8e-6 of the batch (inside the 1e-5 of the split-bf16 kernels);
one whole slice of 16 wrong by 3e-4 is 7.5e-5 of the batch (inside the 1e-4 model contract).  The self-test below builds
both cases.  Rounding error is spread evenly over the slices, so each slice is held to the whole-tensor contract of
test_gpu_parity.py / test_gpu_tc.py:

  2e-6  fp32 operators (DC gradient, sens_reduce / sens_expand_softdc, instance norm, pooling, 2x2 transposed conv, 1x1
        conv, NormUnet prologue / epilogue).  A 320- or 640-point fp32 transform rounds at ~9-10 butterfly levels, the
        operators chain two of them with complex products and a coil sum of 15-16 terms: some 40 roundings of
        u = 2^-24 = 6e-8, rms ~ u * sqrt(40) = 4e-7 per output, 5x under the bound.
  1e-5  split-bf16 tensor-core kernels (tc2_*, tc_conv_bh): every operand is carried as hi + lo bf16 (16-17 significant
        bits), a_lo * b_lo is dropped, ~3e-6 rms per product, plus the tensor core's truncating fp32 accumulation over
        the K chain (the derivation of test_gpu_tc.py).
  2e-6  uconv3 (U-Net 3x3 conv): fp16 hi + lo operands (2^-22), all four products, accumulation chains of <= 12 terms;
        measured 1.2-3.9e-7 per operator, the same as the exact-fp32 kernel (DESIGN.md).
  1e-4  models (rel-L2 of the reconstruction): the project's contract.  The fp32 CPU oracle itself sits 2.7e-5 to
        3.7e-5 from fp64 on E2EVN and 3.4e-5 on CIRIM GRU; a CPU emulation of the split-bf16 arithmetic puts CIRIM 5x8
        at 2.5e-5.

Gradient outputs are compared on their gradient channels only; the eta channels they pass through must be bit-exact.

Batch invariance is bit-identity, no tolerance: every output value is computed by the same arithmetic in the same order
whatever the batch size and whatever position its slice has in the batch (DC rows, tensor-core tiles with a fixed K
chain, instance-norm statistics reduced in a fixed cluster-rank order), so any difference is a bug: a wrong batch
stride, a tile that reads across a slice boundary, a cache keyed on the wrong geometry, a graph replaying stale inputs.

The fp64 references run the oracle (oracle/nets.py, oracle/models.py: plain torch, nothing from mridc_b200) on CUDA
float64 tensors: float64 never takes a TF32 path, so no global torch flag is touched.
"""
import gc

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2

KEYS = ("y", "sensitivity_maps", "mask", "target")
# distance of the fp32 CPU oracle to an fp64 run on one slice of the same geometry, as recorded in DESIGN.md (section 4 and
# the U-Net numerics) and SURVEY.md section 7 (test_gpu_parity.py prints it); not recorded for the brain-geometry CIRIM
FP32_ORACLE_VS_FP64 = {"cirim_gru": 3.4e-5, "cirim_indrnn": 2.0e-7, "e2evn": 2.7e-5, "brain_cirim": None,
                       "brain_e2evn": 3.7e-5}


@pytest.fixture(autouse=True)
def _release_gpu_memory():
    """The B200 machines are shared: hand the cached blocks of each test back to the driver."""
    yield
    gc.collect()
    if torch.cuda.is_available() and torch.cuda.is_initialized():
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- per-slice comparison
def _real64(t):
    t = torch.as_tensor(t)
    return (torch.view_as_real(t) if t.is_complex() else t).double()


def slice_errors(out, ref):
    """-> (rel-L2, max-abs error / max |ref|) of every slice (dim 0) of out against ref, float64 on the CPU."""
    ref = _real64(ref)
    out = _real64(out).to(ref.device)
    assert out.shape == ref.shape, (tuple(out.shape), tuple(ref.shape))
    d = (out - ref).reshape(ref.shape[0], -1)
    r = ref.reshape(ref.shape[0], -1)
    rel = d.norm(dim=1) / r.norm(dim=1).clamp_min(1e-300)
    mx = d.abs().amax(1) / r.abs().amax(1).clamp_min(1e-300)
    return rel.cpu(), mx.cpu()


def check_slices(name, out, ref, tol, slices=None):
    """Every slice's rel-L2 <= tol (NaN fails).  Prints the worst slice, its max-abs error relative to its max |ref| and
    the margin to the tolerance.  ``slices``: the batch indices of the compared slices (default 0 .. n-1)."""
    rel, mx = slice_errors(out, ref)
    ids = list(range(len(rel))) if slices is None else [int(i) for i in slices]
    w = int(torch.nan_to_num(rel, nan=float("inf")).argmax())
    print("[bench shapes] %-50s %2d slices, worst %2d: rel-L2 %.2e  max-abs/max|ref| %.2e  tol %.0e  margin %6.1fx" % (
        name, len(ids), ids[w], rel[w], mx[w], tol, tol / float(rel[w]) if rel[w] != 0 else float("inf")))
    bad = [(ids[i], float(rel[i])) for i in range(len(ids)) if not rel[i] <= tol]
    assert not bad, "%s: slices over the rel-L2 tolerance %.0e: %s" % (name, tol, bad)
    return rel


def test_slice_check_catches_errors_that_whole_tensor_rel_l2_misses():
    """CPU self-test of the helper on the perturbations of the module docstring (16 slices of 320 x 320 x 2)."""
    g = torch.Generator().manual_seed(0)
    ref = torch.randn(16, 320, 320, 2, generator=g, dtype=torch.float64)
    out = ref.clone()
    out[15].view(-1, 2)[5000:5128] *= 1 + 1e-3  # one 128-position tile of the last slice, off by 1e-3
    whole = rel_l2(out, ref)
    rel, mx = slice_errors(out, ref)
    print("one tile: whole-batch rel-L2 %.2e, slice 15 %.2e" % (whole, rel[15]))
    assert whole < 1e-5  # passes the whole-tensor tolerance of the split-bf16 kernels
    assert rel[:15].max() == 0 and rel[15] > 3e-5
    assert abs(mx[15] - 1e-3 * ref[15].view(-1, 2)[5000:5128].abs().max() / ref[15].abs().max()) < 1e-12
    with pytest.raises(AssertionError, match=r"\[\(15, "):
        check_slices("self-test: one tile of slice 15 off by 1e-3", out, ref, 1e-5)
    out = ref.clone()
    out[15] *= 1 + 3e-4  # one whole slice off by 3e-4
    whole = rel_l2(out, ref)
    print("one slice: whole-batch rel-L2 %.2e" % whole)
    assert whole < 1e-4  # passes the model contract
    with pytest.raises(AssertionError, match=r"\[\(15, "):
        check_slices("self-test: slice 15 off by 3e-4", out, ref, 1e-4)
    out[15] = float("nan")
    with pytest.raises(AssertionError, match=r"\[\(15, nan"):
        check_slices("self-test: slice 15 NaN", out, ref, 1e-4)
    rel = check_slices("self-test: exact", ref.clone(), ref, 1e-12, slices=range(100, 116))
    assert rel.max() == 0


# ---------------------------------------------------------------------------------------------- bench workloads
def _inputs(workload):
    """CPU inputs of one bench.py workload, generated exactly as bench.py generates them."""
    import bench
    from mridc_b200 import synth

    if workload in ("cirim_gru", "cirim_indrnn"):
        return bench.build_inputs(16)
    if workload == "e2evn":
        np.random.seed(123)  # Gaussian1DMask draws from the global numpy RNG
        return synth.make_batch(8, 15, 320, 320, mask_func=synth.Gaussian1DMask([0.7], [4]), seed=123, mask_dtype="uint8")
    return synth.make_batch(8, 16, 640, 320, mask_func=synth.Equispaced1DMask([0.04], [8]))


def _model(workload):
    """(eval-mode model, cfg, CPU state dict) with bench.py's seeded weights."""
    import mridc_b200 as mb
    from mridc_b200 import synth

    if "cirim" in workload:
        cfg = synth.cirim_cfg("IndRNN" if workload == "cirim_indrnn" else "GRU")
        torch.manual_seed(1)
        model = mb.CIRIM(cfg).eval()
    else:
        cfg = synth.varnet_cfg()
        torch.manual_seed(1)
        model = mb.VarNet(cfg).eval()
    return model, cfg, {k: v.detach().clone() for k, v in model.state_dict().items()}


def _gpu(d):
    return [d[k].cuda() for k in KEYS]


def _cirim_all(model, y, S, m, tgt):
    """Every estimate of a CIRIM forward: [cascades, time steps, B, H, W] complex."""
    return torch.stack([torch.stack(c) for c in next(model(y, S, m, None, tgt))])


WORKLOADS = ["cirim_gru", "cirim_indrnn", "e2evn", "brain_cirim", "brain_e2evn"]


@pytest.mark.gpu
@pytest.mark.parametrize("workload", WORKLOADS)
def test_model_at_bench_batch_vs_fp64(workload):
    """The five bench workloads at their bench batch (CIRIM 16 slices of 15 x 320 x 320; E2EVN and both brain-geometry
    runs 8 slices) with bench.py's seeded weights and inputs.  The first, middle and last slice against the oracle run
    in fp64 on those slices: rel-L2 <= 1e-4 each (the model contract).  test_batch_invariance_of_the_bench_workloads
    extends this to every slice."""
    from oracle import models as omodels

    model, cfg, sd = _model(workload)
    y, S, m, tgt = _gpu(_inputs(workload))
    model = model.cuda()
    cirim = "cirim" in workload
    out = next(model(y, S, m, None, tgt))[-1][-1] if cirim else model(y, S, m, None, tgt)
    B = y.shape[0]
    idx = [0, B // 2, B - 1]
    del model
    sd64 = {k: v.cuda().double() for k, v in sd.items()}
    fwd = omodels.cirim_forward if cirim else omodels.varnet_forward
    with torch.no_grad():
        ref = fwd(sd64, cfg, y[idx].double(), S[idx].double(), m, None, tgt[idx])
    ref = ref[-1][-1] if cirim else ref
    rel = check_slices("%s B=%d vs fp64 oracle" % (workload, B), out[idx], ref, 1e-4, slices=idx)
    floor = FP32_ORACLE_VS_FP64[workload]
    print("[bench shapes] %-50s CUDA vs fp64 %s | fp32 oracle vs fp64 %s" % (
        workload, " ".join("%.2e" % float(e) for e in rel), "%.1e" % floor if floor else "not recorded"))


# ---------------------------------------------------------------------------------------------- RIM operators
@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["cirim_gru", "brain_cirim"])
def test_dc_hybrid_gradient_at_bench_batch_vs_fp64(workload):
    """dc_hybrid_prepare + the single-kernel hybrid-form gradient, the way CIRIM's time loop runs it: 16 slices of
    15 x 320 x 320 (the bench's equispaced 4x uint8 mask, not centred, backward norm) and 8 brain slices of
    16 x 640 x 320 (whose prepare takes the 640-point strided transform).  fp32 NHWC output vs fp64, per slice; the G8
    output mode (split-bf16 conv input with its replicate border) == fp32 output through mrb_g8_from_nhwc4, byte for
    byte."""
    from mridc_b200 import _lib, _ops
    from oracle import nets as onets

    y, S, m, _ = _gpu(_inputs(workload))
    B, C, H, W, _ = y.shape
    g = torch.Generator(device="cuda").manual_seed(H)
    eta = torch.randn((B, H, W, 2), device="cuda", generator=g)
    mcan = _ops.canonical_mask(m, B, H, W)[0]
    yh = _ops.dc_hybrid_prepare(y, mcan, False)
    assert yh is not None
    g4 = _ops.dc_rim_grad(eta, y, S, mcan, 1.0, False, "backward", nhwc=True, y_hybrid=yh)
    assert torch.equal(g4[..., :2], eta)
    ref = onets.log_likelihood_gradient(eta.double(), y.double(), S.double(), m, 1.0, False, "backward", [-2, -1], 1)
    check_slices("dc_rim_grad hybrid %dx%dx%d B=%d" % (C, H, W, B), g4[..., 2:].permute(0, 3, 1, 2), ref[:, 2:], 2e-6)
    del ref
    lib = _lib.load()
    ga = torch.zeros(lib.mrb_g8_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    _lib.check(lib.mrb_g8_from_nhwc4(_lib.ptr(g4), _lib.ptr(ga), B, H, W, _lib.stream_ptr()))
    gb = torch.zeros_like(ga)
    _ops.dc_rim_grad(eta, y, S, mcan, 1.0, False, "backward", out=gb, nhwc=2, y_hybrid=yh)
    assert torch.equal(ga, gb)


@pytest.mark.gpu
def test_dc_three_pass_2d_masks_at_bench_batch_vs_fp64():
    """The general three-pass gradient (what 2-D masks take) on the bench's 16 slices of 15 x 320 x 320: one shared 2-D
    mask and one 2-D mask per slice, both uint8 of density 0.25, vs fp64 per slice."""
    import bench
    from mridc_b200 import _ops
    from oracle import nets as onets

    y, S, _, _ = _gpu(bench.build_inputs(16))
    B, C, H, W, _ = y.shape
    g = torch.Generator(device="cuda").manual_seed(3)
    eta = torch.randn((B, H, W, 2), device="cuda", generator=g)
    for label, shape in (("shared 2-D mask", (1, 1, H, W, 1)), ("per-slice 2-D masks", (B, 1, H, W, 1))):
        m = (torch.rand(shape, device="cuda", generator=g) < 0.25).to(torch.uint8)
        out = _ops.dc_rim_grad(eta, y, S, m, 1.0, False, "backward")
        assert torch.equal(out[:, :2], eta.permute(0, 3, 1, 2))
        ref = onets.log_likelihood_gradient(eta.double(), y.double(), S.double(), m, 1.0, False, "backward", [-2, -1], 1)
        check_slices("dc_rim_grad three-pass, %s B=%d" % (label, B), out[:, 2:], ref[:, 2:], 2e-6)
        del out, ref


@pytest.mark.gpu
def test_tc2_kernels_at_bench_batch_vs_fp64():
    """The regulariser kernels of a CIRIM time step at the bench batch, 16 slices of 320 x 320 on BH buffers
    ([B][H+4][W+4][64 hi | 64 lo bf16]): there every CTA of the persistent kernels walks many tiles and tiles cross slice
    boundaries of the flattened position space.  conv5x5x4 fed from G8, ConvGRU and IndRNN cells, the dilation-2 3x3
    conv and the final 3x3 tap-GEMM conv with the eta update, each vs fp64 per slice (split-bf16: 1e-5)."""
    from mridc_b200 import _lib
    from oracle import nets as onets

    lib = _lib.load()
    st = _lib.stream_ptr()
    B, H, W = 16, 320, 320
    nb = lib.mrb_bh_bytes(B, H, W)
    g = torch.Generator(device="cuda").manual_seed(16)

    def randn(*shape, scale=1.0):
        return torch.randn(shape, device="cuda", generator=g) * scale

    def to_bh(t):
        buf = torch.empty(nb, dtype=torch.uint8, device="cuda")
        _lib.check(lib.mrb_bh_from_nhwc(_lib.ptr(t), _lib.ptr(buf), B, H, W, st))
        return buf

    def from_bh(buf):
        out = torch.empty((B, H, W, 64), device="cuda")
        _lib.check(lib.mrb_bh_to_nhwc(_lib.ptr(buf), _lib.ptr(out), B, H, W, st))
        return out.permute(0, 3, 1, 2)

    def poisoned():
        return torch.full((nb,), 0x7F, dtype=torch.uint8, device="cuda")

    def nchw64(t):
        return t.permute(0, 3, 1, 2).double()

    x4, w1, b1 = randn(B, H, W, 4), randn(64, 4, 5, 5, scale=0.2), randn(64)
    g8 = torch.zeros(lib.mrb_g8_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    _lib.check(lib.mrb_g8_from_nhwc4(_lib.ptr(x4), _lib.ptr(g8), B, H, W, st))
    ob = poisoned()
    _lib.check(lib.mrb_tc2_conv5x5x4(_lib.ptr(g8), _lib.ptr(w1), _lib.ptr(b1), _lib.ptr(ob), B, H, W, 1, st))
    ref = onets.conv_nonlinear(nchw64(x4), w1.double(), b1.double(), 5, 1, "relu")
    check_slices("mrb_tc2_conv5x5x4 (G8 -> BH) B=16", from_bh(ob), ref, 1e-5)
    del g8, x4, ref

    x, h = randn(B, H, W, 64), randn(B, H, W, 64)
    xb, hb = to_bh(x), to_bh(h)
    x64, h64 = nchw64(x), nchw64(h)
    del x, h
    wih, whh, bih = randn(192, 64, 1, 1, scale=0.1), randn(192, 64, 1, 1, scale=0.1), randn(192)
    pk = torch.empty(lib.mrb_tc2_gru_packed_bytes(), dtype=torch.uint8, device="cuda")
    _lib.check(lib.mrb_tc2_pack_gru(_lib.ptr(wih), _lib.ptr(whh), _lib.ptr(pk), 64, 64, st))
    ob = poisoned()
    _lib.check(lib.mrb_tc2_gru(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pk), _lib.ptr(bih), _lib.ptr(ob), B, H, W, st))
    ref = onets.conv_gru_cell(x64, h64, wih.double(), bih.double(), whh.double(), 1, 1)
    check_slices("mrb_tc2_gru B=16", from_bh(ob), ref, 1e-5)
    del ref

    wi, bi, hh = randn(64, 64, 1, 1, scale=0.1), randn(64), randn(1, 64, 1, 1, scale=0.5)
    pi = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, 1), device="cuda")
    _lib.check(lib.mrb_tc_pack_conv(_lib.ptr(wi), _lib.ptr(pi), 64, 64, 1, st))
    hhd = hh.reshape(-1).contiguous()
    ob = poisoned()
    _lib.check(lib.mrb_tc2_indrnn(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pi), _lib.ptr(bi), _lib.ptr(hhd), _lib.ptr(ob), B, H, W,
                                  st))
    ref = onets.indrnn_cell(x64, h64, wi.double(), bi.double(), hh.double(), 1, 1)
    check_slices("mrb_tc2_indrnn B=16", from_bh(ob), ref, 1e-5)
    del ref, h64, hb

    w2, b2 = randn(64, 64, 3, 3, scale=0.05), randn(64)
    p2 = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, 3), device="cuda")
    _lib.check(lib.mrb_tc_pack_conv(_lib.ptr(w2), _lib.ptr(p2), 64, 64, 3, st))
    ob = poisoned()
    _lib.check(lib.mrb_tc_conv_bh(_lib.ptr(xb), _lib.ptr(p2), _lib.ptr(b2), _lib.ptr(ob), B, H, W, 64, 3, 2, 1, st))
    ref = onets.conv_nonlinear(x64, w2.double(), b2.double(), 3, 2, "relu")
    check_slices("mrb_tc_conv_bh 3x3 dilation 2 B=16", from_bh(ob), ref, 1e-5)
    del ref, ob

    w3, b3, eta = randn(2, 64, 3, 3, scale=0.05), randn(2), randn(B, H, W, 2)
    o = torch.full((B, H, W, 2), float("nan"), device="cuda")
    _lib.check(lib.mrb_tc2_final_conv(_lib.ptr(xb), _lib.ptr(w3), _lib.ptr(b3), _lib.ptr(eta), _lib.ptr(o), B, H, W, st))
    ref = eta.double() + onets.conv_nonlinear(x64, w3.double(), b3.double(), 3, 1, None).permute(0, 2, 3, 1)
    check_slices("mrb_tc2_final_conv + eta B=16", o, ref, 1e-5)


# ---------------------------------------------------------------------------------------------- VarNet operators
@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["e2evn", "brain_e2evn"])
def test_sens_operators_at_bench_batch_vs_fp64(workload):
    """E2EVN's data-consistency halves on its 8 bench slices, 15 x 320 x 320 (col_softdc320) and 16 x 640 x 320
    (col_softdc640): sens_reduce of the bench k-space, sens_expand_softdc with and without the soft-DC epilogue (pred of
    the expansion's magnitude, dc_weight 0.8, the bench's uint8 column mask), vs fp64 per slice."""
    from mridc_b200 import _ops
    from oracle import nets as onets

    y, S, m, _ = _gpu(_inputs(workload))
    B, C, H, W, _ = y.shape
    y64, S64 = y.double(), S.double()
    red = _ops.sens_reduce(y, S, False, "backward")
    check_slices("sens_reduce %dx%dx%d B=%d" % (C, H, W, B), red, onets.sens_reduce(y64, S64, False, "backward", [-2, -1], 1)[:, 0],
                 2e-6)
    g = torch.Generator(device="cuda").manual_seed(H)
    img = torch.randn((B, H, W, 2), device="cuda", generator=g)
    E = onets.sens_expand(img.double().unsqueeze(1), S64, False, "backward", [-2, -1])
    out = _ops.sens_expand_softdc(img, S, None, None, None, None, None, True, False, "backward")
    check_slices("sens_expand (no_dc) %dx%dx%d B=%d" % (C, H, W, B), out, E, 2e-6)
    pred = torch.randn(y.shape, device="cuda", generator=g) * E.std().item()
    dcw = torch.tensor([0.8], device="cuda")
    out = _ops.sens_expand_softdc(img, S, pred, pred, y, m, dcw, False, False, "backward")
    p64 = pred.double()
    ref = p64 - torch.where(m.bool(), p64 - y64, torch.zeros((), dtype=torch.float64, device="cuda")) * 0.8 - E
    check_slices("sens_expand_softdc %dx%dx%d B=%d" % (C, H, W, B), out, ref, 2e-6)


def _instnorm_cluster_size(HW):
    """CTAs per plane of the single-pass instance norm (mrb_instnorm_lrelu): the smallest power of two <= 8 that leaves
    each CTA at most 64 KB of the plane."""
    cs = 1
    while cs < 8 and (HW * 4 + cs - 1) // cs > 65536:
        cs *= 2
    return cs


def _record_unet_launches(monkeypatch, model, args):
    """Run ``model(*args)`` once and return the distinct U-Net launches it made: (kind, integer arguments) in first-seen
    order, plus the weight of the first 3x3 conv seen with each shape."""
    from mridc_b200 import _lib, unet

    lib = _lib.load()
    seen = {}

    def note(kind, ints, extra=None):
        seen.setdefault((kind, ints), extra)

    conv0, norm0 = unet._conv3x3, unet._instnorm_lrelu

    def conv3x3(x, weight, x_bs, N, Cin, H, W, normalised=True):
        note("conv3x3", (x_bs, N, Cin, weight.shape[0], H, W, int(bool(normalised))), weight)
        return conv0(x, weight, x_bs, N, Cin, H, W, normalised)

    def instnorm_lrelu(x, x_bs, out, out_bs, N, C, HW, slope=0.2, eps=1e-5):
        note("instnorm_lrelu", (x_bs, out_bs, N, C, HW, int(out.data_ptr() == x.data_ptr())))
        return norm0(x, x_bs, out, out_bs, N, C, HW, slope, eps)

    def wrap(name):
        fn = getattr(lib, name)

        def call(*a):
            note(name, tuple(v for v in a if isinstance(v, int)))  # the shapes and strides; pointers are ctypes objects
            return fn(*a)
        return call

    with monkeypatch.context() as mp:
        mp.setattr(unet, "_conv3x3", conv3x3)
        mp.setattr(unet, "_instnorm_lrelu", instnorm_lrelu)
        for name in ("mrb_avgpool2", "mrb_conv_transpose2x2", "mrb_conv1x1", "mrb_normunet_in", "mrb_normunet_out"):
            mp.setattr(lib, name, wrap(name))
        model(*args)
        torch.cuda.synchronize()
    return seen


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["e2evn", "brain_e2evn"])
def test_unet_launches_of_e2evn_at_bench_batch_vs_fp64(workload, monkeypatch):
    """Every distinct U-Net launch E2EVN makes at its bench batch (8 slices, 15 x 320 x 320 and 16 x 640 x 320), taken from
    one recorded forward, re-run on its own with the recorded shapes and batch strides on seeded data (the model's own 3x3
    weights) and compared with fp64 per slice: uconv3 (2e-6), instance norm + LeakyReLU in place and into the concat
    buffer (every cluster size the launcher picks), 2x2 average pool, 2x2 transposed conv, 1x1 conv, NormUnet prologue
    and epilogue (fp32 operators, 2e-6).  Nothing outside a strided destination is written."""
    from mridc_b200 import _lib, unet

    model, _, _ = _model(workload)
    args = _gpu(_inputs(workload))
    launches = _record_unet_launches(monkeypatch, model.cuda(), (args[0], args[1], args[2], None, args[3]))
    del model, args
    lib = _lib.load()
    st = _lib.stream_ptr()
    g = torch.Generator(device="cuda").manual_seed(7)
    kinds = sorted(set(k for k, _ in launches))
    assert kinds == sorted(["conv3x3", "instnorm_lrelu", "mrb_avgpool2", "mrb_conv_transpose2x2", "mrb_conv1x1",
                            "mrb_normunet_in", "mrb_normunet_out"]), kinds
    clusters = sorted(set(_instnorm_cluster_size(a[4]) for k, a in launches if k == "instnorm_lrelu"))
    print("[bench shapes] %s: %d distinct U-Net launches, instance-norm cluster sizes %s" % (workload, len(launches), clusters))
    assert clusters == ([1, 4, 8] if "brain" in workload else [1, 2, 8]), clusters

    def rows(N, bs, scale=1.0, shift=0.0):
        return torch.randn((N, bs), device="cuda", generator=g) * scale + shift

    def nan_rows(N, bs):
        return torch.full((N, bs), float("nan"), device="cuda")

    for (kind, a), weight in launches.items():
        tag = "%s %s B=8 %s" % (kind.replace("mrb_", ""), workload, a)
        if kind == "conv3x3":
            x_bs, N, Cin, Cout, H, W, normalised = a
            x = rows(N, x_bs)
            out = unet._conv3x3(x, weight, x_bs, N, Cin, H, W, bool(normalised))
            ref = F.conv2d(x[:, :Cin * H * W].reshape(N, Cin, H, W).double(), weight.detach().double(), padding=1)
            check_slices(tag, out, ref, 2e-6)
        elif kind == "instnorm_lrelu":
            x_bs, out_bs, N, C, HW, inplace = a
            x = rows(N, x_bs, 1.5, 0.3)
            ref = F.leaky_relu(F.instance_norm(x[:, :C * HW].reshape(N, C, HW).double(), eps=1e-5), 0.2)
            out = x if inplace else nan_rows(N, out_bs)
            unet._instnorm_lrelu(x, x_bs, out, out_bs, N, C, HW)
            check_slices(tag, out[:, :C * HW].reshape(N, C, HW), ref, 2e-6)
            if not inplace:
                assert torch.isnan(out[:, C * HW:]).all()
        elif kind == "mrb_avgpool2":
            x_bs, out_bs, N, C, H, W = a
            x, out = rows(N, x_bs), nan_rows(N, out_bs)
            _lib.check(lib.mrb_avgpool2(_lib.ptr(x), x_bs, _lib.ptr(out), out_bs, N, C, H, W, st))
            n = C * (H // 2) * (W // 2)
            check_slices(tag, out[:, :n], F.avg_pool2d(x[:, :C * H * W].reshape(N, C, H, W).double(), 2).reshape(N, n), 2e-6)
            assert torch.isnan(out[:, n:]).all()
        elif kind == "mrb_conv_transpose2x2":
            x_bs, out_bs, N, Cin, Cout, H, W = a
            x, out = rows(N, x_bs), nan_rows(N, out_bs)
            w = torch.randn((Cin, Cout, 2, 2), device="cuda", generator=g) / Cin ** 0.5
            _lib.check(lib.mrb_conv_transpose2x2(_lib.ptr(x), x_bs, _lib.ptr(w), _lib.ptr(out), out_bs, N, Cin, Cout, H, W, st))
            n = Cout * 4 * H * W
            ref = F.conv_transpose2d(x[:, :Cin * H * W].reshape(N, Cin, H, W).double(), w.double(), stride=2)
            check_slices(tag, out[:, :n], ref.reshape(N, n), 2e-6)
            assert torch.isnan(out[:, n:]).all()
        elif kind == "mrb_conv1x1":
            x_bs, out_bs, N, Cin, Cout, HW = a
            x, out = rows(N, x_bs), nan_rows(N, out_bs)
            w = torch.randn((Cout, Cin), device="cuda", generator=g) / Cin ** 0.5
            b = torch.randn((Cout,), device="cuda", generator=g)
            _lib.check(lib.mrb_conv1x1(_lib.ptr(x), x_bs, _lib.ptr(w), _lib.ptr(b), _lib.ptr(out), out_bs, N, Cin, Cout, HW, st))
            ref = torch.einsum("oc,nch->noh", w.double(), x[:, :Cin * HW].reshape(N, Cin, HW).double()) + b.double()[:, None]
            check_slices(tag, out[:, :Cout * HW].reshape(N, Cout, HW), ref, 2e-6)
            assert torch.isnan(out[:, Cout * HW:]).all()
        elif kind == "mrb_normunet_in":
            B, C, HW, normalize = a
            x = rows(B, C * HW * 2, 2.0, 0.5)
            out = nan_rows(B, 2 * C * HW)
            ms = torch.empty((B, 2, 2), device="cuda")
            stats = torch.empty((4 * B,), dtype=torch.float64, device="cuda")
            _lib.check(lib.mrb_normunet_in(_lib.ptr(x), _lib.ptr(out), _lib.ptr(ms), B, C, HW, normalize, _lib.ptr(stats), st))
            planes = x.double().reshape(B, C * HW, 2).permute(0, 2, 1)  # [B, re | im, C * HW]
            if normalize:
                mean, std = planes.mean(-1, keepdim=True), planes.std(-1, keepdim=True)
                check_slices(tag + " mean/std", ms, torch.cat((mean, std), -1), 2e-6)
                planes = (planes - mean) / std
            check_slices(tag, out, planes.reshape(B, 2 * C * HW), 2e-6)
        elif kind == "mrb_normunet_out":
            B, C, HW, normalize = a
            x = rows(B, 2 * C * HW)
            ms = torch.stack((torch.randn((B, 2), device="cuda", generator=g),
                              torch.rand((B, 2), device="cuda", generator=g) + 0.5), -1).contiguous()  # (mean, std > 0)
            out = nan_rows(B, C * HW * 2)
            _lib.check(lib.mrb_normunet_out(_lib.ptr(x), _lib.ptr(ms), _lib.ptr(out), B, C, HW, normalize, st))
            planes = x.double().reshape(B, 2, C * HW)
            if normalize:
                planes = planes * ms[:, :, 1:].double() + ms[:, :, :1].double()
            check_slices(tag, out, planes.permute(0, 2, 1).reshape(B, -1), 2e-6)


# ---------------------------------------------------------------------------------------------- batch invariance
@pytest.mark.gpu
def test_batch_invariance_of_the_bench_workloads():
    """One process, in this order: CIRIM (bench weights and inputs) at 16 slices; every slice alone, twice (the second
    call replays the captured CUDA graph of the time loop); the 16 slices permuted; per-slice column masks [16, 1, 1, W, 1]
    against each slice run alone with its own mask; the brain-geometry CIRIM, E2EVN and brain-geometry E2EVN at 8 slices
    against each slice alone; CIRIM at 16 slices again.  Every estimate of every slice (all cascades and time steps for
    CIRIM) is bit-identical wherever the slice appears, so geometry-keyed caches (zero state, static hybrid k-space,
    graphs, packed weights) survive the changes of geometry in between."""
    from mridc_b200 import synth

    model, _, _ = _model("cirim_gru")
    model = model.cuda()
    host = _inputs("cirim_gru")
    y, S, m, tgt = _gpu(host)
    B = y.shape[0]
    base = _cirim_all(model, y, S, m, tgt)
    singles = 0
    for i in range(B):
        one = [t[i:i + 1].contiguous() for t in (y, S)] + [m, tgt[i:i + 1].contiguous()]  # the same tensors both calls
        for call in ("eager", "graph replay"):
            assert torch.equal(_cirim_all(model, *one), base[:, :, i:i + 1]), "CIRIM slice %d alone (%s)" % (i, call)
            singles += 1
    assert any(isinstance(gr, tuple) for blk in model.cirim for gr in blk._tc_engine._graphs.values())
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(5)).cuda()
    assert torch.equal(_cirim_all(model, y[perm], S[perm], m, tgt[perm]), base[:, :, perm]), "CIRIM permuted"
    print("[bench shapes] CIRIM 16 slices: %d single-slice runs and the permuted batch bit-identical" % singles)

    # per-slice column masks: the fully sampled k-space of each slice under its own mask, on the scale of the bench's y
    mf = synth.RandomMask1D([0.08], [4])
    mps = torch.stack([mf((1, 320, 320, 2), seed=s)[0].reshape(1, 1, 320, 1) for s in range(B)])  # [B, 1, 1, W, 1]
    k = host["kspace"]
    scale = host["y"].flatten(1).norm(dim=1) / (k * host["mask"]).flatten(1).norm(dim=1)
    yps = (k * mps * scale.view(-1, 1, 1, 1, 1)).cuda()
    mps = mps.to(torch.uint8).cuda()
    assert len(set(tuple(t.flatten().tolist()) for t in mps.cpu())) == B
    full = _cirim_all(model, yps, S, mps, tgt)
    for i in range(B):
        assert torch.equal(_cirim_all(model, yps[i:i + 1], S[i:i + 1], mps[i:i + 1], tgt[i:i + 1]), full[:, :, i:i + 1]), \
            "CIRIM per-slice masks, slice %d" % i
    del full, yps, mps

    for workload in ("brain_cirim", "e2evn", "brain_e2evn"):
        vn = None if workload == "brain_cirim" else _model(workload)[0].cuda()
        yb, Sb, mb, tb = _gpu(_inputs(workload))

        def run(i=None):  # -> [B, ...] (slices first); the whole batch, or slice i alone
            sel = slice(None) if i is None else slice(i, i + 1)
            if vn is not None:
                return vn(yb[sel], Sb[sel], mb, None, tb[sel])
            return _cirim_all(model, yb[sel], Sb[sel], mb, tb[sel]).movedim(2, 0)

        full = run()
        for i in range(yb.shape[0]):
            assert torch.equal(run(i), full[i:i + 1]), "%s slice %d alone" % (workload, i)
        print("[bench shapes] %s 8 slices: every slice alone bit-identical" % workload)
        del vn, full, yb, Sb, tb

    assert torch.equal(_cirim_all(model, y, S, m, tgt), base), "CIRIM 16 slices after the other geometries"
