"""GPU: tensor-core (tcgen05 / TMEM, bf16 hi/lo split) RIM regulariser kernels against the CPU oracle and the
exact-fp32 CUDA-core kernels.  Tolerance: rel-L2 <= 1e-5 per operator: every operand is carried as hi + lo bf16
(16-17 significant bits) and a_lo*b_lo is dropped, ~3e-6 rms per product, plus the tensor core's truncating fp32
accumulation over the K chain.  Plain BF16 would sit at ~4e-3, plain TF32 at ~5e-4; the end-to-end budget is 1e-4
(rel-L2 on the reconstruction) and a CPU emulation of this arithmetic over CIRIM 5x8 lands at 2.5e-5."""
import numpy as np
import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu


def _diag(out_nchw, ref, tol, what):
    """rel-L2 check that reports where the error sits (pixels / channels) when it fails."""
    e = rel_l2(out_nchw, ref)
    print("[tc parity] %-16s rel-L2 %.2e (tol %.0e)" % (what, e, tol))  # visible with pytest -s
    if e >= tol:
        o = torch.as_tensor(out_nchw).detach().cpu().float()
        d = (o - ref).abs()
        idx = (d > 10 * tol * ref.abs().max()).nonzero()
        W = ref.shape[-1]
        msg = "%s: rel-L2 %.3e >= %.1e; %d bad elems; chans %s; pixels %s" % (
            what, e, tol, idx.shape[0], sorted(set(int(i[1]) for i in idx))[:64],
            sorted(set(int(i[2]) * W + int(i[3]) for i in idx))[:64])
        raise AssertionError(msg)


def _pack(w, k):
    from mridc_b200 import _lib

    lib = _lib.load()
    w = w.contiguous()
    p = torch.empty(lib.mrb_tc_packed_floats(0, w.shape[0], 64, k), device="cuda")
    _lib.check(lib.mrb_tc_pack_conv(_lib.ptr(w), _lib.ptr(p), w.shape[0], 64, k, _lib.stream_ptr()))
    return p


def test_dc_nhwc_layout_matches_nchw():
    from mridc_b200 import _ops

    g = torch.Generator(device="cuda").manual_seed(1)
    B, C, H, W = 2, 5, 24, 20
    y = torch.randn(B, C, H, W, 2, device="cuda", generator=g)
    S = torch.randn(B, C, H, W, 2, device="cuda", generator=g)
    eta = torch.randn(B, H, W, 2, device="cuda", generator=g)
    m = (torch.rand(1, 1, 1, W, 1, device="cuda", generator=g) < 0.5).float()
    a = _ops.dc_rim_grad(eta, y, S, m, 1.0, True, "ortho")
    b = _ops.dc_rim_grad(eta, y, S, m, 1.0, True, "ortho", nhwc=True)
    assert torch.equal(a, b.permute(0, 3, 1, 2))


@pytest.mark.parametrize("layer", ["GRU", "IndRNN"])
def test_rim_block_tc_vs_fp32_and_oracle(monkeypatch, layer):
    """The shipped geometries (64 filters, GRU or IndRNN with k=1): tensor-core engine == exact-fp32 kernels == oracle."""
    from mridc_b200 import synth
    from mridc_b200.rim import RIMBlock
    from mridc_b200.rim_tc import RimTcEngine
    from oracle import nets as onets

    cfg = synth.cirim_cfg(layer, centered=True, normalization="ortho")
    kw = {k: cfg[k] for k in ("recurrent_layer", "conv_filters", "conv_kernels", "conv_dilations", "conv_bias",
                              "recurrent_filters", "recurrent_kernels", "recurrent_dilations", "recurrent_bias",
                              "depth", "time_steps", "conv_dim", "no_dc", "fft_centered", "fft_normalization",
                              "spatial_dims", "coil_dim", "dimensionality")}
    torch.manual_seed(3)
    blk = RIMBlock(**kw).eval()
    with torch.no_grad():
        for st in blk.layers:
            st.convs.conv_layer.bias.normal_(0, 0.1)
            st.rnn.ih.bias.normal_(0, 0.1)
            if layer == "IndRNN":  # the default init (std 1/128) makes the recurrent term numerically invisible
                st.rnn.hh.normal_(0, 0.5)
                st.rnn.ih.weight.normal_(0, 0.1)
    sd = {k: v.detach().clone() for k, v in blk.state_dict().items()}
    batch = synth.make_batch(2, 6, 48, 40, centered=True, normalization="ortho")
    y, S, m = batch["y"], batch["sensitivity_maps"], batch["mask"]
    with torch.no_grad():
        ref, ref_h = onets.rim_block(sd, dict(cfg), y.clone(), y, S, m, None, None, 1.0, False)
    blk = blk.cuda()
    assert RimTcEngine.supported(blk)
    etas, hx = blk(y.cuda(), y.cuda(), S.cuda(), m.cuda(), None, None, 1.0, False)
    assert blk._tc_engine and len(etas) == 8
    assert hx[0].shape == (2, 64, 48, 40)
    for a, b in zip(etas, ref):  # 8 time steps of split-bf16 convs: ~3e-6 per operator, budget 3e-5 per block
        assert rel_l2(a, b) < 3e-5
    assert rel_l2(hx[0], ref_h[0]) < 3e-5 and rel_l2(hx[1], ref_h[1]) < 3e-5
    monkeypatch.setenv("MRIDC_B200_DISABLE_TC", "1")
    etas32, hx32 = blk(y.cuda(), y.cuda(), S.cuda(), m.cuda(), None, None, 1.0, False)
    assert rel_l2(etas[-1], etas32[-1]) < 3e-5 and rel_l2(hx[1], hx32[1]) < 3e-5
    # continuing from given hidden states (NCHW in, as the reference API)
    monkeypatch.delenv("MRIDC_B200_DISABLE_TC")
    e2, h2 = blk(etas, y.cuda(), S.cuda(), m.cuda(), None, [t.contiguous() for t in hx32], 1.0, True)
    with torch.no_grad():
        r2, _ = onets.rim_block(sd, dict(cfg), ref, y, S, m, None, [t.clone() for t in ref_h], 1.0, True)
    assert rel_l2(e2[-1], r2[-1]) < 5e-5


def _bh_roundtrip(x_nhwc):
    """fp32 [B,H,W,64] -> BH -> (raw BH view [B,H+4,W+4,128] bf16, fp32 back)"""
    from mridc_b200 import _lib

    lib = _lib.load()
    st = _lib.stream_ptr()
    B, H, W, _ = x_nhwc.shape
    bh = torch.empty(lib.mrb_bh_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    _lib.check(lib.mrb_bh_from_nhwc(_lib.ptr(x_nhwc), _lib.ptr(bh), B, H, W, st))
    back = torch.empty_like(x_nhwc)
    _lib.check(lib.mrb_bh_to_nhwc(_lib.ptr(bh), _lib.ptr(back), B, H, W, st))
    return bh, back


@pytest.mark.parametrize("B,H,W", [(1, 16, 8), (2, 37, 45), (2, 5, 100), (1, 320, 320)])
def test_tc2_gru_vs_oracle(B, H, W):
    """Second-generation GRU kernel (TMA + smem operands, BH activations): converters, cell arithmetic, replicate border."""
    from mridc_b200 import _lib
    from oracle import nets as onets

    lib = _lib.load()
    st = _lib.stream_ptr()
    g = torch.Generator().manual_seed(H + 1)
    x = torch.randn(B, 64, H, W, generator=g)
    h = torch.randn(B, 64, H, W, generator=g)
    wih = torch.randn(192, 64, 1, 1, generator=g) * 0.1
    whh = torch.randn(192, 64, 1, 1, generator=g) * 0.1
    bih = torch.randn(192, generator=g)
    ref = onets.conv_gru_cell(x, h, wih, bih, whh, 1, 1)
    xd, hd = x.permute(0, 2, 3, 1).contiguous().cuda(), h.permute(0, 2, 3, 1).contiguous().cuda()
    xb, xback = _bh_roundtrip(xd)
    hb, _ = _bh_roundtrip(hd)
    assert rel_l2(xback, xd) < 4e-6  # hi + lo carries 16-17 significant bits
    raw = xb.view(torch.bfloat16).view(B, H + 4, W + 4, 128).float()
    assert torch.equal(raw[:, 0, 0], raw[:, 2, 2]) and torch.equal(raw[:, -1, -1], raw[:, -3, -3])  # replicate border
    assert torch.equal(raw[:, 1, 5 % (W + 4)], raw[:, 2, min(max(5 % (W + 4), 2), W + 1)])
    wd, w2d, bd = wih.cuda().contiguous(), whh.cuda().contiguous(), bih.cuda()
    pk = torch.empty(lib.mrb_tc2_gru_packed_bytes(), dtype=torch.uint8, device="cuda")
    _lib.check(lib.mrb_tc2_pack_gru(_lib.ptr(wd), _lib.ptr(w2d), _lib.ptr(pk), 64, 64, st))
    ob = torch.full((lib.mrb_bh_bytes(B, H, W),), 0x7f, dtype=torch.uint8, device="cuda")  # poison: every byte must be written
    # garbage (NaN patterns) in the border of x must not reach any interior result
    xb.view(torch.bfloat16).view(B, H + 4, W + 4, 128)[:, :2] = float("nan")
    xb.view(torch.bfloat16).view(B, H + 4, W + 4, 128)[:, :, -2:] = float("nan")
    _lib.check(lib.mrb_tc2_gru(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pk), _lib.ptr(bd), _lib.ptr(ob), B, H, W, st))
    _lib.check(lib.mrb_bh_fix_border(_lib.ptr(ob), B, H, W, st))
    out = torch.empty_like(xd)
    _lib.check(lib.mrb_bh_to_nhwc(_lib.ptr(ob), _lib.ptr(out), B, H, W, st))
    _diag(out.permute(0, 3, 1, 2), ref, 1e-5, "gru (tc2)")
    rawo = ob.view(torch.bfloat16).view(B, H + 4, W + 4, 128).float()
    inner = rawo[:, 2:-2, 2:-2]
    pad = torch.nn.functional.pad(inner.permute(0, 3, 1, 2), (2, 2, 2, 2), mode="replicate").permute(0, 2, 3, 1)
    assert torch.equal(pad, rawo)  # the replicate border of the output is complete and exact
    # run-to-run determinism (eight launches at the full size, see the IndRNN twin below)
    for rep in range(8 if H >= 320 else 2):
        ob2 = torch.full_like(ob, 0x11 if rep % 2 else 0x7f)
        _lib.check(lib.mrb_tc2_gru(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pk), _lib.ptr(bd), _lib.ptr(ob2), B, H, W, st))
        _lib.check(lib.mrb_bh_fix_border(_lib.ptr(ob2), B, H, W, st))
        assert torch.equal(ob, ob2), rep


@pytest.mark.parametrize("B,H,W", [(1, 16, 8), (2, 37, 45), (1, 320, 320)])
def test_tc2_indrnn_vs_oracle(B, H, W):
    """IndRNN cell on BH activations (ind2_kernel): ReLU(W_ih x + b + hh * h), with and without bias; deterministic."""
    from mridc_b200 import _lib
    from oracle import nets as onets

    lib = _lib.load()
    st = _lib.stream_ptr()
    g = torch.Generator().manual_seed(W + 7)
    x = torch.randn(B, 64, H, W, generator=g)
    h = torch.randn(B, 64, H, W, generator=g)
    wih = torch.randn(64, 64, 1, 1, generator=g) * 0.1
    bih = torch.randn(64, generator=g)
    hh = torch.randn(1, 64, 1, 1, generator=g) * 0.5
    xb, _ = _bh_roundtrip(x.permute(0, 2, 3, 1).contiguous().cuda())
    hb, _ = _bh_roundtrip(h.permute(0, 2, 3, 1).contiguous().cuda())
    pk = _pack(wih.cuda(), 1)
    hhd = hh.reshape(-1).cuda()
    for bias in (bih, None):
        ref = onets.indrnn_cell(x, h, wih, bias, hh, 1, 1)
        bd = None if bias is None else bias.cuda()
        ob = torch.full((lib.mrb_bh_bytes(B, H, W),), 0x7f, dtype=torch.uint8, device="cuda")
        _lib.check(lib.mrb_tc2_indrnn(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pk), _lib.ptr(bd), _lib.ptr(hhd), _lib.ptr(ob), B, H, W,
                                      st))
        out = torch.empty(B, H, W, 64, device="cuda")
        _lib.check(lib.mrb_bh_to_nhwc(_lib.ptr(ob), _lib.ptr(out), B, H, W, st))
        _diag(out.permute(0, 3, 1, 2), ref, 1e-5, "indrnn (tc2)")
        # bit-reproducible run to run: eight launches (the refill of an h box once overtook the epilogue's last loads of it,
        # about one tile in 800 -- DESIGN 4.3)
        for rep in range(8 if H >= 320 else 2):
            ob2 = torch.full_like(ob, 0x11 if rep % 2 else 0x7f)
            _lib.check(lib.mrb_tc2_indrnn(_lib.ptr(xb), _lib.ptr(hb), _lib.ptr(pk), _lib.ptr(bd), _lib.ptr(hhd), _lib.ptr(ob2), B, H,
                                          W, st))
            assert torch.equal(ob, ob2), rep


@pytest.mark.parametrize("B,H,W", [(2, 37, 45), (1, 64, 32), (2, 33, 28), (1, 320, 320), (1, 12, 30)])
def test_tc2_bh_conv_ops_vs_oracle(B, H, W):
    """The convolutions of the time step on BH activations: conv5x5 (fp32 gradient -> G8 -> BH), conv3x3 (BH -> BH, replicate
    padding = the BH border), final conv (BH -> eta)."""
    from mridc_b200 import _lib
    from oracle import nets as onets

    lib = _lib.load()
    st = _lib.stream_ptr()
    g = torch.Generator().manual_seed(W)
    nb = lib.mrb_bh_bytes(B, H, W)

    def from_bh(buf):
        out = torch.empty(B, H, W, 64, device="cuda")
        _lib.check(lib.mrb_bh_to_nhwc(_lib.ptr(buf), _lib.ptr(out), B, H, W, st))
        return out.permute(0, 3, 1, 2)

    x4 = torch.randn(B, 4, H, W, generator=g)
    w1 = torch.randn(64, 4, 5, 5, generator=g) * 0.2
    b1 = torch.randn(64, generator=g)
    x4d, b1d = x4.permute(0, 2, 3, 1).contiguous().cuda(), b1.cuda()
    # bulk-copy-fed: fp32 gradient -> G8 -> BH, weights split on the fly, with and without bias / ReLU
    g8 = torch.zeros(lib.mrb_g8_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    _lib.check(lib.mrb_g8_from_nhwc4(_lib.ptr(x4d), _lib.ptr(g8), B, H, W, st))
    w1d = w1.cuda()
    for bias, relu in ((b1d, 1), (None, 0)):
        refg = onets.conv_nonlinear(x4, w1, None if bias is None else b1, 5, 1, "relu" if relu else None)
        ob = torch.full((nb,), 0x7f, dtype=torch.uint8, device="cuda")
        _lib.check(lib.mrb_tc2_conv5x5x4(_lib.ptr(g8), _lib.ptr(w1d), _lib.ptr(bias), _lib.ptr(ob), B, H, W, relu, st))
        _diag(from_bh(ob), refg, 1e-5, "conv5x5x4 (g8)")
        ob2 = torch.empty_like(ob)
        _lib.check(lib.mrb_tc2_conv5x5x4(_lib.ptr(g8), _lib.ptr(w1d), _lib.ptr(bias), _lib.ptr(ob2), B, H, W, relu, st))
        assert torch.equal(from_bh(ob), from_bh(ob2))

    x = torch.randn(B, 64, H, W, generator=g)
    xd = x.permute(0, 2, 3, 1).contiguous().cuda()
    xb, _ = _bh_roundtrip(xd)
    for dil, relu in ((2, 1), (1, 0)):
        w2 = torch.randn(64, 64, 3, 3, generator=g) * 0.05
        b2 = torch.randn(64, generator=g)
        ref = onets.conv_nonlinear(x, w2, b2, 3, dil, "relu" if relu else None)
        p2, b2d = _pack(w2.cuda(), 3), b2.cuda()
        ob = torch.full((nb,), 0x7f, dtype=torch.uint8, device="cuda")
        _lib.check(lib.mrb_tc_conv_bh(_lib.ptr(xb), _lib.ptr(p2), _lib.ptr(b2d), _lib.ptr(ob), B, H, W, 64, 3, dil, relu, st))
        _diag(from_bh(ob), ref, 1e-5, "conv3x3 dil %d (bh)" % dil)
        ob2 = torch.empty_like(ob)
        _lib.check(lib.mrb_tc_conv_bh(_lib.ptr(xb), _lib.ptr(p2), _lib.ptr(b2d), _lib.ptr(ob2), B, H, W, 64, 3, dil, relu, st))
        a_, b_ = from_bh(ob), from_bh(ob2)
        assert torch.equal(a_, b_)  # run-to-run determinism (interior)

    w3 = torch.randn(2, 64, 3, 3, generator=g) * 0.05
    eta = torch.randn(B, H, W, 2, generator=g)
    ref = eta + onets.conv_nonlinear(x, w3, None, 3, 1, None).permute(0, 2, 3, 1)
    o2 = torch.empty(B, H, W, 2, device="cuda")
    w3d, etad = w3.cuda(), eta.cuda()
    _lib.check(lib.mrb_conv_c2_bh_residual(_lib.ptr(xb), _lib.ptr(w3d), None, _lib.ptr(etad), _lib.ptr(o2), B, H, W, st))
    e = rel_l2(o2, ref)
    print("[tc parity] %-16s rel-L2 %.2e" % ("conv_c2 (bh)", e))
    assert e < 5e-6  # exact fp32 arithmetic on x = hi + lo (2^-18 relative representation error)
    # tensor-core tap GEMM + clamped gather: never reads the BH border (poisoned here), with and without bias
    xp = xb.clone()
    v = xp.view(torch.bfloat16).view(B, H + 4, W + 4, 128)
    v[:, :2] = float("nan"); v[:, -2:] = float("nan"); v[:, :, :2] = float("nan"); v[:, :, -2:] = float("nan")
    for bias in (None, torch.randn(2, generator=g)):
        refb = ref if bias is None else ref + bias
        o3 = torch.full((B, H, W, 2), float("nan"), device="cuda")
        bdev = None if bias is None else bias.cuda()
        bd = None if bias is None else _lib.ptr(bdev)
        _lib.check(lib.mrb_tc2_final_conv(_lib.ptr(xp), _lib.ptr(w3d), bd, _lib.ptr(etad), _lib.ptr(o3), B, H, W, st))
        e = rel_l2(o3, refb)
        print("[tc parity] %-16s rel-L2 %.2e" % ("final conv (tc2)", e))
        assert e < 1e-5
        o4 = torch.empty_like(o3)
        _lib.check(lib.mrb_tc2_final_conv(_lib.ptr(xp), _lib.ptr(w3d), bd, _lib.ptr(etad), _lib.ptr(o4), B, H, W, st))
        assert torch.equal(o3, o4)


@pytest.mark.parametrize("centered", [False, True])
def test_dc_direct_g8_output_equals_converter(centered):
    """The W = 320 row-form DC kernel writing the regulariser's G8 input itself (split + replicate border) == fp32 output
    followed by the converter, byte for byte (guards untouched)."""
    from mridc_b200 import _lib, _ops

    lib = _lib.load()
    B, C, H, W = 2, 5, 9, 320
    g = torch.Generator().manual_seed(11)
    y = torch.randn(B, C, H, W, 2, generator=g)
    S = torch.randn(B, C, H, W, 2, generator=g)
    eta = torch.randn(B, H, W, 2, generator=g)
    m = (torch.rand(1, 1, 1, W, 1, generator=g) < 0.3).float()
    y, S, eta, m = (y * m).cuda(), S.cuda(), eta.cuda(), m.cuda()
    yh = _ops.dc_hybrid_prepare(y, m, centered)
    g4 = _ops.dc_rim_grad(eta, y, S, m, 1.0, centered, "ortho", nhwc=True, y_hybrid=yh)
    ga = torch.zeros(lib.mrb_g8_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    _lib.check(lib.mrb_g8_from_nhwc4(_lib.ptr(g4), _lib.ptr(ga), B, H, W, _lib.stream_ptr()))
    gb = torch.zeros_like(ga)
    _ops.dc_rim_grad(eta, y, S, m, 1.0, centered, "ortho", out=gb, nhwc=2, y_hybrid=yh)
    assert torch.equal(ga, gb)
    assert int((ga != 0).sum()) > ga.numel() // 2


@pytest.mark.parametrize("N,Cin,Cout,H,W", [(2, 2, 14, 32, 48), (1, 14, 14, 37, 45), (2, 28, 56, 20, 24), (1, 56, 56, 16, 16),
                                            (2, 56, 28, 40, 40), (1, 64, 70, 12, 11), (1, 14, 14, 320, 320)])
def test_unet_conv3x3_tc_vs_oracle(N, Cin, Cout, H, W):
    """U-Net 3x3 conv (zero padding, no bias) on tcgen05: any channel counts up to 64 inputs, odd sizes, input read in place
    from a wider (concat) buffer, output written with a batch stride; run-to-run deterministic."""
    from mridc_b200 import _lib

    lib = _lib.load()
    st = _lib.stream_ptr()
    g = torch.Generator().manual_seed(Cin * 100 + Cout)
    xfull = torch.randn(N, Cin + 3, H, W, generator=g)
    w = torch.randn(Cout, Cin, 3, 3, generator=g) * (1.0 / (3.0 * Cin ** 0.5))
    ref = torch.nn.functional.conv2d(xfull[:, 3:], w, None, padding=1)
    xd, wraw = xfull.cuda(), w.cuda()
    wd = torch.empty(lib.mrb_tc2_unet_packed_bytes(Cin, Cout), dtype=torch.uint8, device="cuda")
    _lib.check(lib.mrb_tc2_unet_pack(_lib.ptr(wraw), _lib.ptr(wd), Cin, Cout, st))
    xv = xd[:, 3:]  # channels [3, 3 + Cin) of the wider buffer: batch stride (Cin + 3) H W
    outfull = torch.full((N, Cout + 2, H, W), float("nan"), device="cuda")
    ov = outfull[:, 2:]
    _lib.check(lib.mrb_tc2_unet_conv3x3(_lib.ptr(xv), (Cin + 3) * H * W, _lib.ptr(wd), _lib.ptr(ov), (Cout + 2) * H * W, N, Cin,
                                        Cout, H, W, st))
    _diag(ov, ref, 2e-6, "unet conv3x3 %d->%d" % (Cin, Cout))  # fp16 split: the tolerance of the fp32 kernels
    assert torch.isnan(outfull[:, :2]).all()  # nothing outside the destination channels is written
    o2 = torch.empty((N, Cout, H, W), device="cuda")
    _lib.check(lib.mrb_tc2_unet_conv3x3(_lib.ptr(xv), (Cin + 3) * H * W, _lib.ptr(wd), _lib.ptr(o2), Cout * H * W, N, Cin, Cout,
                                        H, W, st))
    assert torch.equal(o2, ov)


@pytest.mark.parametrize("B,H,W", [(1, 8, 32), (1, 12, 28), (3, 5, 40), (1, 12, 20)])
def test_cirim_tiny_images_on_the_bh_engine_or_the_fp32_loop(monkeypatch, B, H, W):
    """Images smaller than a tile / a TMA box (the final tap GEMM falls back to the CUDA-core kernel below 16 padded rows);
    below the engine's width of 28 the block runs the exact-fp32 loop."""
    import mridc_b200 as mb
    from mridc_b200 import synth
    from mridc_b200.rim_tc import RimTcEngine
    from oracle import models as omodels

    runs = []
    tc_run = RimTcEngine.run
    monkeypatch.setattr(RimTcEngine, "run", lambda self, *a, **k: runs.append(W) or tc_run(self, *a, **k))

    cfg = synth.cirim_cfg("GRU", num_cascades=1, centered=True, normalization="ortho")
    batch = synth.make_batch(B, 3, H, W, centered=True, normalization="ortho")
    torch.manual_seed(5)
    model = mb.CIRIM(cfg).eval()
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    with torch.no_grad():
        ref = omodels.cirim_forward(sd, cfg, batch["y"], batch["sensitivity_maps"], batch["mask"], None, batch["target"])
    out = next(model.cuda()(batch["y"].cuda(), batch["sensitivity_maps"].cuda(), batch["mask"].cuda(), None,
                            batch["target"].cuda()))
    e = rel_l2(out[-1][-1], ref[-1][-1])
    print("[tc parity] tiny CIRIM %dx%dx%d rel-L2 %.2e" % (B, H, W, e))
    assert e < 3e-5
    assert model.cirim[0]._tc_engine  # the block geometry is the engine's; only the width decides
    assert bool(runs) == (W >= 28)


def test_cirim_graph_replay_equals_eager(monkeypatch):
    """CUDA-graph replay of the time loop (third call with the same input tensors) == eager launches, bit for bit; new
    eta values, new k-space values in the same tensors and a different cascade state are all picked up."""
    import mridc_b200 as mb
    from mridc_b200 import synth

    cfg = synth.cirim_cfg("GRU", num_cascades=2)
    batch = synth.make_batch(2, 6, 64, 48)
    torch.manual_seed(4)
    model = mb.CIRIM(cfg).cuda().eval()
    y, S, m, tgt = (batch[k].cuda() for k in ("y", "sensitivity_maps", "mask", "target"))

    def run():
        return torch.stack([torch.stack(c) for c in next(model(y, S, m, None, tgt))])

    monkeypatch.setenv("MRIDC_B200_GRAPHS", "0")
    ref = run()
    monkeypatch.setenv("MRIDC_B200_GRAPHS", "auto")  # 2 x 64 x 48 pixels: launch-bound -> graphs
    a = run()   # eager (first sight of these tensors)
    b = run()   # captures + replays
    c = run()   # replays
    assert any(isinstance(g, tuple) for blk in model.cirim for g in blk._tc_engine._graphs.values())
    assert torch.equal(a, ref) and torch.equal(b, ref) and torch.equal(c, ref)
    y.mul_(0.5)  # same tensors, new contents
    d = run()
    monkeypatch.setenv("MRIDC_B200_GRAPHS", "0")
    assert torch.equal(d, run()) and not torch.equal(d, ref)
