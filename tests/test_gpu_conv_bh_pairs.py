"""mrb_tc_conv_bh (tc_kernel) on the geometries its work dealing creates, per slice against fp64 (split-bf16: 1e-5).

tc_kernel reads the A operand of tap (ky, kx) as one TMA box per (tile, kernel row) seen kx*dil rows further on through a
shifted SWIZZLE_128B descriptor, runs two consecutive 128-position tiles on each streamed weight chunk, and deals the
tiles left after the last full round of pairs partly as single tiles.  The rows below reach each of those cases:

  single taps      weights that are zero except at one tap: the output is one shifted product, so a wrong row shift or
                   swizzle phase of the descriptor shows up as a wrong tap instead of being averaged with correct ones;
  pair geometry    an odd tile count (the tail holds single tiles), pairs whose tiles lie in two slices, first and last
                   tiles whose boxes reach outside the tensor (zero-filled by TMA), at k = 3 / dil 1, k = 3 / dil 2, k = 5;
  batch invariance a slice alone and inside a batch of 16 (where it runs in pairs) gives the same bits.
"""
import pytest
import torch

from test_gpu_bench_shapes import check_slices


def _lib():
    from mridc_b200 import _lib

    return _lib, _lib.load(), _lib.stream_ptr()


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _conv(x, w, b, k, dil, relu=1):
    """fp32 NHWC x -> (raw BH output bytes, NCHW fp32 interior)"""
    L, lib, st = _lib()
    B, H, W, _ = x.shape
    xb = torch.empty(lib.mrb_bh_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    L.check(lib.mrb_bh_from_nhwc(L.ptr(x), L.ptr(xb), B, H, W, st))
    pk = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, k), device="cuda")
    L.check(lib.mrb_tc_pack_conv(L.ptr(w), L.ptr(pk), 64, 64, k, st))
    ob = torch.full((lib.mrb_bh_bytes(B, H, W),), 0x7F, dtype=torch.uint8, device="cuda")
    L.check(lib.mrb_tc_conv_bh(L.ptr(xb), L.ptr(pk), L.ptr(b), L.ptr(ob), B, H, W, 64, k, dil, relu, st))
    out = torch.empty((B, H, W, 64), device="cuda")
    L.check(lib.mrb_bh_to_nhwc(L.ptr(ob), L.ptr(out), B, H, W, st))
    return ob, out.permute(0, 3, 1, 2)


def _ref(x, w, b, k, dil, relu=True):
    from oracle import nets as onets

    return onets.conv_nonlinear(x.permute(0, 3, 1, 2).double(), w.double(), None if b is None else b.double(), k, dil,
                                "relu" if relu else None)


def _weights(g, k):
    return torch.randn((64, 64, k, k), device="cuda", generator=g) * (1.0 / (64 * k * k)) ** 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("k,dil", [(5, 1), (3, 2)])
def test_single_tap_reads_its_shifted_rows(k, dil):
    """One non-zero tap at a time, every tap of the kernel: the box row shift kx*dil takes every value 0..4 between the
    two geometries, i.e. every row phase of the 8-row swizzle pattern a tap can start at, and both halves (hi, lo)."""
    B, H, W = 3, 30, 37
    g = _gen(80 + k)
    x = torch.randn((B, H, W, 64), device="cuda", generator=g)
    full = _weights(g, k)
    b = torch.randn(64, device="cuda", generator=g)
    for ky in range(k):
        for kx in range(k):
            w = torch.zeros_like(full)
            w[:, :, ky, kx] = full[:, :, ky, kx] * k
            _, out = _conv(x, w, b, k, dil, relu=0)
            check_slices("tc_conv_bh k=%d dil=%d tap (%d, %d) only" % (k, dil, ky, kx), out, _ref(x, w, b, k, dil, False),
                         1e-5)


# (B, H, W): tile counts on both sides of the 148-CTA pair rounds
#   41 x 28 x 32: (H+4)(W+4) = 9 tiles per slice exactly, 369 tiles (odd): the pairs (8, 9), (26, 27), ... lie in two
#                 slices, one round of pairs and 73 single tiles;
#   2 x 320 x 320: 1641 tiles (odd), five rounds of pairs, then 13 pairs and 135 single tiles; tiles straddle slices;
#   3 x 64 x 100: 166 tiles, no full round: 18 pairs and 130 single tiles.
PAIR_SHAPES = [(41, 28, 32), (2, 320, 320), (3, 64, 100)]


@pytest.mark.gpu
@pytest.mark.parametrize("k,dil", [(3, 1), (3, 2), (5, 1)])
@pytest.mark.parametrize("B,H,W", PAIR_SHAPES)
def test_pair_geometry_per_slice(B, H, W, k, dil):
    g = _gen(90 + B + k + dil)
    x = torch.randn((B, H, W, 64), device="cuda", generator=g)
    w = _weights(g, k)
    b = torch.randn(64, device="cuda", generator=g)
    _, out = _conv(x, w, b, k, dil)
    check_slices("tc_conv_bh %dx%dx%d k=%d dil=%d" % (B, H, W, k, dil), out, _ref(x, w, b, k, dil), 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("k,dil", [(3, 2), (5, 1)])
def test_slice_alone_and_in_a_batch_of_16_give_the_same_bits(k, dil):
    """16 x 64 x 64 is 578 tiles (one round of pairs, then 134 pairs and 14 single tiles); one slice alone is 37 single
    tiles.  The interior of the BH output (the conv result, hi and lo) must match bit for bit."""
    B, H, W = 16, 64, 64
    g = _gen(120 + k)
    x = torch.randn((B, H, W, 64), device="cuda", generator=g)
    w = _weights(g, k)
    b = torch.randn(64, device="cuda", generator=g)
    ob, out = _conv(x, w, b, k, dil)
    check_slices("tc_conv_bh B=16 k=%d dil=%d" % (k, dil), out, _ref(x, w, b, k, dil), 1e-5)
    full = ob.view(torch.int16).reshape(B, H + 4, W + 4, 128)[:, 2:H + 2, 2:W + 2]
    for s in (0, 5, 15):
        one, _ = _conv(x[s:s + 1].contiguous(), w, b, k, dil)
        alone = one.view(torch.int16).reshape(1, H + 4, W + 4, 128)[0, 2:H + 2, 2:W + 2]
        assert torch.equal(alone, full[s]), "slice %d differs alone and inside the batch (k=%d dil=%d)" % (s, k, dil)
