"""CPU: the other consumers of the DC operator (SURVEY 8 (f) 2 / 4).

(1) The oracle restatement (oracle/consumers.py) against the committed reference vectors (tests/golden/consumers.npz,
    produced by the unmodified reference modules, oracle/make_golden.py::gen_consumers).
(2) Host logic of the product modules: their composition (axis handling, state-dict layout, signs, hidden-state plumbing)
    is run with the CUDA operator wrappers swapped for the oracle's CPU functions -- test scaffolding only, the package
    itself has no CPU path -- and compared with the same vectors.  The CUDA operators themselves are covered by the
    ``-m gpu`` twin of this file (tests/test_gpu_consumers.py).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from oracle import consumers as oc
from oracle import mri as omri

NRM3 = ["backward", "ortho", "forward"]
SD = [-2, -1]


def T(a):
    return torch.from_numpy(np.asarray(a))


def W(g, prefix):
    """weights stored as prefix + key.replace('.', '_')"""
    return {k[len(prefix):]: T(v) for k, v in g.items() if k.startswith(prefix)}


def load_sd(module, g, prefix):
    flat = W(g, prefix)
    sd = {k: flat[k.replace(".", "_")] for k in module.state_dict().keys()}
    module.load_state_dict(sd, strict=True)
    return sd


# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_sigmanet_layers_golden(golden):
    g = golden("consumers")
    for i in range(int(g["nsig"])):
        cen, nrm = bool(g["sig%d_cfg" % i][0]), NRM3[int(g["sig%d_cfg" % i][1])]
        x, y, S, m = (T(g["sig%d_%s" % (i, k)]) for k in ("x", "y", "smaps", "mask"))
        assert torch.allclose(oc.data_gd(x, y, S, m, 0.7, cen, nrm, SD), T(g["sig%d_gd" % i]), rtol=1e-6, atol=1e-6)
        assert torch.allclose(oc.data_vs(x, y, S, m, 0.3, 0.6, cen, nrm, SD), T(g["sig%d_vs" % i]), rtol=1e-6, atol=1e-6)
        if "sig%d_cg" % i in g:
            assert rel_l2(oc.prox_cg(x, 0.5, y, S, m, 1e-6, 6, cen, nrm, SD), g["sig%d_cg" % i]) < 1e-5
    x, y, S, m = (T(g["dun_" + k]) for k in ("x", "y", "smaps", "mask"))
    x1 = oc.data_gd(x, y, S, m, 0.4, True, "ortho", SD)
    assert x1.shape == g["dun_gd1"].shape == (3, 10, 12, 2)  # per-coil images after the first layer (dunet.py:186)
    assert torch.allclose(oc.data_gd(x1, y, S, m, 0.4, True, "ortho", SD), T(g["dun_gd2"]), rtol=1e-6, atol=1e-6)
    assert torch.allclose(oc.dc_layer(T(g["dcl_x"]), T(g["dcl_y"]), T(g["dcl_mask"]), 0.25, False, "ortho", SD),
                          T(g["dcl_out"]), rtol=1e-6, atol=1e-6)


def _ccnn_reg(g):
    w = W(g, "ccnn_w_")
    return lambda x: F.conv2d(F.relu(F.conv2d(x, w["0_weight"], w["0_bias"], padding=1)), w["2_weight"], w["2_bias"], padding=1)


def test_oracle_blocks_golden(golden):
    g = golden("consumers")
    reg = _ccnn_reg(g)
    for i, no_dc in enumerate((False, True)):
        pred, y, S, m = (T(g["ccnn%d_%s" % (i, k)]) for k in ("pred", "y", "S", "mask"))
        out = oc.cascadenet_block(reg, torch.tensor([0.8]), pred, y, S, m, True, "ortho", SD, 1, no_dc)
        assert rel_l2(out, g["ccnn%d_out" % i]) < 1e-6
    isd = {k: T(v) for k, v in ((k2, g["rvn_init_" + k2.replace(".", "_")]) for k2 in
                                ("conv_blocks.0.1.weight", "conv_blocks.0.1.bias", "conv_blocks.1.1.weight",
                                 "conv_blocks.1.1.bias", "out_blocks.0.0.weight", "out_blocks.0.0.bias",
                                 "out_blocks.1.0.weight", "out_blocks.1.0.bias"))}
    assert rel_l2(oc.recurrent_init(isd, (1, 2), 2, 2, T(g["rvn_img0"])), g["rvn_h0"]) < 1e-6


# ---------------------------------------------------------------------------------------------------------------------
class _OracleUtils:
    """oracle functions behind the signatures of mridc_b200.utils (test scaffolding)."""

    @staticmethod
    def complex_mul(x, y, _conj_y=False):
        return omri.complex_mul(x, omri.complex_conj(y) if _conj_y else y)

    complex_conj = staticmethod(omri.complex_conj)
    complex_abs = staticmethod(omri.complex_abs)


class _OracleOps:
    """oracle functions behind the signatures of mridc_b200._ops (test scaffolding)."""
    ACT_NONE, ACT_RELU, ACT_LEAKY, PAD_ZERO, PAD_REPLICATE = 0, 1, 2, 0, 1

    @staticmethod
    def check_spatial_dims(sd, ndim_complex=4):
        return None

    @staticmethod
    def sens_reduce(x, S, cen, nrm, out=None, ws=None):
        return omri.complex_mul(omri.ifft2(x, cen, nrm, SD), omri.complex_conj(S)).sum(1)

    @staticmethod
    def sens_expand_softdc(img, S, base, pred, y, mask, dc_weight, no_dc, cen, nrm, out=None, ws=None):
        B, C, H, Wd, _ = S.shape
        E = omri.fft2(omri.complex_mul(img.reshape(B, 1, H, Wd, 2), S), cen, nrm, SD)
        if no_dc:
            return E
        return base - torch.where(mask.bool(), pred - y, torch.zeros(1)) * dc_weight - E

    @staticmethod
    def conv2d(x, weight, bias, k, dil, pad_mode, act=0, **kw):
        p = dil * (k - 1) // 2
        x = F.pad(x, (p, p, p, p), mode="replicate" if pad_mode == 1 else "constant")
        out = F.conv2d(x, weight, bias, dilation=dil)
        return F.relu(out) if act == 1 else out


@pytest.fixture
def cpu_ops(monkeypatch):
    import mridc_b200._lib as lib
    import mridc_b200.cascadenet as cas
    import mridc_b200.data_consistency as dcm
    import mridc_b200.recurrentvarnet as rvn

    monkeypatch.setattr(lib, "require_cuda", lambda t, name="tensor", dtype=torch.float32: t)
    for mod in (dcm,):
        monkeypatch.setattr(mod, "fft", omri)
        monkeypatch.setattr(mod, "utils", _OracleUtils)
    for mod in (cas, rvn):
        monkeypatch.setattr(mod, "_ops", _OracleOps)
    return None


def test_host_logic_sigmanet_layers(golden, cpu_ops):
    import mridc_b200 as mb

    g = golden("consumers")
    for i in range(int(g["nsig"])):
        cen, nrm = bool(g["sig%d_cfg" % i][0]), NRM3[int(g["sig%d_cfg" % i][1])]
        x, y, S, m = (T(g["sig%d_%s" % (i, k)]) for k in ("x", "y", "smaps", "mask"))
        kw = dict(fft_centered=cen, fft_normalization=nrm, spatial_dims=SD)
        assert rel_l2(mb.DataGDLayer(0.7, **kw)(x, y, S, m), g["sig%d_gd" % i]) < 1e-6
        assert rel_l2(mb.DataVSLayer(0.3, 0.6, **kw)(x, y, S, m), g["sig%d_vs" % i]) < 1e-6
        if "sig%d_cg" % i in g:
            assert rel_l2(mb.DataProxCGLayer(0.5, tol=1e-6, iter=6, **kw)(x, y, S, m), g["sig%d_cg" % i]) < 1e-5
    x, y, S, m = (T(g["dun_" + k]) for k in ("x", "y", "smaps", "mask"))
    gd = mb.DataGDLayer(0.4, fft_centered=True, fft_normalization="ortho", spatial_dims=SD)
    assert rel_l2(gd(gd(x, y, S, m), y, S, m), g["dun_gd2"]) < 1e-6
    assert rel_l2(mb.DataVSLayer(0.2, 0.5)(x, y, S, m), g["dun_vs"]) < 1e-6
    dl = mb.DCLayer(0.25, fft_centered=False, fft_normalization="ortho", spatial_dims=SD)
    assert rel_l2(dl(T(g["dcl_x"]), T(g["dcl_y"]), T(g["dcl_mask"])), g["dcl_out"]) < 1e-6
    # parameter names of the reference modules
    assert list(mb.DataGDLayer(0.1).state_dict()) == ["data_weight"]
    assert list(mb.DataProxCGLayer(0.1).state_dict()) == ["lambdaa"]
    assert list(mb.DataVSLayer(0.1, 0.2).state_dict()) == ["alpha", "beta"]
    assert list(mb.DCLayer().state_dict()) == ["lambda_"]
    assert list(mb.DataIDLayer().state_dict()) == []


def test_host_logic_cascadenet_and_recurrentvarnet(golden, cpu_ops):
    import mridc_b200 as mb

    g = golden("consumers")

    class Reg(torch.nn.Module):
        def forward(self, x):
            return _ccnn_reg(g)(x)

    for i, no_dc in enumerate((False, True)):
        pred, y, S, m = (T(g["ccnn%d_%s" % (i, k)]) for k in ("pred", "y", "S", "mask"))
        blk = mb.CascadeNetBlock(Reg(), True, "ortho", SD, 1, no_dc)
        blk.dc_weight.data.fill_(0.8)
        assert rel_l2(blk(pred, y, S, m), g["ccnn%d_out" % i]) < 1e-6
    init = mb.RecurrentInit(2, 8, (8, 8), (1, 2), depth=2, multiscale_depth=2)
    load_sd(init, g, "rvn_init_")
    blk = mb.RecurrentVarNetBlock(2, 8, 2, True, "ortho", SD, 1)
    load_sd(blk, g, "rvn_blk_")
    y, S, m, cur = (T(g["rvn_" + k]) for k in ("y", "S", "mask", "cur"))
    h0 = init(T(g["rvn_img0"]))
    assert rel_l2(h0, g["rvn_h0"]) < 1e-6
    k1, h1 = blk(cur, y, m, S, h0)
    k2, h2 = blk(k1, y, m, S, h1)
    assert rel_l2(k1, g["rvn_k1"]) < 1e-6 and rel_l2(h1, g["rvn_h1"]) < 1e-6
    assert rel_l2(k2, g["rvn_k2"]) < 2e-6 and rel_l2(h2, g["rvn_h2"]) < 2e-6
    k1n, h1n = blk(cur, y, m, S, None)  # zero initial state
    assert rel_l2(k1n, g["rvn_k1n"]) < 1e-6 and rel_l2(h1n, g["rvn_h1n"]) < 1e-6


def test_initialisers_follow_the_reference_rng_order(golden):
    """Same seed => the reference's random-init weights (module construction order and initialisers), against the weights
    the reference modules drew for tests/golden (stored with '.' in the keys replaced by '_'): RecurrentInit followed by a
    RecurrentVarNetBlock from one seed, the NormUnet of a qVarNetBlock and the JRSCIRIM blocks."""
    import mridc_b200 as mb
    from oracle.make_golden import JRS_CASES, JRS_RIM

    def check(g, prefix, module, skip=()):
        keys = [k[len(prefix):] for k in g if k.startswith(prefix)]
        sd = module.state_dict()
        assert keys == [k.replace(".", "_") for k in sd], prefix
        for k, v in sd.items():
            if k not in skip:
                assert torch.equal(T(g[prefix + k.replace(".", "_")]), v), prefix + k

    g = golden("consumers")
    torch.manual_seed(6)
    init = mb.RecurrentInit(2, 8, (8, 8), (1, 2), depth=2, multiscale_depth=2)
    blk = mb.RecurrentVarNetBlock(2, 8, 2, True, "ortho", SD, 1)
    check(g, "rvn_init_", init)
    check(g, "rvn_blk_", blk, skip=("learning_rate",))  # set to 0.9 after construction
    torch.manual_seed(7)
    unet = mb.NormUnet(chans=4, num_pools=2, in_chans=8, out_chans=8, padding_size=3)
    check(g, "qvn_w_", mb.qVarNetBlock(unet, True, "ortho", SD, 2, False), skip=("dc_weight",))
    g = golden("jrscirim")
    for idx, (name, sp, in_ch, mag, slices) in enumerate(JRS_CASES):
        torch.manual_seed(40 + idx)
        check(g, "jrs%d_w_" % idx, mb.JRSCIRIMBlock(dict(JRS_RIM), dict(sp), in_ch, mag, True, "ortho", SD, 2, 2, slices,
                                                   "SENSE", True))


def test_oracle_jrscirim_golden(golden):
    """JRSCIRIMBlock restatement (CIRIM cascades + segmentation head) against the reference's own outputs."""
    from oracle.make_golden import JRS_CASES, JRS_RIM

    g = golden("jrscirim")
    hp = dict(JRS_RIM, fft_centered=True, fft_normalization="ortho", spatial_dims=SD, coil_dim=1)
    for idx, (name, sp, in_ch, mag, slices) in enumerate(JRS_CASES):
        p = "jrs%d_" % idx
        y, S, m, init, target = (T(g[p + k]) for k in ("y", "S", "mask", "init", "target"))
        sd = {k[len(p + "w_"):]: T(v) for k, v in g.items() if k.startswith(p + "w_")}
        # stored keys have '.' replaced by '_': rebuild the dotted names from a reference-shaped module
        import mridc_b200 as mb
        blk = mb.JRSCIRIMBlock(dict(JRS_RIM), dict(sp), in_ch, mag, True, "ortho", SD, 2, 2, slices, "SENSE", True)
        sd = {k: sd[k.replace(".", "_")] for k in blk.state_dict().keys()}
        no_init = torch.zeros(2, slices) if slices > 1 else torch.zeros(1)
        with torch.no_grad():
            rec, seg = oc.jrscirim_block(sd, hp, 2, True, "unet" if "UNet" in sp["segmentation_module"] else "conv", sp, in_ch,
                                         mag, slices, y, S, m, init if idx == 1 else no_init, target)
        rec = torch.view_as_real(torch.stack([torch.stack(c) for c in rec]))
        assert rel_l2(rec, g[p + "rec"]) < 1e-5, name
        assert rel_l2(seg, g[p + "seg"]) < 1e-4, name
