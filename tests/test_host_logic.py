"""CPU: host-side logic of the drop-in layer (no compute calls): parameter/key compatibility with the reference,
initialiser parity, error behaviour, masks, sharding arithmetic."""
import numpy as np
import pytest
import torch

RIM_HP = dict(conv_filters=[16, 16, 2], conv_kernels=[5, 3, 3], conv_dilations=[1, 2, 1],
              conv_bias=[True, True, False], recurrent_filters=[16, 16, 0], recurrent_kernels=[1, 1, 0],
              recurrent_dilations=[1, 1, 0], recurrent_bias=[True, True, False])
LAYERS = ["GRU", "IndRNN", "MGU"]  # layer codes of the golden configs


def assert_reference_init(g, prefix, sd, skip=()):
    """`sd`, the state_dict of a module built right after torch.manual_seed(s), against the weights the reference module
    got from the same seed (stored under `prefix` by oracle/make_golden.py): same keys in the same order, same values bit
    for bit.  `skip` names parameters the generator overwrote after construction."""
    keys = [k[len(prefix):] for k in g if k.startswith(prefix)]
    assert keys == list(sd), prefix
    for k in keys:
        if k not in skip:
            assert torch.equal(torch.from_numpy(g[prefix + k]), sd[k]), prefix + k


def test_masks_bit_exact_vs_reference_golden(golden):
    from mridc_b200 import synth

    g = golden("masks")
    cases = [("random", synth.RandomMask1D, [0.08], [4], (1, 320, 320, 2), 123),
             ("random8", synth.RandomMask1D, [0.04], [8], (1, 640, 320, 2), 7),
             ("equi", synth.Equispaced1DMask, [0.08], [4], (1, 320, 320, 2), 123),
             ("equi8", synth.Equispaced1DMask, [0.04], [8], (1, 640, 320, 2), 123),
             ("equi_multi", synth.Equispaced1DMask, [0.08, 0.04], [4, 8], (1, 218, 170, 2), (1, 2, 3))]
    for name, cls, cf, acc, shape, seed in cases:
        m, a = cls(cf, acc)(shape, seed)
        assert m.dtype == torch.float32 and tuple(m.shape) == g[name].shape
        assert np.array_equal(m.numpy(), g[name]), name
        assert a == int(g[name + "_acc"])
    for name, acc in (("gauss4", 4), ("gauss8", 8)):
        np.random.seed(123)
        m, _ = synth.Gaussian1DMask([0.7], [acc])((1, 320, 320, 2), 0, scale=0.02)
        assert np.array_equal(m.numpy(), g[name]), name
        assert abs(m.mean().item() - 1.0 / acc) < 0.05
    # seeded masks do not disturb the generator's state and are reproducible
    f = synth.Equispaced1DMask([0.08], [4])
    assert torch.equal(f((1, 64, 64, 2), 5)[0], f((1, 64, 64, 2), 5)[0])
    with pytest.raises(ValueError):
        synth.RandomMask1D([0.08], [4, 8])


def test_state_dict_keys_match_reference_layout(golden):
    """Reference state_dicts (stored in the golden files) load strictly into the drop-in modules."""
    import mridc_b200 as mb

    g = golden("rim")
    blk = mb.RIMBlock(recurrent_layer="GRU", depth=2, time_steps=8, conv_dim=2, no_dc=True, **RIM_HP)
    blk.load_state_dict(golden.weights(g, "rim0_w_"), strict=True)
    assert sorted(blk.state_dict()) == sorted(golden.weights(g, "rim0_w_"))
    blk = mb.RIMBlock(recurrent_layer="IndRNN", depth=2, time_steps=8, conv_dim=2, no_dc=True, **RIM_HP)
    blk.load_state_dict(golden.weights(g, "rim2_w_"), strict=True)
    blk = mb.RIMBlock(recurrent_layer="GRU", depth=2, time_steps=8, conv_dim=2, no_dc=False, **RIM_HP)
    assert "dc_weight" in blk.state_dict()
    g = golden("unet_vn")
    vb = mb.VarNetBlock(mb.NormUnet(chans=4, num_pools=2, padding_size=11))
    vb.load_state_dict(golden.weights(g, "vn0_w_"), strict=True)
    full = mb.CIRIM(dict(RIM_HP, recurrent_layer="GRU", depth=2, time_steps=5, conv_dim=2, no_dc=True,
                         num_cascades=3, dimensionality=2, keep_eta=True, fft_centered=False,
                         fft_normalization="backward", spatial_dims=[-2, -1], coil_dim=1,
                         coil_combination_method="SENSE"))
    assert full.time_steps == 8  # rounded up to a multiple of 8 (cirim.py:51)
    keys = set(full.state_dict())
    assert "dc_weight" in keys and "cirim.2.layers.1.rnn.hh.weight" in keys
    assert "cirim.0.final_layer.0.conv_layer.weight" in keys and "cirim.0.final_layer.0.conv_layer.bias" not in keys
    # SURVEY 8a: 94,080 parameters per GRU cascade at 64 filters
    big = mb.RIMBlock(recurrent_layer="GRU", conv_filters=[64, 64, 2], conv_kernels=[5, 3, 3],
                      conv_dilations=[1, 2, 1], conv_bias=[True, True, False], recurrent_filters=[64, 64, 0],
                      recurrent_kernels=[1, 1, 0], recurrent_dilations=[1, 1, 0], recurrent_bias=[True, True, False],
                      depth=2, time_steps=8, conv_dim=2, no_dc=True)
    assert sum(p.numel() for p in big.parameters()) == 94080
    vn = mb.VarNetBlock(mb.NormUnet(chans=14, num_pools=2, padding_size=11))
    assert sum(p.numel() for p in vn.parameters()) == 89267


def test_initialisers_reproduce_reference_weights(golden):
    """Same seed -> same random-init weights as the reference modules (same init calls in the same order): every RIMBlock
    (GRU / IndRNN / MGU, 2-D and 3-D), NormUnet and VarNetBlock whose reference weights are stored in tests/golden."""
    import mridc_b200 as mb
    from oracle.make_golden import RIM_HP as GOLDEN_RIM_HP

    g = golden("rim")
    for i in range(int(g["nrim"])):
        layer, rk, no_dc = (int(v) for v in g["rim%d_cfg" % i][:3])
        torch.manual_seed(1 + i)
        blk = mb.RIMBlock(**dict(GOLDEN_RIM_HP, recurrent_layer=LAYERS[layer], recurrent_kernels=[rk, rk, 0],
                                 no_dc=bool(no_dc)))
        assert_reference_init(g, "rim%d_w_" % i, blk.state_dict())
    g = golden("rim3d")
    for i in range(int(g["nrim"])):
        layer, steps = int(g["rim%d_cfg" % i][0]), int(g["rim%d_cfg" % i][3])
        torch.manual_seed(40 + i)
        blk = mb.RIMBlock(**dict(GOLDEN_RIM_HP, recurrent_layer=LAYERS[layer], no_dc=True, time_steps=steps, conv_dim=3,
                                 dimensionality=3))
        assert_reference_init(g, "rim%d_w_" % i, blk.state_dict())
    g = golden("unet_vn")
    for i in range(int(g["nunet"])):
        chans, pools, padsz = (int(v) for v in g["unet%d_cfg" % i])
        torch.manual_seed(5 + i)
        assert_reference_init(g, "unet%d_w_" % i, mb.NormUnet(chans=chans, num_pools=pools, padding_size=padsz).state_dict())
    for j in range(int(g["nvn"])):
        torch.manual_seed(40 + j)
        vb = mb.VarNetBlock(mb.NormUnet(chans=4, num_pools=2, padding_size=11), no_dc=bool(g["vn%d_cfg" % j][2]))
        assert_reference_init(g, "vn%d_w_" % j, vb.state_dict(), skip=("dc_weight",))  # set to 0.7 after construction


def test_error_behaviour_matches_reference_texts():
    import mridc_b200 as mb

    x = torch.zeros(2, 3, 4, 2)
    with pytest.raises(ValueError, match="Tensors do not have separate complex dim."):
        mb.complex_mul(x[..., :1], x)
    with pytest.raises(ValueError, match="Tensor does not have separate complex dim."):
        mb.complex_conj(x[..., :1])
    with pytest.raises(ValueError, match="Output type not supported."):
        mb.coil_combination(x, x, method="espirit")
    with pytest.raises(ValueError, match="len\\(shift\\) must match len\\(dim\\)"):
        mb.roll(x, [1], [0, 1])
    with pytest.raises(ValueError, match="Invalid shapes."):
        mb.center_crop(x, (9, 1))
    with pytest.raises(ValueError, match="Please specify a proper recurrent layer type."):
        mb.RIMBlock(recurrent_layer="LSTM", depth=2, conv_dim=2, **RIM_HP)
    with pytest.raises(ValueError, match="Please specify a proper nonlinearity"):
        mb.ConvNonlinear(4, 8, 2, 3, 1, True, "gelu")
    # no CPU fallback anywhere on the compute path
    for fn in (lambda: mb.fft2(x), lambda: mb.ifft2(x), lambda: mb.complex_abs(x), lambda: mb.rss(x, 1),
               lambda: mb.sense(x, x, 1), lambda: mb.fftshift(x)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn()
    # crops are pure index arithmetic and work on any device, bit exact
    a = torch.arange(6 * 8).reshape(6, 8)
    assert torch.equal(mb.center_crop(a, (2, 4)), a[2:4, 2:6])
    assert torch.equal(mb.check_stacked_complex(x), torch.view_as_complex(x))


def test_partition_and_shard_arithmetic():
    from mridc_b200 import sharding

    assert sharding.partition(10, 4) == [(0, 3), (3, 6), (6, 9), (9, 10)]
    assert sharding.partition(8, 8) == [(i, i + 1) for i in range(8)]
    assert sharding.partition(3, 8)[3:] == [(3, 3)] * 5
    assert sharding.partition(0, 2) == [(0, 0), (0, 0)]
    for n in range(0, 40):
        for w in (1, 2, 3, 8):
            p = sharding.partition(n, w)
            assert p[0][0] == 0 and p[-1][1] == n and all(a[1] == b[0] for a, b in zip(p, p[1:]))
    y = torch.arange(10).reshape(10, 1)
    m = torch.ones(1, 5)
    (ys, ms, none), (a, b) = sharding.shard_slices([y, m, None], rank=1, world_size=4)
    assert (a, b) == (3, 6) and torch.equal(ys, y[3:6]) and ms is m and none is None
    with pytest.raises(ValueError):
        sharding.partition(4, 0)


def test_synth_batch_shapes_and_determinism():
    from mridc_b200 import synth

    b1 = synth.make_batch(2, 4, 32, 24, centered=True, normalization="ortho")
    b2 = synth.make_batch(2, 4, 32, 24, centered=True, normalization="ortho")
    assert b1["y"].shape == (2, 4, 32, 24, 2) and b1["mask"].shape == (1, 1, 1, 24, 1)
    assert b1["mask"].dtype == torch.uint8 and b1["target"].dtype == torch.complex64
    assert all(torch.equal(b1[k], b2[k]) for k in ("y", "sensitivity_maps", "mask", "target"))
    # masked columns of y are exactly zero; sampled ones are not
    m = b1["mask"].bool().reshape(-1)
    assert torch.count_nonzero(b1["y"][..., ~m, :]) == 0 and torch.count_nonzero(b1["y"][..., m, :]) > 0
    assert not torch.equal(b1["y"][0], b1["y"][1])


def test_host_prefetcher_rejects_cpu_device():
    import pytest
    import mridc_b200 as mb

    with pytest.raises(RuntimeError, match="CUDA device"):
        mb.HostPrefetcher([], "cpu")


def test_qcirim_ctor_errors():
    import mridc_b200 as mb
    from mridc_b200 import synth

    with pytest.raises(ValueError, match="Only 2D is currently supported"):
        mb.qCIRIM(dict(synth.qcirim_cfg(filters=8), quantitative_module_dimensionality=3))
    with pytest.raises(ValueError, match="does not support explicit DC"):
        mb.qCIRIM(dict(synth.qcirim_cfg(filters=8), quantitative_module_no_dc=False))
    with pytest.raises(NotImplementedError):
        mb.qCIRIM(dict(synth.qcirim_cfg(filters=8), use_reconstruction_module=True))
    # no CPU fallback on the quantitative path either
    m = torch.zeros(1, 4, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mb.SignalForwardModel("MEGRE")(m, m, m, m)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mb.RescaleByMax.reverse(torch.zeros(1, 4, 4, 4), torch.ones(4))


def test_qrim_initialisers_reproduce_reference_weights(golden):
    """qRIMBlock (GRU / IndRNN / MGU) and the cascades of qCIRIM against the reference weights stored in tests/golden."""
    import mridc_b200 as mb
    from oracle.make_golden import QRIM_HP, oqnets_cfg

    g = golden("qmri")
    hp = {k: v for k, v in QRIM_HP.items() if k != "time_steps"}
    for i in range(int(g["nblk"])):
        torch.manual_seed(40 + i)
        blk = mb.qRIMBlock(recurrent_layer=LAYERS[int(g["blk%d_cfg" % i][0])], depth=2, time_steps=QRIM_HP["time_steps"],
                           conv_dim=2, no_dc=True, linear_forward_model=mb.SignalForwardModel(sequence="MEGRE"), **hp)
        assert_reference_init(g, "blk%d_w_" % i, blk.state_dict())
    torch.manual_seed(77)
    assert_reference_init(g, "model_w_", mb.qCIRIM(oqnets_cfg(num_cascades=2)).state_dict())


def test_sens_net_initialiser_and_bookkeeping_match_reference(golden):
    """BaseSensitivityModel against the reference's weights and low-frequency bookkeeping stored in tests/golden; a VarNet
    with use_sens_net builds that network first (base.py:81-94), so it draws the same weights from the same seed."""
    import mridc_b200 as mb
    from mridc_b200 import synth
    from oracle import nets as onets

    g = golden("sens")
    for i in range(int(g["nsens"])):
        chans, pools, mtype, _, _, normalize, mcenter, nlf = (int(v) for v in g["sens%d_cfg" % i])
        kw = dict(mask_type=["1D", "2D"][mtype], normalize=bool(normalize), mask_center=bool(mcenter))
        torch.manual_seed(60 + i)
        assert_reference_init(g, "sens%d_w_" % i, mb.BaseSensitivityModel(chans, pools, **kw).state_dict())
        cfg = dict(synth.varnet_cfg(num_cascades=1), use_sens_net=True, sens_chans=chans, sens_pools=pools,
                   sens_mask_type=kw["mask_type"], sens_normalize=kw["normalize"], sens_mask_center=kw["mask_center"])
        torch.manual_seed(60 + i)
        sd = mb.VarNet(cfg).state_dict()
        assert_reference_init(g, "sens%d_w_" % i, {k[len("sens_net."):]: v for k, v in sd.items() if k.startswith("sens_net.")})
        pad, n = mb.BaseSensitivityModel.get_pad_and_num_low_freqs(torch.from_numpy(g["sens%d_mask" % i]),
                                                                   None if nlf < 0 else nlf)
        assert np.array_equal(pad.numpy(), g["sens%d_pad" % i]) and np.array_equal(n.numpy(), g["sens%d_nlf" % i]), i
    # more masks and low-frequency counts: the restatement, pinned to the same stored vectors by test_oracle_golden.py
    gen = torch.Generator().manual_seed(3)
    for _ in range(5):
        m = (torch.rand(3, 1, 1, 24, 1, generator=gen) < 0.5).float()
        m[:, 0, 0, 10:14, 0] = 1
        for nlf in (None, 0, 4):
            pa, na = onets.sens_pad_and_num_low_freqs(m, nlf)
            pb, nb = mb.BaseSensitivityModel.get_pad_and_num_low_freqs(m, nlf)
            assert torch.equal(pa, pb) and torch.equal(na, nb)


def _replay_apply_mask(golden, device):
    """tests/golden/apply_mask.npz (oracle/make_golden.py::gen_apply_mask): the reference's apply_mask
    (common/parts/utils.py:293-343) on seeded k-space -- data, mask and acceleration must come back bit for bit,
    including the cleared sign of zeros (":341 + 0.0"), the padding zeroing (:332-335) and the mask fftshift (:337-338)."""
    from mridc_b200 import synth, utils as mutils

    g = golden("apply_mask")
    for i in range(int(g["nam"])):
        kind, shift = (int(v) for v in g["am%d_cfg" % i])
        cf, acc = [float(v) for v in g["am%d_cf" % i]], [int(v) for v in g["am%d_accs" % i]]
        seed = g["am%d_seed" % i]
        seed = int(seed) if seed.ndim == 0 else tuple(int(v) for v in seed)
        pad = tuple(int(v) for v in g["am%d_pad" % i])
        pad = None if pad == (-1, -1) else pad
        if kind == 2:  # 2-D equispaced mask drawn by the reference, replayed through a fixed mask function
            raw, racc = torch.from_numpy(g["am%d_raw" % i]), float(g["am%d_acc" % i])

            def fn(shape, seed, half_scan_percentage=0.0, scale=0.02, _m=raw, _a=racc):
                return _m.clone(), _a
        else:
            fn = (synth.Equispaced1DMask if kind == 0 else synth.RandomMask1D)(cf, acc)
        data = torch.from_numpy(g["am%d_in" % i]).to(device)
        out, mask, a = mutils.apply_mask(data, fn, seed=seed, padding=pad, shift=bool(shift))
        assert out.device == data.device and mask.device == data.device
        ref = torch.from_numpy(g["am%d_out" % i])
        assert torch.equal(out.cpu(), ref), i
        assert torch.equal(torch.signbit(out.cpu()), torch.signbit(ref)), i
        assert torch.equal(mask.cpu(), torch.from_numpy(g["am%d_mask" % i])), i
        assert float(a) == float(g["am%d_acc" % i]), i


def test_apply_mask_golden(golden):
    _replay_apply_mask(golden, "cpu")
