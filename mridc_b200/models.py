"""Drop-ins for the reconstruction models named by the north star: CIRIM, VarNet (E2EVN), UNet, ZF.

Constructor ``Model(cfg, trainer=None)`` reads the same flat cfg keys as the reference and ``forward`` has the
same signature and return structure (CIRIM.forward is a *generator*, as in the reference).  Only the inference
path is implemented: the Lightning/NeMo base class (training steps, losses, data loaders, exp-manager) is out
of scope (SURVEY.md section 2, rows 9/17) -- ``trainer`` is accepted and ignored, loss keys are not read.

  CIRIM   mridc/collections/reconstruction/models/cirim.py:25-197
  VarNet  mridc/collections/reconstruction/models/vn.py:22-142
  UNet    mridc/collections/reconstruction/models/unet.py:21-121
  ZF      mridc/collections/reconstruction/models/zf.py:20-100
  PICS    mridc/collections/reconstruction/models/pics.py (BART `pics`; here FISTA on the GPU, mridc_b200.pics)
  qCIRIM  mridc/collections/quantitative/models/qcirim.py:21-341 (quantitative module; BASELINE.json configs[4])
"""
import math
from typing import Any, Generator, List, Mapping, Union

import torch
import torch.nn as nn

from . import _lib, _ops, pics, utils
from .qrim import RescaleByMax, SignalForwardModel, qRIMBlock
from .rim import RIMBlock
from .sensitivity import BaseSensitivityModel
from .unet import NormUnet
from .varnet import VarNetBlock

__all__ = ["CIRIM", "VarNet", "UNet", "ZF", "PICS", "qCIRIM"]


def _cfg_dict(cfg) -> dict:
    if isinstance(cfg, Mapping):
        return dict(cfg)
    try:  # OmegaConf DictConfig without importing omegaconf
        return dict(cfg.items())
    except Exception as exc:
        raise TypeError("cfg must be a mapping (dict / DictConfig)") from exc


def _listify(v):
    return list(v) if v is not None and not isinstance(v, (int, float, str, bool)) else v


class _BaseModel(nn.Module):
    """Inference-only stand-in for BaseMRIReconstructionModel(ModelPT) (reconstruction/models/base.py:56)."""

    def __init__(self, cfg, trainer=None):
        super().__init__()
        self._cfg = _cfg_dict(cfg)
        self.trainer = trainer
        # base.py:81-94: the sensitivity network is built by the base class, i.e. BEFORE the cascades (same RNG order).
        # As in the reference it is applied by the caller of ``forward`` (``sensitivity_maps = model.sens_net(kspace,
        # mask)``, base.py:234-235 / :300-301 / :392-393), not inside it.
        self.use_sens_net = self._cfg.get("use_sens_net")
        if self.use_sens_net:
            c = self._cfg
            self.sens_net = BaseSensitivityModel(
                c.get("sens_chans"), c.get("sens_pools"), fft_centered=c.get("fft_centered"),
                fft_normalization=c.get("fft_normalization"), spatial_dims=_listify(c.get("spatial_dims")),
                coil_dim=c.get("coil_dim"), mask_type=c.get("sens_mask_type"), normalize=c.get("sens_normalize"),
                mask_center=c.get("sens_mask_center"))

    @property
    def cfg(self):
        return self._cfg


class CIRIM(_BaseModel):
    """Cascades of Independently Recurrent Inference Machines, cirim.py:25."""

    def __init__(self, cfg, trainer=None):
        super().__init__(cfg, trainer)
        c = self._cfg
        self.recurrent_filters = _listify(c.get("recurrent_filters"))
        self.time_steps = 8 * math.ceil(c.get("time_steps") / 8)  # cirim.py:51
        self.no_dc = c.get("no_dc")
        self.fft_centered = c.get("fft_centered")
        self.fft_normalization = c.get("fft_normalization")
        self.spatial_dims = _listify(c.get("spatial_dims"))
        self.coil_dim = c.get("coil_dim")
        self.num_cascades = c.get("num_cascades")
        self.cirim = nn.ModuleList([
            RIMBlock(
                recurrent_layer=c.get("recurrent_layer"),
                conv_filters=_listify(c.get("conv_filters")),
                conv_kernels=_listify(c.get("conv_kernels")),
                conv_dilations=_listify(c.get("conv_dilations")),
                conv_bias=_listify(c.get("conv_bias")),
                recurrent_filters=self.recurrent_filters,
                recurrent_kernels=_listify(c.get("recurrent_kernels")),
                recurrent_dilations=_listify(c.get("recurrent_dilations")),
                recurrent_bias=_listify(c.get("recurrent_bias")),
                depth=c.get("depth"),
                time_steps=self.time_steps,
                conv_dim=c.get("conv_dim"),
                no_dc=self.no_dc,
                fft_centered=self.fft_centered,
                fft_normalization=self.fft_normalization,
                spatial_dims=self.spatial_dims,
                coil_dim=self.coil_dim,
                dimensionality=c.get("dimensionality"),
            )
            for _ in range(self.num_cascades)
        ])
        self.keep_eta = c.get("keep_eta")
        self.coil_combination_method = c.get("coil_combination_method")
        # cirim.py:92-94: rnn_weights_init touches only Linear/Embedding/LayerNorm -> a no-op for these convs
        self.dc_weight = nn.Parameter(torch.ones(1))  # cirim.py:112 (unused by forward, kept for checkpoints)
        self.accumulate_estimates = True

    @torch.no_grad()
    def forward(self, y: torch.Tensor, sensitivity_maps: torch.Tensor, mask: torch.Tensor, init_pred: torch.Tensor,
                target: torch.Tensor) -> Union[Generator, torch.Tensor]:
        """cirim.py:115-165 -- yields list[num_cascades] of list[time_steps] of complex [B, h, w]."""
        _lib.require_cuda(y, "y")
        prediction = y  # cirim.py:146 clones; nothing below mutates y, so the copy is not needed
        init_pred = None if init_pred is None or init_pred.dim() < 4 else init_pred
        hx = None
        sigma = 1.0
        cascades_etas = []
        y = y.contiguous()
        hybrid_cache = {}  # hybrid-space k-space of y: prepared by the first cascade, reused by the others
        for i, cascade in enumerate(self.cirim):
            prediction, _ = cascade(prediction, y, sensitivity_maps, mask, init_pred, hx, sigma,
                                    keep_eta=False if i == 0 else self.keep_eta, y_hybrid=hybrid_cache, want_hx=False)
            cascades_etas.append([self.process_intermediate_pred(pred, sensitivity_maps, target)
                                  for pred in prediction])
        yield cascades_etas

    def process_intermediate_pred(self, pred, sensitivity_maps, target, do_coil_combination=False):
        """cirim.py:167-197."""
        if not self.no_dc or do_coil_combination:
            if self.coil_combination_method == "SENSE" and self.coil_dim == 1:
                _ops.check_spatial_dims(self.spatial_dims)
                pred = _ops.sens_reduce(pred, sensitivity_maps, self.fft_centered, self.fft_normalization)
            else:
                from . import fft as _fft
                pred = _fft.ifft2(pred, centered=self.fft_centered, normalization=self.fft_normalization,
                                  spatial_dims=self.spatial_dims)
                pred = utils.coil_combination(pred, sensitivity_maps, method=self.coil_combination_method,
                                              dim=self.coil_dim)
        pred = torch.view_as_complex(pred)
        _, pred = utils.center_crop_to_smallest(target, pred)
        return pred


def _ifft_combine(y, sensitivity_maps, method, centered, normalization, spatial_dims, coil_dim):
    """ifft2 + coil_combination: one fused operator for SENSE, two kernels for RSS."""
    if method == "SENSE" and coil_dim == 1 and y.dim() == 5:
        _ops.check_spatial_dims(spatial_dims)
        return _ops.sens_reduce(y, sensitivity_maps, centered, normalization)
    from . import fft as _fft
    img = _fft.ifft2(y, centered=centered, normalization=normalization, spatial_dims=spatial_dims)
    return utils.coil_combination(img, sensitivity_maps, method=method, dim=coil_dim)


class VarNet(_BaseModel):
    """End-to-End Variational Network, vn.py:22."""

    def __init__(self, cfg, trainer=None):
        super().__init__(cfg, trainer)
        c = self._cfg
        self.no_dc = c.get("no_dc")
        self.fft_centered = c.get("fft_centered")
        self.fft_normalization = c.get("fft_normalization")
        self.spatial_dims = _listify(c.get("spatial_dims"))
        self.coil_dim = c.get("coil_dim")
        self.num_cascades = c.get("num_cascades")
        self.cascades = nn.ModuleList([
            VarNetBlock(
                NormUnet(chans=c.get("channels"), num_pools=c.get("pooling_layers"),
                         padding_size=c.get("padding_size"), normalize=c.get("normalize")),
                fft_centered=self.fft_centered, fft_normalization=self.fft_normalization,
                spatial_dims=self.spatial_dims, coil_dim=self.coil_dim, no_dc=self.no_dc)
            for _ in range(self.num_cascades)
        ])
        self.coil_combination_method = c.get("coil_combination_method")
        self.dc_weight = nn.Parameter(torch.ones(1))  # vn.py:91
        self.accumulate_estimates = False

    @torch.no_grad()
    def forward(self, y: torch.Tensor, sensitivity_maps: torch.Tensor, mask: torch.Tensor, init_pred: torch.Tensor,
                target: torch.Tensor) -> torch.Tensor:
        """vn.py:94-142."""
        _lib.require_cuda(y, "y")
        estimation = y
        for cascade in self.cascades:
            estimation = cascade(estimation, y, sensitivity_maps, mask)
        estimation = _ifft_combine(estimation, sensitivity_maps, self.coil_combination_method, self.fft_centered,
                                   self.fft_normalization, self.spatial_dims, self.coil_dim)
        estimation = torch.view_as_complex(estimation)
        _, estimation = utils.center_crop_to_smallest(target, estimation)
        return estimation


class UNet(_BaseModel):
    """U-Net on the zero-filled SENSE image, unet.py:21."""

    def __init__(self, cfg, trainer=None):
        super().__init__(cfg, trainer)
        c = self._cfg
        self.fft_centered = c.get("fft_centered")
        self.fft_normalization = c.get("fft_normalization")
        self.spatial_dims = _listify(c.get("spatial_dims"))
        self.coil_dim = c.get("coil_dim")
        self.unet = NormUnet(chans=c.get("channels"), num_pools=c.get("pooling_layers"),
                             padding_size=c.get("padding_size"), normalize=c.get("normalize"))
        self.coil_combination_method = c.get("coil_combination_method")
        self.accumulate_estimates = False

    @torch.no_grad()
    def forward(self, y: torch.Tensor, sensitivity_maps: torch.Tensor, mask: torch.Tensor, init_pred: torch.Tensor,
                target: torch.Tensor) -> torch.Tensor:
        """unet.py:77-121."""
        eta = torch.view_as_complex(_ifft_combine(y, sensitivity_maps, self.coil_combination_method,
                                                  self.fft_centered, self.fft_normalization, self.spatial_dims,
                                                  self.coil_dim))
        _, eta = utils.center_crop_to_smallest(target, eta)
        out = self.unet(torch.view_as_real(eta.unsqueeze(self.coil_dim)).contiguous())
        return torch.view_as_complex(out).squeeze(self.coil_dim)


class ZF(_BaseModel):
    """Zero-filled reconstruction, zf.py:20.  NB: forward has no ``init_pred`` (zf.py:62-68)."""

    def __init__(self, cfg, trainer=None):
        super().__init__(cfg, trainer)
        c = self._cfg
        self.coil_combination_method = c.get("coil_combination_method")
        self.fft_centered = c.get("fft_centered")
        self.fft_normalization = c.get("fft_normalization")
        self.spatial_dims = _listify(c.get("spatial_dims"))
        self.coil_dim = c.get("coil_dim")

    @torch.no_grad()
    def forward(self, y: torch.Tensor, sensitivity_maps: torch.Tensor, mask: torch.Tensor,
                target: torch.Tensor = None) -> Union[list, Any]:
        """zf.py:62-100."""
        pred = _ifft_combine(y, sensitivity_maps, self.coil_combination_method.upper(), self.fft_centered,
                             self.fft_normalization, self.spatial_dims, self.coil_dim)
        pred = utils.check_stacked_complex(pred)
        _, pred = utils.center_crop_to_smallest(target, pred)
        return pred


class PICS(_BaseModel):
    """l1-wavelet compressed-sensing SENSE reconstruction, the classical baseline of upstream ``PICS`` (which calls BART
    ``pics``).  Solved here by ``mridc_b200.pics.l1_wavelet_recon`` with the contract of DESIGN.md section 4.8: cfg
    ``reg_wt`` is lamda, ``num_iters`` the number of FISTA iterations."""

    def __init__(self, cfg, trainer=None):
        super().__init__(cfg, trainer)
        c = self._cfg
        self.reg_wt = c.get("reg_wt")
        self.num_iters = c.get("num_iters")
        self.fft_centered = c.get("fft_centered")
        self.fft_normalization = c.get("fft_normalization")
        self.spatial_dims = _listify(c.get("spatial_dims"))
        self.coil_dim = c.get("coil_dim")
        _ops.check_spatial_dims(self.spatial_dims)
        if self.coil_dim is not None and self.coil_dim != 1:
            raise NotImplementedError("mridc_b200 PICS takes k-space as [B, C, H, W, 2] (coil_dim 1); got %s" % (
                self.coil_dim,))

    @torch.no_grad()
    def forward(self, y: torch.Tensor, sensitivity_maps: torch.Tensor, mask: torch.Tensor,
                init_pred: torch.Tensor = None, target: torch.Tensor = None) -> torch.Tensor:
        """-> complex [B, H, W], cropped to ``target``.  ``init_pred`` is unused: FISTA starts from zero."""
        pred = pics.l1_wavelet_recon(y, sensitivity_maps, mask, self.reg_wt, self.num_iters, self.fft_centered,
                                     self.fft_normalization)
        pred = torch.view_as_complex(pred)
        if target is not None:
            _, pred = utils.center_crop_to_smallest(target, pred)
        return pred


class qCIRIM(_BaseModel):
    """quantitative Cascades of Independently Recurrent Inference Machines, qcirim.py:21 -- the quantitative module
    (R2*, S0, B0, phi mapping from multi-echo k-space).  ``use_reconstruction_module`` (a CIRIM per echo followed by a
    least-squares re-fit of the maps, qcirim.py:185-245) is not on the BASELINE configs[4] path and raises."""

    def __init__(self, cfg, trainer=None):
        super().__init__(cfg, trainer)
        c = self._cfg
        dimensionality = c.get("quantitative_module_dimensionality")
        if dimensionality != 2:
            raise ValueError(f"Only 2D is currently supported for qMRI models.Found {dimensionality}")  # qcirim.py:45-49
        if not c.get("quantitative_module_no_dc"):
            raise ValueError("qCIRIM does not support explicit DC component.")  # :51-53
        self.fft_centered = c.get("fft_centered")
        self.fft_normalization = c.get("fft_normalization")
        self.spatial_dims = _listify(c.get("spatial_dims"))
        self.coil_dim = c.get("coil_dim")
        self.coil_combination_method = c.get("coil_combination_method")
        self.shift_B0_input = c.get("shift_B0_input")
        self.cirim = nn.ModuleList([])
        self.use_reconstruction_module = c.get("use_reconstruction_module")
        if self.use_reconstruction_module:
            raise NotImplementedError(
                "mridc_b200: qCIRIM with use_reconstruction_module=True is out of scope (SURVEY 8f rank 2)")
        self.qcirim = nn.ModuleList([
            qRIMBlock(
                recurrent_layer=c.get("quantitative_module_recurrent_layer"),
                conv_filters=_listify(c.get("quantitative_module_conv_filters")),
                conv_kernels=_listify(c.get("quantitative_module_conv_kernels")),
                conv_dilations=_listify(c.get("quantitative_module_conv_dilations")),
                conv_bias=_listify(c.get("quantitative_module_conv_bias")),
                recurrent_filters=_listify(c.get("quantitative_module_recurrent_filters")),
                recurrent_kernels=_listify(c.get("quantitative_module_recurrent_kernels")),
                recurrent_dilations=_listify(c.get("quantitative_module_recurrent_dilations")),
                recurrent_bias=_listify(c.get("quantitative_module_recurrent_bias")),
                depth=c.get("quantitative_module_depth"),
                time_steps=c.get("quantitative_module_time_steps"),
                conv_dim=c.get("quantitative_module_conv_dim"),
                no_dc=c.get("quantitative_module_no_dc"),
                linear_forward_model=SignalForwardModel(
                    sequence=c.get("quantitative_module_signal_forward_model_sequence")),
                fft_centered=self.fft_centered,
                fft_normalization=self.fft_normalization,
                spatial_dims=self.spatial_dims,
                coil_dim=self.coil_dim,
                coil_combination_method=self.coil_combination_method,
                dimensionality=dimensionality,
            )
            for _ in range(c.get("quantitative_module_num_cascades"))
        ])
        self.accumulate_estimates = c.get("quantitative_module_accumulate_estimates")
        self.gamma = torch.tensor(_listify(c.get("quantitative_module_gamma_regularization_factors")))  # :141
        self.preprocessor = RescaleByMax

    @torch.no_grad()
    def forward(self, R2star_map_init: torch.Tensor, S0_map_init: torch.Tensor, B0_map_init: torch.Tensor,
                phi_map_init: torch.Tensor, TEs: List, y: torch.Tensor, sensitivity_maps: torch.Tensor,
                mask_brain: torch.Tensor, sampling_mask: torch.Tensor) -> Union[Generator, torch.Tensor]:
        """qcirim.py:145-312 -- yields [pred, R2star, S0, B0, phi] where pred is an empty tensor (no reconstruction
        module) and every map entry is list[num_cascades] of list[time_steps] of [B, H, W]."""
        _lib.require_cuda(y, "y")
        g = [float(self.gamma[k]) for k in range(4)]
        # :247-250 (x / gamma: a true division, the block multiplies the factor back in, qrim_block.py:196-199)
        maps = [_lib.require_cuda(m, n) / g[k] for k, (m, n) in enumerate(
            ((R2star_map_init, "R2star_map_init"), (S0_map_init, "S0_map_init"), (B0_map_init, "B0_map_init"),
             (phi_map_init, "phi_map_init")))]
        prediction = y  # :252 clones; nothing below writes to y
        eta = None
        hx = None
        cascades = [[], [], [], []]
        for i, cascade in enumerate(self.qcirim):
            prediction, hx = cascade(prediction, y, maps[0], maps[1], maps[2], maps[3], TEs, sensitivity_maps,
                                     sampling_mask, eta, hx, self.gamma, keep_eta=i != 0)
            maps = [prediction[-1][:, k] for k in range(4)]  # :279-284
            steps = [self.process_intermediate_pred(pred, None, None, False, _abs=True) for pred in prediction]
            for k in range(4):
                cascades[k].append([s[k] for s in steps])
        yield [torch.empty([]), cascades[0], cascades[1], cascades[2], cascades[3]]

    def process_intermediate_pred(self, pred, sensitivity_maps, target, do_coil_combination=False, _abs=False):
        """qcirim.py:314-341: RescaleByMax.reverse(pred, gamma) split into the four maps.  ``_abs`` folds the caller's
        ``torch.abs(pred)`` (:300) into the same kernel."""
        x = self.preprocessor.reverse(pred, self.gamma, _take_abs=_abs)
        return x[:, 0, ...], x[:, 1, ...], x[:, 2, ...], x[:, 3, ...]
