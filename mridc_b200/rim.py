"""Drop-ins for the RIM building blocks of the reference (B200 kernels behind the same module API).

  log_likelihood_gradient   mridc/collections/reconstruction/models/rim/rim_utils.py:11-67
  ConvNonlinear / ConvRNNStack  .../rim/conv_layers.py:36-123 / :8-33
  ConvGRUCell / ConvMGUCell / IndRNNCell  .../rim/rnn_cells.py:93-127 / :230-261 / :367-391
  RIMBlock                  .../rim/rim_block.py:15-269

Parameters live in the same sub-module / attribute names as the reference so that a reference
``state_dict`` loads key-for-key (SURVEY.md section 8a "Weights"); the ``torch.nn`` layer objects are
used only as parameter holders and for their initialisers -- the arithmetic is the sm_100a kernels.
Inference only (no autograd through the kernels).
"""
from typing import Any, Optional, Sequence, Tuple, Union

import os

import torch
import torch.nn as nn

from . import _lib, _ops

__all__ = ["log_likelihood_gradient", "ConvNonlinear", "ConvRNNStack", "ConvGRUCell", "ConvMGUCell", "IndRNNCell",
           "RIMBlock"]


def log_likelihood_gradient(eta: torch.Tensor, masked_kspace: torch.Tensor, sense: torch.Tensor, mask: torch.Tensor,
                            sigma: float, fft_centered: bool, fft_normalization: str, spatial_dims: Sequence[int],
                            coil_dim: int) -> torch.Tensor:
    """rim_utils.py:11-67 as one fused data-consistency operator; returns [B, 4, H, W]."""
    if coil_dim == 0:
        coil_dim += 1  # rim_utils.py:41-42
    if coil_dim != 1:
        raise NotImplementedError("mridc_b200: fused RIM gradient expects coil_dim == 1 ([B, C, H, W, 2] data)")
    _ops.check_spatial_dims(spatial_dims)
    return _ops.dc_rim_grad(eta, masked_kspace, sense, mask, sigma, fft_centered, fft_normalization)


def _pad_amount(dilation, kernel_size):
    return (dilation * (kernel_size - 1)) // 2


def _require_2d(conv_dim, who):
    if conv_dim != 2:
        raise NotImplementedError("mridc_b200: %s supports conv_dim == 2 only (got %s)" % (who, conv_dim))


def _require_2d_or_3d(conv_dim, who):
    if conv_dim not in (2, 3):
        raise NotImplementedError("mridc_b200: %s supports conv_dim 2 and 3 (got %s)" % (who, conv_dim))


def _conv3d_dchw(x, w5, bias, k, dil, pad_mode, act=_ops.ACT_NONE, slope=0.0, add=None, add_scale=None, residual=None):
    """'same' 3-D convolution of the slice stack x [D, Cin, H, W] (torch's unbatched Conv3d input [Cin, D, H, W] with the
    slice axis leading) with w5 [Cout, Cin, k, k, k]: the depth taps are k launches of the batched 2-D kernel over the
    (replicate- or zero-) shifted stack, each adding the previous partial sum in its epilogue; bias, the optional
    ``add_scale * add`` term, the activation and the channels-last residual belong to the last launch.
    -> [D, Cout, H, W] (or [D, H, W, Cout] with ``residual``)."""
    x = x.contiguous()
    D = x.shape[0]
    pad = _pad_amount(dil, k)
    ar = torch.arange(D, device=x.device)
    ones = None
    acc = None
    for kd in range(k):
        off = kd * dil - pad
        if off == 0:
            xk = x
        elif pad_mode == _ops.PAD_REPLICATE:
            xk = x.index_select(0, (ar + off).clamp_(0, D - 1))
        else:  # zero padding: slices outside the stack contribute nothing
            lo, hi = max(0, -off), min(D, D - off)
            if hi <= lo:
                continue
            xk = torch.zeros_like(x)
            xk[lo:hi] = x[lo + off:hi + off]
        last = kd == k - 1
        a, a_s = acc, None
        if acc is not None:
            if ones is None:
                ones = torch.ones(w5.shape[0], dtype=torch.float32, device=x.device)
            a_s = ones
        if last and add is not None:
            extra = add.contiguous() * add_scale.reshape(1, -1, 1, 1)
            a = extra if a is None else a + extra
            if ones is None:
                ones = torch.ones(w5.shape[0], dtype=torch.float32, device=x.device)
            a_s = ones
        acc = _ops.conv2d(xk, w5[:, :, kd].contiguous(), bias if last else None, k, dil, pad_mode,
                          act if last else _ops.ACT_NONE, slope if last else 0.0, add=a, add_scale=a_s,
                          residual=residual if last else None)
    return acc


class ConvRNNStack(nn.Module):
    """conv_layers.py:8-33."""

    def __init__(self, convs, rnn):
        super().__init__()
        self.convs = convs
        self.rnn = rnn

    def forward(self, x, hidden):
        return self.rnn(self.convs(x), hidden)


class ConvNonlinear(nn.Module):
    """conv_layers.py:36-123: ReplicationPad(dil*(k-1)//2) -> Conv(padding=0) -> ReLU / LeakyReLU / identity."""

    def __init__(self, input_size, features, conv_dim, kernel_size, dilation, bias, nonlinear="relu"):
        super().__init__()
        _require_2d_or_3d(conv_dim, "ConvNonlinear")
        if kernel_size % 2 != 1:
            raise NotImplementedError("mridc_b200: ConvNonlinear supports odd kernel sizes only")
        self.input_size = input_size
        self.features = features
        self.kernel_size = kernel_size
        self.dilation = dilation
        self.bias = bias
        self.conv_dim = conv_dim
        if nonlinear is not None and nonlinear.upper() == "RELU":
            self._act, self._slope = _ops.ACT_RELU, 0.0
        elif nonlinear is not None and nonlinear.upper() == "LEAKYRELU":
            self._act, self._slope = _ops.ACT_LEAKY, 0.01  # torch.nn.LeakyReLU() default slope
        elif nonlinear is None:
            self._act, self._slope = _ops.ACT_NONE, 0.0
        else:
            raise ValueError("Please specify a proper nonlinearity")
        conv_class = nn.Conv3d if conv_dim == 3 else nn.Conv2d  # conv_layers.py:96-104
        self.conv_layer = conv_class(in_channels=input_size, out_channels=features, kernel_size=kernel_size, padding=0,
                                     dilation=dilation, bias=bias)
        self.reset_parameters()

    def reset_parameters(self):
        torch.nn.init.kaiming_normal_(self.conv_layer.weight, nonlinearity="relu")
        if self.conv_layer.bias is not None:
            nn.init.zeros_(self.conv_layer.bias)

    def check_forward_input(self, _input):
        if _input.size(1) != self.input_size:
            raise RuntimeError(f"input has inconsistent input_size: got {_input.size(1)}, expected {self.input_size}")

    def forward(self, _input, residual_nhwc: Optional[torch.Tensor] = None):
        if self.conv_dim == 3:
            # unbatched Conv3d input [C, D, H, W] (rim_block.py:230-231) -> [F, D, H, W]
            out = self.forward_dchw(_input.permute(1, 0, 2, 3), residual_nhwc)
            return out if residual_nhwc is not None else out.permute(1, 0, 2, 3)
        self.check_forward_input(_input)
        return _ops.conv2d(_input, self.conv_layer.weight, self.conv_layer.bias, self.kernel_size, self.dilation,
                           _ops.PAD_REPLICATE, self._act, self._slope, residual=residual_nhwc)

    def forward_dchw(self, x, residual_nhwc: Optional[torch.Tensor] = None):
        """conv_dim == 3 on the slice stack [D, C, H, W] (ReplicationPad3d + Conv3d, conv_layers.py:72-76,:123)."""
        self.check_forward_input(x)
        return _conv3d_dchw(x, self.conv_layer.weight, self.conv_layer.bias, self.kernel_size, self.dilation,
                            _ops.PAD_REPLICATE, self._act, self._slope, residual=residual_nhwc)


def _reject_3d_gates(conv_dim, _input):
    """The reference builds the GRU / MGU gates as nn.Conv2d whatever conv_dim says (rnn_cells.py:23-38, :160-175) and
    then feeds them the 5-D tensors of :114-116 / :249-251: the same failure, with the same text."""
    if conv_dim == 3:
        raise RuntimeError("Expected 3D (unbatched) or 4D (batched) input to conv2d, but got input of size: %s"
                           % list(_input.unsqueeze(0).shape))


class _CellBase(nn.Module):
    def check_forward_input(self, _input):
        if _input.size(1) != self.input_size:
            raise RuntimeError(f"input has inconsistent input_size: got {_input.size(1)}, expected {self.input_size}")

    def check_forward_hidden(self, _input, hx, hidden_label=""):
        if _input.size(0) != hx.size(0):
            raise RuntimeError(
                f"Input batch size {_input.size(0)} doesn't match hidden{hidden_label} batch size {hx.size(0)}")
        if hx.size(1) != self.hidden_size:
            raise RuntimeError(
                f"hidden{hidden_label} has inconsistent hidden_size: got {hx.size(1)}, expected {self.hidden_size}")

    @staticmethod
    def orthotogonalize_weights(weights, chunks=1):
        return torch.cat([nn.init.orthogonal_(w) for w in weights.chunk(chunks, 0)], 0)


class ConvGRUCell(_CellBase):
    """rnn_cells.py:8-127."""

    def __init__(self, input_size, hidden_size, conv_dim, kernel_size, dilation=1, bias=True):
        super().__init__()
        _require_2d_or_3d(conv_dim, "ConvGRUCell")
        self.input_size, self.hidden_size, self.bias, self.conv_dim = input_size, hidden_size, bias, conv_dim
        self.kernel_size, self.dilation = kernel_size, dilation
        pad = _pad_amount(dilation, kernel_size)
        self.ih = nn.Conv2d(input_size, 3 * hidden_size, kernel_size, padding=pad, dilation=dilation, bias=bias)
        self.hh = nn.Conv2d(hidden_size, 3 * hidden_size, kernel_size, padding=pad, dilation=dilation, bias=False)
        self.reset_parameters()

    def reset_parameters(self):
        self.ih.weight.data = self.orthotogonalize_weights(self.ih.weight.data)
        self.hh.weight.data = self.orthotogonalize_weights(self.hh.weight.data)
        if self.bias is True:
            nn.init.zeros_(self.ih.bias)

    def forward(self, _input, hx):
        _reject_3d_gates(self.conv_dim, _input)
        self.check_forward_input(_input)
        self.check_forward_hidden(_input, hx)
        lib = _lib.load()
        _input, hx = _input.contiguous(), hx.contiguous()
        N, _, H, W = _input.shape
        out = torch.empty_like(hx)
        if self.kernel_size == 1:
            _lib.check(lib.mrb_gru_cell_1x1(_lib.ptr(_input), _lib.ptr(hx), _lib.ptr(self.ih.weight),
                                            _lib.ptr(self.ih.bias), _lib.ptr(self.hh.weight), _lib.ptr(out), N,
                                            self.input_size, self.hidden_size, H * W, _lib.stream_ptr()))
            return out
        ih = _ops.conv2d(_input, self.ih.weight, self.ih.bias, self.kernel_size, self.dilation, _ops.PAD_ZERO)
        hh = _ops.conv2d(hx, self.hh.weight, None, self.kernel_size, self.dilation, _ops.PAD_ZERO)
        _lib.check(lib.mrb_gru_gates(_lib.ptr(ih), _lib.ptr(hh), _lib.ptr(hx), _lib.ptr(out), N, self.hidden_size,
                                     H * W, _lib.stream_ptr()))
        return out


class ConvMGUCell(_CellBase):
    """rnn_cells.py:130-261."""

    def __init__(self, input_size, hidden_size, conv_dim, kernel_size, dilation=1, bias=True):
        super().__init__()
        _require_2d_or_3d(conv_dim, "ConvMGUCell")
        self.input_size, self.hidden_size, self.bias, self.conv_dim = input_size, hidden_size, bias, conv_dim
        self.kernel_size, self.dilation = kernel_size, dilation
        pad = _pad_amount(dilation, kernel_size)
        self.ih = nn.Conv2d(input_size, 2 * hidden_size, kernel_size, padding=pad, dilation=dilation, bias=bias)
        self.hh = nn.Conv2d(hidden_size, 2 * hidden_size, kernel_size, padding=pad, dilation=dilation, bias=False)
        self.reset_parameters()

    def reset_parameters(self):
        self.ih.weight.data = self.orthotogonalize_weights(self.ih.weight.data)
        self.hh.weight.data = self.orthotogonalize_weights(self.hh.weight.data)
        nn.init.xavier_uniform_(self.ih.weight, nn.init.calculate_gain("relu"))
        nn.init.xavier_uniform_(self.hh.weight)
        if self.bias is True:
            nn.init.zeros_(self.ih.bias)

    def forward(self, _input, hx):
        _reject_3d_gates(self.conv_dim, _input)
        self.check_forward_input(_input)
        self.check_forward_hidden(_input, hx)
        _input, hx = _input.contiguous(), hx.contiguous()
        N, _, H, W = _input.shape
        ih = _ops.conv2d(_input, self.ih.weight, self.ih.bias, self.kernel_size, self.dilation, _ops.PAD_ZERO)
        hh = _ops.conv2d(hx, self.hh.weight, None, self.kernel_size, self.dilation, _ops.PAD_ZERO)
        out = torch.empty_like(hx)
        _lib.check(_lib.load().mrb_mgu_gates(_lib.ptr(ih), _lib.ptr(hh), _lib.ptr(hx), _lib.ptr(out), N,
                                             self.hidden_size, H * W, _lib.stream_ptr()))
        return out


class IndRNNCell(_CellBase):
    """rnn_cells.py:264-391."""

    def __init__(self, input_size, hidden_size, conv_dim, kernel_size, dilation=1, bias=True):
        super().__init__()
        _require_2d_or_3d(conv_dim, "IndRNNCell")
        self.input_size, self.hidden_size, self.bias, self.conv_dim = input_size, hidden_size, bias, conv_dim
        self.kernel_size, self.dilation = kernel_size, dilation
        pad = _pad_amount(dilation, kernel_size)
        conv_class = nn.Conv3d if conv_dim == 3 else nn.Conv2d  # rnn_cells.py:295-312
        self.ih = conv_class(input_size, hidden_size, kernel_size, padding=pad, dilation=dilation, bias=bias)
        self.hh = nn.Parameter(
            nn.init.normal_(torch.empty(*((1, hidden_size) + (1,) * conv_dim)),
                            std=1.0 / (hidden_size * (1 + kernel_size**2))))
        self.reset_parameters()

    def reset_parameters(self):
        self.ih.weight.data = self.orthotogonalize_weights(self.ih.weight.data)
        nn.init.normal_(self.ih.weight, std=1.0 / (self.hidden_size * (1 + self.kernel_size**2)))
        if self.bias is True:
            nn.init.zeros_(self.ih.bias)

    def forward(self, _input, hx):
        if self.conv_dim == 3:
            # rnn_cells.py:386-391: _input [C, D, H, W], hx [D, C, H, W] -> [1, C, D, H, W]
            return self.forward_dchw(_input.permute(1, 0, 2, 3), hx).permute(1, 0, 2, 3).unsqueeze(0)
        self.check_forward_input(_input)
        self.check_forward_hidden(_input, hx)
        # ReLU(ih(x) + hh * h) with the recurrent term and ReLU fused into the conv epilogue (rnn_cells.py:391)
        return _ops.conv2d(_input, self.ih.weight, self.ih.bias, self.kernel_size, self.dilation, _ops.PAD_ZERO,
                           _ops.ACT_RELU, 0.0, add=hx.contiguous(), add_scale=self.hh.reshape(-1))


def _indrnn_forward_dchw(self, x, hx):
    """conv_dim == 3 on slice stacks [D, C, H, W]: ReLU(Conv3d(x) + hh * h), zero padding (rnn_cells.py:297-304,:391)."""
    self.check_forward_input(x)
    self.check_forward_hidden(x, hx)
    return _conv3d_dchw(x, self.ih.weight, self.ih.bias, self.kernel_size, self.dilation, _ops.PAD_ZERO, _ops.ACT_RELU,
                        0.0, add=hx, add_scale=self.hh.reshape(-1))


IndRNNCell.forward_dchw = _indrnn_forward_dchw


class RIMBlock(nn.Module):
    """rim_block.py:15-269.  dimensionality == 3 (inputs [batch, slices, coils, H, W, 2], conv_dim == 3) runs like the
    reference: folded to batch*slices for the data-consistency gradient (:168-180), the regulariser's 3-D convolutions
    over the stack of batch*slices images (:230-246).  As in the reference only the IndRNN cell has a 3-D path."""

    def __init__(self, recurrent_layer=None, conv_filters=None, conv_kernels=None, conv_dilations=None,
                 conv_bias=None, recurrent_filters=None, recurrent_kernels=None, recurrent_dilations=None,
                 recurrent_bias=None, depth: int = 2, time_steps: int = 8, conv_dim: int = 2, no_dc: bool = False,
                 fft_centered: bool = True, fft_normalization: str = "ortho",
                 spatial_dims: Optional[Tuple[int, int]] = None, coil_dim: int = 1, dimensionality: int = 2,
                 consecutive_slices: int = 1):
        super().__init__()
        self.conv_dim = conv_dim
        self.input_size = depth * 2
        self.time_steps = time_steps
        self.layers = nn.ModuleList()
        conv_layer = None
        for (
            (conv_features, conv_k_size, conv_dilation, l_conv_bias, nonlinear),
            (rnn_features, rnn_k_size, rnn_dilation, rnn_bias, rnn_type),
        ) in zip(
            zip(conv_filters, conv_kernels, conv_dilations, conv_bias, ["relu", "relu", None]),
            zip(recurrent_filters, recurrent_kernels, recurrent_dilations, recurrent_bias,
                [recurrent_layer, recurrent_layer, None]),
        ):
            conv_layer = None
            if conv_features != 0:
                conv_layer = ConvNonlinear(self.input_size, conv_features, conv_dim=conv_dim, kernel_size=conv_k_size,
                                           dilation=conv_dilation, bias=l_conv_bias, nonlinear=nonlinear)
                self.input_size = conv_features
            if rnn_features != 0 and rnn_type is not None:
                if rnn_type.upper() == "GRU":
                    rnn_cls = ConvGRUCell
                elif rnn_type.upper() == "MGU":
                    rnn_cls = ConvMGUCell
                elif rnn_type.upper() == "INDRNN":
                    rnn_cls = IndRNNCell
                else:
                    raise ValueError("Please specify a proper recurrent layer type.")
                rnn_layer = rnn_cls(self.input_size, rnn_features, conv_dim=conv_dim, kernel_size=rnn_k_size,
                                    dilation=rnn_dilation, bias=rnn_bias)
                self.input_size = rnn_features
                self.layers.append(ConvRNNStack(conv_layer, rnn_layer))
        self.final_layer = nn.Sequential(conv_layer)
        self.recurrent_filters = recurrent_filters
        self.fft_centered = fft_centered
        self.fft_normalization = fft_normalization
        self.spatial_dims = spatial_dims if spatial_dims is not None else [-2, -1]
        self.coil_dim = coil_dim
        self.no_dc = no_dc
        if not self.no_dc:
            self.dc_weight = nn.Parameter(torch.ones(1))
            self.zero = torch.zeros(1, 1, 1, 1, 1)
        self.dimensionality = dimensionality
        self.consecutive_slices = consecutive_slices
        self._tc_engine = None  # built lazily on the first forward (tensor-core path, rim_tc.py)

    @torch.no_grad()
    def forward(self, pred: torch.Tensor, masked_kspace: torch.Tensor, sense: torch.Tensor, mask: torch.Tensor,
                eta: torch.Tensor = None, hx: torch.Tensor = None, sigma: float = 1.0,
                keep_eta: bool = False, y_hybrid: Optional[dict] = None,
                want_hx: bool = True) -> Tuple[Any, Union[list, torch.Tensor, None]]:
        """rim_block.py:134-269.  Not in the reference signature: ``y_hybrid``, a dict the caller keeps across cascades so
        that the hybrid-space k-space of ``masked_kspace`` (dc_hybrid_prepare) is computed once per slice batch; and
        ``want_hx=False``, with which a caller that drops the hidden states (CIRIM.forward) spares their export."""
        _ops.check_spatial_dims(self.spatial_dims)
        if self.coil_dim != 1:
            raise NotImplementedError("mridc_b200: RIMBlock expects coil_dim == 1")
        stack = self.dimensionality == 3 or self.consecutive_slices > 1
        if stack:  # rim_block.py:168-180: [batch, slices, coils, H, W, 2] -> [batch * slices, coils, H, W, 2]
            if self.conv_dim != 3:
                # the reference hands [4, batch*slices, H, W] to its Conv2d layers here, which only type-checks when
                # batch*slices happens to equal the channel count
                raise NotImplementedError("mridc_b200: slice stacks (dimensionality 3 / consecutive_slices > 1) need "
                                          "conv_dim == 3")
            fold = lambda t: t.reshape([t.shape[0] * t.shape[1], *t.shape[2:]])
            pred = pred[-1].detach() if isinstance(pred, (tuple, list)) else fold(pred)
            masked_kspace, mask, sense = fold(masked_kspace), fold(mask), fold(sense)
            if eta is not None and eta.dim() == 5:
                eta = fold(eta)  # :213-214
        elif self.conv_dim != 2:
            raise NotImplementedError("mridc_b200: conv_dim == 3 needs dimensionality == 3")
        if isinstance(pred, list):
            pred = pred[-1].detach()  # rim_block.py:185-186
        masked_kspace = _lib.require_cuda(masked_kspace, "masked_kspace").contiguous()
        sense = _lib.require_cuda(sense, "sense").contiguous()
        B, C, H, W, _ = masked_kspace.shape
        hx_given = hx is not None
        hx = list(hx) if hx_given else None  # zero initial state (:188-193): created below, only where it is read
        ws = torch.empty((2, B, C, H, W, 2), dtype=torch.float32, device=masked_kspace.device)
        if eta is None or eta.ndim < 3:  # :195-211
            eta = pred if keep_eta else _ops.sens_reduce(pred, sense, self.fft_centered, self.fft_normalization, ws=ws)
        mcan = _ops.canonical_mask(mask, B, H, W)[0]  # canonicalise once for the whole time loop
        # 1-D column masks: hybrid-space k-space once per forward -> single-kernel gradient in the time loop
        yhyb = None
        if not os.environ.get("MRIDC_B200_DC_3PASS"):
            key = (masked_kspace.data_ptr(), masked_kspace._version, mcan.data_ptr(), mcan._version, bool(self.fft_centered))
            if y_hybrid is not None and y_hybrid.get("key") == key:
                yhyb = y_hybrid["yh"]
            else:
                yhyb = _ops.dc_hybrid_prepare(masked_kspace, mcan, self.fft_centered, ws=ws[0])
                if y_hybrid is not None:
                    # keep the tensors alive with the entry: a recycled allocation can then never alias the key
                    y_hybrid.update(key=key, yh=yhyb, y=masked_kspace, mask=mcan)
        etas = []
        final = self.final_layer[0]
        from .rim_tc import RimTcEngine

        if self._tc_engine is None:
            self._tc_engine = RimTcEngine(self) if RimTcEngine.supported(self) else False
        use_tc = bool(self._tc_engine) and self._tc_engine.covers(W) and _lib.require_cuda(eta, "eta") is not None
        if use_tc:
            # tensor-core (tcgen05, split-bf16) engine for the whole time loop
            etas, hx = self._tc_engine.run(eta, masked_kspace, sense, mcan, sigma, hx if hx_given else None, ws, yhyb,
                                           want_hx=want_hx or not self.no_dc)
        if not use_tc and hx is None:
            # the tensor-core engine reads a shared, cached zero state instead: two 26 MB-per-slice fills per cascade
            # were 2.6 % of the CIRIM step at 16 slices
            hx = [masked_kspace.new_zeros((B, f, H, W)) for f in self.recurrent_filters if f != 0]
        for _ in range(0 if use_tc else self.time_steps):  # :217-249 (generic exact-fp32 kernels)
            grad_eta = _ops.dc_rim_grad(eta, masked_kspace, sense, mcan, sigma, self.fft_centered,
                                        self.fft_normalization, ws=ws, y_hybrid=yhyb)
            if stack:
                # [batch*slices, 4, H, W] is the slice stack [D, C, H, W] of the 3-D convolutions (:230-246)
                for h, convrnn in enumerate(self.layers):
                    grad_eta = convrnn.convs.forward_dchw(grad_eta)
                    if not hasattr(convrnn.rnn, "forward_dchw"):
                        _reject_3d_gates(3, grad_eta.permute(1, 0, 2, 3))  # GRU / MGU: fails like the reference
                    hx[h] = convrnn.rnn.forward_dchw(grad_eta, hx[h])
                    grad_eta = hx[h]
                eta = final.forward_dchw(grad_eta, residual_nhwc=eta.contiguous())
                etas.append(eta)
                continue
            for h, convrnn in enumerate(self.layers):
                hx[h] = convrnn(grad_eta, hx[h])
                grad_eta = hx[h]
            # final conv (no bias/activation in the shipped configs) fused with eta + grad.permute(0,2,3,1)
            eta = final(grad_eta, residual_nhwc=eta.contiguous())
            etas.append(eta)
        if self.no_dc:
            return etas, hx  # :253-254
        if mask.dtype != torch.bool:
            # same failure mode as the reference's torch.where(mask, ...) (rim_block.py:256)
            raise RuntimeError("where expected condition to be a boolean tensor, but got a tensor with dtype %s"
                               % mask.dtype)
        dcw = self.dc_weight.detach()
        current_kspace = [
            _ops.sens_expand_softdc(e, sense, masked_kspace, pred, masked_kspace, mcan, dcw, False, self.fft_centered,
                                    self.fft_normalization, ws=ws)
            for e in etas
        ]  # :256-267: masked_kspace - soft_dc - fft2(S * e)
        return current_kspace, hx
