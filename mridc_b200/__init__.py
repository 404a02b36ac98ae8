"""mridc_b200 -- B200-native (sm_100a) drop-in for mridc's unrolled-reconstruction inference hot path.

Python surface = the reference's own API for this path (``mridc.collections.common.parts`` fft/utils functions,
RIM / VarNet / U-Net blocks, CIRIM / VarNet / UNet / ZF ``forward``); the arithmetic is hand-written CUDA behind
the C-ABI of ``include/mridc_b200.h`` (``libmridc_b200.so``).  No CPU fallback.
"""
from .fft import fft2, ifft2, fftshift, ifftshift, roll, roll_one_dim  # noqa: F401
from .utils import (  # noqa: F401
    complex_mul, complex_conj, complex_abs, complex_abs_sq, check_stacked_complex, rss, rss_complex, sense,
    coil_combination, apply_mask, mask_center, batched_mask_center, center_crop, complex_center_crop,
    center_crop_to_smallest, to_tensor, tensor_to_complex_np, is_none,
)
from .rim import (  # noqa: F401
    log_likelihood_gradient, ConvNonlinear, ConvRNNStack, ConvGRUCell, ConvMGUCell, IndRNNCell, RIMBlock,
)
from .unet import NormUnet, Unet, ConvBlock, TransposeConvBlock  # noqa: F401
from .varnet import VarNetBlock  # noqa: F401
from .sensitivity import BaseSensitivityModel  # noqa: F401
from .qrim import (  # noqa: F401
    RescaleByMax, SignalForwardModel, expand_op, analytical_log_likelihood_gradient, qRIMBlock,
)
from .data_consistency import (  # noqa: F401
    DataIDLayer, DataGDLayer, DataProxCGLayer, ConjugateGradient, DataVSLayer, DCLayer,
)
from .cascadenet import CascadeNetBlock  # noqa: F401
from .recurrentvarnet import Conv2dGRU, RecurrentInit, RecurrentVarNetBlock  # noqa: F401
from .qvarnet import qVarNetBlock  # noqa: F401
from .jrscirim import JRSCIRIMBlock  # noqa: F401
from .models import CIRIM, VarNet, UNet, ZF, PICS, qCIRIM  # noqa: F401
from .pipeline import HostPrefetcher  # noqa: F401
from .transforms import MRIDataTransforms, assemble_reconstructions, save_reconstructions  # noqa: F401
from .espirit import espirit_maps  # noqa: F401
from .pics import l1_wavelet_recon  # noqa: F401
from . import metrics  # noqa: F401

__version__ = "0.1.0"
