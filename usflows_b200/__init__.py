"""usflows_b200 -- B200-native (sm_100a) evaluation of USFlows normalising flows.

Drop-in for the hot path of aai-institute/USFlows: `Flow` / `USFlow` `log_prob`, `sample`, `backward`,
`_forward` over LU / Householder affine layers, additive masked couplings with MLP conditioners, scale,
leaky-ReLU and permute layers, Laplace / Normal / Lp-radial base densities, DenseNN and (vector-branch) ConvNet
conditioners.  Python host code calls hand-written
CUDA (tcgen05 + TMEM + TMA contractions, fused elementwise kernels) through the C ABI in
include/usflows_b200.h.  CUDA tensors only -- there is no CPU fallback.
"""
from . import distributions, nn, transforms  # noqa: F401
from .distributions import Chi, Gamma, GammaMM, LogNormalMM, WeibullMM, Independent, Laplace, LogNormal, Normal, RadialDistribution  # noqa: F401
from .engine import get_precision, set_chunk_rows, set_precision  # noqa: F401
from .flows import Flow, USFlow  # noqa: F401
from .ops import dequantize, quantize  # noqa: F401
from .nn import (AdditiveAffineNN, BottleneckConv, CondConvNet, CondConvNet2D, ConditionalDenseNN, ConvNet, ConvNet2D, DenseNN, GatedConv, GatedConvND, GatedMLP,  # noqa: F401
                 LayerNormChannels, LayerNormChannelsND, LayerNormVector)
from .optim import SophiaG  # noqa: F401
from .transforms import Bijective1x1Conv2d, MaskedAffineCoupling, PlaneBijectiveLinearTransform  # noqa: F401
from .transforms import (AffineTransform, BaseTransform, BlockAffineTransform, BlockLUTransform,  # noqa: F401
                         CompositeRotation, HouseholderTransform, InverseTransform, LeakyReLUTransform, LUTransform,
                         MaskedCoupling, Permute, Rotation, ScaleTransform, SequentialAffineTransform)

__version__ = "0.1.0"
