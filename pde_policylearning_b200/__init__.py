"""B200-native Fourier-neural-operator hot path (SpectralConv fwd+bwd and its pointwise neighbours).

The arithmetic lives in libb2no.so (hand-written CUDA for sm_100a behind the C ABI in include/b2no.h);
this package is the host-side mirror of the reference's operator interface.  There is no CPU fallback."""
from . import _lib  # noqa: F401
from .ops import SpecGeom, set_precision  # noqa: F401
from .functional import (spectral_block, pointwise_conv, pointwise_conv2, mlp_head, rel_l2_loss,  # noqa: F401
                         rno_gate)
from .modules import (  # noqa: F401
    ComplexDenseWeight, SpectralConv, SpectralConv1d, SpectralConv2d, SpectralConv3d, SubConv,
    FactorizedSpectralConv, FactorizedSpectralConv1d, FactorizedSpectralConv2d, FactorizedSpectralConv3d,
    Lifting, Projection, MLP, SoftGating, FNOBlocks, FNO, FNO1d, FNO2d, FNO3d, FNO2dObserver, LpLoss,
    RnoSpectralConv2d, FourierLayer2d, RNO_cell, RNO_layer, SpectralConvWithFC, SpectralRegressor, RNO2d,
    RNO2dObserver, PinoSpectralConv3d, MultiplicativeNet, PINObserver2d, PlanePredHead, PINObserverFullField,
    PolicyModel2D, PinoSpectralConv2d, PinoFNO2d,
)
from .pino_loss import channelflow_pino_loss, fdm_ns_vorticity, get_forcing, pino_training_loss  # noqa: F401
from .convert import convert_  # noqa: F401
from .optim import FusedAdam, GraphedTrainStep, HostBatchPipeline  # noqa: F401

__version__ = "0.1.0"
