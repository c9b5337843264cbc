"""b200wave: the B200-native (sm_100a) wavelet + SSIM hot path of
KevynUtopia/Frequency-Aware-Inverse-Consistent-OCTA-Super-Resolution.

Drop-in surface (same names and signatures as the reference):

* ``DWTForward``, ``DWTInverse`` and the aliases ``DWT``, ``IDWT``, ``DWT2D``, ``IDWT2D``
  (``pytorch_wavelets/__init__.py:24-33``), ``dwt.lowlevel.AFB2D`` / ``SFB2D`` / ``afb2d`` / ``sfb2d``
* ``DWT1DForward``, ``DWT1DInverse`` (aliases ``DWT1D``, ``IDWT1D``), ``dwt.lowlevel.AFB1D`` / ``SFB1D``
* ``SWTForward`` and its periodic inverse ``SWTInverse`` (the reference has no usable one), ``dwt.lowlevel.afb2d_atrous`` /
  ``sfb2d_atrous``
* ``SSIM``, ``ssim`` (``ssim.py``)
* ``freq.high_pass``, ``freq.low_pass`` (``utils.py:93-117``) and the batched ``freq.gaussian_split``
* ``HostPipeline``: host-buffer front end (chunked, stream-overlapped H2D | kernels | D2H)

Everything computes in hand-written CUDA kernels behind ``torch.ops.b200wave``;
there is no CPU path.
"""
from . import ops  # noqa: F401  (registers torch.ops.b200wave.*)
from . import dwt  # noqa: F401
from .dwt import lowlevel  # noqa: F401
from .dwt.transform2d import DWTForward, DWTInverse, SWTForward, SWTInverse
from .dwt.transform1d import DWT1DForward, DWT1DInverse
from .ssim import SSIM, ssim
from .wavelets import Wavelet, wavelist  # noqa: F401
from .hostpipe import HostPipeline
from . import freq  # noqa: F401  (utils.high_pass / low_pass, SURVEY 8f row 1)
from . import fsd  # noqa: F401  (FS_Discriminator*.filter_wavelet, SURVEY 8f row 2)
from . import losses  # noqa: F401  (TVLoss, SURVEY 8f row 4)
from .losses import TVLoss, phase_consistency_loss

__version__ = "0.1.0"

DWT = DWTForward
IDWT = DWTInverse
DWT2D = DWT
IDWT2D = IDWT
DWT1D = DWT1DForward
IDWT1D = DWT1DInverse

__all__ = ["DWTForward", "DWTInverse", "DWT", "IDWT", "DWT2D", "IDWT2D", "DWT1DForward", "DWT1DInverse", "DWT1D", "IDWT1D", "SWTForward",
           "SWTInverse",           "SSIM", "ssim", "lowlevel",
           "Wavelet", "wavelist", "HostPipeline", "TVLoss", "phase_consistency_loss", "__version__"]
