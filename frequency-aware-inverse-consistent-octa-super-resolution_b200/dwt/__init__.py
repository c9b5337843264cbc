"""Discrete wavelet transform path (mirror of ``pytorch_wavelets.dwt``): 2-D and 1-D."""
from . import lowlevel  # noqa: F401
from .transform2d import DWTForward, DWTInverse, SWTForward, SWTInverse  # noqa: F401
from .transform1d import DWT1DForward, DWT1DInverse  # noqa: F401
