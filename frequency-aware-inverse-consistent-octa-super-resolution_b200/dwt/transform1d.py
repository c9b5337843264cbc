"""``DWT1DForward`` / ``DWT1DInverse`` -- drop-in for ``pytorch_wavelets/dwt/transform1d.py:7-115`` (SURVEY.md 8f
row 3): same constructor arguments, buffer names (``h0``, ``h1`` / ``g0``, ``g1``, shape (1, 1, L)), ``(yl, yh)`` layout
with the finest scale first, ``None`` detail entries = zeros, the 'unpad' of odd lengths.  Each level is one launch of
the 1-D analysis / synthesis kernel (``csrc/dwt1d.cu``) through ``lowlevel.AFB1D`` / ``SFB1D``.  CUDA-only.
"""
import torch.nn as nn

from . import lowlevel
from ..wavelets import as_wavelet, is_wavelet


def _taps_of(wave, names):
    if isinstance(wave, str):
        wave = as_wavelet(wave)
    if is_wavelet(wave):
        return tuple(getattr(wave, n) for n in names)
    assert len(wave) == 2
    return wave[0], wave[1]


class DWT1DForward(nn.Module):
    """transform1d.py:7-62.  ``forward(x)``: x (N, C, L) -> (yl, [yh_1 (finest), ..., yh_J])."""

    def __init__(self, J=1, wave="db1", mode="zero"):
        super().__init__()
        h0, h1 = _taps_of(wave, ("dec_lo", "dec_hi"))
        filts = lowlevel.prep_filt_afb1d(h0, h1)
        self.register_buffer("h0", filts[0])
        self.register_buffer("h1", filts[1])
        self.J = J
        self.mode = mode

    def forward(self, x):
        assert x.ndim == 3, "Can only handle 3d inputs (N, C, L)"
        highs = []
        x0 = x
        mode = lowlevel.mode_to_int(self.mode)
        lowlevel._is_f64(x, self.h0)   # double input needs double filters and vice versa
        for _ in range(self.J):
            x0, x1 = lowlevel.AFB1D.apply(x0, self.h0, self.h1, mode)
            highs.append(x1)
        return x0, highs


class DWT1DInverse(nn.Module):
    """transform1d.py:65-115.  ``forward((yl, yh))`` -> (N, C, L)."""

    def __init__(self, wave="db1", mode="zero"):
        super().__init__()
        g0, g1 = _taps_of(wave, ("rec_lo", "rec_hi"))
        filts = lowlevel.prep_filt_sfb1d(g0, g1)
        self.register_buffer("g0", filts[0])
        self.register_buffer("g1", filts[1])
        self.mode = mode

    def forward(self, coeffs):
        x0, highs = coeffs
        assert x0.ndim == 3, "Can only handle 3d inputs (N, C, L)"
        mode = lowlevel.mode_to_int(self.mode)
        lowlevel._is_f64(x0, self.g0)
        for x1 in highs[::-1]:
            # 'unpad' (transform1d.py:110-112) as a view: the kernel takes the row stride
            if x1 is not None and x0.shape[-1] > x1.shape[-1]:
                x0 = x0[..., :-1]
            x0 = lowlevel.SFB1D.apply(x0, x1, self.g0, self.g1, mode)   # x1 None = zeros, never materialised (:106-107)
        return x0
