"""Wavelet front end of the frequency discriminators (``FS_DiscriminatorA/B.filter_wavelet``, model.py:166-179 and
222-235): one Haar/reflect analysis level, band selection and the ``* 0.5 + 0.5`` normalisation of the detail bands.

The reference computes all four sub-bands, then slices, scales and concatenates them with separate elementwise
kernels.  Here the selection and the affine map sit in the analysis kernel's store epilogue
(``b200w_afb2d_ex_f32``): a band that the discriminator does not look at is never written, and with one input
channel the ``(N, 1, 3, H', W')`` detail tensor *is* ``torch.cat((LH, HL, HH), 1)`` -- a view, no copy.

Double inputs (the reference's double mode: discriminators built under ``torch.set_default_dtype(torch.float64)``) go
through ``b200w_afb2d_ex_f64``, the fp64 direct kernel with the same epilogue; see ``module_taps`` for the dtype rules.

    filt = WaveletFilter(cs='cat', variant='B')          # model.py:190-192 defaults of FS_DiscriminatorB
    dwt, ximg = filt(x)                                  # == FS_DiscriminatorB.filter_wavelet(x)
"""
import numpy as np
import torch
import torch.nn as nn

from . import ops, ops64
from .dwt import lowlevel
from .dwt.transform2d import _filters_from

_FORMATS = ("sum", "each", "cat")


def _select(x, taps, mode, want_low, want_highs, norm):
    scale, shift = (0.5, 0.5) if norm else (1.0, 0.0)
    op = ops64.afb2d_select if x.dtype == torch.float64 else ops.afb2d_select
    return op(x, taps[0], taps[1], taps[2], taps[3], mode, want_low, want_highs, scale, shift)


def filter_wavelet(x, cs="sum", norm=True, variant="A", taps=None, mode="reflect"):
    """``FS_Discriminator{variant}.filter_wavelet(x, norm)`` for the band format ``cs``.

    Returns what the reference returns: ``(LL, x)`` for A/'sum' (model.py:171-172), ``(HH, x)`` for B/'sum'
    (model.py:227-228), ``(LL, LH, HL, HH, x)`` for 'each', ``(cat((LH, HL, HH), 1), x)`` for 'cat'.  ``taps`` are the
    four host tap tuples of a ``DWTForward`` (default: haar, as at model.py:140,190).  A float64 ``x`` is filtered in
    double (with double haar taps by default), a float32 one in fp32.
    """
    fmt = cs.lower()
    if fmt not in _FORMATS:
        raise NotImplementedError('Wavelet format [{:s}] not recognized'.format(cs))
    if taps is None:
        taps = _haar_taps(x.dtype == torch.float64)
    m = lowlevel.mode_to_int(mode)
    lowlevel.int_to_mode(m)
    if fmt == "sum" and variant.upper() == "A":
        low, _ = _select(x, taps, m, True, False, norm)
        return low, x
    if fmt == "each":
        low, highs = _select(x, taps, m, True, True, norm)
        return low, highs[:, :, 0], highs[:, :, 1], highs[:, :, 2], x
    _, highs = _select(x, taps, m, False, True, norm)
    if fmt == "sum":                      # variant B looks at the diagonal band only
        return highs[:, :, 2], x
    n, c, _, h, w = highs.shape
    if c == 1:
        return highs.view(n, 3, h, w), x  # cat((LH, HL, HH), 1) of single-channel bands is the band axis itself
    return highs.transpose(1, 2).reshape(n, 3 * c, h, w), x


_HAAR = {}


def _haar_taps(f64):
    """The four host tap tuples of a haar ``DWTForward``: time-reversed dec_lo / dec_hi (prep_filt_afb2d), rounded to
    fp32 as a module built under the float32 default holds them, or kept in double for double inputs."""
    if f64 not in _HAAR:
        lo, hi = _filters_from("haar", ("dec_lo", "dec_hi"))[:2]
        dt = np.float64 if f64 else np.float32
        lo, hi = (tuple(float(v) for v in np.asarray(f, dtype=np.float64)[::-1].astype(dt)) for f in (lo, hi))
        # DWTForward passes its *_col buffers into AFB2D's row slots (pw/dwt/transform2d.py:70-71)
        _HAAR[f64] = (lo, hi, lo, hi)
    return _HAAR[f64]


def module_taps(x, filters):
    """Host taps of a module's ``(h0_col, h1_col, h0_row, h1_row)`` buffers for input ``x``.  A double ``x`` needs
    float64 buffers (a module built under ``torch.set_default_dtype(torch.float64)``) and raises like the reference's
    convolution otherwise; a float32 ``x`` takes the fp32 path whatever the buffers hold."""
    if x.dtype == torch.float64:
        lowlevel._is_f64(x, filters[0])
    return tuple(lowlevel.host_taps(f) for f in filters)


class WaveletFilter(nn.Module):
    """Module form: holds the same ``h0_col .. h1_row`` buffers as the ``DWTForward(J=1, wave='haar',
    mode='reflect')`` the reference discriminators own, so their ``DWT2.*`` state-dict entries load."""

    def __init__(self, cs="sum", variant="A", wave="haar", mode="reflect"):
        super().__init__()
        if cs.lower() not in _FORMATS:
            raise NotImplementedError('Wavelet format [{:s}] not recognized'.format(cs))
        filts = lowlevel.prep_filt_afb2d(*_filters_from(wave, ("dec_lo", "dec_hi")))
        for name, f in zip(("h0_col", "h1_col", "h0_row", "h1_row"), filts):
            self.register_buffer(name, f)
        self.cs = cs
        self.variant = variant
        self.mode = mode

    def forward(self, x, norm=True):
        taps = module_taps(x, (self.h0_col, self.h1_col, self.h0_row, self.h1_row))
        return filter_wavelet(x, self.cs, norm, self.variant, taps, self.mode)
