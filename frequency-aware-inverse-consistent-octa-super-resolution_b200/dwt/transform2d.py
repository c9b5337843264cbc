"""``DWTForward`` / ``DWTInverse`` -- drop-in for ``pytorch_wavelets.dwt.transform2d``.

Same constructor arguments and defaults, same registered buffer names and shapes
(``h0_col, h1_col (1,1,L,1)``, ``h0_row, h1_row (1,1,1,L)``; ``g*`` likewise) so
``state_dict``s of the reference's ``FS_Discriminator*`` (``model.py:140,190``)
stay loadable, same ``(yl, [yh_1 (finest) .. yh_J])`` output structure
(``pw/dwt/transform2d.py:7-148``).  Every level is one fused sm_100a kernel.
"""
import torch.nn as nn

from . import lowlevel
from .. import ops, ops64
from ..wavelets import as_wavelet, is_wavelet


def _filters_from(wave, attrs):
    """``wave`` -> (col_lo, col_hi, row_lo, row_hi) raw taps, like pw/dwt/transform2d.py:22-33."""
    if isinstance(wave, str):
        wave = as_wavelet(wave)
    if is_wavelet(wave):
        lo, hi = getattr(wave, attrs[0]), getattr(wave, attrs[1])
        return lo, hi, lo, hi
    if len(wave) == 2:
        return wave[0], wave[1], wave[0], wave[1]
    if len(wave) == 4:
        return wave[0], wave[1], wave[2], wave[3]
    raise ValueError("wave must be a name, a Wavelet, or a tuple of 2 or 4 filters")


class DWTForward(nn.Module):
    """2-D DWT decomposition of an image batch.

    Args:
        J (int): number of levels.
        wave (str | Wavelet | tuple(ndarray)): wavelet name, an object with ``dec_lo``/``dec_hi``
            (e.g. ``pywt.Wavelet``), or ``(h0, h1)`` / ``(h0_col, h1_col, h0_row, h1_row)`` arrays.
        mode (str): 'zero', 'symmetric', 'reflect', 'periodic' or 'periodization'.
    """

    def __init__(self, J=1, wave='db1', mode='zero'):
        super().__init__()
        filts = lowlevel.prep_filt_afb2d(*_filters_from(wave, ('dec_lo', 'dec_hi')))
        for name, f in zip(('h0_col', 'h1_col', 'h0_row', 'h1_row'), filts):
            self.register_buffer(name, f)
        self.J = J
        self.mode = mode

    def forward(self, x):
        """x: (N, C, H, W) -> (yl, yh); yl (N, C, H', W'), yh[j] (N, C, 3, H'', W'') holding LH, HL, HH,
        finest scale first."""
        mode = lowlevel.mode_to_int(self.mode)
        lowlevel.int_to_mode(mode)
        # NB the *_col buffers go into AFB2D's *_row slots at pw/dwt/transform2d.py:70-71: the "col" filters
        # therefore run along W and the "row" filters along H.  The J-level loop over AFB2D.apply is one launch.
        taps = [lowlevel.host_taps(f) for f in (self.h0_col, self.h1_col, self.h0_row, self.h1_row)]
        yh = []
        ll = x
        J = int(self.J)
        if lowlevel._is_f64(x, self.h0_col):   # the reference's double mode: level by level through the fp64 kernels
            for _ in range(J):
                ll, high = ops64.afb2d(ll, taps[0], taps[1], taps[2], taps[3], mode)
                yh.append(high)
            return ll, yh
        while J > 0:   # chunks of at most MAX_LEVELS levels per launch
            n = min(J, ops.MAX_LEVELS)
            outs = ops.DWT2Function.apply(ll, taps[0], taps[1], taps[2], taps[3], mode, n)
            ll = outs[0]
            yh.extend(outs[1:])
            J -= n
        return ll, yh


class DWTInverse(nn.Module):
    """2-D inverse DWT; ``forward((yl, yh))`` reconstructs the image.  ``None`` entries of ``yh`` count as
    zeros (no zero tensor is materialised: the kernel skips the three detail bands)."""

    def __init__(self, wave='db1', mode='zero'):
        super().__init__()
        filts = lowlevel.prep_filt_sfb2d(*_filters_from(wave, ('rec_lo', 'rec_hi')))
        for name, f in zip(('g0_col', 'g1_col', 'g0_row', 'g1_row'), filts):
            self.register_buffer(name, f)
        self.mode = mode

    def forward(self, coeffs):
        yl, yh = coeffs
        mode = lowlevel.mode_to_int(self.mode)
        lowlevel.int_to_mode(mode)
        taps = [lowlevel.host_taps(f) for f in (self.g0_col, self.g1_col, self.g0_row, self.g1_row)]
        yh = list(yh)
        ll = yl
        if lowlevel._is_f64(yl, self.g0_col):   # double mode: pw/dwt/transform2d.py:134-148 level by level
            for h in yh[::-1]:
                if h is not None:
                    if ll.shape[-2] > h.shape[-2]:
                        ll = ll[..., :-1, :]
                    if ll.shape[-1] > h.shape[-1]:
                        ll = ll[..., :-1]
                ll = ops64.sfb2d(ll, h, taps[0], taps[1], taps[2], taps[3], mode, -1, -1)
            return ll
        # the loop over SFB2D.apply incl. the 'unpad' crop (a level reconstructed from an odd-sized input is one
        # sample too large, pw/dwt/transform2d.py:141-145) is one launch; the crop is a strided read
        while yh:
            chunk = yh[-ops.MAX_LEVELS:]
            yh = yh[:-ops.MAX_LEVELS]
            ll = ops.IDWT2Function.apply(taps[0], taps[1], taps[2], taps[3], mode, ll, *chunk)
        return ll


class SWTForward(nn.Module):
    """2-D stationary (undecimated) wavelet transform, drop-in for ``pw/dwt/transform2d.py:151-212``: same constructor
    arguments and buffers; ``forward(x)`` returns a list of J tensors.  Each level is one launch of the a-trous kernel
    (``csrc/swt.cu``) with dilation 2**j.

    What the reference actually does (and this module reproduces): ``afb2d_atrous`` returns (N, 4C, H, W) -- not the
    (N, C, 4, H, W) of its docstring -- so with J = 1 that is the shape of the single coefficient tensor; its default
    mode ``'periodization'`` raises ``ValueError("Unkown pad type")`` inside ``mypad``; and for J > 1 its
    ``ll = y[:, :, 0]`` slices a row of the 4-D tensor and the next level fails.  Here J > 1 follows the documented
    intent instead: the next level's input is the (lo, lo) band of every channel.
    """

    def __init__(self, J=1, wave="db1", mode="periodization"):
        super().__init__()
        h0_col, h1_col, h0_row, h1_row = _filters_from(wave, ("dec_lo", "dec_hi"))
        filts = lowlevel.prep_filt_afb2d(h0_col, h1_col, h0_row, h1_row)
        self.register_buffer("h0_col", filts[0])
        self.register_buffer("h1_col", filts[1])
        self.register_buffer("h0_row", filts[2])
        self.register_buffer("h1_row", filts[3])
        self.J = J
        self.mode = mode

    def forward(self, x):
        ll = x
        coeffs = []
        filts = (self.h0_col, self.h1_col, self.h0_row, self.h1_row)
        lowlevel._is_f64(x, self.h0_col)   # double input needs double filters and vice versa
        for j in range(self.J):
            y = lowlevel.afb2d_atrous(ll, filts, self.mode, 2 ** j)
            coeffs.append(y)
            n, c4, h, w = y.shape
            ll = y.view(n, c4 // 4, 4, h, w)[:, :, 0]
        return coeffs


class SWTInverse(nn.Module):
    """Inverse of ``SWTForward`` with ``mode='periodic'``; ``forward(coeffs)`` takes the list ``SWTForward`` returns
    (finest level first, each (N, 4C, H, W)) and gives back the (N, C, H, W) image.  Buffers ``g0_col, g1_col, g0_row,
    g1_row`` as in ``DWTInverse``.  Each level is one launch of the a-trous synthesis kernel (``csrc/swt_inverse.cu``)
    with dilation 2**j, coarsest first; it starts from band 0 of the coarsest level, read in place, and never reads band
    0 of the finer levels.

    The reference offers no usable inverse (its ``swt_inverse.py`` is unfinished and not exported), so the semantics
    are defined here (DESIGN.md K12): each axis is undone by the synthesis pair of the wavelet, halved.  Only periodic
    extension has an exact undecimated inverse; any other mode raises ``ValueError`` at construction.
    """

    def __init__(self, wave="db1", mode="periodic"):
        super().__init__()
        if mode != "periodic":
            raise ValueError("SWTInverse: only periodic extension (mode='periodic') has an exact undecimated inverse; "
                             "got mode %r" % (mode,))
        filts = lowlevel.prep_filt_sfb2d(*_filters_from(wave, ("rec_lo", "rec_hi")))
        for name, f in zip(("g0_col", "g1_col", "g0_row", "g1_row"), filts):
            self.register_buffer(name, f)
        self.mode = mode

    def forward(self, coeffs):
        coeffs = list(coeffs)
        if not coeffs:
            raise ValueError("SWTInverse: coeffs is empty; expected the list SWTForward returns")
        shape = tuple(coeffs[0].shape)
        if len(shape) != 4 or shape[1] % 4:
            raise ValueError("SWTInverse: coefficients must be (N, 4C, H, W), got %s" % (shape,))
        for j, c in enumerate(coeffs):
            if tuple(c.shape) != shape:
                raise ValueError("SWTInverse: coeffs[%d] has shape %s, coeffs[0] %s; every level must have the same "
                                 "shape" % (j, tuple(c.shape), shape))
            lowlevel._is_f64(c, self.g0_col)   # double coefficients need double filters and vice versa
        filts = (self.g0_col, self.g1_col, self.g0_row, self.g1_row)
        ll = coeffs[-1][:, 0::4]
        for j in range(len(coeffs) - 1, -1, -1):
            ll = lowlevel.sfb2d_atrous(coeffs[j], filts, self.mode, 2 ** j, ll=ll)
        return ll
