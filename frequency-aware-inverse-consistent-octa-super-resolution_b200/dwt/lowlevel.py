"""Host-side mirror of ``pytorch_wavelets.dwt.lowlevel`` for the 2-D DWT path.

Same names, positional signatures, integer mode codes and error behaviour as
the reference (``pw`` = ``/root/reference/pytorch_wavelets/pytorch_wavelets``):
``AFB2D`` / ``SFB2D`` (``pw/dwt/lowlevel.py:312-365, 647-694``), ``afb2d`` /
``sfb2d`` (``:427-472, 600-644``), ``mode_to_int`` / ``int_to_mode``
(``:274-309``) and ``prep_filt_*`` (``:870-975``).  The arithmetic itself runs
in the fused sm_100a kernels behind ``torch.ops.b200wave`` (see ``ops.py``).
"""
import weakref

import numpy as np
import torch

from .. import ops, ops64

_MODES = {"zero": 0, "symmetric": 1, "per": 2, "periodization": 2, "constant": 3, "reflect": 4, "replicate": 5,
          "periodic": 6}
_INT_TO_MODE = {0: "zero", 1: "symmetric", 2: "periodization", 3: "constant", 4: "reflect", 5: "replicate",
                6: "periodic"}


def mode_to_int(mode):
    """pw/dwt/lowlevel.py:274-290."""
    try:
        return _MODES[mode]
    except (KeyError, TypeError):
        raise ValueError("Unkown pad type: {}".format(mode))


def int_to_mode(mode):
    """pw/dwt/lowlevel.py:293-309."""
    try:
        return _INT_TO_MODE[mode]
    except (KeyError, TypeError):
        raise ValueError("Unkown pad type: {}".format(mode))


# ---------------------------------------------------------------------------------------------------
# Host copies of filter tensors.  The kernels take their taps by value (constant bank), so a filter that
# lives on the GPU (a module buffer after ``.to(device)``) is read back ONCE and remembered; later calls
# with the same tensor object (same storage, same version counter) are free and never synchronise, which
# also keeps the ops CUDA-graph capturable after a warm-up call.
# ---------------------------------------------------------------------------------------------------
_tap_cache = {}


def host_taps(f):
    """Filter (tensor / ndarray / sequence) -> tuple of python floats, in storage order."""
    if isinstance(f, torch.Tensor):
        key = id(f)
        hit = _tap_cache.get(key)
        if hit is not None:
            ref, version, ptr, taps = hit
            if ref() is f and version == f._version and ptr == f.data_ptr():
                return taps
        taps = tuple(float(v) for v in f.detach().reshape(-1).cpu().tolist())
        if len(_tap_cache) > 256:
            for k in [k for k, v in _tap_cache.items() if v[0]() is None]:
                del _tap_cache[k]
        _tap_cache[key] = (weakref.ref(f), f._version, f.data_ptr(), taps)
        return taps
    return tuple(float(v) for v in np.asarray(f, dtype=np.float64).ravel())


def _is_f64(x, filt):
    """Double inputs are served when the module's filters are double too (built under
    ``torch.set_default_dtype(torch.float64)``, as the reference requires: with fp32 filters its conv raises)."""
    if x.dtype != torch.float64:
        if x.dtype == torch.float32 and filt.dtype == torch.float64:
            raise RuntimeError("expected scalar type Double but found Float: the module holds float64 filters (built "
                               "under torch.set_default_dtype(torch.float64)); pass double inputs, as with the reference")
        return False
    if filt.dtype != torch.float64:
        raise RuntimeError("expected scalar type Float but found Double: the module holds float32 filters; build it "
                           "under torch.set_default_dtype(torch.float64) for double inputs (as with the reference)")
    return True


def _as_taps(f, reverse):
    """Non-tensor filters are converted like afb1d/sfb1d do (lowlevel.py:120-125, 232-237)."""
    if isinstance(f, torch.Tensor):
        return host_taps(f)
    taps = host_taps(f)
    return taps[::-1] if reverse else taps


class AFB2D(object):
    """Single-level 2-D analysis: ``AFB2D.apply(x, h0_row, h1_row, h0_col, h1_col, mode)
    -> (low, highs)`` (pw/dwt/lowlevel.py:312-365).  ``h*_row`` filter along W (dim 3), ``h*_col``
    along H (dim 2); tensors are assumed already time-reversed (``prep_filt_afb2d``); ``mode`` is the
    integer code of ``mode_to_int``.  Differentiable w.r.t. ``x`` with the reference's backward."""

    @staticmethod
    def apply(x, h0_row, h1_row, h0_col, h1_col, mode):
        int_to_mode(mode)  # validates the code, ValueError("Unkown pad type") otherwise
        op = ops64.afb2d if x.dtype == torch.float64 else ops.afb2d
        return op(x, _as_taps(h0_row, True), _as_taps(h1_row, True),
                  _as_taps(h0_col, True), _as_taps(h1_col, True), int(mode))


class SFB2D(object):
    """Single-level 2-D synthesis: ``SFB2D.apply(low, highs, g0_row, g1_row, g0_col, g1_col, mode)
    -> y`` (pw/dwt/lowlevel.py:647-694).  Deviation from the reference (documented in DESIGN.md): the
    gradient of ``highs`` is produced even when ``low`` does not require grad (the reference returns
    ``None`` there, lowlevel.py:685)."""

    @staticmethod
    def apply(low, highs, g0_row, g1_row, g0_col, g1_col, mode):
        int_to_mode(mode)
        op = ops64.sfb2d if low.dtype == torch.float64 else ops.sfb2d
        return op(low, highs, _as_taps(g0_row, False), _as_taps(g1_row, False),
                  _as_taps(g0_col, False), _as_taps(g1_col, False), int(mode), -1, -1)


class AFB1D(object):
    """Single-level 1-D analysis: ``AFB1D.apply(x, h0, h1, mode) -> (x0, x1)`` on (N, C, L) tensors
    (pw/dwt/lowlevel.py:368-424).  ``h0`` / ``h1`` as stored by ``prep_filt_afb1d`` (time-reversed).  Differentiable
    w.r.t. ``x`` with the reference's backward (synthesis with the same taps, cropped to the input length)."""

    @staticmethod
    def apply(x, h0, h1, mode):
        int_to_mode(mode)
        op = ops64.afb1d if x.dtype == torch.float64 else ops.afb1d
        return op(x, _as_taps(h0, True), _as_taps(h1, True), int(mode))


class SFB1D(object):
    """Single-level 1-D synthesis: ``SFB1D.apply(low, high, g0, g1, mode) -> y`` (pw/dwt/lowlevel.py:697-743).  As for
    ``SFB2D``, ``high.grad`` is produced even when ``low`` needs none (the reference returns ``None``, :735)."""

    @staticmethod
    def apply(low, high, g0, g1, mode):
        int_to_mode(mode)
        op = ops64.sfb1d if low.dtype == torch.float64 else ops.sfb1d
        return op(low, high, _as_taps(g0, False), _as_taps(g1, False), int(mode), -1)


def afb2d_atrous(x, filts, mode="periodization", dilation=1):
    """One undecimated 2-D analysis level (pw/dwt/lowlevel.py:475-521): x (N, C, H, W) -> (N, 4C, H, W), channel
    4c + 2a + e = (W filter a, then H filter e) of input channel c -- what the reference's two grouped convolutions
    return (its docstring promises (N, C, 4, H, W); ``y.view(N, C, 4, H, W)`` is that).  ``filts`` = (h0, h1) or
    (h0_col, h1_col, h0_row, h1_row), arrays or prepped tensors.  The reference's default mode ``'periodization'`` is
    unknown to ``mypad`` and raises ``ValueError("Unkown pad type")`` there; so it does here."""
    if len(filts) == 2:
        filts = (filts[0], filts[1], filts[0], filts[1])
    elif len(filts) != 4:
        raise ValueError("Unknown form for input filts")
    h0_col, h1_col, h0_row, h1_row = filts
    if mode in ("per", "periodization") or mode not in _MODES:
        raise ValueError("Unkown pad type: {}".format(mode))
    op = ops64.swt2d if x.dtype == torch.float64 else ops.swt2d
    return op(x, _as_taps(h0_row, True), _as_taps(h1_row, True), _as_taps(h0_col, True), _as_taps(h1_col, True),
              mode_to_int(mode), int(dilation))


def sfb2d_atrous(y, filts, mode="periodic", dilation=1, ll=None):
    """One undecimated 2-D synthesis level, the functional mirror of ``afb2d_atrous`` and the inverse of it in periodic
    mode: y (N, 4C, H, W) as ``afb2d_atrous`` returns it -> (N, C, H, W).  ``ll`` (N, C, H, W) replaces band 0 of ``y``
    (the low band reconstructed from the coarser levels; default: band 0 of ``y`` itself).  ``filts`` = (g0, g1) or
    (g0_col, g1_col, g0_row, g1_row): synthesis taps, arrays or ``prep_filt_sfb2d`` tensors; ``*_row`` run along W,
    ``*_col`` along H, as the analysis filters of ``afb2d_atrous`` do.  Only ``mode='periodic'`` has an exact
    undecimated inverse; any other mode raises ``ValueError``."""
    if len(filts) == 2:
        filts = (filts[0], filts[1], filts[0], filts[1])
    elif len(filts) != 4:
        raise ValueError("Unknown form for input filts")
    if mode != "periodic":
        raise ValueError("sfb2d_atrous: only periodic extension ('periodic') has an exact undecimated inverse, got %r"
                         % (mode,))
    g0_col, g1_col, g0_row, g1_row = filts
    if ll is None:
        ll = y[:, 0::4]
    op = ops64.iswt2d if y.dtype == torch.float64 else ops.iswt2d
    return op(ll, y, _as_taps(g0_row, False), _as_taps(g1_row, False), _as_taps(g0_col, False),
              _as_taps(g1_col, False), int(dilation))


def _four_filters(filts, prep, device=None):
    """Normalise the ``filts`` argument of afb2d / sfb2d to (col_lo, col_hi, row_lo, row_hi) tensors.
    A pair means "same filters on both axes"; raw arrays go through ``prep``; prepared tensors are
    used as they are (a pair of column tensors is transposed to get the row ones)."""
    filts = list(filts)
    if len(filts) not in (2, 4):
        raise ValueError("Unknown form for input filts")
    if not all(isinstance(f, torch.Tensor) for f in filts):
        return prep(*filts, device=device)
    if len(filts) == 4:
        return tuple(filts)
    lo, hi = filts
    return lo, hi, lo.transpose(2, 3), hi.transpose(2, 3)


def afb2d(x, filts, mode="zero"):
    """Functional single-level analysis (pw/dwt/lowlevel.py:427-472): returns (N, 4C, H', W') with the
    sub-bands of channel c at 4c..4c+3 in the order ll, lh, hl, hh."""
    c_lo, c_hi, r_lo, r_hi = _four_filters(filts, prep_filt_afb2d, x.device)
    low, highs = AFB2D.apply(x, r_lo, r_hi, c_lo, c_hi, mode_to_int(mode))
    n, c, h, w = low.shape
    return torch.cat([low.unsqueeze(2), highs], dim=2).reshape(n, 4 * c, h, w)


def sfb2d(ll, lh, hl, hh, filts, mode="zero"):
    """Functional single-level synthesis (pw/dwt/lowlevel.py:600-644)."""
    c_lo, c_hi, r_lo, r_hi = _four_filters(filts, prep_filt_sfb2d)
    return SFB2D.apply(ll, torch.stack([lh, hl, hh], dim=2), r_lo, r_hi, c_lo, c_hi, mode_to_int(mode))


def _filter_pair(lo, hi, device, reverse):
    dt = torch.get_default_dtype()
    out = []
    for f in (lo, hi):
        a = np.asarray(f, dtype=np.float64).ravel()
        if reverse:
            a = a[::-1].copy()
        out.append(torch.tensor(a, device=device, dtype=dt).reshape(1, 1, -1))
    return out[0], out[1]


def _to_2d(col_pair, row_pair):
    return (col_pair[0].reshape(1, 1, -1, 1), col_pair[1].reshape(1, 1, -1, 1),
            row_pair[0].reshape(1, 1, 1, -1), row_pair[1].reshape(1, 1, 1, -1))


def prep_filt_sfb1d(g0, g1, device=None):
    """Synthesis taps as (1,1,L) tensors of the default dtype, NOT mirrored (pw/dwt/lowlevel.py:902-922)."""
    return _filter_pair(g0, g1, device, reverse=False)


def prep_filt_sfb2d(g0_col, g1_col, g0_row=None, g1_row=None, device=None):
    """(g0_col, g1_col) as (1,1,L,1) and (g0_row, g1_row) as (1,1,1,L) (pw/dwt/lowlevel.py:870-899)."""
    col = prep_filt_sfb1d(g0_col, g1_col, device)
    row = col if g0_row is None else prep_filt_sfb1d(g0_row, g1_row, device)
    return _to_2d(col, row)


def prep_filt_afb1d(h0, h1, device=None):
    """Analysis taps, time-reversed because the filter bank correlates (pw/dwt/lowlevel.py:956-975)."""
    return _filter_pair(h0, h1, device, reverse=True)


def prep_filt_afb2d(h0_col, h1_col, h0_row=None, h1_row=None, device=None):
    """pw/dwt/lowlevel.py:925-953.  (The reference's ``h0_row=None`` branch has a typo, :945, that
    leaves ``h1_row`` undefined; here it means "same as the column filters", as its docstring says.)"""
    col = prep_filt_afb1d(h0_col, h1_col, device)
    row = col if h0_row is None else prep_filt_afb1d(h0_row, h1_row, device)
    return _to_2d(col, row)
