"""Double-precision ops ``b200wave64::*`` (the reference's fp64 mode: modules built under
``torch.set_default_dtype(torch.float64)``, ``tests/test_dwt.py:132-160``, or double images for SSIM and TVLoss).

Same contract as the fp32 ops in ``ops.py`` and ``losses.py`` -- outputs allocated by torch, launch on the current
stream, CUDA-only, the same backward structure -- on double tensors with double taps:

* ``afb2d`` / ``sfb2d``: the one-thread-per-output direct kernels of ``csrc/dwt.cu`` instantiated for ``double``;
  ``DWTForward`` / ``DWTInverse`` run fp64 transforms level by level through them (precision, not speed, is the point
  of this path).  ``afb2d`` backward = ``sfb2d`` with the analysis taps + crop, ``sfb2d`` backward = ``afb2d`` with the
  synthesis taps.
* ``afb1d`` / ``sfb1d`` (``csrc/dwt1d.cu``), ``swt2d`` / ``swt2d_adjoint`` (``csrc/swt.cu``), ``iswt2d``
  (``csrc/swt_inverse.cu``), ``tv_sums`` / ``tv_grad``
  (``csrc/tv.cu``): the fp32 kernels instantiated for ``double``.  As in fp32, ``losses.TVLoss`` differentiates
  ``tv_sums`` through ``tv_grad`` (once differentiable).
* ``ssim_fwd`` / ``ssim_bwd`` (``csrc/ssim_f64.cu``): ``win`` is the DENSE ws x ws window, row-major (in double the
  reference's window is the fp32 rounding of an outer product, which is not separable).
* ``afb2d_select`` (``b200w_afb2d_ex_f64``): the discriminators' ``filter_wavelet`` level (``fsd.py``) on the direct
  kernel; backward = ``sfb2d`` of ``(dlow, hi_scale * dhighs)``, as ``ops.afb2d_select``.
* ``freq_mask_`` / ``abs_sign`` / ``sign_mul`` (``csrc/freq.cu``): the pointwise passes of ``freq.gaussian_split`` on
  complex128 / double tensors; the mask is rounded to fp32 as the reference stores it.
"""
import torch

from . import _cabi
from .ops import (_check_mode, _check_swt_mode, _mode_name, _planes_view, _rows_view, _stream, coeff_len, idwt_len,
                  iswt2d_backward, iswt_adjoint_taps, iswt_layout)

_LIB = torch.library.Library("b200wave64", "DEF")
_LIB.define("afb2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode) -> (Tensor, Tensor)")
_LIB.define("sfb2d(Tensor low, Tensor? highs, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
            "int out_h, int out_w) -> Tensor")
_LIB.define("afb1d(Tensor x, float[] h0, float[] h1, int mode) -> (Tensor, Tensor)")
_LIB.define("sfb1d(Tensor low, Tensor? high, float[] g0, float[] g1, int mode, int out_len) -> Tensor")
_LIB.define("swt2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, int dilation) -> Tensor")
_LIB.define("swt2d_adjoint(Tensor dy, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, int dilation) "
            "-> Tensor")
_LIB.define("iswt2d(Tensor ll, Tensor y, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int dilation) -> Tensor")
_LIB.define("ssim_fwd(Tensor img1, Tensor img2, float[] win, bool size_average, int n_maps) -> (Tensor, Tensor)")
_LIB.define("ssim_bwd(Tensor img1, Tensor img2, Tensor maps, Tensor grad_out, float[] win, bool size_average, "
            "bool need_d2) -> (Tensor, Tensor)")
_LIB.define("tv_sums(Tensor x) -> Tensor")
_LIB.define("tv_grad(Tensor x, Tensor grad_out, float ch, float cw) -> Tensor")
_LIB.define("afb2d_select(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, bool want_low, "
            "bool want_highs, float hi_scale, float hi_shift) -> (Tensor, Tensor)")
_LIB.define("freq_mask_(Tensor(a!) spec, int rows, int cols, float radius, bool highpass) -> Tensor(a!)")
_LIB.define("abs_sign(Tensor x, float sign) -> Tensor")
_LIB.define("sign_mul(Tensor g, Tensor x, float sign) -> Tensor")


def _require_cuda_f64(t, name):
    if not t.is_cuda:
        raise RuntimeError("b200wave64::%s is CUDA-only (sm_100a); there is no CPU fallback -- got a %s tensor"
                           % (name, t.device))
    if t.dtype != torch.float64:
        raise RuntimeError("b200wave64::%s: expected scalar type Double but found %s" % (name, t.dtype))


def _taps(*lists):
    return [_cabi.taps_array_f64(v)[0] for v in lists]


def _afb2d_cuda(x, w_lo, w_hi, h_lo, h_hi, mode):
    _check_mode(mode)
    _require_cuda_f64(x, "afb2d")
    if x.dim() != 4:
        raise IndexError("b200wave64::afb2d expects a 4-D (N, C, H, W) tensor, got %d-D" % x.dim())
    lib = _cabi.load()
    N, C, H, W = x.shape
    Lw, Lh = len(w_lo), len(h_lo)
    Ho, Wo = coeff_len(H, Lh, mode), coeff_len(W, Lw, mode)
    low = torch.empty((N, C, Ho, Wo), device=x.device, dtype=torch.float64)
    highs = torch.empty((N, C, 3, Ho, Wo), device=x.device, dtype=torch.float64)
    if low.numel() == 0:
        return low, highs
    xk, ps, rs = _planes_view(x)
    a = _taps(w_lo, w_hi, h_lo, h_hi)
    with torch.cuda.device(x.device):
        rc = lib.b200w_afb2d_f64(xk.data_ptr(), ps, rs, N * C, H, W, a[0], a[1], Lw, a[2], a[3], Lh, int(mode),
                                 low.data_ptr(), highs.data_ptr(), _stream())
    _cabi.check(rc, _mode_name(mode))
    return low, highs


def _sfb2d_cuda(low, highs, w_lo, w_hi, h_lo, h_hi, mode, out_h, out_w):
    _check_mode(mode)
    _require_cuda_f64(low, "sfb2d")
    if low.dim() != 4:
        raise IndexError("b200wave64::sfb2d expects a 4-D (N, C, h, w) tensor, got %d-D" % low.dim())
    lib = _cabi.load()
    N, C, h, w = low.shape
    if highs is not None:
        _require_cuda_f64(highs, "sfb2d")
        if tuple(highs.shape) != (N, C, 3, h, w):
            raise RuntimeError("b200wave64::sfb2d: highs must be (N, C, 3, h, w) = %s, got %s"
                               % ((N, C, 3, h, w), tuple(highs.shape)))
    Lw, Lh = len(w_lo), len(h_lo)
    oh = idwt_len(h, Lh, mode) if out_h < 0 else out_h
    ow = idwt_len(w, Lw, mode) if out_w < 0 else out_w
    y = torch.empty((N, C, oh, ow), device=low.device, dtype=torch.float64)
    if y.numel() == 0:
        return y
    lk, ps, rs = _planes_view(low)
    hk = None if highs is None else highs.contiguous()
    a = _taps(w_lo, w_hi, h_lo, h_hi)
    with torch.cuda.device(low.device):
        rc = lib.b200w_sfb2d_f64(lk.data_ptr(), ps, rs, None if hk is None else hk.data_ptr(), N * C, h, w, a[0], a[1],
                                 Lw, a[2], a[3], Lh, int(mode), y.data_ptr(), oh, ow, _stream())
    _cabi.check(rc, _mode_name(mode))
    return y


def _afb2d_fake(x, w_lo, w_hi, h_lo, h_hi, mode):
    N, C, H, W = x.shape
    Ho, Wo = coeff_len(H, len(h_lo), mode), coeff_len(W, len(w_lo), mode)
    return x.new_empty((N, C, Ho, Wo)), x.new_empty((N, C, 3, Ho, Wo))


def _sfb2d_fake(low, highs, w_lo, w_hi, h_lo, h_hi, mode, out_h, out_w):
    N, C, h, w = low.shape
    oh = idwt_len(h, len(h_lo), mode) if out_h < 0 else out_h
    ow = idwt_len(w, len(w_lo), mode) if out_w < 0 else out_w
    return low.new_empty((N, C, oh, ow))


def _afb2d_setup(ctx, inputs, output):
    x, w_lo, w_hi, h_lo, h_hi, mode = inputs
    ctx.taps = (w_lo, w_hi, h_lo, h_hi)
    ctx.mode = mode
    ctx.in_hw = (x.shape[-2], x.shape[-1])
    ctx.set_materialize_grads(False)


def _afb2d_backward(ctx, dlow, dhighs):
    dx = None
    if ctx.needs_input_grad[0]:
        if dlow is None and dhighs is None:
            return None, None, None, None, None, None
        if dlow is None:
            n, c, _, h, w = dhighs.shape
            dlow = dhighs.new_zeros((n, c, h, w))
        H, W = ctx.in_hw
        dx = torch.ops.b200wave64.sfb2d(dlow, dhighs, *ctx.taps, ctx.mode, H, W)     # lowlevel.py:356-364
    return dx, None, None, None, None, None


def _sfb2d_setup(ctx, inputs, output):
    low, highs, w_lo, w_hi, h_lo, h_hi, mode, out_h, out_w = inputs
    ctx.taps = (w_lo, w_hi, h_lo, h_hi)
    ctx.mode = mode
    ctx.has_highs = highs is not None
    ctx.cropped = tuple(output.shape[-2:]) != (idwt_len(low.shape[-2], len(h_lo), mode),
                                               idwt_len(low.shape[-1], len(w_lo), mode))


def _sfb2d_backward(ctx, dy):
    dlow = dhighs = None
    need_low = ctx.needs_input_grad[0]
    need_high = ctx.has_highs and ctx.needs_input_grad[1]
    if need_low or need_high:
        if ctx.cropped:
            raise RuntimeError("b200wave64::sfb2d: backward through a cropped synthesis is not defined")
        dlow, dhighs = torch.ops.b200wave64.afb2d(dy, *ctx.taps, ctx.mode)                # lowlevel.py:687-693
        if not need_low:
            dlow = None
        if not need_high:
            dhighs = None
    return dlow, dhighs, None, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------- afb2d_select
def _afb2d_select_cuda(x, w_lo, w_hi, h_lo, h_hi, mode, want_low, want_highs, hi_scale, hi_shift):
    """One analysis level that writes only the sub-bands asked for, the detail bands as hi_scale*v + hi_shift; an
    output that is not wanted comes back with 0 elements."""
    _check_mode(mode)
    _require_cuda_f64(x, "afb2d_select")
    if x.dim() != 4:
        raise IndexError("b200wave64::afb2d_select expects a 4-D (N, C, H, W) tensor, got %d-D" % x.dim())
    if not (want_low or want_highs):
        raise ValueError("afb2d_select: at least one of the low-pass / detail outputs must be requested")
    lib = _cabi.load()
    N, C, H, W = x.shape
    Lw, Lh = len(w_lo), len(h_lo)
    if len(w_hi) != Lw or len(h_hi) != Lh:
        raise RuntimeError("low- and high-pass filters must have the same length along an axis")
    Ho, Wo = coeff_len(H, Lh, mode), coeff_len(W, Lw, mode)
    low = torch.empty((N, C, Ho, Wo) if want_low else (0,), device=x.device, dtype=torch.float64)
    highs = torch.empty((N, C, 3, Ho, Wo) if want_highs else (0,), device=x.device, dtype=torch.float64)
    if N * C * Ho * Wo == 0:
        return low, highs
    xk, ps, rs = _planes_view(x)
    a = _taps(w_lo, w_hi, h_lo, h_hi)
    with torch.cuda.device(x.device):
        rc = lib.b200w_afb2d_ex_f64(xk.data_ptr(), ps, rs, N * C, H, W, a[0], a[1], Lw, a[2], a[3], Lh, int(mode),
                                    low.data_ptr() if want_low else None, highs.data_ptr() if want_highs else None,
                                    float(hi_scale), float(hi_shift), _stream())
    _cabi.check(rc, _mode_name(mode))
    return low, highs


def _afb2d_select_fake(x, w_lo, w_hi, h_lo, h_hi, mode, want_low, want_highs, hi_scale, hi_shift):
    N, C, H, W = x.shape
    Ho, Wo = coeff_len(H, len(h_lo), mode), coeff_len(W, len(w_lo), mode)
    return (x.new_empty((N, C, Ho, Wo) if want_low else (0,)),
            x.new_empty((N, C, 3, Ho, Wo) if want_highs else (0,)))


def _afb2d_select_setup(ctx, inputs, output):
    x, w_lo, w_hi, h_lo, h_hi, mode, want_low, want_highs, hi_scale, _ = inputs
    ctx.taps = (w_lo, w_hi, h_lo, h_hi)
    ctx.mode = mode
    ctx.in_shape = tuple(x.shape)
    ctx.want = (want_low, want_highs)
    ctx.hi_scale = hi_scale
    ctx.set_materialize_grads(False)


def _afb2d_select_backward(ctx, dlow, dhighs):
    none = (None,) * 10
    if not ctx.needs_input_grad[0]:
        return none
    want_low, want_highs = ctx.want
    dlow = dlow if want_low else None
    dhighs = dhighs if want_highs else None
    if dlow is None and dhighs is None:
        return none
    N, C, H, W = ctx.in_shape
    if dlow is None:
        dlow = dhighs.new_zeros((N, C) + tuple(dhighs.shape[-2:]))
    if dhighs is not None and ctx.hi_scale != 1.0:
        dhighs = dhighs * ctx.hi_scale   # d(hi_scale * v + hi_shift) / dv
    # AFB2D.backward's pseudo-adjoint (lowlevel.py:356-364); a missing detail gradient is never materialised
    dx = torch.ops.b200wave64.sfb2d(dlow, dhighs, *ctx.taps, ctx.mode, H, W)
    return (dx,) + none[1:]


# ------------------------------------------------------------------------------------------- 1-D banks
def _afb1d_cuda(x, h0, h1, mode):
    _check_mode(mode)
    _require_cuda_f64(x, "afb1d")
    if x.dim() != 3:
        raise IndexError("b200wave64::afb1d expects a 3-D (N, C, L) tensor, got %d-D" % x.dim())
    if len(h0) != len(h1):
        raise RuntimeError("low- and high-pass filters must have the same length")
    lib = _cabi.load()
    N, C, n = x.shape
    m = coeff_len(n, len(h0), mode)
    lo = torch.empty((N, C, m), device=x.device, dtype=torch.float64)
    hi = torch.empty((N, C, m), device=x.device, dtype=torch.float64)
    if lo.numel() == 0:
        return lo, hi
    xk, rs = _rows_view(x)
    a = _taps(h0, h1)
    with torch.cuda.device(x.device):
        rc = lib.b200w_afb1d_f64(xk.data_ptr(), rs, N * C, n, a[0], a[1], len(h0), int(mode), lo.data_ptr(),
                                 hi.data_ptr(), _stream())
    _cabi.check(rc, _mode_name(mode))
    return lo, hi


def _sfb1d_cuda(low, high, g0, g1, mode, out_len):
    _check_mode(mode)
    _require_cuda_f64(low, "sfb1d")
    if low.dim() != 3:
        raise IndexError("b200wave64::sfb1d expects 3-D (N, C, L) tensors, got %d-D" % low.dim())
    if high is not None:
        _require_cuda_f64(high, "sfb1d")
        if high.shape != low.shape:
            raise RuntimeError("b200wave64::sfb1d: low %s and high %s must have the same shape"
                               % (tuple(low.shape), tuple(high.shape)))
    lib = _cabi.load()
    N, C, m = low.shape
    n = idwt_len(m, len(g0), mode) if out_len < 0 else out_len
    y = torch.empty((N, C, n), device=low.device, dtype=torch.float64)
    if y.numel() == 0:
        return y
    lk, rs = _rows_view(low)
    hk = None if high is None else high.contiguous()
    a = _taps(g0, g1)
    with torch.cuda.device(low.device):
        rc = lib.b200w_sfb1d_f64(lk.data_ptr(), rs, None if hk is None else hk.data_ptr(), N * C, m, a[0], a[1],
                                 len(g0), int(mode), n, y.data_ptr(), _stream())
    _cabi.check(rc, _mode_name(mode))
    return y


def _afb1d_fake(x, h0, h1, mode):
    N, C, n = x.shape
    m = coeff_len(n, len(h0), mode)
    return x.new_empty((N, C, m)), x.new_empty((N, C, m))


def _sfb1d_fake(low, high, g0, g1, mode, out_len):
    N, C, m = low.shape
    return low.new_empty((N, C, idwt_len(m, len(g0), mode) if out_len < 0 else out_len))


def _afb1d_setup(ctx, inputs, output):
    x, h0, h1, mode = inputs
    ctx.taps = (h0, h1)
    ctx.mode = mode
    ctx.n = x.shape[-1]
    ctx.set_materialize_grads(False)


def _afb1d_backward(ctx, dlo, dhi):
    dx = None
    if ctx.needs_input_grad[0]:
        if dlo is None and dhi is None:
            return None, None, None, None
        if dlo is None:
            dlo = torch.zeros_like(dhi)
        dx = torch.ops.b200wave64.sfb1d(dlo, dhi, ctx.taps[0], ctx.taps[1], ctx.mode, ctx.n)   # lowlevel.py:417-422
    return dx, None, None, None


def _sfb1d_setup(ctx, inputs, output):
    low, high, g0, g1, mode, out_len = inputs
    ctx.taps = (g0, g1)
    ctx.mode = mode
    ctx.has_high = high is not None
    ctx.cropped = output.shape[-1] != idwt_len(low.shape[-1], len(g0), mode)


def _sfb1d_backward(ctx, dy):
    dlo = dhi = None
    need_lo = ctx.needs_input_grad[0]
    need_hi = ctx.has_high and ctx.needs_input_grad[1]
    if need_lo or need_hi:
        if ctx.cropped:
            raise RuntimeError("b200wave64::sfb1d: backward through a cropped synthesis is not defined "
                               "(the crop only exists inside AFB1D.backward)")
        dlo, dhi = torch.ops.b200wave64.afb1d(dy, ctx.taps[0], ctx.taps[1], ctx.mode)    # lowlevel.py:736-742
        if not need_lo:
            dlo = None
        if not need_hi:
            dhi = None
    return dlo, dhi, None, None, None, None


# ------------------------------------------------------------------------------------------- a trous (SWT)
def _swt_call(fn_name, t, w_lo, w_hi, h_lo, h_hi, mode, dilation, planes, H, W, out):
    lib = _cabi.load()
    if not (len(w_lo) == len(w_hi) == len(h_lo) == len(h_hi)):
        raise RuntimeError("b200wave64::swt2d: all four filters must have the same length")
    a = _taps(w_lo, w_hi, h_lo, h_hi)
    with torch.cuda.device(t.device):
        rc = getattr(lib, fn_name)(t.data_ptr(), planes, H, W, a[0], a[1], a[2], a[3], len(w_lo), int(dilation),
                                   int(mode), out.data_ptr(), _stream())
    _cabi.check(rc, _mode_name(mode))


def _swt2d_cuda(x, w_lo, w_hi, h_lo, h_hi, mode, dilation):
    _check_swt_mode(mode)
    _require_cuda_f64(x, "swt2d")
    if x.dim() != 4:
        raise IndexError("b200wave64::swt2d expects a 4-D (N, C, H, W) tensor, got %d-D" % x.dim())
    N, C, H, W = x.shape
    y = torch.empty((N, 4 * C, H, W), device=x.device, dtype=torch.float64)
    if y.numel():
        _swt_call("b200w_swt2d_fwd_f64", x.contiguous(), w_lo, w_hi, h_lo, h_hi, mode, dilation, N * C, H, W, y)
    return y


def _swt2d_adjoint_cuda(dy, w_lo, w_hi, h_lo, h_hi, mode, dilation):
    _check_swt_mode(mode)
    _require_cuda_f64(dy, "swt2d_adjoint")
    N, C4, H, W = dy.shape
    dx = torch.empty((N, C4 // 4, H, W), device=dy.device, dtype=torch.float64)
    if dx.numel():
        _swt_call("b200w_swt2d_bwd_f64", dy.contiguous(), w_lo, w_hi, h_lo, h_hi, mode, dilation, N * (C4 // 4), H, W,
                  dx)
    return dx


def _swt2d_setup(ctx, inputs, output):
    x, w_lo, w_hi, h_lo, h_hi, mode, dilation = inputs
    ctx.args = (w_lo, w_hi, h_lo, h_hi, mode, dilation)


def _swt2d_backward(ctx, dy):
    dx = None
    if ctx.needs_input_grad[0]:
        dx = torch.ops.b200wave64.swt2d_adjoint(dy, *ctx.args)
    return dx, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------- inverse SWT
def _iswt2d_cuda(ll, y, w_lo, w_hi, h_lo, h_hi, dilation):
    _require_cuda_f64(ll, "iswt2d")
    _require_cuda_f64(y, "iswt2d")
    if not (len(w_lo) == len(w_hi) == len(h_lo) == len(h_hi)):
        raise RuntimeError("b200wave64::iswt2d: all four filters must have the same length")
    lk, ps, yk = iswt_layout(ll, y, "b200wave64::iswt2d")
    N, C4, H, W = yk.shape
    x = torch.empty((N, C4 // 4, H, W), device=y.device, dtype=torch.float64)
    if x.numel() == 0:
        return x
    lib = _cabi.load()
    a = _taps(w_lo, w_hi, h_lo, h_hi)
    with torch.cuda.device(y.device):
        rc = lib.b200w_iswt2d_f64(lk.data_ptr(), ps, yk.data_ptr(), N * (C4 // 4), H, W, a[0], a[1], a[2], a[3],
                                  len(w_lo), int(dilation), x.data_ptr(), _stream())
    _cabi.check(rc)
    return x


def _iswt2d_setup(ctx, inputs, output):
    ll, y, w_lo, w_hi, h_lo, h_hi, dilation = inputs
    ctx.taps = iswt_adjoint_taps(w_lo, w_hi, h_lo, h_hi)
    ctx.dilation = dilation


def _iswt2d_backward(ctx, dx):
    return iswt2d_backward(torch.ops.b200wave64.swt2d, ctx, dx)


# ------------------------------------------------------------------------------------------- ssim
def _ssim_common(img1, img2, win, name):
    _require_cuda_f64(img1, name)
    _require_cuda_f64(img2, name)
    if img1.dim() != 4 or img1.shape != img2.shape:
        raise RuntimeError("b200wave64::%s expects two (N, C, H, W) tensors of equal shape, got %s and %s"
                           % (name, tuple(img1.shape), tuple(img2.shape)))
    ws = int(round(len(win) ** 0.5))
    if ws * ws != len(win) or ws % 2 == 0 or ws > _cabi.SSIM_MAX_WINDOW:
        raise RuntimeError("b200wave64::%s: the window must be ws x ws taps with ws odd and <= %d, got %d taps"
                           % (name, _cabi.SSIM_MAX_WINDOW, len(win)))
    return ws


def _ssim_fwd_cuda(img1, img2, win, size_average, n_maps):
    ws = _ssim_common(img1, img2, win, "ssim_fwd")
    lib = _cabi.load()
    img1, img2 = img1.contiguous(), img2.contiguous()
    N, C, H, W = img1.shape
    out = torch.empty(() if size_average else (N,), device=img1.device, dtype=torch.float64)
    maps = torch.empty((n_maps, N, C, H, W), device=img1.device, dtype=torch.float64)
    ws_bytes = lib.b200w_ssim_workspace_bytes_f64(N, C, H, W)
    work = torch.empty((max(ws_bytes, 8) // 8,), device=img1.device, dtype=torch.float64)
    a_win, _ = _cabi.taps_array_f64(win)
    with torch.cuda.device(img1.device):
        rc = lib.b200w_ssim_fwd_f64(img1.data_ptr(), img2.data_ptr(), N, C, H, W, a_win, ws, int(size_average),
                                    int(n_maps), maps.data_ptr() if n_maps else None, out.data_ptr(),
                                    work.data_ptr(), ws_bytes, _stream())
    _cabi.check(rc)
    return out, maps


def _ssim_fwd_fake(img1, img2, win, size_average, n_maps):
    N, C, H, W = img1.shape
    return img1.new_empty(() if size_average else (N,)), img1.new_empty((n_maps, N, C, H, W))


def _ssim_bwd_cuda(img1, img2, maps, grad_out, win, size_average, need_d2):
    ws = _ssim_common(img1, img2, win, "ssim_bwd")
    lib = _cabi.load()
    img1, img2, maps = img1.contiguous(), img2.contiguous(), maps.contiguous()
    N, C, H, W = img1.shape
    n_maps = maps.shape[0]
    if n_maps not in (3, 4) or (need_d2 and n_maps != 4):
        raise RuntimeError("b200wave64::ssim_bwd: forward saved %d derivative maps, not enough for this backward"
                           % n_maps)
    g = grad_out.to(device=img1.device, dtype=torch.float64).contiguous()
    if g.numel() != (1 if size_average else N):
        raise RuntimeError("b200wave64::ssim_bwd: grad_out has %d elements" % g.numel())
    d1 = torch.empty_like(img1)
    d2 = torch.empty_like(img2) if need_d2 else torch.empty((0,), device=img1.device, dtype=torch.float64)
    a_win, _ = _cabi.taps_array_f64(win)
    with torch.cuda.device(img1.device):
        rc = lib.b200w_ssim_bwd_f64(img1.data_ptr(), img2.data_ptr(), maps.data_ptr(), n_maps, g.data_ptr(),
                                    N, C, H, W, a_win, ws, int(size_average), d1.data_ptr(),
                                    d2.data_ptr() if need_d2 else None, _stream())
    _cabi.check(rc)
    return d1, d2


def _ssim_bwd_fake(img1, img2, maps, grad_out, win, size_average, need_d2):
    return torch.empty_like(img1), (torch.empty_like(img2) if need_d2 else img1.new_empty((0,)))


def _ssim_setup(ctx, inputs, output):
    img1, img2, win, size_average, n_maps = inputs
    _, maps = output
    ctx.save_for_backward(img1, img2, maps)
    ctx.win = win
    ctx.size_average = size_average
    ctx.n_maps = n_maps
    ctx.set_materialize_grads(False)


def _ssim_backward(ctx, dval, dmaps):
    need1, need2 = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    if not (need1 or need2) or dval is None:
        return None, None, None, None, None
    if ctx.n_maps < 3 or (need2 and ctx.n_maps < 4):
        raise RuntimeError("b200wave64::ssim_fwd was called with n_maps=%d, which does not support the requested "
                           "gradient (use 3 for d/dimg1, 4 for both)" % ctx.n_maps)
    img1, img2, maps = ctx.saved_tensors
    d1, d2 = torch.ops.b200wave64.ssim_bwd(img1, img2, maps, dval, ctx.win, ctx.size_average, bool(need2))
    return (d1 if need1 else None), (d2 if need2 else None), None, None, None


# ------------------------------------------------------------------------------------------- TV
def _check_tv(x, name):
    _require_cuda_f64(x, name)
    if x.dim() != 4:
        raise IndexError("b200wave64::%s expects a 4-D (N, C, H, W) tensor, got %d-D" % (name, x.dim()))


def _tv_sums_cuda(x):
    """(2,) double tensor: sum of squared vertical / horizontal forward differences (model.py:28-29)."""
    _check_tv(x, "tv_sums")
    lib = _cabi.load()
    xc = x.contiguous()
    n, c, h, w = xc.shape
    out = torch.zeros(2, device=x.device, dtype=torch.float64)
    if xc.numel() == 0:
        return out
    ws = torch.empty(int(lib.b200w_tv_workspace_bytes_f64(n * c, h)), device=x.device, dtype=torch.uint8)
    with torch.cuda.device(x.device):
        rc = lib.b200w_tv_fwd_f64(xc.data_ptr(), n * c, h, w, ws.data_ptr(), ws.numel(), out.data_ptr(), _stream())
    _cabi.check(rc, "tv")
    return out


def _tv_grad_cuda(x, grad_out, ch, cw):
    _check_tv(x, "tv_grad")
    lib = _cabi.load()
    xc = x.contiguous()
    n, c, h, w = xc.shape
    dx = torch.empty_like(xc)
    if xc.numel() == 0:
        return dx
    g = grad_out.reshape(-1)[:1].to(torch.float64).contiguous()
    with torch.cuda.device(x.device):
        rc = lib.b200w_tv_bwd_f64(xc.data_ptr(), g.data_ptr(), float(ch), float(cw), n * c, h, w, dx.data_ptr(),
                                  _stream())
    _cabi.check(rc, "tv")
    return dx


# ------------------------------------------------------------------------------------------- frequency split
def _require_freq(t, name, dtype):
    if not t.is_cuda:
        raise RuntimeError("b200wave64::%s is CUDA-only (sm_100a); there is no CPU fallback -- got a %s tensor"
                           % (name, t.device))
    if t.dtype != dtype:
        raise RuntimeError("b200wave64::%s: expected %s but found %s" % (name, dtype, t.dtype))


def _freq_mask_cuda(spec, rows, cols, radius, highpass):
    _require_freq(spec, "freq_mask_", torch.complex128)
    if not spec.is_contiguous() or spec.shape[-2] != rows or spec.shape[-1] != cols // 2 + 1:
        raise RuntimeError("b200wave64::freq_mask_ expects the contiguous half spectrum (..., %d, %d), got %s"
                           % (rows, cols // 2 + 1, tuple(spec.shape)))
    if spec.numel() == 0:
        return spec
    planes = spec.numel() // (rows * (cols // 2 + 1))
    with torch.cuda.device(spec.device):
        rc = _cabi.load().b200w_freq_mask_c128(spec.data_ptr(), planes, rows, cols, float(radius),
                                               int(bool(highpass)), _stream())
    _cabi.check(rc)
    return spec


def _abs_sign_cuda(x, sign):
    _require_freq(x, "abs_sign", torch.float64)
    x = x.contiguous()
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = _cabi.load().b200w_abs_sign_f64(x.data_ptr(), y.data_ptr(), x.numel(), float(sign), _stream())
    _cabi.check(rc)
    return y


def _sign_mul_cuda(g, x, sign):
    _require_freq(g, "sign_mul", torch.float64)
    _require_freq(x, "sign_mul", torch.float64)
    g, x = g.contiguous(), x.contiguous()
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = _cabi.load().b200w_sign_mul_f64(g.data_ptr(), x.data_ptr(), out.data_ptr(), x.numel(), float(sign),
                                             _stream())
    _cabi.check(rc)
    return out


def _cpu_refuse(name):
    def impl(*args, **kwargs):
        raise RuntimeError("b200wave64::%s is CUDA-only (sm_100a): there is no CPU fallback. Move the tensors to "
                           "a B200 (`.cuda()`)." % name)
    return impl


_LIB.impl("afb2d", _afb2d_cuda, "CUDA")
_LIB.impl("sfb2d", _sfb2d_cuda, "CUDA")
_LIB.impl("afb1d", _afb1d_cuda, "CUDA")
_LIB.impl("sfb1d", _sfb1d_cuda, "CUDA")
_LIB.impl("swt2d", _swt2d_cuda, "CUDA")
_LIB.impl("swt2d_adjoint", _swt2d_adjoint_cuda, "CUDA")
_LIB.impl("iswt2d", _iswt2d_cuda, "CUDA")
_LIB.impl("ssim_fwd", _ssim_fwd_cuda, "CUDA")
_LIB.impl("ssim_bwd", _ssim_bwd_cuda, "CUDA")
_LIB.impl("tv_sums", _tv_sums_cuda, "CUDA")
_LIB.impl("tv_grad", _tv_grad_cuda, "CUDA")
_LIB.impl("afb2d_select", _afb2d_select_cuda, "CUDA")
_LIB.impl("freq_mask_", _freq_mask_cuda, "CUDA")
_LIB.impl("abs_sign", _abs_sign_cuda, "CUDA")
_LIB.impl("sign_mul", _sign_mul_cuda, "CUDA")
for _name in ("afb2d", "sfb2d", "afb1d", "sfb1d", "swt2d", "swt2d_adjoint", "ssim_fwd", "ssim_bwd", "tv_sums",
              "tv_grad", "afb2d_select", "freq_mask_", "abs_sign", "sign_mul", "iswt2d"):
    _LIB.impl(_name, _cpu_refuse(_name), "CPU")
torch.library.register_fake("b200wave64::afb2d", _afb2d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::sfb2d", _sfb2d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::afb1d", _afb1d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::sfb1d", _sfb1d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::swt2d", lambda x, wl, wh, hl, hh, mode, d:
                            x.new_empty((x.shape[0], 4 * x.shape[1], x.shape[2], x.shape[3])), lib=_LIB)
torch.library.register_fake("b200wave64::swt2d_adjoint", lambda dy, wl, wh, hl, hh, mode, d:
                            dy.new_empty((dy.shape[0], dy.shape[1] // 4, dy.shape[2], dy.shape[3])), lib=_LIB)
torch.library.register_fake("b200wave64::ssim_fwd", _ssim_fwd_fake, lib=_LIB)
torch.library.register_fake("b200wave64::ssim_bwd", _ssim_bwd_fake, lib=_LIB)
torch.library.register_fake("b200wave64::tv_sums", lambda x: x.new_empty((2,)), lib=_LIB)
torch.library.register_fake("b200wave64::tv_grad", lambda x, g, ch, cw: torch.empty_like(x), lib=_LIB)
torch.library.register_autograd("b200wave64::afb2d", _afb2d_backward, setup_context=_afb2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::sfb2d", _sfb2d_backward, setup_context=_sfb2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::afb1d", _afb1d_backward, setup_context=_afb1d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::sfb1d", _sfb1d_backward, setup_context=_sfb1d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::swt2d", _swt2d_backward, setup_context=_swt2d_setup, lib=_LIB)
torch.library.register_fake("b200wave64::iswt2d", lambda ll, y, wl, wh, hl, hh, d:
                            y.new_empty((y.shape[0], y.shape[1] // 4, y.shape[2], y.shape[3])), lib=_LIB)
torch.library.register_autograd("b200wave64::iswt2d", _iswt2d_backward, setup_context=_iswt2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::ssim_fwd", _ssim_backward, setup_context=_ssim_setup, lib=_LIB)
torch.library.register_fake("b200wave64::afb2d_select", _afb2d_select_fake, lib=_LIB)
torch.library.register_autograd("b200wave64::afb2d_select", _afb2d_select_backward, setup_context=_afb2d_select_setup,
                                lib=_LIB)

afb2d = torch.ops.b200wave64.afb2d
sfb2d = torch.ops.b200wave64.sfb2d
afb1d = torch.ops.b200wave64.afb1d
sfb1d = torch.ops.b200wave64.sfb1d
swt2d = torch.ops.b200wave64.swt2d
swt2d_adjoint = torch.ops.b200wave64.swt2d_adjoint
iswt2d = torch.ops.b200wave64.iswt2d
ssim_fwd = torch.ops.b200wave64.ssim_fwd
ssim_bwd = torch.ops.b200wave64.ssim_bwd
tv_sums = torch.ops.b200wave64.tv_sums
tv_grad = torch.ops.b200wave64.tv_grad
afb2d_select = torch.ops.b200wave64.afb2d_select
freq_mask_ = torch.ops.b200wave64.freq_mask_
abs_sign = torch.ops.b200wave64.abs_sign
sign_mul = torch.ops.b200wave64.sign_mul
