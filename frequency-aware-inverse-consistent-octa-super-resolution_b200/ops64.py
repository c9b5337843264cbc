"""Double-precision single-level ops ``b200wave::afb2d_f64`` / ``sfb2d_f64`` (the reference's fp64 mode: modules built
under ``torch.set_default_dtype(torch.float64)``, ``tests/test_dwt.py:132-160``).

Same contract as the fp32 ops in ``ops.py`` -- outputs allocated by torch, launch on the current stream, CUDA-only, the
reference's hand-written backward (``afb2d`` backward = ``sfb2d`` with the analysis taps + crop, ``sfb2d`` backward =
``afb2d`` with the synthesis taps) -- on double tensors with double taps, through the one-thread-per-output direct
kernels of ``csrc/dwt.cu``, instantiated for ``double``.  ``DWTForward`` / ``DWTInverse`` run fp64 transforms level by level through these ops
(precision, not speed, is the point of this path).
"""
import torch

from . import _cabi
from .ops import _check_mode, _mode_name, _planes_view, _stream, coeff_len, idwt_len

_LIB = torch.library.Library("b200wave64", "DEF")
_LIB.define("afb2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode) -> (Tensor, Tensor)")
_LIB.define("sfb2d(Tensor low, Tensor? highs, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
            "int out_h, int out_w) -> Tensor")


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


def _cpu_refuse(name):
    def impl(*args, **kwargs):
        raise RuntimeError("b200wave64::%s is CUDA-only (sm_100a): there is no CPU fallback. Move the tensors to "
                           "a B200 (`.cuda()`)." % name)
    return impl


_LIB.impl("afb2d", _afb2d_cuda, "CUDA")
_LIB.impl("sfb2d", _sfb2d_cuda, "CUDA")
_LIB.impl("afb2d", _cpu_refuse("afb2d"), "CPU")
_LIB.impl("sfb2d", _cpu_refuse("sfb2d"), "CPU")
torch.library.register_fake("b200wave64::afb2d", _afb2d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::sfb2d", _sfb2d_fake, lib=_LIB)
torch.library.register_autograd("b200wave64::afb2d", _afb2d_backward, setup_context=_afb2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::sfb2d", _sfb2d_backward, setup_context=_sfb2d_setup, lib=_LIB)

afb2d = torch.ops.b200wave64.afb2d
sfb2d = torch.ops.b200wave64.sfb2d
