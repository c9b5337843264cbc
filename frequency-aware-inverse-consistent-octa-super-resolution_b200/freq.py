"""Fourier-domain Gaussian frequency split -- host mirror of ``utils.py:71-117`` of the reference
(``guais_low_pass`` / ``guais_high_pass`` / ``high_pass`` / ``low_pass``), SURVEY.md section 8f row 1.

``train.py:173-213`` calls ``utils.high_pass(real_A[0], i=10)`` / ``utils.low_pass(real_A[0], i=8)`` eight times per
step; each call rebuilds the mask with two Python loops on the host, uploads it, and filters ONE image with a complex
``fft2``.  Here the transform is batched over every plane, uses the half spectrum (``rfft2`` / ``irfft2``, cuFFT), and
the mask is evaluated inside the pointwise kernel (``csrc/freq.cu``) -- no mask tensor, no fftshift, no host work.

* ``high_pass(timg, i=4)`` / ``low_pass(timg, i=10)``: same signature and result as the reference (``timg`` is
  ``(1, H, W)``; the result is ``(H, W)``; ``low_pass`` returns ``-|.|`` exactly like ``utils.py:117``).
* ``gaussian_split(x, radius, highpass, sign)``: the batched form for ``(..., H, W)`` tensors.
Differentiable: the filter is linear and self-adjoint (real, even mask), ``abs`` back-propagates ``sgn``.
float32 and float64 images are served; float64 is the reference's double mode (complex128 FFTs, the mask evaluated in
double and rounded to fp32 as ``torch.from_numpy(mask).float()`` stores it), through the ``ops64`` twins of the ops.
"""
import ctypes

import torch
from torch.autograd.function import once_differentiable

from . import _cabi, ops64

_LIB = torch.library.Library("b200wave_freq", "DEF")
_LIB.define("mask_(Tensor(a!) spec, int rows, int cols, float radius, bool highpass) -> Tensor(a!)")
_LIB.define("abs_sign(Tensor x, float sign) -> Tensor")
_LIB.define("sign_mul(Tensor g, Tensor x, float sign) -> Tensor")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require(t, name, dtype):
    if not t.is_cuda:
        raise RuntimeError("b200wave_freq::%s is CUDA-only (sm_100a); there is no CPU fallback -- got a %s tensor"
                           % (name, t.device))
    if t.dtype != dtype:
        raise RuntimeError("b200wave_freq::%s: expected %s but found %s" % (name, dtype, t.dtype))


def _mask_cuda(spec, rows, cols, radius, highpass):
    _require(spec, "mask_", torch.complex64)
    if not spec.is_contiguous() or spec.shape[-2] != rows or spec.shape[-1] != cols // 2 + 1:
        raise RuntimeError("b200wave_freq::mask_ expects the contiguous half spectrum (..., %d, %d), got %s"
                           % (rows, cols // 2 + 1, tuple(spec.shape)))
    if spec.numel() == 0:
        return spec
    planes = spec.numel() // (rows * (cols // 2 + 1))
    with torch.cuda.device(spec.device):
        rc = _cabi.load().b200w_freq_mask_c64(spec.data_ptr(), planes, rows, cols, float(radius), int(bool(highpass)),
                                              _stream())
    _cabi.check(rc)
    return spec


def _abs_sign_cuda(x, sign):
    _require(x, "abs_sign", torch.float32)
    x = x.contiguous()
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = _cabi.load().b200w_abs_sign_f32(x.data_ptr(), y.data_ptr(), x.numel(), float(sign), _stream())
    _cabi.check(rc)
    return y


def _sign_mul_cuda(g, x, sign):
    _require(g, "sign_mul", torch.float32)
    _require(x, "sign_mul", torch.float32)
    g, x = g.contiguous(), x.contiguous()
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        rc = _cabi.load().b200w_sign_mul_f32(g.data_ptr(), x.data_ptr(), out.data_ptr(), x.numel(), float(sign), _stream())
    _cabi.check(rc)
    return out


def _cpu_refuse(name):
    def impl(*args, **kwargs):
        raise RuntimeError("b200wave_freq::%s is CUDA-only (sm_100a): there is no CPU fallback." % name)
    return impl


_LIB.impl("mask_", _mask_cuda, "CUDA")
_LIB.impl("abs_sign", _abs_sign_cuda, "CUDA")
_LIB.impl("sign_mul", _sign_mul_cuda, "CUDA")
for _name in ("mask_", "abs_sign", "sign_mul"):
    _LIB.impl(_name, _cpu_refuse(_name), "CPU")


# (mask_, abs_sign, sign_mul) by dtype: fp32 here, float64 / complex128 in ops64 (the reference's double mode)
_OPS = {torch.float32: (torch.ops.b200wave_freq.mask_, torch.ops.b200wave_freq.abs_sign,
                        torch.ops.b200wave_freq.sign_mul),
        torch.float64: (ops64.freq_mask_, ops64.abs_sign, ops64.sign_mul)}


def _filter(x, radius, highpass):
    """irfft2(mask * rfft2(x)) over the last two dims (cuFFT + the in-place mask kernel)."""
    rows, cols = x.shape[-2:]
    spec = torch.fft.rfft2(x).contiguous()
    _OPS[x.dtype][0](spec, rows, cols, float(radius), bool(highpass))
    return torch.fft.irfft2(spec, s=(rows, cols))


class _GaussianSplit(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, radius, highpass, sign):
        y = _filter(x, radius, highpass)
        ctx.save_for_backward(y)
        ctx.args = (radius, highpass, sign)
        return _OPS[y.dtype][1](y, float(sign))

    @staticmethod
    @once_differentiable   # the backward kernels have no autograd formula of their own: double backward raises
    def backward(ctx, g):
        (y,) = ctx.saved_tensors
        radius, highpass, sign = ctx.args
        t = _OPS[y.dtype][2](g, y, float(sign))
        return _filter(t, radius, highpass), None, None, None   # the filter is self-adjoint


def gaussian_split(x, radius, highpass, sign=1.0):
    """``sign * |ifft2(mask_r * fft2(x))|`` over the last two dims of a real fp32 or float64 CUDA tensor, batched over
    the rest.  float64 follows the reference's double mode: complex128 FFTs, the mask rounded to fp32."""
    if not x.is_cuda:
        raise RuntimeError("b200wave.freq is CUDA-only (sm_100a); there is no CPU fallback -- got a %s tensor" % x.device)
    if x.dtype not in _OPS:
        raise RuntimeError("b200wave.freq: expected scalar type Float but found %s" % x.dtype)
    if x.dim() < 2:
        raise ValueError("b200wave.freq expects (..., H, W)")
    return _GaussianSplit.apply(x, float(radius), bool(highpass), float(sign))


def high_pass(timg, i=4):
    """utils.py:93-103 -- ``timg`` is (1, H, W) (the reference filters ``timg[0]``); returns (H, W)."""
    return gaussian_split(timg[0], i, True, 1.0)


def low_pass(timg, i=10):
    """utils.py:105-117 -- returns ``-|.|`` like the reference (``iimg*-1``)."""
    return gaussian_split(timg[0], i, False, -1.0)
