"""Double-precision ops ``b200wave64::*`` (the reference's fp64 mode: modules built under
``torch.set_default_dtype(torch.float64)``, ``tests/test_dwt.py:132-160``, or double images for SSIM and TVLoss).

Same contract as the fp32 ops -- outputs allocated by torch, launch on the current stream, CUDA-only, the same
backward structure -- on double tensors with double taps.  The bodies are the fp32 ops' own (``ops.py``, ``losses.py``,
``freq.py``) bound to ``ops.F64``; this module defines and registers the ops:

* ``afb2d`` / ``sfb2d``: the one-thread-per-output direct kernels of ``csrc/dwt.cu`` instantiated for ``double``;
  ``DWTForward`` / ``DWTInverse`` run fp64 transforms level by level through them (precision, not speed, is the point
  of this path).  ``afb2d`` backward = ``sfb2d`` with the analysis taps + crop, ``sfb2d`` backward = ``afb2d`` with the
  synthesis taps.
* ``afb1d`` / ``sfb1d`` (``csrc/dwt1d.cu``), ``swt2d`` / ``swt2d_adjoint`` (``csrc/swt.cu``), ``iswt2d``
  (``csrc/swt_inverse.cu``), ``tv_sums`` / ``tv_grad``
  (``csrc/tv.cu``): the fp32 kernels instantiated for ``double``.  As in fp32, ``losses.TVLoss`` differentiates
  ``tv_sums`` through ``tv_grad`` (once differentiable).
* ``ssim_fwd`` / ``ssim_bwd`` (``csrc/ssim_f64.cu``): ``win`` is the DENSE ws x ws window, row-major (in double the
  reference's window is the fp32 rounding of an outer product, which is not separable).  ``msssim_scale`` /
  ``msssim_scale_bwd``: one MS-SSIM scale on the same kernels, as ``ops.msssim_scale``.
* ``afb2d_select`` (``b200w_afb2d_ex_f64``): the discriminators' ``filter_wavelet`` level (``fsd.py``) on the direct
  kernel; backward = ``sfb2d`` of ``(dlow, hi_scale * dhighs)``, as ``ops.afb2d_select``.
* ``freq_mask_`` / ``abs_sign`` / ``sign_mul`` (``csrc/freq.cu``): the pointwise passes of ``freq.gaussian_split`` on
  complex128 / double tensors; the mask is rounded to fp32 as the reference stores it.
"""
import functools

import torch

from . import freq, losses, ops
from .ops import F64

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
_LIB.define("msssim_scale(Tensor img1, Tensor img2, float[] win, bool cs, bool pool, int n_maps) "
            "-> (Tensor, Tensor, Tensor, Tensor)")
_LIB.define("msssim_scale_bwd(Tensor img1, Tensor img2, Tensor maps, Tensor grad_out, float[] win, Tensor? up1, "
            "Tensor? up2, bool need_d2) -> (Tensor, Tensor)")
_LIB.define("tv_sums(Tensor x) -> Tensor")
_LIB.define("tv_grad(Tensor x, Tensor grad_out, float ch, float cw) -> Tensor")
_LIB.define("afb2d_select(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, bool want_low, "
            "bool want_highs, float hi_scale, float hi_shift) -> (Tensor, Tensor)")
_LIB.define("freq_mask_(Tensor(a!) spec, int rows, int cols, float radius, bool highpass) -> Tensor(a!)")
_LIB.define("abs_sign(Tensor x, float sign) -> Tensor")
_LIB.define("sign_mul(Tensor g, Tensor x, float sign) -> Tensor")

_LIB.impl("afb2d", functools.partial(ops._afb2d_cuda, F64), "CUDA")
_LIB.impl("sfb2d", functools.partial(ops._sfb2d_cuda, F64), "CUDA")
_LIB.impl("afb1d", functools.partial(ops._afb1d_cuda, F64), "CUDA")
_LIB.impl("sfb1d", functools.partial(ops._sfb1d_cuda, F64), "CUDA")
_LIB.impl("swt2d", functools.partial(ops._swt2d_cuda, F64), "CUDA")
_LIB.impl("swt2d_adjoint", functools.partial(ops._swt2d_adjoint_cuda, F64), "CUDA")
_LIB.impl("iswt2d", functools.partial(ops._iswt2d_cuda, F64), "CUDA")
_LIB.impl("ssim_fwd", functools.partial(ops._ssim_fwd_cuda, F64), "CUDA")
_LIB.impl("ssim_bwd", functools.partial(ops._ssim_bwd_cuda, F64), "CUDA")
_LIB.impl("msssim_scale", functools.partial(ops._msssim_scale_cuda, F64), "CUDA")
_LIB.impl("msssim_scale_bwd", functools.partial(ops._msssim_scale_bwd_cuda, F64), "CUDA")
_LIB.impl("tv_sums", functools.partial(losses._tv_sums_cuda, F64), "CUDA")
_LIB.impl("tv_grad", functools.partial(losses._tv_grad_cuda, F64), "CUDA")
_LIB.impl("afb2d_select", functools.partial(ops._afb2d_select_cuda, F64), "CUDA")
_LIB.impl("freq_mask_", functools.partial(freq._mask_cuda, F64), "CUDA")
_LIB.impl("abs_sign", functools.partial(freq._abs_sign_cuda, F64), "CUDA")
_LIB.impl("sign_mul", functools.partial(freq._sign_mul_cuda, F64), "CUDA")
for _name in ("afb2d", "sfb2d", "afb1d", "sfb1d", "swt2d", "swt2d_adjoint", "ssim_fwd", "ssim_bwd", "tv_sums",
              "tv_grad", "afb2d_select", "freq_mask_", "abs_sign", "sign_mul", "iswt2d", "msssim_scale",
              "msssim_scale_bwd"):
    _LIB.impl(_name, ops._cpu_refuse(F64.ns, _name), "CPU")
torch.library.register_fake("b200wave64::afb2d", ops._afb2d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::sfb2d", ops._sfb2d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::afb1d", ops._afb1d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::sfb1d", ops._sfb1d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::swt2d", ops._swt2d_fake, lib=_LIB)
torch.library.register_fake("b200wave64::swt2d_adjoint", ops._swt2d_adjoint_fake, lib=_LIB)
torch.library.register_fake("b200wave64::ssim_fwd", ops._ssim_fwd_fake, lib=_LIB)
torch.library.register_fake("b200wave64::ssim_bwd", ops._ssim_bwd_fake, lib=_LIB)
torch.library.register_fake("b200wave64::tv_sums", losses._tv_sums_fake, lib=_LIB)
torch.library.register_fake("b200wave64::tv_grad", losses._tv_grad_fake, lib=_LIB)
torch.library.register_autograd("b200wave64::afb2d", functools.partial(ops._afb2d_backward, F64),
                                setup_context=ops._afb2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::sfb2d", functools.partial(ops._sfb2d_backward, F64),
                                setup_context=ops._sfb2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::afb1d", functools.partial(ops._afb1d_backward, F64),
                                setup_context=ops._afb1d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::sfb1d", functools.partial(ops._sfb1d_backward, F64),
                                setup_context=ops._sfb1d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::swt2d", functools.partial(ops._swt2d_backward, F64),
                                setup_context=ops._swt2d_setup, lib=_LIB)
torch.library.register_fake("b200wave64::iswt2d", ops._iswt2d_fake, lib=_LIB)
torch.library.register_autograd("b200wave64::iswt2d", functools.partial(ops._iswt2d_backward, F64),
                                setup_context=ops._iswt2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave64::ssim_fwd", functools.partial(ops._ssim_backward, F64),
                                setup_context=ops._ssim_setup, lib=_LIB)
torch.library.register_fake("b200wave64::msssim_scale", ops._msssim_scale_fake, lib=_LIB)
torch.library.register_fake("b200wave64::msssim_scale_bwd", ops._msssim_scale_bwd_fake, lib=_LIB)
torch.library.register_autograd("b200wave64::msssim_scale", functools.partial(ops._msssim_scale_backward, F64),
                                setup_context=ops._msssim_scale_setup, lib=_LIB)
torch.library.register_fake("b200wave64::afb2d_select", ops._afb2d_select_fake, lib=_LIB)
torch.library.register_autograd("b200wave64::afb2d_select", functools.partial(ops._afb2d_select_backward, F64),
                                setup_context=ops._afb2d_select_setup, lib=_LIB)

afb2d = torch.ops.b200wave64.afb2d
sfb2d = torch.ops.b200wave64.sfb2d
afb1d = torch.ops.b200wave64.afb1d
sfb1d = torch.ops.b200wave64.sfb1d
swt2d = torch.ops.b200wave64.swt2d
swt2d_adjoint = torch.ops.b200wave64.swt2d_adjoint
iswt2d = torch.ops.b200wave64.iswt2d
ssim_fwd = torch.ops.b200wave64.ssim_fwd
ssim_bwd = torch.ops.b200wave64.ssim_bwd
msssim_scale = torch.ops.b200wave64.msssim_scale
msssim_scale_bwd = torch.ops.b200wave64.msssim_scale_bwd
tv_sums = torch.ops.b200wave64.tv_sums
tv_grad = torch.ops.b200wave64.tv_grad
afb2d_select = torch.ops.b200wave64.afb2d_select
freq_mask_ = torch.ops.b200wave64.freq_mask_
abs_sign = torch.ops.b200wave64.abs_sign
sign_mul = torch.ops.b200wave64.sign_mul
