"""Reduction-style losses of the training step that sit beside the wavelet / SSIM path (SURVEY.md 8f row 4).

``TVLoss`` -- drop-in for ``model.py:17-33`` (constructed at ``train.py:98``): same constructor argument, same scalar
``TVLoss_weight * 2 * (h_tv / count_h + w_tv / count_w) / batch_size``.  The reference slices ``x`` four times,
subtracts, squares and reduces (about ten elementwise passes and as many again in autograd's backward); here the two
sums come out of one pass over ``x`` (``b200w_tv_fwd_f32``) and the gradient out of one more (``b200w_tv_bwd_f32``).
Double images run through the same kernels instantiated for double (``b200w_tv_fwd_f64`` / ``b200w_tv_bwd_f64``), as
the reference computes in the images' dtype.

``phase_consistency_loss`` -- drop-in for ``model.py:36-58`` (constructed at ``train.py:94``): minus the cosine
similarity of the masked log-amplitude spectra of ``x[0]`` and ``y[0]``.  The reference rebuilds the rows x cols mask
with two Python loops on the host per call, runs two complex ``fft2`` + ``fftshift`` and ~10 elementwise / reduction
kernels.  Here: ``rfft2`` of both images (cuFFT, half spectrum), one kernel for the three inner products with the mask
evaluated in place (``b200w_phase_sums_c64``), one kernel for the gradient w.r.t. both spectra
(``b200w_phase_grad_c64``); autograd's own ``rfft2`` backward carries it to the images.
CUDA-only, like the rest of the package.
"""
import ctypes

import torch
from torch.autograd.function import once_differentiable
import torch.nn as nn

from . import _cabi, ops64

_LIB = torch.library.Library("b200wave_losses", "DEF")
_LIB.define("tv_sums(Tensor x) -> Tensor")
_LIB.define("tv_grad(Tensor x, Tensor grad_out, float ch, float cw) -> Tensor")
_LIB.define("phase_sums(Tensor fx, Tensor fy, int cols, float radius) -> Tensor")
_LIB.define("phase_grad(Tensor fx, Tensor fy, int cols, float radius, Tensor sums, Tensor grad_out, float eps) "
            "-> (Tensor, Tensor)")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check(x, name):
    if not x.is_cuda:
        raise RuntimeError("b200wave_losses::%s is CUDA-only (sm_100a); there is no CPU fallback -- got a %s tensor"
                           % (name, x.device))
    if x.dtype != torch.float32:
        raise RuntimeError("b200wave_losses::%s: expected scalar type Float but found %s" % (name, x.dtype))
    if x.dim() != 4:
        raise IndexError("b200wave_losses::%s expects a 4-D (N, C, H, W) tensor, got %d-D" % (name, x.dim()))


def _tv_sums_cuda(x):
    """(2,) tensor: sum of squared vertical / horizontal forward differences (model.py:28-29)."""
    _check(x, "tv_sums")
    lib = _cabi.load()
    xc = x.contiguous()
    n, c, h, w = xc.shape
    out = torch.zeros(2, device=x.device, dtype=torch.float32)
    if xc.numel() == 0:
        return out
    ws = torch.empty(int(lib.b200w_tv_workspace_bytes(n * c, h)), device=x.device, dtype=torch.uint8)
    with torch.cuda.device(x.device):
        rc = lib.b200w_tv_fwd_f32(xc.data_ptr(), n * c, h, w, ws.data_ptr(), ws.numel(), out.data_ptr(), _stream())
    _cabi.check(rc, "tv")
    return out


def _tv_grad_cuda(x, grad_out, ch, cw):
    _check(x, "tv_grad")
    lib = _cabi.load()
    xc = x.contiguous()
    n, c, h, w = xc.shape
    dx = torch.empty_like(xc)
    if xc.numel() == 0:
        return dx
    g = grad_out.reshape(-1)[:1].to(torch.float32).contiguous()
    with torch.cuda.device(x.device):
        rc = lib.b200w_tv_bwd_f32(xc.data_ptr(), g.data_ptr(), float(ch), float(cw), n * c, h, w, dx.data_ptr(),
                                  _stream())
    _cabi.check(rc, "tv")
    return dx


def _check_spec(f, name):
    if not f.is_cuda:
        raise RuntimeError("b200wave_losses::%s is CUDA-only (sm_100a); there is no CPU fallback -- got a %s tensor"
                           % (name, f.device))
    if f.dtype != torch.float32 or f.dim() != 4 or f.shape[-1] != 2:
        raise RuntimeError("b200wave_losses::%s expects view_as_real of a (C, rows, cols/2+1) complex64 half spectrum"
                           % name)


def _phase_sums_cuda(fx, fy, cols, radius):
    """(3,) tensor <a_x,a_y>, <a_x,a_x>, <a_y,a_y> from the two half spectra (view_as_real, (C, rows, cols/2+1, 2))."""
    _check_spec(fx, "phase_sums")
    _check_spec(fy, "phase_sums")
    if fx.shape != fy.shape or fx.shape[2] != cols // 2 + 1:
        raise RuntimeError("b200wave_losses::phase_sums: spectra of different shapes / not the half spectrum of `cols`")
    lib = _cabi.load()
    fx, fy = fx.contiguous(), fy.contiguous()
    planes, rows = fx.shape[0], fx.shape[1]
    out = torch.empty(3, device=fx.device, dtype=torch.float32)
    ws = torch.empty(int(lib.b200w_phase_workspace_bytes(planes, rows, cols)), device=fx.device, dtype=torch.uint8)
    with torch.cuda.device(fx.device):
        rc = lib.b200w_phase_sums_c64(fx.data_ptr(), fy.data_ptr(), planes, rows, cols, float(radius), ws.data_ptr(),
                                      ws.numel(), out.data_ptr(), _stream())
    _cabi.check(rc, "phase_consistency_loss")
    return out


def _phase_grad_cuda(fx, fy, cols, radius, sums, grad_out, eps):
    _check_spec(fx, "phase_grad")
    _check_spec(fy, "phase_grad")
    lib = _cabi.load()
    fx, fy = fx.contiguous(), fy.contiguous()
    planes, rows = fx.shape[0], fx.shape[1]
    gx, gy = torch.empty_like(fx), torch.empty_like(fy)
    g = grad_out.reshape(-1)[:1].to(torch.float32).contiguous()
    with torch.cuda.device(fx.device):
        rc = lib.b200w_phase_grad_c64(fx.data_ptr(), fy.data_ptr(), planes, rows, cols, float(radius),
                                      sums.contiguous().data_ptr(), g.data_ptr(), float(eps), gx.data_ptr(),
                                      gy.data_ptr(), _stream())
    _cabi.check(rc, "phase_consistency_loss")
    return gx, gy


def _cpu_refuse(name):
    def impl(*args, **kwargs):
        raise RuntimeError("b200wave_losses::%s is CUDA-only (sm_100a): there is no CPU fallback. Move the tensors "
                           "to a B200 (`.cuda()`)." % name)
    return impl


_LIB.impl("tv_sums", _tv_sums_cuda, "CUDA")
_LIB.impl("tv_grad", _tv_grad_cuda, "CUDA")
_LIB.impl("tv_sums", _cpu_refuse("tv_sums"), "CPU")
_LIB.impl("tv_grad", _cpu_refuse("tv_grad"), "CPU")
_LIB.impl("phase_sums", _phase_sums_cuda, "CUDA")
_LIB.impl("phase_grad", _phase_grad_cuda, "CUDA")
_LIB.impl("phase_sums", _cpu_refuse("phase_sums"), "CPU")
_LIB.impl("phase_grad", _cpu_refuse("phase_grad"), "CPU")
torch.library.register_fake("b200wave_losses::phase_sums", lambda fx, fy, cols, radius: fx.new_empty((3,)), lib=_LIB)
torch.library.register_fake("b200wave_losses::phase_grad",
                            lambda fx, fy, cols, radius, sums, g, eps: (torch.empty_like(fx), torch.empty_like(fy)),
                            lib=_LIB)
torch.library.register_fake("b200wave_losses::tv_sums", lambda x: x.new_empty((2,)), lib=_LIB)
torch.library.register_fake("b200wave_losses::tv_grad", lambda x, g, ch, cw: torch.empty_like(x), lib=_LIB)


class _TV(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight):
        n, c, h, w = x.shape
        count_h = c * (h - 1) * w          # model.py:26-27 via _tensor_size
        count_w = c * h * (w - 1)
        f64 = x.dtype == torch.float64
        sums = ops64.tv_sums(x) if f64 else torch.ops.b200wave_losses.tv_sums(x)
        ctx.save_for_backward(x)
        ctx.f64 = f64
        ctx.scales = (weight, n, count_h, count_w)
        # the same arithmetic as model.py:30 (a zero count divides by zero exactly as the reference does)
        return weight * 2 * (sums[0] / count_h + sums[1] / count_w) / n

    @staticmethod
    @once_differentiable   # the backward kernels have no autograd formula of their own: double backward raises
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        weight, n, count_h, count_w = ctx.scales
        ch = weight * 2.0 / (n * count_h) if count_h else float("nan")
        cw = weight * 2.0 / (n * count_w) if count_w else float("nan")
        grad = ops64.tv_grad if ctx.f64 else torch.ops.b200wave_losses.tv_grad
        return grad(x, g, ch, cw), None


class TVLoss(nn.Module):
    """``model.TVLoss`` (model.py:17-33)."""

    def __init__(self, TVLoss_weight=1):
        super().__init__()
        self.TVLoss_weight = TVLoss_weight

    def forward(self, x):
        return _TV.apply(x, self.TVLoss_weight)

    def _tensor_size(self, t):
        return t.size()[1] * t.size()[2] * t.size()[3]


class _PhaseCos(torch.autograd.Function):
    """-cosine_similarity(m * log|Fx|, m * log|Fy|) as a function of the two half spectra (complex64)."""

    EPS = 1e-8      # torch.cosine_similarity's default, model.py:58

    @staticmethod
    def forward(ctx, fx, fy, cols, radius):
        rx, ry = torch.view_as_real(fx), torch.view_as_real(fy)
        sums = torch.ops.b200wave_losses.phase_sums(rx, ry, cols, radius)
        ctx.save_for_backward(rx, ry, sums)
        ctx.geom = (cols, radius)
        norms = sums[1:].sqrt().clamp_min(_PhaseCos.EPS)
        return -sums[0] / (norms[0] * norms[1])

    @staticmethod
    @once_differentiable   # the backward kernels have no autograd formula of their own: double backward raises
    def backward(ctx, g):
        rx, ry, sums = ctx.saved_tensors
        cols, radius = ctx.geom
        gx, gy = torch.ops.b200wave_losses.phase_grad(rx, ry, cols, radius, sums, g, _PhaseCos.EPS)
        return torch.view_as_complex(gx), torch.view_as_complex(gy), None, None


class phase_consistency_loss(nn.Module):
    """``model.phase_consistency_loss`` (model.py:36-58): only the first batch element of ``x`` and ``y`` enters, as in
    the reference (``x[0]``, ``y[0]``); radius 5."""

    def __init__(self):
        super().__init__()

    def forward(self, x, y):
        radius = 5
        for t, name in ((x, "x"), (y, "y")):
            if not t.is_cuda:
                raise RuntimeError("b200wave.phase_consistency_loss is CUDA-only (sm_100a); there is no CPU fallback "
                                   "-- got a %s tensor for %s" % (t.device, name))
            if t.dim() != 4:
                raise IndexError("phase_consistency_loss expects 4-D (N, C, H, W) tensors, got %d-D" % t.dim())
        if x.shape[1:] != y.shape[1:]:
            raise RuntimeError("phase_consistency_loss: x[0] and y[0] must have the same shape")
        fx = torch.fft.rfft2(x[0].float())
        fy = torch.fft.rfft2(y[0].float())
        return _PhaseCos.apply(fx, fy, int(x.shape[-1]), float(radius))
