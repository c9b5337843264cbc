"""Multi-scale SSIM (Wang, Simoncelli and Bovik, 2003) built from this package's Gaussian-window SSIM.

``ms_ssim(img1, img2, window_size=11, size_average=True, weights=None)`` and the module
``MS_SSIM(window_size=11, size_average=True, weights=None)``.  The reference has no MS-SSIM; the semantics are
defined here so that one scale *is* ``b200wave.ssim``:

* scales ``x(0) = img``, ``x(j+1) = F.avg_pool2d(x(j), 2)`` (floor pooling: an odd last row or column is dropped);
* at every scale the terms of ``ssim.py:17-37`` as ``b200wave.ssim`` computes them: the same window (float32: the
  11-tap Gaussian applied separably; float64: the dense window ``ssim()`` builds), zero-padded "same" blur,
  ``C1 = 0.01**2``, ``C2 = 0.03**2``;
* for the scales ``j < M - 1`` the per-sample mean of the contrast-structure map ``cs = A2 / B2``, for the last scale
  the per-sample mean of the SSIM map;
* ``MS[n] = prod_j relu(v_j[n]) ** w_j``, ``MS.mean()`` when ``size_average`` else ``MS`` of shape (N,).

``weights`` defaults to Wang et al.'s five, so ``M = len(weights)``.  A sample clamped to 0 gets a zero gradient.

Each scale is one op (``ops.msssim_scale`` / ``ops64.msssim_scale``): the SSIM forward kernel with a cs epilogue and
the 2x2 pooling of both images written from inside it, so the next scale's input costs no extra pass.  Its backward
is one launch of the SSIM backward kernel that also adds the pooling's transpose of the coarser scale's gradient.
The combination of the (M, N) values runs in torch and never touches full-size tensors.
"""
import math
import numbers

import torch

from . import ops, ops64
from .ssim import _check_window, _win2d_taps, _win_taps

WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def _check_weights(weights):
    if weights is None:
        return WEIGHTS
    try:
        w = tuple(weights)
    except TypeError:
        raise ValueError("MS-SSIM weights must be a sequence of numbers, got %r" % (weights,)) from None
    if not w or any(isinstance(v, bool) or not isinstance(v, numbers.Real) or not math.isfinite(v) or v < 0
                    for v in w):
        raise ValueError("MS-SSIM weights must be a non-empty sequence of finite, non-negative numbers, got %r"
                         % (weights,))
    return tuple(float(v) for v in w)


def ms_ssim(img1, img2, window_size=11, size_average=True, weights=None):
    _check_window(window_size)
    w = _check_weights(weights)
    if img1.dim() != 4 or img1.shape != img2.shape:
        raise RuntimeError("ms_ssim expects two (N, C, H, W) tensors of equal shape, got %s and %s"
                           % (tuple(img1.shape), tuple(img2.shape)))
    M = len(w)
    H, W = img1.shape[-2:]
    if min(H, W) < 2 ** (M - 1):
        raise ValueError("ms_ssim with %d scales needs images of at least %d x %d pixels, got %d x %d"
                         % (M, 2 ** (M - 1), 2 ** (M - 1), H, W))
    if img1.dtype == torch.float64:
        scale, ssim_fwd, win = ops64.msssim_scale, ops64.ssim_fwd, _win2d_taps(window_size)
    else:
        scale, ssim_fwd, win = ops.msssim_scale, ops.ssim_fwd, _win_taps(window_size)
    grad = torch.is_grad_enabled()
    need1 = grad and img1.requires_grad
    need2 = grad and img2.requires_grad
    a, b = img1, img2
    if need2 and not need1:
        # cs and SSIM are symmetric in their arguments: the tensor that needs the gradient goes first at every scale,
        # so each forward stores 3 derivative maps instead of 4
        a, b = img2, img1
    n_maps = 4 if (need1 and need2) else (3 if (need1 or need2) else 0)
    vals = []
    for _ in range(M - 1):
        v, _, a, b = scale(a, b, win, True, True, n_maps)
        if n_maps != 4:   # the second image needs no gradient: keep its pooled copy out of the graph
            b = b.detach()
        vals.append(v)
    if M == 1:   # one scale is b200wave.ssim, bit for bit
        vals.append(ssim_fwd(a, b, win, False, n_maps)[0])
    else:
        vals.append(scale(a, b, win, False, False, n_maps)[0])
    ms = None
    for v, wj in zip(vals, w):
        # relu(v) ** wj with a zero gradient where v <= 0 (not 0 * inf)
        pos = v > 0
        t = torch.where(pos, torch.where(pos, v, torch.ones_like(v)) ** wj, 0.0 if wj > 0 else 1.0)
        ms = t if ms is None else ms * t
    return ms.mean() if size_average else ms


class MS_SSIM(torch.nn.Module):
    def __init__(self, window_size=11, size_average=True, weights=None):
        super(MS_SSIM, self).__init__()
        _check_window(window_size)
        self.window_size = window_size
        self.size_average = size_average
        self.weights = _check_weights(weights)

    def forward(self, img1, img2):
        return ms_ssim(img1, img2, self.window_size, self.size_average, self.weights)
