"""Gaussian-window SSIM -- drop-in for the reference's ``ssim.py``.

``SSIM(window_size=11, size_average=True)(img1, img2)`` and
``ssim(img1, img2, window_size=11, size_average=True)`` keep the reference's
signatures (``ssim.py:39-73``); ``gaussian`` / ``create_window`` build the same
fp32 window (``ssim.py:7-15``).  The five blurs, the SSIM map, its reduction
and the backward run in two fused sm_100a kernels (``csrc/ssim.cu``).

Double images run through the fp64 kernels (``csrc/ssim_f64.cu``), which apply
the dense 2-D window the reference applies in double: built in the default
dtype current when it is (re)built, rounded with ``.float()``, cast to the
images' dtype (``ssim.py:7-15, 50-73``).
"""
from math import exp

import torch

from . import ops, ops64
from .dwt.lowlevel import host_taps


def gaussian(window_size, sigma):
    """Normalised 1-D Gaussian as an fp32 tensor, computed like ssim.py:7-9."""
    gauss = torch.tensor([exp(-(x - window_size // 2) ** 2 / float(2 * sigma ** 2)) for x in range(window_size)],
                         dtype=torch.float32)
    return gauss / gauss.sum()


def create_window(window_size, channel):
    """(channel, 1, ws, ws) window = outer product of the 1-D Gaussian (ssim.py:11-15)."""
    w1 = gaussian(window_size, 1.5).unsqueeze(1)
    w2 = w1.mm(w1.t()).float().unsqueeze(0).unsqueeze(0)
    return w2.expand(channel, 1, window_size, window_size).contiguous()


_win_cache = {}


def _check_window(window_size):
    """The fused kernel holds an odd window of at most 11 taps (the reference's default and only use, train.py:97).
    The reference itself accepts any size (an even one yields an (H+1) x (W+1) map); anything else is refused here,
    loudly and before any device work."""
    if not isinstance(window_size, int) or window_size < 1 or window_size > 11 or window_size % 2 == 0:
        raise ValueError("b200wave.SSIM / ssim support odd window sizes 1..11 (got %r): the fused sm_100a kernel is "
                         "built for the reference's 11-tap Gaussian window and smaller odd ones" % (window_size,))


def _win_taps(window_size):
    _check_window(window_size)
    taps = _win_cache.get(window_size)
    if taps is None:
        taps = tuple(float(v) for v in gaussian(window_size, 1.5).tolist())
        _win_cache[window_size] = taps
    return taps


def _reference_window(window_size, channel):
    """The window as ssim.py:7-15 builds it: 1-D Gaussian and outer product in the CURRENT default dtype (the
    reference's ``torch.Tensor([...])``), rounded with ``.float()``.  Under a float64 default it is not the outer
    product of an fp32 Gaussian, and not separable."""
    dt = torch.get_default_dtype()
    gauss = torch.tensor([exp(-(x - window_size // 2) ** 2 / float(2 * 1.5 ** 2)) for x in range(window_size)],
                         dtype=dt)
    w1 = (gauss / gauss.sum()).unsqueeze(1)
    w2 = w1.mm(w1.t()).float().unsqueeze(0).unsqueeze(0)
    return w2.expand(channel, 1, window_size, window_size).contiguous()


_win2d_cache = {}


def _win2d_taps(window_size):
    """ssim() rebuilds the window on every call (ssim.py:65-73): the same taps, cached by the default dtype."""
    _check_window(window_size)
    key = (window_size, torch.get_default_dtype())
    taps = _win2d_cache.get(key)
    if taps is None:
        taps = tuple(float(v) for v in _reference_window(window_size, 1).double().reshape(-1).tolist())
        _win2d_cache[key] = taps
    return taps


def _ssim(img1, img2, window, window_size, channel, size_average=True):
    """ssim.py:17-37.  For fp32 images ``window`` is accepted for signature compatibility; the kernel applies the
    separable form of the same Gaussian (the 2-D window is its outer product).  For double images the kernel applies
    ``window`` tap by tap (``None``: the window ``ssim()`` builds)."""
    if img1.dim() != 4 or img1.shape != img2.shape:
        raise RuntimeError("ssim expects two (N, C, H, W) tensors of equal shape, got %s and %s"
                           % (tuple(img1.shape), tuple(img2.shape)))
    if img1.dtype == torch.float64:
        fwd = ops64.ssim_fwd
        ws2 = window_size * window_size
        win = _win2d_taps(window_size) if window is None else host_taps(window)[:ws2]
    else:
        fwd = ops.ssim_fwd
        win = _win_taps(window_size)
    grad = torch.is_grad_enabled()
    need1 = grad and img1.requires_grad
    need2 = grad and img2.requires_grad
    if need2 and not need1:
        # SSIM is symmetric in its arguments: put the tensor that needs the gradient first so the
        # forward stores 3 derivative maps instead of 4
        val, _ = fwd(img2, img1, win, bool(size_average), 3)
        return val
    n_maps = 4 if need2 else (3 if need1 else 0)
    val, _ = fwd(img1, img2, win, bool(size_average), n_maps)
    return val


class SSIM(torch.nn.Module):
    def __init__(self, window_size=11, size_average=True):
        super(SSIM, self).__init__()
        _check_window(window_size)
        self.window_size = window_size
        self.size_average = size_average
        self.channel = 1
        self.window = create_window(window_size, self.channel)

    def forward(self, img1, img2):
        channel = img1.size(1)
        if channel != self.channel or self.window.dtype != img1.dtype or self.window.device != img1.device:
            # kept as a plain attribute, lazily re-created like ssim.py:50-60; in double the kernel applies these taps
            build = _reference_window if img1.dtype == torch.float64 else create_window
            self.window = build(self.window_size, channel).to(device=img1.device, dtype=img1.dtype)
            self.channel = channel
        return _ssim(img1, img2, self.window, self.window_size, channel, self.size_average)


def ssim(img1, img2, window_size=11, size_average=True):
    return _ssim(img1, img2, None, window_size, img1.size(1), size_average)
