"""CPU oracle for MS-SSIM -- TEST INFRASTRUCTURE ONLY.

Plain-numpy float64 restatement of ``b200wave.ms_ssim`` (the reference has no MS-SSIM) on top of
``ssim_oracle.ssim_terms`` / ``blur_same``: scales ``x(j+1) = avg_pool2d(x(j), 2)`` (floor), the per-sample mean of
the contrast-structure map ``A2 / B2`` at every scale but the last, of the SSIM map at the last, and
``MS = prod_j relu(v_j) ** w_j``.  The backward is the closed form: the derivative maps of cs or S, blurred back to
each scale's images, and the transpose of the pooling (each coarse gradient spread as 0.25 over its 2x2 block).
"""
import numpy as np

from . import ssim_oracle
from .ssim_oracle import blur_same

WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def pool2(x):
    """F.avg_pool2d(x, 2): an odd last row or column is dropped."""
    h, w = x.shape[-2] // 2 * 2, x.shape[-1] // 2 * 2
    return 0.25 * (x[..., 0:h:2, 0:w:2] + x[..., 0:h:2, 1:w:2] + x[..., 1:h:2, 0:w:2] + x[..., 1:h:2, 1:w:2])


def pool2_transpose(g, shape):
    out = np.zeros(shape, dtype=g.dtype)
    h, w = g.shape[-2] * 2, g.shape[-1] * 2
    for dy in (0, 1):
        for dx in (0, 1):
            out[..., dy:h:2, dx:w:2] += 0.25 * g
    return out


def _scales(img1, img2, M):
    xs = [(img1, img2)]
    for _ in range(M - 1):
        xs.append((pool2(xs[-1][0]), pool2(xs[-1][1])))
    return xs


def _scale_maps(x1, x2, last, window_size):
    """Per-pixel value map of one scale and its derivatives w.r.t. mu1, mu2, E[x1^2] (= E[x2^2]) and E[x1 x2]."""
    w, mu1, mu2, A1, A2, B1, B2 = ssim_oracle.ssim_terms(x1, x2, window_size)
    if last:
        v = (A1 * A2) / (B1 * B2)
        d_mu1 = 2 * mu2 * (A2 - A1) / (B1 * B2) - 2 * mu1 * v * (1 / B1 - 1 / B2)
        d_mu2 = 2 * mu1 * (A2 - A1) / (B1 * B2) - 2 * mu2 * v * (1 / B1 - 1 / B2)
        d_e = -v / B2
        d_e12 = 2 * A1 / (B1 * B2)
    else:
        v = A2 / B2
        d_mu1 = 2 * (mu1 * v - mu2) / B2
        d_mu2 = 2 * (mu2 * v - mu1) / B2
        d_e = -v / B2
        d_e12 = 2 / B2
    return w, v, (d_mu1, d_mu2, d_e, d_e12)


def scale_values(img1, img2, M, window_size=11):
    """(M, N): per-sample mean of cs at scales 0..M-2 and of the SSIM map at scale M-1."""
    xs = _scales(img1, img2, M)
    return np.stack([_scale_maps(a, b, j == M - 1, window_size)[1].mean(axis=(1, 2, 3)) for j, (a, b) in enumerate(xs)])


def ms_ssim(img1, img2, window_size=11, size_average=True, weights=WEIGHTS):
    v = scale_values(img1, img2, len(weights), window_size)
    ms = np.prod([np.maximum(v[j], 0) ** w for j, w in enumerate(weights)], axis=0)
    return ms.mean() if size_average else ms


def ms_ssim_backward(img1, img2, grad_out=1.0, window_size=11, size_average=True, weights=WEIGHTS):
    """Gradients (d/dimg1, d/dimg2) of ``ms_ssim`` times ``grad_out`` (scalar, or shape (N,) without size_average)."""
    M = len(weights)
    N = img1.shape[0]
    xs = _scales(img1, img2, M)
    v = scale_values(img1, img2, M, window_size)
    f = np.stack([np.maximum(v[j], 0) ** w for j, w in enumerate(weights)])
    go = np.full(N, float(grad_out) / N) if size_average else np.asarray(grad_out, dtype=np.float64).reshape(N)
    acc1 = acc2 = None
    for j in range(M - 1, -1, -1):
        x1, x2 = xs[j]
        others = np.prod([f[k] for k in range(M) if k != j], axis=0) if M > 1 else np.ones(N)
        pos = v[j] > 0
        dv = np.where(pos, weights[j] * np.where(pos, v[j], 1.0) ** (weights[j] - 1), 0.0) * others * go
        w, _, (d_mu1, d_mu2, d_e, d_e12) = _scale_maps(x1, x2, j == M - 1, window_size)
        g = (dv / np.prod(x1.shape[1:])).reshape(N, 1, 1, 1)
        # the window is symmetric and the blur zero padded => self-adjoint
        d1 = blur_same(g * d_mu1, w) + 2 * x1 * blur_same(g * d_e, w) + x2 * blur_same(g * d_e12, w)
        d2 = blur_same(g * d_mu2, w) + 2 * x2 * blur_same(g * d_e, w) + x1 * blur_same(g * d_e12, w)
        if acc1 is not None:
            d1 = d1 + pool2_transpose(acc1, x1.shape)
            d2 = d2 + pool2_transpose(acc2, x2.shape)
        acc1, acc2 = d1, d2
    return acc1, acc2
