"""CPU oracle for the undecimated (a trous) 2-D synthesis bank of ``SWTInverse`` -- TEST INFRASTRUCTURE ONLY.

Plain-numpy (float64) restatement of the formula DESIGN.md K12 defines, written directly with modulo indexing (and
deliberately not derived from ``swt_oracle``'s adjoint, so that the two stay independent): with d = dilation and
pl = floor(L d / 2) - d,

    x[r, c] = sum_{a,e} sum_{jh,jw} (gH_e[jh] / 2) (gW_a[jw] / 2) y_{2a+e}[(r - d jh + pl) mod H, (c - d jw + pl) mod W]

where y_0 is the low band of the coarser level and y_1..y_3 are bands 1..3 of this level (channel 4c + 2a + e, a = the
filter along W, e = the one along H), gW = (g0_row, g1_row), gH = (g0_col, g1_col) the synthesis taps, not reversed.
Only tests may import it.
"""
import numpy as np


def _bands(ll, y):
    y = np.asarray(y, dtype=np.float64)
    n, c4, h, w = y.shape
    yb = y.reshape(n, c4 // 4, 4, h, w)
    return [np.asarray(ll, dtype=np.float64), yb[:, :, 1], yb[:, :, 2], yb[:, :, 3]]


def _taps(g0_col, g1_col, g0_row, g1_row):
    f = lambda t: np.asarray(t, dtype=np.float64).ravel()
    return (f(g0_col), f(g1_col)), (f(g0_row), f(g1_row))


def sfb2d_atrous(ll, y, g0_col, g1_col, g0_row, g1_row, dilation=1):
    """One level: ll (N, C, H, W) and y (N, 4C, H, W) -> x (N, C, H, W)."""
    bands = _bands(ll, y)
    gH, gW = _taps(g0_col, g1_col, g0_row, g1_row)
    L, d = gH[0].size, dilation
    pl = (L * d) // 2 - d
    _, _, H, W = bands[0].shape
    r, c = np.arange(H), np.arange(W)
    x = np.zeros_like(bands[0])
    for a in (0, 1):
        for e in (0, 1):
            yb = bands[2 * a + e]
            for jh in range(L):
                rows = yb[:, :, (r - d * jh + pl) % H, :]
                for jw in range(L):
                    x += (0.5 * gH[e][jh]) * (0.5 * gW[a][jw]) * rows[:, :, :, (c - d * jw + pl) % W]
    return x


def sfb2d_atrous_transpose(dx, g0_col, g1_col, g0_row, g1_row, dilation=1):
    """Transpose of ``sfb2d_atrous``: dx (N, C, H, W) -> (d_ll (N, C, H, W), d_y (N, 4C, H, W) with band 0 zero).
    Each term reads a cyclic shift of a band, so its transpose is the opposite shift."""
    dx = np.asarray(dx, dtype=np.float64)
    gH, gW = _taps(g0_col, g1_col, g0_row, g1_row)
    L, d = gH[0].size, dilation
    pl = (L * d) // 2 - d
    n, ch, H, W = dx.shape
    r, c = np.arange(H), np.arange(W)
    g = np.zeros((n, ch, 4, H, W))
    for a in (0, 1):
        for e in (0, 1):
            for jh in range(L):
                rows = dx[:, :, (r + d * jh - pl) % H, :]
                for jw in range(L):
                    g[:, :, 2 * a + e] += (0.5 * gH[e][jh]) * (0.5 * gW[a][jw]) * rows[:, :, :, (c + d * jw - pl) % W]
    d_ll = g[:, :, 0].copy()
    g[:, :, 0] = 0
    return d_ll, g.reshape(n, 4 * ch, H, W)


def iswt(coeffs, g0_col, g1_col, g0_row, g1_row):
    """SWTInverse: coeffs[j] (N, 4C, H, W), finest first, dilation 2**j -> x (N, C, H, W)."""
    y = np.asarray(coeffs[-1], dtype=np.float64)
    n, c4, h, w = y.shape
    ll = y.reshape(n, c4 // 4, 4, h, w)[:, :, 0]
    for j in range(len(coeffs) - 1, -1, -1):
        ll = sfb2d_atrous(ll, coeffs[j], g0_col, g1_col, g0_row, g1_row, 2 ** j)
    return ll


def iswt_transpose(dx, J, g0_col, g1_col, g0_row, g1_row):
    """Gradients of every coeffs[j] of ``iswt`` for the upstream gradient dx."""
    grads = [None] * J
    g = np.asarray(dx, dtype=np.float64)
    for j in range(J):
        g, grads[j] = sfb2d_atrous_transpose(g, g0_col, g1_col, g0_row, g1_row, 2 ** j)
    n, c, h, w = g.shape
    grads[J - 1].reshape(n, c, 4, h, w)[:, :, 0] = g   # the top level's band 0 is the starting ll
    return grads
