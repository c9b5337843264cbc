"""GPU: the double-precision paths of SSIM, the 1-D DWT, SWTForward and TVLoss (the reference's double mode) against
the float64 goldens of the unmodified reference and the float64 oracle, at 1e-12 relative (max|a-b| / max|b|)."""
import os
import sys

import numpy as np
import pytest
import torch

import b200wave
from b200wave.dwt import lowlevel
from b200wave.losses import TVLoss
from oracle import dwt_oracle, ssim_oracle, swt_oracle
from helpers import load_dwt1d_cases, load_ssim_cases, load_swt_cases, load_tv_cases, rel_err

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "pywt_standin"))

DEV = "cuda"
RTOL_F64 = 1e-12
SSIM_CASES = load_ssim_cases()
DWT1D_CASES = load_dwt1d_cases()
SWT_CASES = load_swt_cases()
TV_CASES = load_tv_cases()


def dd(a, grad=False):
    return torch.tensor(np.asarray(a, dtype=np.float64), device=DEV, requires_grad=grad)


@pytest.fixture
def double_mode():
    """Modules built under torch.set_default_dtype(torch.float64), as the reference's double tests do."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        yield
    finally:
        torch.set_default_dtype(old)


# ------------------------------------------------------------------------------------------- SSIM
@pytest.mark.parametrize("via", ["module", "function"])
@pytest.mark.parametrize("case", SSIM_CASES, ids=[c["id"] for c in SSIM_CASES])
def test_golden_ssim_double(case, via):
    """Double images, window built under the float32 default (the goldens' setting): value, d1 and d2."""
    sa = bool(case["size_average"])
    fn = b200wave.SSIM(window_size=11, size_average=sa) if via == "module" else \
        (lambda x, y: b200wave.ssim(x, y, window_size=11, size_average=sa))
    a, b = dd(case["img1"], True), dd(case["img2"], True)
    val = fn(a, b)
    assert val.dtype == torch.float64
    assert rel_err(np.atleast_1d(val.detach().cpu().numpy()), np.atleast_1d(case["val"])) < RTOL_F64
    val.backward(dd(case["gout"]) if not sa else None)
    if np.abs(case["d1"]).max() > 1e-12:
        assert rel_err(a.grad.cpu(), case["d1"]) < RTOL_F64
        assert rel_err(b.grad.cpu(), case["d2"]) < RTOL_F64
    else:   # ssim(x, x): the gradient vanishes up to double rounding of O(1/NCHW) terms
        assert a.grad.abs().max().item() < 1e-12
    # only img2 needs a gradient: the forward swaps the arguments and stores 3 maps
    a2, b2 = dd(case["img1"]), dd(case["img2"], True)
    val2 = fn(a2, b2)
    assert torch.equal(val2.detach(), val.detach())
    val2.backward(dd(case["gout"]) if not sa else None)
    assert a2.grad is None
    if np.abs(case["d2"]).max() > 1e-12:
        assert rel_err(b2.grad.cpu(), case["d2"]) < RTOL_F64


@pytest.mark.parametrize("ws", [1, 3, 5, 7, 9, 11])
def test_ssim_double_default_window_vs_oracle(ws, double_mode, monkeypatch):
    """Under the float64 default the window is the fp32 rounding of a float64 outer product: the kernel applies the
    module's taps.  The oracle is given that same window."""
    rng = np.random.default_rng(ws)
    shape = (3, 2, 37, 53)
    x = rng.random(shape)
    y = np.clip(x + 0.1 * rng.standard_normal(shape), 0, 1)
    mod = b200wave.SSIM(window_size=ws, size_average=False)
    a, b = dd(x, True), dd(y, True)
    val = mod(a, b)
    win = mod.window[0, 0].cpu().numpy()
    assert mod.window.dtype == torch.float64
    monkeypatch.setattr(ssim_oracle, "window2d", lambda window_size=11: win)
    assert rel_err(val.detach().cpu(), ssim_oracle.ssim(x, y, ws, False)) < RTOL_F64
    gout = np.linspace(0.5, 1.5, 3)
    val.backward(dd(gout))
    o1, o2 = ssim_oracle.ssim_backward(x, y, gout, ws, False)
    assert rel_err(a.grad.cpu(), o1) < RTOL_F64 and rel_err(b.grad.cpu(), o2) < RTOL_F64
    v = b200wave.ssim(dd(x), dd(y), window_size=ws)   # ssim() builds the same window per call
    assert rel_err(np.atleast_1d(v.cpu().numpy()), np.atleast_1d(ssim_oracle.ssim(x, y, ws, True))) < RTOL_F64


def test_ssim_double_full_size_cfg3():
    """cfg3 (256 x 1 x 400 x 400) in double: identity, symmetry, per-sample means, finite difference, agreement with
    the fp32 kernel, bit-reproducibility, and CUDA-graph replay of forward + backward."""
    g = torch.Generator(device=DEV).manual_seed(0)
    x = torch.rand((256, 1, 400, 400), generator=g, device=DEV, dtype=torch.float64)
    y = (x + 0.1 * torch.randn(x.shape, generator=g, device=DEV, dtype=torch.float64)).clamp_(0, 1)
    with torch.no_grad():
        assert abs(b200wave.ssim(x, x).item() - 1.0) < 1e-15
        s_xy, s_yx = b200wave.ssim(x, y), b200wave.ssim(y, x)
        assert abs(s_xy.item() - s_yx.item()) < 1e-14
        per = b200wave.ssim(x, y, size_average=False)
        assert per.shape == (256,) and abs(per.mean().item() - s_xy.item()) < 1e-14
        s32 = b200wave.ssim(x.float(), y.float())
        assert abs(s32.item() - s_xy.item()) < 1e-5
        assert torch.equal(b200wave.ssim(x, y), s_xy)
    xg = x.clone().requires_grad_(True)
    b200wave.ssim(xg, y).backward()
    # random magnitudes, signs of the gradient: along a direction with random signs the derivative of the mean is only
    # O(1e-5) here, and the double rounding of the two values (~1e-16 / (2 eps) = 5e-12) would swamp a 1e-7 comparison
    d = torch.randn(x.shape, generator=g, device=DEV, dtype=torch.float64).abs_() * xg.grad.sign()
    eps = 1e-5
    with torch.no_grad():
        fd = (b200wave.ssim(x + eps * d, y) - b200wave.ssim(x - eps * d, y)) / (2 * eps)
    an = (xg.grad * d).sum()
    assert abs(fd.item() - an.item()) <= 1e-7 * abs(an.item())
    g1 = xg.grad.clone()
    xg.grad = None
    b200wave.ssim(xg, y).backward()
    assert torch.equal(xg.grad, g1)

    # graph capture of forward + backward (small shape: the graph holds its own buffers)
    xs, ys = x[:8].clone(), y[:8].clone()
    xs.requires_grad_(True)

    def step():
        xs.grad = None
        v = b200wave.ssim(xs, ys)
        v.backward()
        return v.detach(), xs.grad.clone()

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            ve, ge = step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    xs.grad = None
    with torch.cuda.graph(graph):
        v = b200wave.ssim(xs, ys)
        v.backward()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(v.detach(), ve) and torch.equal(xs.grad, ge)


def test_mixed_dtypes_raise(double_mode):
    x64 = torch.rand((1, 1, 32, 32), device=DEV, dtype=torch.float64)
    x32 = x64.float()
    for a, b in ((x32, x64), (x64, x32)):
        with pytest.raises(RuntimeError, match="expected scalar type"):
            b200wave.SSIM()(a, b)
        with pytest.raises(RuntimeError, match="expected scalar type"):
            b200wave.ssim(a, b)
    f64_1d, f64_swt = b200wave.DWT1DForward(wave="db2").to(DEV), b200wave.SWTForward(wave="db2", mode="zero").to(DEV)
    torch.set_default_dtype(torch.float32)
    f32_1d, f32_swt = b200wave.DWT1DForward(wave="db2").to(DEV), b200wave.SWTForward(wave="db2", mode="zero").to(DEV)
    i32_1d = b200wave.DWT1DInverse(wave="db2").to(DEV)
    for fwd, t in ((f64_1d, x32[0]), (f32_1d, x64[0]), (f64_swt, x32), (f32_swt, x64)):
        with pytest.raises(RuntimeError, match="expected scalar type"):
            fwd(t)
    with pytest.raises(RuntimeError, match="expected scalar type"):
        i32_1d((x64[0][..., :17], [x64[0][..., :17]]))


# ------------------------------------------------------------------------------------------- 1-D DWT
@pytest.mark.parametrize("case", DWT1D_CASES, ids=[c["id"] for c in DWT1D_CASES])
def test_golden_dwt1d_double(case, double_mode):
    J, mode = case["J"], case["mode"]
    xfm = b200wave.DWT1DForward(J=J, wave=(case["h0"][::-1].copy(), case["h1"][::-1].copy()), mode=mode).to(DEV)
    ifm = b200wave.DWT1DInverse(wave=(case["g0"], case["g1"]), mode=mode).to(DEV)
    assert xfm.h0.dtype == torch.float64
    x = dd(case["x"], True)
    yl, yh = xfm(x)
    assert yl.dtype == torch.float64 and rel_err(yl.detach().cpu(), case["yl"]) < RTOL_F64
    for j in range(J):
        assert rel_err(yh[j].detach().cpu(), case["yh%d" % j]) < RTOL_F64
    (dx,) = torch.autograd.grad([yl] + list(yh), x, [dd(case["gl"])] + [dd(case["gh%d" % j]) for j in range(J)])
    assert rel_err(dx.cpu(), case["dx"]) < RTOL_F64
    cl = dd(case["yl"], True)
    ch = [dd(case["yh%d" % j], True) for j in range(J)]
    rec = ifm((cl, ch))
    assert rec.dtype == torch.float64 and rel_err(rec.detach().cpu(), case["rec"]) < RTOL_F64
    grads = torch.autograd.grad(rec, [cl] + ch, dd(case["gy"]))
    assert rel_err(grads[0].cpu(), case["dcl"]) < RTOL_F64
    for j in range(J):
        assert rel_err(grads[1 + j].cpu(), case["dch%d" % j]) < RTOL_F64


@pytest.mark.parametrize("wave", ["haar", "db4", "db8"])
@pytest.mark.parametrize("mode", ["zero", "symmetric", "reflect", "periodic", "periodization"])
def test_oracle_dwt1d_long_signals_double(wave, mode, double_mode):
    rng = np.random.default_rng(len(wave) * 7 + len(mode))
    xn = rng.standard_normal((3, 2, 100003))
    xfm = b200wave.DWT1DForward(J=3, wave=wave, mode=mode).to(DEV)
    ifm = b200wave.DWT1DInverse(wave=wave, mode=mode).to(DEV)
    h0, h1 = xfm.h0.flatten().cpu().numpy(), xfm.h1.flatten().cpu().numpy()
    yl, yh = xfm(dd(xn))
    lo = xn
    for j in range(3):
        lo, hi = dwt_oracle.afb1d(lo, h0, h1, mode)
        assert rel_err(yh[j].cpu(), hi) < RTOL_F64
    assert rel_err(yl.cpu(), lo) < RTOL_F64
    rec = ifm((yl, yh))
    assert rel_err(rec[..., :xn.shape[-1]].cpu(), xn) < 1e-11      # perfect reconstruction up to the wavelet's taps
    xs = dd(np.ascontiguousarray(np.repeat(xn, 2, axis=-1)))[..., ::2]
    yl2, _ = xfm(xs)
    assert torch.equal(yl2, yl)


# ------------------------------------------------------------------------------------------- SWT
@pytest.mark.parametrize("case", SWT_CASES, ids=[c["id"] for c in SWT_CASES])
def test_golden_swt_level_double(case):
    filts = tuple(dd(case[k]) for k in ("h0_col", "h1_col", "h0_row", "h1_row"))
    x = dd(case["x"], True)
    y = lowlevel.afb2d_atrous(x, filts, case["mode"], case["dilation"])
    assert y.dtype == torch.float64 and rel_err(y.detach().cpu(), case["y"]) < RTOL_F64
    (dx,) = torch.autograd.grad(y, x, dd(case["gy"]))
    assert rel_err(dx.cpu(), case["dx"]) < RTOL_F64


@pytest.mark.parametrize("mode", ["zero", "symmetric", "reflect", "periodic"])
def test_oracle_swt_forward_module_double(mode, double_mode):
    rng = np.random.default_rng(31)
    xn = rng.standard_normal((2, 2, 304, 304))
    xfm = b200wave.SWTForward(J=3, wave="db2", mode=mode).to(DEV)
    fl = [getattr(xfm, k).flatten().cpu().numpy() for k in ("h0_col", "h1_col", "h0_row", "h1_row")]
    x = dd(xn, True)
    coeffs = xfm(x)
    ll = xn
    for j in range(3):
        y = swt_oracle.afb2d_atrous(ll, *fl, mode, 2 ** j)
        assert coeffs[j].dtype == torch.float64 and rel_err(coeffs[j].detach().cpu(), y) < RTOL_F64
        ll = y.reshape(2, 2, 4, 304, 304)[:, :, 0]
    g = [rng.standard_normal(c.shape) for c in coeffs]
    (dx,) = torch.autograd.grad(coeffs, x, [dd(t) for t in g])
    d = np.zeros((2, 2, 304, 304))
    for j in range(2, -1, -1):
        gj = g[j].reshape(2, 2, 4, 304, 304).copy()
        gj[:, :, 0] += d
        d = swt_oracle.afb2d_atrous_backward(gj.reshape(2, 8, 304, 304), *fl, mode, 2 ** j)
    assert rel_err(dx.cpu(), d) < RTOL_F64


# ------------------------------------------------------------------------------------------- TV
@pytest.mark.parametrize("case", TV_CASES, ids=[c["id"] for c in TV_CASES])
def test_golden_tv_loss_double(case):
    x = dd(case["x"], True)
    loss = TVLoss(case["weight"])(x)
    assert loss.dtype == torch.float64 and loss.dim() == 0
    assert abs(loss.item() - case["loss"]) <= RTOL_F64 * abs(case["loss"])
    loss.backward()
    assert x.grad.dtype == torch.float64 and rel_err(x.grad.cpu(), case["dx"]) < RTOL_F64
