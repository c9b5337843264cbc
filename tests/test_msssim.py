"""MS-SSIM (DESIGN.md K13): the float64 oracle against an independent torch restatement and against the SSIM oracle
(CPU), argument checks of the functional, the module and the C entry points (CPU), and on the GPU parity with the
oracle, the one-scale case against b200wave.ssim, identities, float64, gradcheck and graph capture."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import b200wave
from b200wave import _cabi, compat, ops, ops64
from b200wave.ssim import _win2d_taps, _win_taps, create_window
from oracle import msssim_oracle, ssim_oracle
from helpers import RTOL_F32, rel_err

DEV = "cuda"
W5 = msssim_oracle.WEIGHTS
# float32 gradients with more than one scale: the coarse scales' pooled images vary little around their mean, so the
# moment differences E[x^2] - mu^2 cancel more digits there, and their per-pixel gradient weight is 4^j larger.
# Measured against the float64 kernels on a B200: 1e-6 at M = 1 (plain SSIM), 3e-6 at M = 2, 0.9-1.3e-5 at M = 5
# (8x1x256^2 to 256x1x400^2).  Values stay within RTOL_F32.
GRAD_RTOL_MS = 3e-5


def torch_ms_ssim(x, y, weights, size_average=True, ws=11):
    """Independent restatement in torch float64: dense F.conv2d with the window of ssim.py, avg_pool2d, autograd."""
    win = create_window(ws, x.shape[1]).double()
    vals = []
    for j in range(len(weights)):
        if j:
            x, y = F.avg_pool2d(x, 2), F.avg_pool2d(y, 2)
        conv = lambda t: F.conv2d(t, win, padding=ws // 2, groups=x.shape[1])
        mu1, mu2 = conv(x), conv(y)
        s11, s22, s12 = conv(x * x) - mu1 * mu1, conv(y * y) - mu2 * mu2, conv(x * y) - mu1 * mu2
        cs = (2 * s12 + 0.03 ** 2) / (s11 + s22 + 0.03 ** 2)
        if j == len(weights) - 1:
            cs = (2 * mu1 * mu2 + 0.01 ** 2) / (mu1 * mu1 + mu2 * mu2 + 0.01 ** 2) * cs
        vals.append(cs.mean(dim=(1, 2, 3)))
    ms = 1.0
    for v, w in zip(vals, weights):
        ms = ms * torch.relu(v) ** w
    return ms.mean() if size_average else ms


def pair(shape, seed, noise=0.1):
    rng = np.random.default_rng(seed)
    x = rng.random(shape)
    y = np.clip(x + noise * rng.standard_normal(shape), 0, 1)
    return x, y


# ------------------------------------------------------------------------------------------- CPU: oracle
@pytest.mark.parametrize("shape,weights", [((2, 1, 32, 40), W5), ((2, 3, 37, 53), W5[:3]), ((1, 2, 16, 16), W5),
                                           ((3, 1, 24, 20), (0.5, 0.0, 1.5))])
@pytest.mark.parametrize("size_average", [True, False])
def test_oracle_matches_torch_restatement(shape, weights, size_average):
    x, y = pair(shape, 1)
    tx, ty = torch.tensor(x, requires_grad=True), torch.tensor(y, requires_grad=True)
    want = torch_ms_ssim(tx, ty, weights, size_average)
    gout = np.linspace(0.5, 1.5, shape[0]) if not size_average else 1.0
    want.backward(torch.tensor(gout) if not size_average else None)
    got = msssim_oracle.ms_ssim(x, y, 11, size_average, weights)
    assert rel_err(np.atleast_1d(got), np.atleast_1d(want.detach().numpy())) <= 1e-12
    d1, d2 = msssim_oracle.ms_ssim_backward(x, y, gout, 11, size_average, weights)
    assert rel_err(d1, tx.grad.numpy()) <= 1e-12
    assert rel_err(d2, ty.grad.numpy()) <= 1e-12


def test_oracle_one_scale_is_ssim():
    x, y = pair((3, 2, 29, 33), 2)
    for sa in (True, False):
        assert rel_err(np.atleast_1d(msssim_oracle.ms_ssim(x, y, 11, sa, (1.0,))),
                       np.atleast_1d(ssim_oracle.ssim(x, y, 11, sa))) <= 1e-12
        gout = 1.0 if sa else np.array([0.3, 1.0, 2.0])
        for a, b in zip(msssim_oracle.ms_ssim_backward(x, y, gout, 11, sa, (1.0,)),
                        ssim_oracle.ssim_backward(x, y, gout, 11, sa)):
            assert rel_err(a, b) <= 1e-12


# ------------------------------------------------------------------------------------------- CPU: host checks
def test_exports_and_compat_namespace():
    assert b200wave.ms_ssim is b200wave.msssim.ms_ssim and b200wave.MS_SSIM is b200wave.msssim.MS_SSIM
    assert "ms_ssim" in b200wave.__all__ and "MS_SSIM" in b200wave.__all__
    ssim_mod = b200wave.SSIM.__module__
    import sys
    assert not hasattr(sys.modules[ssim_mod], "ms_ssim") and not hasattr(sys.modules[ssim_mod], "MS_SSIM")
    assert callable(compat.install)


@pytest.mark.parametrize("weights", [[], (0.5, -0.1), (0.5, float("nan")), (1.0, float("inf")), ("a",), 3, (True,)])
def test_bad_weights_raise(weights):
    x = torch.zeros((1, 1, 64, 64))
    with pytest.raises(ValueError, match="weights"):
        b200wave.ms_ssim(x, x, weights=weights)
    with pytest.raises(ValueError, match="weights"):
        b200wave.MS_SSIM(weights=weights)


@pytest.mark.parametrize("ws", [0, 2, 13, 4.0])
def test_bad_window_raises(ws):
    x = torch.zeros((1, 1, 64, 64))
    with pytest.raises(ValueError, match="odd window sizes"):
        b200wave.ms_ssim(x, x, window_size=ws)
    with pytest.raises(ValueError, match="odd window sizes"):
        b200wave.MS_SSIM(window_size=ws)


def test_too_small_and_mismatched_images_raise():
    with pytest.raises(ValueError, match="at least 16 x 16"):
        b200wave.ms_ssim(torch.zeros((1, 1, 15, 64)), torch.zeros((1, 1, 15, 64)))
    with pytest.raises(ValueError, match="at least 4 x 4"):
        b200wave.MS_SSIM(weights=(1, 1, 1))(torch.zeros((1, 1, 64, 3)), torch.zeros((1, 1, 64, 3)))
    with pytest.raises(RuntimeError, match="equal shape"):
        b200wave.ms_ssim(torch.zeros((1, 1, 32, 32)), torch.zeros((1, 1, 32, 33)))
    with pytest.raises(RuntimeError, match="equal shape"):
        b200wave.ms_ssim(torch.zeros((1, 32, 32)), torch.zeros((1, 32, 32)))


def test_cpu_tensors_are_refused():
    for dt in (torch.float32, torch.float64):
        x = torch.rand((1, 1, 32, 32), dtype=dt)
        with pytest.raises(RuntimeError, match="CUDA-only"):
            b200wave.ms_ssim(x, x)
        with pytest.raises(RuntimeError, match="CUDA-only"):
            b200wave.ms_ssim(x, x, weights=(1.0,))
    x4 = torch.rand((1, 1, 8, 8), dtype=torch.float64)
    for op, x in ((ops.msssim_scale, x4.float()), (ops64.msssim_scale, x4)):
        with pytest.raises(RuntimeError, match="CUDA-only"):
            op(x, x, [1.0], True, True, 0)


BOGUS = ctypes.c_void_p(256)


def test_entry_points_return_status_codes_before_any_launch():
    lib = _cabi.load()
    w1d = {ws: _cabi.taps_array([1.0 / ws] * ws)[0] for ws in (4, 11, 13)}
    w2d = {ws: _cabi.taps_array_f64([1.0 / ws ** 2] * ws * ws)[0] for ws in (4, 11, 13)}

    def fwd(i1=BOGUS, i2=BOGUS, N=2, C=3, H=40, W=70, ws=11, win=True, cs=1, n_maps=0, maps=BOGUS, out=BOGUS,
            p1=BOGUS, p2=BOGUS, work=BOGUS, nbytes=None):
        def make(k):
            w = (w1d if k == 0 else w2d)[ws] if win else None
            nb = nbytes if nbytes is not None else (lib.b200w_ssim_workspace_bytes(N, C, H, W) if k == 0
                                                    else lib.b200w_ssim_workspace_bytes_f64(N, C, H, W))
            return (i1, i2, N, C, H, W, w, ws, cs, n_maps, maps, out, p1, p2, work, nb, None)
        return make

    E = _cabi
    cases = [(fwd(i1=None, N=0), E.ERR_NULL_POINTER), (fwd(out=None, ws=4), E.ERR_NULL_POINTER),
             (fwd(N=0, ws=4), E.ERR_BAD_SHAPE), (fwd(W=0), E.ERR_BAD_SHAPE), (fwd(n_maps=2, ws=4), E.ERR_BAD_SHAPE),
             (fwd(n_maps=3, maps=None, ws=4), E.ERR_NULL_POINTER), (fwd(p2=None, ws=4), E.ERR_NULL_POINTER),
             (fwd(p1=None, H=1), E.ERR_NULL_POINTER), (fwd(H=1, ws=4), E.ERR_BAD_SHAPE),
             (fwd(W=1, ws=4), E.ERR_BAD_SHAPE), (fwd(ws=4), E.ERR_BAD_WINDOW), (fwd(ws=13), E.ERR_BAD_WINDOW),
             (fwd(win=False), E.ERR_BAD_WINDOW), (fwd(work=None), E.ERR_WORKSPACE), (fwd(nbytes=8), E.ERR_WORKSPACE),
             (fwd(nbytes=8, p1=None, p2=None, H=1, cs=0), E.ERR_WORKSPACE)]
    for make, want in cases:
        c32 = lib.b200w_msssim_scale_fwd_f32(*make(0))
        c64 = lib.b200w_msssim_scale_fwd_f64(*make(1))
        assert c32 == c64 == want, (make(1), c32, c64, want)

    def bwd(i1=BOGUS, i2=BOGUS, maps=BOGUS, n_maps=3, g=BOGUS, N=2, C=3, H=40, W=70, ws=11, win=True, up1=BOGUS,
            up2=None, d1=BOGUS, d2=None):
        def make(k):
            w = (w1d if k == 0 else w2d)[ws] if win else None
            return (i1, i2, maps, n_maps, g, N, C, H, W, w, ws, up1, up2, d1, d2, None)
        return make

    cases = [(bwd(maps=None, ws=4), E.ERR_NULL_POINTER), (bwd(g=None, N=0), E.ERR_NULL_POINTER),
             (bwd(d1=None), E.ERR_NULL_POINTER), (bwd(N=0, ws=4), E.ERR_BAD_SHAPE),
             (bwd(n_maps=2, ws=4), E.ERR_BAD_SHAPE), (bwd(n_maps=3, d2=BOGUS, ws=4), E.ERR_BAD_SHAPE),
             (bwd(up2=BOGUS, ws=4), E.ERR_BAD_SHAPE), (bwd(H=1, ws=4), E.ERR_BAD_SHAPE),
             (bwd(up1=None, up2=BOGUS, n_maps=4, d2=BOGUS, W=1, ws=4), E.ERR_BAD_SHAPE),
             (bwd(ws=4), E.ERR_BAD_WINDOW), (bwd(ws=13), E.ERR_BAD_WINDOW), (bwd(win=False), E.ERR_BAD_WINDOW)]
    for make, want in cases:
        c32 = lib.b200w_msssim_scale_bwd_f32(*make(0))
        c64 = lib.b200w_msssim_scale_bwd_f64(*make(1))
        assert c32 == c64 == want, (make(1), c32, c64, want)


# ------------------------------------------------------------------------------------------- GPU
SHAPES = [((8, 1, 256, 256), 5), ((2, 3, 37, 53), 3), ((1, 1, 16, 16), 5), ((256, 1, 400, 400), 5)]
SHAPE_IDS = ["%s-M%d" % ("x".join(map(str, s)), m) for s, m in SHAPES]


def _grads(x, y, need, dtype, size_average, weights, gout):
    tx = torch.tensor(x, device=DEV, dtype=dtype, requires_grad=need in ("1", "both"))
    ty = torch.tensor(y, device=DEV, dtype=dtype, requires_grad=need in ("2", "both"))
    val = b200wave.ms_ssim(tx, ty, size_average=size_average, weights=weights)
    val.backward(None if size_average else torch.tensor(gout, device=DEV, dtype=dtype))
    return val.detach().cpu().numpy(), tx.grad, ty.grad


@pytest.mark.gpu
@pytest.mark.parametrize("shape,M", SHAPES, ids=SHAPE_IDS)
def test_parity_with_oracle(shape, M):
    """Samples are independent, so at the cfg3 shape the oracle (numpy, dense window) runs on the first K samples
    only: their per-sample values, and their gradients (the mean's gradient is 1/N of each sample's)."""
    x, y = pair(shape, 3)
    N = shape[0]
    K = N if N * shape[2] * shape[3] <= 8 * 256 * 256 else 2
    weights = W5[:M]
    gtol = RTOL_F32 if M == 1 else GRAD_RTOL_MS
    for sa in (True, False):
        gout = np.full(N, 1.0 / N) if sa else np.linspace(0.5, 1.5, N)
        want = msssim_oracle.ms_ssim(x[:K], y[:K], 11, False, weights)
        o1, o2 = msssim_oracle.ms_ssim_backward(x[:K], y[:K], gout[:K], 11, False, weights)
        for need in ("1", "2", "both"):
            val, g1, g2 = _grads(x.astype(np.float32), y.astype(np.float32), need, torch.float32, sa, weights,
                                 None if sa else gout)
            if sa and K == N:
                assert rel_err(np.atleast_1d(val), np.atleast_1d(want.mean())) <= RTOL_F32, need
            elif not sa:
                assert rel_err(val[:K], want) <= RTOL_F32, need
            if need in ("1", "both"):
                assert rel_err(g1[:K].cpu(), o1) <= gtol, need
            if need in ("2", "both"):
                assert rel_err(g2[:K].cpu(), o2) <= gtol, need
            assert (g1 is None) == (need == "2") and (g2 is None) == (need == "1")
    if K < N:   # the mean over all samples is the mean of the per-sample values
        a = torch.tensor(x, device=DEV, dtype=torch.float32)
        b = torch.tensor(y, device=DEV, dtype=torch.float32)
        per = b200wave.ms_ssim(a, b, size_average=False, weights=weights)
        assert abs(b200wave.ms_ssim(a, b, weights=weights).item() - per.double().mean().item()) <= 1e-6
        assert rel_err(per[:K].cpu(), want) <= RTOL_F32


@pytest.mark.gpu
def test_pooled_outputs_are_avg_pool2d():
    for dt, op in ((torch.float32, ops.msssim_scale), (torch.float64, ops64.msssim_scale)):
        win = _win_taps(11) if dt == torch.float32 else _win2d_taps(11)
        for shape in ((2, 3, 37, 53), (1, 1, 130, 67), (3, 1, 64, 64)):
            a = torch.rand(shape, device=DEV, dtype=dt)
            b = torch.rand(shape, device=DEV, dtype=dt)
            _, _, p1, p2 = op(a, b, win, True, True, 0)
            assert torch.equal(p1, F.avg_pool2d(a, 2)) and torch.equal(p2, F.avg_pool2d(b, 2))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_one_scale_is_ssim(dtype):
    x, y = pair((4, 3, 61, 75), 4)
    a, b = torch.tensor(x, device=DEV, dtype=dtype), torch.tensor(y, device=DEV, dtype=dtype)
    per = b200wave.ms_ssim(a, b, size_average=False, weights=(1.0,))
    assert torch.equal(per, b200wave.ssim(a, b, size_average=False))
    assert abs(b200wave.ms_ssim(a, b, weights=(1.0,)).item() - b200wave.ssim(a, b).item()) <= 1e-6
    ag = a.clone().requires_grad_(True)
    bg = b.clone().requires_grad_(True)
    ag2 = a.clone().requires_grad_(True)
    bg2 = b.clone().requires_grad_(True)
    b200wave.ms_ssim(ag, bg, weights=(1.0,), size_average=False).sum().backward()
    b200wave.ssim(ag2, bg2, size_average=False).sum().backward()
    assert torch.equal(ag.grad, ag2.grad) and torch.equal(bg.grad, bg2.grad)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,M", [((8, 1, 256, 256), 5), ((2, 3, 37, 53), 3), ((1, 1, 16, 16), 5)])
def test_identity_is_exactly_one(shape, M):
    x = torch.rand(shape, device=DEV)
    assert b200wave.ms_ssim(x, x, weights=W5[:M]).item() == 1.0
    assert torch.equal(b200wave.ms_ssim(x, x, weights=W5[:M], size_average=False), torch.ones(shape[0], device=DEV))
    v = b200wave.ms_ssim(x.double(), x.double(), weights=W5[:M], size_average=False)
    assert (v - 1).abs().max().item() <= 2.0 ** -52


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_inverted_image_gives_zero_with_zero_finite_gradient(dtype):
    x = torch.rand((2, 1, 64, 64), device=DEV, dtype=dtype)
    a = x.clone().requires_grad_(True)
    b = (1 - x).requires_grad_(True)
    val = b200wave.ms_ssim(a, b)
    val.backward()
    assert val.item() == 0.0
    for g in (a.grad, b.grad):
        assert torch.isfinite(g).all() and not g.any()


@pytest.mark.gpu
@pytest.mark.parametrize("shape,M", SHAPES[:3], ids=SHAPE_IDS[:3])
def test_double_matches_oracle(shape, M):
    x, y = pair(shape, 5)
    weights = W5[:M]
    for sa in (True, False):
        gout = 1.0 if sa else np.linspace(0.5, 1.5, shape[0])
        val, g1, g2 = _grads(x, y, "both", torch.float64, sa, weights, gout)
        assert rel_err(np.atleast_1d(val), np.atleast_1d(msssim_oracle.ms_ssim(x, y, 11, sa, weights))) <= 1e-12
        o1, o2 = msssim_oracle.ms_ssim_backward(x, y, gout, 11, sa, weights)
        assert rel_err(g1.cpu(), o1) <= 1e-12 and rel_err(g2.cpu(), o2) <= 1e-12


@pytest.mark.gpu
def test_gradcheck_double():
    x, y = pair((2, 1, 12, 10), 6, noise=0.3)
    a = torch.tensor(x, device=DEV, requires_grad=True)
    b = torch.tensor(y, device=DEV, requires_grad=True)
    assert torch.autograd.gradcheck(lambda p, q: b200wave.ms_ssim(p, q, size_average=False, weights=(0.3, 0.7)),
                                    (a, b), eps=1e-6, atol=1e-8)


@pytest.mark.gpu
def test_graph_replay_matches_eager():
    x, y = pair((4, 2, 96, 80), 7)
    a = torch.tensor(x, device=DEV, dtype=torch.float32, requires_grad=True)
    b = torch.tensor(y, device=DEV, dtype=torch.float32)
    crit = b200wave.MS_SSIM(weights=W5[:4])

    def step():
        return torch.autograd.grad(crit(a, b), a)[0]

    eager = step()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
    with torch.no_grad():
        b.copy_(torch.tensor(pair((4, 2, 96, 80), 8)[1], device=DEV))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, step())


@pytest.mark.gpu
def test_mixed_dtypes_and_cpu_raise():
    a = torch.rand((1, 1, 32, 32), device=DEV)
    with pytest.raises(RuntimeError, match="expected scalar type"):
        b200wave.ms_ssim(a, a.double())
    with pytest.raises(RuntimeError, match="expected scalar type"):
        b200wave.ms_ssim(a.double(), a)
    with pytest.raises(RuntimeError):
        b200wave.ms_ssim(a, a.cpu())
