"""SWTInverse, the periodic inverse of SWTForward (DESIGN.md K12): the float64 oracle against the identity and against
the adjoint route (CPU), argument validation of the module and of the C entry points, what the compiler makes of the
kernel (CPU), and on the GPU the round trip, parity with the oracle and with the adjoint route, gradients and graph
capture."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import b200wave
from b200wave import _build, _cabi, ops, ops64
from b200wave.dwt import lowlevel
from b200wave.wavelets import as_wavelet
from oracle import iswt_oracle, swt_oracle
from helpers import rel_err

DEV = "cuda"
WAVES = ["haar", "db2", "db3", "db4", "db8", "bior2.4"]
SIZES = [(37, 53), (64, 64), (9, 12)]


def analysis_taps(wave):
    """(h0_col, h1_col, h0_row, h1_row) as SWTForward's buffers hold them: the decomposition taps, reversed."""
    w = as_wavelet(wave)
    lo, hi = np.asarray(w.dec_lo, np.float64)[::-1], np.asarray(w.dec_hi, np.float64)[::-1]
    return lo, hi, lo, hi


def synthesis_taps(wave):
    w = as_wavelet(wave)
    lo, hi = np.asarray(w.rec_lo, np.float64), np.asarray(w.rec_hi, np.float64)
    return lo, hi, lo, hi


def forward_oracle(x, J, h):
    coeffs, ll = [], x
    for j in range(J):
        y = swt_oracle.afb2d_atrous(ll, *h, "periodic", 2 ** j)
        coeffs.append(y)
        n, c4, hh, ww = y.shape
        ll = y.reshape(n, c4 // 4, 4, hh, ww)[:, :, 0]
    return coeffs


def with_band0(ll, y):
    n, c4, h, w = y.shape
    z = np.array(y, dtype=np.float64).reshape(n, c4 // 4, 4, h, w)
    z[:, :, 0] = ll
    return z.reshape(n, c4, h, w)


# ------------------------------------------------------------------------------------------- CPU: oracle
@pytest.mark.parametrize("size", SIZES, ids=["%dx%d" % s for s in SIZES])
@pytest.mark.parametrize("wave", WAVES)
def test_oracle_inverts_the_forward(wave, size):
    x = np.random.default_rng(1).standard_normal((1, 2) + size)
    rec = iswt_oracle.iswt(forward_oracle(x, 3, analysis_taps(wave)), *synthesis_taps(wave))
    assert rel_err(rec, x) <= 1e-12


@pytest.mark.parametrize("size", SIZES, ids=["%dx%d" % s for s in SIZES])
@pytest.mark.parametrize("wave", WAVES)
def test_oracle_matches_the_adjoint_route(wave, size):
    """One level = the adjoint of the analysis level with the halved synthesis taps, applied to (ll, bands 1..3)."""
    rng = np.random.default_rng(2)
    g = synthesis_taps(wave)
    half = [0.5 * t for t in g]
    for d in (1, 2, 4):
        ll = rng.standard_normal((2, 1) + size)
        y = rng.standard_normal((2, 4) + size)
        got = iswt_oracle.sfb2d_atrous(ll, y, *g, d)
        want = swt_oracle.afb2d_atrous_backward(with_band0(ll, y), *half, "periodic", d)
        assert rel_err(got, want) <= 1e-12


def test_oracle_transpose_is_the_transpose():
    rng = np.random.default_rng(3)
    g = synthesis_taps("db3")
    coeffs = [rng.standard_normal((1, 8, 11, 14)) for _ in range(3)]
    dx = rng.standard_normal((1, 2, 11, 14))
    grads = iswt_oracle.iswt_transpose(dx, 3, *g)
    lhs = float((iswt_oracle.iswt(coeffs, *g) * dx).sum())
    top = coeffs[-1].reshape(1, 2, 4, 11, 14)[:, :, 0]
    masked = [with_band0(np.zeros_like(top), c) for c in coeffs[:-1]] + [coeffs[-1]]
    rhs = float(sum((m * gr).sum() for m, gr in zip(masked, grads)))
    assert abs(lhs - rhs) <= 1e-12 * abs(lhs) + 1e-12
    for gr in grads[:-1]:
        assert not gr.reshape(1, 2, 4, 11, 14)[:, :, 0].any()


# ------------------------------------------------------------------------------------------- CPU: host logic
@pytest.mark.parametrize("mode", ["zero", "symmetric", "reflect", "periodization"])
def test_modes_other_than_periodic_raise(mode):
    with pytest.raises(ValueError, match="only periodic extension"):
        b200wave.SWTInverse(wave="db2", mode=mode)
    with pytest.raises(ValueError, match="only periodic extension"):
        lowlevel.sfb2d_atrous(torch.zeros((1, 4, 8, 8)), synthesis_taps("db2"), mode=mode)


def test_exports_and_buffers():
    assert b200wave.SWTInverse is b200wave.dwt.SWTInverse and "SWTInverse" in b200wave.__all__
    m = b200wave.SWTInverse(wave="db3")
    w = as_wavelet("db3")
    assert m.g0_col.shape == (1, 1, 6, 1) and m.g0_row.shape == (1, 1, 1, 6)
    assert np.array_equal(m.g1_row.flatten().numpy(), np.asarray(w.rec_hi, np.float32))
    ref = b200wave.DWTInverse(wave="db3")
    for k in ("g0_col", "g1_col", "g0_row", "g1_row"):
        assert torch.equal(getattr(m, k), getattr(ref, k))


def test_malformed_coeffs_raise():
    inv = b200wave.SWTInverse(wave="db2")
    with pytest.raises(ValueError, match="empty"):
        inv([])
    with pytest.raises(ValueError, match="same shape"):
        inv([torch.zeros((1, 4, 16, 16)), torch.zeros((1, 4, 16, 15))])
    with pytest.raises(ValueError, match="4C"):
        inv([torch.zeros((1, 6, 16, 16))])
    with pytest.raises(ValueError, match="4C"):
        inv([torch.zeros((4, 16, 16))])
    # double mode as in SWTForward: float64 coefficients need float64 buffers and vice versa
    with pytest.raises(RuntimeError, match="expected scalar type Float"):
        inv([torch.zeros((1, 4, 16, 16), dtype=torch.float64)])
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        inv64 = b200wave.SWTInverse(wave="db2")
    finally:
        torch.set_default_dtype(old)
    with pytest.raises(RuntimeError, match="expected scalar type Double"):
        inv64([torch.zeros((1, 4, 16, 16), dtype=torch.float64), torch.zeros((1, 4, 16, 16))])


def test_ops_refuse_cpu_tensors():
    taps = [0.5, 0.5]
    for op, dt in ((ops.iswt2d, torch.float32), (ops64.iswt2d, torch.float64)):
        y = torch.zeros((1, 4, 8, 8), dtype=dt)
        with pytest.raises(RuntimeError, match="CUDA-only"):
            op(y[:, 0::4], y, taps, taps, taps, taps, 1)


BOGUS = ctypes.c_void_p(256)


def test_entry_points_return_the_same_codes_before_any_launch():
    lib = _cabi.load()
    t2 = (_cabi.taps_array([0.5, 0.5])[0], _cabi.taps_array_f64([0.5, 0.5])[0])
    t1 = (_cabi.taps_array([1.0])[0], _cabi.taps_array_f64([1.0])[0])
    t4 = (_cabi.taps_array([0.1] * 4)[0], _cabi.taps_array_f64([0.1] * 4)[0])

    def call(ll=BOGUS, ps=None, y=BOGUS, planes=1, H=8, W=8, taps=t2, L=2, d=1, x=BOGUS):
        return lambda k: (ll, H * W if ps is None else ps, y, planes, H, W, *([taps[k] if taps else None] * 4), L, d,
                          x, None)

    cases = [(call(ll=None), _cabi.ERR_NULL_POINTER), (call(y=None), _cabi.ERR_NULL_POINTER),
             (call(x=None), _cabi.ERR_NULL_POINTER), (call(taps=None), _cabi.ERR_NULL_POINTER),
             (call(L=0), _cabi.ERR_BAD_TAPS), (call(L=_cabi.MAX_TAPS + 1), _cabi.ERR_BAD_TAPS),
             (call(taps=t1, L=1), _cabi.ERR_BAD_TAPS), (call(d=0), _cabi.ERR_BAD_SHAPE),
             (call(H=0), _cabi.ERR_BAD_SHAPE), (call(W=0), _cabi.ERR_BAD_SHAPE), (call(planes=0), _cabi.ERR_BAD_SHAPE),
             (call(H=50000, W=50000), _cabi.ERR_BAD_SHAPE), (call(ps=63), _cabi.ERR_BAD_SHAPE),
             # floor(L d / 2) > 3 min(H, W): db2 at d = 16 needs 11 x 11
             (call(H=10, W=11, taps=t4, L=4, d=16), _cabi.ERR_BAD_SHAPE),
             (call(H=11, W=10, taps=t4, L=4, d=16), _cabi.ERR_BAD_SHAPE)]
    for make, want in cases:
        c32 = lib.b200w_iswt2d_f32(*make(0))
        c64 = lib.b200w_iswt2d_f64(*make(1))
        assert c32 == c64 == want, (make(1), c32, c64, want)


@pytest.mark.skipif(_build.find_nvcc() is None, reason="needs nvcc")
def test_kernel_does_not_spill(tmp_path):
    cmd = [_build.find_nvcc()] + _build.NVCC_FLAGS + ["-Xptxas", "-v", "-I", _build.INCLUDE, "-I", _build.CSRC, "-c",
                                                      os.path.join(_build.CSRC, "swt_inverse.cu"),
                                                      "-o", str(tmp_path / "swt_inverse.o")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    out = res.stdout + res.stderr
    kernels = re.findall(r"Compiling entry function '(\S+)'", out)
    assert sorted(k for k in kernels if "iswt2d_kernel" in k) == sorted(
        ["_ZN5b200w13iswt2d_kernelIfEEvNS_10IswtParamsIT_EE", "_ZN5b200w13iswt2d_kernelIdEEvNS_10IswtParamsIT_EE"])
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", out)
    assert len(spills) == 2 and all(s == ("0", "0") for s in spills), out


# ------------------------------------------------------------------------------------------- GPU
def module_taps(m, names):
    return [getattr(m, k).flatten().cpu().numpy().astype(np.float64) for k in names]


def make_pair(wave, J, dtype):
    old = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        if isinstance(wave, tuple):
            fwd_wave, inv_wave = wave
        else:
            fwd_wave = inv_wave = wave
        return (b200wave.SWTForward(J=J, wave=fwd_wave, mode="periodic").to(DEV),
                b200wave.SWTInverse(wave=inv_wave).to(DEV))
    finally:
        torch.set_default_dtype(old)


def tensor_rel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


def _db2_mixed():
    """Different filters on the two axes: db2 along H, its time-reversed pair (analysis with the synthesis taps and
    back) along W.  Swapping the axes of the inverse does not reconstruct, so this pins the orientation."""
    w = as_wavelet("db2")
    return ((w.dec_lo, w.dec_hi, w.rec_lo, w.rec_hi), (w.rec_lo, w.rec_hi, w.dec_lo, w.dec_hi))


ROUND_TRIPS = [((64, 1, 304, 304), "db3", 3), ((8, 3, 1024, 1024), "db2", 5), ((8, 3, 1024, 1024), "db8", 5),
               ((2, 2, 37, 53), "bior2.4", 3), ((2, 3, 40, 56), "mixed", 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape,wave,J", ROUND_TRIPS, ids=["%s-%s-J%d" % ("x".join(map(str, s)), w, j)
                                                           for s, w, j in ROUND_TRIPS])
def test_round_trip(shape, wave, J, dtype):
    fwd, inv = make_pair(_db2_mixed() if wave == "mixed" else wave, J, dtype)
    gen = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn(shape, device=DEV, dtype=dtype, generator=gen)
    coeffs = fwd(x)
    before = _cabi.kernel_launches()
    rec = inv(coeffs)
    torch.cuda.synchronize()
    # one launch per level, no copies (the top ll is read in place)
    assert _cabi.kernel_launches() - before == J
    assert all(k.startswith("iswt2d_kernel") for k in _cabi.recent_kernels(J))
    assert rec.shape == x.shape and rec.dtype == dtype
    assert tensor_rel(rec, x) <= (1e-5 if dtype == torch.float32 else 1e-12)
    if wave == "mixed":   # the axes swapped do not reconstruct
        a, b = _db2_mixed()
        _, inv_swapped = make_pair((a, (b[2], b[3], b[0], b[1])), J, dtype)
        assert tensor_rel(inv_swapped(coeffs), x) > 1e-2


PARITY = [((2, 3, 37, 53), "db3", (1, 2, 4)), ((1, 2, 11, 11), "db2", (16,)), ((3, 1, 29, 17), "bior2.4", (1, 4)),
          ((2, 1, 64, 300), "db8", (1, 8))]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape,wave,dils", PARITY, ids=["%s-%s" % ("x".join(map(str, s)), w) for s, w, _ in PARITY])
def test_level_matches_oracle(shape, wave, dils, dtype):
    """Random coefficients, one level per dilation; 11 x 11 is the smallest plane the shape rule admits for db2 at
    d = 16 (the taps wrap the plane several times)."""
    rng = np.random.default_rng(7)
    g = synthesis_taps(wave)
    tol = 1e-5 if dtype == torch.float32 else 1e-12
    n, c, h, w = shape
    for d in dils:
        ll = rng.standard_normal((n, c, h, w))
        y = rng.standard_normal((n, 4 * c, h, w))
        got = lowlevel.sfb2d_atrous(torch.tensor(y, device=DEV, dtype=dtype), g, dilation=d,
                                    ll=torch.tensor(ll, device=DEV, dtype=dtype))
        assert rel_err(got.cpu(), iswt_oracle.sfb2d_atrous(ll, y, *g, d)) <= tol
    if (h, w) == (11, 11):   # one row or column less is refused
        y = torch.zeros((1, 4, 10, 11), device=DEV, dtype=dtype)
        with pytest.raises(_cabi.B200WaveError):
            lowlevel.sfb2d_atrous(y, g, dilation=16)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_non_contiguous_inputs(dtype):
    rng = np.random.default_rng(8)
    g = synthesis_taps("db2")
    y_t = torch.tensor(rng.standard_normal((2, 12, 33, 80)), device=DEV, dtype=dtype)[:, :, :, ::5]   # (2, 12, 33, 16)
    ll_t = torch.tensor(rng.standard_normal((2, 3, 16, 33)), device=DEV, dtype=dtype).transpose(2, 3)  # (2, 3, 33, 16)
    assert not y_t.is_contiguous() and not ll_t.is_contiguous()
    for d in (1, 4):
        got = lowlevel.sfb2d_atrous(y_t, g, dilation=d, ll=ll_t)
        want = iswt_oracle.sfb2d_atrous(ll_t.cpu().numpy(), y_t.cpu().numpy(), *g, d)
        assert rel_err(got.cpu(), want) <= (1e-5 if dtype == torch.float32 else 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("wave", ["haar", "db2", "db8"])
def test_kernel_matches_adjoint_route(wave):
    gen = torch.Generator(device=DEV).manual_seed(9)
    g = synthesis_taps(wave)
    half = [[0.5 * float(v) for v in t] for t in g]
    for shape, d in (((4, 1, 304, 304), 1), ((2, 2, 304, 304), 4), ((2, 1, 512, 512), 16)):
        y = torch.randn((shape[0], 4 * shape[1]) + shape[2:], device=DEV, generator=gen)
        ll = torch.randn(shape, device=DEV, generator=gen)
        got = lowlevel.sfb2d_atrous(y, g, dilation=d, ll=ll)
        y0 = y.clone()
        y0.view(shape[0], shape[1], 4, *shape[2:])[:, :, 0] = ll
        want = ops.swt2d_adjoint(y0, half[2], half[3], half[0], half[1], ops.PERIODIC, d)
        assert tensor_rel(got, want) <= 1e-5


@pytest.mark.gpu
def test_gradcheck_double():
    fwd, inv = make_pair("db2", 2, torch.float64)
    x = torch.randn((1, 2, 12, 10), device=DEV, dtype=torch.float64)
    coeffs = [c.detach().requires_grad_(True) for c in fwd(x)]
    assert torch.autograd.gradcheck(lambda a, b: inv([a, b]), tuple(coeffs), eps=1e-6, atol=1e-9)


@pytest.mark.gpu
def test_gradients_match_oracle_transpose():
    rng = np.random.default_rng(10)
    _, inv = make_pair("db2", 3, torch.float32)
    g = synthesis_taps("db2")
    coeffs = [torch.tensor(rng.standard_normal((2, 8, 304, 304)), device=DEV, dtype=torch.float32,
                           requires_grad=True) for _ in range(3)]
    dx = rng.standard_normal((2, 2, 304, 304))
    grads = torch.autograd.grad(inv(coeffs), coeffs, torch.tensor(dx, device=DEV, dtype=torch.float32))
    want = iswt_oracle.iswt_transpose(dx, 3, *g)
    for j in range(3):
        assert rel_err(grads[j].cpu(), want[j]) <= 1e-5
        if j < 2:
            assert not grads[j].view(2, 2, 4, 304, 304)[:, :, 0].any()


@pytest.mark.gpu
def test_graph_capture_matches_eager():
    fwd, inv = make_pair("db3", 3, torch.float32)
    x = torch.randn((2, 3, 128, 96), device=DEV)
    coeffs = [c.clone() for c in fwd(x)]
    eager = inv(coeffs)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        inv(coeffs)   # warm-up: the filter taps are read back once, outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = inv(coeffs)
    for c in coeffs:
        c.mul_(2.0)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, 2.0 * eager) or tensor_rel(out, 2.0 * eager) <= 1e-6
    assert tensor_rel(out, 2.0 * x) <= 1e-5
