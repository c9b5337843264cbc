"""The double-precision frequency split (``freq.gaussian_split`` / ``high_pass`` / ``low_pass``) and the discriminators'
wavelet front end (``fsd.filter_wavelet`` / ``WaveletFilter`` / ``compat.patch_model``), i.e. the reference's double
mode of ``utils.py:71-117`` and ``model.py:166-179, 222-235``.

CPU: argument checks of the new entry points in the order of their fp32 counterparts, the CUDA-only refusal of the new
ops, the dtype dispatch of ``fsd``, and what the compiler makes of ``csrc/freq.cu``.
GPU: against the numpy float64 oracles at 1e-12 relative (max|a-b| / max|b|); the frequency-split oracle with its mask
rounded to fp32 as the reference stores it (``torch.from_numpy(mask).float()``)."""
import ctypes
import types

import numpy as np
import pytest
import torch

import b200wave
from b200wave import _build, _cabi, compat, freq, fsd, ops64
from oracle import freq_oracle, fsd_oracle
from helpers import rel_err
from test_f64_host import _compile, _nvcc_is_12_9

RTOL_F64 = 1e-12
DEV = "cuda"
BOGUS = ctypes.c_void_p(256)


@pytest.fixture(scope="module")
def lib():
    return _cabi.load()


@pytest.fixture
def double_mode():
    """Modules built under torch.set_default_dtype(torch.float64), as the reference's double mode builds them."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        yield
    finally:
        torch.set_default_dtype(old)


def _same_codes(lib, name32, name64, calls):
    """Each call is a function (0 = fp32 arguments, 1 = fp64 arguments) -> args; both must return the same code,
    before any launch (the pointers are bogus)."""
    for make in calls:
        c32 = getattr(lib, name32)(*make(0))
        c64 = getattr(lib, name64)(*make(1))
        assert c32 == c64, (name64, make(1), c32, c64)
        assert c64 not in (_cabi.OK, _cabi.ERR_LAUNCH), (name64, c64)


# ---------------------------------------------------------------------------------------------- CPU: C ABI
def test_afb2d_ex_f64_matches_fp32_checks(lib):
    t = {L: (_cabi.taps_array([0.1] * L)[0], _cabi.taps_array_f64([0.1] * L)[0]) for L in (1, 2, 6)}

    def call(x=BOGUS, planes=1, H=8, W=8, Lw=2, Lh=2, null_tap=False, mode=0, low=BOGUS, highs=BOGUS):
        def make(k):
            tw, th = t.get(Lw, t[2])[k], t.get(Lh, t[2])[k]
            return (x, H * W, W, planes, H, W, tw, None if null_tap else tw, Lw, th, th, Lh, mode, low, highs, 0.5, 0.5,
                    None)
        return make

    calls = [call(mode=3, x=None), call(mode=5, planes=0), call(x=None, planes=0), call(low=None, highs=None),
             call(planes=0, Lw=0), call(W=0), call(Lw=0), call(Lh=_cabi.MAX_TAPS + 1), call(null_tap=True, H=0),
             call(null_tap=True), call(H=1, Lh=1, W=4, Lw=6, mode=4), call(H=1, W=1, Lw=1, Lh=1),
             call(H=4, W=4, Lw=6, Lh=6, mode=4), call(H=16, W=4, Lw=6, Lh=6, mode=4, low=None),
             call(H=4, W=16, Lw=2, Lh=6, mode=2, highs=None), call(H=4, W=4, Lw=6, Lh=6, mode=2)]
    _same_codes(lib, "b200w_afb2d_ex_f32", "b200w_afb2d_ex_f64", calls)
    assert lib.b200w_afb2d_ex_f64(*call(mode=3, x=None)(1)) == _cabi.ERR_BAD_MODE          # the mode first
    assert lib.b200w_afb2d_ex_f64(*call(low=None, highs=None)(1)) == _cabi.ERR_NULL_POINTER
    assert lib.b200w_afb2d_ex_f64(*call(null_tap=True)(1)) == _cabi.ERR_BAD_TAPS           # as fill_taps reports it


def test_freq_entry_points_match_fp32_checks(lib):
    def mask(spec=BOGUS, planes=2, rows=8, cols=8, radius=4.0, hp=1):
        return lambda k: (spec, planes, rows, cols, radius, hp, None)

    calls = [mask(spec=None, planes=0), mask(planes=0), mask(rows=0), mask(cols=-1), mask(radius=0.0),
             mask(radius=-1.0), mask(radius=float("nan")), mask(rows=1 << 20, cols=1 << 14)]
    _same_codes(lib, "b200w_freq_mask_c64", "b200w_freq_mask_c128", calls)

    for name in ("abs_sign", "sign_mul"):
        nptr = 2 if name == "abs_sign" else 3
        for k in range(nptr):
            ptrs = [BOGUS] * nptr
            ptrs[k] = None
            _same_codes(lib, "b200w_%s_f32" % name, "b200w_%s_f64" % name, [lambda _, p=ptrs: (*p, 8, 1.0, None)])
        # n == 0 is a no-op that launches nothing, in both precisions
        assert getattr(lib, "b200w_%s_f64" % name)(*([BOGUS] * nptr), 0, 1.0, None) == _cabi.OK


def test_header_declares_the_new_entry_points():
    from test_cabi_symbols import declared_functions
    new = {"b200w_afb2d_ex_f64", "b200w_freq_mask_c128", "b200w_abs_sign_f64", "b200w_sign_mul_f64"}
    assert new <= set(declared_functions()) and new <= set(_cabi.SYMBOLS)


# ---------------------------------------------------------------------------------------------- CPU: ops
def test_new_ops_refuse_cpu_tensors():
    x = torch.rand((1, 1, 8, 8), dtype=torch.float64)
    spec = torch.fft.rfft2(x).contiguous()
    taps = [0.5, 0.5]
    calls = [(ops64.afb2d_select, (x, taps, taps, taps, taps, 4, True, True, 0.5, 0.5)),
             (ops64.freq_mask_, (spec, 8, 8, 4.0, True)), (ops64.abs_sign, (x, 1.0)), (ops64.sign_mul, (x, x, 1.0))]
    for op, args in calls:
        with pytest.raises(RuntimeError, match="b200wave64::.*CUDA-only"):
            op(*args)


def _filter_ns(fn):
    """Which op namespace a call reaches, read from the CPU refusal of the op."""
    with pytest.raises(RuntimeError, match="CUDA-only") as ei:
        fn()
    return str(ei.value).split("::")[0]


def test_fsd_dtype_dispatch():
    """float64 x + float64 module -> double op; float64 x + float32 module -> the reference's dtype error; float32 x
    -> the fp32 op whatever the module holds; the bare function dispatches on x alone."""
    x64 = torch.rand((1, 1, 8, 8), dtype=torch.float64)
    x32 = x64.float()
    f32 = fsd.WaveletFilter(cs="cat", variant="B")
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        f64 = fsd.WaveletFilter(cs="cat", variant="B")
    finally:
        torch.set_default_dtype(old)
    assert f64.h0_col.dtype == torch.float64 and f32.h0_col.dtype == torch.float32
    assert _filter_ns(lambda: f64(x64)) == "b200wave64"
    assert _filter_ns(lambda: f64(x32)) == "b200wave"
    assert _filter_ns(lambda: f32(x32)) == "b200wave"
    with pytest.raises(RuntimeError, match="expected scalar type Float but found Double"):
        f32(x64)
    assert _filter_ns(lambda: fsd.filter_wavelet(x64, "sum")) == "b200wave64"
    assert _filter_ns(lambda: fsd.filter_wavelet(x32, "sum")) == "b200wave"


def test_fsd_haar_taps_per_dtype():
    """The bare function's default taps are those of a haar DWTForward built under the matching default dtype."""
    old = torch.get_default_dtype()
    try:
        for dt in (torch.float32, torch.float64):
            torch.set_default_dtype(dt)
            xfm = b200wave.DWTForward(J=1, wave="haar", mode="reflect")
            x = torch.zeros(1, dtype=dt)
            taps = fsd.module_taps(x, (xfm.h0_col, xfm.h1_col, xfm.h0_row, xfm.h1_row))
            assert fsd._haar_taps(dt == torch.float64) == taps
    finally:
        torch.set_default_dtype(old)
    assert fsd._haar_taps(True) != fsd._haar_taps(False)


class _Disc(torch.nn.Module):
    """Stand-in for FS_DiscriminatorA/B (model.py:140-142, 190-192): owns DWT2 = DWTForward(J=1, 'haar', 'reflect')."""

    def __init__(self, cs):
        super().__init__()
        self.DWT2 = b200wave.DWTForward(J=1, wave="haar", mode="reflect")
        self.cs = cs

    def filter_wavelet(self, x, norm=True):
        raise AssertionError("not patched")


def _patched():
    return compat.patch_model(types.SimpleNamespace(FS_DiscriminatorA=type("A", (_Disc,), {}),
                                                    FS_DiscriminatorB=type("B", (_Disc,), {})))


def test_patch_model_dtype_dispatch():
    mod = _patched()
    x64 = torch.rand((1, 1, 8, 8), dtype=torch.float64)
    with pytest.raises(RuntimeError, match="expected scalar type Float but found Double"):
        mod.FS_DiscriminatorB("cat").filter_wavelet(x64)
    assert _filter_ns(lambda: mod.FS_DiscriminatorA("sum").filter_wavelet(x64.float())) == "b200wave"
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        d = mod.FS_DiscriminatorB("cat")
    finally:
        torch.set_default_dtype(old)
    assert _filter_ns(lambda: d.filter_wavelet(x64)) == "b200wave64"
    assert _filter_ns(lambda: d.filter_wavelet(x64.float())) == "b200wave"


# ---------------------------------------------------------------------------------------------- CPU: compiler output
# float kernels of csrc/freq.cu: (registers, SASS instructions) of the non-template kernels they replace (nvcc 12.9)
FREQ_FLOAT_KERNELS = {"freq_mask_kernelI6float2fE": (24, 176), "abs_sign_kernelIfE": (21, 80),
                      "sign_mul_kernelIfE": (18, 64)}


@pytest.mark.skipif(_build.find_nvcc() is None, reason="needs nvcc")
def test_freq_kernels_do_not_spill_and_float_code_is_unchanged(tmp_path):
    info, ninstr = _compile("freq.cu", tmp_path)
    assert all(v["spill"] == (0, 0) for v in info.values()), info
    assert [k for k in info if "freq_mask_kernelI7double2dE" in k] and [k for k in info if "abs_sign_kernelIdE" in k]
    if not _nvcc_is_12_9():
        return
    for short, (regs, n) in FREQ_FLOAT_KERNELS.items():
        names = [k for k in info if short in k]
        assert len(names) == 1, (short, list(info))
        assert info[names[0]]["regs"] == regs and ninstr[names[0]] == n, (short, info[names[0]], ninstr[names[0]])


# ---------------------------------------------------------------------------------------------- GPU: frequency split
def dd(a, grad=False):
    return torch.tensor(np.asarray(a, dtype=np.float64), device=DEV, requires_grad=grad)


@pytest.fixture
def fp32_mask_oracle(monkeypatch):
    """freq_oracle with the mask rounded to fp32 after it is built in float64 (1 - m included), as utils.py stores it."""
    exact = freq_oracle.gaussian_mask
    monkeypatch.setattr(freq_oracle, "gaussian_mask",
                        lambda *a: exact(*a).astype(np.float32).astype(np.float64))
    return exact


SPLIT_SHAPES = [(255, 256), (256, 255), (64, 64), (33, 47), (3, 2, 96, 80), (2, 1, 1, 40, 31)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SPLIT_SHAPES, ids=["x".join(map(str, s)) for s in SPLIT_SHAPES])
@pytest.mark.parametrize("radius", [4, 8, 10])
def test_gaussian_split_double_matches_oracle(shape, radius, fp32_mask_oracle):
    rng = np.random.default_rng(radius * 1000 + shape[-1])
    x = rng.random(shape)
    g = rng.standard_normal(shape)
    for hp, sign in ((True, 1.0), (False, -1.0)):
        tx = dd(x, True)
        out = freq.gaussian_split(tx, radius, hp, sign)
        assert out.dtype == torch.float64 and out.shape == tx.shape
        want = freq_oracle.split(x, radius, hp, sign)
        assert rel_err(out.detach().cpu(), want) < RTOL_F64
        out.backward(dd(g))
        assert rel_err(tx.grad.cpu(), freq_oracle.split_backward(x, g, radius, hp, sign)) < RTOL_F64


@pytest.mark.gpu
def test_gaussian_split_double_pins_the_fp32_mask(monkeypatch):
    """Without the fp32 rounding of the mask the result would miss the tolerance: the check above pins the rounding."""
    x = np.random.default_rng(3).random((2, 128, 96))
    for hp, sign, r in ((True, 1.0, 10), (False, -1.0, 8)):
        out = freq.gaussian_split(dd(x), r, hp, sign).cpu()
        assert rel_err(out, freq_oracle.split(x, r, hp, sign)) > 100 * RTOL_F64
        exact = freq_oracle.gaussian_mask
        with monkeypatch.context() as m:
            m.setattr(freq_oracle, "gaussian_mask", lambda *a: exact(*a).astype(np.float32).astype(np.float64))
            assert rel_err(out, freq_oracle.split(x, r, hp, sign)) < RTOL_F64


@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(255, 256), (256, 255), (76, 76)])
def test_high_low_pass_double(hw, fp32_mask_oracle):
    x = np.random.default_rng(hw[0]).random((1,) + hw)
    for fn, ofn, i in ((freq.high_pass, freq_oracle.high_pass, 10), (freq.low_pass, freq_oracle.low_pass, 8)):
        out = fn(dd(x), i=i)
        assert out.dtype == torch.float64 and tuple(out.shape) == hw and out.is_contiguous()
        assert rel_err(out.cpu(), ofn(x, i)) < RTOL_F64


@pytest.mark.gpu
def test_gaussian_split_other_dtypes_still_raise():
    x = torch.rand((1, 8, 8), device=DEV)
    for bad in (x.half(), x.bfloat16(), x.to(torch.complex64), x.double().to(torch.complex128)):
        with pytest.raises(RuntimeError, match="expected scalar type Float"):
            freq.gaussian_split(bad, 4, True)


@pytest.mark.gpu
def test_double_pointwise_kernels_on_misaligned_and_odd_tensors():
    """abs_sign / sign_mul in double take the double2 loop on 16-byte aligned tensors and the scalar loop on the odd
    last element or a misaligned view; every path gives the elementwise result exactly."""
    y = torch.rand(1001, device=DEV, dtype=torch.float64) - 0.5
    y[7] = 0.0
    for off, n in ((0, 1000), (0, 999), (1, 999), (1, 1000)):
        v = y[off:off + n]
        assert torch.equal(ops64.abs_sign(v, -1.0), -v.abs())
        gg = torch.rand_like(v)
        assert torch.equal(ops64.sign_mul(gg, v, -1.0), -gg * torch.sign(v))
        assert torch.equal(ops64.sign_mul(gg, v, 1.0), gg * torch.sign(v))


# ---------------------------------------------------------------------------------------------- GPU: filter_wavelet
FSD_SHAPES = [(2, 1, 64, 64), (3, 1, 33, 47), (2, 3, 30, 22), (1, 1, 256, 256), (4, 1, 2, 2)]


def _unfused(ll, hi, cs, norm, variant):
    h = hi * 0.5 + 0.5 if norm else hi
    if cs == "sum":
        return (ll,) if variant == "A" else (h[:, :, 2],)
    if cs == "each":
        return ll, h[:, :, 0], h[:, :, 1], h[:, :, 2]
    return (torch.cat((h[:, :, 0], h[:, :, 1], h[:, :, 2]), 1),)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", FSD_SHAPES, ids=["x".join(map(str, s)) for s in FSD_SHAPES])
def test_filter_wavelet_double_matches_oracle_and_unfused_route(shape, double_mode):
    rng = np.random.default_rng(shape[-1] + shape[1])
    xn = rng.standard_normal(shape)
    xfm = b200wave.DWTForward(J=1, wave="haar", mode="reflect").to(DEV)
    x = dd(xn)
    ll, (hi,) = xfm(x)
    for variant in "AB":
        for cs in ("sum", "each", "cat"):
            filt = fsd.WaveletFilter(cs=cs, variant=variant).to(DEV)
            assert filt.h0_col.dtype == torch.float64
            for norm in (True, False):
                tx = dd(xn, True)
                res = filt(tx, norm)
                assert res[-1] is tx
                got = res[:-1]
                want = _unfused(ll, hi, cs, norm, variant)
                assert len(got) == len(want)
                for a, b in zip(got, want):
                    assert a.dtype == torch.float64 and torch.equal(a, b), (variant, cs, norm)
                for a, b in zip(got, fsd.filter_wavelet(x, cs, norm, variant)[:-1]):   # bare function, double haar
                    assert torch.equal(a, b)
                ora = fsd_oracle.filter_wavelet(xn, cs, norm, variant)
                for a, b in zip(got, ora):
                    assert rel_err(a.detach().cpu(), b) < RTOL_F64
                gs = [rng.standard_normal(tuple(a.shape)) for a in got]
                (dx,) = torch.autograd.grad(list(got), tx, [dd(v) for v in gs])
                want_dx = fsd_oracle.filter_wavelet_backward(gs, shape, cs, norm, variant)
                assert dx.dtype == torch.float64 and rel_err(dx.cpu(), want_dx) < RTOL_F64


@pytest.mark.gpu
def test_filter_wavelet_double_other_filters_and_views(double_mode):
    """Longer filters and other modes, and strided inputs, through the same double epilogue."""
    rng = np.random.default_rng(5)
    for wave, mode, shape in [("db2", "symmetric", (2, 1, 96, 70)), ("db4", "zero", (1, 2, 31, 77)),
                              ("db3", "periodization", (2, 1, 64, 100)), ("db8", "periodic", (1, 1, 40, 36))]:
        x = dd(rng.standard_normal(shape))
        for xs in (x, x[..., 1:]):
            ll, (hi,) = b200wave.DWTForward(J=1, wave=wave, mode=mode).to(DEV)(xs)
            got = fsd.WaveletFilter(cs="each", wave=wave, mode=mode).to(DEV)(xs)
            assert torch.equal(got[0], ll)
            for b in range(3):
                assert torch.equal(got[1 + b], hi[:, :, b] * 0.5 + 0.5)
            cat = fsd.WaveletFilter(cs="cat", variant="B", wave=wave, mode=mode).to(DEV)(xs, False)[0]
            assert torch.equal(cat, torch.cat((hi[:, :, 0], hi[:, :, 1], hi[:, :, 2]), 1))
    with pytest.raises(ValueError):
        ops64.afb2d_select(x, [1.0, 1.0], [1.0, -1.0], [1.0, 1.0], [1.0, -1.0], 4, False, False, 1.0, 0.0)
    with pytest.raises(RuntimeError, match="expected scalar type Float"):   # float16 keeps raising as before
        fsd.filter_wavelet(x.half(), "sum")


@pytest.mark.gpu
def test_patch_model_double_mode():
    mod = _patched()
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        a, b = mod.FS_DiscriminatorA("sum").to(DEV), mod.FS_DiscriminatorB("cat").to(DEV)
    finally:
        torch.set_default_dtype(old)
    xn = np.random.default_rng(1).standard_normal((2, 1, 64, 64))
    for disc, variant, cs in ((a, "A", "sum"), (b, "B", "cat")):
        for norm in (True, False):
            got, x = disc.filter_wavelet(dd(xn), norm)
            assert got.dtype == torch.float64
            assert rel_err(got.cpu(), fsd_oracle.filter_wavelet(xn, cs, norm, variant)[0]) < RTOL_F64


@pytest.mark.gpu
def test_filter_wavelet_fp32_unchanged():
    """float32 inputs keep the fp32 path: bit-identical to the fp32 unfused route, whether the module holds float32 or
    float64 buffers."""
    xn = np.random.default_rng(2).standard_normal((3, 1, 64, 96)).astype(np.float32)
    x = torch.tensor(xn, device=DEV)
    ll, (hi,) = b200wave.DWTForward(J=1, wave="haar", mode="reflect").to(DEV)(x)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        f64 = {(cs, v): fsd.WaveletFilter(cs=cs, variant=v).to(DEV) for cs in ("sum", "each", "cat") for v in "AB"}
    finally:
        torch.set_default_dtype(old)
    for (cs, variant), filt64 in f64.items():
        filt32 = fsd.WaveletFilter(cs=cs, variant=variant).to(DEV)
        for norm in (True, False):
            want = _unfused(ll, hi, cs, norm, variant)
            for got in (filt32(x, norm)[:-1], filt64(x, norm)[:-1], fsd.filter_wavelet(x, cs, norm, variant)[:-1]):
                assert len(got) == len(want)
                for a, b in zip(got, want):
                    assert a.dtype == torch.float32 and torch.equal(a, b), (variant, cs, norm)
