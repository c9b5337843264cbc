"""CPU: the double-precision entry points of SSIM, the 1-D DWT, SWT and TV -- argument validation in the order of
their fp32 counterparts, the SSIM window the double path applies, the CUDA-only refusal of the new ops, and what the
compiler makes of the kernels (no spills; the float instantiations of the templated kernels unchanged)."""
import ctypes
import os
import re
import subprocess
import sys
from math import exp

import pytest
import torch

import b200wave
from b200wave import _build, _cabi, ops64

ssim_mod = sys.modules[b200wave.SSIM.__module__]   # the module; the package exports the function ssim


@pytest.fixture(scope="module")
def lib():
    return _cabi.load()


BOGUS = ctypes.c_void_p(256)


def _pair(values):
    return _cabi.taps_array(values)[0], _cabi.taps_array_f64(values)[0]


def _same_codes(lib, name32, name64, calls):
    """Each call is a function (taps32_or_64 selector) -> args; both entry points must return the same code."""
    for make in calls:
        c32 = getattr(lib, name32)(*make(0))
        c64 = getattr(lib, name64)(*make(1))
        assert c32 == c64, (name64, make(1), c32, c64)
        # every call must be refused before a launch: the pointers are bogus, and on a GPU a launch would fault
        assert c64 not in (_cabi.OK, _cabi.ERR_LAUNCH), (name64, c64)


def test_1d_entry_points_match_fp32_checks(lib):
    t2, t6 = _pair([0.5, 0.5]), _pair([0.1] * 6)

    def afb(x=BOGUS, rows=1, n=16, taps=t2, L=2, mode=0, lo=BOGUS, hi=BOGUS):
        return lambda k: (x, n, rows, n, taps[k] if taps else None, taps[k] if taps else None, L, mode, lo, hi, None)

    calls = [afb(x=None, mode=3), afb(lo=None), afb(hi=None), afb(taps=None, L=0), afb(mode=3, rows=0), afb(mode=5),
             afb(rows=0, L=0), afb(n=0), afb(L=0), afb(L=_cabi.MAX_TAPS + 1), afb(n=4, taps=t6, L=6, mode=2),
             afb(n=2, taps=t6, L=6, mode=4)]
    _same_codes(lib, "b200w_afb1d_f32", "b200w_afb1d_f64", calls)

    def sfb(lo=BOGUS, rows=1, m=8, taps=t2, L=2, mode=0, out_len=16, y=BOGUS):
        return lambda k: (lo, m, None, rows, m, taps[k] if taps else None, taps[k] if taps else None, L, mode, out_len,
                          y, None)

    calls = [sfb(lo=None, mode=3), sfb(y=None), sfb(taps=None), sfb(mode=3, rows=0), sfb(rows=0, L=0), sfb(m=0),
             sfb(out_len=0), sfb(L=0), sfb(L=99), sfb(m=2, taps=t6, L=6, mode=2, out_len=4), sfb(out_len=17),
             sfb(out_len=17, mode=2)]
    _same_codes(lib, "b200w_sfb1d_f32", "b200w_sfb1d_f64", calls)


def test_swt_entry_points_match_fp32_checks(lib):
    t2, t1, t6 = _pair([0.5, 0.5]), _pair([1.0]), _pair([0.1] * 6)
    for which in ("fwd", "bwd"):
        def call(x=BOGUS, planes=1, H=8, W=8, taps=t2, L=2, d=1, mode=0, y=BOGUS):
            return lambda k: (x, planes, H, W, *([taps[k] if taps else None] * 4), L, d, mode, y, None)

        calls = [call(x=None, mode=2), call(y=None), call(taps=None, mode=2), call(mode=2, planes=0), call(planes=0),
                 call(d=0), call(H=50000, W=50000), call(L=0), call(L=_cabi.MAX_TAPS + 1), call(taps=t1, L=1),
                 call(H=3, W=3, taps=t6, L=6, mode=4), call(H=2, W=2, taps=t6, L=6, d=4)]
        _same_codes(lib, "b200w_swt2d_%s_f32" % which, "b200w_swt2d_%s_f64" % which, calls)


def test_tv_entry_points_match_fp32_checks(lib):
    assert lib.b200w_tv_workspace_bytes_f64(3, 40) == 2 * lib.b200w_tv_workspace_bytes(3, 40) > 0
    assert lib.b200w_tv_workspace_bytes_f64(0, 40) == 0
    need = lib.b200w_tv_workspace_bytes_f64(3, 40)

    def fwd(x=BOGUS, planes=3, H=40, W=8, ws=BOGUS, nbytes=need, out=BOGUS):
        return lambda k: (x, planes, H, W, ws, nbytes, out, None)

    calls = [fwd(x=None, planes=0), fwd(out=None), fwd(ws=None, planes=0), fwd(planes=0, nbytes=0), fwd(W=0),
             fwd(planes=1 << 30, H=1 << 10), fwd(nbytes=lib.b200w_tv_workspace_bytes(3, 40))]
    _same_codes(lib, "b200w_tv_fwd_f32", "b200w_tv_fwd_f64", calls[:-1])
    # float partials do not fit double ones: the fp32 size is too small for the double entry point
    assert lib.b200w_tv_fwd_f64(*calls[-1](1)) == _cabi.ERR_WORKSPACE

    def bwd(x=BOGUS, g=BOGUS, planes=3, H=40, W=8, dx=BOGUS):
        return lambda k: (x, g, 1.0, 1.0, planes, H, W, dx, None)

    calls = [bwd(x=None, planes=0), bwd(g=None), bwd(dx=None), bwd(planes=0), bwd(H=0),
             bwd(planes=1 << 30, H=1 << 10)]
    _same_codes(lib, "b200w_tv_bwd_f32", "b200w_tv_bwd_f64", calls)


def test_ssim_entry_points_match_fp32_checks(lib):
    """Same codes and order as b200w_ssim_fwd_f32 / _bwd_f32; the fp64 ones take the dense ws x ws window."""
    w1d = {ws: _cabi.taps_array([1.0 / ws] * ws)[0] for ws in (1, 4, 11, 13)}
    w2d = {ws: _cabi.taps_array_f64([1.0 / ws ** 2] * ws * ws)[0] for ws in (1, 4, 11, 13)}
    need = lib.b200w_ssim_workspace_bytes_f64(2, 3, 40, 70)
    assert need > 0 and lib.b200w_ssim_workspace_bytes_f64(0, 3, 40, 70) == 0

    def fwd(i1=BOGUS, i2=BOGUS, N=2, C=3, H=40, W=70, ws=11, win=True, n_maps=0, maps=BOGUS, out=BOGUS, work=BOGUS,
            nbytes=None):
        def make(k):
            w = (w1d if k == 0 else w2d)[ws] if win else None
            nb = nbytes if nbytes is not None else (lib.b200w_ssim_workspace_bytes(N, C, H, W) if k == 0 else need)
            return (i1, i2, N, C, H, W, w, ws, 1, n_maps, maps, out, work, nb, None)
        return make

    calls = [fwd(i1=None, N=0), fwd(out=None, ws=4), fwd(N=0, ws=4), fwd(W=0), fwd(n_maps=2, ws=4),
             fwd(n_maps=3, maps=None, ws=4), fwd(ws=4), fwd(ws=13), fwd(win=False), fwd(work=None), fwd(nbytes=8)]
    _same_codes(lib, "b200w_ssim_fwd_f32", "b200w_ssim_fwd_f64", calls)
    assert lib.b200w_ssim_fwd_f64(*fwd(ws=4)(1)) == _cabi.ERR_BAD_WINDOW
    assert lib.b200w_ssim_fwd_f64(*fwd(nbytes=need - 1)(1)) == _cabi.ERR_WORKSPACE

    def bwd(i1=BOGUS, i2=BOGUS, maps=BOGUS, n_maps=3, g=BOGUS, N=2, C=3, H=40, W=70, ws=11, win=True, d1=BOGUS,
            d2=None):
        def make(k):
            w = (w1d if k == 0 else w2d)[ws] if win else None
            return (i1, i2, maps, n_maps, g, N, C, H, W, w, ws, 1, d1, d2, None)
        return make

    calls = [bwd(maps=None, ws=4), bwd(g=None, N=0), bwd(d1=None), bwd(N=0, ws=4), bwd(n_maps=2, ws=4),
             bwd(n_maps=3, d2=BOGUS, ws=4), bwd(ws=4), bwd(ws=13), bwd(win=False)]
    _same_codes(lib, "b200w_ssim_bwd_f32", "b200w_ssim_bwd_f64", calls)


def _restated_window(ws):
    """ssim.py:7-15 as written (torch.Tensor follows the default dtype), then .float() and the cast to double."""
    gauss = torch.Tensor([exp(-(x - ws // 2) ** 2 / float(2 * 1.5 ** 2)) for x in range(ws)])
    g = gauss / gauss.sum()
    w1 = g.unsqueeze(1)
    return w1.mm(w1.t()).float().unsqueeze(0).unsqueeze(0).double()


@pytest.mark.parametrize("default", [torch.float32, torch.float64])
def test_double_window_is_the_references(default):
    old = torch.get_default_dtype()
    torch.set_default_dtype(default)
    try:
        for ws in (1, 3, 5, 7, 9, 11):
            want = _restated_window(ws)
            got = torch.tensor(ssim_mod._win2d_taps(ws), dtype=torch.float64).reshape(1, 1, ws, ws)
            assert torch.equal(got, want)
            mod = b200wave.SSIM(window_size=ws)
            x = torch.rand((1, 2, 16, 16), dtype=torch.float64)
            with pytest.raises(RuntimeError, match="CUDA-only"):   # the window is rebuilt before the kernel refuses
                mod(x, x)
            assert mod.window.dtype == torch.float64 and mod.window.shape == (2, 1, ws, ws)
            assert torch.equal(mod.window, want.expand(2, 1, ws, ws))
        if default == torch.float64:   # not the fp32 outer product: the window is not separable
            assert not torch.equal(_restated_window(11), ssim_mod.create_window(11, 1).double())
    finally:
        torch.set_default_dtype(old)


def test_new_ops_refuse_cpu_tensors():
    x4 = torch.rand((1, 1, 8, 8), dtype=torch.float64)
    x3 = x4[0]
    taps = [0.5, 0.5]
    calls = [(ops64.afb1d, (x3, taps, taps, 0)), (ops64.sfb1d, (x3, x3, taps, taps, 0, -1)),
             (ops64.swt2d, (x4, taps, taps, taps, taps, 0, 1)), (ops64.swt2d_adjoint, (x4, taps, taps, taps, taps, 0, 1)),
             (ops64.ssim_fwd, (x4, x4, [1.0], True, 0)),
             (ops64.ssim_bwd, (x4, x4, x4.expand(3, 1, 1, 8, 8), torch.ones((), dtype=torch.float64), [1.0], True,
                               False)),
             (ops64.tv_sums, (x4,)), (ops64.tv_grad, (x4, torch.ones((), dtype=torch.float64), 1.0, 1.0))]
    for op, args in calls:
        with pytest.raises(RuntimeError, match="CUDA-only"):
            op(*args)


# ---------------------------------------------------------------------------------------------- compiler output
def _compile(src, tmp_path):
    nvcc = _build.find_nvcc()
    obj = str(tmp_path / (src + ".o"))
    cmd = [nvcc] + _build.NVCC_FLAGS + ["-Xptxas", "-v", "-I", _build.INCLUDE, "-I", _build.CSRC, "-c",
                                        os.path.join(_build.CSRC, src), "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    info = {}
    cur = None
    for line in res.stdout.splitlines() + res.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            info.setdefault(cur, {})["spill"] = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            info.setdefault(cur, {})["regs"] = int(m.group(1))
    sass = subprocess.run([os.path.join(os.path.dirname(nvcc), "cuobjdump"), "-sass", obj], capture_output=True,
                          text=True).stdout
    ninstr, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            ninstr[cur] = 0
        elif cur and re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+\S", line):
            ninstr[cur] += 1
    return info, ninstr


def _nvcc_is_12_9():
    nvcc = _build.find_nvcc()
    if nvcc is None:
        return False
    return "release 12.9" in subprocess.run([nvcc, "--version"], capture_output=True, text=True).stdout


# float instantiations: (registers, SASS instructions) of the non-template kernels they replace (nvcc 12.9, -O3)
FLOAT_KERNELS = {
    "dwt1d.cu": {"afb1d_kernel": (32, 632), "sfb1d_kernel": (29, 1160)},
    "swt.cu": {"swt2d_fwd_kernel": (30, 912), "swt2d_bwd_kernel": (39, 904)},
    "tv.cu": {"tv_fwd_kernel": (80, 520), "tv_finalize_kernel": (32, 328), "tv_bwd_kernel": (123, 720)},
}


@pytest.mark.skipif(_build.find_nvcc() is None, reason="needs nvcc")
@pytest.mark.parametrize("src", ["dwt1d.cu", "swt.cu", "tv.cu", "ssim_f64.cu"])
def test_kernels_do_not_spill_and_float_code_is_unchanged(src, tmp_path):
    info, ninstr = _compile(src, tmp_path)
    assert info and all(v["spill"] == (0, 0) for v in info.values()), info
    if src == "ssim_f64.cu" or not _nvcc_is_12_9():
        return
    for short, (regs, n) in FLOAT_KERNELS[src].items():
        names = [k for k in info if re.search(r"\d%sIfE" % short, k)]
        assert len(names) == 1, (short, list(info))
        assert info[names[0]]["regs"] == regs and ninstr[names[0]] == n, (short, info[names[0]], ninstr[names[0]])
