"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the public modules /
torch.ops.b200wave (which bind the C ABI), against
  * the committed golden vectors produced by the unmodified reference, and
  * the numpy oracle on seeded inputs,
within the north_star tolerance 1e-5 relative (max|a-b| / max|b| per tensor, fp32), plus
size-independent properties at BASELINE.json's full sizes."""
import os
import sys

import numpy as np
import pytest
import torch

import b200wave
from b200wave import lowlevel
from oracle import dwt_oracle, freq_oracle, fsd_oracle, ssim_oracle, tv_oracle
from helpers import (RTOL_F32, case_filters, load_dwt1d_cases, load_dwt_cases, load_freq_cases, load_fsd_cases,
                     load_phase_cases, load_ssim_cases, load_swt_cases, load_tv_cases, rel_err)

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "pywt_standin"))

DWT_CASES = load_dwt_cases()
SSIM_CASES = load_ssim_cases()
DEV = "cuda"


def cu(a, grad=False):
    return torch.tensor(np.asarray(a), dtype=torch.float32, device=DEV, requires_grad=grad)


def modules_for(case):
    hc, hr, gc, gr = case_filters(case)
    # buffers hold reversed analysis taps; the constructor wants them un-reversed (it reverses)
    xfm = b200wave.DWTForward(J=case["J"], wave=(hc[0][::-1], hc[1][::-1], hr[0][::-1], hr[1][::-1]),
                              mode=case["mode"]).to(DEV)
    ifm = b200wave.DWTInverse(wave=(gc[0], gc[1], gr[0], gr[1]), mode=case["mode"]).to(DEV)
    return xfm, ifm


@pytest.mark.parametrize("case", DWT_CASES, ids=[c["id"] for c in DWT_CASES])
def test_golden_dwt_forward_backward(case):
    xfm, ifm = modules_for(case)
    J = case["J"]
    x = cu(case["x"], grad=True)
    yl, yh = xfm(x)
    assert yl.is_contiguous() and all(h.is_contiguous() for h in yh)       # tests/test_dwt.py:47-50
    assert rel_err(yl.detach().cpu(), case["yl"]) < RTOL_F32
    for j in range(J):
        assert tuple(yh[j].shape) == case["yh%d" % j].shape
        assert rel_err(yh[j].detach().cpu(), case["yh%d" % j]) < RTOL_F32
    (dx,) = torch.autograd.grad([yl] + list(yh), x, [cu(case["gyl"])] + [cu(case["gyh%d" % j]) for j in range(J)])
    assert rel_err(dx.cpu(), case["dx"]) < RTOL_F32


@pytest.mark.parametrize("case", DWT_CASES, ids=[c["id"] for c in DWT_CASES])
def test_golden_idwt_forward_backward(case):
    xfm, ifm = modules_for(case)
    J = case["J"]
    cl = cu(case["yl"], grad=True)
    ch = [cu(case["yh%d" % j], grad=True) for j in range(J)]
    rec = ifm((cl, ch))
    assert rec.is_contiguous()
    assert rel_err(rec.detach().cpu(), case["recon"]) < RTOL_F32
    grads = torch.autograd.grad(rec, [cl] + ch, cu(case["grec"]))
    assert rel_err(grads[0].cpu(), case["dcl"]) < RTOL_F32
    for j in range(J):
        assert rel_err(grads[1 + j].cpu(), case["dch%d" % j]) < RTOL_F32


@pytest.fixture
def double_mode():
    """The reference's fp64 mode: modules are built under torch.set_default_dtype(torch.float64) (tests/test_dwt.py:17-25)."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        yield
    finally:
        torch.set_default_dtype(old)


RTOL_F64 = 1e-12      # double arithmetic against the float64 goldens (the reference itself was run in float64)


@pytest.mark.parametrize("case", DWT_CASES, ids=[c["id"] for c in DWT_CASES])
def test_golden_dwt_double(case, double_mode):
    """The reference's `test_equal_double` mode (tests/test_dwt.py:132-160): float64 modules and inputs through the fp64
    kernels against the float64 goldens -- forward, inverse and both gradient chains, at double precision."""
    xfm, ifm = modules_for(case)
    assert xfm.h0_col.dtype == torch.float64 and ifm.g0_col.dtype == torch.float64
    J = case["J"]
    dd = lambda a, grad=False: torch.tensor(np.asarray(a, dtype=np.float64), device=DEV, requires_grad=grad)
    x = dd(case["x"], True)
    yl, yh = xfm(x)
    assert yl.dtype == torch.float64 and yl.is_contiguous() and all(h.is_contiguous() for h in yh)
    assert rel_err(yl.detach().cpu(), case["yl"]) < RTOL_F64
    for j in range(J):
        assert rel_err(yh[j].detach().cpu(), case["yh%d" % j]) < RTOL_F64
    (dx,) = torch.autograd.grad([yl] + list(yh), x, [dd(case["gyl"])] + [dd(case["gyh%d" % j]) for j in range(J)])
    assert rel_err(dx.cpu(), case["dx"]) < RTOL_F64
    cl = dd(case["yl"], True)
    ch = [dd(case["yh%d" % j], True) for j in range(J)]
    rec = ifm((cl, ch))
    assert rec.dtype == torch.float64 and rel_err(rec.detach().cpu(), case["recon"]) < RTOL_F64
    grads = torch.autograd.grad(rec, [cl] + ch, dd(case["grec"]))
    assert rel_err(grads[0].cpu(), case["dcl"]) < RTOL_F64
    for j in range(J):
        assert rel_err(grads[1 + j].cpu(), case["dch%d" % j]) < RTOL_F64


def test_double_mode_full_plane_and_mixed_dtypes(double_mode):
    """A BASELINE-sized plane in double against the oracle (perfect reconstruction at 1e-12); fp32 input into fp64
    modules and fp64 input into fp32 modules raise, as the reference's convolutions do."""
    rng = np.random.default_rng(17)
    xn = rng.standard_normal((2, 1, 304, 304))
    xfm = b200wave.DWTForward(J=3, wave="db3", mode="symmetric").to(DEV)
    ifm = b200wave.DWTInverse(wave="db3", mode="symmetric").to(DEV)
    h = (xfm.h0_col.flatten().cpu().numpy(), xfm.h1_col.flatten().cpu().numpy())
    x = torch.tensor(xn, device=DEV)
    yl, yh = xfm(x)
    oyl, oyh = dwt_oracle.dwt_forward(xn, 3, h, h, "symmetric")
    assert rel_err(yl.cpu(), oyl) < RTOL_F64
    for a, b in zip(yh, oyh):
        assert rel_err(a.cpu(), b) < RTOL_F64
    assert rel_err(ifm((yl, yh)).cpu(), xn) < 1e-11
    rec0 = ifm((yl, [None, None, None]))
    assert rec0.dtype == torch.float64
    with pytest.raises(RuntimeError, match="expected scalar type"):
        xfm(x.float())


def _wave_taps(name):
    import pywt  # the stand-in (test infrastructure)
    w = pywt.Wavelet(name)
    return w


def guarded(a, grad=False, guard=4096):
    """The array as a CUDA tensor that lives in the middle of a NaN-filled buffer: a kernel that reads before or
    behind a tensor it was given picks up NaNs (the parity check then fails) instead of silently reading mapped
    allocator memory.  compute-sanitizer is closed on this pool, so this is the in-tree substitute for global reads."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    buf = torch.full((a.size + 2 * guard,), float("nan"), dtype=torch.float32, device=DEV)
    view = buf[guard:guard + a.size].view(a.shape)
    view.copy_(torch.from_numpy(a))
    view._guard_buf = buf
    return view.requires_grad_(grad)


def guards_intact(t):
    buf = t._guard_buf
    g = (buf.numel() - t.numel()) // 2
    return bool(torch.isnan(buf[:g]).all() and torch.isnan(buf[g + t.numel():]).all())


def roundtrip_vs_oracle(wave, J, mode, shape, seed=None):
    """DWT, IDWT and the backward of both on seeded inputs against the numpy oracle; every tensor handed to the
    library sits between NaN guard bands."""
    rng = np.random.default_rng(hash((wave, J, mode)) % (2 ** 32) if seed is None else seed)
    x = rng.standard_normal(shape).astype(np.float32)
    xfm = b200wave.DWTForward(J=J, wave=wave, mode=mode).to(DEV)
    ifm = b200wave.DWTInverse(wave=wave, mode=mode).to(DEV)
    hc = (xfm.h0_col.flatten().cpu().numpy().astype(np.float64), xfm.h1_col.flatten().cpu().numpy().astype(np.float64))
    gc = (ifm.g0_col.flatten().cpu().numpy().astype(np.float64), ifm.g1_col.flatten().cpu().numpy().astype(np.float64))
    tx = guarded(x, grad=True)
    yl, yh = xfm(tx)
    oyl, oyh = dwt_oracle.dwt_forward(x.astype(np.float64), J, hc, hc, mode)
    assert rel_err(yl.detach().cpu(), oyl) < RTOL_F32
    for a, b in zip(yh, oyh):
        assert rel_err(a.detach().cpu(), b) < RTOL_F32
    rec = ifm((yl, yh))
    orec = dwt_oracle.dwt_inverse(oyl, oyh, gc, gc, mode)
    assert rel_err(rec.detach().cpu(), orec) < RTOL_F32
    # the inverse once more on coefficients that sit between guard bands themselves
    gl = guarded(yl.detach().cpu().numpy())
    ghs = [guarded(t.detach().cpu().numpy()) for t in yh]
    assert rel_err(ifm((gl, ghs)).cpu(), orec) < RTOL_F32
    assert guards_intact(gl) and all(guards_intact(t) for t in ghs)
    # full chain backward == oracle restatement of the reference's custom backwards
    g = rng.standard_normal(orec.shape).astype(np.float32)
    rec.backward(guarded(g))
    assert guards_intact(tx)
    # oracle: SFB2D.backward chain (finest first), then AFB2D.backward chain (coarsest first)
    dy = g.astype(np.float64)
    dhs = []
    in_shapes = [x.shape[-2:]] + [h.shape[-2:] for h in oyh[:-1]]
    for j in range(J):
        dlow, dhigh = dwt_oracle.sfb2d_backward(dy, gc[0], gc[1], gc[0], gc[1], mode)
        dhs.append(dhigh)
        if j + 1 < J:
            tgt = oyh[j + 1].shape[-2:]
            L = len(gc[0])
            full = tuple(2 * m if mode == "periodization" else 2 * m - L + 2 for m in tgt)
            pad = np.zeros(dlow.shape[:2] + full)
            pad[..., :dlow.shape[-2], :dlow.shape[-1]] = dlow
            dy = pad
    d = dlow
    for j in reversed(range(J)):
        d = dwt_oracle.afb2d_backward(d, dhs[j], hc[0], hc[1], hc[0], hc[1], mode, in_shapes[j])
    assert rel_err(tx.grad.cpu(), d) < RTOL_F32
    # perfect reconstruction (tests/test_dwt.py:64) where the sizes allow it
    if all(s % (2 ** J) == 0 for s in shape[-2:]) or mode != "periodization":
        r = rec.detach().cpu().numpy()[..., :shape[-2], :shape[-1]]
        assert np.abs(r - x).max() < 2e-4 * max(1.0, np.abs(x).max())


@pytest.mark.parametrize("wave,J,mode,shape", [
    ("haar", 3, "zero", (8, 1, 304, 304)),            # BASELINE cfg1
    ("db3", 3, "symmetric", (4, 1, 304, 304)),        # BASELINE cfg2 shape, smaller batch for the oracle
    ("db2", 3, "periodization", (3, 2, 127, 100)),
    ("db4", 2, "reflect", (2, 3, 99, 100)),
    ("db5", 2, "periodic", (2, 2, 65, 130)),
    ("db8", 2, "symmetric", (2, 1, 200, 333)),
    ("db6", 1, "zero", (1, 1, 31, 257)),
    ("db7", 1, "periodization", (1, 2, 64, 65)),
    ("bior2.4", 2, "periodization", (2, 2, 64, 64)),
    ("db1", 1, "reflect", (5, 1, 256, 256)),          # model.py:140 (haar/J=1/reflect on 256x256)
    ("db10", 1, "symmetric", (1, 1, 70, 90)),         # 20 taps: direct kernel
    # 16-byte aligned rows: the streaming kernels (ring + border classes, several segments / warps per row)
    ("db4", 2, "periodic", (2, 1, 128, 96)),
    ("db8", 2, "symmetric", (1, 1, 160, 200)),        # 16 taps: shifting accumulator ring
    ("db5", 3, "zero", (3, 1, 96, 160)),
    ("db2", 3, "reflect", (2, 2, 200, 104)),
    ("db1", 4, "zero", (2, 1, 128, 256)),
    ("db6", 2, "periodization", (1, 1, 96, 128)),
    ("db3", 2, "symmetric", (3, 1, 304, 304)),        # cfg2 geometry
    ("db3", 3, "symmetric", (6, 1, 304, 304)),        # cfg2 itself: the inverse crops 80 -> 79 ('unpad'), its backward
                                                      # runs the analysis chain over a zero-extended row / column
    ("db2", 3, "zero", (5, 1, 300, 296)),             # crops at two levels, zero padding, through the owner kernels
    ("db7", 2, "periodization", (1, 1, 256, 132)),
])
def test_oracle_dwt_roundtrip_seeded(wave, J, mode, shape):
    roundtrip_vs_oracle(wave, J, mode, shape)


# Full-plane oracle parity at the sizes of the cfg5 sweep (BASELINE configs[4]): here different code runs than on the
# small golden images -- many ring segments per row, the ticketed multi-level chain over big planes, sub-band widths
# 513 .. 519 with 4-byte aligned rows, the shifting accumulator ring of the long filters at scale; an odd size, whose
# rows are not 16-byte aligned (the stream kernel's 4-byte copies) in the forward chain and the inverse's backward.
_LARGE = [(size, wave, mode, J) for size in (1024, 2048) for wave in ("db1", "db4", "db8")
          for mode in ("zero", "symmetric", "periodization") for J in (1, 5)] + [(1023, "db4", "symmetric", 5)]


@pytest.mark.parametrize("size,wave,mode,J", _LARGE, ids=["%d-%s-%s-J%d" % c for c in _LARGE])
def test_oracle_parity_large_planes(size, wave, mode, J):
    roundtrip_vs_oracle(wave, J, mode, (2 if size == 1024 else 1, 1, size, size), seed=size + J)


def test_oracle_parity_sweep_batch():
    """One cfg5 point at its real batch geometry, cut to what the oracle finishes in seconds: 6 planes of 1024 x 1024
    (more planes than one CTA wave leaves idle) and an odd-sized plane (1023 x 1025: unaligned rows, odd sub-bands)."""
    roundtrip_vs_oracle("db3", 3, "symmetric", (6, 1, 1024, 1024), seed=7)
    roundtrip_vs_oracle("db4", 4, "symmetric", (1, 2, 1023, 1025), seed=8)


def test_full_size_properties_cfg2():
    """BASELINE cfg2 at full size (64x1x304x304, db3, symmetric, J=3): perfect reconstruction, linearity,
    contiguity -- size-independent properties instead of an oracle run."""
    torch.manual_seed(0)
    x = torch.rand(64, 1, 304, 304, device=DEV)
    z = torch.rand(64, 1, 304, 304, device=DEV)
    xfm = b200wave.DWTForward(J=3, wave="db3", mode="symmetric").to(DEV)
    ifm = b200wave.DWTInverse(wave="db3", mode="symmetric").to(DEV)
    yl, yh = xfm(x)
    assert [tuple(h.shape) for h in yh] == [(64, 1, 3, 154, 154), (64, 1, 3, 79, 79), (64, 1, 3, 42, 42)]
    assert tuple(yl.shape) == (64, 1, 42, 42)
    rec = ifm((yl, yh))
    assert tuple(rec.shape) == (64, 1, 304, 304)
    assert (rec - x).abs().max().item() < 1e-5
    zl, zh = xfm(z)
    sl, sh = xfm(2.0 * x - 3.0 * z)
    assert (sl - (2.0 * yl - 3.0 * zl)).abs().max().item() < 1e-4
    for a, b, c in zip(sh, yh, zh):
        assert (a - (2.0 * b - 3.0 * c)).abs().max().item() < 1e-4
    # every plane is independent: a batch slice transforms to the slice of the transform
    yl8, yh8 = xfm(x[8:16])
    assert torch.equal(yl8, yl[8:16]) and all(torch.equal(a, b[8:16]) for a, b in zip(yh8, yh))


def test_commutativity_of_subbands():
    """tests/test_dwt.py:163-197: reconstructing from one sub-band at a time and summing == reconstructing all."""
    torch.manual_seed(1)
    x = torch.randn(5, 4, 64, 64, device=DEV)
    for wave, J, mode in [("db3", 2, "symmetric"), ("db2", 3, "periodization"), ("db4", 2, "zero")]:
        xfm = b200wave.DWTForward(J=J, wave=wave, mode=mode).to(DEV)
        ifm = b200wave.DWTInverse(wave=wave, mode=mode).to(DEV)
        yl, yh = xfm(x)
        full = ifm((yl, yh))
        zeros = [torch.zeros_like(h) for h in yh]
        parts = ifm((yl, zeros))
        for j in range(J):
            for b in range(3):
                only = list(zeros)
                t = torch.zeros_like(yh[j])
                t[:, :, b] = yh[j][:, :, b]
                only[j] = t
                parts = parts + ifm((torch.zeros_like(yl), only))
        assert (parts - full).abs().max().item() < 1e-4
        # None == zeros for the detail bands (pw/dwt/transform2d.py:137-139); single level so no 'unpad' is skipped
        if J == 1:
            assert torch.equal(ifm((yl, [None])), ifm((yl, zeros)))
    xfm = b200wave.DWTForward(J=1, wave="db3", mode="zero").to(DEV)
    ifm = b200wave.DWTInverse(wave="db3", mode="zero").to(DEV)
    yl, yh = xfm(x)
    assert torch.allclose(ifm((yl, [None])), ifm((yl, [torch.zeros_like(yh[0])])), atol=1e-6)


def test_gradients_match_time_reversed_filters():
    """tests/test_dwt.py:200-299: AFB2D backward == DWTInverse with (dec_lo[::-1], dec_hi[::-1]); SFB2D backward
    == DWTForward with those filters -- for modes where the reference's backward is the true adjoint."""
    torch.manual_seed(2)
    w = b200wave.Wavelet("db3")
    for mode in ("zero", "periodization"):
        xfm = b200wave.DWTForward(J=1, wave="db3", mode=mode).to(DEV)
        ifm_t = b200wave.DWTInverse(wave=(w.dec_lo[::-1], w.dec_hi[::-1]), mode=mode).to(DEV)
        x = torch.randn(5, 6, 128, 128, device=DEV, requires_grad=True)
        yl, yh = xfm(x)
        gl, gh = torch.randn_like(yl), torch.randn_like(yh[0])
        (dx,) = torch.autograd.grad([yl, yh[0]], x, [gl, gh])
        ref = ifm_t((gl, [gh]))
        assert (dx - ref[..., :128, :128]).abs().max().item() < 1e-4


def test_mixed_and_odd_length_filters_direct_kernel():
    """4-tuple wave with different lengths per axis and an odd-length filter exercise the direct kernels."""
    rng = np.random.default_rng(11)
    x = rng.standard_normal((2, 2, 40, 52)).astype(np.float32)
    h_w = (rng.standard_normal(5), rng.standard_normal(5))     # odd length, along W ("col" slot)
    h_h = (rng.standard_normal(4), rng.standard_normal(4))
    for mode in ("zero", "symmetric", "periodic", "reflect"):
        xfm = b200wave.DWTForward(J=1, wave=(h_w[0], h_w[1], h_h[0], h_h[1]), mode=mode).to(DEV)
        ifm = b200wave.DWTInverse(wave=(h_w[0], h_w[1], h_h[0], h_h[1]), mode=mode).to(DEV)
        yl, yh = xfm(cu(x))
        f = lambda t: t.flatten().cpu().numpy().astype(np.float64)
        oyl, oyh = dwt_oracle.dwt_forward(x.astype(np.float64), 1, (f(xfm.h0_col), f(xfm.h1_col)),
                                          (f(xfm.h0_row), f(xfm.h1_row)), mode)
        assert rel_err(yl.cpu(), oyl) < RTOL_F32 and rel_err(yh[0].cpu(), oyh[0]) < RTOL_F32
        rec = ifm((yl, yh))
        orec = dwt_oracle.dwt_inverse(oyl, oyh, (f(ifm.g0_col), f(ifm.g1_col)), (f(ifm.g0_row), f(ifm.g1_row)), mode)
        assert rel_err(rec.cpu(), orec) < RTOL_F32


def test_strided_and_noncontiguous_inputs():
    torch.manual_seed(3)
    base = torch.randn(4, 3, 70, 90, device=DEV)
    xfm = b200wave.DWTForward(J=1, wave="db2", mode="symmetric").to(DEV)
    views = [base[:, :, 3:67, 5:85], base[:, 1:2], base[::2], base.transpose(2, 3), base[:, :, :, ::2]]
    for v in views:
        a_l, a_h = xfm(v)
        b_l, b_h = xfm(v.contiguous())
        assert torch.equal(a_l, b_l) and torch.equal(a_h[0], b_h[0])
    # a three-level chain on rows that are not 16-byte aligned (the stream kernel with 4-byte copies) against the
    # contiguous copy (16-byte copies): bit-identical, forward and backward
    from b200wave import _cabi
    big = torch.randn(2, 1, 1030, 1030, device=DEV)
    xfm = b200wave.DWTForward(J=3, wave="db3", mode="symmetric").to(DEV)
    xu = big.clone().requires_grad_()
    xc = big[..., 3:1027, 5:1029].contiguous().requires_grad_()
    a_l, a_h = xfm(xu[..., 3:1027, 5:1029])
    assert _cabi.recent_kernels(1) == ["afb_stream_kernel"]
    b_l, b_h = xfm(xc)
    assert torch.equal(a_l, b_l) and all(torch.equal(a, b) for a, b in zip(a_h, b_h))
    gl, gh = torch.randn_like(a_l), [torch.randn_like(h) for h in a_h]
    (da,) = torch.autograd.grad([a_l] + a_h, xu, [gl] + gh)
    (db,) = torch.autograd.grad([b_l] + b_h, xc, [gl] + gh)
    assert torch.equal(da[..., 3:1027, 5:1029], db)


def test_error_behaviour_on_gpu():
    x = torch.zeros(1, 1, 16, 16, device=DEV)
    for bad in ("constant", "replicate"):            # accepted by mode_to_int, rejected downstream
        with pytest.raises(ValueError, match="Unkown pad type: %s" % bad):
            b200wave.DWTForward(mode=bad).to(DEV)(x)
    with pytest.raises(RuntimeError, match="expected scalar type Float"):
        b200wave.DWTForward().to(DEV)(x.double())
    with pytest.raises(IndexError):
        b200wave.DWTForward().to(DEV)(x[0])
    with pytest.raises(RuntimeError, match="reflect"):
        b200wave.DWTForward(wave="db4", mode="reflect").to(DEV)(torch.zeros(1, 1, 4, 4, device=DEV))
    # empty batch
    yl, yh = b200wave.DWTForward(J=2, wave="db2").to(DEV)(torch.zeros(0, 3, 16, 16, device=DEV))
    assert yl.shape == (0, 3, 6, 6) and yh[0].shape == (0, 3, 3, 9, 9)


def test_functional_afb2d_sfb2d():
    torch.manual_seed(4)
    x = torch.randn(2, 3, 32, 48, device=DEV)
    w = b200wave.Wavelet("db2")
    y = lowlevel.afb2d(x, (w.dec_lo, w.dec_hi), mode="periodization")
    assert y.shape == (2, 12, 16, 24)
    y5 = y.reshape(2, 3, 4, 16, 24)
    rec = lowlevel.sfb2d(y5[:, :, 0].contiguous(), y5[:, :, 1], y5[:, :, 2], y5[:, :, 3], (w.rec_lo, w.rec_hi),
                         mode="periodization")
    assert (rec - x).abs().max().item() < 1e-5


# ------------------------------------------------------------------------------------------- SSIM
@pytest.mark.parametrize("case", SSIM_CASES, ids=[c["id"] for c in SSIM_CASES])
def test_golden_ssim(case):
    a, b = cu(case["img1"], grad=True), cu(case["img2"], grad=True)
    mod = b200wave.SSIM(window_size=11, size_average=case["size_average"])
    val = mod(a, b)
    assert rel_err(np.atleast_1d(val.detach().cpu().numpy()), np.atleast_1d(case["val"])) < RTOL_F32
    val.backward(cu(case["gout"]) if not case["size_average"] else None)
    scale = np.abs(case["d1"]).max()
    if scale > 1e-12:
        assert rel_err(a.grad.cpu(), case["d1"]) < RTOL_F32
        assert rel_err(b.grad.cpu(), case["d2"]) < RTOL_F32
    else:   # ssim(x, x): zero gradient up to fp32 rounding of O(1/NCHW) terms
        assert a.grad.abs().max().item() < 1e-9


@pytest.mark.parametrize("shape,size_average", [
    ((2, 1, 400, 400), True),        # BASELINE cfg3 shape, small batch for the oracle
    ((3, 2, 67, 131), False),        # odd sizes: scalar staging path, partial strips
    ((1, 3, 31, 64), True),
    ((2, 1, 304, 304), True),        # cfg1
    ((1, 1, 9, 7), True),            # smaller than the window
])
def test_oracle_ssim_seeded(shape, size_average):
    rng = np.random.default_rng(abs(hash(shape)) % (2 ** 32))
    x = rng.random(shape).astype(np.float32)
    y = np.clip(x + 0.1 * rng.standard_normal(shape), 0, 1).astype(np.float32)
    a, b = cu(x, grad=True), cu(y, grad=True)
    val = b200wave.ssim(a, b, window_size=11, size_average=size_average)
    oval = ssim_oracle.ssim(x.astype(np.float64), y.astype(np.float64), 11, size_average)
    assert rel_err(np.atleast_1d(val.detach().cpu().numpy()), np.atleast_1d(oval)) < RTOL_F32
    gout = np.linspace(0.5, 1.5, shape[0]) if not size_average else 1.0
    val.backward(cu(gout) if not size_average else None)
    o1, o2 = ssim_oracle.ssim_backward(x.astype(np.float64), y.astype(np.float64), gout, 11, size_average)
    assert rel_err(a.grad.cpu(), o1) < RTOL_F32
    assert rel_err(b.grad.cpu(), o2) < RTOL_F32


def test_ssim_grad_only_second_argument_and_identity():
    rng = np.random.default_rng(5)
    x = rng.random((2, 2, 40, 56)).astype(np.float32)
    y = rng.random((2, 2, 40, 56)).astype(np.float32)
    a, b = cu(x), cu(y, grad=True)
    val = b200wave.ssim(a, b)
    val.backward()
    _, o2 = ssim_oracle.ssim_backward(x.astype(np.float64), y.astype(np.float64))
    assert rel_err(b.grad.cpu(), o2) < RTOL_F32 and a.grad is None
    with torch.no_grad():
        assert abs(b200wave.ssim(a, a).item() - 1.0) < 1e-6
    # smaller odd windows go through the same kernel with zero outer taps
    v5 = b200wave.ssim(a, b.detach(), window_size=5).item()
    assert abs(v5 - ssim_oracle.ssim(x.astype(np.float64), y.astype(np.float64), 5)) < 1e-6


def test_full_size_properties_cfg3():
    """BASELINE cfg3 at full size (256x1x400x400): symmetry, identity, per-sample means average to the global mean,
    batch independence."""
    torch.manual_seed(0)
    x = torch.rand(256, 1, 400, 400, device=DEV)
    y = (x + 0.1 * torch.randn_like(x)).clamp_(0, 1)
    s_xy = b200wave.ssim(x, y)
    s_yx = b200wave.ssim(y, x)
    assert abs(s_xy.item() - s_yx.item()) < 1e-6
    assert abs(b200wave.ssim(x, x).item() - 1.0) < 1e-6
    per = b200wave.ssim(x, y, size_average=False)
    assert per.shape == (256,) and abs(per.double().mean().item() - s_xy.item()) < 1e-6
    per8 = b200wave.ssim(x[8:16], y[8:16], size_average=False)
    assert torch.allclose(per8, per[8:16], atol=1e-6)
    xg = x.clone().requires_grad_(True)
    b200wave.SSIM()(xg, y).backward()
    assert xg.grad.shape == x.shape and torch.isfinite(xg.grad).all()
    # the mean's gradient is O(1/NCHW); directional derivative check against a finite difference
    d = torch.randn_like(x)
    eps = 1e-2
    fd = (b200wave.ssim(x + eps * d, y).double() - b200wave.ssim(x - eps * d, y).double()) / (2 * eps)
    an = (xg.grad.double() * d.double()).sum()
    assert abs(fd.item() - an.item()) < 2e-3 * max(1e-3, abs(an.item())) + 1e-6


def test_host_pipeline_matches_direct_call():
    """b200wave.HostPipeline (chunked, stream-overlapped host-buffer front end) == the plain device call."""
    torch.manual_seed(5)
    xfm = b200wave.DWTForward(J=2, wave="db3", mode="symmetric").to(DEV)
    ifm = b200wave.DWTInverse(wave="db3", mode="symmetric").to(DEV)

    def step(x, g):
        x.grad = None
        yl, yh = xfm(x)
        rec = ifm((yl, yh))
        rec.backward(g)
        return rec, x.grad

    xh = torch.rand(10, 1, 76, 76).pin_memory().requires_grad_(True)
    gh = torch.randn(10, 1, 76, 76).pin_memory()
    xd = xh.detach().to(DEV).requires_grad_(True)
    rec_ref, dx_ref = step(xd, gh.to(DEV))
    for chunks, graph in [(1, False), (3, False), (4, True), (5, True)]:
        pipe = b200wave.HostPipeline(step, (xh, gh), chunks=chunks, graph=graph)
        for _ in range(2):   # second call exercises buffer reuse
            rec, dx = pipe((xh, gh))
        assert rec.shape == rec_ref.shape and dx.shape == dx_ref.shape
        assert rel_err(rec, rec_ref.detach().cpu()) < 1e-6
        assert rel_err(dx, dx_ref.detach().cpu()) < 1e-6


@pytest.mark.parametrize("env", ["B200W_FORCE_DIRECT=1", "B200W_OWNER=2", "B200W_OWNER=0", "B200W_TMA=0",
                                 "B200W_TMA=0 B200W_OWNER=2",
                                 "B200W_TMA_NOBOXES=1 B200W_OWNER=2", "B200W_TMA_G=2 B200W_TMA_D=2 B200W_OWNER=2"])
def test_alternative_kernel_paths(env):
    """The same golden / oracle cases through the other implementations of the path (the env switches are read
    once per process, hence a child pytest): direct kernels (with the store epilogue of filter_wavelet), the owner
    kernels forced onto every multi-level shape that fits (TMA-staged ones first; B200W_TMA=0: the cp.async ones), the
    ticketed chain kernels alone, the TMA kernels with row-by-row staging of the extension rows / with few streams and
    the shallowest ring."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    child_env = dict(os.environ)
    for kv in env.split():
        k, v = kv.split("=")
        child_env[k] = v
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_parity.py"), "-q", "-x",
                          "-m", "gpu", "-k", "golden_dwt or golden_idwt or oracle_dwt_roundtrip or commutativity or "
                          "owner_kernel or filter_wavelet",
                          "-p", "no:cacheprovider"],
                         cwd=root, env=child_env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                         timeout=1500)
    assert res.returncode == 0, res.stdout[-3000:]


@pytest.mark.parametrize("env", ["B200W_OWNER=0", "B200W_OWNER=2", "B200W_TMA=0"])
def test_large_planes_other_policies(env):
    """The large-plane oracle comparisons through the other kernel-selection policies (child pytest: the switches are
    read once per process)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    child_env = dict(os.environ)
    for kv in env.split():
        k, v = kv.split("=")
        child_env[k] = v
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_parity.py"), "-q", "-x",
                          "-m", "gpu", "-k", "large_planes and not other_policies and not 2048-db8 or sweep_batch",
                          "-p", "no:cacheprovider"],
                         cwd=root, env=child_env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                         timeout=1500)
    assert res.returncode == 0, res.stdout[-3000:]


@pytest.mark.parametrize("env", ["", "B200W_TMA=0", "B200W_OWNER=0"])
def test_bounds_build(env):
    """The B200W_BOUNDS debug build of the library (device-side checks of every shared-memory access, staged copy and
    global store of the stream / owner / TMA kernels against the CTA's shared-memory size and the buffers the launch
    was given; a violation traps) through the golden, owner-shape and one large-plane case: the in-tree substitute for
    compute-sanitizer, which is closed on this pool.  The library is built by `python -m b200wave._build --bounds`
    (minutes of nvcc time, so it is not part of the default build; it travels with the snapshot)."""
    import subprocess
    from b200wave import _build
    stamp = os.path.join(_build.LIB_DIR, "libb200wave_bounds.stamp")
    fresh = os.path.exists(_build.BOUNDS_LIB_PATH) and os.path.exists(stamp) and \
        open(stamp).read().strip() == _build._source_hash() + "+bounds"
    if not fresh:
        if os.environ.get("B200W_BUILD_BOUNDS") == "1" and _build.find_nvcc():
            _build.build_bounds()
        else:
            pytest.skip("libb200wave_bounds.so is missing or stale: python -m b200wave._build --bounds")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    child_env = dict(os.environ)
    child_env["B200W_LIBRARY"] = _build.BOUNDS_LIB_PATH
    for kv in env.split():
        k, v = kv.split("=")
        child_env[k] = v
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_parity.py"), "-q", "-x",
                          "-m", "gpu", "-k", "golden_dwt or golden_idwt or owner_kernel or 1024-db4-symmetric-J5 or "
                          "1024-db1-zero-J5 or sweep_batch", "-p", "no:cacheprovider"],
                         cwd=root, env=child_env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                         timeout=2400)
    if res.returncode != 0:   # the device printf repeats per thread: show the first few violations and pytest's summary
        lines = res.stdout.splitlines()
        hits = [ln.strip() for ln in lines if "B200W_BOUNDS" in ln][:6]
        tail = [ln for ln in lines if ln.startswith(("FAILED", "ERROR")) or " passed" in ln or " failed" in ln][-4:]
        pytest.fail("\n".join(hits + tail) or res.stdout[-3000:])


FREQ_CASES = load_freq_cases()


@pytest.mark.parametrize("case", FREQ_CASES, ids=[c["id"] for c in FREQ_CASES])
def test_golden_freq_split(case):
    """b200wave.freq.high_pass / low_pass (same signature as utils.py:93-117) vs the reference's own outputs."""
    from b200wave import freq
    t = cu(case["x"])
    out = freq.high_pass(t, i=case["radius"]) if case["highpass"] else freq.low_pass(t, i=case["radius"])
    assert tuple(out.shape) == case["y"].shape and out.is_contiguous()
    assert rel_err(out.cpu(), case["y"]) < RTOL_F32


def test_freq_split_batched_and_gradient():
    """Batched form == per-image calls == float64 oracle; gradient == oracle (self-adjoint filter, sgn through abs)."""
    from b200wave import freq
    rng = np.random.default_rng(11)
    x = rng.random((3, 2, 96, 80)).astype(np.float32)
    g = rng.standard_normal((3, 2, 96, 80)).astype(np.float32)
    for radius, hp, sign in [(10, True, 1.0), (8, False, -1.0)]:
        tx = cu(x, grad=True)
        out = freq.gaussian_split(tx, radius, hp, sign)
        ref = freq_oracle.split(x, radius, hp, sign)
        assert rel_err(out.detach().cpu(), ref) < RTOL_F32
        one = (freq.high_pass if hp else freq.low_pass)(cu(x[1, 1][None]), i=radius)
        assert rel_err(one.cpu(), ref[1, 1]) < RTOL_F32
        out.backward(cu(g))
        assert rel_err(tx.grad.cpu(), freq_oracle.split_backward(x, g, radius, hp, sign)) < RTOL_F32
    with pytest.raises(RuntimeError, match="CUDA-only"):
        freq.high_pass(torch.rand(1, 8, 8))


def test_more_levels_than_one_launch_holds():
    """J > B200W_MAX_LEVELS (8): DWTForward / DWTInverse split the chain into several launches."""
    rng = np.random.default_rng(7)
    x = rng.standard_normal((1, 2, 600, 520)).astype(np.float32)
    J = 9
    xfm = b200wave.DWTForward(J=J, wave="db1", mode="zero").to(DEV)
    ifm = b200wave.DWTInverse(wave="db1", mode="zero").to(DEV)
    hc = (xfm.h0_col.flatten().cpu().numpy().astype(np.float64), xfm.h1_col.flatten().cpu().numpy().astype(np.float64))
    gc = (ifm.g0_col.flatten().cpu().numpy().astype(np.float64), ifm.g1_col.flatten().cpu().numpy().astype(np.float64))
    tx = cu(x, grad=True)
    yl, yh = xfm(tx)
    assert len(yh) == J
    oyl, oyh = dwt_oracle.dwt_forward(x.astype(np.float64), J, hc, hc, "zero")
    assert rel_err(yl.detach().cpu(), oyl) < RTOL_F32
    for a, b in zip(yh, oyh):
        assert rel_err(a.detach().cpu(), b) < RTOL_F32
    rec = ifm((yl, yh))
    orec = dwt_oracle.dwt_inverse(oyl, oyh, gc, gc, "zero")
    assert rel_err(rec.detach().cpu(), orec) < RTOL_F32
    rec.sum().backward()
    assert tx.grad is not None and torch.isfinite(tx.grad).all()


FSD_CASES = load_fsd_cases()


@pytest.mark.parametrize("case", FSD_CASES, ids=[c["id"] for c in FSD_CASES])
def test_golden_filter_wavelet(case):
    """b200wave.fsd.WaveletFilter vs FS_DiscriminatorA/B.filter_wavelet (model.py:166-179, 222-235): the reference's
    own outputs and input gradients."""
    from b200wave import fsd
    filt = fsd.WaveletFilter(cs=case["cs"], variant=case["variant"]).to(DEV)
    x = cu(case["x"], grad=True)
    res = filt(x, case["norm"])
    assert res[-1] is x and len(res) - 1 == len(case["y"])
    for got, want in zip(res[:-1], case["y"]):
        assert tuple(got.shape) == want.shape
        assert rel_err(got.detach().cpu(), want) < RTOL_F32
    (dx,) = torch.autograd.grad(list(res[:-1]), x, [cu(g) for g in case["g"]])
    assert rel_err(dx.cpu(), case["dx"]) < RTOL_F32


@pytest.mark.parametrize("shape", [(8, 1, 256, 256), (3, 1, 304, 304), (2, 1, 1024, 1024), (2, 2, 130, 74),
                                   (1, 1, 67, 93), (5, 1, 2, 2)])
def test_filter_wavelet_matches_unfused_path(shape):
    """The store epilogue (skipped bands, 0.5*v+0.5) is bit-identical to DWTForward followed by the reference's
    slicing and scaling (0.5*v is exact, so the fused multiply-add rounds like the separate multiply and add) -- at
    the training crop size (train.py: 256x256), the BASELINE sizes and ragged ones; and it matches the oracle."""
    from b200wave import fsd
    rng = np.random.default_rng(shape[-1])
    xn = rng.standard_normal(shape).astype(np.float32)
    x = cu(xn)
    xfm = b200wave.DWTForward(J=1, wave="haar", mode="reflect").to(DEV)
    ll, (hi,) = xfm(x)
    for variant in "AB":
        for cs in ("sum", "each", "cat"):
            for norm in (True, False):
                got = fsd.filter_wavelet(x, cs, norm, variant)[:-1]
                h = hi * 0.5 + 0.5 if norm else hi
                if cs == "sum":
                    want = (ll,) if variant == "A" else (h[:, :, 2],)
                elif cs == "each":
                    want = (ll, h[:, :, 0], h[:, :, 1], h[:, :, 2])
                else:
                    want = (torch.cat((h[:, :, 0], h[:, :, 1], h[:, :, 2]), 1),)
                assert len(got) == len(want)
                for a, b in zip(got, want):
                    assert torch.equal(a, b), (variant, cs, norm)
                ora = fsd_oracle.filter_wavelet(xn, cs, norm, variant)
                for a, b in zip(got, ora):
                    assert rel_err(a.cpu(), b) < RTOL_F32


def test_filter_wavelet_other_filters_and_errors():
    """Longer filters and other modes go through the same epilogue (stream ring with 16- and 4-byte copies, border
    items)."""
    from b200wave import fsd, ops
    rng = np.random.default_rng(5)
    for wave, mode, shape in [("db2", "symmetric", (2, 1, 96, 200)), ("db4", "zero", (1, 2, 301, 77)),
                              ("db3", "periodization", (2, 1, 64, 1000)), ("db8", "periodic", (1, 1, 200, 136))]:
        x = cu(rng.standard_normal(shape).astype(np.float32))
        ll, (hi,) = b200wave.DWTForward(J=1, wave=wave, mode=mode).to(DEV)(x)
        filt = fsd.WaveletFilter(cs="each", wave=wave, mode=mode).to(DEV)
        got = filt(x)
        assert torch.equal(got[0], ll)
        for b in range(3):
            assert torch.equal(got[1 + b], hi[:, :, b] * 0.5 + 0.5)
        cat = fsd.WaveletFilter(cs="cat", variant="B", wave=wave, mode=mode).to(DEV)(x, False)[0]
        assert torch.equal(cat, torch.cat((hi[:, :, 0], hi[:, :, 1], hi[:, :, 2]), 1))
        # a strided view: rows that are not 16-byte aligned (4-byte copies into the stream kernel's ring)
        xs = x[..., 1:]
        lls, (his,) = b200wave.DWTForward(J=1, wave=wave, mode=mode).to(DEV)(xs)
        gs = filt(xs)
        assert torch.equal(gs[0], lls) and torch.equal(gs[3], his[:, :, 2] * 0.5 + 0.5)
    with pytest.raises(NotImplementedError, match="not recognized"):
        fsd.filter_wavelet(x, cs="avg")
    with pytest.raises(RuntimeError, match="CUDA-only"):
        fsd.filter_wavelet(torch.rand(1, 1, 8, 8))
    with pytest.raises(ValueError):
        t = ops.afb2d_select(x, [1.0, 1.0], [1.0, -1.0], [1.0, 1.0], [1.0, -1.0], 4, False, False, 1.0, 0.0)


def test_patch_model_swaps_the_discriminator_methods():
    """compat.patch_model on a stand-in for the reference's model module: classes that, like FS_DiscriminatorA/B
    (model.py:140-142, 190-192), own ``DWT2 = DWTForward(J=1, 'haar', 'reflect')`` and ``cs``."""
    import types
    from b200wave import compat

    class A(torch.nn.Module):
        def __init__(self, cs):
            super().__init__()
            self.DWT2 = b200wave.DWTForward(J=1, wave="haar", mode="reflect")
            self.cs = cs

        def filter_wavelet(self, x, norm=True):
            raise AssertionError("not patched")

    class B(A):
        pass

    mod = compat.patch_model(types.SimpleNamespace(FS_DiscriminatorA=A, FS_DiscriminatorB=B))
    case = [c for c in FSD_CASES if c["variant"] == "B" and c["cs"] == "cat"][0]
    got, x = mod.FS_DiscriminatorB("cat").to(DEV).filter_wavelet(cu(case["x"]), case["norm"])
    assert rel_err(got.cpu(), case["y"][0]) < RTOL_F32
    case = [c for c in FSD_CASES if c["variant"] == "A" and c["cs"] == "sum"][0]
    got, x = mod.FS_DiscriminatorA("sum").to(DEV).filter_wavelet(cu(case["x"]), case["norm"])
    assert rel_err(got.cpu(), case["y"][0]) < RTOL_F32
    assert mod.TVLoss is b200wave.TVLoss and mod.phase_consistency_loss is b200wave.phase_consistency_loss


_OWNER_GRID = [((12, 1, 128, 160), w, m, 3) for w in ("haar", "db2", "db3", "db4", "db5", "db8")
               for m in ("zero", "symmetric", "reflect", "periodic", "periodization")]


@pytest.mark.parametrize("shape,wave,mode,J", [((64, 1, 76, 76), "db3", "symmetric", 3),
                                               ((160, 1, 50, 66), "db2", "reflect", 2),
                                               ((40, 2, 75, 83), "haar", "zero", 4),
                                               ((80, 1, 64, 96), "db4", "periodization", 3),
                                               ((37, 2, 61, 47), "db5", "periodic", 2),
                                               ((16, 1, 256, 256), "db3", "zero", 3),
                                               ((8, 1, 512, 384), "db2", "zero", 4),     # first level(s) as a chain launch
                                               ((8, 1, 640, 512), "db4", "symmetric", 5),
                                               ((24, 1, 128, 192), "db4", "zero", 2),
                                               ((64, 1, 304, 304), "db3", "symmetric", 3)] + _OWNER_GRID)
def test_owner_kernel_shapes(shape, wave, mode, J):
    """Shapes the default policy hands to the owner kernel (small planes with 16-byte aligned rows, J > 1; parts of a
    plane overlap by the rows the deeper levels need) against the oracle, forward, inverse and gradient -- including
    every padding mode x filter length on one shape (zero rows / wrapped rows / long filters in every code path)."""
    rng = np.random.default_rng(J * 100 + shape[-1])
    xn = rng.standard_normal(shape).astype(np.float32)
    xfm = b200wave.DWTForward(J=J, wave=wave, mode=mode).to(DEV)
    h = (xfm.h0_col.flatten().cpu().numpy().astype(np.float64), xfm.h1_col.flatten().cpu().numpy().astype(np.float64))
    yl_o, yh_o = dwt_oracle.dwt_forward(xn.astype(np.float64), J, h, h, mode)
    x = cu(xn, grad=True)
    yl, yh = xfm(x)
    assert rel_err(yl.detach().cpu(), yl_o) < RTOL_F32
    for a, b in zip(yh, yh_o):
        assert rel_err(a.detach().cpu(), b) < RTOL_F32
    # synthesis chain on the same coefficients (owner kernel of the inverse transform)
    ifm = b200wave.DWTInverse(wave=wave, mode=mode).to(DEV)
    g = (ifm.g0_col.flatten().cpu().numpy().astype(np.float64), ifm.g1_col.flatten().cpu().numpy().astype(np.float64))
    rec = ifm((yl.detach(), [t.detach() for t in yh]))
    assert rel_err(rec.cpu(), dwt_oracle.dwt_inverse(yl_o, yh_o, g, g, mode)) < RTOL_F32
    rec0 = ifm((yl.detach(), [None] * J))                    # detail bands absent = zeros (and no 'unpad' crops)
    if rec0.shape == rec.shape:
        assert rel_err(rec0.cpu(), dwt_oracle.dwt_inverse(yl_o, [np.zeros_like(t) for t in yh_o], g, g, mode)) < RTOL_F32
    # gradient: the reference's AFB2D.backward chain, level by level
    gl = rng.standard_normal(yl_o.shape).astype(np.float32)
    gh = [rng.standard_normal(b.shape).astype(np.float32) for b in yh_o]
    (dx,) = torch.autograd.grad([yl] + list(yh), x, [cu(gl)] + [cu(g) for g in gh])
    d = gl.astype(np.float64)
    sizes = [xn.shape[-2:]] + [b.shape[-2:] for b in yh_o[:-1]]
    for j in range(J - 1, -1, -1):
        d = dwt_oracle.afb2d_backward(d, gh[j].astype(np.float64), h[0], h[1], h[0], h[1], mode, sizes[j])
    assert rel_err(dx.cpu(), d) < RTOL_F32


TV_CASES = load_tv_cases()


@pytest.mark.parametrize("case", TV_CASES, ids=[c["id"] for c in TV_CASES])
def test_golden_tv_loss(case):
    """b200wave.losses.TVLoss vs the reference module's own value and input gradient (model.py:17-33)."""
    from b200wave.losses import TVLoss
    x = cu(case["x"], grad=True)
    loss = TVLoss(case["weight"])(x)
    assert loss.dim() == 0
    assert abs(loss.item() - case["loss"]) <= RTOL_F32 * abs(case["loss"])
    loss.backward()
    assert rel_err(x.grad.cpu(), case["dx"]) < RTOL_F32


DWT1D_CASES = load_dwt1d_cases()


@pytest.mark.parametrize("case", DWT1D_CASES, ids=[c["id"] for c in DWT1D_CASES])
def test_golden_dwt1d_forward_inverse_backward(case):
    """b200wave.DWT1DForward / DWT1DInverse vs the unmodified reference (transform1d.py): coefficients, reconstruction,
    the input gradient (AFB1D.backward chain) and the coefficient gradients (SFB1D.backward chain)."""
    J, mode = case["J"], case["mode"]
    xfm = b200wave.DWT1DForward(J=J, wave=(case["h0"][::-1].copy(), case["h1"][::-1].copy()), mode=mode).to(DEV)
    ifm = b200wave.DWT1DInverse(wave=(case["g0"], case["g1"]), mode=mode).to(DEV)
    assert np.allclose(xfm.h0.flatten().cpu().numpy(), case["h0"]) and tuple(xfm.h0.shape) == (1, 1, len(case["h0"]))
    x = cu(case["x"], grad=True)
    yl, yh = xfm(x)
    assert yl.is_contiguous() and all(t.is_contiguous() for t in yh) and len(yh) == J
    assert rel_err(yl.detach().cpu(), case["yl"]) < RTOL_F32
    for j in range(J):
        assert rel_err(yh[j].detach().cpu(), case["yh%d" % j]) < RTOL_F32
    (dx,) = torch.autograd.grad([yl] + list(yh), x, [cu(case["gl"])] + [cu(case["gh%d" % j]) for j in range(J)])
    assert rel_err(dx.cpu(), case["dx"]) < RTOL_F32
    cl = cu(case["yl"], grad=True)
    ch = [cu(case["yh%d" % j], grad=True) for j in range(J)]
    rec = ifm((cl, ch))
    assert rec.is_contiguous() and rel_err(rec.detach().cpu(), case["rec"]) < RTOL_F32
    grads = torch.autograd.grad(rec, [cl] + ch, cu(case["gy"]))
    assert rel_err(grads[0].cpu(), case["dcl"]) < RTOL_F32
    for j in range(J):
        assert rel_err(grads[1 + j].cpu(), case["dch%d" % j]) < RTOL_F32


@pytest.mark.parametrize("wave", ["haar", "db4", "db8"])
@pytest.mark.parametrize("mode", ["zero", "symmetric", "reflect", "periodic", "periodization"])
def test_oracle_dwt1d_long_signals(wave, mode):
    """Long odd-length signals (many CTAs, interior fast path + both border paths), every padding mode, against the
    oracle; perfect reconstruction; absent detail bands = zeros; strided (non-contiguous) input rows."""
    rng = np.random.default_rng(len(wave) * 7 + len(mode))
    xn = rng.standard_normal((3, 2, 100003)).astype(np.float32)
    xfm = b200wave.DWT1DForward(J=3, wave=wave, mode=mode).to(DEV)
    ifm = b200wave.DWT1DInverse(wave=wave, mode=mode).to(DEV)
    h0, h1 = (xfm.h0.flatten().cpu().numpy().astype(np.float64), xfm.h1.flatten().cpu().numpy().astype(np.float64))
    g0, g1 = (ifm.g0.flatten().cpu().numpy().astype(np.float64), ifm.g1.flatten().cpu().numpy().astype(np.float64))
    yl, yh = xfm(cu(xn))
    lo = xn.astype(np.float64)
    for j in range(3):
        lo, hi = dwt_oracle.afb1d(lo, h0, h1, mode)
        assert rel_err(yh[j].cpu(), hi) < RTOL_F32
    assert rel_err(yl.cpu(), lo) < RTOL_F32
    rec = ifm((yl, yh))
    if mode in ("periodization",):
        assert rec.shape[-1] == xn.shape[-1] + 1          # odd length: the reference returns the even extension
    assert rel_err(rec[..., :xn.shape[-1]].cpu(), xn) < RTOL_F32
    r = lo
    for j in range(2, -1, -1):
        z = np.zeros_like(yh[j].cpu().numpy(), dtype=np.float64)
        if r.shape[-1] > z.shape[-1]:
            r = r[..., :-1]
        r = dwt_oracle.sfb1d(r, z, g0, g1, mode)
    rec0 = ifm((yl, [None, None, None]))
    if rec0.shape == r.shape:      # without detail bands the reference applies no 'unpad' (transform1d.py:106-112)
        assert rel_err(rec0.cpu(), r) < RTOL_F32
    xs = cu(np.ascontiguousarray(np.repeat(xn, 2, axis=-1)))[..., ::2]      # sample stride 2 -> copied, same result
    yl2, _ = xfm(xs)
    assert torch.equal(yl2, yl)
    xr = cu(np.concatenate([xn, xn], axis=-1))[..., :xn.shape[-1]]          # row stride != length: taken as a view
    yl3, _ = xfm(xr)
    assert torch.equal(yl3, yl)


def test_dwt1d_error_behaviour():
    with pytest.raises(ValueError, match="Unkown pad type"):
        b200wave.DWT1DForward(mode="constant")(cu(np.zeros((1, 1, 16), np.float32)))
    with pytest.raises(AssertionError):
        b200wave.DWT1DForward()(cu(np.zeros((1, 1, 4, 4), np.float32)))
    with pytest.raises(RuntimeError, match="CUDA-only"):
        b200wave.DWT1DForward()(torch.zeros(1, 1, 16))


SWT_CASES = load_swt_cases()


@pytest.mark.parametrize("case", SWT_CASES, ids=[c["id"] for c in SWT_CASES])
def test_golden_swt_level(case):
    """lowlevel.afb2d_atrous (one level of SWTForward) vs the unmodified reference function: output and the input
    gradient autograd derives there (lowlevel.py:475-521)."""
    from b200wave.dwt import lowlevel
    filts = tuple(cu(case[k]) for k in ("h0_col", "h1_col", "h0_row", "h1_row"))
    x = cu(case["x"], grad=True)
    y = lowlevel.afb2d_atrous(x, filts, case["mode"], case["dilation"])
    assert tuple(y.shape) == case["y"].shape and y.is_contiguous()
    assert rel_err(y.detach().cpu(), case["y"]) < RTOL_F32
    (dx,) = torch.autograd.grad(y, x, cu(case["gy"]))
    assert rel_err(dx.cpu(), case["dx"]) < RTOL_F32


@pytest.mark.parametrize("mode", ["zero", "symmetric", "reflect", "periodic"])
def test_oracle_swt_forward_module(mode):
    """SWTForward, J = 3 (dilations 1, 2, 4) on a BASELINE-sized plane against the oracle, and its gradient; J > 1
    feeds the (lo, lo) band of every channel to the next level (the documented intent; the reference cannot run J > 1)."""
    from oracle import swt_oracle
    rng = np.random.default_rng(31)
    xn = rng.standard_normal((2, 2, 304, 304)).astype(np.float32)
    xfm = b200wave.SWTForward(J=3, wave="db2", mode=mode).to(DEV)
    fl = [getattr(xfm, k).flatten().cpu().numpy().astype(np.float64) for k in ("h0_col", "h1_col", "h0_row", "h1_row")]
    x = cu(xn, grad=True)
    coeffs = xfm(x)
    assert len(coeffs) == 3 and all(tuple(c.shape) == (2, 8, 304, 304) for c in coeffs)
    ll = xn.astype(np.float64)
    refs = []
    for j in range(3):
        y = swt_oracle.afb2d_atrous(ll, *fl, mode, 2 ** j)
        refs.append(y)
        assert rel_err(coeffs[j].detach().cpu(), y) < RTOL_F32
        ll = y.reshape(2, 2, 4, 304, 304)[:, :, 0]
    g = [rng.standard_normal(c.shape).astype(np.float32) for c in coeffs]
    (dx,) = torch.autograd.grad(coeffs, x, [cu(t) for t in g])
    d = np.zeros((2, 2, 304, 304))
    for j in range(2, -1, -1):
        gj = g[j].astype(np.float64).reshape(2, 2, 4, 304, 304).copy()
        gj[:, :, 0] += d                      # the next level read this level's (lo, lo) band
        d = swt_oracle.afb2d_atrous_backward(gj.reshape(2, 8, 304, 304), *fl, mode, 2 ** j)
    assert rel_err(dx.cpu(), d) < RTOL_F32


PHASE_CASES = load_phase_cases()
# fp32 FFT: the log-amplitude of weak bins carries the transform's absolute error (~1e-7 * sqrt(H W) * max|F|), and the
# gradient divides by |F|^2 once more -- so the input gradients are compared at 2e-4 of their maximum, the value at 1e-5
PHASE_GRAD_RTOL = 2e-4


@pytest.mark.parametrize("case", PHASE_CASES, ids=[c["id"] for c in PHASE_CASES])
def test_golden_phase_consistency_loss(case):
    """b200wave.phase_consistency_loss vs the reference module's own value and input gradients (model.py:36-58)."""
    x, y = cu(case["x"], grad=True), cu(case["y"], grad=True)
    loss = b200wave.phase_consistency_loss()(x, y)
    assert loss.dim() == 0
    assert abs(loss.item() - case["loss"]) <= RTOL_F32
    loss.backward()
    assert rel_err(x.grad.cpu(), case["dx"]) < PHASE_GRAD_RTOL
    assert rel_err(y.grad.cpu(), case["dy"]) < PHASE_GRAD_RTOL
    if x.shape[0] > 1:      # only the first batch element enters (model.py:52,55)
        assert float(x.grad[1:].abs().max()) == 0.0


def test_phase_consistency_loss_train_size():
    """The crop size of the training step (train.py: 256 x 256 single-channel) against the oracle; upstream gradient
    other than 1; identical images give -1."""
    from oracle import phase_oracle
    rng = np.random.default_rng(9)
    xn = rng.random((4, 1, 256, 256)).astype(np.float32)
    yn = np.clip(xn + 0.1 * rng.standard_normal(xn.shape), 0, 1).astype(np.float32)
    crit = b200wave.phase_consistency_loss()
    x, y = cu(xn, grad=True), cu(yn)
    loss = crit(x, y)
    assert abs(loss.item() - phase_oracle.phase_consistency_loss(xn, yn)) <= RTOL_F32
    (loss * 2.5).backward()
    assert rel_err(x.grad.cpu(), 2.5 * phase_oracle.phase_consistency_grad(xn, yn, 0)) < PHASE_GRAD_RTOL
    assert abs(crit(cu(xn), cu(xn)).item() + 1.0) < 1e-6


def test_tv_loss_full_size_and_scaled_gradient():
    """BASELINE-sized batch against the oracle; an upstream gradient other than 1; non-contiguous input."""
    from b200wave.losses import TVLoss
    rng = np.random.default_rng(2)
    xn = rng.random((64, 1, 304, 304)).astype(np.float32)
    x = cu(xn, grad=True)
    crit = TVLoss()
    loss = crit(x)
    assert abs(loss.item() - tv_oracle.tv_loss(xn)) <= RTOL_F32 * tv_oracle.tv_loss(xn)
    (loss * 3.0).backward()
    assert rel_err(x.grad.cpu(), tv_oracle.tv_loss_backward(xn, 3.0)) < RTOL_F32
    xt = cu(xn[:4]).transpose(2, 3)               # strided view
    ref = tv_oracle.tv_loss(np.ascontiguousarray(xn[:4].transpose(0, 1, 3, 2)))
    assert abs(float(crit(xt)) - ref) <= RTOL_F32 * ref
    a = float(crit(cu(xn[:2])))
    assert a == float(crit(cu(xn[:2])))            # fixed-order reduction: bit-reproducible
