"""CPU: the C-ABI shared library builds for sm_100a, loads without a GPU, exports every symbol that
include/b200wave.h declares, and its host-only entry points / argument validation behave."""
import ctypes
import os
import re
import subprocess

import pytest

import b200wave  # noqa: F401
from b200wave import _build, _cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200wave.h")


@pytest.fixture(scope="module")
def lib():
    return _cabi.load()


def declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200w_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    names = declared_functions()
    assert names == sorted(_cabi.SYMBOLS), (names, sorted(_cabi.SYMBOLS))


def test_library_exports_every_declared_symbol(lib):
    raw = ctypes.CDLL(_cabi.library_path())
    for name in declared_functions():
        assert hasattr(raw, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", _cabi.library_path()], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (b200w_\w+)", out))
    assert exported == set(declared_functions())


def test_library_is_sm100a_only():
    cuobjdump = os.path.join(os.path.dirname(_build.find_nvcc()), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", _cabi.library_path()], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, out


def test_host_only_entry_points(lib):
    assert lib.b200w_abi_version() == _cabi.ABI_VERSION
    assert lib.b200w_dwt_coeff_len(304, 6, 1) == 154
    assert lib.b200w_dwt_coeff_len(127, 6, 2) == 64
    assert lib.b200w_idwt_len(66, 6, 1) == 128 and lib.b200w_idwt_len(64, 6, 2) == 128
    assert lib.b200w_dwt_coeff_len(10, 4, 3) == _cabi.ERR_BAD_MODE      # 'constant' is rejected downstream
    assert lib.b200w_dwt_coeff_len(10, 4, 5) == _cabi.ERR_BAD_MODE      # 'replicate' too
    assert lib.b200w_status_string(_cabi.ERR_BAD_MODE) == b"Unkown pad type"
    assert lib.b200w_ssim_workspace_bytes(2, 3, 400, 400) > 0
    assert lib.b200w_ssim_workspace_bytes(0, 3, 400, 400) == 0


def test_argument_validation_happens_before_any_launch(lib):
    """These calls must return an error code without touching the (absent) GPU."""
    taps, n = _cabi.taps_array([0.5, 0.5])
    bogus = ctypes.c_void_p(256)
    args = (bogus, 64, 8, 1, 8, 8, taps, taps, n, taps, taps, n)
    assert lib.b200w_afb2d_f32(*args, 3, bogus, bogus, None) == _cabi.ERR_BAD_MODE
    assert lib.b200w_afb2d_f32(None, 64, 8, 1, 8, 8, taps, taps, n, taps, taps, n, 0, bogus, bogus, None) \
        == _cabi.ERR_NULL_POINTER
    assert lib.b200w_afb2d_f32(bogus, 64, 8, 1, 8, 8, taps, taps, 0, taps, taps, n, 0, bogus, bogus, None) \
        == _cabi.ERR_BAD_TAPS
    assert lib.b200w_afb2d_f32(bogus, 64, 8, 0, 8, 8, taps, taps, n, taps, taps, n, 0, bogus, bogus, None) \
        == _cabi.ERR_BAD_SHAPE
    t6, n6 = _cabi.taps_array([0.1] * 6)
    # reflect padding needs pad < dimension (torch F.pad rule): 4-sample axis, 6 taps -> pad 4
    assert lib.b200w_afb2d_f32(bogus, 16, 4, 1, 4, 4, t6, t6, n6, t6, t6, n6, 4, bogus, bogus, None) \
        == _cabi.ERR_REFLECT_PAD
    assert lib.b200w_afb2d_f32(bogus, 16, 4, 1, 4, 4, t6, t6, n6, t6, t6, n6, 2, bogus, bogus, None) \
        == _cabi.ERR_PER_TOO_SHORT
    # synthesis: out larger than the natural output
    assert lib.b200w_sfb2d_f32(bogus, 16, 4, None, 1, 4, 4, taps, taps, n, taps, taps, n, 0, bogus, 9, 8, None) \
        == _cabi.ERR_BAD_SHAPE
    w11, nw = _cabi.taps_array([1.0 / 11] * 11)
    w4, nw4 = _cabi.taps_array([0.25] * 4)
    assert lib.b200w_ssim_fwd_f32(bogus, bogus, 1, 1, 8, 8, w4, nw4, 1, 0, None, bogus, bogus, 1024, None) \
        == _cabi.ERR_BAD_WINDOW
    assert lib.b200w_ssim_fwd_f32(bogus, bogus, 1, 1, 8, 8, w11, nw, 1, 0, None, bogus, None, 0, None) \
        == _cabi.ERR_WORKSPACE
    with pytest.raises(ValueError, match="Unkown pad type: constant"):
        _cabi.check(_cabi.ERR_BAD_MODE, "constant")
    with pytest.raises(_cabi.B200WaveError):
        _cabi.check(_cabi.ERR_BAD_SHAPE)


def test_f64_argument_validation_happens_before_any_launch(lib):
    """b200w_afb2d_f64 / b200w_sfb2d_f64: bad arguments come back as status codes without touching the (absent) GPU.
    Unlike the fp32 entry points they check the data pointers before the mode and report null taps as
    ERR_NULL_POINTER; outputs of more than 2^31-1 pixels per plane are ERR_BAD_SHAPE."""
    t2, n2 = _cabi.taps_array_f64([0.5, 0.5])
    t6, n6 = _cabi.taps_array_f64([0.1] * 6)
    t1, n1 = _cabi.taps_array_f64([1.0])
    bogus = ctypes.c_void_p(256)

    def taps(w=(t2, n2), h=(t2, n2)):   # (w_lo, w_hi, Lw, h_lo, h_hi, Lh)
        return (w[0], w[0], w[1], h[0], h[0], h[1])

    def afb(x=bogus, planes=1, H=8, W=8, tp=taps(), mode=0, low=bogus, highs=bogus):
        return lib.b200w_afb2d_f64(x, H * W, W, planes, H, W, *tp, mode, low, highs, None)

    assert afb(x=None, mode=3) == _cabi.ERR_NULL_POINTER                  # pointers before the mode
    assert afb(low=None) == _cabi.ERR_NULL_POINTER
    assert afb(highs=None) == _cabi.ERR_NULL_POINTER
    assert afb(mode=3, planes=0) == _cabi.ERR_BAD_MODE                    # mode before the shape
    assert afb(mode=5) == _cabi.ERR_BAD_MODE
    assert afb(planes=0, tp=taps(w=(None, n2))) == _cabi.ERR_BAD_SHAPE    # shape before the taps
    assert afb(H=0) == _cabi.ERR_BAD_SHAPE
    assert afb(tp=taps(w=(None, 0))) == _cabi.ERR_NULL_POINTER            # null taps before the tap count
    assert afb(tp=(t2, t2, n2, t2, None, n2)) == _cabi.ERR_NULL_POINTER
    assert afb(tp=taps(w=(t2, 0))) == _cabi.ERR_BAD_TAPS
    assert afb(tp=taps(h=(t2, _cabi.MAX_TAPS + 1))) == _cabi.ERR_BAD_TAPS
    # reflect padding needs pad < dimension: 4-sample axis, 6 taps -> pad 4; the taps are checked first
    assert afb(H=4, W=4, tp=taps((t6, n6), (t6, n6)), mode=4) == _cabi.ERR_REFLECT_PAD
    assert afb(H=16, W=4, tp=taps((t6, n6), (t6, n6)), mode=4) == _cabi.ERR_REFLECT_PAD
    assert afb(H=4, W=4, tp=taps((t6, 0), (t6, n6)), mode=4) == _cabi.ERR_BAD_TAPS
    assert afb(H=4, W=4, tp=taps((t6, n6), (t6, n6)), mode=2) == _cabi.ERR_PER_TOO_SHORT
    assert afb(H=4, W=16, tp=taps((t2, n2), (t6, n6)), mode=2) == _cabi.ERR_PER_TOO_SHORT
    assert afb(H=1, W=8, tp=taps(h=(t1, n1))) == _cabi.ERR_BAD_SHAPE        # zero output rows
    assert afb(H=100000, W=100000) == _cabi.ERR_BAD_SHAPE                   # 50000^2 output pixels

    def sfb(low=bogus, planes=1, h=4, w=4, tp=taps(), mode=0, y=bogus, out_h=8, out_w=8):
        return lib.b200w_sfb2d_f64(low, h * w, w, None, planes, h, w, *tp, mode, y, out_h, out_w, None)

    assert sfb(low=None, mode=3) == _cabi.ERR_NULL_POINTER
    assert sfb(y=None) == _cabi.ERR_NULL_POINTER
    assert sfb(mode=3, planes=0) == _cabi.ERR_BAD_MODE
    assert sfb(planes=0, tp=taps(w=(None, n2))) == _cabi.ERR_BAD_SHAPE
    assert sfb(w=0) == _cabi.ERR_BAD_SHAPE
    assert sfb(out_w=0) == _cabi.ERR_BAD_SHAPE
    assert sfb(tp=taps(w=(None, 0))) == _cabi.ERR_NULL_POINTER
    assert sfb(tp=(t2, t2, n2, t2, None, n2)) == _cabi.ERR_NULL_POINTER
    assert sfb(tp=taps(w=(t2, 0))) == _cabi.ERR_BAD_TAPS
    assert sfb(tp=taps(h=(t2, _cabi.MAX_TAPS + 1))) == _cabi.ERR_BAD_TAPS
    assert sfb(h=2, w=2, tp=taps((t6, n6), (t6, n6)), mode=2, out_h=4, out_w=4) == _cabi.ERR_PER_TOO_SHORT
    assert sfb(h=8, w=2, tp=taps((t6, n6), (t6, n6)), mode=2, out_h=4, out_w=4) == _cabi.ERR_PER_TOO_SHORT
    assert sfb(h=2, w=8, tp=taps((t6, 0), (t6, n6)), mode=2, out_h=4, out_w=4) == _cabi.ERR_BAD_TAPS
    assert sfb(h=2, w=2, tp=taps((t6, n6), (t6, n6)), mode=2, out_h=99) == _cabi.ERR_PER_TOO_SHORT
    # synthesis: out larger than the natural output (idwt_len)
    assert sfb(out_h=9) == _cabi.ERR_BAD_SHAPE
    assert sfb(out_w=9, mode=1) == _cabi.ERR_BAD_SHAPE
    assert sfb(out_h=9, mode=2) == _cabi.ERR_BAD_SHAPE
    assert sfb(tp=taps((t6, n6), (t6, n6)), out_h=5, out_w=4) == _cabi.ERR_BAD_SHAPE
    assert sfb(h=50000, w=50000, out_h=100000, out_w=100000) == _cabi.ERR_BAD_SHAPE   # 10^10 output pixels


def test_multilevel_entry_points_validate_before_any_launch(lib):
    """b200w_dwt2_f32 / b200w_idwt2_f32: workspace sizing is host arithmetic and bad arguments come back as status
    codes without touching the (absent) GPU."""
    t6, n6 = _cabi.taps_array([0.1] * 6)
    bogus = ctypes.c_void_p(256)
    # cfg2: 64 planes of 304x304, db3 (6 taps), symmetric, J=3 -> LL scratch of levels 0 and 1 + counters
    ws3 = lib.b200w_dwt2_workspace_bytes(64, 304, 304, 6, 6, 1, 3, None)
    ll0 = 64 * 154 * 156 * 4     # rows padded to a multiple of 4 floats
    ll1 = 64 * 79 * 80 * 4
    assert ws3 >= ll0 + ll1 and ws3 < ll0 + ll1 + 4096
    assert lib.b200w_dwt2_workspace_bytes(64, 304, 304, 6, 6, 1, 1, None) == 0          # J == 1 needs none
    assert lib.b200w_dwt2_workspace_bytes(64, 304, 304, 6, 6, 3, 3, None) == 0          # bad mode
    pads = _cabi.int_array([0, 0, 1, 1, 0, 1])
    assert lib.b200w_dwt2_workspace_bytes(64, 304, 304, 6, 6, 1, 3, pads) > ws3         # zero-extended levels
    highs = _cabi.ptr_array([None, None, None])
    highs[0] = highs[1] = highs[2] = 256
    common = (bogus, 304 * 304, 304, 64, 304, 304, t6, t6, n6, t6, t6, n6)
    assert lib.b200w_dwt2_f32(*common, 1, 3, None, bogus, highs, None, 0, None) == _cabi.ERR_WORKSPACE
    assert lib.b200w_dwt2_f32(*common, 1, 3, None, bogus, highs, bogus, 16, None) == _cabi.ERR_WORKSPACE
    assert lib.b200w_dwt2_f32(*common, 1, 9, None, bogus, highs, bogus, ws3, None) == _cabi.ERR_BAD_SHAPE
    assert lib.b200w_dwt2_f32(*common, 5, 3, None, bogus, highs, bogus, ws3, None) == _cabi.ERR_BAD_MODE
    assert lib.b200w_dwt2_f32(*common, 1, 3, None, None, highs, bogus, ws3, None) == _cabi.ERR_NULL_POINTER
    bad_pads = _cabi.int_array([0, 0, 2, 0, 0, 0])
    assert lib.b200w_dwt2_f32(*common, 1, 3, bad_pads, bogus, highs, bogus, ws3, None) == _cabi.ERR_BAD_SHAPE

    hs, ws = _cabi.int_array([154, 79, 42]), _cabi.int_array([154, 79, 42])
    ohs, ows = _cabi.int_array([304, 154, 80]), _cabi.int_array([304, 154, 80])
    wsi = lib.b200w_idwt2_workspace_bytes(64, 3, ohs, ows)
    assert wsi >= 64 * (154 * 156 + 80 * 80) * 4
    assert lib.b200w_idwt2_workspace_bytes(64, 1, ohs, ows) == 0
    syn = (bogus, 42 * 42, 42, highs, 64, hs, ws, t6, t6, n6, t6, t6, n6)
    assert lib.b200w_idwt2_f32(*syn, 1, 3, ohs, ows, bogus, None, 0, None) == _cabi.ERR_WORKSPACE
    too_big = _cabi.int_array([305, 154, 80])
    assert lib.b200w_idwt2_f32(*syn, 1, 3, too_big, ows, bogus, bogus, wsi, None) == _cabi.ERR_BAD_SHAPE
    small_prev = _cabi.int_array([304, 153, 80])    # level 0 needs a 154-row low-pass, level 1 only yields 153
    assert lib.b200w_idwt2_f32(*syn, 1, 3, small_prev, ows, bogus, bogus, wsi, None) == _cabi.ERR_BAD_SHAPE
    assert lib.b200w_idwt2_f32(*syn, 1, 3, ohs, ows, None, bogus, wsi, None) == _cabi.ERR_NULL_POINTER
