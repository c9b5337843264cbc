"""``torch.library`` custom ops ``b200wave::*`` -- the thin layer between the
Python modules and the C ABI.

Each op takes device tensors plus host scalars / tap lists, allocates its
outputs with torch (the library never allocates) and launches on torch's
current stream, so the ops are asynchronous and CUDA-graph capturable.
CUDA-only: there is deliberately no CPU implementation.

Autograd follows the reference's hand-written backward passes, not the
mathematical adjoint (SURVEY.md 8a-Q1):

* ``afb2d`` backward  = ``sfb2d`` with the same (reversed) analysis taps, cropped
  to the input size                       (pw/dwt/lowlevel.py:349-365)
* ``sfb2d`` backward  = ``afb2d`` of ``dy`` with the synthesis taps as
  correlation kernels                     (pw/dwt/lowlevel.py:682-694)
* ``ssim_fwd`` backward = ``ssim_bwd`` (closed form of autograd through ssim.py:17-37)
"""
import ctypes

import torch
from torch.autograd.function import once_differentiable

from . import _cabi

_LIB = torch.library.Library("b200wave", "DEF")

_LIB.define("afb2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode) -> (Tensor, Tensor)")
_LIB.define("afb2d_select(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, bool want_low, "
            "bool want_highs, float hi_scale, float hi_shift) -> (Tensor, Tensor)")
_LIB.define("sfb2d(Tensor low, Tensor? highs, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
            "int out_h, int out_w) -> Tensor")
_LIB.define("dwt2(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, int J, int[] pad_hw) "
            "-> Tensor[]")
_LIB.define("idwt2(Tensor yl, Tensor?[] yh, int[] hw, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
            "int[] out_hw) -> Tensor")
_LIB.define("afb1d(Tensor x, float[] h0, float[] h1, int mode) -> (Tensor, Tensor)")
_LIB.define("sfb1d(Tensor low, Tensor? high, float[] g0, float[] g1, int mode, int out_len) -> Tensor")
_LIB.define("swt2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, int dilation) -> Tensor")
_LIB.define("swt2d_adjoint(Tensor dy, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, int dilation) "
            "-> Tensor")
_LIB.define("iswt2d(Tensor ll, Tensor y, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int dilation) -> Tensor")
_LIB.define("ssim_fwd(Tensor img1, Tensor img2, float[] win, bool size_average, int n_maps) -> (Tensor, Tensor)")
_LIB.define("ssim_bwd(Tensor img1, Tensor img2, Tensor maps, Tensor grad_out, float[] win, bool size_average, "
            "bool need_d2) -> (Tensor, Tensor)")

MAX_LEVELS = _cabi.MAX_LEVELS

_INT_TO_MODE = {0: "zero", 1: "symmetric", 2: "periodization", 3: "constant", 4: "reflect", 5: "replicate",
                6: "periodic"}


def _mode_name(mode):
    return _INT_TO_MODE.get(int(mode), mode)


def coeff_len(n, l, mode):
    """pywt.dwt_coeff_len as used at pw/dwt/lowlevel.py:153 (host arithmetic only)."""
    return (n + 1) // 2 if mode == 2 else (n + l - 1) // 2


def idwt_len(m, l, mode):
    return 2 * m if mode == 2 else 2 * m - l + 2


def _check_mode(mode):
    if mode not in (0, 1, 2, 4, 6):
        raise ValueError("Unkown pad type: {}".format(_mode_name(mode)))


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_cuda_f32(t, name):
    if not t.is_cuda:
        raise RuntimeError("b200wave::%s is CUDA-only (sm_100a); there is no CPU fallback -- got a %s tensor"
                           % (name, t.device))
    if t.dtype != torch.float32:
        raise RuntimeError("b200wave::%s: expected scalar type Float but found %s" % (name, t.dtype))


def _planes_view(t):
    """(N,C,H,W) tensor -> (tensor to keep alive, plane_stride, row_stride); copies only when the
    layout cannot be expressed as planes with unit column stride."""
    n, c, h, w = t.shape
    sn, sc, sh, sw = t.stride()
    ok = (sw == 1 or w == 1) and (n == 1 or c == 1 or sn == c * sc)
    if not ok:
        t = t.contiguous()
        sn, sc, sh, sw = t.stride()
    plane_stride = sc if c > 1 else (sn if n > 1 else h * sh)
    return t, plane_stride, sh


# ------------------------------------------------------------------------------------------- afb2d
def _afb2d_cuda(x, w_lo, w_hi, h_lo, h_hi, mode):
    _check_mode(mode)
    _require_cuda_f32(x, "afb2d")
    if x.dim() != 4:
        raise IndexError("b200wave::afb2d expects a 4-D (N, C, H, W) tensor, got %d-D" % x.dim())
    lib = _cabi.load()
    N, C, H, W = x.shape
    Lw, Lh = len(w_lo), len(h_lo)
    if len(w_hi) != Lw or len(h_hi) != Lh:
        raise RuntimeError("low- and high-pass filters must have the same length along an axis")
    Ho, Wo = coeff_len(H, Lh, mode), coeff_len(W, Lw, mode)
    low = torch.empty((N, C, Ho, Wo), device=x.device, dtype=torch.float32)
    highs = torch.empty((N, C, 3, Ho, Wo), device=x.device, dtype=torch.float32)
    if low.numel() == 0:
        return low, highs
    xk, ps, rs = _planes_view(x)
    a_wl, _ = _cabi.taps_array(w_lo)
    a_wh, _ = _cabi.taps_array(w_hi)
    a_hl, _ = _cabi.taps_array(h_lo)
    a_hh, _ = _cabi.taps_array(h_hi)
    with torch.cuda.device(x.device):
        rc = lib.b200w_afb2d_f32(xk.data_ptr(), ps, rs, N * C, H, W, a_wl, a_wh, Lw, a_hl, a_hh, Lh, int(mode),
                                 low.data_ptr(), highs.data_ptr(), _stream())
    _cabi.check(rc, _mode_name(mode))
    return low, highs


def _afb2d_fake(x, w_lo, w_hi, h_lo, h_hi, mode):
    N, C, H, W = x.shape
    Ho, Wo = coeff_len(H, len(h_lo), mode), coeff_len(W, len(w_lo), mode)
    return x.new_empty((N, C, Ho, Wo)), x.new_empty((N, C, 3, Ho, Wo))


# ------------------------------------------------------------------------------------------- afb2d_select
def _afb2d_select_cuda(x, w_lo, w_hi, h_lo, h_hi, mode, want_low, want_highs, hi_scale, hi_shift):
    """One analysis level that writes only the sub-bands asked for, the detail bands as hi_scale*v + hi_shift
    (FS_Discriminator.filter_wavelet, model.py:166-179): an output that is not wanted comes back with 0 elements
    and costs no HBM traffic."""
    _check_mode(mode)
    _require_cuda_f32(x, "afb2d_select")
    if x.dim() != 4:
        raise IndexError("b200wave::afb2d_select expects a 4-D (N, C, H, W) tensor, got %d-D" % x.dim())
    if not (want_low or want_highs):
        raise ValueError("afb2d_select: at least one of the low-pass / detail outputs must be requested")
    lib = _cabi.load()
    N, C, H, W = x.shape
    Lw, Lh = len(w_lo), len(h_lo)
    if len(w_hi) != Lw or len(h_hi) != Lh:
        raise RuntimeError("low- and high-pass filters must have the same length along an axis")
    Ho, Wo = coeff_len(H, Lh, mode), coeff_len(W, Lw, mode)
    low = torch.empty((N, C, Ho, Wo) if want_low else (0,), device=x.device, dtype=torch.float32)
    highs = torch.empty((N, C, 3, Ho, Wo) if want_highs else (0,), device=x.device, dtype=torch.float32)
    if N * C * Ho * Wo == 0:
        return low, highs
    xk, ps, rs = _planes_view(x)
    a_wl, _ = _cabi.taps_array(w_lo)
    a_wh, _ = _cabi.taps_array(w_hi)
    a_hl, _ = _cabi.taps_array(h_lo)
    a_hh, _ = _cabi.taps_array(h_hi)
    with torch.cuda.device(x.device):
        rc = lib.b200w_afb2d_ex_f32(xk.data_ptr(), ps, rs, N * C, H, W, a_wl, a_wh, Lw, a_hl, a_hh, Lh, int(mode),
                                    low.data_ptr() if want_low else None, highs.data_ptr() if want_highs else None,
                                    float(hi_scale), float(hi_shift), _stream())
    _cabi.check(rc, _mode_name(mode))
    return low, highs


def _afb2d_select_fake(x, w_lo, w_hi, h_lo, h_hi, mode, want_low, want_highs, hi_scale, hi_shift):
    N, C, H, W = x.shape
    Ho, Wo = coeff_len(H, len(h_lo), mode), coeff_len(W, len(w_lo), mode)
    return (x.new_empty((N, C, Ho, Wo) if want_low else (0,)),
            x.new_empty((N, C, 3, Ho, Wo) if want_highs else (0,)))


def _afb2d_select_setup(ctx, inputs, output):
    x, w_lo, w_hi, h_lo, h_hi, mode, want_low, want_highs, hi_scale, _ = inputs
    ctx.taps = (w_lo, w_hi, h_lo, h_hi)
    ctx.mode = mode
    ctx.in_shape = tuple(x.shape)
    ctx.want = (want_low, want_highs)
    ctx.hi_scale = hi_scale
    ctx.set_materialize_grads(False)


def _afb2d_select_backward(ctx, dlow, dhighs):
    none = (None,) * 10
    if not ctx.needs_input_grad[0]:
        return none
    want_low, want_highs = ctx.want
    dlow = dlow if want_low else None
    dhighs = dhighs if want_highs else None
    if dlow is None and dhighs is None:
        return none
    N, C, H, W = ctx.in_shape
    w_lo, w_hi, h_lo, h_hi = ctx.taps
    if dlow is None:
        dlow = dhighs.new_zeros((N, C) + tuple(dhighs.shape[-2:]))
    if dhighs is not None and ctx.hi_scale != 1.0:
        dhighs = dhighs * ctx.hi_scale   # d(hi_scale * v + hi_shift) / dv
    # same pseudo-adjoint as AFB2D.backward (lowlevel.py:356-364); a missing detail gradient is never materialised
    dx = torch.ops.b200wave.sfb2d(dlow, dhighs, w_lo, w_hi, h_lo, h_hi, ctx.mode, H, W)
    return (dx,) + none[1:]


# ------------------------------------------------------------------------------------------- sfb2d
def _sfb2d_cuda(low, highs, w_lo, w_hi, h_lo, h_hi, mode, out_h, out_w):
    _check_mode(mode)
    _require_cuda_f32(low, "sfb2d")
    if low.dim() != 4:
        raise IndexError("b200wave::sfb2d expects a 4-D (N, C, h, w) lowpass tensor, got %d-D" % low.dim())
    lib = _cabi.load()
    N, C, h, w = low.shape
    Lw, Lh = len(w_lo), len(h_lo)
    if len(w_hi) != Lw or len(h_hi) != Lh:
        raise RuntimeError("low- and high-pass filters must have the same length along an axis")
    if highs is not None:
        _require_cuda_f32(highs, "sfb2d")
        if tuple(highs.shape) != (N, C, 3, h, w):
            raise RuntimeError("b200wave::sfb2d: highs must have shape %s, got %s"
                               % ((N, C, 3, h, w), tuple(highs.shape)))
        highs = highs.contiguous()
    full_h, full_w = idwt_len(h, Lh, mode), idwt_len(w, Lw, mode)
    oh = full_h if out_h < 0 else out_h
    ow = full_w if out_w < 0 else out_w
    y = torch.empty((N, C, oh, ow), device=low.device, dtype=torch.float32)
    if y.numel() == 0:
        return y
    lk, ps, rs = _planes_view(low)
    a_wl, _ = _cabi.taps_array(w_lo)
    a_wh, _ = _cabi.taps_array(w_hi)
    a_hl, _ = _cabi.taps_array(h_lo)
    a_hh, _ = _cabi.taps_array(h_hi)
    with torch.cuda.device(low.device):
        rc = lib.b200w_sfb2d_f32(lk.data_ptr(), ps, rs, None if highs is None else highs.data_ptr(), N * C, h, w,
                                 a_wl, a_wh, Lw, a_hl, a_hh, Lh, int(mode), y.data_ptr(), oh, ow, _stream())
    _cabi.check(rc, _mode_name(mode))
    return y


def _sfb2d_fake(low, highs, w_lo, w_hi, h_lo, h_hi, mode, out_h, out_w):
    N, C, h, w = low.shape
    oh = idwt_len(h, len(h_lo), mode) if out_h < 0 else out_h
    ow = idwt_len(w, len(w_lo), mode) if out_w < 0 else out_w
    return low.new_empty((N, C, oh, ow))


# ------------------------------------------------------------------------------------------- multi-level chains
def dwt2_level_dims(H, W, Lh, Lw, mode, J, pad_hw=()):
    """Output (Ho, Wo) of every level of the analysis chain (host arithmetic)."""
    dims = []
    h, w = H, W
    for j in range(J):
        ph, pw = (pad_hw[2 * j], pad_hw[2 * j + 1]) if (pad_hw and j > 0) else (0, 0)
        h, w = coeff_len(h + ph, Lh, mode), coeff_len(w + pw, Lw, mode)
        dims.append((h, w))
    return dims


def _dwt2_cuda(x, w_lo, w_hi, h_lo, h_hi, mode, J, pad_hw):
    """J analysis levels in one launch; returns [yl, yh_0 (finest), ..., yh_{J-1}]."""
    _check_mode(mode)
    _require_cuda_f32(x, "dwt2")
    if x.dim() != 4:
        raise IndexError("b200wave::dwt2 expects a 4-D (N, C, H, W) tensor, got %d-D" % x.dim())
    if not 1 <= J <= _cabi.MAX_LEVELS:
        raise RuntimeError("b200wave::dwt2 supports 1..%d levels per call, got %d" % (_cabi.MAX_LEVELS, J))
    if pad_hw and len(pad_hw) != 2 * J:
        raise RuntimeError("pad_hw must hold 2*J entries")
    lib = _cabi.load()
    N, C, H, W = x.shape
    Lw, Lh = len(w_lo), len(h_lo)
    if len(w_hi) != Lw or len(h_hi) != Lh:
        raise RuntimeError("low- and high-pass filters must have the same length along an axis")
    dims = dwt2_level_dims(H, W, Lh, Lw, mode, J, pad_hw)
    yl = torch.empty((N, C) + dims[-1], device=x.device, dtype=torch.float32)
    highs = [torch.empty((N, C, 3, h, w), device=x.device, dtype=torch.float32) for h, w in dims]
    if x.numel() == 0 or N * C == 0:
        return [yl] + highs
    xk, ps, rs = _planes_view(x)
    pads = _cabi.int_array(pad_hw) if pad_hw else None
    # the intermediate low-pass images and the per-plane completion counters live in the workspace
    ws_bytes = lib.b200w_dwt2_workspace_bytes(N * C, H, W, Lw, Lh, int(mode), int(J), pads)
    work = torch.empty((max(ws_bytes, 4),), device=x.device, dtype=torch.uint8)
    a_wl, _ = _cabi.taps_array(w_lo)
    a_wh, _ = _cabi.taps_array(w_hi)
    a_hl, _ = _cabi.taps_array(h_lo)
    a_hh, _ = _cabi.taps_array(h_hi)
    with torch.cuda.device(x.device):
        rc = lib.b200w_dwt2_f32(xk.data_ptr(), ps, rs, N * C, H, W, a_wl, a_wh, Lw, a_hl, a_hh, Lh, int(mode), int(J),
                                pads, yl.data_ptr(), _cabi.ptr_array(highs), work.data_ptr(), ws_bytes, _stream())
    _cabi.check(rc, _mode_name(mode))
    return [yl] + highs


def _dwt2_fake(x, w_lo, w_hi, h_lo, h_hi, mode, J, pad_hw):
    N, C, H, W = x.shape
    dims = dwt2_level_dims(H, W, len(h_lo), len(w_lo), mode, J, pad_hw)
    return [x.new_empty((N, C) + dims[-1])] + [x.new_empty((N, C, 3) + d) for d in dims]


def _idwt2_cuda(yl, yh, hw, w_lo, w_hi, h_lo, h_hi, mode, out_hw):
    """J synthesis levels in one launch.  hw = 2*J ints (h_j, w_j): sub-band size of level j (yh index, finest
    first); out_hw = 2*J ints (per-level output size, a crop of the natural one) or [] for the natural sizes."""
    _check_mode(mode)
    _require_cuda_f32(yl, "idwt2")
    if yl.dim() != 4:
        raise IndexError("b200wave::idwt2 expects a 4-D (N, C, h, w) lowpass tensor, got %d-D" % yl.dim())
    J = len(yh)
    if not 1 <= J <= _cabi.MAX_LEVELS:
        raise RuntimeError("b200wave::idwt2 supports 1..%d levels per call, got %d" % (_cabi.MAX_LEVELS, J))
    if len(hw) != 2 * J or (out_hw and len(out_hw) != 2 * J):
        raise RuntimeError("hw / out_hw must hold 2*J entries")
    lib = _cabi.load()
    N, C = yl.shape[:2]
    Lw, Lh = len(w_lo), len(h_lo)
    if len(w_hi) != Lw or len(h_hi) != Lh:
        raise RuntimeError("low- and high-pass filters must have the same length along an axis")
    hs, ws = list(hw[0::2]), list(hw[1::2])
    if yl.shape[-2] < hs[-1] or yl.shape[-1] < ws[-1]:
        raise RuntimeError("b200wave::idwt2: yl %s is smaller than the coarsest sub-bands (%d, %d)"
                           % (tuple(yl.shape), hs[-1], ws[-1]))
    kept = []
    for j, h in enumerate(yh):
        if h is not None:
            _require_cuda_f32(h, "idwt2")
            if tuple(h.shape) != (N, C, 3, hs[j], ws[j]):
                raise RuntimeError("b200wave::idwt2: yh[%d] must have shape %s, got %s"
                                   % (j, (N, C, 3, hs[j], ws[j]), tuple(h.shape)))
            h = h.contiguous()
        kept.append(h)
    if out_hw:
        ohs, ows = list(out_hw[0::2]), list(out_hw[1::2])
    else:
        ohs = [idwt_len(h, Lh, mode) for h in hs]
        ows = [idwt_len(w, Lw, mode) for w in ws]
    y = torch.empty((N, C, ohs[0], ows[0]), device=yl.device, dtype=torch.float32)
    if y.numel() == 0:
        return y
    lk, ps, rs = _planes_view(yl)
    a_oh, a_ow = _cabi.int_array(ohs), _cabi.int_array(ows)
    ws_bytes = lib.b200w_idwt2_workspace_bytes(N * C, J, a_oh, a_ow)
    work = torch.empty((max(ws_bytes, 4),), device=yl.device, dtype=torch.uint8)
    a_wl, _ = _cabi.taps_array(w_lo)
    a_wh, _ = _cabi.taps_array(w_hi)
    a_hl, _ = _cabi.taps_array(h_lo)
    a_hh, _ = _cabi.taps_array(h_hi)
    with torch.cuda.device(yl.device):
        rc = lib.b200w_idwt2_f32(lk.data_ptr(), ps, rs, _cabi.ptr_array(kept), N * C, _cabi.int_array(hs),
                                 _cabi.int_array(ws), a_wl, a_wh, Lw, a_hl, a_hh, Lh, int(mode), J,
                                 a_oh, a_ow, y.data_ptr(), work.data_ptr(), ws_bytes, _stream())
    _cabi.check(rc, _mode_name(mode))
    return y


def _idwt2_fake(yl, yh, hw, w_lo, w_hi, h_lo, h_hi, mode, out_hw):
    N, C = yl.shape[:2]
    if out_hw:
        return yl.new_empty((N, C, out_hw[0], out_hw[1]))
    return yl.new_empty((N, C, idwt_len(hw[0], len(h_lo), mode), idwt_len(hw[1], len(w_lo), mode)))


class DWT2Function(torch.autograd.Function):
    """All J analysis levels of ``DWTForward`` as one autograd node / one launch.  Backward = the chain of the
    reference's ``AFB2D.backward`` (pw/dwt/lowlevel.py:349-365): synthesis with the same (reversed) analysis taps,
    every level cropped to the size of the corresponding forward input -- again one launch."""

    @staticmethod
    def forward(ctx, x, w_lo, w_hi, h_lo, h_hi, mode, J):
        outs = torch.ops.b200wave.dwt2(x, w_lo, w_hi, h_lo, h_hi, mode, J, [])
        ctx.taps = (w_lo, w_hi, h_lo, h_hi)
        ctx.mode = mode
        ctx.J = J
        # AFB2D saves only shapes, never x (lowlevel.py:337-338)
        ctx.in_hw = [tuple(x.shape[-2:])] + [tuple(h.shape[-2:]) for h in outs[1:J]]
        ctx.sub_hw = [tuple(h.shape[-2:]) for h in outs[1:]]
        ctx.nc = tuple(x.shape[:2])
        ctx.set_materialize_grads(False)
        return tuple(outs)

    @staticmethod
    @once_differentiable   # the backward kernels have no autograd formula of their own: double backward raises
    def backward(ctx, gyl, *gyh):
        if not ctx.needs_input_grad[0] or (gyl is None and all(g is None for g in gyh)):
            return (None,) * 7
        J = ctx.J
        if gyl is None:
            ref = next(g for g in gyh if g is not None)
            gyl = ref.new_zeros(ctx.nc + ctx.sub_hw[-1])
        w_lo, w_hi, h_lo, h_hi = ctx.taps
        hw = [v for d in ctx.sub_hw for v in d]
        out_hw = [v for d in ctx.in_hw for v in d]
        dx = torch.ops.b200wave.idwt2(gyl, list(gyh), hw, w_lo, w_hi, h_lo, h_hi, ctx.mode, out_hw)
        return (dx,) + (None,) * 6


class IDWT2Function(torch.autograd.Function):
    """All J synthesis levels of ``DWTInverse`` (incl. the 'unpad' crops, transform2d.py:141-145) as one node / one
    launch.  Backward = the chain of the reference's ``SFB2D.backward`` (lowlevel.py:682-694): analysis of dy with
    the un-reversed synthesis taps as correlators; where the forward cropped ll, autograd hands SFB2D.backward the
    gradient padded with a zero row / column -- reproduced by the kernel's zero extension."""

    @staticmethod
    def forward(ctx, w_lo, w_hi, h_lo, h_hi, mode, yl, *yh):
        J = len(yh)
        Lw, Lh = len(w_lo), len(h_lo)
        # sub-band size per level: a None entry means "zeros of the current ll size" (transform2d.py:137-139)
        hw = [None] * J
        pads = [0] * (2 * J)   # zero extension of the backward chain's level inputs
        cur = tuple(yl.shape[-2:])
        for j in range(J - 1, -1, -1):
            if yh[j] is None:
                hw[j] = cur
            else:
                hw[j] = tuple(yh[j].shape[-2:])
                if hw[j][0] > cur[0] or hw[j][1] > cur[1]:
                    raise RuntimeError("DWTInverse: yh[%d] %s is larger than the lowpass it is combined with %s"
                                       % (j, hw[j], cur))
            if j < J - 1:   # ll came out of level j+1 with size `cur`; the forward used its top-left hw[j] block
                pads[2 * (j + 1)], pads[2 * (j + 1) + 1] = cur[0] - hw[j][0], cur[1] - hw[j][1]
            cur = (idwt_len(hw[j][0], Lh, mode), idwt_len(hw[j][1], Lw, mode))
        flat_hw = [v for d in hw for v in d]
        y = torch.ops.b200wave.idwt2(yl, list(yh), flat_hw, w_lo, w_hi, h_lo, h_hi, mode, [])
        ctx.taps = (w_lo, w_hi, h_lo, h_hi)
        ctx.mode = mode
        ctx.J = J
        ctx.pads = pads
        ctx.yl_hw = tuple(yl.shape[-2:])
        ctx.coarse_hw = hw[J - 1]
        ctx.present = [h is not None for h in yh]
        return y

    @staticmethod
    @once_differentiable   # the backward kernels have no autograd formula of their own: double backward raises
    def backward(ctx, dy):
        J = ctx.J
        need_l = ctx.needs_input_grad[5]
        need_h = [ctx.present[j] and ctx.needs_input_grad[6 + j] for j in range(J)]
        if dy is None or not (need_l or any(need_h)):
            return (None,) * (6 + J)
        if max(ctx.pads) > 1:
            raise RuntimeError("DWTInverse backward: lowpass more than one sample larger than its sub-bands")
        w_lo, w_hi, h_lo, h_hi = ctx.taps
        pads = ctx.pads if any(ctx.pads) else []
        outs = torch.ops.b200wave.dwt2(dy, w_lo, w_hi, h_lo, h_hi, ctx.mode, J, pads)
        dyl = outs[0] if need_l else None
        if dyl is not None and tuple(dyl.shape[-2:]) != ctx.yl_hw:   # yl itself was cropped by the forward
            dyl = torch.nn.functional.pad(dyl, (0, ctx.yl_hw[1] - dyl.shape[-1], 0, ctx.yl_hw[0] - dyl.shape[-2]))
        dyh = [outs[1 + j] if need_h[j] else None for j in range(J)]
        return (None,) * 5 + (dyl,) + tuple(dyh)


# ------------------------------------------------------------------------------------------- autograd (DWT)
def _afb2d_setup(ctx, inputs, output):
    x, w_lo, w_hi, h_lo, h_hi, mode = inputs
    ctx.taps = (w_lo, w_hi, h_lo, h_hi)
    ctx.mode = mode
    ctx.in_hw = (x.shape[-2], x.shape[-1])   # AFB2D saves only the shape, not x (lowlevel.py:337-338)
    ctx.set_materialize_grads(False)


def _afb2d_backward(ctx, dlow, dhighs):
    dx = None
    if ctx.needs_input_grad[0]:
        if dlow is None and dhighs is None:
            return None, None, None, None, None, None
        if dlow is None:
            n, c, _, h, w = dhighs.shape
            dlow = dhighs.new_zeros((n, c, h, w))
        w_lo, w_hi, h_lo, h_hi = ctx.taps
        H, W = ctx.in_hw
        # synthesis with the saved analysis taps, cropped to the forward input (lowlevel.py:356-364)
        dx = torch.ops.b200wave.sfb2d(dlow, dhighs, w_lo, w_hi, h_lo, h_hi, ctx.mode, H, W)
    return dx, None, None, None, None, None


def _sfb2d_setup(ctx, inputs, output):
    low, highs, w_lo, w_hi, h_lo, h_hi, mode, out_h, out_w = inputs
    ctx.taps = (w_lo, w_hi, h_lo, h_hi)
    ctx.mode = mode
    ctx.has_highs = highs is not None
    ctx.cropped = tuple(output.shape[-2:]) != (idwt_len(low.shape[-2], len(h_lo), mode),
                                               idwt_len(low.shape[-1], len(w_lo), mode))


def _sfb2d_backward(ctx, dy):
    dlow = dhighs = None
    need_low = ctx.needs_input_grad[0]
    need_high = ctx.has_highs and ctx.needs_input_grad[1]
    if need_low or need_high:
        if ctx.cropped:
            raise RuntimeError("b200wave::sfb2d: backward through a cropped synthesis is not defined "
                               "(the crop only exists inside AFB2D.backward)")
        w_lo, w_hi, h_lo, h_hi = ctx.taps
        # analysis of dy with the un-reversed synthesis taps as correlators (lowlevel.py:687-693)
        dlow, dhighs = torch.ops.b200wave.afb2d(dy, w_lo, w_hi, h_lo, h_hi, ctx.mode)
        if not need_low:
            dlow = None
        if not need_high:
            dhighs = None
    return dlow, dhighs, None, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------- 1-D banks
def _rows_view(t):
    """(N, C, L) tensor -> (tensor to keep alive, row stride): rows must be equally spaced with unit sample stride."""
    n, c, l = t.shape
    sn, sc, sl = t.stride()
    ok = (sl == 1 or l == 1) and (n == 1 or c == 1 or sn == c * sc)
    if not ok:
        t = t.contiguous()
        sn, sc, sl = t.stride()
    return t, (sc if c > 1 else (sn if n > 1 else l))


def _afb1d_cuda(x, h0, h1, mode):
    _check_mode(mode)
    _require_cuda_f32(x, "afb1d")
    if x.dim() != 3:
        raise IndexError("b200wave::afb1d expects a 3-D (N, C, L) tensor, got %d-D" % x.dim())
    if len(h0) != len(h1):
        raise RuntimeError("low- and high-pass filters must have the same length")
    lib = _cabi.load()
    N, C, n = x.shape
    m = coeff_len(n, len(h0), mode)
    lo = torch.empty((N, C, m), device=x.device, dtype=torch.float32)
    hi = torch.empty((N, C, m), device=x.device, dtype=torch.float32)
    if lo.numel() == 0:
        return lo, hi
    xk, rs = _rows_view(x)
    a0, _ = _cabi.taps_array(h0)
    a1, _ = _cabi.taps_array(h1)
    with torch.cuda.device(x.device):
        rc = lib.b200w_afb1d_f32(xk.data_ptr(), rs, N * C, n, a0, a1, len(h0), int(mode), lo.data_ptr(), hi.data_ptr(),
                                 _stream())
    _cabi.check(rc, _mode_name(mode))
    return lo, hi


def _afb1d_fake(x, h0, h1, mode):
    N, C, n = x.shape
    m = coeff_len(n, len(h0), mode)
    return x.new_empty((N, C, m)), x.new_empty((N, C, m))


def _sfb1d_cuda(low, high, g0, g1, mode, out_len):
    _check_mode(mode)
    _require_cuda_f32(low, "sfb1d")
    if low.dim() != 3:
        raise IndexError("b200wave::sfb1d expects 3-D (N, C, L) tensors, got %d-D" % low.dim())
    if high is not None:
        _require_cuda_f32(high, "sfb1d")
        if high.shape != low.shape:
            raise RuntimeError("b200wave::sfb1d: low %s and high %s must have the same shape"
                               % (tuple(low.shape), tuple(high.shape)))
    lib = _cabi.load()
    N, C, m = low.shape
    full = idwt_len(m, len(g0), mode)
    n = full if out_len < 0 else out_len
    y = torch.empty((N, C, n), device=low.device, dtype=torch.float32)
    if y.numel() == 0:
        return y
    lk, rs = _rows_view(low)
    hk = None if high is None else high.contiguous()
    a0, _ = _cabi.taps_array(g0)
    a1, _ = _cabi.taps_array(g1)
    with torch.cuda.device(low.device):
        rc = lib.b200w_sfb1d_f32(lk.data_ptr(), rs, None if hk is None else hk.data_ptr(), N * C, m, a0, a1, len(g0),
                                 int(mode), n, y.data_ptr(), _stream())
    _cabi.check(rc, _mode_name(mode))
    return y


def _sfb1d_fake(low, high, g0, g1, mode, out_len):
    N, C, m = low.shape
    return low.new_empty((N, C, idwt_len(m, len(g0), mode) if out_len < 0 else out_len))


def _afb1d_setup(ctx, inputs, output):
    x, h0, h1, mode = inputs
    ctx.taps = (h0, h1)
    ctx.mode = mode
    ctx.n = x.shape[-1]                      # AFB1D saves only the length (lowlevel.py:398)
    ctx.set_materialize_grads(False)


def _afb1d_backward(ctx, dlo, dhi):
    dx = None
    if ctx.needs_input_grad[0]:
        if dlo is None and dhi is None:
            return None, None, None, None
        if dlo is None:
            dlo = torch.zeros_like(dhi)
        # synthesis with the saved analysis taps, cropped to the forward input (lowlevel.py:417-422)
        dx = torch.ops.b200wave.sfb1d(dlo, dhi, ctx.taps[0], ctx.taps[1], ctx.mode, ctx.n)
    return dx, None, None, None


def _sfb1d_setup(ctx, inputs, output):
    low, high, g0, g1, mode, out_len = inputs
    ctx.taps = (g0, g1)
    ctx.mode = mode
    ctx.has_high = high is not None
    ctx.cropped = output.shape[-1] != idwt_len(low.shape[-1], len(g0), mode)


def _sfb1d_backward(ctx, dy):
    dlo = dhi = None
    need_lo = ctx.needs_input_grad[0]
    need_hi = ctx.has_high and ctx.needs_input_grad[1]
    if need_lo or need_hi:
        if ctx.cropped:
            raise RuntimeError("b200wave::sfb1d: backward through a cropped synthesis is not defined "
                               "(the crop only exists inside AFB1D.backward)")
        # analysis of dy with the un-reversed synthesis taps as correlators (lowlevel.py:736-742)
        dlo, dhi = torch.ops.b200wave.afb1d(dy, ctx.taps[0], ctx.taps[1], ctx.mode)
        if not need_lo:
            dlo = None
        if not need_hi:
            dhi = None
    return dlo, dhi, None, None, None, None


# ------------------------------------------------------------------------------------------- a trous (SWT)
def _check_swt_mode(mode):
    if mode not in (0, 1, 4, 6):     # mypad: zero, symmetric, reflect, periodic (lowlevel.py:28-88)
        raise ValueError("Unkown pad type: {}".format(_mode_name(mode)))


def _swt_call(fn_name, t, w_lo, w_hi, h_lo, h_hi, mode, dilation, planes, H, W, out):
    lib = _cabi.load()
    if not (len(w_lo) == len(w_hi) == len(h_lo) == len(h_hi)):
        raise RuntimeError("b200wave::swt2d: all four filters must have the same length")
    a_wl, _ = _cabi.taps_array(w_lo)
    a_wh, _ = _cabi.taps_array(w_hi)
    a_hl, _ = _cabi.taps_array(h_lo)
    a_hh, _ = _cabi.taps_array(h_hi)
    with torch.cuda.device(t.device):
        rc = getattr(lib, fn_name)(t.data_ptr(), planes, H, W, a_wl, a_wh, a_hl, a_hh, len(w_lo), int(dilation),
                                   int(mode), out.data_ptr(), _stream())
    _cabi.check(rc, _mode_name(mode))


def _swt2d_cuda(x, w_lo, w_hi, h_lo, h_hi, mode, dilation):
    _check_swt_mode(mode)
    _require_cuda_f32(x, "swt2d")
    if x.dim() != 4:
        raise IndexError("b200wave::swt2d expects a 4-D (N, C, H, W) tensor, got %d-D" % x.dim())
    N, C, H, W = x.shape
    y = torch.empty((N, 4 * C, H, W), device=x.device, dtype=torch.float32)
    if y.numel():
        _swt_call("b200w_swt2d_fwd_f32", x.contiguous(), w_lo, w_hi, h_lo, h_hi, mode, dilation, N * C, H, W, y)
    return y


def _swt2d_adjoint_cuda(dy, w_lo, w_hi, h_lo, h_hi, mode, dilation):
    _check_swt_mode(mode)
    _require_cuda_f32(dy, "swt2d_adjoint")
    N, C4, H, W = dy.shape
    dx = torch.empty((N, C4 // 4, H, W), device=dy.device, dtype=torch.float32)
    if dx.numel():
        _swt_call("b200w_swt2d_bwd_f32", dy.contiguous(), w_lo, w_hi, h_lo, h_hi, mode, dilation, N * (C4 // 4), H, W, dx)
    return dx


def _swt2d_setup(ctx, inputs, output):
    x, w_lo, w_hi, h_lo, h_hi, mode, dilation = inputs
    ctx.args = (w_lo, w_hi, h_lo, h_hi, mode, dilation)


def _swt2d_backward(ctx, dy):
    dx = None
    if ctx.needs_input_grad[0]:
        dx = torch.ops.b200wave.swt2d_adjoint(dy, *ctx.args)
    return dx, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------- inverse SWT
PERIODIC = 6


def iswt_layout(ll, y, name):
    """Checks the shapes of one inverse-SWT level and returns (ll as (tensor, plane stride), dense y); copies only what
    the kernel cannot read in place: ll needs unit column stride, row stride W and uniform plane spacing."""
    if ll.dim() != 4 or y.dim() != 4:
        raise IndexError("%s expects 4-D ll (N, C, H, W) and y (N, 4C, H, W), got %d-D and %d-D"
                         % (name, ll.dim(), y.dim()))
    N, C4, H, W = y.shape
    if C4 % 4 or tuple(ll.shape) != (N, C4 // 4, H, W):
        raise RuntimeError("%s: y must be (N, 4C, H, W) and ll (N, C, H, W), got %s and %s"
                           % (name, tuple(y.shape), tuple(ll.shape)))
    lk, ps, rs = _planes_view(ll)
    if rs != W and H > 1:
        lk = ll.contiguous()
        ps = H * W
    return lk, ps, y.contiguous()


def iswt_adjoint_taps(w_lo, w_hi, h_lo, h_hi):
    """The inverse level is (1/4) x the transpose of an analysis level with the synthesis taps: halved taps (exact)."""
    return [[0.5 * float(v) for v in t] for t in (w_lo, w_hi, h_lo, h_hi)]


def _iswt2d_cuda(ll, y, w_lo, w_hi, h_lo, h_hi, dilation):
    _require_cuda_f32(ll, "iswt2d")
    _require_cuda_f32(y, "iswt2d")
    if not (len(w_lo) == len(w_hi) == len(h_lo) == len(h_hi)):
        raise RuntimeError("b200wave::iswt2d: all four filters must have the same length")
    lk, ps, yk = iswt_layout(ll, y, "b200wave::iswt2d")
    N, C4, H, W = yk.shape
    x = torch.empty((N, C4 // 4, H, W), device=y.device, dtype=torch.float32)
    if x.numel() == 0:
        return x
    lib = _cabi.load()
    a = [_cabi.taps_array(t)[0] for t in (w_lo, w_hi, h_lo, h_hi)]
    with torch.cuda.device(y.device):
        rc = lib.b200w_iswt2d_f32(lk.data_ptr(), ps, yk.data_ptr(), N * (C4 // 4), H, W, a[0], a[1], a[2], a[3],
                                  len(w_lo), int(dilation), x.data_ptr(), _stream())
    _cabi.check(rc)
    return x


def _iswt2d_setup(ctx, inputs, output):
    ll, y, w_lo, w_hi, h_lo, h_hi, dilation = inputs
    ctx.taps = iswt_adjoint_taps(w_lo, w_hi, h_lo, h_hi)
    ctx.dilation = dilation


def iswt2d_backward(swt2d_op, ctx, dx):
    """Transpose of the level: the analysis kernel with the halved synthesis taps; band 0 of its output is the gradient
    of ll, bands 1..3 that of y (whose band 0 the level never reads)."""
    need_ll, need_y = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    if dx is None or not (need_ll or need_y):
        return (None,) * 7
    g = swt2d_op(dx, *ctx.taps, PERIODIC, ctx.dilation)
    N, C4, H, W = g.shape
    g5 = g.view(N, C4 // 4, 4, H, W)
    dll = g5[:, :, 0].clone() if need_ll else None
    dy = None
    if need_y:
        g5[:, :, 0] = 0
        dy = g
    return (dll, dy) + (None,) * 5


def _iswt2d_backward(ctx, dx):
    return iswt2d_backward(torch.ops.b200wave.swt2d, ctx, dx)


# ------------------------------------------------------------------------------------------- ssim
def _ssim_common(img1, img2, win, name):
    _require_cuda_f32(img1, name)
    _require_cuda_f32(img2, name)
    if img1.dim() != 4 or img1.shape != img2.shape:
        raise RuntimeError("b200wave::%s expects two (N, C, H, W) tensors of equal shape, got %s and %s"
                           % (name, tuple(img1.shape), tuple(img2.shape)))
    if len(win) % 2 == 0 or len(win) > _cabi.SSIM_MAX_WINDOW:
        raise RuntimeError("b200wave::%s: window size must be odd and <= %d, got %d"
                           % (name, _cabi.SSIM_MAX_WINDOW, len(win)))


def _ssim_fwd_cuda(img1, img2, win, size_average, n_maps):
    _ssim_common(img1, img2, win, "ssim_fwd")
    lib = _cabi.load()
    img1, img2 = img1.contiguous(), img2.contiguous()
    N, C, H, W = img1.shape
    out = torch.empty(() if size_average else (N,), device=img1.device, dtype=torch.float32)
    maps = torch.empty((n_maps, N, C, H, W), device=img1.device, dtype=torch.float32)
    ws_bytes = lib.b200w_ssim_workspace_bytes(N, C, H, W)
    work = torch.empty((max(ws_bytes, 4) // 4,), device=img1.device, dtype=torch.float32)
    a_win, nwin = _cabi.taps_array(win)
    with torch.cuda.device(img1.device):
        rc = lib.b200w_ssim_fwd_f32(img1.data_ptr(), img2.data_ptr(), N, C, H, W, a_win, nwin, int(size_average),
                                    int(n_maps), maps.data_ptr() if n_maps else None, out.data_ptr(),
                                    work.data_ptr(), ws_bytes, _stream())
    _cabi.check(rc)
    return out, maps


def _ssim_fwd_fake(img1, img2, win, size_average, n_maps):
    N, C, H, W = img1.shape
    return img1.new_empty(() if size_average else (N,)), img1.new_empty((n_maps, N, C, H, W))


def _ssim_bwd_cuda(img1, img2, maps, grad_out, win, size_average, need_d2):
    _ssim_common(img1, img2, win, "ssim_bwd")
    lib = _cabi.load()
    img1, img2, maps = img1.contiguous(), img2.contiguous(), maps.contiguous()
    N, C, H, W = img1.shape
    n_maps = maps.shape[0]
    if n_maps not in (3, 4) or (need_d2 and n_maps != 4):
        raise RuntimeError("b200wave::ssim_bwd: forward saved %d derivative maps, not enough for this backward"
                           % n_maps)
    g = grad_out.to(device=img1.device, dtype=torch.float32).contiguous()
    if g.numel() != (1 if size_average else N):
        raise RuntimeError("b200wave::ssim_bwd: grad_out has %d elements" % g.numel())
    d1 = torch.empty_like(img1)
    d2 = torch.empty_like(img2) if need_d2 else torch.empty((0,), device=img1.device, dtype=torch.float32)
    a_win, nwin = _cabi.taps_array(win)
    with torch.cuda.device(img1.device):
        rc = lib.b200w_ssim_bwd_f32(img1.data_ptr(), img2.data_ptr(), maps.data_ptr(), n_maps, g.data_ptr(),
                                    N, C, H, W, a_win, nwin, int(size_average), d1.data_ptr(),
                                    d2.data_ptr() if need_d2 else None, _stream())
    _cabi.check(rc)
    return d1, d2


def _ssim_bwd_fake(img1, img2, maps, grad_out, win, size_average, need_d2):
    return torch.empty_like(img1), (torch.empty_like(img2) if need_d2 else img1.new_empty((0,)))


def _ssim_setup(ctx, inputs, output):
    img1, img2, win, size_average, n_maps = inputs
    _, maps = output
    ctx.save_for_backward(img1, img2, maps)
    ctx.win = win
    ctx.size_average = size_average
    ctx.n_maps = n_maps
    ctx.set_materialize_grads(False)


def _ssim_backward(ctx, dval, dmaps):
    need1, need2 = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    if not (need1 or need2) or dval is None:
        return None, None, None, None, None
    if ctx.n_maps < 3 or (need2 and ctx.n_maps < 4):
        raise RuntimeError("b200wave::ssim_fwd was called with n_maps=%d, which does not support the requested "
                           "gradient (use 3 for d/dimg1, 4 for both)" % ctx.n_maps)
    img1, img2, maps = ctx.saved_tensors
    d1, d2 = torch.ops.b200wave.ssim_bwd(img1, img2, maps, dval, ctx.win, ctx.size_average, bool(need2))
    return (d1 if need1 else None), (d2 if need2 else None), None, None, None


_LIB.impl("afb2d", _afb2d_cuda, "CUDA")
_LIB.impl("sfb2d", _sfb2d_cuda, "CUDA")
_LIB.impl("dwt2", _dwt2_cuda, "CUDA")
_LIB.impl("idwt2", _idwt2_cuda, "CUDA")
_LIB.impl("ssim_fwd", _ssim_fwd_cuda, "CUDA")
_LIB.impl("ssim_bwd", _ssim_bwd_cuda, "CUDA")
_LIB.impl("afb2d_select", _afb2d_select_cuda, "CUDA")
_LIB.impl("afb1d", _afb1d_cuda, "CUDA")
_LIB.impl("swt2d", _swt2d_cuda, "CUDA")
_LIB.impl("swt2d_adjoint", _swt2d_adjoint_cuda, "CUDA")
_LIB.impl("sfb1d", _sfb1d_cuda, "CUDA")
_LIB.impl("iswt2d", _iswt2d_cuda, "CUDA")


def _cpu_refuse(name):
    def impl(*args, **kwargs):
        raise RuntimeError("b200wave::%s is CUDA-only (sm_100a): there is no CPU fallback. Move the tensors to "
                           "a B200 (`.cuda()`)." % name)
    return impl


for _name in ("afb2d", "afb2d_select", "sfb2d", "dwt2", "idwt2", "ssim_fwd", "ssim_bwd", "afb1d", "sfb1d", "swt2d",
              "swt2d_adjoint", "iswt2d"):
    _LIB.impl(_name, _cpu_refuse(_name), "CPU")

torch.library.register_fake("b200wave::afb2d", _afb2d_fake, lib=_LIB)
torch.library.register_fake("b200wave::sfb2d", _sfb2d_fake, lib=_LIB)
torch.library.register_fake("b200wave::afb2d_select", _afb2d_select_fake, lib=_LIB)
torch.library.register_autograd("b200wave::afb2d_select", _afb2d_select_backward, setup_context=_afb2d_select_setup,
                                lib=_LIB)
torch.library.register_fake("b200wave::dwt2", _dwt2_fake, lib=_LIB)
torch.library.register_fake("b200wave::afb1d", _afb1d_fake, lib=_LIB)
torch.library.register_fake("b200wave::swt2d", lambda x, wl, wh, hl, hh, mode, d:
                            x.new_empty((x.shape[0], 4 * x.shape[1], x.shape[2], x.shape[3])), lib=_LIB)
torch.library.register_fake("b200wave::swt2d_adjoint", lambda dy, wl, wh, hl, hh, mode, d:
                            dy.new_empty((dy.shape[0], dy.shape[1] // 4, dy.shape[2], dy.shape[3])), lib=_LIB)
torch.library.register_autograd("b200wave::swt2d", _swt2d_backward, setup_context=_swt2d_setup, lib=_LIB)
torch.library.register_fake("b200wave::sfb1d", _sfb1d_fake, lib=_LIB)
torch.library.register_fake("b200wave::iswt2d", lambda ll, y, wl, wh, hl, hh, d:
                            y.new_empty((y.shape[0], y.shape[1] // 4, y.shape[2], y.shape[3])), lib=_LIB)
torch.library.register_autograd("b200wave::iswt2d", _iswt2d_backward, setup_context=_iswt2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave::afb1d", _afb1d_backward, setup_context=_afb1d_setup, lib=_LIB)
torch.library.register_autograd("b200wave::sfb1d", _sfb1d_backward, setup_context=_sfb1d_setup, lib=_LIB)
torch.library.register_fake("b200wave::idwt2", _idwt2_fake, lib=_LIB)
torch.library.register_fake("b200wave::ssim_fwd", _ssim_fwd_fake, lib=_LIB)
torch.library.register_fake("b200wave::ssim_bwd", _ssim_bwd_fake, lib=_LIB)
torch.library.register_autograd("b200wave::afb2d", _afb2d_backward, setup_context=_afb2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave::sfb2d", _sfb2d_backward, setup_context=_sfb2d_setup, lib=_LIB)
torch.library.register_autograd("b200wave::ssim_fwd", _ssim_backward, setup_context=_ssim_setup, lib=_LIB)

afb2d = torch.ops.b200wave.afb2d
afb2d_select = torch.ops.b200wave.afb2d_select
sfb2d = torch.ops.b200wave.sfb2d
dwt2 = torch.ops.b200wave.dwt2
idwt2 = torch.ops.b200wave.idwt2
ssim_fwd = torch.ops.b200wave.ssim_fwd
ssim_bwd = torch.ops.b200wave.ssim_bwd
afb1d = torch.ops.b200wave.afb1d
swt2d = torch.ops.b200wave.swt2d
swt2d_adjoint = torch.ops.b200wave.swt2d_adjoint
iswt2d = torch.ops.b200wave.iswt2d
sfb1d = torch.ops.b200wave.sfb1d


def ssim_bench_kernels(sets, win):
    """The kernels one SSIM forward + backward step launches, for bench.py's per-kernel timing: yields
    (name, fn(i), algorithmic bytes per pixel, FP32-pipe lane operations per pixel).  ``sets`` = [(img1, img2), ...].
    Lane operations: a packed FFMA2 occupies the FP32 pipe for two lanes' worth (tools/micro/ffma2.cu), so it counts 2.
    Forward (4 moments): horizontal 4 x 12 (11 taps in 6 pairs) + 3 products + 4 pair sums, vertical 4 x 11, SSIM map +
    3 derivative maps 33 = 132.  Backward (3 maps): horizontal 3 x 12 + 3, vertical 4 x 11 (the 4th lane idles), 6 = 89."""
    n = len(sets)
    saved = [ssim_fwd(s[0].detach(), s[1], win, True, 3)[1] for s in sets]
    gout = torch.ones((), device=sets[0][0].device)
    return [
        ("ssim_fwd", lambda i: ssim_fwd(sets[i % n][0].detach(), sets[i % n][1], win, True, 3), 4 * (2 + 3), 132),
        ("ssim_bwd", lambda i: ssim_bwd(sets[i % n][0].detach(), sets[i % n][1], saved[i % n], gout, win, True, False),
         4 * (5 + 1), 89),
    ]
