"""CPU: the torch op surface of the package -- every op's schema and the dispatch keys that have a kernel, the CUDA-only
refusal of CPU tensors, and the output shapes of every op with a fake implementation, in both precisions."""
import re

import pytest
import torch

import b200wave  # noqa: F401  (registers every op)

NAMESPACES = ("b200wave", "b200wave64", "b200wave_losses", "b200wave_freq")
KEYS = ("CUDA", "CPU", "Meta", "Autograd")

_ALL = "CUDA CPU Meta Autograd"
_NO_AUTOGRAD = "CUDA CPU Meta"
_CUDA_CPU = "CUDA CPU"
SURFACE = [
    ("b200wave64::abs_sign(Tensor x, float sign) -> Tensor", _CUDA_CPU),
    ("b200wave64::afb1d(Tensor x, float[] h0, float[] h1, int mode) -> (Tensor, Tensor)", _ALL),
    ("b200wave64::afb2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode) "
     "-> (Tensor, Tensor)", _ALL),
    ("b200wave64::afb2d_select(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
     "bool want_low, bool want_highs, float hi_scale, float hi_shift) -> (Tensor, Tensor)", _ALL),
    ("b200wave64::freq_mask_(Tensor(a!) spec, int rows, int cols, float radius, bool highpass) -> Tensor(a!)",
     _CUDA_CPU),
    ("b200wave64::iswt2d(Tensor ll, Tensor y, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int dilation) "
     "-> Tensor", _ALL),
    ("b200wave64::msssim_scale(Tensor img1, Tensor img2, float[] win, bool cs, bool pool, int n_maps) "
     "-> (Tensor, Tensor, Tensor, Tensor)", _ALL),
    ("b200wave64::msssim_scale_bwd(Tensor img1, Tensor img2, Tensor maps, Tensor grad_out, float[] win, Tensor? up1, "
     "Tensor? up2, bool need_d2) -> (Tensor, Tensor)", _NO_AUTOGRAD),
    ("b200wave64::sfb1d(Tensor low, Tensor? high, float[] g0, float[] g1, int mode, int out_len) -> Tensor", _ALL),
    ("b200wave64::sfb2d(Tensor low, Tensor? highs, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
     "int out_h, int out_w) -> Tensor", _ALL),
    ("b200wave64::sign_mul(Tensor g, Tensor x, float sign) -> Tensor", _CUDA_CPU),
    ("b200wave64::ssim_bwd(Tensor img1, Tensor img2, Tensor maps, Tensor grad_out, float[] win, bool size_average, "
     "bool need_d2) -> (Tensor, Tensor)", _NO_AUTOGRAD),
    ("b200wave64::ssim_fwd(Tensor img1, Tensor img2, float[] win, bool size_average, int n_maps) -> (Tensor, Tensor)",
     _ALL),
    ("b200wave64::swt2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, int dilation) "
     "-> Tensor", _ALL),
    ("b200wave64::swt2d_adjoint(Tensor dy, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
     "int dilation) -> Tensor", _NO_AUTOGRAD),
    ("b200wave64::tv_grad(Tensor x, Tensor grad_out, float ch, float cw) -> Tensor", _NO_AUTOGRAD),
    ("b200wave64::tv_sums(Tensor x) -> Tensor", _NO_AUTOGRAD),
    ("b200wave::afb1d(Tensor x, float[] h0, float[] h1, int mode) -> (Tensor, Tensor)", _ALL),
    ("b200wave::afb2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode) -> (Tensor, Tensor)",
     _ALL),
    ("b200wave::afb2d_select(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
     "bool want_low, bool want_highs, float hi_scale, float hi_shift) -> (Tensor, Tensor)", _ALL),
    ("b200wave::dwt2(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, int J, int[] pad_hw) "
     "-> Tensor[]", _NO_AUTOGRAD),
    ("b200wave::idwt2(Tensor yl, Tensor?[] yh, int[] hw, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, "
     "int mode, int[] out_hw) -> Tensor", _NO_AUTOGRAD),
    ("b200wave::iswt2d(Tensor ll, Tensor y, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int dilation) "
     "-> Tensor", _ALL),
    ("b200wave::msssim_scale(Tensor img1, Tensor img2, float[] win, bool cs, bool pool, int n_maps) "
     "-> (Tensor, Tensor, Tensor, Tensor)", _ALL),
    ("b200wave::msssim_scale_bwd(Tensor img1, Tensor img2, Tensor maps, Tensor grad_out, float[] win, Tensor? up1, "
     "Tensor? up2, bool need_d2) -> (Tensor, Tensor)", _NO_AUTOGRAD),
    ("b200wave::sfb1d(Tensor low, Tensor? high, float[] g0, float[] g1, int mode, int out_len) -> Tensor", _ALL),
    ("b200wave::sfb2d(Tensor low, Tensor? highs, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
     "int out_h, int out_w) -> Tensor", _ALL),
    ("b200wave::ssim_bwd(Tensor img1, Tensor img2, Tensor maps, Tensor grad_out, float[] win, bool size_average, "
     "bool need_d2) -> (Tensor, Tensor)", _NO_AUTOGRAD),
    ("b200wave::ssim_fwd(Tensor img1, Tensor img2, float[] win, bool size_average, int n_maps) -> (Tensor, Tensor)",
     _ALL),
    ("b200wave::swt2d(Tensor x, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, int dilation) "
     "-> Tensor", _ALL),
    ("b200wave::swt2d_adjoint(Tensor dy, float[] w_lo, float[] w_hi, float[] h_lo, float[] h_hi, int mode, "
     "int dilation) -> Tensor", _NO_AUTOGRAD),
    ("b200wave_freq::abs_sign(Tensor x, float sign) -> Tensor", _CUDA_CPU),
    ("b200wave_freq::mask_(Tensor(a!) spec, int rows, int cols, float radius, bool highpass) -> Tensor(a!)",
     _CUDA_CPU),
    ("b200wave_freq::sign_mul(Tensor g, Tensor x, float sign) -> Tensor", _CUDA_CPU),
    ("b200wave_losses::phase_grad(Tensor fx, Tensor fy, int cols, float radius, Tensor sums, Tensor grad_out, "
     "float eps) -> (Tensor, Tensor)", _NO_AUTOGRAD),
    ("b200wave_losses::phase_sums(Tensor fx, Tensor fy, int cols, float radius) -> Tensor", _NO_AUTOGRAD),
    ("b200wave_losses::tv_grad(Tensor x, Tensor grad_out, float ch, float cw) -> Tensor", _NO_AUTOGRAD),
    ("b200wave_losses::tv_sums(Tensor x) -> Tensor", _NO_AUTOGRAD),
]


def _op_names():
    return sorted(n for n in torch._C._dispatch_get_all_op_names() if n.split("::")[0] in NAMESPACES)


def _packet(name):
    ns, op = name.split("::")
    return getattr(getattr(torch.ops, ns), op)


def test_schemas_and_dispatch_keys():
    got = [(str(_packet(n).default._schema),
            " ".join(k for k in KEYS if torch._C._dispatch_has_kernel_for_dispatch_key(n, k))) for n in _op_names()]
    assert got == SURFACE


def _cpu_args(name):
    """Arguments of the op's schema with CPU tensors of the op's dtype (complex for a spectrum)."""
    dtype = torch.float64 if name.startswith("b200wave64::") else torch.float32
    args = []
    for a in _packet(name).default._schema.arguments:
        t = str(a.type)
        x = torch.zeros((1, 1, 8, 8), dtype=dtype)
        if a.name == "spec":
            x = x.to(dtype.to_complex())
        args.append({"Tensor": x, "Optional[Tensor]": x, "List[Tensor]": [x], "List[Optional[Tensor]]": [x],
                     "List[float]": [0.5, 0.5], "List[int]": [], "int": 1, "float": 1.0, "bool": True}[t])
    return args


@pytest.mark.parametrize("name", [e[0].split("(")[0] for e in SURFACE])
def test_every_op_refuses_cpu_tensors(name):
    with pytest.raises(RuntimeError, match=re.escape("%s is CUDA-only" % name)):
        _packet(name)(*_cpu_args(name))


def _ns(op, dtype):
    """Namespace of a twin op: float64 ones are b200wave64::*, float32 TV ones b200wave_losses::*."""
    if dtype == torch.float64:
        return "b200wave64"
    return "b200wave_losses" if op.startswith("tv_") else "b200wave"


def _meta_cases(dtype):
    """(op name without namespace, args, expected output shapes) of every op with a fake in this precision."""
    x = torch.empty((4, 2, 37, 50), device="meta", dtype=dtype)
    low, highs = x.new_empty((4, 2, 21, 27)), x.new_empty((4, 2, 3, 21, 27))
    x1, lo1 = x.new_empty((4, 2, 37)), x.new_empty((4, 2, 19))
    y4 = x.new_empty((4, 8, 37, 50))
    w6, w2 = [0.1] * 6, [0.5] * 2
    win = [0.2] * 5 if dtype == torch.float32 else [0.04] * 25
    maps, g = x.new_empty((3, 4, 2, 37, 50)), x.new_empty(())
    gn = x.new_empty((4,))
    half = (4, 2, 18, 25)
    return [
        ("afb2d", (x, w6, w6, w6, w6, 1), [(4, 2, 21, 27), (4, 2, 3, 21, 27)]),
        ("afb2d_select", (x, w6, w6, w6, w6, 1, True, False, 0.5, 0.5), [(4, 2, 21, 27), (0,)]),
        ("afb2d_select", (x, w6, w6, w2, w2, 2, False, True, 0.5, 0.5), [(0,), (4, 2, 3, 19, 25)]),
        ("sfb2d", (low, highs, w6, w6, w6, w6, 1, -1, -1), [(4, 2, 38, 50)]),
        ("sfb2d", (low, None, w6, w6, w6, w6, 1, 37, 49), [(4, 2, 37, 49)]),
        ("afb1d", (x1, w6, w6, 2), [(4, 2, 19), (4, 2, 19)]),
        ("sfb1d", (lo1, lo1, w6, w6, 2, -1), [(4, 2, 38)]),
        ("sfb1d", (lo1, None, w6, w6, 2, 37), [(4, 2, 37)]),
        ("swt2d", (x, w2, w2, w2, w2, 0, 2), [(4, 8, 37, 50)]),
        ("swt2d_adjoint", (y4, w2, w2, w2, w2, 0, 2), [(4, 2, 37, 50)]),
        ("iswt2d", (x, y4, w2, w2, w2, w2, 1), [(4, 2, 37, 50)]),
        ("ssim_fwd", (x, x, win, False, 3), [(4,), (3, 4, 2, 37, 50)]),
        ("ssim_fwd", (x, x, win, True, 0), [(), (0, 4, 2, 37, 50)]),
        ("ssim_bwd", (x, x, maps, g, win, True, True), [(4, 2, 37, 50), (4, 2, 37, 50)]),
        ("ssim_bwd", (x, x, maps, gn, win, False, False), [(4, 2, 37, 50), (0,)]),
        ("msssim_scale", (x, x, win, True, True, 3), [(4,), (3, 4, 2, 37, 50), half, half]),
        ("msssim_scale", (x, x, win, False, False, 4), [(4,), (4, 4, 2, 37, 50), (0,), (0,)]),
        ("msssim_scale_bwd", (x, x, maps, gn, win, x.new_empty(half), None, True), [(4, 2, 37, 50), (4, 2, 37, 50)]),
        ("msssim_scale_bwd", (x, x, maps, gn, win, None, None, False), [(4, 2, 37, 50), (0,)]),
        ("tv_sums", (x,), [(2,)]),
        ("tv_grad", (x, g, 1.0, 1.0), [(4, 2, 37, 50)]),
    ]


def _fp32_only_cases():
    x = torch.empty((4, 2, 37, 50), device="meta")
    w6 = [0.1] * 6
    fx = torch.empty((2, 16, 9, 2), device="meta")
    return [
        ("b200wave", "dwt2", (x, w6, w6, w6, w6, 1, 2, []), [(4, 2, 13, 16), (4, 2, 3, 21, 27), (4, 2, 3, 13, 16)]),
        ("b200wave", "idwt2", (x.new_empty((4, 2, 13, 16)), [None, None], [21, 27, 13, 16], w6, w6, w6, w6, 1, []),
         [(4, 2, 38, 50)]),
        ("b200wave", "idwt2", (x.new_empty((4, 2, 13, 16)), [None, None], [21, 27, 13, 16], w6, w6, w6, w6, 1,
                               [37, 50, 21, 27]), [(4, 2, 37, 50)]),
        ("b200wave_losses", "phase_sums", (fx, fx, 16, 5.0), [(3,)]),
        ("b200wave_losses", "phase_grad", (fx, fx, 16, 5.0, fx.new_empty((3,)), fx.new_empty(()), 1e-8),
         [(2, 16, 9, 2), (2, 16, 9, 2)]),
    ]


def _check_meta(ns, op, args, shapes, dtype):
    out = getattr(getattr(torch.ops, ns), op)(*args)
    out = list(out) if isinstance(out, (tuple, list)) else [out]
    assert [tuple(t.shape) for t in out] == shapes, (ns, op)
    assert all(t.device.type == "meta" and t.dtype == dtype for t in out), (ns, op)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_fake_shapes_in_both_precisions(dtype):
    for op, args, shapes in _meta_cases(dtype):
        _check_meta(_ns(op, dtype), op, args, shapes, dtype)


def test_fake_shapes_of_fp32_only_ops():
    for ns, op, args, shapes in _fp32_only_cases():
        _check_meta(ns, op, args, shapes, torch.float32)


def test_every_fake_is_covered():
    """The cases above reach every op that has a Meta kernel."""
    have = {n for n in _op_names() if torch._C._dispatch_has_kernel_for_dispatch_key(n, "Meta")}
    covered = {_ns(op, dt) + "::" + op for dt in (torch.float32, torch.float64) for op, _, _ in _meta_cases(dt)}
    covered |= {ns + "::" + op for ns, op, _, _ in _fp32_only_cases()}
    assert covered == have
