"""Golden vectors for the 1-D DWT, from the UNMODIFIED reference (``pytorch_wavelets/dwt/transform1d.py`` over
``lowlevel.AFB1D`` / ``SFB1D``).

    python tests/golden/make_golden_1d.py        # writes tests/golden/dwt1d_cases.npz

Build container only (needs /root/reference and the ``pywt`` stand-in).  Cases follow the reference's own
parametrisation (tests/test_dwt1d.py:28-39 on (5, 4, 64) scaled to (2, 3, 64); the odd lengths of :81-88) plus a long
filter.  float64 on fp32-valued inputs.  Per case: the forward coefficients, the reconstruction, the input gradient of
the forward transform for random upstream gradients (AFB1D.backward chain) and the coefficient gradients of the inverse
(SFB1D.backward chain); the prepped filter buffers as the modules hold them.  Every case is replayed through the numpy
oracle (``dwt_oracle.afb1d`` / ``sfb1d``) and the worst deviation is printed.
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("B200W_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle", "pywt_standin"))
sys.path.insert(0, os.path.join(REF, "pytorch_wavelets"))
warnings.filterwarnings("ignore")
import torch  # noqa: E402

torch.set_default_dtype(torch.float64)
from pytorch_wavelets.dwt.transform1d import DWT1DForward, DWT1DInverse  # noqa: E402  (the reference)

from oracle import dwt_oracle  # noqa: E402
from helpers import save_golden  # noqa: E402  (keeps every golden file under 1 MB)

CASES = []
for wave, J, mode in [("db1", 1, "zero"), ("db1", 3, "zero"), ("db3", 1, "symmetric"), ("db3", 2, "reflect"),
                      ("db2", 3, "periodization"), ("db2", 3, "periodic"), ("db4", 2, "zero"), ("db3", 3, "symmetric"),
                      ("bior2.4", 2, "periodization")]:
    CASES.append((wave, J, mode, (2, 3, 64)))
for length in (64, 127, 99):
    for mode in ("symmetric", "periodization"):
        CASES.append(("db3", 3, mode, (2, 2, length)))
CASES.append(("db8", 2, "symmetric", (1, 2, 75)))
CASES.append(("db8", 1, "zero", (1, 1, 40)))

out = {"ncases": len(CASES)}
rng = np.random.default_rng(11)
worst = 0.0


def f32(a):
    return a.astype(np.float32).astype(np.float64)


for k, (wave, J, mode, shape) in enumerate(CASES):
    xn = f32(rng.standard_normal(shape))
    xfm, ifm = DWT1DForward(J=J, wave=wave, mode=mode), DWT1DInverse(wave=wave, mode=mode)
    x = torch.from_numpy(xn).requires_grad_(True)
    yl, yh = xfm(x)
    gl = f32(rng.standard_normal(tuple(yl.shape)))
    gh = [f32(rng.standard_normal(tuple(t.shape))) for t in yh]
    (dx,) = torch.autograd.grad([yl] + list(yh), x, [torch.from_numpy(gl)] + [torch.from_numpy(g) for g in gh])
    cl = yl.detach().clone().requires_grad_(True)
    ch = [t.detach().clone().requires_grad_(True) for t in yh]
    rec = ifm((cl, ch))
    gy = f32(rng.standard_normal(tuple(rec.shape)))
    grads = torch.autograd.grad(rec, [cl] + ch, torch.from_numpy(gy))
    pre = "d%02d/" % k
    out[pre + "wave"], out[pre + "J"], out[pre + "mode"] = wave, J, mode
    out[pre + "x"] = xn
    out[pre + "h0"], out[pre + "h1"] = xfm.h0.numpy().ravel(), xfm.h1.numpy().ravel()
    out[pre + "g0"], out[pre + "g1"] = ifm.g0.numpy().ravel(), ifm.g1.numpy().ravel()
    out[pre + "yl"] = yl.detach().numpy()
    out[pre + "gl"], out[pre + "gy"] = gl, gy
    out[pre + "dx"] = dx.numpy()
    out[pre + "rec"] = rec.detach().numpy()
    out[pre + "dcl"] = grads[0].numpy()
    for j in range(J):
        out[pre + "yh%d" % j] = yh[j].detach().numpy()
        out[pre + "gh%d" % j] = gh[j]
        out[pre + "dch%d" % j] = grads[1 + j].numpy()
    # oracle replay (forward + inverse)
    h0, h1, g0, g1 = out[pre + "h0"], out[pre + "h1"], out[pre + "g0"], out[pre + "g1"]
    lo = xn
    for j in range(J):
        lo, hi = dwt_oracle.afb1d(lo, h0, h1, mode)
        worst = max(worst, float(np.abs(hi - out[pre + "yh%d" % j]).max()))
    worst = max(worst, float(np.abs(lo - out[pre + "yl"]).max()))
    r = out[pre + "yl"]
    for j in range(J - 1, -1, -1):
        hi = out[pre + "yh%d" % j]
        if r.shape[-1] > hi.shape[-1]:
            r = r[..., :-1]
        r = dwt_oracle.sfb1d(r, hi, g0, g1, mode)
    worst = max(worst, float(np.abs(r - out[pre + "rec"]).max()))
save_golden("dwt1d_cases", out)
print("dwt1d cases: %d, worst |oracle - reference| = %.3e" % (len(CASES), worst))
