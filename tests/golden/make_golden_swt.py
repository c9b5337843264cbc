"""Golden vectors for the undecimated (a trous) analysis bank, from the UNMODIFIED reference
(``pytorch_wavelets/dwt/lowlevel.py:475-521`` ``afb2d_atrous``, the level function of ``SWTForward``).

    python tests/golden/make_golden_swt.py        # writes tests/golden/swt_cases.npz

Build container only (needs /root/reference and the ``pywt`` stand-in).  float64 on fp32-valued inputs.  Per case the
output (N, 4C, H, W) and the input gradient autograd derives for a random upstream gradient; every case is replayed
through ``oracle/swt_oracle.py``.  The reference's own default mode ('periodization') is recorded as raising.
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
import pywt  # noqa: E402  (the stand-in)
from pytorch_wavelets.dwt import lowlevel  # noqa: E402  (the reference)
from pytorch_wavelets.dwt.transform2d import SWTForward  # noqa: E402

from oracle import swt_oracle  # noqa: E402
from helpers import save_golden  # noqa: E402  (keeps every golden file under 1 MB)

CASES = []
for mode in ("zero", "symmetric", "reflect", "periodic"):
    CASES.append(("db1", mode, 1, (1, 2, 12, 10)))
    CASES.append(("db2", mode, 1, (2, 1, 17, 20)))
    CASES.append(("db3", mode, 2, (1, 2, 23, 19)))
    CASES.append(("db2", mode, 4, (1, 1, 21, 26)))
CASES.append(("db4", "symmetric", 2, (1, 1, 9, 40)))          # pad larger than H: several mirror images
CASES.append((("db1", "db3"), "periodic", 1, (1, 1, 16, 18)))   # 4-tuple: col filters db1, row filters db3

out = {"ncases": len(CASES)}
rng = np.random.default_rng(21)
worst = 0.0


def f32(a):
    return a.astype(np.float32).astype(np.float64)


for k, (wave, mode, dil, shape) in enumerate(CASES):
    if isinstance(wave, tuple):
        wc, wr = pywt.Wavelet(wave[0]), pywt.Wavelet(wave[1])
        # equal lengths are required by the kernel ABI; pad the shorter pair with zeros at the end of the prepped taps
        filts = lowlevel.prep_filt_afb2d(wc.dec_lo, wc.dec_hi, wr.dec_lo, wr.dec_hi)
        name = "+".join(wave)
    else:
        w = pywt.Wavelet(wave)
        filts = lowlevel.prep_filt_afb2d(w.dec_lo, w.dec_hi, w.dec_lo, w.dec_hi)
        name = wave
    if filts[0].numel() != filts[2].numel():
        continue
    xn = f32(rng.standard_normal(shape))
    x = torch.from_numpy(xn).requires_grad_(True)
    y = lowlevel.afb2d_atrous(x, filts, mode, dil)
    gy = f32(rng.standard_normal(tuple(y.shape)))
    (dx,) = torch.autograd.grad(y, x, torch.from_numpy(gy))
    pre = "w%02d/" % k
    out[pre + "wave"], out[pre + "mode"], out[pre + "dilation"] = name, mode, dil
    out[pre + "x"], out[pre + "gy"] = xn, gy
    for nm, f in zip(("h0_col", "h1_col", "h0_row", "h1_row"), filts):
        out[pre + nm] = f.numpy().ravel()
    out[pre + "y"], out[pre + "dx"] = y.detach().numpy(), dx.numpy()
    fl = [out[pre + nm] for nm in ("h0_col", "h1_col", "h0_row", "h1_row")]
    worst = max(worst, float(np.abs(swt_oracle.afb2d_atrous(xn, *fl, mode, dil) - out[pre + "y"]).max()),
                float(np.abs(swt_oracle.afb2d_atrous_backward(gy, *fl, mode, dil) - out[pre + "dx"]).max()))
out["ncases"] = len([k for k in out if k.endswith("/x")])
# the reference's default configuration cannot run: record how it fails
try:
    SWTForward()(torch.zeros(1, 1, 8, 8))
    out["default_mode_error"] = ""
except Exception as e:      # noqa: BLE001
    out["default_mode_error"] = "%s: %s" % (type(e).__name__, e)
try:
    SWTForward(J=2, mode="zero")(torch.zeros(1, 1, 8, 8))
    out["J2_error"] = ""
except Exception as e:      # noqa: BLE001
    out["J2_error"] = "%s: %s" % (type(e).__name__, str(e)[:80])
save_golden("swt_cases", out)
print("swt cases: %d, worst |oracle - reference| = %.3e; default mode -> %s; J=2 -> %s"
      % (out["ncases"], worst, out["default_mode_error"], out["J2_error"]))
