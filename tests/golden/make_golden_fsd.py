"""Golden vectors for the discriminators' wavelet front end, from the UNMODIFIED reference ``model.py``.

    python tests/golden/make_golden_fsd.py        # writes tests/golden/fsd_cases.npz

Build container only (needs /root/reference and the ``pywt`` stand-in, PyWavelets is not installed).  ``model.py``
imports packages that are not installed here (tkinter, cv2, torchvision, ...); empty stand-in modules let it import.
``FS_DiscriminatorA/B.filter_wavelet`` (model.py:166-179, 222-235) are called unbound on a small object that holds
what the methods read (``DWT2`` -- the reference's own ``DWTForward(J=1, 'haar', 'reflect')`` -- and ``cs``), so no
convolutional discriminator has to be built.  float64 on fp32-valued inputs; each case also stores the input gradient
autograd gives for fixed upstream gradients.
"""
import os
import sys
import types
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("B200W_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle", "pywt_standin"))
warnings.filterwarnings("ignore")
import torch  # noqa: E402


class _Stub(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        sub = _Stub(self.__name__ + "." + name)
        setattr(self, name, sub)
        return sub

    def __call__(self, *a, **k):
        return None


for name in ["skimage", "skimage.metrics", "skimage.io", "skimage.measure", "matplotlib", "matplotlib.pyplot", "cv2",
             "tqdm", "torchvision", "torchvision.utils", "torchvision.transforms", "torchvision.models", "PIL",
             "PIL.Image", "visdom", "tkinter"]:
    if name not in sys.modules:
        try:
            __import__(name)
        except Exception:
            sys.modules[name] = _Stub(name)

sys.path.insert(0, os.path.join(REF, "pytorch_wavelets"))
sys.path.insert(0, REF)
torch.set_default_dtype(torch.float64)
import model as ref_model  # noqa: E402  (the reference)
from pytorch_wavelets import DWTForward  # noqa: E402  (the reference)

from oracle import fsd_oracle  # noqa: E402
from helpers import save_golden  # noqa: E402  (keeps every golden file under 1 MB)

# (variant, cs, norm, (N, C, H, W)); train.py feeds (N, 1, 256, 256) crops, FS_DiscriminatorA cs='sum', B cs='cat'
CASES = [("A", "sum", True, (2, 1, 64, 64)), ("B", "cat", True, (2, 1, 64, 64)),
         ("A", "each", True, (1, 1, 37, 41)), ("B", "sum", True, (1, 1, 40, 52)),
         ("A", "cat", False, (1, 1, 31, 36)), ("B", "each", False, (2, 2, 24, 20)),
         ("B", "cat", True, (2, 3, 18, 28)), ("A", "sum", False, (1, 2, 33, 33))]

out = {"ncases": len(CASES)}
rng = np.random.default_rng(7)
worst = 0.0
for k, (variant, cs, norm, shape) in enumerate(CASES):
    cls = ref_model.FS_DiscriminatorA if variant == "A" else ref_model.FS_DiscriminatorB
    holder = types.SimpleNamespace(DWT2=DWTForward(J=1, wave='haar', mode='reflect'), cs=cs)
    x = torch.from_numpy(rng.standard_normal(shape).astype(np.float32).astype(np.float64)).requires_grad_(True)
    res = cls.filter_wavelet(holder, x, norm)
    assert res[-1] is x
    bands = res[:-1]
    grads = [torch.from_numpy(rng.standard_normal(tuple(b.shape)).astype(np.float32).astype(np.float64)) for b in bands]
    torch.autograd.backward(list(bands), grads)
    pre = "w%02d/" % k
    out[pre + "x"] = x.detach().numpy()
    out[pre + "variant"] = variant
    out[pre + "cs"] = cs
    out[pre + "norm"] = norm
    out[pre + "nbands"] = len(bands)
    for i, (b, g) in enumerate(zip(bands, grads)):
        out[pre + "y%d" % i] = b.detach().numpy()
        out[pre + "g%d" % i] = g.numpy()
    out[pre + "dx"] = x.grad.numpy()
    mine = fsd_oracle.filter_wavelet(out[pre + "x"], cs, norm, variant)
    for i, m in enumerate(mine):
        worst = max(worst, float(np.abs(m - out[pre + "y%d" % i]).max()))
    dxo = fsd_oracle.filter_wavelet_backward([g.numpy() for g in grads], shape, cs, norm, variant)
    worst = max(worst, float(np.abs(dxo - out[pre + "dx"]).max()))

save_golden("fsd_cases", out)
print("fsd cases: %d, worst |oracle - reference| = %.3e" % (len(CASES), worst))
