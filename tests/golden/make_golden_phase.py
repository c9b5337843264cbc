"""Golden vectors for phase_consistency_loss, from the UNMODIFIED reference ``model.py`` (:36-58).

    python tests/golden/make_golden_phase.py        # writes tests/golden/phase_cases.*.npz

Build container only (needs /root/reference and the ``pywt`` stand-in).  ``model.py`` imports packages that are not
installed here and hard-codes ``.cuda()`` on the mask (:50); empty stand-in modules and a no-op ``Tensor.cuda`` let the
unmodified module run on CPU (as in make_golden_freq.py).  float64 on fp32-valued inputs; each case stores the loss and
both input gradients for an upstream gradient of 1.
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
torch.Tensor.cuda = lambda self, *a, **k: self      # model.py:50 calls .cuda() on the mask
torch.Tensor.float = lambda self, *a, **k: self     # ... after .float(): keep the float64 golden arithmetic
import model as ref_model  # noqa: E402  (the reference)

from oracle import phase_oracle  # noqa: E402
from helpers import save_golden  # noqa: E402  (keeps every golden file under 1 MB)

CASES = [(2, 1, 64, 64), (1, 1, 256, 256), (3, 2, 37, 41), (1, 3, 16, 50), (2, 1, 33, 8), (1, 1, 128, 96)]
out = {"ncases": len(CASES)}
rng = np.random.default_rng(5)
worst = 0.0
for k, shape in enumerate(CASES):
    xn = rng.random(shape).astype(np.float32).astype(np.float64)
    yn = np.clip(xn + 0.2 * rng.standard_normal(shape), 0, 1).astype(np.float32).astype(np.float64)
    x = torch.from_numpy(xn).requires_grad_(True)
    y = torch.from_numpy(yn).requires_grad_(True)
    loss = ref_model.phase_consistency_loss()(x, y)
    loss.backward()
    pre = "p%02d/" % k
    out[pre + "x"], out[pre + "y"] = xn, yn
    out[pre + "loss"] = float(loss)
    out[pre + "dx"], out[pre + "dy"] = x.grad.numpy(), y.grad.numpy()
    worst = max(worst, abs(phase_oracle.phase_consistency_loss(xn, yn) - float(loss)),
                float(np.abs(phase_oracle.phase_consistency_grad(xn, yn, 0) - out[pre + "dx"]).max()
                      / np.abs(out[pre + "dx"]).max()),
                float(np.abs(phase_oracle.phase_consistency_grad(xn, yn, 1) - out[pre + "dy"]).max()
                      / np.abs(out[pre + "dy"]).max()))
save_golden("phase_cases", out)
print("phase cases: %d, worst |oracle - reference| = %.3e" % (len(CASES), worst))
