"""Golden vectors for the total-variation loss, from the UNMODIFIED reference ``model.py`` (``TVLoss``, :17-33).

    python tests/golden/make_golden_tv.py        # writes tests/golden/tv_cases.npz

Build container only (needs /root/reference and the ``pywt`` stand-in).  ``model.py`` imports packages that are not
installed here; empty stand-in modules let it import (as in make_golden_fsd.py).  float64 on fp32-valued inputs; each
case stores the loss and the input gradient for an upstream gradient of 1.
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

from oracle import tv_oracle  # noqa: E402
from helpers import save_golden  # noqa: E402  (keeps every golden file under 1 MB)

CASES = [((2, 1, 64, 64), 1), ((1, 1, 256, 256), 1), ((3, 2, 37, 41), 0.5), ((1, 3, 5, 300), 2), ((2, 1, 130, 7), 1),
         ((1, 1, 2, 2), 1)]
out = {"ncases": len(CASES)}
rng = np.random.default_rng(3)
worst = 0.0
for k, (shape, weight) in enumerate(CASES):
    x = torch.from_numpy(rng.random(shape).astype(np.float32).astype(np.float64)).requires_grad_(True)
    loss = ref_model.TVLoss(weight)(x)
    loss.backward()
    pre = "t%02d/" % k
    out[pre + "x"] = x.detach().numpy()
    out[pre + "weight"] = float(weight)
    out[pre + "loss"] = float(loss)
    out[pre + "dx"] = x.grad.numpy()
    worst = max(worst, abs(tv_oracle.tv_loss(out[pre + "x"], weight) - float(loss)) / abs(float(loss)),
                float(np.abs(tv_oracle.tv_loss_backward(out[pre + "x"], 1.0, weight) - out[pre + "dx"]).max()))
save_golden("tv_cases", out)
print("tv cases: %d, worst |oracle - reference| = %.3e" % (len(CASES), worst))
