"""Golden vectors for the Fourier-domain frequency split, from the UNMODIFIED reference ``utils.py``.

    python tests/golden/make_golden_freq.py        # writes tests/golden/freq_cases.*.npz

Build container only (needs /root/reference).  ``utils.py`` imports packages that are not installed here (skimage,
matplotlib, ...) and hard-codes ``.cuda()`` on the mask (``utils.py:97,110``); empty stand-in modules and a no-op
``Tensor.cuda`` let the unmodified functions run on CPU.  Inputs are fp32-valued; the reference computes in
complex64/fp32 here exactly as it does in ``train.py``.
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
             "tqdm", "torchvision", "torchvision.utils", "torchvision.transforms", "PIL", "PIL.Image", "visdom", "tkinter"]:
    if name not in sys.modules:
        try:
            __import__(name)
        except Exception:
            sys.modules[name] = _Stub(name)

torch.Tensor.cuda = lambda self, *a, **k: self      # utils.py:97,110 call .cuda() on the mask
sys.path.insert(0, REF)
import utils as ref_utils  # noqa: E402  (the reference)

from oracle import freq_oracle  # noqa: E402
from helpers import save_golden  # noqa: E402  (keeps every golden file under 1 MB)

CASES = [  # (H, W, radius, highpass) -- train.py:173-213 uses i = 10, 8, 5, 14 on 256x256
    (256, 256, 10, True), (256, 256, 8, False), (128, 128, 5, True), (128, 128, 14, False),
    (64, 48, 4, True), (33, 40, 10, False), (50, 37, 3, True), (31, 31, 6, False),
]

out = {"ncases": len(CASES)}
rng = np.random.default_rng(2024)
worst = 0.0
for k, (h, w, r, hp) in enumerate(CASES):
    x = rng.random((1, h, w)).astype(np.float32)
    t = torch.tensor(x)
    y = (ref_utils.high_pass(t, i=r) if hp else ref_utils.low_pass(t, i=r)).numpy()
    o = freq_oracle.high_pass(x, r) if hp else freq_oracle.low_pass(x, r)
    err = np.abs(o - y).max() / np.abs(y).max()
    worst = max(worst, err)
    pre = "f%02d/" % k
    out[pre + "x"] = x
    out[pre + "y"] = y.astype(np.float32)      # the reference computes in fp32
    out[pre + "radius"] = r
    out[pre + "highpass"] = int(hp)
print("oracle (float64) vs reference (fp32 fft): worst rel err %.2e" % worst)
print("wrote", save_golden("freq_cases", out))
