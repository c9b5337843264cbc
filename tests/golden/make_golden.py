"""Generate golden vectors by running the UNMODIFIED reference in the build container.

    python tests/golden/make_golden.py            # writes tests/golden/*.npz

Needs ``/root/reference`` (read-only mount, build container only) and the
``pywt`` stand-in under ``oracle/pywt_standin`` (PyWavelets is not installed).
The reference runs on CPU in float64 (``torch.set_default_dtype``), on inputs
whose values are exactly representable in float32 so the fp32 CUDA path sees
identical inputs.  The script also replays every case through the numpy oracle
and prints the worst deviation (it must be ~1e-13).

The committed ``.npz`` files are what travels to the GPU box; nothing in the
test-suite reads ``/root/reference`` at run time.
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
sys.path.insert(0, REF)

warnings.filterwarnings("ignore")
import torch  # noqa: E402

torch.set_default_dtype(torch.float64)
import pywt  # noqa: E402  (the stand-in)
from pytorch_wavelets import DWTForward, DWTInverse  # noqa: E402  (the reference)
import ssim as ref_ssim  # noqa: E402  (the reference)

from oracle import dwt_oracle, ssim_oracle  # noqa: E402
from helpers import save_golden  # noqa: E402  (keeps every golden file under 1 MB)

# (name, wave, J, mode, (N, C, H, W))
DWT_CASES = []
# the reference's own parametrisation, tests/test_dwt.py:28-41, on a small image
for wave, J, mode in [("db1", 1, "zero"), ("db1", 3, "zero"), ("db3", 1, "symmetric"),
                      ("db3", 2, "reflect"), ("db2", 3, "periodization"), ("db2", 3, "periodic"),
                      ("db4", 2, "zero"), ("db3", 3, "symmetric"), ("bior2.4", 2, "periodization")]:
    DWT_CASES.append((wave, J, mode, (1, 2, 36, 28)))
# odd shapes, tests/test_dwt.py:84-129 scaled down
for size in [(32, 32), (31, 31), (30, 31), (26, 25), (25, 26)]:
    DWT_CASES.append(("db3", 3, "symmetric", (1, 2) + size))
    DWT_CASES.append(("db3", 2, "periodization", (1, 2) + size))
DWT_CASES.append(("haar", 1, "reflect", (2, 1, 16, 20)))          # model.py:140 configuration
DWT_CASES.append(("db2", 2, "periodic", (1, 1, 19, 23)))
DWT_CASES.append(("db8", 1, "symmetric", (1, 1, 40, 36)))
DWT_CASES.append(("db8", 1, "zero", (1, 1, 37, 41)))
# 4-tuple wave: haar as "col" (runs along W), db2 as "row" (runs along H) -- SURVEY 8a-Q2
DWT_CASES.append((("haar", "db2"), 2, "symmetric", (1, 2, 16, 24)))


def f32_valued(rng, shape, kind="randn"):
    a = rng.standard_normal(shape) if kind == "randn" else rng.random(shape)
    return a.astype(np.float32).astype(np.float64)


def wave_args(wave):
    if isinstance(wave, tuple):
        a, b = pywt.Wavelet(wave[0]), pywt.Wavelet(wave[1])
        dec = (a.dec_lo, a.dec_hi, b.dec_lo, b.dec_hi)
        rec = (a.rec_lo, a.rec_hi, b.rec_lo, b.rec_hi)
        return dec, rec
    return wave, wave


def run_dwt_case(idx, wave, J, mode, shape, rng):
    dec, rec = wave_args(wave)
    xfm = DWTForward(J=J, wave=dec, mode=mode)
    ifm = DWTInverse(wave=rec, mode=mode)
    x = torch.tensor(f32_valued(rng, shape), requires_grad=True)
    yl, yh = xfm(x)
    # AFB2D.backward chain
    gyl = torch.tensor(f32_valued(rng, tuple(yl.shape)))
    gyh = [torch.tensor(f32_valued(rng, tuple(h.shape))) for h in yh]
    (dx,) = torch.autograd.grad([yl] + list(yh), x, [gyl] + gyh)
    # SFB2D forward + backward chain on detached coefficients
    cl = yl.detach().clone().requires_grad_(True)
    ch = [h.detach().clone().requires_grad_(True) for h in yh]
    recon = ifm((cl, ch))
    grec = torch.tensor(f32_valued(rng, tuple(recon.shape)))
    dcs = torch.autograd.grad(recon, [cl] + ch, grec)
    out = {"x": x.detach().numpy(), "yl": yl.detach().numpy(), "gyl": gyl.numpy(), "dx": dx.numpy(),
           "recon": recon.detach().numpy(), "grec": grec.numpy(), "dcl": dcs[0].numpy(),
           "J": np.int64(J), "mode": np.array(mode),
           "wave": np.array(wave if isinstance(wave, str) else "|".join(wave))}
    for j in range(J):
        out["yh%d" % j] = yh[j].detach().numpy()
        out["gyh%d" % j] = gyh[j].numpy()
        out["dch%d" % j] = dcs[1 + j].numpy()
    # prepped filter buffers exactly as the reference modules hold them
    for nm in ("h0_col", "h1_col", "h0_row", "h1_row"):
        out[nm] = getattr(xfm, nm).numpy().ravel()
    for nm in ("g0_col", "g1_col", "g0_row", "g1_row"):
        out[nm] = getattr(ifm, nm).numpy().ravel()

    # ---- replay through the numpy oracle
    worst = 0.0
    h_col = (out["h0_col"], out["h1_col"])
    h_row = (out["h0_row"], out["h1_row"])
    g_col = (out["g0_col"], out["g1_col"])
    g_row = (out["g0_row"], out["g1_row"])
    oyl, oyh = dwt_oracle.dwt_forward(out["x"], J, h_col, h_row, mode)
    worst = max(worst, np.abs(oyl - out["yl"]).max())
    for j in range(J):
        worst = max(worst, np.abs(oyh[j] - out["yh%d" % j]).max())
    orec = dwt_oracle.dwt_inverse(out["yl"], [out["yh%d" % j] for j in range(J)], g_col, g_row, mode)
    worst = max(worst, np.abs(orec - out["recon"]).max())
    return out, worst


def run_ssim_case(name, a, b, size_average):
    t1 = torch.tensor(a, dtype=torch.float64, requires_grad=True)
    t2 = torch.tensor(b, dtype=torch.float64, requires_grad=True)
    # the window must be built as in normal fp32 use (ssim.py:7-15 under the
    # default dtype float32) and only then cast to the images' dtype (ssim.py:58)
    torch.set_default_dtype(torch.float32)
    try:
        val = ref_ssim.SSIM(window_size=11, size_average=size_average)(t1, t2)
    finally:
        torch.set_default_dtype(torch.float64)
    if size_average:
        gout = np.float64(1.0)
        val.backward()
    else:
        gout = np.linspace(0.5, 1.5, a.shape[0])
        val.backward(torch.tensor(gout))
    out = {"img1": a, "img2": b, "val": val.detach().numpy(), "gout": gout,
           "d1": t1.grad.numpy(), "d2": t2.grad.numpy(), "size_average": np.bool_(size_average)}
    oval = ssim_oracle.ssim(a, b, 11, size_average)
    o1, o2 = ssim_oracle.ssim_backward(a, b, gout, 11, size_average)
    worst = max(np.abs(oval - out["val"]).max(), np.abs(o1 - out["d1"]).max() / np.abs(out["d1"]).max(),
                np.abs(o2 - out["d2"]).max() / np.abs(out["d2"]).max())
    return out, worst


def main():
    rng = np.random.default_rng(20261018)
    worst_all = 0.0
    bundle = {}
    for i, (wave, J, mode, shape) in enumerate(DWT_CASES):
        out, worst = run_dwt_case(i, wave, J, mode, shape, rng)
        worst_all = max(worst_all, worst)
        for k, v in out.items():
            bundle["c%02d/%s" % (i, k)] = v
        print("dwt case %02d %-14s J=%d %-14s %s  oracle-vs-ref %.2e" % (i, wave, J, mode, shape, worst))
    bundle["ncases"] = np.int64(len(DWT_CASES))
    save_golden("dwt_cases", bundle)

    sb = {}
    x = f32_valued(rng, (2, 3, 24, 31), "rand")
    noisy = np.clip(x + 0.1 * f32_valued(rng, x.shape), 0, 1).astype(np.float32).astype(np.float64)
    indep = f32_valued(rng, x.shape, "rand")
    n = 0
    for nm, b in (("noisy", noisy), ("indep", indep)):
        for sa in (True, False):
            out, worst = run_ssim_case(nm, x, b, sa)
            worst_all = max(worst_all, worst)
            for k, v in out.items():
                sb["s%02d/%s" % (n, k)] = v
            print("ssim case %02d %-6s size_average=%s val=%s oracle-vs-ref %.2e" % (n, nm, sa, out["val"], worst))
            n += 1
    # known answer: ssim(x, x) == 1
    out, worst = run_ssim_case("same", x, x.copy(), True)
    for k, v in out.items():
        sb["s%02d/%s" % (n, k)] = v
    print("ssim case %02d same val=%s" % (n, out["val"]))
    n += 1
    sb["ncases"] = np.int64(n)
    save_golden("ssim_cases", sb)
    print("worst oracle-vs-reference deviation: %.3e" % worst_all)
    assert worst_all < 1e-10, worst_all


if __name__ == "__main__":
    main()
