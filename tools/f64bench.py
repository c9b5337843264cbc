"""Double-precision paths on the B200: fp64 SSIM forward (+3 derivative maps) and backward at the cfg3 shape
(256 x 1 x 400 x 400, 328 MB per double image, larger than L2), against the incumbent for this mode -- a torch
restatement of the reference's _ssim (ssim.py:17-37: five dense grouped F.conv2d + pointwise, autograd backward) in
double on the same card -- the 1-D / a trous kernels in double against fp32, and the frequency split's pointwise
kernels and filter_wavelet in double against fp32 (achieved GB/s against the HBM peak).  Times are CUDA events around
`--iters` launches after `--warmup`.  Prints one JSON line with the card name and power limit read in the same run.

    python tools/f64bench.py [--iters 20] [--warmup 3] [--dfma-per-s X]

`--dfma-per-s` (from tools/micro/dfma.cu) adds the fp64 SSIM kernels' share of that DFMA ceiling.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import b200wave  # noqa: E402
from b200wave import ops, ops64  # noqa: E402

SSIM_MOD = sys.modules[b200wave.SSIM.__module__]


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers still stand with the torch device name
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def reference_ssim(img1, img2, window, ws, channel):
    """ssim.py:17-37 in the images' dtype."""
    mu1 = F.conv2d(img1, window, padding=ws // 2, groups=channel)
    mu2 = F.conv2d(img2, window, padding=ws // 2, groups=channel)
    mu1_sq, mu2_sq, mu1_mu2 = mu1.pow(2), mu2.pow(2), mu1 * mu2
    sigma1_sq = F.conv2d(img1 * img1, window, padding=ws // 2, groups=channel) - mu1_sq
    sigma2_sq = F.conv2d(img2 * img2, window, padding=ws // 2, groups=channel) - mu2_sq
    sigma12 = F.conv2d(img1 * img2, window, padding=ws // 2, groups=channel) - mu1_mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    m = ((2 * mu1_mu2 + C1) * (2 * sigma12 + C2)) / ((mu1_sq + mu2_sq + C1) * (sigma1_sq + sigma2_sq + C2))
    return m.mean()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dfma-per-s", type=float, default=None)
    args = ap.parse_args()
    dev = "cuda"
    res = {"card": card()}
    it, wu = args.iters, args.warmup

    # ---- SSIM at cfg3
    N, C, H, W, ws = 256, 1, 400, 400, 11
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand((N, C, H, W), generator=g, device=dev, dtype=torch.float64)
    y = (x + 0.1 * torch.randn(x.shape, generator=g, device=dev, dtype=torch.float64)).clamp_(0, 1)
    win = SSIM_MOD._win2d_taps(ws)
    _, maps = ops64.ssim_fwd(x, y, win, True, 3)
    gout = torch.ones((), device=dev, dtype=torch.float64)
    t_fwd = timed(lambda: ops64.ssim_fwd(x, y, win, True, 3), it, wu)
    t_bwd = timed(lambda: ops64.ssim_bwd(x, y, maps, gout, win, True, False), it, wu)
    px = N * C * H * W
    ssim = {"shape": [N, C, H, W], "fwd_ms": t_fwd, "bwd_ms": t_bwd, "step_ms": t_fwd + t_bwd,
            "fwd_dfma_per_s": px * 4 * ws * ws / (t_fwd * 1e-3), "bwd_dfma_per_s": px * 3 * ws * ws / (t_bwd * 1e-3)}
    if args.dfma_per_s:
        ssim["fwd_share_of_dfma_ceiling"] = ssim["fwd_dfma_per_s"] / args.dfma_per_s
        ssim["bwd_share_of_dfma_ceiling"] = ssim["bwd_dfma_per_s"] / args.dfma_per_s
    del maps
    window = torch.tensor(win, device=dev, dtype=torch.float64).reshape(1, 1, ws, ws).expand(C, 1, ws, ws).contiguous()
    xr = x.clone().requires_grad_(True)

    def torch_step():
        xr.grad = None
        reference_ssim(xr, y, window, ws, C).backward()

    t_torch = timed(torch_step, max(3, it // 4), 1)
    with torch.no_grad():
        vk = b200wave.ssim(x, y).item()
        vt = reference_ssim(x, y, window, ws, C).item()
    ssim.update({"torch_f64_conv2d_step_ms": t_torch, "speedup_vs_torch_f64": t_torch / (t_fwd + t_bwd),
                 "value_kernel": vk, "value_torch": vt})
    x32, y32 = x.float(), y.float()
    w1 = SSIM_MOD._win_taps(ws)
    _, m32 = ops.ssim_fwd(x32, y32, w1, True, 3)
    g32 = gout.float()
    ssim["fp32_step_ms"] = timed(lambda: ops.ssim_fwd(x32, y32, w1, True, 3), it, wu) + \
        timed(lambda: ops.ssim_bwd(x32, y32, m32, g32, w1, True, False), it, wu)
    res["ssim_cfg3"] = ssim
    del x, y, xr, x32, y32, m32
    torch.cuda.empty_cache()

    # ---- 1-D at 64 x 2^20 (db4, symmetric) and SWT at 64 x 304^2 (db2, zero, dilation 1): double vs fp32
    from b200wave.wavelets import as_wavelet
    wv = as_wavelet("db4")
    h0, h1 = tuple(wv.dec_lo[::-1]), tuple(wv.dec_hi[::-1])
    g0, g1 = tuple(wv.rec_lo), tuple(wv.rec_hi)
    one_d = {}
    for name, dt, mod in (("f64", torch.float64, ops64), ("f32", torch.float32, ops)):
        s = torch.randn((64, 1, 1 << 20), device=dev, dtype=dt)
        lo, hi = mod.afb1d(s, h0, h1, 1)
        one_d[name + "_afb1d_ms"] = timed(lambda: mod.afb1d(s, h0, h1, 1), it, wu)
        one_d[name + "_sfb1d_ms"] = timed(lambda: mod.sfb1d(lo, hi, g0, g1, 1, -1), it, wu)
    res["dwt1d_64x2^20_db4"] = one_d
    w2 = as_wavelet("db2")
    a0, a1 = tuple(w2.dec_lo[::-1]), tuple(w2.dec_hi[::-1])
    swt = {}
    for name, dt, fwd, adj in (("f64", torch.float64, ops64.swt2d, ops64.swt2d_adjoint),
                               ("f32", torch.float32, ops.swt2d, torch.ops.b200wave.swt2d_adjoint)):
        s = torch.randn((64, 1, 304, 304), device=dev, dtype=dt)
        yy = fwd(s, a0, a1, a0, a1, 0, 1)
        swt[name + "_fwd_ms"] = timed(lambda: fwd(s, a0, a1, a0, a1, 0, 1), it, wu)
        swt[name + "_adjoint_ms"] = timed(lambda: adj(yy, a0, a1, a0, a1, 0, 1), it, wu)
    res["swt_64x304^2_db2"] = swt
    res.update(freq_and_fsd(it, wu))
    print(json.dumps(res))


def hbm_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json"
    except (OSError, KeyError, ValueError):
        return 7700.0, "data sheet (MEASURED_PEAKS.json absent)"


def freq_and_fsd(it, wu):
    """Double frequency split (mask kernel on the complex128 half spectrum, abs kernel) and double filter_wavelet at
    64 x 256^2 (the spectrum and the image fit the 126 MB L2) and 64 x 1024^2 (they do not), with the fp32 kernels
    beside them.  Algorithmic bytes per call: mask 2 x the bin (16 B/bin fp32 complex64 -> 32 B/bin complex128), abs
    2 x the pixel; filter_wavelet reads the image once and writes LL (cs='sum', A) or the three detail bands
    (cs='cat', B) at a quarter of the pixels: fp64 8 B/px in + 2 or 6 B/px out (fp32 half of that, DESIGN K6)."""
    from b200wave import freq, fsd
    peak, src = hbm_peak_gbs()
    dev = "cuda"
    out = {"hbm_peak_gbs": peak, "hbm_peak_source": src}
    for side in (256, 1024):
        key = "64x%d^2" % side
        r = {}
        for name, dt in (("f64", torch.float64), ("f32", torch.float32)):
            mask_, abs_sign = freq._ops(dt)[:2]
            es = torch.finfo(dt).bits // 8
            x = torch.rand((64, 1, side, side), device=dev, dtype=dt)
            spec = torch.fft.rfft2(x).contiguous()
            bins, px = spec.numel(), x.numel()
            t_mask = timed(lambda: mask_(spec, side, side, 10.0, True), it, wu)
            t_abs = timed(lambda: abs_sign(x, 1.0), it, wu)
            t_split = timed(lambda: freq.gaussian_split(x, 10, True), it, wu)
            r[name + "_mask_ms"] = t_mask
            r[name + "_mask_gbs"] = 4 * es * bins / (t_mask * 1e6)
            r[name + "_abs_ms"] = t_abs
            r[name + "_abs_gbs"] = 2 * es * px / (t_abs * 1e6)
            r[name + "_split_fwd_ms"] = t_split
            for cs, variant, out_b in (("sum", "A", 1), ("cat", "B", 3)):
                t = timed(lambda: fsd.filter_wavelet(x, cs, True, variant), it, wu)
                r["%s_fsd_%s%s_ms" % (name, cs, variant)] = t
                r["%s_fsd_%s%s_gbs" % (name, cs, variant)] = (es + out_b * es / 4) * px / (t * 1e6)
            for k in [k for k in r if k.startswith(name) and k.endswith("_gbs")]:
                r[k[:-4] + "_share_of_hbm_peak"] = r[k] / peak
            del x, spec
            torch.cuda.empty_cache()
        out["freq_fsd_" + key] = r
    return out


if __name__ == "__main__":
    main()
