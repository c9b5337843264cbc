"""Kernel micro-benchmark: per-launch duration of single levels / SSIM kernels (CUDA graph of back-to-back
launches over rotating inputs larger than L2, CUDA events).

    python tools/kbench.py [dwt|ssim|swt|iswt|dwt1d|fsd|freq|tv|all]
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import b200wave  # noqa: E402
from b200wave import lowlevel, ops  # noqa: E402
from b200wave.ssim import _win_taps  # noqa: E402

PEAK = 6538.9
dev = "cuda"


def timeit(fn, nsets, reps=60):
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    keep = []
    with torch.cuda.graph(g):
        for i in range(reps):
            keep.append(fn(i))
            if len(keep) > nsets:
                keep.pop(0)
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


def dwt_case(n, h, w, wave, mode):
    xfm = b200wave.DWTForward(J=1, wave=wave, mode=mode).to(dev)
    ifm = b200wave.DWTInverse(wave=wave, mode=mode).to(dev)
    m = lowlevel.mode_to_int(mode)
    nbytes_in = 4 * n * h * w
    nsets = max(2, int(2 * 126e6 * 1.05 / nbytes_in) + 1)
    xs = [torch.rand(n, 1, h, w, device=dev) for _ in range(nsets)]
    with torch.no_grad():
        cs = [xfm(x) for x in xs]
        ho, wo = cs[0][0].shape[-2:]
        by = 4 * n * (h * w + 4 * ho * wo)
        ta = timeit(lambda i: lowlevel.AFB2D.apply(xs[i % nsets], xfm.h0_col, xfm.h1_col, xfm.h0_row, xfm.h1_row, m), nsets)
        ts = timeit(lambda i: lowlevel.SFB2D.apply(cs[i % nsets][0], cs[i % nsets][1][0], ifm.g0_col, ifm.g1_col,
                                                   ifm.g0_row, ifm.g1_row, m), nsets)
    print("dwt %-5s %-13s %4dx%4dx%4d  afb %7.1f us %6.0f GB/s (%4.1f%%)   sfb %7.1f us %6.0f GB/s (%4.1f%%)" % (
        wave, mode, n, h, w, ta * 1e6, by / ta / 1e9, by / ta / 1e9 / PEAK * 100, ts * 1e6, by / ts / 1e9,
        by / ts / 1e9 / PEAK * 100), flush=True)


def ssim_case(n, h, w):
    nsets = max(2, int(2 * 126e6 / (8 * n * h * w)) + 1)
    a = [torch.rand(n, 1, h, w, device=dev) for _ in range(nsets)]
    b = [(t + 0.1 * torch.randn_like(t)).clamp_(0, 1) for t in a]
    win = _win_taps(11)
    g = torch.ones((), device=dev)
    with torch.no_grad():
        t0 = timeit(lambda i: ops.ssim_fwd(a[i % nsets], b[i % nsets], win, True, 0), nsets, 20)
        t3 = timeit(lambda i: ops.ssim_fwd(a[i % nsets], b[i % nsets], win, True, 3), nsets, 20)
        maps = [ops.ssim_fwd(a[i], b[i], win, True, 3)[1] for i in range(nsets)]
        tb = timeit(lambda i: ops.ssim_bwd(a[i % nsets], b[i % nsets], maps[i % nsets], g, win, True, False), nsets, 20)
    px = n * h * w
    print("ssim %4dx%4dx%4d  fwd(no maps) %7.1f us %6.1f Gpx/s %5.0f GB/s | fwd+3maps %7.1f us %5.0f GB/s | "
          "bwd %7.1f us %5.0f GB/s | fwd+bwd algorithmic 20 B/px: %5.0f GB/s (%4.1f%%)" % (
              n, h, w, t0 * 1e6, px / t0 / 1e9, 8 * px / t0 / 1e9, t3 * 1e6, 20 * px / t3 / 1e9, tb * 1e6,
              24 * px / tb / 1e9, 20 * px / (t3 + tb) / 1e9, 20 * px / (t3 + tb) / 1e9 / PEAK * 100), flush=True)


def freq_case(n, h, w, radius=10):
    """Fourier-domain split (utils.py:93-117 batched): whole call and the pointwise kernels alone."""
    import time
    import numpy as np
    from b200wave import freq
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle import freq_oracle
    nsets = max(2, int(2 * 126e6 * 1.05 / (4 * n * h * w)) + 1)
    xs = [torch.rand(n, 1, h, w, device=dev) for _ in range(nsets)]
    specs = [torch.fft.rfft2(x).contiguous() for x in xs]
    with torch.no_grad():
        t_all = timeit(lambda i: freq.gaussian_split(xs[i % nsets], radius, True, 1.0), nsets)
        t_mask = timeit(lambda i: torch.ops.b200wave_freq.mask_(specs[i % nsets], h, w, float(radius), True), nsets)
        t_abs = timeit(lambda i: torch.ops.b200wave_freq.abs_sign(xs[i % nsets], 1.0), nsets)
    px = n * h * w
    mask_bytes = 16 * n * h * (w // 2 + 1)
    xc = xs[0][:4].cpu().numpy()
    t0 = time.perf_counter()
    freq_oracle.split(xc, radius, True, 1.0)
    t_cpu = (time.perf_counter() - t0) / 4 * n
    print("freq %4dx%4dx%4d r=%d  split %7.1f us %6.1f Gpx/s | mask kernel %6.1f us %5.0f GB/s (%4.1f%%) | abs kernel %6.1f us "
          "%5.0f GB/s (%4.1f%%) | numpy fp64 (1 core) %8.1f ms" % (
              n, h, w, radius, t_all * 1e6, px / t_all / 1e9, t_mask * 1e6, mask_bytes / t_mask / 1e9,
              mask_bytes / t_mask / 1e9 / PEAK * 100, t_abs * 1e6, 8 * px / t_abs / 1e9, 8 * px / t_abs / 1e9 / PEAK * 100,
              t_cpu * 1e3), flush=True)


def fsd_case(n, h, w):
    """filter_wavelet (model.py:166-179, 222-235): fused store epilogue vs DWTForward + slicing/scaling/cat."""
    import b200wave
    from b200wave import fsd
    nsets = max(2, int(2 * 126e6 * 1.05 / (8 * n * h * w)) + 1)
    xs = [torch.randn(n, 1, h, w, device=dev) for _ in range(nsets)]
    xfm = b200wave.DWTForward(J=1, wave="haar", mode="reflect").to(dev)

    def unfused(x, cs):
        ll, (hi,) = xfm(x)
        if cs == "sum":
            return ll
        lh, hl, hh = hi[:, :, 0] * 0.5 + 0.5, hi[:, :, 1] * 0.5 + 0.5, hi[:, :, 2] * 0.5 + 0.5
        return torch.cat((lh, hl, hh), 1)

    px = n * h * w
    with torch.no_grad():
        for cs, variant, bytes_px in (("sum", "A", 4 + 1), ("cat", "B", 4 + 3)):
            t_f = timeit(lambda i: fsd.filter_wavelet(xs[i % nsets], cs, True, variant), nsets)
            t_u = timeit(lambda i: unfused(xs[i % nsets], cs), nsets)
            gbs = bytes_px * px / t_f / 1e9
            print("fsd %4dx%4dx%4d cs=%-3s fused %7.1f us %6.0f GB/s (%4.1f%% of peak, %d B/px) | unfused %7.1f us | x%.2f" % (
                n, h, w, cs, t_f * 1e6, gbs, gbs / PEAK * 100, bytes_px, t_u * 1e6, t_u / t_f), flush=True)


def dwt1d_case(rows, n, wave, mode):
    """1-D analysis / synthesis level (AFB1D / SFB1D): 8 B per input sample in either direction."""
    import b200wave
    nsets = max(2, int(2 * 126e6 * 1.05 / (4 * rows * n)) + 1)
    xs = [torch.randn(rows, 1, n, device=dev) for _ in range(nsets)]
    xfm = b200wave.DWT1DForward(J=1, wave=wave, mode=mode).to(dev)
    ifm = b200wave.DWT1DInverse(wave=wave, mode=mode).to(dev)
    with torch.no_grad():
        cs = [xfm(x) for x in xs]
        t_a = timeit(lambda i: xfm(xs[i % nsets]), nsets)
        t_s = timeit(lambda i: ifm(cs[i % nsets]), nsets)
    b = 8.0 * rows * n
    print("dwt1d %-5s %-13s %5dx%8d  afb1d %7.1f us %6.0f GB/s (%4.1f%%)   sfb1d %7.1f us %6.0f GB/s (%4.1f%%)" % (
        wave, mode, rows, n, t_a * 1e6, b / t_a / 1e9, b / t_a / 1e9 / PEAK * 100, t_s * 1e6, b / t_s / 1e9,
        b / t_s / 1e9 / PEAK * 100), flush=True)


def swt_case(n, h, w, wave, mode, dilation):
    """One undecimated level (afb2d_atrous): 4 B in + 16 B out per pixel."""
    from b200wave.dwt import lowlevel
    import b200wave
    nsets = max(2, int(2 * 126e6 * 1.05 / (4 * n * h * w)) + 1)
    xs = [torch.randn(n, 1, h, w, device=dev) for _ in range(nsets)]
    m = b200wave.SWTForward(J=1, wave=wave, mode=mode).to(dev)
    filts = (m.h0_col, m.h1_col, m.h0_row, m.h1_row)
    with torch.no_grad():
        t = timeit(lambda i: lowlevel.afb2d_atrous(xs[i % nsets], filts, mode, dilation), nsets)
    b = 20.0 * n * h * w
    print("swt   %-5s %-10s d=%d %4dx%4dx%4d  %7.1f us %6.0f GB/s (%4.1f%%)" % (
        wave, mode, dilation, n, h, w, t * 1e6, b / t / 1e9, b / t / 1e9 / PEAK * 100), flush=True)


def iswt_case(n, h, w, wave, dilation):
    """One level of SWTInverse (the a-trous synthesis kernel) and the same level through the adjoint route (the analysis
    kernel's gather-form adjoint with the halved synthesis taps, swt2d_adjoint); ll is band 0 of the coefficients, as at
    the top level.  Algorithmic bytes 20 B/px: 4 planes read, 1 written."""
    nsets = max(2, int(2 * 126e6 * 1.05 / (16 * n * h * w)) + 1)
    ys = [torch.randn(n, 4, h, w, device=dev) for _ in range(nsets)]
    m = b200wave.SWTInverse(wave=wave).to(dev)
    filts = (m.g0_col, m.g1_col, m.g0_row, m.g1_row)
    half = ops.iswt_adjoint_taps(*[lowlevel.host_taps(f) for f in (m.g0_row, m.g1_row, m.g0_col, m.g1_col)])
    with torch.no_grad():
        ref = ops.swt2d_adjoint(ys[0], *half, ops.PERIODIC, dilation)
        err = ((lowlevel.sfb2d_atrous(ys[0], filts, "periodic", dilation) - ref).abs().max() / ref.abs().max()).item()
        tk = timeit(lambda i: lowlevel.sfb2d_atrous(ys[i % nsets], filts, "periodic", dilation), nsets)
        ta = timeit(lambda i: ops.swt2d_adjoint(ys[i % nsets], *half, ops.PERIODIC, dilation), nsets, 10)
    b = 20.0 * n * h * w
    print("iswt  %-5s d=%-2d %4dx%4dx%4d  kernel %8.1f us %6.0f GB/s (%4.1f%%) | adjoint route %9.1f us %6.0f GB/s "
          "(%4.1f%%) | x%.1f | rel diff %.1e" % (
              wave, dilation, n, h, w, tk * 1e6, b / tk / 1e9, b / tk / 1e9 / PEAK * 100, ta * 1e6, b / ta / 1e9,
              b / ta / 1e9 / PEAK * 100, ta / tk, err), flush=True)


what = (sys.argv[1] if len(sys.argv) > 1 else "all") if __name__ == "__main__" else "none"
if what in ("iswt", "all"):
    import subprocess
    print("device:", subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                     "-i", "0"], capture_output=True, text=True).stdout.strip(), flush=True)
    for wave in ("haar", "db2", "db8"):
        iswt_case(64, 304, 304, wave, 1)
        for d in (1, 4, 16):
            iswt_case(64, 1024, 1024, wave, d)
if what in ("dwt1d", "all"):
    dwt1d_case(64, 1 << 20, "db3", "symmetric")
    dwt1d_case(64, 1 << 20, "haar", "zero")
    dwt1d_case(64, 1 << 20, "db8", "periodization")
    dwt1d_case(4096, 4096, "db3", "symmetric")
if what in ("swt", "all"):
    swt_case(64, 304, 304, "db2", "symmetric", 1)
    swt_case(64, 1024, 1024, "db2", "symmetric", 1)
    swt_case(64, 1024, 1024, "db2", "periodic", 4)
    swt_case(64, 1024, 1024, "haar", "zero", 1)
if what in ("fsd", "all"):
    fsd_case(8, 256, 256)
    fsd_case(64, 256, 256)
    fsd_case(64, 304, 304)
    fsd_case(64, 1024, 1024)
if what in ("freq", "all"):
    freq_case(64, 256, 256)
    freq_case(256, 256, 256)
    freq_case(64, 1024, 1024)
if what in ("dwt", "all"):
    dwt_case(64, 304, 304, "db3", "symmetric")
    dwt_case(64, 154, 154, "db3", "symmetric")
    dwt_case(64, 79, 79, "db3", "symmetric")
    dwt_case(64, 304, 304, "haar", "zero")
    dwt_case(64, 1024, 1024, "db3", "symmetric")
    dwt_case(64, 1024, 1024, "haar", "zero")
    dwt_case(64, 1024, 1024, "db8", "symmetric")
    dwt_case(16, 2048, 2048, "db4", "zero")
    dwt_case(64, 1024, 1024, "db2", "periodization")
if what in ("ssim", "all"):
    ssim_case(256, 400, 400)
    ssim_case(64, 1024, 1024)
    ssim_case(8, 304, 304)


def tv_case(n, h, w):
    """TVLoss (model.py:17-33): fused sums / gradient kernels vs the reference's slicing arithmetic in torch."""
    from b200wave.losses import TVLoss
    nsets = max(2, int(2 * 126e6 * 1.05 / (4 * n * h * w)) + 1)
    xs = [torch.rand(n, 1, h, w, device=dev) for _ in range(nsets)]
    crit = TVLoss()

    def ref(x):
        b, hx, wx = x.size(0), x.size(2), x.size(3)
        ch, cw = x[:, :, 1:, :].numel() // b, x[:, :, :, 1:].numel() // b
        h_tv = torch.pow(x[:, :, 1:, :] - x[:, :, :hx - 1, :], 2).sum()
        w_tv = torch.pow(x[:, :, :, 1:] - x[:, :, :, :wx - 1], 2).sum()
        return 2 * (h_tv / ch + w_tv / cw) / b

    g = torch.ones((), device=dev)
    with torch.no_grad():
        t_f = timeit(lambda i: torch.ops.b200wave_losses.tv_sums(xs[i % nsets]), nsets)
        t_b = timeit(lambda i: torch.ops.b200wave_losses.tv_grad(xs[i % nsets], g, 1e-6, 1e-6), nsets)
        t_r = timeit(lambda i: ref(xs[i % nsets]), nsets)
    px = n * h * w
    print("tv %4dx%4dx%4d  sums %7.1f us %5.0f GB/s (%4.1f%%) | grad %7.1f us %5.0f GB/s (%4.1f%%) | torch forward (reference arithmetic) %7.1f us x%.1f" % (
        n, h, w, t_f * 1e6, 4 * px / t_f / 1e9, 4 * px / t_f / 1e9 / PEAK * 100, t_b * 1e6, 8 * px / t_b / 1e9,
        8 * px / t_b / 1e9 / PEAK * 100, t_r * 1e6, t_r / t_f), flush=True)


if what in ("tv", "all"):
    tv_case(8, 256, 256)
    tv_case(64, 304, 304)
    tv_case(64, 1024, 1024)
