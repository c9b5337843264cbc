#!/usr/bin/env python
"""Benchmark of the wavelet + SSIM hot path (driver contract: ONE JSON line on stdout from rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2|cfg1|cfg3|sweep1024] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input:
  cfg2 (default, BASELINE.json configs[1]): DWTForward(J=3, db3, symmetric) -> DWTInverse -> backward through both,
        on a 64x1x304x304 batch per GPU (SURVEY.md 8d);
  cfg1: haar/zero/J=3 round trip + SSIM(recon, x), no grad, 8x1x304x304;
  cfg3: SSIM fwd+bwd (grad w.r.t. img1), 256x1x400x400;
  sweep1024: one point of the configs[4] sweep, DWT+IDWT J=3 db3 symmetric fwd+bwd on 64x1x1024x1024.
value  = Mpix/s (input pixels N*C*H*W per step) with inputs resident in HBM, steps replayed from CUDA graphs
         captured through the public modules, rotating over input sets that together exceed the L2;
e2e    = the same step through the public API starting from pinned HOST buffers, host<->device copies inside the
         timed region;
roofline     = the slowest kernel the step launches (for J > 1 the multi-level chain kernels), timed alone with CUDA
               events: its algorithmic bytes / time against the measured HBM peak (MEASURED_PEAKS.json);
workloads    = the other BASELINE configs in the same run (device-resident value + roofline each), so every config is
               driver-measured, not only the headline one;
reference_gpu = the UNMODIFIED reference modules (oracle/_ref, staged by `make -C oracle ref`) on the same GPU, its own
               F.conv2d composition, CUDA events -- the incumbent on this hardware (reported, not part of any timed region
               of ours);
cpu_baseline = the reference's CPU path on the host cores: the unmodified reference (kind "reference") when it is
               staged, else the C/OpenMP port oracle/c/ref_port.c (kind "port").
--impl reference times that CPU path only (rank 0) and prints the same line with "impl": "reference".
--dump-outputs DIR writes what the last timed step of the headline workload returned (rank 0) as DIR/<name>.npy, so
that two builds run with the same arguments, and therefore on the same seeded inputs, can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "wavelet+SSIM fwd/bwd Mpix/s"
UNIT = "Mpix/s"
L2_BYTES = 126 * 1024 * 1024

WORKLOADS = {
    "cfg2": dict(desc="cfg2: DWT+IDWT J=3 db3 symmetric fwd+bwd, 64x1x304x304 per GPU", kind="dwt",
                 shape=(64, 1, 304, 304), wave="db3", mode="symmetric", J=3, grad=True, ssim=False),
    "cfg1": dict(desc="cfg1: DWT+IDWT J=3 haar zero round trip + SSIM, no grad, 8x1x304x304 per GPU", kind="dwt",
                 shape=(8, 1, 304, 304), wave="haar", mode="zero", J=3, grad=False, ssim=True),
    "cfg3": dict(desc="cfg3: SSIM 11x11 fwd+bwd (grad img1), 256x1x400x400 per GPU", kind="ssim",
                 shape=(256, 1, 400, 400)),
    "sweep1024": dict(desc="cfg5 point: DWT+IDWT J=3 db3 symmetric fwd+bwd, 64x1x1024x1024 per GPU", kind="dwt",
                      shape=(64, 1, 1024, 1024), wave="db3", mode="symmetric", J=3, grad=True, ssim=False),
}
SECONDARY = ["cfg1", "cfg3", "sweep1024"]   # reported under "workloads" next to the headline


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of that kernel on this workload, from the committed
    `ncu --set full` captures (profiles/traffic.json); None when there is no capture for it."""
    for name in ("traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                v = json.load(fh).get(workload, {}).get(kernel)
            if v is not None:
                return v
        except (OSError, ValueError):
            pass
    return None


def host_copy_bound(n_gpus):
    """Measured pinned-memory copy bandwidth of the box with `n_gpus` ranks copying at once, both directions busy
    (profiles/pcie_probe.json, written from tools/pcie_probe.py runs under torchrun): GB/s per rank per direction."""
    try:
        with open(os.path.join(ROOT, "profiles", "pcie_probe.json")) as fh:
            e = json.load(fh).get(str(n_gpus))
        return (float(e["duplex_gbs_per_rank_per_direction"]), e.get("source")) if e else (None, None)
    except (OSError, ValueError, KeyError):
        return None, None


def level_sizes(h, w, L, J, mode):
    out = []
    for _ in range(J):
        h = (h + 1) // 2 if mode == "periodization" else (h + L - 1) // 2
        w = (w + 1) // 2 if mode == "periodization" else (w + L - 1) // 2
        out.append((h, w))
    return out


def dwt_pass_bytes(shape, L, J, mode):
    """Algorithmic bytes of one transform pass (SURVEY.md 8d): 4*NC*(n0 + 3*sum n_j + n_J)."""
    n, c, h, w = shape
    sizes = level_sizes(h, w, L, J, mode)
    coeffs = 3 * sum(a * b for a, b in sizes) + sizes[-1][0] * sizes[-1][1]
    return 4 * n * c * (h * w + coeffs)


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed regions run."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv = None
            self.err = repr(e)

    def _reasons(self):
        nv = self.nv
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10,
                 "applications_clocks_setting": 0x2}
        return [k for k, bit in names.items() if mask & bit]

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                self.samples.append((mhz, util))
                self.reasons.update(self._reasons())
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        busy = [m for m, u in self.samples if u > 0] or [m for m, _ in self.samples]
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------- CPU reference arm
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        return os.cpu_count() or 1


def _sized_run(make, run, n, steps, warmup, budget_s, cores):
    """Times `steps` calls of run(batch) on a sub-batch sized (from one probe) to fit about budget_s seconds."""
    probe_b = max(1, min(n, 2 * cores))
    probe = make(probe_b)
    run(probe)
    t0 = time.perf_counter()
    run(probe)
    per_img = (time.perf_counter() - t0) / probe_b
    total = max(1, steps + warmup)
    b = int(max(1, min(n, budget_s / (total * per_img))))
    batch = make(b)
    for _ in range(warmup):
        run(batch)
    t0 = time.perf_counter()
    for _ in range(steps):
        run(batch)
    return b, time.perf_counter() - t0


def cpu_reference_unmodified(workload, steps, warmup, budget_s):
    """The reference's own modules (oracle/_ref: pytorch_wavelets + ssim.py, unmodified) on the host cores."""
    import torch
    from oracle import ref_runner
    pw, ss = ref_runner.load()
    cfg = WORKLOADS[workload]
    n, c, h, w = cfg["shape"]
    cores = host_cores()
    torch.set_num_threads(cores)   # torchrun exports OMP_NUM_THREADS=1 for its workers: ask for the cores explicitly
    gen = torch.Generator().manual_seed(0)
    if cfg["kind"] == "dwt":
        xfm = pw.DWTForward(J=cfg["J"], wave=cfg["wave"], mode=cfg["mode"])
        ifm = pw.DWTInverse(wave=cfg["wave"], mode=cfg["mode"])
        crit = ss.SSIM() if cfg["ssim"] else None

        def run(batch):
            x, g = batch
            if cfg["grad"]:
                x.grad = None
                rec = ifm(xfm(x))
                rec.backward(g)
            else:
                with torch.no_grad():
                    rec = ifm(xfm(x))
                    if crit is not None:
                        crit(rec, x)

        def make(b):
            return (torch.rand((b, c, h, w), generator=gen).requires_grad_(cfg["grad"]),
                    torch.randn((b, c, h, w), generator=gen))
    else:
        crit = ss.SSIM()

        def run(batch):
            x, y = batch
            x.grad = None
            crit(x, y).backward()

        def make(b):
            x = torch.rand((b, c, h, w), generator=gen)
            y = (x + 0.1 * torch.randn((b, c, h, w), generator=gen)).clamp_(0, 1)
            return x.requires_grad_(True), y
    b, dt = _sized_run(make, run, n, steps, warmup, budget_s, cores)
    mpix = b * c * h * w / 1e6
    return {"value": mpix * steps / dt, "unit": UNIT, "cores": cores, "kind": "reference",
            "sample": "%d of %d images per step (%s), %d steps, unmodified pytorch_wavelets + ssim.py (oracle/_ref) on "
                      "torch CPU, %d threads" % (b, n, "x".join(map(str, (b, c, h, w))), steps, cores),
            "ms_per_step": dt / steps * 1e3}


def cpu_reference_port(workload, steps, warmup, budget_s):
    """The C/OpenMP port of the reference's CPU path (oracle/c/ref_port.c) on all host cores."""
    import numpy as np
    from oracle import c_port, dwt_oracle, ssim_oracle
    sys.path.insert(0, os.path.join(ROOT, "oracle", "pywt_standin"))
    import pywt  # stand-in: tap source of the oracle side
    cfg = WORKLOADS[workload]
    rng = np.random.default_rng(0)
    n, c, h, w = cfg["shape"]
    cores = c_port.use_all_cores()   # not OMP_NUM_THREADS: torchrun pins that to 1 for its workers

    if cfg["kind"] == "dwt":
        wv = pywt.Wavelet(cfg["wave"])
        hf = tuple(np.asarray(t, np.float32) for t in dwt_oracle.prep_afb(wv.dec_lo, wv.dec_hi))
        gf = (np.asarray(wv.rec_lo, np.float32), np.asarray(wv.rec_hi, np.float32))
        win2d = ssim_oracle.window2d(11)

        def run(batch):
            x = batch["x"]
            if cfg["grad"]:
                c_port.dwt_roundtrip_fwd_bwd(x, batch["g"], cfg["J"], hf, hf, gf, gf, cfg["mode"])
            else:
                yl, yh = c_port.dwt_forward(x, cfg["J"], hf, hf, cfg["mode"])
                rec = c_port.dwt_inverse(yl, yh, gf, gf, cfg["mode"])
                if cfg["ssim"]:
                    c_port.ssim(rec, x, win2d, True)

        def make(b):
            return {"x": rng.random((b, c, h, w), dtype=np.float32),
                    "g": rng.standard_normal((b, c, h, w)).astype(np.float32)}
    else:
        win2d = ssim_oracle.window2d(11)

        def run(batch):
            c_port.ssim(batch["x"], batch["y"], win2d, True, None, True, False)

        def make(b):
            x = rng.random((b, c, h, w), dtype=np.float32)
            return {"x": x, "y": np.clip(x + 0.1 * rng.standard_normal(x.shape).astype(np.float32), 0, 1)}

    b, dt = _sized_run(make, run, n, steps, warmup, budget_s, cores)
    mpix = b * c * h * w / 1e6
    return {"value": mpix * steps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d of %d images per step (%s), %d steps, C/OpenMP port of the reference's CPU path "
                      "(oracle/c/ref_port.c; the unmodified reference is not staged under oracle/_ref)" %
                      (b, n, "x".join(map(str, (b, c, h, w))), steps),
            "ms_per_step": dt / steps * 1e3}


def cpu_reference(workload, steps, warmup, budget_s=60.0):
    from oracle import ref_runner
    if ref_runner.available():
        return cpu_reference_unmodified(workload, steps, warmup, budget_s)
    return cpu_reference_port(workload, steps, warmup, budget_s)


# ----------------------------------------------------------------------------------------------- GPU arm
def build_step(cfg, dev, modules):
    """The step of a workload through the given modules (ours or the reference's): returns (step, make_set,
    set_bytes, step_bytes, extras)."""
    import torch
    n, c, h, w = cfg["shape"]
    if cfg["kind"] == "dwt":
        xfm = modules.DWTForward(J=cfg["J"], wave=cfg["wave"], mode=cfg["mode"]).to(dev)
        ifm = modules.DWTInverse(wave=cfg["wave"], mode=cfg["mode"]).to(dev)
        crit = modules.SSIM() if cfg["ssim"] else None
        L = xfm.h0_col.numel()
        passes = 4 if cfg["grad"] else 2
        step_bytes = passes * dwt_pass_bytes(cfg["shape"], L, cfg["J"], cfg["mode"]) + (8 * n * c * h * w if crit else 0)

        def step(x, g):
            if cfg["grad"]:
                x.grad = None
                yl, yh = xfm(x)
                rec = ifm((yl, yh))
                rec.backward(g)
                return rec, x.grad
            with torch.no_grad():
                yl, yh = xfm(x)
                rec = ifm((yl, yh))
                val = crit(rec, x) if crit else None
            return rec, val

        def make_set():
            x = torch.rand(n, c, h, w, device=dev, requires_grad=cfg["grad"])
            g = torch.randn(n, c, h, w, device=dev)
            return x, g
        extras = {"xfm": xfm, "ifm": ifm, "L": L}
    else:
        crit = modules.SSIM()
        step_bytes = 20 * n * c * h * w

        def step(x, y):
            x.grad = None
            val = crit(x, y)
            val.backward()
            return val, x.grad

        def make_set():
            x = torch.rand(n, c, h, w, device=dev)
            y = (x + 0.1 * torch.randn_like(x)).clamp_(0, 1)
            return x.requires_grad_(True), y
        extras = {}
    return step, make_set, 2 * 4 * n * c * h * w, step_bytes, extras


def step_output_names(cfg):
    """Names of the tensors the step of build_step returns, in order."""
    if cfg["kind"] == "ssim":
        return ("ssim", "dx")
    return ("rec", "dx") if cfg["grad"] else ("rec", "ssim")


DUMP_BYTES = 60 * 1024 * 1024   # all dumped arrays together; the .npy headers stay well inside 64 MB


def dump_outputs(out_dir, names, outputs):
    """Writes each output tensor as out_dir/<name>.npy (float32 or float64).  An output larger than its share of
    DUMP_BYTES is written as a fixed sample: the elements of its flattened array at the sorted indices that
    numpy.random.default_rng(0).choice(numel, k, replace=False) draws.  Returns what was written."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    pairs = [(name, t.detach()) for name, t in zip(names, outputs) if t is not None]
    written = {}
    for name, t in pairs:
        if t.dtype not in (torch.float32, torch.float64):
            t = t.float()
        flat = t.reshape(-1)
        k = DUMP_BYTES // len(pairs) // flat.element_size()
        entry = {"shape": list(t.shape), "dtype": str(t.dtype).replace("torch.", "")}
        if flat.numel() > k:
            idx = np.sort(np.random.default_rng(0).choice(flat.numel(), k, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
            entry["sampled"] = k
        np.save(os.path.join(out_dir, name + ".npy"), flat.cpu().numpy() if "sampled" in entry else t.cpu().numpy())
        written[name] = entry
    return written


def capture_graphs(step, sets):
    import torch
    graphs = []
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for s in sets:
            step(*s)
    torch.cuda.current_stream().wait_stream(side)
    for s in sets:
        gph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gph):
            out = step(*s)
        graphs.append((gph, out))
    torch.cuda.synchronize()
    return graphs


def time_kernel(fn, nsets, reps):
    """Average duration of one launch: `reps` launches over rotating inputs captured into one CUDA graph (no host
    launch gaps, outputs from the graph's pool), timed with events on the stream."""
    import torch
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    gph = torch.cuda.CUDAGraph()
    keep = []
    with torch.cuda.graph(gph):
        for i in range(reps):
            keep.append(fn(i))
            if len(keep) > nsets:
                keep.pop(0)
    gph.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    gph.replay()
    b.record()
    torch.cuda.synchronize()
    del keep
    return a.elapsed_time(b) / reps * 1e-3


def kernel_rooflines(name, cfg, sets, extras, reps, peak, peak_src):
    """Times the kernels the step of this workload launches, each alone; returns (roofline of the slowest, table)."""
    import torch
    from b200wave import _cabi, lowlevel
    n, c, h, w = cfg["shape"]
    nsets = len(sets)
    kernels = {}
    with torch.no_grad():
        if cfg["kind"] == "dwt":
            xfm, ifm, L = extras["xfm"], extras["ifm"], extras["L"]
            mode = lowlevel.mode_to_int(cfg["mode"])
            ho, wo = level_sizes(h, w, L, 1, cfg["mode"])[0]
            lvl_bytes = 4 * n * c * (h * w + 4 * ho * wo)
            t_afb = time_kernel(lambda i: lowlevel.AFB2D.apply(sets[i % nsets][0].detach(), xfm.h0_col, xfm.h1_col,
                                                               xfm.h0_row, xfm.h1_row, mode), nsets, reps)
            k_afb = _cabi.recent_kernels(1)[0]
            ll1 = [lowlevel.AFB2D.apply(s[0].detach(), xfm.h0_col, xfm.h1_col, xfm.h0_row, xfm.h1_row, mode)
                   for s in sets]
            t_sfb = time_kernel(lambda i: lowlevel.SFB2D.apply(ll1[i % nsets][0], ll1[i % nsets][1], ifm.g0_col,
                                                               ifm.g1_col, ifm.g0_row, ifm.g1_row, mode), nsets, reps)
            k_sfb = _cabi.recent_kernels(1)[0]
            del ll1
            kernels = {"afb2d_level1": {"s": t_afb, "GB/s": lvl_bytes / t_afb / 1e9, "bytes": lvl_bytes, "sass": k_afb},
                       "sfb2d_level1": {"s": t_sfb, "GB/s": lvl_bytes / t_sfb / 1e9, "bytes": lvl_bytes, "sass": k_sfb}}
            slowest = "afb2d_level1" if t_afb >= t_sfb else "sfb2d_level1"
            if cfg["J"] > 1:
                # the kernels the step actually launches: one chain kernel per J-level transform (forward and
                # backward passes use the same two kernels)
                chain_bytes = dwt_pass_bytes(cfg["shape"], L, cfg["J"], cfg["mode"])
                coeffs = [xfm(s[0].detach()) for s in sets]
                t_dwt = time_kernel(lambda i: xfm(sets[i % nsets][0].detach()), nsets, reps)
                k_dwt = _cabi.recent_kernels(1)[0]
                t_idwt = time_kernel(lambda i: ifm(coeffs[i % nsets]), nsets, reps)
                k_idwt = _cabi.recent_kernels(1)[0]
                del coeffs
                kernels["dwt2_chain"] = {"s": t_dwt, "GB/s": chain_bytes / t_dwt / 1e9, "bytes": chain_bytes,
                                         "sass": k_dwt, "levels": cfg["J"]}
                kernels["idwt2_chain"] = {"s": t_idwt, "GB/s": chain_bytes / t_idwt / 1e9, "bytes": chain_bytes,
                                          "sass": k_idwt, "levels": cfg["J"]}
                slowest = "dwt2_chain" if t_dwt >= t_idwt else "idwt2_chain"
        else:
            kernels = ssim_kernels(sets, n * c * h * w, nsets, reps)
            slowest = max(kernels, key=lambda k: kernels[k]["s"])
    k = kernels[slowest]
    roof = {"bound": "hbm", "kernel": slowest, "achieved": k["GB/s"], "peak": peak, "unit": "GB/s",
            "frac": k["GB/s"] / peak, "traffic": ncu_traffic(name, slowest), "peak_source": peak_src,
            "algorithmic_bytes_per_launch": k["bytes"], "launch_us": k["s"] * 1e6, "sass": k.get("sass"),
            "note": "timed alone: %d launches over rotating inputs > L2 in one CUDA graph, CUDA events" % reps}
    if "fp32_ceiling_GB/s" in k:
        roof["fp32_ceiling"] = {"GB/s": k["fp32_ceiling_GB/s"], "frac_of_ceiling": k["GB/s"] / k["fp32_ceiling_GB/s"],
                                "note": k.get("fp32_note")}
    return roof, kernels


def ssim_kernels(sets, px, nsets, reps):
    """The SSIM kernels of a forward + backward step, each timed alone.  The FP32-FMA ceiling (SURVEY.md 8d: the 11-tap
    separable passes cost more FMAs per byte than the HBM ridge) is printed beside the HBM numbers."""
    import torch
    from b200wave import ops
    from b200wave.ssim import _win_taps
    win = _win_taps(11)
    dev = sets[0][0].device
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    try:
        import pynvml
        pynvml.nvmlInit()
        mhz = pynvml.nvmlDeviceGetMaxClockInfo(pynvml.nvmlDeviceGetHandleByIndex(dev.index or 0), pynvml.NVML_CLOCK_SM)
    except Exception:
        mhz = 1965
    fma_per_s = sms * 128 * mhz * 1e6   # scalar FP32 FMA lanes of the whole chip
    out = {}
    for key, fn, nbytes, fma_px in ops.ssim_bench_kernels(sets, win):
        t = time_kernel(fn, nsets, reps)
        ceil_px_s = fma_per_s / fma_px
        out[key] = {"s": t, "GB/s": nbytes * px / t / 1e9, "bytes": nbytes * px, "Gpx/s": px / t / 1e9,
                    "fp32_ceiling_GB/s": nbytes * ceil_px_s / 1e9,
                    "fp32_note": "%d FP32-pipe lane operations per pixel (FFMA2 = 2) on %d SMs x 128 lanes x %d MHz" % (fma_px, sms, mhz),
                    "sass": next((k for k in __import__("b200wave")._cabi.recent_kernels(2) if "stream" in k), None)}
    return out


def run_value(step, sets, steps, warmup, use_graph):
    """Device-resident timing of `steps` steps rotating over the input sets; returns (ms total, graphs or None)."""
    import torch
    nsets = len(sets)
    graphs = None
    if use_graph:
        try:
            graphs = capture_graphs(step, sets)
        except Exception as e:  # pragma: no cover
            print("graph capture failed, timing eager launches: %r" % (e,), file=sys.stderr)
            graphs = None

    def run_step(i):
        """Runs step i; returns its outputs (for a replay, the graph's output tensors, which it has just rewritten)."""
        if graphs is not None:
            graphs[i % nsets][0].replay()
            return graphs[i % nsets][1]
        return step(*sets[i % nsets])
    return run_step, graphs


def reference_gpu_leg(name, dev, steps=10):
    """The unmodified reference modules on this GPU (eager: its padding builds index arrays on the host every call,
    so it cannot be graph-captured), CUDA events around `steps` steps after 3 warm-up steps."""
    import torch
    from oracle import ref_runner
    if not ref_runner.available():
        return {"unavailable": "oracle/_ref not staged (make -C oracle ref)"}
    cfg = WORKLOADS[name]

    class Mods(object):
        pass
    pw, ss = ref_runner.load()
    Mods.DWTForward, Mods.DWTInverse, Mods.SSIM = pw.DWTForward, pw.DWTInverse, ss.SSIM
    try:
        step, make_set, set_bytes, _, _ = build_step(cfg, dev, Mods)
        nsets = max(2, -(-2 * L2_BYTES // set_bytes))
        sets = [make_set() for _ in range(nsets)]
        for i in range(3):
            step(*sets[i % nsets])
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            step(*sets[i % nsets])
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        n, c, h, w = cfg["shape"]
        del sets
        torch.cuda.empty_cache()
        return {"ms_per_step": ms, "value": n * c * h * w / 1e6 / (ms / 1e3), "unit": UNIT, "steps": steps,
                "impl": "unmodified pytorch_wavelets / ssim.py (oracle/_ref) on cuda, eager, same step and shapes"}
    except Exception as e:  # pragma: no cover
        return {"unavailable": "reference failed on cuda: %r" % (e,)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-workloads", action="store_true", help="skip the secondary workloads / reference_gpu legs")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replays")
    ap.add_argument("--e2e-chunks", type=int, default=1,
                    help="batch chunks of the host-buffer pipeline (e2e); consecutive steps already overlap their "
                         "uploads and downloads, and one chunk per step measured best (profiles/r01_notes.md)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of the headline workload as DIR/<name>.npy "
                         "(a fixed sample of an output that does not fit %d MB)" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = WORKLOADS[args.workload]

    if args.impl == "reference":
        if rank != 0:
            return 0
        base = cpu_reference(args.workload, args.steps, args.warmup)
        line = {"metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": base["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": cfg["desc"]}, "impl": "reference",
                "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    import b200wave

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    saved_stdout = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # keep stdout to the one JSON line: NCCL printf()s its version banner there when the first communicator is
        # created, so file descriptor 1 points at stderr until the line is printed
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)

    n, c, h, w = cfg["shape"]
    mpix_step = n * c * h * w / 1e6
    torch.manual_seed(1234 + rank)
    from b200wave import _cabi
    peak, peak_src = hbm_peak()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def measure(name, wcfg, steps, warmup, with_e2e, dump_dir=None):
        """value (+ e2e) of one workload on every rank, max over ranks; the kernel rooflines on rank 0; with dump_dir,
        rank 0 writes the outputs of the last timed step there."""
        wn, wc, wh, ww = wcfg["shape"]
        step, make_set, set_bytes, step_bytes, extras = build_step(wcfg, dev, b200wave)
        nsets = max(2, -(-2 * L2_BYTES // set_bytes))  # inputs alone exceed 2x L2 across the rotation
        sets = [make_set() for _ in range(nsets)]
        # warm-up (also fills the host tap cache so graph capture never synchronises)
        for i in range(max(3, min(warmup, nsets))):
            step(*sets[i % nsets])
        torch.cuda.synchronize()
        before = _cabi.kernel_launches()
        step(*sets[0])
        torch.cuda.synchronize()
        per_step = _cabi.kernel_launches() - before
        if per_step <= 0:
            raise RuntimeError("the step launched none of the library's kernels: refusing to report a number")
        step_kernels = _cabi.recent_kernels(per_step)
        run_step, graphs = run_value(step, sets, steps, warmup, not args.no_graph)
        for i in range(warmup):
            run_step(i)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            out = run_step(i)
        ev1.record()
        barrier()
        ms = all_max(ev0.elapsed_time(ev1))
        dumped = dump_outputs(dump_dir, step_output_names(wcfg), out) if dump_dir and rank == 0 else None
        res = {"desc": wcfg["desc"], "ms_per_step": ms / steps, "steps": steps,
               "value": world * wn * wc * wh * ww / 1e6 * steps / (ms / 1e3), "unit": UNIT,
               "step_algorithmic_bytes": step_bytes, "step_hbm_frac": (step_bytes / (ms / steps * 1e-3) / 1e9) / peak,
               "gpu_launches_per_step": per_step, "step_kernels": step_kernels,
               "replay": "cuda-graph" if graphs is not None else "eager",
               "l2": "rotating %d input sets (%.0f MB) > 2x 126 MB L2; outputs re-allocated per set"
                     % (nsets, nsets * set_bytes / 1e6)}
        if dumped is not None:
            res["dump_outputs"] = dumped
        if with_e2e:
            # The public host-buffer call (b200wave.HostPipeline): every step copies that step's inputs from pinned
            # host memory, runs the same step, and copies the results back; H2D copy, kernels and D2H copy overlap
            # on three streams and consecutive steps stream through those queues back to back.
            from b200wave import HostPipeline
            host_in = [tuple(t.detach().cpu().pin_memory().requires_grad_(t.requires_grad) for t in s) for s in sets[:2]]
            chunks = 1 if wcfg["kind"] == "ssim" else args.e2e_chunks   # a scalar mean does not split into chunks
            pipe = HostPipeline(step, host_in[0], chunks=chunks, graph=not args.no_graph)
            h2d, d2h = pipe.bytes_per_call(host_in[0])
            e2e_steps = max(3, min(steps, 50))
            for i in range(3):
                pipe(host_in[i % len(host_in)], sync=False)
            pipe.join()
            barrier()
            ev0.record()
            for i in range(e2e_steps):
                pipe(host_in[i % len(host_in)], sync=False)   # steps stream through the three queues back to back
            pipe.join()              # the timed region ends when the last step's results are in host memory
            ev1.record()
            barrier()
            e2e_ms = all_max(ev0.elapsed_time(ev1))
            res["e2e"] = {"value": world * wn * wc * wh * ww / 1e6 * e2e_steps / (e2e_ms / 1e3), "unit": UNIT,
                          "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / e2e_steps,
                          "steps": e2e_steps,
                          "api": "b200wave.HostPipeline(step, chunks=%d): pinned host -> H2D | kernels | D2H overlapped "
                                 "on three streams" % len(pipe.bounds)}
            gbs, src = host_copy_bound(world)
            if gbs:   # the step cannot be faster than its own copies at the box's measured duplex copy rate
                bound_ms = max(h2d, d2h) / (gbs * 1e9) * 1e3
                res["e2e"]["host_bound"] = {"duplex_gbs_per_rank_per_direction": gbs, "bound_ms_per_step": bound_ms,
                                            "source": src,
                                            "note": "probe taken on one box of the pool; boxes differ by +-30 % at "
                                                    "N > 1, so a fraction above 1 means this box's host side is faster"}
                res["e2e"]["frac_of_host_bound"] = bound_ms / (e2e_ms / e2e_steps)
            del pipe, host_in
        if rank == 0:
            graphs = None   # free the pools before the kernel timings allocate their own
            res["roofline"], res["kernels"] = kernel_rooflines(name, wcfg, sets, extras, max(20, min(steps, 100)),
                                                               peak, peak_src)
        del sets
        torch.cuda.empty_cache()
        return res

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    main_res = measure(args.workload, cfg, args.steps, args.warmup, True, args.dump_outputs)
    clocks = sampler.stop() if sampler else None

    # the other BASELINE configs, device-resident value + roofline each (every rank runs them so that the per-rank
    # work stays symmetric; they are skipped under --no-workloads)
    others = {}
    if not args.no_workloads:
        for name in SECONDARY:
            if name == args.workload:
                continue
            try:
                r = measure(name, WORKLOADS[name], max(5, min(args.steps, 30)), 3, False)
                others[name] = {k: r[k] for k in ("desc", "ms_per_step", "value", "unit", "step_hbm_frac", "steps",
                                                  "gpu_launches_per_step", "step_kernels") if k in r}
                if "roofline" in r:
                    others[name]["roofline"] = r["roofline"]
                    others[name]["kernels"] = r["kernels"]
            except Exception as e:  # pragma: no cover
                others[name] = {"error": repr(e)}

    ref_gpu = None
    cpu = None
    if rank == 0 and world == 1:
        if not args.no_workloads:
            ref_gpu = {name: reference_gpu_leg(name, dev) for name in ("cfg2", "cfg3")}
        if not args.no_cpu_baseline:
            cpu = cpu_reference(args.workload, steps=5, warmup=1, budget_s=15.0)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    elif rank == 0:
        cpu = {"skipped": "n_gpus > 1: the CPU baseline is reported by the N=1 run only"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": main_res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["desc"], "per_gpu_batch": n, "global_batch": n * world,
                       "parallelism": "batch-sharded x%d, no data-path collective" % world,
                       "replay": main_res["replay"], "l2": main_res["l2"]},
            "step_algorithmic_bytes": main_res["step_algorithmic_bytes"],
            "step_hbm_frac": main_res["step_hbm_frac"],
            "e2e": main_res["e2e"],
            "gpu_launches": main_res["gpu_launches_per_step"] * args.steps, "step_kernels": main_res["step_kernels"],
            "roofline": main_res.get("roofline"), "kernels": main_res.get("kernels"),
            "workloads": others, "reference_gpu": ref_gpu, "cpu_baseline": cpu, "clocks": clocks,
            "library_build": _cabi.build_hash(),
        }
        if "dump_outputs" in main_res:
            line["dump_outputs"] = {"dir": args.dump_outputs, "arrays": main_res["dump_outputs"]}
        if saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
