"""Time lost between the chain kernels of the cfg2 step.

    python tools/gapbench.py [--reps N] [--rounds R]

The cfg2 step of bench.py (DWTForward(J=3, db3, symmetric) -> DWTInverse -> backward through both, 64x1x304x304)
launches four chain kernels: analysis, synthesis, analysis, synthesis.  This tool times, over rotating inputs that
together exceed 2x the 126 MB L2, each inside one CUDA graph of N launches / steps, with CUDA events:
  (a) the analysis chain (DWTForward) launched back to back alone, and the synthesis chain (DWTInverse) likewise;
  (b) the step itself, built through the public modules exactly as bench.py builds it;
  (c) (b) against sum(a) = 2 x analysis + 2 x synthesis: what alternating the two kernels costs beyond their own
      launch-to-launch time.
It repeats the three timings R times (interleaved) and prints every round and the medians, with the card's name, power
limit and SM clock.
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import b200wave  # noqa: E402
import bench  # noqa: E402

L2_BYTES = 126 * 1024 * 1024


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), (s.strip() for s in out.split(","))))
    except Exception as e:   # the numbers still stand with the torch device name
        return {"name": torch.cuda.get_device_name(0), "power.limit": "unknown (%s)" % e}


def graph_time(fn, nsets, reps):
    """Mean time of one fn(i) over `reps` calls captured into one CUDA graph (outputs kept alive for one rotation)."""
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
    times = []
    for _ in range(3):
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) / reps * 1e3)
    del keep, g
    return statistics.median(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200, help="launches / steps per graph")
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "gapbench needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.manual_seed(1234)
    cfg = bench.WORKLOADS["cfg2"]
    step, make_set, set_bytes, _, extras = bench.build_step(cfg, dev, b200wave)
    xfm, ifm = extras["xfm"], extras["ifm"]
    nsets = max(2, -(-2 * L2_BYTES // set_bytes))
    sets = [make_set() for _ in range(nsets)]
    with torch.no_grad():
        coeffs = [xfm(s[0].detach()) for s in sets]
    from b200wave import _cabi

    def t_afb():
        with torch.no_grad():
            return graph_time(lambda i: xfm(sets[i % nsets][0].detach()), nsets, args.reps)

    def t_sfb():
        with torch.no_grad():
            return graph_time(lambda i: ifm(coeffs[i % nsets]), nsets, args.reps)

    def t_step():
        return graph_time(lambda i: step(*sets[i % nsets]), nsets, args.reps)

    print("card:", card())
    print("cfg2: %s, %d rotating input sets (%.0f MB), %d launches / steps per graph" % (
        cfg["desc"], nsets, nsets * set_bytes / 1e6, args.reps))
    before = _cabi.kernel_launches()
    step(*sets[0])
    torch.cuda.synchronize()
    print("step kernels:", _cabi.recent_kernels(_cabi.kernel_launches() - before))
    rows = []
    for r in range(args.rounds):
        a, s, b = t_afb(), t_sfb(), t_step()
        rows.append((a, s, b))
        print("round %d: (a) analysis %.2f us, synthesis %.2f us; (b) step %.2f us; sum(a) %.2f us; (c) b - sum(a) %.2f us"
              % (r, a, s, b, 2 * a + 2 * s, b - 2 * a - 2 * s), flush=True)
    med = [statistics.median(x) for x in zip(*rows)]
    a, s, b = med
    print("median: (a) analysis %.2f us, synthesis %.2f us; (b) step %.2f us; sum(a) %.2f us; (c) b - sum(a) %.2f us"
          % (a, s, b, 2 * a + 2 * s, b - 2 * a - 2 * s))
    print("card after:", card())


if __name__ == "__main__":
    main()
