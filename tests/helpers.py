"""Shared helpers for the test-suite (oracle access, golden-case loading, error metric)."""
import glob
import io
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# north_star tolerance: 1e-5 relative (fp32), measured as max|a-b| / max|b| per tensor (BASELINE.md 5)
RTOL_F32 = 1e-5

# every golden file stays below 1 MB; a set that does not fit is written as several parts
GOLDEN_FILE_BYTES = 1000 * 1000


def _golden_paths(name):
    single = os.path.join(GOLDEN, name + ".npz")
    parts = glob.glob(os.path.join(GOLDEN, name + ".[0-9]*.npz"))
    return [single] if os.path.exists(single) else sorted(parts, key=lambda p: int(p.rsplit(".", 2)[1]))


def _npz_bytes(arrays):
    buf = io.BytesIO()
    np.savez_compressed(buf, **arrays)
    return buf.tell()


def save_golden(name, arrays):
    """Writes the golden set ``name`` (a dict of arrays) as tests/golden/<name>.npz, or, when that file would not stay
    under GOLDEN_FILE_BYTES, as <name>.1.npz, <name>.2.npz, ... each holding whole arrays.  load_golden reads either
    form."""
    for p in _golden_paths(name):
        os.remove(p)
    parts = [arrays]
    if _npz_bytes(arrays) >= GOLDEN_FILE_BYTES:
        parts, cur, cur_bytes = [], {}, 0
        for key, value in arrays.items():
            size = _npz_bytes({key: value})
            if cur and cur_bytes + size > 0.9 * GOLDEN_FILE_BYTES:
                parts.append(cur)
                cur, cur_bytes = {}, 0
            cur[key] = value
            cur_bytes += size
        parts.append(cur)
    names = [name + ".npz"] if len(parts) == 1 else ["%s.%d.npz" % (name, i + 1) for i in range(len(parts))]
    for fname, part in zip(names, parts):
        path = os.path.join(GOLDEN, fname)
        np.savez_compressed(path, **part)
        assert os.path.getsize(path) < GOLDEN_FILE_BYTES, (path, "one array alone is too large for a golden file")
    return names


def load_golden(name):
    """The arrays of the golden set ``name`` written by save_golden, as a dict."""
    paths = _golden_paths(name)
    if not paths:
        raise FileNotFoundError("no golden set %r under %s" % (name, GOLDEN))
    out = {}
    for p in paths:
        with np.load(p) as z:
            out.update((k, z[k]) for k in z.files)
    return out


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    denom = np.abs(b).max()
    if denom == 0:
        return np.abs(a).max()
    return np.abs(a - b).max() / denom


def load_dwt_cases():
    z = load_golden("dwt_cases")
    n = int(z["ncases"])
    cases = []
    for i in range(n):
        pre = "c%02d/" % i
        case = {k[len(pre):]: z[k] for k in z if k.startswith(pre)}
        case["J"] = int(case["J"])
        case["mode"] = str(case["mode"])
        case["wave"] = str(case["wave"])
        case["id"] = "%02d-%s-J%d-%s-%dx%d" % (i, case["wave"], case["J"], case["mode"],
                                               case["x"].shape[-2], case["x"].shape[-1])
        cases.append(case)
    return cases


def load_ssim_cases():
    z = load_golden("ssim_cases")
    n = int(z["ncases"])
    cases = []
    for i in range(n):
        pre = "s%02d/" % i
        case = {k[len(pre):]: z[k] for k in z if k.startswith(pre)}
        case["size_average"] = bool(case["size_average"])
        case["id"] = "%02d-sa%d" % (i, case["size_average"])
        cases.append(case)
    return cases


def case_filters(case):
    """(h_col, h_row, g_col, g_row) pairs of prepped taps as the reference's buffers hold them."""
    return ((case["h0_col"], case["h1_col"]), (case["h0_row"], case["h1_row"]),
            (case["g0_col"], case["g1_col"]), (case["g0_row"], case["g1_row"]))


def load_freq_cases():
    z = load_golden("freq_cases")
    cases = []
    for i in range(int(z["ncases"])):
        pre = "f%02d/" % i
        case = {k[len(pre):]: z[k] for k in z if k.startswith(pre)}
        case["radius"] = int(case["radius"])
        case["highpass"] = bool(case["highpass"])
        case["id"] = "%02d-%s-r%d-%dx%d" % (i, "high" if case["highpass"] else "low", case["radius"],
                                            case["x"].shape[-2], case["x"].shape[-1])
        cases.append(case)
    return cases


def load_fsd_cases():
    z = load_golden("fsd_cases")
    cases = []
    for i in range(int(z["ncases"])):
        pre = "w%02d/" % i
        case = {k[len(pre):]: z[k] for k in z if k.startswith(pre)}
        case["variant"] = str(case["variant"])
        case["cs"] = str(case["cs"])
        case["norm"] = bool(case["norm"])
        n = int(case["nbands"])
        case["y"] = [case["y%d" % b] for b in range(n)]
        case["g"] = [case["g%d" % b] for b in range(n)]
        case["id"] = "%02d-%s-%s-norm%d-%dx%d" % (i, case["variant"], case["cs"], case["norm"],
                                                  case["x"].shape[-2], case["x"].shape[-1])
        cases.append(case)
    return cases


def load_tv_cases():
    z = load_golden("tv_cases")
    cases = []
    for i in range(int(z["ncases"])):
        pre = "t%02d/" % i
        case = {k[len(pre):]: z[k] for k in z if k.startswith(pre)}
        case["weight"] = float(case["weight"])
        case["loss"] = float(case["loss"])
        case["id"] = "%02d-%s-w%g" % (i, "x".join(str(d) for d in case["x"].shape), case["weight"])
        cases.append(case)
    return cases


def load_phase_cases():
    z = load_golden("phase_cases")
    cases = []
    for i in range(int(z["ncases"])):
        pre = "p%02d/" % i
        case = {k[len(pre):]: z[k] for k in z if k.startswith(pre)}
        case["loss"] = float(case["loss"])
        case["id"] = "%02d-%s" % (i, "x".join(str(d) for d in case["x"].shape))
        cases.append(case)
    return cases


def load_dwt1d_cases():
    z = load_golden("dwt1d_cases")
    cases = []
    for i in range(int(z["ncases"])):
        pre = "d%02d/" % i
        case = {k[len(pre):]: z[k] for k in z if k.startswith(pre)}
        case["J"] = int(case["J"])
        case["mode"] = str(case["mode"])
        case["wave"] = str(case["wave"])
        case["id"] = "%02d-%s-J%d-%s-%d" % (i, case["wave"], case["J"], case["mode"], case["x"].shape[-1])
        cases.append(case)
    return cases


def load_swt_cases():
    z = load_golden("swt_cases")
    cases = []
    pres = sorted({k.split("/")[0] for k in z if "/" in k})
    for pre in pres:
        case = {k[len(pre) + 1:]: z[k] for k in z if k.startswith(pre + "/")}
        case["mode"], case["wave"], case["dilation"] = str(case["mode"]), str(case["wave"]), int(case["dilation"])
        case["id"] = "%s-%s-%s-d%d-%dx%d" % (pre, case["wave"], case["mode"], case["dilation"], case["x"].shape[-2],
                                             case["x"].shape[-1])
        cases.append(case)
    return cases
