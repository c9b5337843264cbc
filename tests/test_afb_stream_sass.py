"""CPU: what the compiler makes of the analysis stream and owner kernels (csrc/dwt_stream_afb.cu).  The stream kernel
is built per filter length L and window shift S for two global copy widths: V = 4 (one 16-byte cp.async per ring
slot, rows 16-byte aligned) and V = 1 (four 4-byte cp.async, any other rows).  The 16-byte instantiations, which
every aligned input runs, keep their registers, spills and instruction count; a 4-byte one exists for every L the
templated kernels serve."""
import re

import pytest

from b200wave import _build
from test_f64_host import _compile, _nvcc_is_12_9

# (L, S): (registers, SASS instructions) with nvcc 12.9, -O3; none of them spills
STREAM_16B = {(2, 0): (48, 1000), (4, 2): (71, 1472), (4, 3): (72, 1488), (6, 0): (92, 2016), (6, 2): (92, 2040),
              (8, 1): (96, 2960), (8, 2): (96, 2968), (10, 0): (128, 2712), (12, 2): (128, 3344),
              (12, 3): (128, 3360), (14, 0): (168, 4008), (14, 2): (168, 4016), (16, 1): (168, 4696),
              (16, 2): (168, 4704)}
OWNER = {(2, 0): (105, 1168), (4, 2): (139, 1760), (4, 3): (139, 1784), (6, 0): (148, 2552), (6, 2): (146, 2568),
         (8, 1): (168, 3680), (8, 2): (168, 3680), (10, 0): (213, 2768), (12, 2): (219, 3288), (12, 3): (219, 3344),
         (14, 0): (255, 3888), (14, 2): (255, 3912), (16, 1): (255, 4624), (16, 2): (255, 4624)}


@pytest.mark.skipif(_build.find_nvcc() is None, reason="needs nvcc")
def test_stream_and_owner_kernels_by_copy_width(tmp_path):
    info, ninstr = _compile("dwt_stream_afb.cu", tmp_path)
    stream, owner = {}, {}
    for name in info:
        m = re.search(r"afb_stream_kernelILi(\d+)ELi(\d+)ELi(\d+)EEEv", name)
        if m:
            stream[tuple(int(g) for g in m.groups())] = name
        m = re.search(r"afb_owner_kernelILi(\d+)ELi(\d+)EEEv", name)
        if m:
            owner[(int(m.group(1)), int(m.group(2)))] = name
    assert sorted(k[:2] for k in stream if k[2] == 4) == sorted(STREAM_16B), sorted(stream)
    assert sorted(owner) == sorted(OWNER), sorted(owner)
    assert {k[2] for k in stream} == {1, 4}, sorted(stream)
    assert {k[0] for k in stream if k[2] == 1} == set(range(2, 17, 2)), sorted(stream)
    for (L, S, V), name in stream.items():
        if V == 4 or L <= 8:   # 4-byte copies: haar .. db4 must not spill
            assert info[name]["spill"] == (0, 0), ((L, S, V), info[name])
    for name in owner.values():
        assert info[name]["spill"] == (0, 0), (name, info[name])
    if not _nvcc_is_12_9():
        return
    for (L, S), want in STREAM_16B.items():
        name = stream[(L, S, 4)]
        assert (info[name]["regs"], ninstr[name]) == want, ((L, S), info[name], ninstr[name])
    for key, want in OWNER.items():
        name = owner[key]
        assert (info[name]["regs"], ninstr[name]) == want, (key, info[name], ninstr[name])
