"""CPU: the TMA analysis kernel is built for two parameter-block sizes (table capacities kAfbTabSmall and kAfbTabMax,
csrc/dwt_tma.cuh).  The launch picks the smaller block when the plan's tables fit in it, so the two instantiations of
every filter length must be the same code: same registers, same spills, same instruction count."""
import re

import pytest

from b200wave import _build
from test_f64_host import _compile


@pytest.mark.skipif(_build.find_nvcc() is None, reason="needs nvcc")
def test_both_parameter_blocks_compile_to_the_same_kernel(tmp_path):
    info, ninstr = _compile("dwt_tma_afb.cu", tmp_path)
    by_size = {}
    for name in info:
        m = re.search(r"afb_tma_kernelILi(\d+)ELi(\d+)ELi(\d+)E", name)
        if m:
            by_size.setdefault((int(m.group(1)), int(m.group(2))), {})[int(m.group(3))] = name
    assert len(by_size) == 15, sorted(by_size)   # L = 2, 4, .., 16; both extensions for L >= 4
    for key, sizes in by_size.items():
        assert sorted(sizes) == [2048, 5120], (key, sizes)
        small, large = sizes[2048], sizes[5120]
        assert info[small] == info[large], (key, info[small], info[large])
        assert ninstr[small] == ninstr[large], (key, ninstr[small], ninstr[large])
        if key[0] <= 8:   # haar .. db4
            assert info[small]["spill"] == (0, 0), (key, info[small])
