"""Static checks of the spectrum-trace kernels (cuobjdump on libsa_engine.so, no GPU needed): trace_finalize_kernel and
the pooled four-step rows kernels (large_rows_kernel<.., POOL = true>) keep everything in registers."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "spectral_analyzer_b200", "libsa_engine.so")
pytestmark = pytest.mark.skipif(not shutil.which("cuobjdump") or not os.path.exists(LIB), reason="needs cuobjdump + the built library")


def res_usage():
    out = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, timeout=300).stdout
    return {name: {k: int(v) for k, v in re.findall(r"(\w+)(?:\[0\])?:(\d+)", line)}
            for name, line in re.findall(r"Function (\S+):\n\s*(REG:.*)", out)}


def test_trace_kernels_do_not_spill():
    res = res_usage()
    fin = {k: v for k, v in res.items() if "trace_finalize_kernel" in k}
    pooled = {k: v for k, v in res.items() if re.match(r"_ZN2sa17large_rows_kernelI[fd]Li\d+ELi\d+ELb1EEEv", k)}
    assert len(fin) == 2, sorted(fin)                       # FP32 and FP64 cells
    assert len(pooled) == 5, sorted(pooled)                 # FP32 32768 / 65536, FP64 16384 / 32768 / 65536
    for name, r in {**fin, **pooled}.items():
        assert r["STACK"] == 0 and r["LOCAL"] == 0, (name, r)
