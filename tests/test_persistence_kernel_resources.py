"""Static checks of the persistence histogram kernel (cuobjdump on libsa_engine.so, no GPU needed): both tile widths
keep their counters in shared memory and everything else in registers."""
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


def test_histogram_kernel_does_not_spill():
    hist = {k: v for k, v in res_usage().items() if "persistence_hist_kernel" in k}
    assert len(hist) == 2, sorted(hist)                     # 64- and 128-bin tiles
    for name, r in hist.items():
        assert r["STACK"] == 0 and r["LOCAL"] == 0, (name, r)
        assert r["REG"] <= 64, (name, r)                    # 1024 threads per CTA
