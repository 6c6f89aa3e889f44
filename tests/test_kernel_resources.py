"""Static checks of the built sm_100a code (cuobjdump on libsa_engine.so, no GPU needed): the resource budgets the
occupancy plans in DESIGN.md rely on, and the SASS mnemonics that show the Blackwell features the design claims
(TMA bulk copies completing on mbarriers, packed FP32, cp.async staging) are really in the kernels that claim them."""
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
    res = {}
    for name, line in re.findall(r"Function (\S+):\n\s*(REG:.*)", out):
        res[name] = {k: int(v) for k, v in re.findall(r"(\w+)(?:\[0\])?:(\d+)", line)}
    return res


def sass(mangled):
    return subprocess.run(["cuobjdump", "-sass", "-fun", mangled, LIB], capture_output=True, text=True, timeout=300).stdout


RES = None


def get_res():
    global RES
    if RES is None:
        RES = res_usage()
    return RES


def test_only_sm_100a_code_is_shipped():
    out = subprocess.run(["cuobjdump", "-lelf", LIB], capture_output=True, text=True, timeout=300).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_register_and_stack_budgets():
    res = get_res()
    assert len(res) > 150
    spec = {k: v for k, v in res.items() if "spectrogram_" in k and "kernel" in k}
    # headline: 128 registers -> one 512-thread CTA per SM (4 warps per scheduler), nothing spilled
    head = {k: v for k, v in spec.items() if "spectrogram_tma_kernelIfLi1024E" in k}
    assert len(head) >= 6
    for k, v in head.items():
        assert v["REG"] <= 128 and v["STACK"] == 0 and v["LOCAL"] == 0, (k, v)
    # small-radix-first kernels (2048..16384): 512-thread CTAs need <= 128 registers, no spills
    for k, v in spec.items():
        if "spectrogram_mid_kernel" in k:
            assert v["REG"] <= 128 and v["STACK"] == 0, (k, v)
    # radix-64 kernel: 64 points per thread is a deliberate 255-register design with a bounded spill
    r64 = {k: v for k, v in spec.items() if "spectrogram_r64_kernel" in k}
    assert r64 and all(v["REG"] <= 255 and v["STACK"] <= 256 for v in r64.values()), r64
    # no kernel anywhere keeps a large local frame
    worst = max(res.items(), key=lambda kv: kv[1]["STACK"])
    assert worst[1]["STACK"] <= 256, worst
    # downconverter: 64 registers -> 4 CTAs of 256 threads per SM; the pipelined variant (template flag PIPE, "ELb1ELb1E")
    # carries the next tile's 17 raw samples in registers: <= 85 registers -> 3 CTAs per SM; its cf32 instance ("ILi0E")
    # is software-pipelined at 2 CTAs per SM (<= 128 registers, no spills)
    dc = {k: v for k, v in res.items() if "downconvert_kernel" in k}
    assert dc and any("ELb1ELb1E" in k for k in dc)
    def budget(k):
        if "ELb1ELb1E" not in k:
            return 64, 64
        return (128, 0) if "kernelILi0E" in k else (85, 64)
    assert all(v["REG"] <= budget(k)[0] and v["STACK"] <= budget(k)[1] for k, v in dc.items()), dc


def count(text, pattern):
    return len(re.findall(pattern, text))


def test_headline_kernel_uses_tma_mbarrier_and_packed_fp32():
    s = sass("_ZN2sa22spectrogram_tma_kernelIfLi1024ELi0ELb1EEEvNS_8SpecArgsE")      # <float, 1024, cf32, window>
    assert count(s, r"\bUBLKCP") >= 1                      # cp.async.bulk global -> shared (TMA 1-D)
    assert count(s, r"SYNCS\.ARRIVE\.TRANS64") >= 1 and count(s, r"SYNCS\.PHASECHK\.TRANS64\.TRYWAIT") >= 1
    assert count(s, r"\bFFMA2\b") >= 100 and count(s, r"\bFADD2\b") >= 50 and count(s, r"\bFMUL2\b") >= 30
    assert count(s, r"\bMUFU\.LG2\b") >= 32                # one log2 per bin of the thread
    assert count(s, r"\bLDL\b|\bSTL\b") == 0


def test_radix64_kernel_is_tma_staged_and_mid_kernel_uses_cp_async():
    r64 = sass("_ZN2sa22spectrogram_r64_kernelILi1ELb1EEEvNS_8SpecArgsE")           # ci16, window: BASELINE config 2
    assert count(r64, r"\bUBLKCP") >= 1 and count(r64, r"\bFFMA2\b") >= 200
    res = get_res()
    mid = [k for k in res if "spectrogram_mid_kernelILi2048ELi2ELb0ELb1E" in k]     # cu8 2048 rect, staged: config 4
    assert mid, "config-4 kernel missing"
    s = sass(mid[0])
    assert count(s, r"\bLDGSTS") >= 1                      # cp.async global -> shared staging of the next frame
    assert count(s, r"\bFFMA2\b") >= 100
    assert count(s, r"\bF2I|\bI2F") == 0                   # integer decode and pixel rounding stay on the FMA pipe


def test_row_downconverter_stages_by_cp_async_and_reads_taps_from_the_constant_bank():
    """downconvert_rows_kernel<D, MODE, NT, NBUF>: the raw tile arrives by 16-byte cp.async (LDGSTS.128), the shipped
    variant (MODE 1) has no table loads in its tap loop -- its only shared-memory loads are the raw row (D/2 LDS.128 per
    row and tile variant), the partial sums and nothing else -- and multiplies by taps held in uniform registers loaded
    from the kernel-parameter bank (FFMA ..., UR..)."""
    res = get_res()
    rows = {k: v for k, v in res.items() if "downconvert_rows_kernel" in k}
    assert len(rows) >= 16                                   # D in {4, 8, 16, 32} x (table variant + four shapes)
    for k, v in rows.items():
        assert v["REG"] <= 128 and v["STACK"] <= 64, (k, v)
    name = "_ZN2sa23downconvert_rows_kernelILi0ELi16ELi1ELi128ELi2ELb1EEEvNS_6DcArgsENS_10DcRowsTapsIXT0_EEE"     # C3: cf32, D 16, 128 rows, 2 buffers, swizzled
    assert name in rows and rows[name]["STACK"] == 0 and rows[name]["REG"] <= 80, sorted(rows)      # 6 CTAs of 128 threads per SM
    s = sass(name)
    assert count(s, r"\bLDGSTS\.E\.BYPASS\.128") >= 8          # 8 chunks per thread and tile
    assert count(s, r"\bFFMA R\d+, R\d+(\.reuse)?, UR\d+, R\d+") >= 1800                # ~16 taps x 16 samples x (2 parities x 2 edge variants x 2 byte orders); a few taps ride in vector registers
    assert count(s, r"\bLDS\.128") == 8 * 8                   # the raw row only: 8 chunks x 8 variants of the tap loop (parity, edge, byte order)
    fast = {k: v for k, v in res.items() if "downconvert_rows_fast_kernel" in k}      # box-car mode: 3 CTAs of 128 threads, no spills
    assert len(fast) == 3 and all(v["REG"] <= 128 and v["STACK"] == 0 for v in fast.values()), fast
    table = sass("_ZN2sa23downconvert_rows_kernelILi0ELi16ELi0ELi256ELi1ELb0EEEvNS_6DcArgsENS_10DcRowsTapsIXT0_EEE")
    assert count(table, r"\bLDS\.128") >= 2 * (8 + 3 * 16)     # the ablation variant reads taps and NCO phasors as tables


def test_no_tensor_core_or_library_fft_code():
    out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, timeout=600).stdout
    # DESIGN section 4: no DFT-as-GEMM stage is shipped.  The ONLY kernel with tensor-core / TMEM instructions is the
    # ablation kernel of csrc/tc_ablation.cu (tcgen05.mma -> UTCHMMA, tcgen05.ld -> LDTM), which no product entry point launches.
    per_fn, fn = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = m.group(1)
        elif fn and re.search(r"\b(HMMA|IMMA|UTCHMMA|UTCQMMA|UTCIMMA|QGMMA|LDTM)\b", line):
            per_fn[fn] = per_fn.get(fn, 0) + 1
    assert set(per_fn) == {k for k in per_fn if "tc_spectrogram_kernel" in k} and len(per_fn) == 1, per_fn
    abl = next(iter(per_fn))
    body = out[out.index(abl):]
    body = body[:body.index("Function :", 10)] if "Function :" in body[10:] else body
    assert count(body, r"\bUTCHMMA\b") >= 1 and count(body, r"\bLDTM\b") >= 2          # tcgen05.mma kind::tf32, tcgen05.ld
    syms = subprocess.run(["nm", "-D", LIB], capture_output=True, text=True).stdout
    assert "cufft" not in syms.lower()
