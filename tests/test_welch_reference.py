"""CPU checks of the Welch test support (tests/welch_reference.py): the block-tone input and the norm-wise comparator
reject every indexing mistake a Welch kernel can make by at least 100x the bound of the kernel family the case's nfft
selects, accept an FP32 Welch, and the numpy and C references agree.  tests/test_gpu_welch_matrix.py relies on all
three.

One exception: the FP32 direct DFT kernel's bound grows with sqrt(nfft) (30 sqrt(nfft) 2^-24, 1.9e-4 at 11000 points),
while a one-sample shift or the symmetric window changes a smooth-windowed segment by O(1/nfft).  At direct-kernel
sizes those two mutants are held to 10x the bound; every mistake in which segments are read stays at 100x."""
import numpy as np
import pytest

import welch_reference as wr
from util import NORM_TOL_F32, frame_norm_error

FS = 2.0e6
# (nfft, hop, window, detrend, stride): stride = segments between one slot's consecutive steps (nsplit x FPC)
CASES = [(64, 16, "hann", None, 64), (256, 256, "blackman_harris", "constant", 32), (512, 301, "hamming", "constant", 48),
         (128, 160, "rect", None, 64), (2048, 1024, "hann", None, 16), (16384, 8192, "blackman", "constant", 3),
         (1000, 250, "hann", "constant", 4), (11000, 8000, "blackman", "constant", 4)]
SUBTLE = ("shifted by one", "symmetric window")


def bound(nfft):
    """the bound of the FP32 kernel engine.psd_welch picks for nfft"""
    return wr.tol_of(wr.kernel_of("f32", nfft)[0], nfft)


def margin(nfft, mutant):
    direct = wr.kernel_of("f32", nfft)[0] == "psd_direct_kernel<float>"
    return 10 if direct and mutant in SUBTLE else 100


def err(got, ref):
    return float(frame_norm_error(got[None], ref[None])[0])


def case_input(nfft, hop, detrend, nseg):
    # blocks of half a hop: a block boundary inside every segment, also when the hop leaves gaps; DC offsets when the
    # case removes the mean
    block = max(1, hop // 2)
    n = (nseg - 1) * hop + nfft + hop // 2 + 1          # a tail shorter than a hop, and room for a one-sample shift
    return wr.block_tones(n, nfft, block, seed=nfft + hop, dc_db=0.0 if detrend else None)


def mutants(x, nfft, hop, win, detrend, stride):
    nseg = wr.n_segments(x.size, nfft, hop)
    starts = np.arange(nseg) * hop
    sp = lambda st, **k: wr.segment_power(x, nfft, st, win, detrend, **k)
    db = lambda acc, k=nseg: wr.to_db(acc, k, FS, nfft, win)
    ref = db(sp(starts))
    j = nseg // 2
    twice = starts.copy()
    twice[j] = starts[j - 1]
    subst = starts.copy()
    subst[j - stride] = starts[j]                       # segment s read in place of s - stride
    iters = -(-nseg // stride)
    out = {
        "dropped": db(sp(np.delete(starts, j))),
        "counted twice": db(sp(twice)),
        "s + stride": db(sp(subst)),
        "shifted by one": db(sp(starts + 1)),
        "ragged step dropped": db(sp(starts[:(iters - 1) * stride])),
        "bins off by one": np.roll(ref, 1),
        "nseg + 1": db(sp(starts), nseg + 1),
        "nseg - 1": db(sp(starts), nseg - 1),
    }
    if detrend:
        out["detrend omitted"] = db(wr.segment_power(x, nfft, starts, win, None))
    if win != "rect":                                   # the symmetric rectangle is the periodic one
        out["symmetric window"] = db(sp(starts, symmetric=True))
    return ref, out


@pytest.mark.parametrize("nfft,hop,win,detrend,stride", CASES, ids=["%d-%d-%s" % c[:3] for c in CASES])
def test_mutants_rejected(nfft, hop, win, detrend, stride):
    nseg = 3 * stride + stride // 2 + 3                 # several steps, the last one ragged
    x = case_input(nfft, hop, detrend, nseg)
    assert wr.n_segments(x.size, nfft, hop) == nseg and nseg % stride
    ref, muts = mutants(x, nfft, hop, win, detrend, stride)
    oracle = wr.welch_db(x[:(nseg - 1) * hop + nfft], FS, nfft, hop, win, detrend=detrend)
    assert err(ref, oracle) < 1e-12
    weak = {k: err(v, ref) for k, v in muts.items() if err(v, ref) < margin(nfft, k) * bound(nfft)}
    assert not weak, (bound(nfft), weak)


@pytest.mark.parametrize("nfft,hop,win,detrend,stride", CASES, ids=["%d-%d-%s" % c[:3] for c in CASES])
def test_fp32_welch_accepted(nfft, hop, win, detrend, stride):
    """A Welch computed in complex64 with FP32 accumulation (what the kernels do) stays well inside the bound."""
    nseg = 3 * stride + stride // 2 + 3
    x = case_input(nfft, hop, detrend, nseg).astype(np.complex64)
    ref = wr.welch_db(x.astype(np.complex128), FS, nfft, hop, win, detrend=detrend)
    w = wr.window(win, nfft).astype(np.float32)
    acc = np.zeros(nfft, np.float32)
    for s in range(nseg):
        seg = x[s * hop:s * hop + nfft]
        if detrend:
            seg = seg - seg.mean(dtype=np.complex64)
        f = np.fft.fft(seg * w).astype(np.complex64)
        acc += (f.real * f.real + f.imag * f.imag).astype(np.float32)
    got = wr.to_db(acc.astype(np.float64), nseg, FS, nfft, win)
    assert err(got, ref) < 0.3 * bound(nfft)


@pytest.mark.parametrize("nfft,hop,win,scaling,detrend", [(64, 16, "hann", "density", None),
                                                           (1024, 777, "blackman", "spectrum", "constant"),
                                                           (4096, 4096, "rect", "density", "constant")])
def test_numpy_and_c_references_agree(nfft, hop, win, scaling, detrend):
    x = wr.block_tones(40 * hop + nfft + 5, nfft, hop, seed=nfft, dc_db=-6.0)
    got = wr.welch_sum(x, FS, nfft, hop, win, scaling=scaling, detrend=detrend)
    ref = wr.welch_db(x, FS, nfft, hop, win, scaling=scaling, detrend=detrend)
    assert err(got, ref) < 1e-12


def test_nsplit_table_reaches_every_regime():
    """The sizes the GPU matrix uses put each kernel in each of the four regimes."""
    seen = {}
    for prec, nfft, reg, nseg, hop, win, scaling, detrend in wr.matrix_cases():
        name, fpc, _ = wr.kernel_of(prec, nfft)
        assert wr.regime(nseg, fpc) == reg, (prec, nfft, nseg, reg)
        seen.setdefault(name, set()).add(reg)
    assert len(seen) == 5 + 4 + 8
    for name, regs in seen.items():
        assert regs == {1, 2, 3, 4}, (name, regs)
    assert wr.nsplit_of(10 ** 7, 64) == 64 and wr.nsplit_of(1, 16) == 1 and wr.nsplit_of(8 * 16 + 1, 16) == 2
