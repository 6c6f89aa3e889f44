"""Every Welch PSD kernel against the FP64 oracle on block-tone input, across split, iteration and persistent-wave
boundaries.

The block-tone input of tests/welch_reference.py gives every segment its own tones at its own levels, so a segment
read from the wrong place, read twice, dropped, or summed under another signal's split changes bins by a large fraction
(tests/test_welch_reference.py shows each such mistake lands >= 100x over the bound of its kernel family).  Geometry is restated in
welch_reference.py from fft_core.cuh / spectrogram_mid_kernel.cuh / analysis.cu, and each case asserts the kernel
engine.last_kernel reports, the regime its segment count puts the launch in, and (batch cases) how many waves it spans.

  (a) each kernel engine.psd_welch reaches (FP32 64..16384: general plan to 1024, welch_accum_mid_kernel from 2048;
      FP64 64..8192) in four regimes: fewer segments than frame slots; one CTA per signal with several steps;
      1 < nsplit < 64 with a ragged last step; nsplit = 64 with 10 steps per slot.  Hops below, at and above nfft and
      odd; a tail shorter than a hop; all five windows; both scalings; mean removal on and off (always on with idle
      slots, where the mid kernel transforms zero segments to keep its barriers);
  (b) the batch path (FP32 rows of the downconverter's scratch, down 1, taps [1.0]: the rows are the recording's
      samples) past the persistent mid kernel's first wave: n_sig x nsplit >= 2 W + r tasks, W = SMs x (threads per
      SM / 512) an upper bound of its resident CTAs; signals of different lengths (idle splits); even hop (128-bit
      loads) and odd hop; short annotations between the full ones (NaN-padded rows through the direct kernel, and the
      packed-rows-plus-copies output path); one FP64 batch whose (nsplit, n_sig) grid exceeds one wave;
  (c) the same batch twice is byte-identical (the ticket order is not), PSD-only equals with-IQ;
  (d) several batches (SA_DC_BATCH_MB=1, both schedules, a child process): every signal against the oracle;
  (e) one signal of 4 M segments at 64 points: every frame slot adds 1001 segments in FP32.  This bounds the
      accumulation error only -- with a thousand segments per bin one wrong segment is below the bound.  Its
      reference transforms 4.1 M x 64 = 262 M points, over the ~150 M per case the rest of the module keeps to: the
      64-point kernel has 64 x 64 = 4096 slots at nsplit = 64, so 1000 additions per slot cannot take fewer segments
      (the numpy reference takes about 15 s of the module's time);
  (f) the direct DFT kernel: lengths below 64 and not powers of two, over one kDirectTile (1024), several segments
      with mean removal, and several signals in one launch through the batch's short rows.

Comparator: util.frame_norm_error on the PSD row, E = max_k |A_got - A_ref| / rms_k(A_ref), A = 10^(dB/20) = sqrt(P).
Bounds: util.NORM_TOL_F32 = 1e-5 and util.NORM_TOL_F64 = 1e-12, the spectrogram's, for the general FP32 and FP64
kernels (including the 4 M-segment case).  Two families get their own bound:
  welch_accum_mid_kernel  MID_F32_TOL = 2.5e-5, about 2x its worst E.  Worst E per size and load path (FP64 rows
                          through engine.psd_welch; FP32 rows of the batch with 128-bit loads, even hop; and scalar
                          loads, odd hop):
                                    psd_welch   batch vec   batch scalar
                             2048   5.4e-6      5.4e-6      5.1e-6
                             4096   7.9e-6      6.6e-6      8.4e-6
                             8192   7.3e-6      8.5e-6      9.4e-6
                            16384   7.7e-6      1.22e-5     8.5e-6
                          The error grows with the size and hardly with the path.  It is as large at 16384 points,
                          where FPC = 1 and there is no slot sum, as at 8192.  So it comes from the transform: the
                          small-radix-first plan generates its twiddles by an FP32 recurrence.  Its per-frame error
                          already reaches 4.9e-6 on white noise in the spectrogram matrix.  Here the +-20 dB block gains
                          put the strongest tone bins far above the row rms that E is relative to.  Neither the load
                          path nor the slot sums add measurably.  The worst case is the 16384-point batch with an even
                          hop (8192).
  psd_direct_kernel<float>  direct_f32_tol = max(1e-5, 30 sqrt(nfft) 2^-24): each bin is a sequential FP32 sum of
                          nfft products whose partial sums reach the tone's full amplitude, so the error grows as
                          sqrt(nfft) 2^-24; 30 is about 2.5x the worst measured E / (sqrt(nfft) 2^-24) (11.9, at a
                          1500-point short row of a batch).
Worst E measured on one NVIDIA B200 (power limit 1000 W, max SM clock 1965 MHz):
  welch_accum_kernel<float>         9.0e-7   (1024 points, one segment slot short of a CTA, mean removal)
  welch_accum_mid_kernel<float>     1.22e-5  (table above)
  welch_accum_kernel<double>        2.7e-14
  psd_direct_kernel<double>         1.4e-13
  psd_direct_kernel<float>          E / (sqrt(nfft) 2^-24) = 11.9  (nfft 5 .. 11000)
The module prints these per family and, for the FP32 kernels, per size and path (run with -s).
The whole module, CPU references included, takes about 31 s on that machine.
"""
import json
import os
import subprocess
import sys
import functools

import numpy as np
import pytest
import torch

import welch_reference as wr
from util import frame_norm_error

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FS = 1.0e6
WORST = {}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IDENTITY = np.array([1.0])      # down 1 with this filter: the FP32 rows are the recording's samples
DETAIL = {}                      # (kernel, nfft, path) -> worst E


def note(name, e, nfft, path, case=""):
    """records E under the kernel family (the direct FP32 kernel as E / (sqrt(nfft) 2^-24)) and, per size and path,
    under (kernel, nfft, path)"""
    fam = wr.family(name)
    v = float(e)
    if name == "psd_direct_kernel<float>":
        v = v / (np.sqrt(nfft) * 2.0 ** -24)
        fam += " (E / sqrt(nfft) 2^-24)"
    if v > WORST.get(fam, (0.0, ""))[0]:
        WORST[fam] = (v, "%d %s %s" % (nfft, path, case))
    key = (wr.family(name), nfft, path)
    DETAIL[key] = max(DETAIL.get(key, 0.0), float(e))


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    import time
    t0 = time.time()
    yield
    print("\nworst frame_norm_error per Welch kernel family (module %.0f s):" % (time.time() - t0))
    for k in sorted(WORST):
        print("  %-50s %.3e   at %s" % (k, WORST[k][0], WORST[k][1]))
    print("worst E of the FP32 kernels per size and path:")
    for k in sorted(DETAIL):
        if "<float" in k[0]:
            print("  %-32s %6d  %-14s %.3e" % (k[0], k[1], k[2], DETAIL[k]))


@pytest.fixture(scope="module")
def wave():
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, p.max_threads_per_multi_processor


def check_row(got, ref, name, nfft, path, case=""):
    assert np.isfinite(got).all()
    e = float(frame_norm_error(got[None], ref[None])[0])
    note(name, e, nfft, path, case)
    tol = wr.tol_of(name, nfft)
    assert e <= tol, "%s: E %.3g > %.3g" % (name, e, tol)
    return e


@pytest.fixture
def config(engine):
    def set_(**kw):
        engine.set_analysis_config(**kw)
    yield set_
    engine.reset_analysis_config()


# ---------------- (a) every kernel through engine.psd_welch ----------------

CASES = wr.matrix_cases()


@pytest.mark.parametrize("prec,nfft,reg,nseg,hop,win,scaling,detrend", CASES,
                         ids=["%s-%d-r%d-hop%d-%s" % (c[0], c[1], c[2], c[4], c[5]) for c in CASES])
def test_welch_kernel_regimes(engine, config, prec, nfft, reg, nseg, hop, win, scaling, detrend):
    name, fpc, _ = wr.kernel_of(prec, nfft)
    assert wr.regime(nseg, fpc) == reg
    n = (nseg - 1) * hop + nfft + hop // 3                           # a tail shorter than a hop
    assert wr.n_segments(n, nfft, hop) == nseg
    x = wr.block_tones(n, nfft, max(1, hop // 2), seed=nfft * 10 + reg, dc_db=0.0 if detrend else None)
    config(psd_scaling=scaling, psd_detrend=detrend, psd_precision=prec)
    got = engine.psd_welch(wr.iq_of(x), FS, nfft, hop=hop, window=win)[1]
    assert engine.last_kernel == name
    check_row(got, wr.welch_db(x, FS, nfft, hop, win, scaling, detrend), name, nfft, "psd_welch",
              "r%d hop %d %s %s" % (reg, hop, win, detrend or ""))


# ---------------- (b) / (c) the batch path past the first wave ----------------

@functools.lru_cache(maxsize=2)
def recording(n, seed):
    """cf32 recording of block tones (blocks of 1000 samples: no annotation's segments line up with them)"""
    return wr.block_tones(n, 4096, 1000, seed).astype(np.complex64)


def batch_plan(nfft, hop, n_full, long_nseg, shorts, seed):
    """annotations (start, count, 0, 1, False): one long signal (sets nsplit), n_full - 1 of random shorter lengths,
    and `shorts` (counts below nfft) placed between them"""
    rng = np.random.default_rng(seed)
    counts = [(long_nseg - 1) * hop + nfft + hop // 2]
    counts += [int(nfft + hop * rng.integers(0, 40 * max(1, 16384 // nfft) // 8 + 2) + rng.integers(0, hop))
               for _ in range(n_full - 1)]
    rng.shuffle(counts)
    for j, c in enumerate(shorts):
        counts.insert(1 + (2 * j + 1) * len(counts) // (2 * len(shorts) + 1), c)
    n_rec = max(counts) + (1 << 16)
    anns = [(int(rng.integers(0, n_rec - c)), int(c), 0.0, 1, False) for c in counts]
    return n_rec, anns


def run_batch(engine, raw, anns, nfft, hop, win, want_iq=True):
    return engine.downconvert_psd_batch(raw.view(np.float32), "cf32_le", FS, anns, psd_nfft=nfft, psd_hop=hop,
                                        psd_window=win, want_iq=want_iq)


def batch_path(hop):
    """the load path of the FP32 rows: the mid kernel's 128-bit loads need an even hop (rows start 16-byte aligned)"""
    return "batch vec" if hop % 2 == 0 else "batch scalar"


def check_batch(raw, anns, iqs, psd, nfft, hop, win, name, scaling="density", detrend=None):
    """every row: full annotations against the FP64 Welch of the returned IQ, short ones against the oracle of their
    own length (hop nf / 4) followed by NaN"""
    worst = 0.0
    for i, (s, c, _, _, _) in enumerate(anns):
        iq = iqs[i]
        assert iq.shape == (2, c)
        assert np.array_equal(iq[0] + 1j * iq[1], raw[s:s + c].astype(np.complex128))     # down 1, taps [1.0]
        x = iq[0] + 1j * iq[1]
        if c >= nfft:
            worst = max(worst, check_row(psd[i], wr.welch_db(x, FS, nfft, hop, win, scaling, detrend), name, nfft,
                                         batch_path(hop), "hop %d %s %s" % (hop, win, detrend or "")))
        else:
            assert np.isnan(psd[i, c:]).all()
            check_row(psd[i, :c], wr.welch_db(x, FS, c, max(1, c // 4), win, scaling, detrend),
                      "psd_direct_kernel<double>" if "<double" in name else "psd_direct_kernel<float>", c, "batch")
    return worst


def mid_batch(nfft, hop, wave):
    """a past-wave batch for the mid kernel of nfft points"""
    fpc = wr.F32_MID_FPC[nfft]
    W = wr.wave_ctas(*wave, wr.MID_CTA)
    long_nseg = (wr.MAX_SPLIT - 1) * wr.STEPS * fpc + 5                # nsplit 64
    n_full = -(-(2 * W + 7) // wr.MAX_SPLIT)
    n_rec, anns = batch_plan(nfft, hop, n_full, long_nseg, [nfft // 2 + 3, 1000, nfft // 2 + 3, 77], seed=nfft + hop)
    full = [c for _, c, _, _, _ in anns if c >= nfft]
    ns = wr.nsplit_of(max(wr.n_segments(c, nfft, hop) for c in full), fpc)
    assert ns == wr.MAX_SPLIT and len(full) * ns >= 2 * W + 7
    assert min(wr.n_segments(c, nfft, hop) for c in full) < ns * fpc        # idle splits
    return recording(n_rec, 5), anns


MID_BATCHES = [(n, h) for n in sorted(wr.F32_MID_FPC) for h in (n // 2, n // 2 + 1)]


@pytest.mark.parametrize("nfft,hop", MID_BATCHES, ids=["%d-hop%d" % c for c in MID_BATCHES])
def test_mid_kernel_batch_past_first_wave(engine, config, wave, nfft, hop):
    raw, anns = mid_batch(nfft, hop, wave)
    config(taps=IDENTITY)
    name = "welch_accum_mid_kernel<float,%d>" % nfft
    iqs, psd = run_batch(engine, raw, anns, nfft, hop, "hann")
    assert engine.last_kernel.endswith("+" + name), engine.last_kernel
    check_batch(raw, anns, iqs, psd, nfft, hop, "hann", name)


def test_fp64_batch_past_first_wave(engine, config, wave):
    """FP32 rows into welch_accum_kernel<double, 1024> (FPC 2, 128 threads), grid (64, n_sig) over one wave; every
    annotation full length, so the rows are written in place (contiguous output)."""
    nfft, hop = 1024, 700
    name, fpc, cta = wr.kernel_of("f64", nfft)
    W = wr.wave_ctas(wave[0], 2048, cta)
    n_full = -(-(W + 5) // wr.MAX_SPLIT)
    n_rec, anns = batch_plan(nfft, hop, n_full, (wr.MAX_SPLIT - 1) * wr.STEPS * fpc + 3, [], seed=11)
    ns = wr.nsplit_of(max(wr.n_segments(c, nfft, hop) for _, c, _, _, _ in anns), fpc)
    assert ns * len(anns) > W
    raw = recording(n_rec, 5)
    config(taps=IDENTITY, psd_precision="f64", psd_detrend="constant", psd_scaling="spectrum")
    iqs, psd = run_batch(engine, raw, anns, nfft, hop, "blackman")
    assert engine.last_kernel.endswith("+" + name), engine.last_kernel
    check_batch(raw, anns, iqs, psd, nfft, hop, "blackman", name, "spectrum", "constant")


def test_batch_reproducible(engine, config, wave):
    """Run twice: byte-identical PSD rows although the CTAs draw the tasks in another order; PSD-only equals with-IQ."""
    raw, anns = mid_batch(4096, 2048, wave)
    config(taps=IDENTITY)
    _, a = run_batch(engine, raw, anns, 4096, 2048, "hamming")
    _, b = run_batch(engine, raw, anns, 4096, 2048, "hamming")
    none, c = run_batch(engine, raw, anns, 4096, 2048, "hamming", want_iq=False)
    assert none is None
    assert a.tobytes() == b.tobytes() and a.tobytes() == c.tobytes()


# ---------------- (d) several batches ----------------

CHILD = r'''
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1] + "/tests")
import welch_reference as wr
from util import frame_norm_error
from spectral_analyzer_b200 import Engine
eng = Engine()
eng.set_analysis_config(taps=np.array([1.0]))
nfft, hop = 2048, 1000
rng = np.random.default_rng(3)
raw = wr.block_tones(1 << 22, 4096, 1000, 9).astype(np.complex64)
counts = [int(rng.integers(20000, 110000)) for _ in range(36)]
counts[5], counts[17], counts[30] = 1500, 777, 1500
anns = [(int(rng.integers(0, (1 << 22) - c)), c, 0.0, 1, False) for c in counts]
iqs, psd = eng.downconvert_psd_batch(raw.view(np.float32), "cf32_le", 1e6, anns, psd_nfft=nfft, psd_hop=hop)
kernel = eng.last_kernel
none, psd2 = eng.downconvert_psd_batch(raw.view(np.float32), "cf32_le", 1e6, anns, psd_nfft=nfft, psd_hop=hop, want_iq=False)
out = {"kernel": kernel, "same": bool(psd.tobytes() == psd2.tobytes()), "iq_ok": True, "nan_ok": True, "full": [], "short": []}
for i, (s, c, _, _, _) in enumerate(anns):
    x = raw[s:s + c].astype(np.complex128)
    out["iq_ok"] &= bool(np.array_equal(iqs[i][0] + 1j * iqs[i][1], x))      # down 1, taps [1.0]: the samples
    if c >= nfft:
        e = frame_norm_error(psd[i][None], wr.welch_db(x, 1e6, nfft, hop, "hann")[None])[0]
        out["full"].append(float(e))
    else:
        out["nan_ok"] &= bool(np.isnan(psd[i, c:]).all())
        e = frame_norm_error(psd[i, :c][None], wr.welch_db(x, 1e6, c, c // 4, "hann")[None])[0]
        out["short"].append([c, float(e)])
print(json.dumps(out))
'''


@pytest.mark.parametrize("sched", ["0", "1"])
def test_several_batches_every_signal(sched):
    """36 annotations over a 1 MB batch cut (about 20 batches, both workspaces, the helper stream): every row."""
    env = dict(os.environ, SA_DC_BATCH_MB="1", SA_DC_SCHED=sched)
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["kernel"].endswith("+welch_accum_mid_kernel<float,2048>"), out
    assert out["same"] and out["iq_ok"] and out["nan_ok"], out
    assert len(out["full"]) == 33 and len(out["short"]) == 3
    name = "welch_accum_mid_kernel<float,2048>"
    for e in out["full"]:
        note(name, e, 2048, "batch vec", "several batches, SA_DC_SCHED=" + sched)
        assert e <= wr.tol_of(name, 2048), out
    for c, e in out["short"]:
        note("psd_direct_kernel<float>", e, c, "batch")
        assert e <= wr.direct_f32_tol(c), out


# ---------------- (e) long FP32 accumulation ----------------

def test_long_fp32_accumulation(engine, config):
    """64 points, hop 16: 4 M segments over 64 x 64 frame slots, 1001 FP32 additions per slot and bin."""
    nfft, hop = 64, 16
    name, fpc, _ = wr.kernel_of("f32", nfft)
    nseg = wr.MAX_SPLIT * fpc * 1000 + 37
    assert wr.iterations(nseg, wr.nsplit_of(nseg, fpc), fpc) == 1001
    n = (nseg - 1) * hop + nfft + 5
    x = wr.block_tones_device(n, nfft, hop // 2, seed=64, device=DEV).cpu().numpy()
    torch.cuda.empty_cache()
    config(taps=IDENTITY)
    _, psd = engine.downconvert_psd_batch(x.view(np.float32), "cf32_le", FS, [(0, n, 0.0, 1, False)], psd_nfft=nfft,
                                          psd_hop=hop, psd_window="hann", want_iq=False)
    assert engine.last_kernel.endswith("+" + name)
    acc = wr.segment_power(x, nfft, np.arange(nseg, dtype=np.int64) * hop, "hann", None, slab=1 << 22)
    check_row(psd[0], wr.to_db(acc, nseg, FS, nfft, "hann"), name, nfft, "batch vec", "4 M segments")


# ---------------- (f) direct DFT kernel ----------------

DIRECT = [(5, 3, 4), (33, 11, 9), (48, 48, 3), (32, 7, 20), (1000, 250, 12), (1536, 1536, 5), (3000, 1100, 7),
          (5000, 4999, 4), (11000, 5500, 3)]


@pytest.mark.parametrize("prec", ["f32", "f64"])
@pytest.mark.parametrize("nfft,hop,nseg", DIRECT, ids=["%d-hop%d" % c[:2] for c in DIRECT])
def test_direct_kernel(engine, config, prec, nfft, hop, nseg):
    name = wr.kernel_of(prec, nfft)[0]
    assert name.startswith("psd_direct_kernel")
    n = (nseg - 1) * hop + nfft + hop // 2
    x = wr.block_tones(n, nfft, max(1, hop // 2), seed=nfft + 1, dc_db=-3.0)
    win = wr.WINDOWS[nfft % 5]
    for detrend in (None, "constant"):
        config(psd_detrend=detrend, psd_precision=prec)
        got = engine.psd_welch(wr.iq_of(x), FS, nfft, hop=hop, window=win)[1]
        assert engine.last_kernel == name
        check_row(got, wr.welch_db(x, FS, nfft, hop, win, "density", detrend), name, nfft, "psd_welch")


def test_direct_kernel_several_signals_in_one_launch(engine, config):
    """Only short annotations: one direct launch per length, several signals each (rows NaN padded to psd_nfft)."""
    nfft = 2048
    raw = recording(1 << 20, 5)
    rng = np.random.default_rng(4)
    counts = [1000, 1999, 1000, 1000, 1999, 1000]
    anns = [(int(rng.integers(0, (1 << 20) - c)), c, 0.0, 1, False) for c in counts]
    for prec in ("f32", "f64"):
        config(taps=IDENTITY, psd_precision=prec)
        iqs, psd = run_batch(engine, raw, anns, nfft, 1024, "blackman_harris")
        name = wr.kernel_of(prec, 1001)[0]
        assert engine.last_kernel.endswith("+" + name), engine.last_kernel
        check_batch(raw, anns, iqs, psd, nfft, 1024, "blackman_harris", name)
