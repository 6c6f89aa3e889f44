"""The spectrum-trace references (CPU, tests/trace_reference.py): the trace built from the C oracle's |X|^2 against the
independent numpy restatement, the mean trace against scipy's Welch PSD, F = 1 against the spectrogram oracle, and the
EOF / strict-zero rules of the definition (include/sa_engine.h, sa_spectrum_trace)."""
import numpy as np
import pytest
import scipy.signal as sps

import trace_reference as tr
from oracle import c_oracle as co
from oracle import np_oracle as npo

STATS = ("mean", "max", "min")


def noise(dt, n, seed):
    rng = np.random.default_rng(seed)
    kind = dt.split("_")[0]
    order = "<" if dt.endswith("_le") else ">"
    if kind == "cf32":
        return rng.standard_normal(2 * n).astype(order + "f4")
    if kind == "cf64":
        return rng.standard_normal(2 * n).astype(order + "f8")
    if kind == "ci16":
        return rng.integers(-30000, 30000, 2 * n).astype(order + "i2")
    return rng.integers(0, 256, 2 * n).astype(np.uint8)


@pytest.mark.parametrize("dt,nfft,hop,start,win,F,db_mode", [
    ("cf32_le", 256, 100, 3, "hann", 7, 0), ("ci16_be", 128, 128, 0, "rect", 1, 1),
    ("cu8", 64, 33, 5, "blackman_harris", 20, 0), ("cf64_le", 512, 256, 0, "hamming", 13, 1),
    ("ci8", 256, 300, 1, "blackman", 50, 0)])
def test_c_and_numpy_references_agree(dt, nfft, hop, start, win, F, db_mode):
    n = 60 * hop + nfft
    raw = noise(dt, n, seed=nfft + hop)
    frames = 64                                    # the last frames read past the end: EOF
    a = tr.spectrum_trace(raw, dt, start, nfft, hop, win, frames, F, db_mode=db_mode, eof_fill_db=-140.0)
    b = tr.spectrum_trace_np(raw, dt, start, nfft, hop, win, frames, F, db_mode=db_mode, eof_fill_db=-140.0)
    for s in STATS:
        assert a[s].shape == (-(-frames // F), nfft)
        assert np.abs(a[s] - b[s]).max() < 1e-12, s


SCIPY_WIN = {"rect": "boxcar", "hann": "hann", "blackman_harris": "blackmanharris"}


@pytest.mark.parametrize("win", ["rect", "hann", "blackman_harris"])
@pytest.mark.parametrize("overlap", [False, True], ids=["hop=nfft", "hop=nfft/4"])
def test_mean_trace_is_welch_psd(win, overlap):
    """MEAN over readable frames = the two-sided density Welch PSD (fs = 1, no detrend), fft-shifted, times sum w^2."""
    nfft = 256
    hop = nfft // 4 if overlap else nfft
    raw = noise("cf32_le", 40 * nfft + 17, seed=7)
    x = raw[0::2].astype(np.float64) + 1j * raw[1::2].astype(np.float64)
    frames = (x.size - nfft) // hop + 1
    got = tr.spectrum_trace(raw, "cf32_le", 0, nfft, hop, win, frames, frames, db_mode=co.DB_POWER)["mean"][0]
    _, psd = sps.welch(x, fs=1.0, window=SCIPY_WIN[win], nperseg=nfft, noverlap=nfft - hop, detrend=False,
                       return_onesided=False, scaling="density")
    w = npo.window(win, nfft)
    ref = 10 * np.log10(np.fft.fftshift(psd) * np.sum(w * w) + 1e-20)
    assert np.abs(got - ref).max() < 1e-9


@pytest.mark.parametrize("db_mode", [0, 1])
def test_one_frame_per_row_is_the_spectrogram(db_mode):
    nfft, hop, frames = 256, 192, 40
    raw = noise("ci16_le", 35 * hop + nfft, seed=3)
    ref = co.spectrogram(raw, "ci16_le", 2, nfft, hop, "hann", frames, db_mode=db_mode)
    trc = tr.spectrum_trace(raw, "ci16_le", 2, nfft, hop, "hann", frames, 1, db_mode=db_mode)
    for s in STATS:
        assert np.abs(trc[s] - ref).max() < 1e-9, s


def test_eof_frames_follow_the_definition():
    """EOF frames contribute the power of eof_fill_db, counted in MEAN; a row of only EOF frames is eof_fill_db."""
    nfft, hop, F, eof = 128, 128, 4, -120.0
    raw = noise("cf32_le", 10 * hop + nfft, seed=5)          # frames 0..10 readable, 11.. EOF
    frames = 14
    t = tr.spectrum_trace(raw, "cf32_le", 0, nfft, hop, "rect", frames, F, eof_fill_db=eof, db_mode=co.DB_POWER)
    pw = 10 ** (co.spectrogram(raw, "cf32_le", 0, nfft, hop, "rect", frames, db_mode=co.DB_POWER) / 10) - 1e-20
    pw[11:] = 10 ** (eof / 10) - 1e-20
    for r in range(4):
        blk = pw[r * F:min(frames, (r + 1) * F)]
        assert np.allclose(t["mean"][r], 10 * np.log10(blk.mean(axis=0) + 1e-20), atol=1e-9)
        assert np.allclose(t["max"][r], 10 * np.log10(blk.max(axis=0) + 1e-20), atol=1e-9)
        assert np.allclose(t["min"][r], 10 * np.log10(blk.min(axis=0) + 1e-20), atol=1e-9)
    for s in STATS:
        assert np.allclose(t[s][3], eof, atol=1e-9, rtol=0)                    # frames 12, 13: EOF only


@pytest.mark.parametrize("dt", ["cf64_le", "ri16_le"])
def test_strict_zero_rows_are_constants(dt):
    """cf64 / a datatype without a decode branch under strict_reference: readable frames have P = 0 (-200 dB), EOF
    frames the EOF power; each row is a constant given by its counts."""
    nfft, hop, F = 64, 64, 3
    bps = 16 if dt.startswith("cf64") else 8
    raw = np.zeros(7 * hop * bps + nfft * bps - 1, np.uint8)  # frames 0..6 readable, 7.. EOF
    frames = 10
    for impl in (tr.spectrum_trace, tr.spectrum_trace_np):
        t = impl(raw, dt, 0, nfft, hop, "hann", frames, F, strict_reference=True)
        pe = (10 ** (-150.0 / 20) - 1e-10) ** 2
        lvl = lambda p: 20 * np.log10(np.sqrt(p) + 1e-10)
        want = {"mean": [lvl(0), lvl(0), lvl(2 * pe / 3), lvl(pe)],
                "max": [lvl(0), lvl(0), lvl(pe), lvl(pe)],
                "min": [lvl(0), lvl(0), lvl(0), lvl(pe)]}
        for s in STATS:
            assert t[s].shape == (4, nfft)
            assert np.allclose(t[s], np.array(want[s])[:, None], atol=1e-9, rtol=0), (impl.__name__, s)
