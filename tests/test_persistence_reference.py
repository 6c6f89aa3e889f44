"""Self-tests of tests/persistence_reference.py on the CPU: the quantizer and the oracle comparator accept the histogram
of FP32-rounded oracle dB and of magnitudes perturbed within 0.9 of the error bound, and reject the mutants a wrong
kernel would produce (levels shifted, bins off by one, a frame dropped / counted twice / replaced by its neighbour,
EOF frames omitted, levels reversed, out-of-range values dropped, power dB for magnitude dB).

Input: gain-stepped noise plus a tone, cf32, whose frame gains step by 20 dB from 0 down to -220 dB (the quietest
frames reach |X| ~ 1e-10, where magnitude and power dB differ), so that neighbouring frames land on different levels."""
import numpy as np
import pytest

import persistence_reference as pr
from oracle import c_oracle as co

NFFT, HOP = 64, 64
N_READ = 60                       # readable frames
N_EOF = 3


def gain_stepped(n_frames=N_READ, nfft=NFFT, seed=5):
    rng = np.random.default_rng(seed)
    n = n_frames * nfft
    t = np.arange(n)
    g = np.power(10.0, -(np.arange(n_frames) % 12.0)).repeat(nfft)        # 20 dB per frame, |X| down to ~1e-11
    z = rng.standard_normal((n, 2)) * 0.3
    z[:, 0] += np.cos(2 * np.pi * 0.2 * t)
    z[:, 1] += np.sin(2 * np.pi * 0.2 * t)
    return (z * g[:, None]).astype(np.float32).view(np.uint8).reshape(-1)


RANGES = [(37, -190.0, 10.0), (256, -215.0, 35.0), (2, -120.0, -100.0)]


def oracle_rows(raw, frames, db_mode=0):
    db = co.spectrogram(raw, "cf32_le", 0, NFFT, HOP, "hann", frames, db_mode=db_mode)
    db[N_READ:] = -150.0
    return db


@pytest.fixture(scope="module")
def raw():
    return gain_stepped()


@pytest.mark.parametrize("n_levels,lo_db,hi_db", RANGES)
def test_quantizer_restates_the_definition(n_levels, lo_db, hi_db):
    d = np.array([np.nan, -np.inf, np.inf, lo_db - 1, lo_db, hi_db, hi_db + 5, lo_db + (hi_db - lo_db) / n_levels],
                 np.float32)
    lv = pr.quantize(d, n_levels, lo_db, hi_db, False)
    assert list(lv[:7]) == [0, 0, n_levels - 1, 0, 0, n_levels - 1, n_levels - 1]
    assert lv[7] in (0, 1)                      # the first boundary, up to the FP32 rounding of s
    x = np.linspace(lo_db - 3, hi_db + 3, 10001)
    for f64 in (False, True):
        q = pr.quantize(x, n_levels, lo_db, hi_db, f64)
        assert np.all(np.diff(q) >= 0) and q.min() == 0 and q.max() == n_levels - 1
        ft = np.float64 if f64 else np.float32
        u = (x.astype(ft) - ft(lo_db)) * ft(n_levels / (hi_db - lo_db))
        assert np.array_equal(q, np.where(u >= 1, np.minimum(np.floor(u), n_levels - 1), 0))


@pytest.mark.parametrize("n_levels,lo_db,hi_db", RANGES)
@pytest.mark.parametrize("db_mode", [0, 1])
def test_comparator_accepts_fp32_rows_and_perturbed_magnitudes(raw, n_levels, lo_db, hi_db, db_mode):
    frames = N_READ + N_EOF
    rows = oracle_rows(raw, frames, db_mode)
    counts = pr.histogram(rows.astype(np.float32), n_levels, lo_db, hi_db, False)
    assert np.all(counts.sum(axis=0) == frames)
    rng = np.random.default_rng(n_levels)
    h_lo, h_hi, h_p = pr.oracle_level_histograms(raw, "cf32_le", 0, NFFT, HOP, "hann", frames, n_levels, lo_db, hi_db,
                                                 False, db_mode,
                                                 perturb=lambda m, e: m + 0.9 * e * rng.choice([-1.0, 1.0], m.shape))
    assert pr.counts_within_bounds(counts, h_lo, h_hi, frames) is None
    assert pr.counts_within_bounds(h_p, h_lo, h_hi, frames) is None
    for f64 in (False, True):
        assert pr.check_against_oracle(pr.histogram(rows if f64 else rows.astype(np.float32), n_levels, lo_db, hi_db,
                                                    f64), raw, "cf32_le", 0, NFFT, HOP, "hann", frames, n_levels,
                                       lo_db, hi_db, f64, db_mode) is None


@pytest.mark.parametrize("n_levels,lo_db,hi_db", RANGES[:2])
def test_comparator_rejects_mutants(raw, n_levels, lo_db, hi_db):
    frames = N_READ + N_EOF
    rows = oracle_rows(raw, frames).astype(np.float32)
    h_lo, h_hi = pr.oracle_level_histograms(raw, "cf32_le", 0, NFFT, HOP, "hann", frames, n_levels, lo_db, hi_db, False)
    good = pr.histogram(rows, n_levels, lo_db, hi_db, False)
    assert pr.counts_within_bounds(good, h_lo, h_hi, frames) is None

    def rejects(c):
        return pr.counts_within_bounds(c, h_lo, h_hi, frames) is not None

    lv = pr.quantize(rows, n_levels, lo_db, hi_db, False)
    assert rejects(pr.histogram_of_levels(np.minimum(lv + 1, n_levels - 1), n_levels))      # every level up by one
    assert rejects(pr.histogram_of_levels(np.maximum(lv - 1, 0), n_levels))                 # ... down by one
    assert rejects(np.roll(good, 1, axis=1)) and rejects(np.roll(good, -1, axis=1))         # bins off by one
    for t in (5, 17, N_READ - 1):
        assert rejects(pr.histogram(np.delete(rows, t, axis=0), n_levels, lo_db, hi_db, False))     # dropped
        assert rejects(pr.histogram(np.insert(rows, t, rows[t], axis=0), n_levels, lo_db, hi_db, False))   # twice
        swapped = rows.copy()
        swapped[t] = rows[t - 1]                                                              # replaced by neighbour
        assert rejects(pr.histogram(swapped, n_levels, lo_db, hi_db, False)), t
    assert rejects(pr.histogram(rows[:N_READ], n_levels, lo_db, hi_db, False))              # EOF frames omitted
    assert rejects(good[::-1])                                                              # levels reversed
    inside = (rows >= lo_db) & (rows < hi_db)
    if n_levels == 37:                           # the range clips the tone above and the quiet frames below
        assert (rows < lo_db).any() and (rows >= hi_db).any()
        dropped = np.zeros_like(good)
        np.add.at(dropped, (lv[inside], np.nonzero(inside)[1]), 1)
        assert rejects(dropped)                                                             # out of range dropped
    power = oracle_rows(raw, frames, db_mode=1).astype(np.float32)
    if n_levels == 256:                          # levels of 1 dB reach down to -215 dB, where the two modes differ
        assert rejects(pr.histogram(power, n_levels, lo_db, hi_db, False))                      # power dB for magnitude dB


def test_strict_zero_and_eof_constants():
    """-200 dB is the oracle's row of a zero frame in both db_modes; EOF frames hold eof_fill_db."""
    raw = np.zeros(8 * NFFT * 8, np.uint8)
    for mode in (0, 1):
        db = co.spectrogram(raw, "cf32_le", 0, NFFT, HOP, "hann", 8, db_mode=mode)
        assert np.all(db == -200.0)
        h_lo, h_hi = pr.oracle_level_histograms(raw, "cf64_le", 0, NFFT, HOP, "hann", 7, 37, -190.0, 10.0, True, mode,
                                                eof_fill_db=-150.0, strict_reference=True)
        assert np.array_equal(h_lo, h_hi)
        readable = 8 * NFFT * 8 // (16 * NFFT)                  # cf64: 16 bytes per IQ pair
        want = np.zeros((37, NFFT), np.int64)
        want[pr.quantize(np.array([-200.0]), 37, -190.0, 10.0, True)[0]] += readable
        want[pr.quantize(np.array([-150.0]), 37, -190.0, 10.0, True)[0]] += 7 - readable
        assert np.array_equal(h_lo, want)
    db = co.spectrogram(gain_stepped(4), "cf32_le", 0, NFFT, HOP, "hann", 6)
    assert np.all(db[4:] == -150.0)                             # the oracle's EOF rows


def test_chunk_rule():
    assert pr.level_chunk_frames(1024, 524287) == 524287        # the headline shape is one chunk
    assert pr.level_chunk_frames(65536, 10 ** 6) == 8192
    assert pr.level_chunk_frames(64, 5) == 5
