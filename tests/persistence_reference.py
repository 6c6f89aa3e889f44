"""numpy restatement of the persistence spectrum (sa_spectrum_persistence) and its oracle comparator.

Per frame t and bin k (fft-shifted) d[t][k] is the value of the spectrogram row: FP32 dB on FP32 launches, FP64 dB on
FP64 launches, eof_fill_db for a frame past the end of the buffer, -200 dB for a strict-reference zero decode.  In the
launch's precision, each operation rounded on its own:
    u = (d - min_db) * s,  s = n_levels / (max_db - min_db)   (min_db and s computed in FP64, then rounded)
    level = u >= 1 ? (int)min(u, n_levels - 1) : 0;  counts[level][k] += 1
numpy's float32 / float64 arithmetic rounds every operation, so `quantize` is the kernel's quantizer bit for bit.

`check_against_oracle` holds counts to the FP64 oracle (oracle/sa_oracle.c power-mode rows, streamed in slabs): per frame
the oracle magnitude |X|, the frame's rms magnitude r_t and eps = tol r_t (the bounds util.frame_norm_error enforces);
[|X| - eps, |X| + eps] is taken to dB under the request's db_mode, widened by SLACK_DB, and quantized to levels lo <= hi.
A column passes when it sums to n_frames and, at every level boundary j, #{hi < j} <= sum_{l<j} counts[l] <= #{lo < j}.
EOF and strict-zero frames take their exact levels.
"""
import numpy as np

from oracle import c_oracle as co
from util import NORM_TOL_F32, NORM_TOL_F64

BPS = {"cf32": 8, "ci16": 4, "cu8": 2, "ci8": 2, "cf64": 16}
SLAB = 1 << 22                      # points per oracle call
SLACK_DB = {False: 1e-4, True: 1e-9}    # lg2.approx and the quantizer's rounding (FP32); FP64
LEVEL_CHUNK_BYTES = 512 << 20       # persistence.cu kLevelChunkBytes: level rows per chunk of the device entry


def level_chunk_frames(nfft, n_frames):
    """Frames per chunk of level rows (the chunk rule of DESIGN.md N5)."""
    return min(n_frames, max(1, LEVEL_CHUNK_BYTES // nfft))


def quantize(d, n_levels, min_db, max_db, f64):
    """Levels (int64) of dB values d in the launch's precision (f64: FP64 launch)."""
    ft = np.float64 if f64 else np.float32
    mn, s, top = ft(min_db), ft(n_levels / (max_db - min_db)), ft(n_levels - 1)
    with np.errstate(invalid="ignore", over="ignore"):
        u = (np.asarray(d).astype(ft) - mn) * s
        lv = np.zeros(u.shape, np.int64)
        m = u >= 1
        lv[m] = np.minimum(u[m], top).astype(np.int64)
    return lv


def histogram_of_levels(lv, n_levels):
    """counts [n_levels, nfft] (uint32) of level rows [frames, nfft]."""
    nfft = lv.shape[1]
    idx = (lv.astype(np.int64) * nfft + np.arange(nfft)[None, :]).ravel()
    return np.bincount(idx, minlength=n_levels * nfft).reshape(n_levels, nfft).astype(np.uint32)


def histogram(rows_db, n_levels, min_db, max_db, f64):
    """The persistence counts of dB rows [frames, nfft] (FP32 rows with f64=False, FP64 rows with f64=True)."""
    return histogram_of_levels(quantize(rows_db, n_levels, min_db, max_db, f64), n_levels)


def _layout(buf, datatype, strict_reference):
    kind = datatype.split("_")[0]
    known = kind in BPS
    bps = BPS[kind] if known else 8                                  # Global.getBytesPerSample fallback
    zeros = (not known) or (kind == "cf64" and strict_reference)     # SpectralService.java:60-63
    return bps, zeros, np.ascontiguousarray(buf).view(np.uint8).size


def mag_to_db(m, db_mode):
    return 20 * np.log10(m + 1e-10) if db_mode == 0 else 10 * np.log10(m * m + 1e-20)


def oracle_slabs(buf, datatype, start_sample, nfft, hop, window, n_frames, strict_reference=False):
    """Yields (f0, |X| [nf, nfft] FP64, readable [nf]) over slabs of frames; |X| of strict-zero frames is 0."""
    bps, zeros, cap = _layout(buf, datatype, strict_reference)
    step = max(1, SLAB // nfft)
    for f0 in range(0, n_frames, step):
        nf = min(step, n_frames - f0)
        t = f0 + np.arange(nf)
        readable = (start_sample + t * hop + nfft) * bps <= cap                  # MainController.java:987
        if zeros:
            m = np.zeros((nf, nfft))
        else:
            db = co.spectrogram(buf, datatype, start_sample + f0 * hop, nfft, hop, window, nf, db_mode=co.DB_POWER)
            m = np.sqrt(np.maximum(np.power(10.0, db / 10) - 1e-20, 0.0))
        yield f0, m, readable


def level_bounds(m, readable, n_levels, min_db, max_db, f64, db_mode=0, eof_fill_db=-150.0, zeros=False, tol=None):
    """(lo, hi) levels of oracle magnitudes m [nf, nfft] under the FP32 / FP64 error bound; exact for EOF and zero
    frames."""
    tol = (NORM_TOL_F64 if f64 else NORM_TOL_F32) if tol is None else tol
    eps = tol * np.sqrt(np.mean(m * m, axis=1, keepdims=True))
    with np.errstate(divide="ignore"):
        d_lo = mag_to_db(np.maximum(m - eps, 0.0), db_mode) - SLACK_DB[f64]
        d_hi = mag_to_db(m + eps, db_mode) + SLACK_DB[f64]
    if zeros:
        d_lo[:] = -200.0
        d_hi[:] = -200.0
    d_lo[~readable] = eof_fill_db
    d_hi[~readable] = eof_fill_db
    return quantize(d_lo, n_levels, min_db, max_db, f64), quantize(d_hi, n_levels, min_db, max_db, f64)


def oracle_level_histograms(buf, datatype, start_sample, nfft, hop, window, n_frames, n_levels, min_db, max_db, f64,
                            db_mode=0, eof_fill_db=-150.0, strict_reference=False, tol=None, perturb=None):
    """Histograms (H_lo, H_hi) of the lower / upper level bounds of every frame.  perturb(m, eps) -> m', when given,
    also returns the histogram of the levels of perturbed magnitudes, rounded to the launch's precision."""
    _, zeros, _ = _layout(buf, datatype, strict_reference)
    h_lo = np.zeros((n_levels, nfft), np.int64)
    h_hi = np.zeros((n_levels, nfft), np.int64)
    h_p = np.zeros((n_levels, nfft), np.int64) if perturb else None
    for _, m, readable in oracle_slabs(buf, datatype, start_sample, nfft, hop, window, n_frames, strict_reference):
        lo, hi = level_bounds(m, readable, n_levels, min_db, max_db, f64, db_mode, eof_fill_db, zeros, tol)
        h_lo += histogram_of_levels(lo, n_levels)
        h_hi += histogram_of_levels(hi, n_levels)
        if perturb:
            t = (NORM_TOL_F64 if f64 else NORM_TOL_F32) if tol is None else tol
            eps = t * np.sqrt(np.mean(m * m, axis=1, keepdims=True))
            with np.errstate(divide="ignore"):
                d = mag_to_db(np.maximum(perturb(m, eps), 0.0), db_mode)
            d[~readable] = eof_fill_db
            if zeros:
                d[readable] = -200.0
            h_p += histogram(d.astype(np.float64 if f64 else np.float32), n_levels, min_db, max_db, f64)
    return (h_lo, h_hi, h_p) if perturb else (h_lo, h_hi)


def counts_within_bounds(counts, h_lo, h_hi, n_frames):
    """None when every column sums to n_frames and #{hi < j} <= sum_{l<j} counts[l] <= #{lo < j} at every boundary j;
    else a message naming the first violation."""
    counts = np.asarray(counts, np.int64)
    sums = counts.sum(axis=0)
    if not np.all(sums == n_frames):
        k = int(np.argmax(sums != n_frames))
        return "column %d sums to %d, not %d" % (k, sums[k], n_frames)
    c = np.cumsum(counts, axis=0)[:-1]                # sum_{l<j} counts[l], j = 1 .. n_levels-1
    a = np.cumsum(h_hi, axis=0)[:-1]                  # #{hi < j}
    b = np.cumsum(h_lo, axis=0)[:-1]                  # #{lo < j}
    bad = (c < a) | (c > b)
    if bad.any():
        j, k = np.argwhere(bad)[0]
        return "boundary %d bin %d: %d counts below it, bounds [%d, %d]" % (j + 1, k, c[j, k], a[j, k], b[j, k])
    return None


def check_against_oracle(counts, buf, datatype, start_sample, nfft, hop, window, n_frames, n_levels, min_db, max_db,
                         f64, db_mode=0, eof_fill_db=-150.0, strict_reference=False):
    h_lo, h_hi = oracle_level_histograms(buf, datatype, start_sample, nfft, hop, window, n_frames, n_levels, min_db,
                                         max_db, f64, db_mode, eof_fill_db, strict_reference)
    return counts_within_bounds(counts, h_lo, h_hi, n_frames)
