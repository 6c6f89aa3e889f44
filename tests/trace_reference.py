"""FP64 references of the spectrum traces (sa_spectrum_trace), built from the oracle's spectrogram restatements.

Row r reduces frames [r F, min((r + 1) F, n_frames)) of the spectrogram; per frame t and bin k (fft-shifted) the power
is P_t[k] = |X_t[k]|^2 (0 for the strict-reference zero decodes: cf64 with strict_reference, or a datatype without a
decode branch), or for a frame past the end of the buffer the power whose level is eof_fill_db.  MEAN = sum P / count
(EOF frames counted), MAX = max P, MIN = min P, each leveled once: 20 log10(sqrt(P) + 1e-10) (db_mode 0) or
10 log10(P + 1e-20) (db_mode 1).

Two independent restatements that check each other (tests/test_oracle_trace.py):
  spectrum_trace     |X|^2 from the C oracle (oracle/sa_oracle.c, power-mode rows, FP64), streamed in slabs of frames;
  spectrum_trace_np  |X|^2 from numpy's FFT on oracle/np_oracle.decode, frame by frame.
"""
import numpy as np

from oracle import c_oracle as co
from oracle import np_oracle as npo

STATS = ("mean", "max", "min")
BPS = {"cf32": 8, "ci16": 4, "cu8": 2, "ci8": 2, "cf64": 16}
SLAB = 1 << 22                      # points per oracle call


def eof_power(db_mode, eof_fill_db):
    if db_mode == 0:
        return max(0.0, 10 ** (eof_fill_db / 20) - 1e-10) ** 2
    return max(0.0, 10 ** (eof_fill_db / 10) - 1e-20)


def level(p, db_mode):
    return 20 * np.log10(np.sqrt(p) + 1e-10) if db_mode == 0 else 10 * np.log10(p + 1e-20)


def _layout(buf, datatype, strict_reference):
    kind = datatype.split("_")[0]
    known = kind in BPS
    bps = BPS[kind] if known else 8                                  # Global.getBytesPerSample fallback
    zeros = (not known) or (kind == "cf64" and strict_reference)     # SpectralService.java:60-63
    return bps, zeros, np.ascontiguousarray(buf).view(np.uint8).size


class _Rows:
    """FP64 running sum / max / min per output row, fed with blocks of consecutive frames."""

    def __init__(self, n_frames, F, nfft):
        self.F, self.n = F, n_frames
        n_rows = -(-n_frames // F)
        self.sum = np.zeros((n_rows, nfft))
        self.max = np.full((n_rows, nfft), -np.inf)
        self.min = np.full((n_rows, nfft), np.inf)

    def add(self, f0, p):
        rows = (f0 + np.arange(p.shape[0])) // self.F
        for r in np.unique(rows):
            blk = p[rows == r]
            self.sum[r] += blk.sum(axis=0)
            np.maximum(self.max[r], blk.max(axis=0), out=self.max[r])
            np.minimum(self.min[r], blk.min(axis=0), out=self.min[r])

    def levels(self, db_mode, stats):
        cnt = np.minimum(self.F, self.n - np.arange(self.sum.shape[0]) * self.F).astype(np.float64)
        val = {"mean": self.sum / cnt[:, None], "max": self.max, "min": self.min}
        return {s: level(val[s], db_mode) for s in STATS if s in stats}


def spectrum_trace(buf, datatype, start_sample, nfft, hop, window, n_frames, frames_per_row, db_mode=0,
                   eof_fill_db=-150.0, strict_reference=False, stats=STATS):
    """{stat: [ceil(n_frames / F), nfft]} FP64 levels, |X|^2 from the C oracle's power-mode rows."""
    bps, zeros, cap = _layout(buf, datatype, strict_reference)
    acc = _Rows(n_frames, frames_per_row, nfft)
    pe = eof_power(db_mode, eof_fill_db)
    step = max(1, SLAB // nfft)
    for f0 in range(0, n_frames, step):
        nf = min(step, n_frames - f0)
        t = f0 + np.arange(nf)
        readable = (start_sample + t * hop + nfft) * bps <= cap                  # MainController.java:987
        if zeros:
            p = np.zeros((nf, nfft))
        else:
            db = co.spectrogram(buf, datatype, start_sample + f0 * hop, nfft, hop, window, nf, db_mode=co.DB_POWER)
            p = np.power(10.0, db / 10) - 1e-20
        p[~readable] = pe
        acc.add(f0, p)
    return acc.levels(db_mode, stats)


def spectrum_trace_np(buf, datatype, start_sample, nfft, hop, window, n_frames, frames_per_row, db_mode=0,
                      eof_fill_db=-150.0, strict_reference=False, stats=STATS):
    """The same from numpy's FFT, frame by frame (independent of oracle/sa_oracle.c)."""
    bps, zeros, cap = _layout(buf, datatype, strict_reference)
    acc = _Rows(n_frames, frames_per_row, nfft)
    pe = eof_power(db_mode, eof_fill_db)
    w = npo.window(window, nfft)
    for t in range(n_frames):
        off = (start_sample + t * hop) * bps
        if off + nfft * bps > cap:
            p = np.full(nfft, pe)
        elif zeros:
            p = np.zeros(nfft)
        else:
            p = np.fft.fftshift(np.abs(np.fft.fft(npo.decode(buf, off, nfft, datatype) * w)) ** 2)
        acc.add(t, p[None, :])
    return acc.levels(db_mode, stats)
