"""Spectrum traces (sa_spectrum_trace / sa_spectrum_trace_device) against the FP64 oracle on the GPU.

Input: seeded, non-repeating white noise plus three tones whose bins stand 3 .. 10 dB above the noise, generated on the
device and quantised per datatype.  The tones stay weak on purpose: the norm-wise comparator divides by the rms of a
row, so a tone far above the noise would multiply the FP32 error of its bin (and the float32 rounding of its dB value)
by its peak-to-rms ratio, up to sqrt(nfft).
Trace rows are compared as frames on linear magnitude within NORM_TOL_F32 / NORM_TOL_F64: MEAN and MAX with
util.frame_norm_error against their own rows; MIN against the scale of the frames it was taken from, the rms of the
reference MEAN row (the minimum of F powers is about 1/F of their mean, so the MIN row's own rms is no error scale for
the transform).  MEAN also stays within 1e-3 dB on the bins within 40 dB of the row maximum, in rows of at least 7
frames (a one-frame mean is a single periodogram, whose Rayleigh nulls reach into that range).

  (a) every in-SM family x decode kind (FP32: cf32 LE/BE, ci16, cu8 / ci8, 64 .. 16384; FP64: cf64 and the others,
      64 .. 8192), rect and windowed, aligned and unaligned, on 2 W + r frames with EOF frames in the last row; F in
      {1, 7, 3*256 + 5, n_frames} with all three statistics, and each statistic alone (MAX / MIN bit-identical to the
      three-statistic launch);
  (b) the four-step sizes, FP32 and FP64, over at least two workspace chunks;
  (c) one row of all three statistics over 2^17 + 5 frames at 1024 points, run twice (MAX / MIN bit-identical);
  (d) the host entry against the device entry over more host chunks than pipeline slots (small SA_CHUNK_MB);
  (e) strict-reference zero decodes (constant rows) on the host and device paths; (f) every argument error.
Each case asserts the transform kernel the dispatch reports.
"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import trace_reference as tr
from oracle import c_oracle as co
from spectral_analyzer_b200 import _capi
from util import NORM_TOL_F32, NORM_TOL_F64, frame_norm_error

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BPS = {"cf32": 8, "ci16": 4, "cu8": 2, "ci8": 2, "cf64": 16}
VARIANTS = {"cf32": ("cf32_le", "cf32_be"), "ci16": ("ci16_le", "ci16_be"), "c8": ("cu8", "ci8"),
            "cf64": ("cf64_le", "cf64_be")}
WINDOWS = ["hann", "hamming", "blackman", "blackman_harris"]
P_F32 = {64: 8, 128: 16, 256: 16, 512: 32, 1024: 32, 2048: 32, 4096: 32, 8192: 32, 16384: 32}
P_F64 = {64: 8, 128: 16, 256: 16, 512: 16, 1024: 16, 2048: 16, 4096: 16, 8192: 16}
STATS = ("mean", "max", "min")
PE_MAG = (10 ** (-150.0 / 20) - 1e-10) ** 2          # the power of an EOF frame (eof_fill_db = -150, MAG_1E10)


def dk_name(dt):
    k = dt.split("_")[0]
    return "c8" if k in ("cu8", "ci8") else k


def expected_kernel(prec, nfft, dt, win, aligned):
    """The spectrogram dispatch (engine.cu launch_spectrogram), with the mid kernel at 4096 points (the radix-64
    kernel has its own store code) and the pooled rows kernel on the four-step path."""
    dk = dk_name(dt)
    if prec == "f64":
        if nfft > 8192:
            return ("large_cols_kernel+large_rows_kernel(pooled)<double,", ",%s,window>" % dk)
        return ("spectrogram_kernel<double,%d,%s,window>" % (nfft, dk), "")
    w = "rect" if win == "rect" else "window"
    if nfft > 16384:
        return ("large_cols_kernel+large_rows_kernel(pooled)<float,", ",%s,%s>" % (dk, w))
    if not aligned or nfft <= 512:
        fam = "spectrogram_kernel"
    elif nfft == 1024:
        fam = "spectrogram_tma_kernel"
    elif nfft == 8192:
        fam = "spectrogram_mid_kernel"
    else:
        fam = "spectrogram_mid_kernel(prefetch)"
    return ("%s<float,%d,%s,%s>" % (fam, nfft, dk, w), "")


def assert_kernel(engine, want):
    name, (pre, suf) = engine.last_kernel, want
    assert (name.startswith(pre) and name.endswith(suf)) if suf else name == pre, (name, want)


@pytest.fixture(scope="module")
def wave():
    p = torch.cuda.get_device_properties(0)
    return lambda nfft, ppt: p.multi_processor_count * (p.max_threads_per_multi_processor // (nfft // ppt))


def tone_noise(dt, n, nfft, seed):
    """White noise (unit variance per component) plus three tones whose bins stand 10, 7 and 3 dB above the noise in an
    nfft-point frame, on the device, as raw bytes of `dt`."""
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    t = torch.arange(n, device=DEV, dtype=torch.float64)
    ph = torch.rand(3, device=DEV, dtype=torch.float64, generator=g) * 2 * np.pi
    z = torch.randn(n, 2, device=DEV, dtype=torch.float64, generator=g)
    for i, (f, snr_db) in enumerate(((0.1234567, 10.0), (-0.3141593, 7.0), (0.4101010, 3.0))):
        a = np.sqrt(2 * 10 ** (snr_db / 10) / nfft)             # |tone bin|^2 = a^2 nfft^2 vs noise 2 nfft per bin
        z[:, 0] += a * torch.cos(2 * np.pi * f * t + ph[i])
        z[:, 1] += a * torch.sin(2 * np.pi * f * t + ph[i])
    kind = dt.split("_")[0]
    if kind == "cf32":
        x = z.float().view(torch.uint8).reshape(-1)
    elif kind == "cf64":
        x = z.contiguous().view(torch.uint8).reshape(-1)
    elif kind == "ci16":
        x = (z * 3000).round().to(torch.int16).view(torch.uint8).reshape(-1)
    elif kind == "cu8":
        x = (z * 20 + 127.5).round().clamp(0, 255).to(torch.uint8).reshape(-1)
    else:
        x = (z * 20).round().clamp(-128, 127).to(torch.int8).view(torch.uint8).reshape(-1)
    if kind in ("cf32", "ci16", "cf64") and not dt.endswith("_le"):
        elem = {"cf32": 4, "ci16": 2, "cf64": 8}[kind]
        x = x.view(-1, elem).flip(1).reshape(-1)
    return x.contiguous()


def level(p):
    return 20 * np.log10(np.sqrt(p) + 1e-10)


def ref_power(host, dt, start, nfft, hop, win, frames):
    """|X_t|^2 of every frame (fft-shifted), EOF frames at the EOF power"""
    n = host.size // BPS[dt.split("_")[0]]
    db = co.spectrogram(host, dt, start, nfft, hop, win, frames, db_mode=co.DB_POWER)
    p = np.power(10.0, db / 10) - 1e-20
    eof = start + np.arange(frames) * hop + nfft > n
    p[eof] = PE_MAG
    return p


def ref_traces(p, F):
    idx = np.arange(0, p.shape[0], F)
    cnt = np.diff(np.append(idx, p.shape[0])).astype(np.float64)
    return {"mean": level(np.add.reduceat(p, idx, axis=0) / cnt[:, None]),
            "max": level(np.maximum.reduceat(p, idx, axis=0)), "min": level(np.minimum.reduceat(p, idx, axis=0))}


def run_trace(engine, d_iq, iq_bytes, dt, nfft, hop, win, frames, start, F, stats=STATS, prec="auto", out="f32", **kw):
    n_rows = -(-frames // F)
    esz = 8 if out == "f64" else 4
    outs = {s: torch.empty(n_rows * nfft * esz, dtype=torch.uint8, device=DEV) for s in stats}
    p = engine.make_params(dt, nfft, hop, win, n_frames=frames, start_sample=start, out=out, precision=prec, **kw)
    ptr = [outs[s].data_ptr() if s in outs else None for s in STATS]
    engine.spectrum_trace_device(d_iq.data_ptr(), iq_bytes, p, F, *ptr, n_rows * nfft * esz,
                                 torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ft = torch.float64 if out == "f64" else torch.float32
    return {s: v.view(ft).view(n_rows, nfft).cpu().numpy() for s, v in outs.items()}


def row_counts(frames, F):
    return np.minimum(F, frames - np.arange(-(-frames // F)) * F)


def check_trace(got, ref, tol, counts):
    """MEAN / MAX: util.frame_norm_error against their own rows; MIN: the same error over the rms of the reference MEAN
    row (see the module docstring); MEAN also 1e-3 dB on the bins within 40 dB of the row maximum in rows of >= 7
    frames.  Returns the worst norm-wise error."""
    worst = 0.0
    for s, g in got.items():
        r = ref[s]
        assert np.isfinite(g).all(), s
        if s == "min":
            a_g, a_r = np.power(10.0, g.astype(np.float64) / 20), np.power(10.0, r / 20)
            e = np.abs(a_g - a_r).max(axis=1) / np.sqrt(np.mean(np.power(10.0, ref["mean"] / 10), axis=1))
        else:
            e = frame_norm_error(g, r)
        assert e.max() <= tol, "%s: worst E %.3g > %.3g at row %d" % (s, e.max(), tol, int(e.argmax()))
        worst = max(worst, float(e.max()))
        if s == "mean":
            strong = (r >= r.max(axis=1, keepdims=True) - 40) & (counts >= 7)[:, None]
            if strong.any():
                d = np.abs(g.astype(np.float64) - r)[strong].max()
                assert d <= 1e-3, "mean: %.3g dB on strong bins" % d
    return worst


# ---------------- (a) in-SM kernels ----------------

def insm_cases():
    out = []
    for k, nfft in enumerate([64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384]):
        for d, dk in enumerate(("cf32", "ci16", "c8")):
            i = len(out)
            dt = VARIANTS[dk][(k + d) % 2]
            win = "rect" if (k + d) % 2 == 0 else WINDOWS[(k + d) % 4]
            aligned = (k + d) % 3 != 2
            if aligned:
                hop, start = [nfft, nfft // 2, nfft + nfft // 8][(k + d) % 3], [0, 16][k % 2]
            else:
                hop, start = ([nfft - 1, 0] if (k + d) % 2 else [nfft, 3])      # odd hop / WAV-style odd start
            out.append(("f32", nfft, dt, win, hop, start, aligned, 3 + i % 5))
    for k, nfft in enumerate([64, 128, 256, 512, 1024, 2048, 4096, 8192]):
        for d, dk in enumerate(("cf64", ("cf32", "ci16", "c8")[k % 3])):
            i = len(out)
            dt = VARIANTS[dk][(k + d) % 2]
            win = (["rect"] + WINDOWS)[(k + d) % 5]
            hop, start = [(nfft, 0), (nfft // 2 + 1, 5), (nfft + nfft // 8, 0)][(k + d) % 3]
            out.append(("f64", nfft, dt, win, hop, start, True, 3 + i % 5))
    return out


def cid(c):
    return "%s-%d-%s-%s-hop%d-start%d" % c[:6]


@pytest.mark.parametrize("prec,nfft,dt,win,hop,start,aligned,r", insm_cases(), ids=[cid(c) for c in insm_cases()])
def test_insm_trace_past_first_wave(engine, wave, prec, nfft, dt, win, hop, start, aligned, r):
    f64 = prec == "f64"
    frames = 2 * wave(nfft, P_F64[nfft] if f64 else P_F32[nfft]) + r
    n = start + (frames - 3) * hop + nfft + hop // 3                   # the last two frames are EOF
    d_iq = tone_noise(dt, n, nfft, seed=nfft * 7 + hop + start)
    host = d_iq.cpu().numpy()
    p = ref_power(host, dt, start, nfft, hop, win, frames)
    tol = NORM_TOL_F64 if f64 else NORM_TOL_F32
    out = "f64" if f64 else "f32"
    want = expected_kernel(prec, nfft, dt, win, aligned)
    Fs = [1, 7, 3 * 256 + 5, frames]
    full = {}
    for F in Fs:
        ref = ref_traces(p, F)
        full[F] = run_trace(engine, d_iq, n * BPS[dt.split("_")[0]], dt, nfft, hop, win, frames, start, F,
                            prec=prec if f64 else "auto", out=out)
        assert_kernel(engine, want)
        check_trace(full[F], ref, tol, row_counts(frames, F))
    for j, s in enumerate(STATS):                                     # each statistic alone
        F = Fs[(j + r) % 4]
        one = run_trace(engine, d_iq, n * BPS[dt.split("_")[0]], dt, nfft, hop, win, frames, start, F, stats=(s,),
                        prec=prec if f64 else "auto", out=out)
        assert_kernel(engine, want)
        if s == "mean":
            check_trace(one, {"mean": ref_traces(p, F)["mean"]}, tol, row_counts(frames, F))
        else:
            assert np.array_equal(one[s], full[F][s]), s


# ---------------- (b) four-step sizes ----------------

FOUR_STEP = [("f32", 32768, "cu8", "hann", 32768, 0, 2048 + 41), ("f32", 65536, "cf32_be", "rect", 65536, 0, 1024 + 23),
             ("f64", 16384, "ci16_le", "hann", 16385, 7, 2048 + 37), ("f64", 32768, "cf64_le", "blackman", 32768, 0, 1024 + 9),
             ("f64", 65536, "cf32_le", "rect", 65536, 0, 512 + 19)]


@pytest.mark.parametrize("prec,nfft,dt,win,hop,start,frames", FOUR_STEP, ids=["%s-%d-%s" % c[:3] for c in FOUR_STEP])
def test_four_step_trace(engine, prec, nfft, dt, win, hop, start, frames):
    chunk = (512 << 20) // (nfft * (16 if prec == "f64" else 8))
    assert frames > chunk                                             # at least two workspace chunks
    n = start + (frames - 3) * hop + nfft + hop // 2
    d_iq = tone_noise(dt, n, nfft, seed=nfft + frames)
    host = d_iq.cpu().numpy()
    tol = NORM_TOL_F64 if prec == "f64" else NORM_TOL_F32
    for F in (7, 3 * 256 + 5, frames):
        got = run_trace(engine, d_iq, n * BPS[dt.split("_")[0]], dt, nfft, hop, win, frames, start, F, prec=prec,
                        out="f64" if prec == "f64" else "f32")
        assert_kernel(engine, expected_kernel(prec, nfft, dt, win, True))
        ref = tr.spectrum_trace(host, dt, start, nfft, hop, win, frames, F)
        check_trace(got, ref, tol, row_counts(frames, F))


# ---------------- (c) long integration ----------------

def test_long_integration_is_bounded_and_reproducible(engine):
    """One row of 2^17 + 5 frames at 1024 points: FP32 cells of at most 256 frames keep MEAN within the norm-wise and
    dB bounds; MAX and MIN are bit-identical between two runs."""
    nfft, hop, frames = 1024, 512, (1 << 17) + 5
    n = (frames - 1) * hop + nfft
    d_iq = tone_noise("cf32_le", n, nfft, seed=17)
    host = d_iq.cpu().numpy()
    a = run_trace(engine, d_iq, n * 8, "cf32_le", nfft, hop, "hann", frames, 0, frames)
    assert_kernel(engine, expected_kernel("f32", nfft, "cf32_le", "hann", True))
    b = run_trace(engine, d_iq, n * 8, "cf32_le", nfft, hop, "hann", frames, 0, frames)
    assert np.array_equal(a["max"], b["max"]) and np.array_equal(a["min"], b["min"])
    check_trace(a, tr.spectrum_trace(host, "cf32_le", 0, nfft, hop, "hann", frames, frames), NORM_TOL_F32,
                row_counts(frames, frames))


# ---------------- (d) host entry against device entry ----------------

HOST_SCRIPT = r"""
import json, sys
import numpy as np, torch
sys.path.insert(0, sys.argv[1])
import spectral_analyzer_b200 as sa
a = json.loads(sys.argv[2])
raw = np.load(a["raw"])
eng = sa.Engine(0)
res = {}
pinned = torch.from_numpy(raw).pin_memory()
for tag, buf in (("pageable", raw), ("pinned", pinned.numpy())):
    got = eng.spectrum_trace(buf, a["dt"], a["nfft"], a["frames"], hop=a["hop"], window=a["win"], start_sample=a["start"],
                             frames_per_row=a["F"], stats=("mean", "max", "min"))
    for s, v in got.items():
        res[tag + "_" + s] = v
    res[tag + "_kernel"] = np.array(eng.last_kernel)
np.savez(a["out"], **res)
"""


@pytest.mark.parametrize("nfft,dt,win,hop,F", [(1024, "cf32_le", "hann", 512, 3 * 256 + 5), (2048, "cu8", "rect", 2048, 100),
                                             (32768, "ci16_le", "blackman_harris", 32768, 5)])
def test_host_entry_matches_device_entry(engine, tmp_path, nfft, dt, win, hop, F):
    bps = BPS[dt.split("_")[0]]
    frames = max(64, (24 << 20) // (hop * bps)) + 3
    n = (frames - 2) * hop + nfft
    d_iq = tone_noise(dt, n, nfft, seed=nfft + F)
    dev = run_trace(engine, d_iq, n * bps, dt, nfft, hop, win, frames, 0, F)
    dev_kernel = engine.last_kernel
    raw = d_iq.cpu().numpy()
    np.save(tmp_path / "raw.npy", raw)
    args = {"raw": str(tmp_path / "raw.npy"), "out": str(tmp_path / "host.npz"), "dt": dt, "nfft": nfft, "frames": frames,
            "hop": hop, "win": win, "start": 0, "F": F}
    env = dict(os.environ, SA_CHUNK_MB="1" if nfft <= 2048 else "4")      # far more chunks than the three slots
    assert frames * hop * bps > 3 * (int(env["SA_CHUNK_MB"]) << 20)
    subprocess.run([sys.executable, "-c", HOST_SCRIPT, ROOT, json.dumps(args)], check=True, env=env, timeout=900)
    host = np.load(tmp_path / "host.npz")
    for tag in ("pageable", "pinned"):
        assert str(host[tag + "_kernel"]) == dev_kernel
        assert np.array_equal(host[tag + "_max"], dev["max"]) and np.array_equal(host[tag + "_min"], dev["min"])
        e = frame_norm_error(host[tag + "_mean"], dev["mean"])
        assert e.max() <= NORM_TOL_F32, e.max()


# ---------------- (e) strict-reference zero decodes ----------------

@pytest.mark.parametrize("dt", ["cf64_le", "ri16_le"])
def test_strict_zero_trace_constants(engine, dt):
    nfft, hop, F, frames = 256, 256, 3, 11
    bps = 16 if dt.startswith("cf64") else 8
    raw = np.random.default_rng(1).integers(0, 256, (frames - 3) * hop * bps + nfft * bps, dtype=np.uint8)
    ref = tr.spectrum_trace(raw, dt, 0, nfft, hop, "hann", frames, F, strict_reference=True)
    got = engine.spectrum_trace(raw, dt, nfft, frames, hop=hop, window="hann", frames_per_row=F, stats=STATS,
                                strict_reference=True)
    d_iq = torch.from_numpy(raw).to(DEV)
    dev = run_trace(engine, d_iq, raw.size, dt, nfft, hop, "hann", frames, 0, F, strict_reference=True)
    for s in STATS:
        assert np.allclose(got[s], ref[s], atol=1e-4, rtol=0) and np.allclose(dev[s], ref[s], atol=1e-4, rtol=0), s
    assert np.allclose(ref["mean"][-1], -150.0) and np.allclose(ref["min"][0], -200.0)


# ---------------- (f) argument errors ----------------

def test_argument_errors(engine):
    L = _capi.lib()
    raw = np.zeros(1 << 16, np.uint8)
    d_iq = torch.zeros(1 << 16, dtype=torch.uint8, device=DEV)
    out = torch.empty(1 << 16, dtype=torch.uint8, device=DEV)
    h_out = np.empty(1 << 16, np.uint8)

    def both(p, F, outs_on, nb, d_ptr=None):
        po = [out.data_ptr() if o else None for o in outs_on]
        ho = [h_out.ctypes.data if o else None for o in outs_on]
        rd = L.sa_spectrum_trace_device(engine.handle, d_ptr or d_iq.data_ptr(), 1 << 16, C.byref(p), F, *po, nb, None)
        rh = L.sa_spectrum_trace(engine.handle, raw.ctypes.data, raw.size, C.byref(p), F, *ho, nb)
        return rd, rh

    p = engine.make_params("cf32_le", 256, 256, "hann", n_frames=10)
    assert both(p, 0, (1, 1, 1), 1 << 16) == (1, 1)                           # frames_per_row == 0
    assert both(p, 3, (0, 0, 0), 1 << 16) == (1, 1)                           # no statistic
    p0 = engine.make_params("cf32_le", 256, 256, "hann", n_frames=0)
    assert both(p0, 3, (1, 0, 0), 1 << 16) == (1, 1)                          # n_frames == 0
    pr = engine.make_params("cf32_le", 256, 256, "hann", n_frames=10, out="rgba8", sample_rate=1.0)
    assert both(pr, 3, (1, 0, 0), 1 << 16) == (1, 1)                          # RGBA
    assert both(p, 3, (0, 1, 1), 4 * 256 * 4 - 1) == (7, 7)                   # 4 rows x 256 x 4 bytes needed
    assert both(p, 3, (0, 1, 1), 4 * 256 * 4) == (0, 0)
    rd = L.sa_spectrum_trace_device(engine.handle, d_iq.data_ptr() + 4, 1 << 15, C.byref(p), 3, out.data_ptr(), None,
                                    None, 1 << 16, None)
    assert rd == 1                                                            # d_iq not aligned to one IQ pair
    torch.cuda.synchronize()
