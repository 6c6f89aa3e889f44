"""Persistence spectra (sa_spectrum_persistence / sa_spectrum_persistence_device) on the GPU.

  (a) exact identity past the first wave: every in-SM family x decode kind (the trace test's case matrix: FP32 cf32
      LE/BE, ci16, cu8 / ci8, 64 .. 16384; FP64 cf64 and the others, 64 .. 8192), rect and windowed, aligned and
      unaligned, both db_modes, n_levels in {2, 37, 256} over ranges that clip on both sides, on 2 W + r frames with EOF
      frames: the counts equal the histogram (tests/persistence_reference.py) of the same engine's F32 rows (FP32
      launches) or F64 rows (FP64 launches) from sa_spectrogram_device, where that runs the same transform kernel;
  (b) the four-step sizes over at least two transform-workspace chunks and two level-row chunks, the same identity;
  (c) one case per family against the FP64 oracle with the comparator of tests/persistence_reference.py, on
      gain-stepped noise plus tones (4096 cf32 aligned included: its level rows come from the mid kernel, its dB rows
      from radix-64);
  (d) the host entry against the device entry, byte for byte, from pageable and pinned memory over many more chunks
      than pipeline slots; (e) a pure tone (every frame of a bin on one level); (f) strict-reference zero decodes,
      EOF-only requests and byte-identical reruns; (g) every argument error; (h) the C++ binding.
Each case asserts the kernels the dispatch reports.
"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import persistence_reference as pr
import test_gpu_spectrum_trace as gt
from spectral_analyzer_b200 import _capi

pytestmark = pytest.mark.gpu
DEV = gt.DEV
ROOT = gt.ROOT
BPS = gt.BPS
HIST = "+persistence_hist_kernel"
LEVELS = [(2, -60.0, 25.0), (37, -10.0, 30.0), (256, 5.0, 28.0)]      # every range clips noise bins on both sides


def transform_kernel(prec, nfft, dt, win, aligned):
    """The transform kernel of a persistence launch: the trace dispatch (the mid kernel at 4096 points), with the rows
    kernel's name on the four-step path."""
    pre, suf = gt.expected_kernel(prec, nfft, dt, win, aligned)
    return pre.replace("(pooled)", ""), suf


def rows_kernel_differs(prec, nfft, dt, aligned):
    """Cases whose dB rows come from another kernel: radix-64 at 4096 points for aligned cf32 / ci16."""
    return prec == "f32" and aligned and nfft == 4096 and gt.dk_name(dt) in ("cf32", "ci16")


def assert_kernels(engine, want):
    """the transform kernel `want` (as gt.assert_kernel), then the histogram kernel"""
    name, (pre, suf) = engine.last_kernel, want
    assert name.endswith(HIST), name
    base = name[:-len(HIST)]
    assert (base.startswith(pre) and base.endswith(suf)) if suf else base == pre, (name, want)


@pytest.fixture(scope="module")
def wave():
    p = torch.cuda.get_device_properties(0)
    return lambda nfft, ppt: p.multi_processor_count * (p.max_threads_per_multi_processor // (nfft // ppt))


def gain_noise(dt, n, nfft, hop, seed):
    """tone_noise with a gain that steps by 10 dB every hop samples over 7 steps, so that neighbouring frames land on
    different levels (raw bytes of `dt` on the device)."""
    raw = gt.tone_noise("cf64_le", n, nfft, seed).view(torch.float64).view(n, 2)
    g = torch.pow(10.0, -((torch.arange(n, device=DEV) // hop) % 7).double() / 2)
    z = raw * g[:, None] * 4
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


def run_persistence(engine, d_iq, iq_bytes, dt, nfft, hop, win, frames, start, n_levels, lo, hi, prec="auto", **kw):
    counts = torch.empty(n_levels * nfft, dtype=torch.int32, device=DEV)
    p = engine.make_params(dt, nfft, hop, win, n_frames=frames, start_sample=start, precision=prec, **kw)
    engine.spectrum_persistence_device(d_iq.data_ptr(), iq_bytes, p, n_levels, lo, hi, counts.data_ptr(),
                                       counts.numel() * 4, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return counts.cpu().numpy().view(np.uint32).reshape(n_levels, nfft)


def run_rows(engine, d_iq, iq_bytes, dt, nfft, hop, win, frames, start, f64, prec="auto", **kw):
    out = torch.empty(frames * nfft, dtype=torch.float64 if f64 else torch.float32, device=DEV)
    p = engine.make_params(dt, nfft, hop, win, n_frames=frames, start_sample=start, precision=prec,
                           out="f64" if f64 else "f32", **kw)
    engine.spectrogram_device(d_iq.data_ptr(), iq_bytes, p, out.data_ptr(), out.numel() * out.element_size(),
                              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out.view(frames, nfft)


def torch_histogram(rows, n_levels, lo, hi, f64, slab=1 << 26):
    """persistence_reference.histogram on the device, slab by slab: every elementwise operation rounds on its own, as
    numpy's and the kernel's do."""
    nfft = rows.shape[1]
    ft = torch.float64 if f64 else torch.float32
    mn = torch.tensor(lo, dtype=torch.float64).to(ft).item()
    s = torch.tensor(n_levels / (hi - lo), dtype=torch.float64).to(ft).item()
    counts = torch.zeros(n_levels * nfft, dtype=torch.int64, device=DEV)
    k = torch.arange(nfft, device=DEV)
    step = max(1, slab // nfft)
    for f0 in range(0, rows.shape[0], step):
        d = rows[f0:f0 + step].to(ft)
        u = torch.mul(torch.sub(d, torch.tensor(mn, dtype=ft, device=DEV)), torch.tensor(s, dtype=ft, device=DEV))
        lv = torch.where(u >= 1, torch.clamp(u, max=n_levels - 1).floor(), torch.zeros_like(u)).long()
        counts += torch.bincount((lv * nfft + k).reshape(-1), minlength=n_levels * nfft)
    return counts.view(n_levels, nfft).cpu().numpy()


def test_torch_histogram_restates_the_reference():
    x = torch.randn(3000, 64, device=DEV, dtype=torch.float64) * 30
    for f64 in (False, True):
        rows = x if f64 else x.float()
        for n_levels, lo, hi in LEVELS:
            assert np.array_equal(torch_histogram(rows, n_levels, lo, hi, f64, slab=1 << 14),
                                  pr.histogram(rows.cpu().numpy(), n_levels, lo, hi, f64))


# ---------------- (a) exact identity, in-SM kernels ----------------

CASES = gt.insm_cases()


@pytest.mark.parametrize("prec,nfft,dt,win,hop,start,aligned,r", CASES, ids=[gt.cid(c) for c in CASES])
def test_insm_counts_are_the_histogram_of_the_rows(engine, wave, prec, nfft, dt, win, hop, start, aligned, r):
    f64 = prec == "f64"
    frames = 2 * wave(nfft, gt.P_F64[nfft] if f64 else gt.P_F32[nfft]) + r
    n = start + (frames - 3) * hop + nfft + hop // 3                   # the last two frames are EOF
    d_iq = gt.tone_noise(dt, n, nfft, seed=nfft * 5 + hop + start)
    nb = n * BPS[dt.split("_")[0]]
    pp = prec if f64 else "auto"
    want = transform_kernel(prec, nfft, dt, win, aligned)
    rows = {}
    for i, (n_levels, lo, hi) in enumerate(LEVELS):
        db_mode = (i + r) % 2
        got = run_persistence(engine, d_iq, nb, dt, nfft, hop, win, frames, start, n_levels, lo, hi, pp, db_mode=db_mode)
        assert_kernels(engine, want)
        assert np.all(got.sum(axis=0) == frames)
        if rows_kernel_differs(prec, nfft, dt, aligned):
            err = pr.check_against_oracle(got, d_iq.cpu().numpy(), dt, start, nfft, hop, win, frames, n_levels, lo, hi,
                                          f64, db_mode)
            assert err is None, err
            continue
        if db_mode not in rows:
            rows[db_mode] = run_rows(engine, d_iq, nb, dt, nfft, hop, win, frames, start, f64, pp, db_mode=db_mode)
            gt.assert_kernel(engine, want)                         # the rows come from the same transform kernel
        ref = torch_histogram(rows[db_mode], n_levels, lo, hi, f64)
        assert np.array_equal(got, ref), (n_levels, int(np.abs(got.astype(np.int64) - ref).sum()))


# ---------------- (b) four-step sizes ----------------

FOUR_STEP = [("f32", 32768, "cu8", "hann", 16384, 0, 16384 + 41), ("f32", 65536, "cf32_be", "rect", 8192, 0, 8192 + 23),
             ("f64", 16384, "ci16_le", "hann", 8191, 7, 32768 + 37), ("f64", 32768, "cf64_le", "blackman", 2048, 0, 16384 + 9),
             ("f64", 65536, "cf32_le", "rect", 8192, 0, 8192 + 19)]


@pytest.mark.parametrize("prec,nfft,dt,win,hop,start,frames", FOUR_STEP, ids=["%s-%d-%s" % c[:3] for c in FOUR_STEP])
def test_four_step_counts_are_the_histogram_of_the_rows(engine, prec, nfft, dt, win, hop, start, frames):
    f64 = prec == "f64"
    assert frames > (512 << 20) // (nfft * (16 if f64 else 8))           # at least two workspace chunks
    assert frames > pr.level_chunk_frames(nfft, frames)                   # at least two level-row chunks
    n = start + (frames - 3) * hop + nfft + hop // 2
    nb = n * BPS[dt.split("_")[0]]
    assert nb < (1200 << 20)
    d_iq = gt.tone_noise(dt, n, nfft, seed=nfft + frames)
    want = transform_kernel(prec, nfft, dt, win, True)
    for i, (n_levels, lo, hi) in enumerate(LEVELS[1:]):
        got = run_persistence(engine, d_iq, nb, dt, nfft, hop, win, frames, start, n_levels, lo, hi, prec, db_mode=i)
        assert_kernels(engine, want)
        rows = run_rows(engine, d_iq, nb, dt, nfft, hop, win, frames, start, f64, prec, db_mode=i)
        gt.assert_kernel(engine, want)
        ref = torch_histogram(rows, n_levels, lo, hi, f64)
        del rows
        assert np.array_equal(got, ref), (n_levels, int(np.abs(got.astype(np.int64) - ref).sum()))


# ---------------- (c) against the FP64 oracle ----------------

ORACLE = [("f32", 256, "cf32_le", "hann", 256, 0, True, 37, -60.0, 40.0),           # general
          ("f32", 1024, "cf32_le", "hann", 512, 0, True, 256, -80.0, 60.0),          # TMA 1024
          ("f32", 4096, "cf32_le", "blackman", 4096, 0, True, 256, -80.0, 80.0),     # 4096 cf32 aligned: mid
          ("f32", 8192, "ci16_be", "rect", 4096, 0, True, 37, 20.0, 140.0),          # mid
          ("f32", 2048, "cu8", "hamming", 2048, 16, True, 2, 0.0, 40.0),              # prefetching mid
          ("f32", 16384, "cf32_le", "hann", 16384, 0, True, 64, -60.0, 100.0),       # prefetching mid, 16384
          ("f32", 1024, "ci8", "rect", 1023, 3, False, 100, -40.0, 60.0),             # unaligned
          ("f64", 2048, "cf64_be", "blackman_harris", 2048, 0, True, 256, -90.0, 70.0)]   # FP64


@pytest.mark.parametrize("prec,nfft,dt,win,hop,start,aligned,n_levels,lo,hi", ORACLE,
                         ids=["%s-%d-%s-%s" % c[:4] for c in ORACLE])
def test_counts_against_oracle(engine, wave, prec, nfft, dt, win, hop, start, aligned, n_levels, lo, hi):
    f64 = prec == "f64"
    frames = 2 * wave(nfft, gt.P_F64[nfft] if f64 else gt.P_F32[nfft]) + 5
    n = start + (frames - 2) * hop + nfft
    d_iq = gain_noise(dt, n, nfft, hop, seed=nfft + n_levels)
    host = d_iq.cpu().numpy()
    for db_mode in (0, 1):
        got = run_persistence(engine, d_iq, host.size, dt, nfft, hop, win, frames, start, n_levels, lo, hi,
                              prec if f64 else "auto", db_mode=db_mode)
        assert_kernels(engine, transform_kernel(prec, nfft, dt, win, aligned))
        err = pr.check_against_oracle(got, host, dt, start, nfft, hop, win, frames, n_levels, lo, hi, f64, db_mode)
        assert err is None, err


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
    res[tag] = eng.spectrum_persistence(buf, a["dt"], a["nfft"], a["frames"], a["levels"], a["lo"], a["hi"], hop=a["hop"],
                                        window=a["win"], start_sample=a["start"])
    res[tag + "_kernel"] = np.array(eng.last_kernel)
np.savez(a["out"], **res)
"""


@pytest.mark.parametrize("nfft,dt,win,hop,levels", [(1024, "cf32_le", "hann", 512, 256), (2048, "cu8", "rect", 2048, 37),
                                                    (32768, "ci16_le", "blackman_harris", 32768, 64)])
def test_host_entry_matches_device_entry(engine, tmp_path, nfft, dt, win, hop, levels):
    bps = BPS[dt.split("_")[0]]
    frames = max(64, (24 << 20) // (hop * bps)) + 3
    n = (frames - 2) * hop + nfft
    d_iq = gain_noise(dt, n, nfft, hop, seed=nfft + levels)
    lo, hi = -20.0, 60.0
    dev = run_persistence(engine, d_iq, n * bps, dt, nfft, hop, win, frames, 0, levels, lo, hi)
    dev_kernel = engine.last_kernel
    raw = d_iq.cpu().numpy()
    np.save(tmp_path / "raw.npy", raw)
    args = {"raw": str(tmp_path / "raw.npy"), "out": str(tmp_path / "host.npz"), "dt": dt, "nfft": nfft, "frames": frames,
            "hop": hop, "win": win, "start": 0, "levels": levels, "lo": lo, "hi": hi}
    env = dict(os.environ, SA_CHUNK_MB="1" if nfft <= 2048 else "4")      # far more chunks than the three slots
    assert frames * hop * bps > 3 * (int(env["SA_CHUNK_MB"]) << 20)
    subprocess.run([sys.executable, "-c", HOST_SCRIPT, ROOT, json.dumps(args)], check=True, env=env, timeout=900)
    host = np.load(tmp_path / "host.npz")
    for tag in ("pageable", "pinned"):
        assert str(host[tag + "_kernel"]) == dev_kernel
        assert host[tag].dtype == np.uint32 and np.array_equal(host[tag], dev), tag


# ---------------- (e) worst contention ----------------

def test_pure_tone_lands_on_one_level(engine):
    """Every frame of an on-bin tone without noise holds the same spectrum: each bin's frames all land on one level,
    the worst case for the shared-memory counters of a tile."""
    nfft, hop, frames = 1024, 1024, (1 << 17) + 7
    n = frames * hop
    t = torch.arange(n, device=DEV, dtype=torch.float64)
    z = torch.stack((torch.cos(2 * np.pi * 37 * t / nfft), torch.sin(2 * np.pi * 37 * t / nfft)), 1)
    d_iq = z.float().contiguous().view(torch.uint8).reshape(-1)
    got = run_persistence(engine, d_iq, n * 8, "cf32_le", nfft, hop, "rect", frames, 0, 256, -250.0, 70.0)
    assert_kernels(engine, transform_kernel("f32", nfft, "cf32_le", "rect", True))
    rows = run_rows(engine, d_iq, n * 8, "cf32_le", nfft, hop, "rect", frames, 0, False)
    assert np.array_equal(got, torch_histogram(rows, 256, -250.0, 70.0, False))
    kt = (37 + nfft // 2) % nfft
    assert got[:, kt].max() == frames                                    # the tone bin: one level
    assert np.all(got.sum(axis=0) == frames)


# ---------------- (f) constants and repeats ----------------

@pytest.mark.parametrize("dt", ["cf64_le", "ri16_le"])
def test_strict_zero_constants(engine, dt):
    nfft, hop, frames, levels, lo, hi = 256, 256, 11, 37, -210.0, -100.0
    bps = 16 if dt.startswith("cf64") else 8
    raw = np.random.default_rng(1).integers(0, 256, (frames - 3) * hop * bps + nfft * bps, dtype=np.uint8)
    f64 = dt.startswith("cf64")
    want = np.zeros((levels, nfft), np.uint32)
    want[pr.quantize(np.array([-200.0]), levels, lo, hi, f64)[0]] += frames - 2
    want[pr.quantize(np.array([-150.0]), levels, lo, hi, f64)[0]] += 2
    got = engine.spectrum_persistence(raw, dt, nfft, frames, levels, lo, hi, hop=hop, window="hann",
                                      strict_reference=True)
    assert np.array_equal(got, want)
    dev = run_persistence(engine, torch.from_numpy(raw).to(DEV), raw.size, dt, nfft, hop, "hann", frames, 0, levels,
                          lo, hi, strict_reference=True)
    assert np.array_equal(dev, want)
    assert engine.last_kernel.startswith("persistence_strict_kernel")       # filled on the caller's stream
    h_lo, h_hi = pr.oracle_level_histograms(raw, dt, 0, nfft, hop, "hann", frames, levels, lo, hi, f64,
                                            strict_reference=True)
    assert np.array_equal(h_lo, want) and np.array_equal(h_hi, want)


@pytest.mark.parametrize("prec,nfft,dt", [("f32", 1024, "cf32_le"), ("f32", 65536, "cu8"), ("f64", 512, "cf64_le")])
def test_eof_only_requests(engine, prec, nfft, dt):
    bps = BPS[dt.split("_")[0]]
    d_iq = torch.zeros(nfft * bps, dtype=torch.uint8, device=DEV)
    frames = 50
    for fill in (-150.0, -37.25, 99.0):
        got = run_persistence(engine, d_iq, nfft * bps, dt, nfft, nfft, "hann", frames, 1, 37, -100.0, 0.0, prec,
                              eof_fill_db=fill)
        want = np.zeros((37, nfft), np.uint32)
        want[pr.quantize(np.array([fill]), 37, -100.0, 0.0, prec == "f64")[0]] = frames
        assert np.array_equal(got, want), fill


def test_reruns_are_byte_identical(engine):
    nfft, hop = 1024, 512
    frames = (1 << 17) + 5
    n = (frames - 1) * hop + nfft
    d_iq = gain_noise("cf32_le", n, nfft, hop, seed=3)
    a = run_persistence(engine, d_iq, n * 8, "cf32_le", nfft, hop, "hann", frames, 0, 256, -40.0, 60.0)
    b = run_persistence(engine, d_iq, n * 8, "cf32_le", nfft, hop, "hann", frames, 0, 256, -40.0, 60.0)
    assert np.array_equal(a, b) and np.all(a.sum(axis=0) == frames)


def test_canvas_fields_are_ignored(engine):
    """out_kind, colormap, sample_rate, min_db and max_db of the params do not take part: canvas params that the
    canvas would refuse (sample_rate 0, max_db <= min_db) or an unknown out_kind count as their F32 rows do."""
    nfft, hop, frames = 512, 256, 301
    n = (frames - 2) * hop + nfft
    d_iq = gain_noise("ci16_le", n, nfft, hop, seed=11)
    ref = run_persistence(engine, d_iq, n * 4, "ci16_le", nfft, hop, "hann", frames, 0, 37, -20.0, 60.0)
    for kw in ({"out": "rgba8", "sample_rate": 0.0, "min_db": 5.0, "max_db": -5.0}, {"out": "f64"}):
        got = run_persistence(engine, d_iq, n * 4, "ci16_le", nfft, hop, "hann", frames, 0, 37, -20.0, 60.0, **kw)
        assert np.array_equal(got, ref), kw
    p = engine.make_params("ci16_le", nfft, hop, "hann", n_frames=frames)
    p.out_kind = 99
    host = np.empty((37, nfft), np.uint32)
    raw = d_iq.cpu().numpy()
    _capi.check(_capi.lib().sa_spectrum_persistence(engine.handle, raw.ctypes.data, raw.size, C.byref(p), 37, -20.0,
                                                    60.0, host.ctypes.data, host.nbytes))
    assert np.array_equal(host, ref)


# ---------------- (g) argument errors ----------------

def test_argument_errors(engine):
    L = _capi.lib()
    raw = np.zeros(1 << 16, np.uint8)
    d_iq = torch.zeros(1 << 16, dtype=torch.uint8, device=DEV)
    out = torch.empty(1 << 18, dtype=torch.uint8, device=DEV)
    h_out = np.empty(1 << 18, np.uint8)

    def both(p, levels, lo, hi, nb, outs=True, d_ptr=None):
        rd = L.sa_spectrum_persistence_device(engine.handle, d_ptr or d_iq.data_ptr(), 1 << 16, C.byref(p), levels, lo,
                                              hi, out.data_ptr() if outs else None, nb, None)
        rh = L.sa_spectrum_persistence(engine.handle, raw.ctypes.data, raw.size, C.byref(p), levels, lo, hi,
                                       h_out.ctypes.data if outs else None, nb)
        return rd, rh

    p = engine.make_params("cf32_le", 256, 256, "hann", n_frames=10)
    big = 1 << 18
    assert both(p, 37, -100.0, 0.0, big) == (0, 0)
    for levels in (0, 1, 257):
        assert both(p, levels, -100.0, 0.0, big) == (1, 1), levels               # n_levels outside 2..256
    for lo, hi in ((0.0, 0.0), (1.0, -1.0), (float("nan"), 0.0), (-100.0, float("inf")), (float("-inf"), 0.0)):
        assert both(p, 37, lo, hi, big) == (1, 1), (lo, hi)                     # not finite, or max_db <= min_db
    assert both(p, 37, -100.0, 0.0, big, outs=False) == (1, 1)                  # NULL output
    assert both(engine.make_params("cf32_le", 256, 256, "hann", n_frames=0), 37, -100.0, 0.0, big) == (1, 1)
    assert both(engine.make_params("cf32_le", 256, 1, "hann", n_frames=1 << 32), 37, -100.0, 0.0, big) == (1, 1)
    assert both(engine.make_params("cf32_le", 250, 256, "hann", n_frames=10), 37, -100.0, 0.0, big) == (1, 1)
    assert both(p, 37, -100.0, 0.0, 37 * 256 * 4 - 1) == (7, 7)                   # SMALL_OUTPUT
    assert both(p, 37, -100.0, 0.0, 37 * 256 * 4) == (0, 0)
    rd = L.sa_spectrum_persistence_device(engine.handle, d_iq.data_ptr() + 4, 1 << 15, C.byref(p), 37, -100.0, 0.0,
                                          out.data_ptr(), big, None)
    assert rd == 1                                                               # d_iq not aligned to one IQ pair
    torch.cuda.synchronize()


# ---------------- (h) C++ binding ----------------

def test_cpp_binding(tmp_path):
    exe = str(tmp_path / "test_persistence")
    lib_dir = os.path.join(ROOT, "spectral_analyzer_b200")
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "test_persistence.cpp"), "-o", exe,
                    "-L", lib_dir, "-lsa_engine", "-Wl,-rpath," + lib_dir], check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    assert "cpp persistence ok" in out
