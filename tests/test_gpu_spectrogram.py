"""GPU parity tests: the CUDA path, called through the C-ABI, against the CPU oracle."""
import glob
import os

import numpy as np
import pytest

from oracle import c_oracle as co
from spectral_analyzer_b200 import synth, SpectralService, EngineError
from util import check_db_parity

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
ALL_DT = ["cf32_le", "cf32_be", "ci16_le", "ci16_be", "cu8", "ci8"]


def test_impulse_and_dc_kat(engine):
    n = 1024
    x = np.zeros(n, complex); x[0] = 1.0
    out = engine.spectrogram(synth.encode(x, "cf32_le"), "cf32_le", n, 1)
    assert np.abs(out - 20 * np.log10(1 + 1e-10)).max() < 1e-5
    out = engine.spectrogram(synth.encode(np.full(n, 0.25), "cf32_le"), "cf32_le", n, 1)[0]
    assert abs(out[n // 2] - 20 * np.log10(0.25 * n)) < 1e-4
    assert (np.delete(out, n // 2) < -100).all()


@pytest.mark.parametrize("dt", ALL_DT)
def test_integer_decode_bit_exact(engine, dt):
    """A length-64 frame holding ONE non-zero sample at n=0 has |X[k]| = |x[0]| in every bin, so the
    decoded value is read back exactly: 20*log10(|v| + 1e-10) must match the FP64 oracle to FP32
    rounding of the dB value -- and, decoded through the FP64 path, to 1e-12."""
    kind = dt.split("_")[0]
    vals = {"ci16": [-32768, -1, 1, 32767, 12345], "cu8": [0, 127, 128, 255, 37], "ci8": [-128, -1, 1, 127, 37],
            "cf32": [1.0, -0.5, 3.0e-5, 12345.678, -1e-3]}[kind]
    for v in vals:
        iq = np.zeros(128, synth.NP_DTYPE[kind])
        if kind == "cu8":
            iq[:] = 0            # cu8 zero level is -127.5/128, so every sample is non-zero: use oracle directly
        iq[0] = v
        raw = iq.astype(("<" if dt.endswith("_le") else ">") + synth.NP_DTYPE[kind]).view(np.uint8)
        ref = co.compute_magnitudes(raw, 0, 64, dt)
        got64 = engine.spectrogram(raw, dt, 64, 1, precision="f64", out_kind="f64")[0]
        assert np.abs(got64 - ref).max() < 1e-9, (dt, v)
        got32 = engine.spectrogram(raw, dt, 64, 1)[0]
        lin = np.abs(10 ** (got32 / 20.0) - 10 ** (ref / 20.0))
        assert lin.max() <= 2e-6 * 10 ** (ref.max() / 20.0), (dt, v)


@pytest.mark.parametrize("nfft", [64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536])
def test_reference_parity_mode_all_sizes(engine, nfft):
    """rect window, hop = nfft, 20*log10(|X|+1e-10): the reference's own framing (SURVEY F3)."""
    frames = 9
    raw = synth.recording(nfft * frames - 17, "cf32_le", seed=nfft)
    ref = co.spectrogram(raw, "cf32_le", 0, nfft, nfft, "rect", frames)
    got = engine.spectrogram(raw, "cf32_le", nfft, frames)
    assert (got[-1] == -150.0).all()                      # EOF row, MainController.java:994-998
    check_db_parity(got[:-1], ref[:-1])


@pytest.mark.parametrize("dt", ALL_DT)
@pytest.mark.parametrize("nfft,win,hop", [(1024, "hann", 512), (4096, "blackman_harris", 4096), (2048, "rect", 2048),
                                          (256, "hamming", 64), (512, "blackman", 300)])
def test_dtypes_windows_hops(engine, dt, nfft, win, hop):
    frames = 13
    raw = synth.recording((frames - 1) * hop + nfft + 5, dt, seed=3)
    ref = co.spectrogram(raw, dt, 5, nfft, hop, win, frames)
    got = engine.spectrogram(raw, dt, nfft, frames, hop=hop, window=win, start_sample=5)
    check_db_parity(got, ref)


@pytest.mark.parametrize("dt", ["cf64_le", "cf64_be", "cf32_le", "ci16_le", "cu8"])
@pytest.mark.parametrize("nfft", [64, 512, 1024, 8192, 16384, 32768, 65536])
def test_fp64_path_tight(engine, dt, nfft):
    frames = 5
    raw = synth.recording(nfft * frames, dt, seed=5)
    for win, hop in (("rect", nfft), ("hann", nfft // 2)):
        ref = co.spectrogram(raw, dt, 0, nfft, hop, win, frames)
        got = engine.spectrogram(raw, dt, nfft, frames, hop=hop, window=win, precision="f64", out_kind="f64")
        check_db_parity(got, ref, strong_tol=1e-9, floor_tol=1e-6)


def test_power_db_mode(engine):
    raw = synth.recording(1024 * 8, "cf32_le", seed=7)
    ref = co.spectrogram(raw, "cf32_le", 0, 1024, 512, "hann", 15, db_mode=co.DB_POWER)
    got = engine.spectrogram(raw, "cf32_le", 1024, 15, hop=512, window="hann", db_mode=1)
    check_db_parity(got, ref, mode_power=True)


def test_golden_fixtures(engine):
    for f in sorted(glob.glob(os.path.join(GOLD, "spec_parity_*.npz"))):
        g = np.load(f)
        dt, nfft, frames = str(g["datatype"]), int(g["nfft"]), int(g["frames"])
        got = engine.spectrogram(g["raw"], dt, nfft, frames)
        assert (got[-1] == -150.0).all()
        check_db_parity(got[:-1], g["img"][:-1])
    g = np.load(os.path.join(GOLD, "spec_c1_mini.npz"))
    got = engine.spectrogram(g["raw"], "cf32_le", 1024, 9, hop=512, window="hann")
    check_db_parity(got, g["img"])


def test_compute_magnitudes_service(engine):
    """The per-frame entry point kept for API compatibility (SpectralService.java:33)."""
    svc = SpectralService(engine)
    raw = synth.recording(5000, "ci16_le", seed=8)
    out = svc.computeMagnitudes(raw, 4 * 123, 1024, "ci16_le")
    assert out.dtype == np.float64 and out.shape == (1024,)
    check_db_parity(out[None], co.compute_magnitudes(raw, 4 * 123, 1024, "ci16_le")[None])
    # odd byte offsets are legal in Java (absolute get on the ByteBuffer)
    out = svc.computeMagnitudes(raw, 3, 256, "ci16_le")
    check_db_parity(out[None], co.compute_magnitudes(raw, 3, 256, "ci16_le")[None])
    with pytest.raises(EngineError) as ei:
        svc.computeMagnitudes(raw, 0, 1000, "ci16_le")       # MathIllegalArgumentException
    assert ei.value.code == 1
    with pytest.raises(EngineError) as ei:
        svc.computeMagnitudes(raw, 4 * 4500, 1024, "ci16_le")  # IndexOutOfBoundsException
    assert ei.value.code == 3
    wf = svc.computeWaterfall(raw, 100, 6, 1024, "ci16_le")
    ref = co.spectrogram(raw, "ci16_le", 100, 1024, 1024, "rect", 6)
    assert (wf[4:] == -150.0).all() and wf.dtype == np.float64
    check_db_parity(wf[:4], ref[:4])


def test_empty_and_ragged(engine):
    raw = synth.recording(100, "cf32_le")
    out = engine.spectrogram(raw, "cf32_le", 256, 3)            # shorter than one frame: all EOF rows
    assert (out == -150.0).all()
    out = engine.spectrogram(raw, "cf32_le", 64, 0)
    assert out.shape == (0, 64)
    out = engine.spectrogram(np.zeros(0, np.uint8), "cf32_le", 64, 2)
    assert (out == -150.0).all()


def test_chunked_host_pipeline_matches_single_chunk(engine, monkeypatch):
    """Frame indexing across chunk boundaries of the H2D/D2H pipeline is exact."""
    import spectral_analyzer_b200 as sa
    raw = synth.recording(1 << 18, "ci16_le", seed=12)
    frames = ((1 << 18) - 1024) // 384 + 3
    a = engine.spectrogram(raw, "ci16_le", 1024, frames, hop=384, window="hann")
    monkeypatch.setenv("SA_CHUNK_MB", "1")
    small = sa.Engine(0)
    small_chunks = small.spectrogram(raw, "ci16_le", 1024, frames, hop=384, window="hann")
    small.close()
    assert np.array_equal(a, small_chunks)
    assert (a[-1] == -150.0).all() and (a[-3] != -150.0).any()


def test_linearity_and_time_shift_properties(engine):
    """Size-independent properties at a larger size than the oracle is asked to handle."""
    n, nfft = 1 << 22, 1024
    x = synth.complex_signal(n, seed=21)
    a = engine.spectrogram(synth.encode(x, "cf32_le"), "cf32_le", nfft, n // nfft)
    b = engine.spectrogram(synth.encode(2.0 * x, "cf32_le"), "cf32_le", nfft, n // nfft)
    strong = a > a.max() - 60
    assert np.abs((b - a)[strong] - 20 * np.log10(2.0)).max() < 1e-4          # homogeneity in dB
    # starting one frame later reproduces rows shifted by one
    c = engine.spectrogram(synth.encode(x, "cf32_le"), "cf32_le", nfft, n // nfft - 1, start_sample=nfft)
    assert np.array_equal(c, a[1:])
    # Parseval on a few frames: sum |X|^2 = N * sum |x|^2
    p = (10 ** (a[:8].astype(np.float64) / 10)).sum(axis=1)
    e = (np.abs(x[:8 * nfft].astype(np.complex64)) ** 2).reshape(8, nfft).sum(axis=1) * nfft
    assert np.abs(p / e - 1).max() < 1e-4


def test_both_1024_kernels_against_oracle(engine):
    """The 1024-point FP32 plan has two kernels: TMA-staged frames (16-byte aligned frame starts) and
    the LDG kernel (any alignment).  Both are checked against the oracle.  The host pipeline copies the
    capture from the first frame on, so an odd start sample alone still gives aligned frames; an odd
    hop does not."""
    raw = synth.recording(1024 * 40, "cf32_le", seed=31)
    ref = co.spectrogram(raw, "cf32_le", 0, 1024, 512, "hann", 70)
    got = engine.spectrogram(raw, "cf32_le", 1024, 70, hop=512, window="hann")
    assert engine.last_kernel == "spectrogram_tma_kernel<float,1024,cf32,window>"
    check_db_parity(got, ref)
    ref_odd = co.spectrogram(raw, "cf32_le", 3, 1024, 512, "hann", 70)
    got_odd = engine.spectrogram(raw, "cf32_le", 1024, 70, hop=512, window="hann", start_sample=3)
    check_db_parity(got_odd, ref_odd)
    ref_ldg = co.spectrogram(raw, "cf32_le", 3, 1024, 513, "hann", 70)
    got_ldg = engine.spectrogram(raw, "cf32_le", 1024, 70, hop=513, window="hann", start_sample=3)
    assert engine.last_kernel == "spectrogram_kernel<float,1024,cf32,window>"
    check_db_parity(got_ldg, ref_ldg)


@pytest.mark.parametrize("cmap", ["Grayscale", "Heatmap"])
@pytest.mark.parametrize("dt,nfft", [("cu8", 2048), ("cf32_le", 1024)])
def test_rgba_epilogue_matches_render(engine, cmap, dt, nfft):
    """SA_OUT_RGBA8 = renderSpectrogram's dB/Hz conversion + getColorForMagnitude
    (MainController.java:1273-1285, :926-957), one pixel per (frame, bin).  Channels may differ by one
    LSB (FP32 dB vs FP64 dB); pixels whose normalised level sits on a Heatmap breakpoint (0.2 / 0.5, where
    the ramp jumps from black to blue) are excluded."""
    frames, fs = 24, 2.4e6
    raw = synth.recording(nfft * frames, dt, seed=17)
    db = co.spectrogram(raw, dt, 0, nfft, nfft, "rect", frames)
    # choose a colour range that spans the image so that all ramp segments are exercised
    conv = 10 * np.log10(fs / nfft) + 20 * np.log10(nfft)
    lo, hi = float(np.percentile(db - conv, 5)), float(db.max() - conv + 3.0)
    ref = co.render_rgba(db, fs, lo, hi, cmap).astype(np.int32)
    got = engine.spectrogram(raw, dt, nfft, frames, out_kind="rgba8", colormap=cmap, sample_rate=fs,
                             min_db=lo, max_db=hi).astype(np.int32)
    assert got.shape == (frames, nfft, 4) and (got[..., 3] == 255).all()
    n = np.clip((db - conv - lo) / (hi - lo), 0, 1)
    safe = np.ones_like(n, bool)
    if cmap == "Heatmap":
        safe = (np.abs(n - 0.2) > 1e-4) & (np.abs(n - 0.5) > 1e-4)
    assert np.abs(got - ref)[safe].max() <= 1
    assert (np.abs(got - ref)[safe] > 0).mean() < 0.05
    assert len(np.unique(ref[..., 0])) > 50 or cmap == "Heatmap"
    # default range of the reference UI (-160 .. -30 dB/Hz)
    got2 = engine.spectrogram(raw, dt, nfft, frames, out_kind="rgba8", colormap=cmap, sample_rate=fs)
    ref2 = co.render_rgba(db, fs, -160.0, -30.0, cmap).astype(np.int32)
    n2 = np.clip((db - conv + 160.0) / 130.0, 0, 1)
    safe2 = (np.abs(n2 - 0.2) > 1e-4) & (np.abs(n2 - 0.5) > 1e-4)
    assert np.abs(got2.astype(np.int32) - ref2)[safe2].max() <= 1


@pytest.mark.parametrize("dt", ["cf32_le", "ci16_be", "cu8"])
@pytest.mark.parametrize("nfft,win,hop", [(32768, "hann", 16384), (65536, "blackman_harris", 65536), (65536, "hann", 5000)])
def test_large_four_step_fp32(engine, dt, nfft, win, hop):
    """nfft above one SM's shared memory: four-step kernels (large_fft_kernels.cuh)."""
    frames = 5
    raw = synth.recording((frames - 2) * hop + nfft + 11, dt, seed=41)       # the last frame runs past EOF
    ref = co.spectrogram(raw, dt, 7, nfft, hop, win, frames)
    got = engine.spectrogram(raw, dt, nfft, frames, hop=hop, window=win, start_sample=7)
    assert (ref[-1] == -150.0).all() and (got[-1] == -150.0).all()
    check_db_parity(got[:-1], ref[:-1])


def test_config5_cf64_65536_hann(engine):
    """BASELINE config 5 in miniature: cf64 recording, 65536-point Hann FFT on the FP64 path."""
    nfft, frames = 65536, 3
    raw = synth.recording(nfft * frames, "cf64_le", seed=5)
    ref = co.spectrogram(raw, "cf64_le", 0, nfft, nfft, "hann", frames)
    got = engine.spectrogram(raw, "cf64_le", nfft, frames, window="hann", out_kind="f64")
    assert got.dtype == np.float64
    check_db_parity(got, ref, strong_tol=1e-9, floor_tol=1e-6)
    # 16-bit stereo WAV: 44-byte header, ci16_le (NonconformingDatasetHelper.java:137-156); the mapped buffer
    # starts after the header (SigMfHelper.java:84), i.e. only 4-byte aligned in the file
    body = synth.recording(1024 * 9, "ci16_le", seed=6)
    wav = np.concatenate([np.zeros(44, np.uint8), body])
    got = engine.spectrogram(wav[44:], "ci16_le", 1024, 9)
    check_db_parity(got, co.spectrogram(body, "ci16_le", 0, 1024, 1024, "rect", 9))


def test_pinned_and_pageable_host_paths_agree(engine, tmp_path):
    """Pinned / registered buffers are DMA'd directly; pageable ones (numpy arrays, an mmapped .sigmf-data file --
    cudaHostRegister refuses file-backed mappings) go through the engine's pinned staging ring."""
    import torch
    n, nfft, hop = 1 << 21, 1024, 512
    raw = synth.recording(n, "ci16_le", seed=44)
    frames = (n - nfft) // hop + 3                                   # two EOF rows
    a = engine.spectrogram(raw, "ci16_le", nfft, frames, hop=hop, window="hann")            # pageable in / out
    pin = torch.empty(raw.size, dtype=torch.uint8, pin_memory=True)
    pin.numpy()[:] = raw
    out = torch.empty((frames, nfft), dtype=torch.float32, pin_memory=True)
    b = engine.spectrogram(pin.numpy(), "ci16_le", nfft, frames, hop=hop, window="hann", out=out.numpy())
    assert np.array_equal(a, b)
    path = tmp_path / "rec.sigmf-data"
    path.write_bytes(raw.tobytes())
    mm = np.memmap(path, dtype=np.uint8, mode="r")
    c = engine.spectrogram(mm, "ci16_le", nfft, frames, hop=hop, window="hann")
    assert np.array_equal(a, c)
    with pytest.raises(EngineError):
        engine.register_host(mm, read_only=True)                    # file-backed: cannot be page-locked
    engine.register_host(raw, read_only=False)                      # anonymous memory can
    d = engine.spectrogram(raw, "ci16_le", nfft, frames, hop=hop, window="hann")
    engine.unregister_host(raw)
    assert np.array_equal(a, d)
    # annotation batch from the mapped file (staged spans)
    iq_m, psd_m = engine.downconvert_psd_batch(mm, "ci16_le", 1e6, [(1000, 600000, 0.1, 16, False), (5, 40000, -0.2, 4, True)], psd_nfft=1024)
    iq_p, psd_p = engine.downconvert_psd_batch(pin.numpy(), "ci16_le", 1e6, [(1000, 600000, 0.1, 16, False), (5, 40000, -0.2, 4, True)], psd_nfft=1024)
    assert all(np.array_equal(x, y) for x, y in zip(iq_m, iq_p)) and np.array_equal(psd_m, psd_p)


@pytest.mark.parametrize("nfft,dt,prec", [(32768, "ci16_le", "f32"), (65536, "cf32_le", "f32"), (16384, "cf64_le", "f64")])
def test_four_step_through_the_chunked_host_pipeline(monkeypatch, nfft, dt, prec):
    """Several host chunks of a four-step size are in flight on different streams: every slot has its own
    workspace (a shared one would be overwritten by the next chunk's column step)."""
    import spectral_analyzer_b200 as sa
    frames, hop = 41, nfft // 2
    raw = synth.recording((frames - 1) * hop + nfft, dt, seed=77)
    ref = co.spectrogram(raw, dt, 0, nfft, hop, "hann", frames)
    monkeypatch.setenv("SA_CHUNK_MB", "1")
    eng = sa.Engine(0)
    kind = "f64" if prec == "f64" else "f32"
    for _ in range(3):          # repeated: a workspace race would be timing dependent
        got = eng.spectrogram(raw, dt, nfft, frames, hop=hop, window="hann", precision=prec, out_kind=kind)
        if prec == "f64":
            check_db_parity(got, ref, strong_tol=1e-9, floor_tol=1e-6)
        else:
            check_db_parity(got, ref)
    eng.close()


def test_index_overflow_is_rejected_not_wrapped(engine):
    """Frame indexing is 64-bit (MainController.java:984 extended): requests whose sample or output offsets would
    wrap are refused with INVALID_ARG before anything is launched."""
    raw = synth.recording(4096, "cf32_le", seed=1)
    out = np.empty((1, 1024), np.float32)
    for kw in (dict(n_frames=1 << 40, hop=1 << 30), dict(n_frames=2, hop=1 << 62), dict(n_frames=1, start_sample=1 << 63),
               dict(n_frames=1 << 60, hop=1)):
        with pytest.raises(EngineError) as ei:
            engine.spectrogram(raw, "cf32_le", 1024, kw.pop("n_frames"), out=out, **kw)
        assert ei.value.code == 1
    # large but representable offsets past EOF give fill rows
    got = engine.spectrogram(raw, "cf32_le", 1024, 2, hop=1024, start_sample=1 << 40)
    assert (got == -150.0).all()


@pytest.mark.parametrize("nfft", [256, 1024, 16384])
@pytest.mark.parametrize("mode", [0, 1])
def test_fp64_db_epilogue_over_the_dynamic_range(engine, nfft, mode):
    """The FP64 dB epilogue switches between a table-driven log (|X|^2 >= 1e-10) and the literal
    20 log10(sqrt(p) + 1e-10) per thread: frames of white noise scaled from 1e-13 to 1e100 cover both sides of the
    threshold, exact zeros and the 1e-10 floor.  White noise keeps every bin within ~25 dB of the frame's maximum,
    so ALL bins are held to the FP64 tolerance of 1e-9 dB."""
    amps = [0.0, 1e-13, 1e-9, 3e-8, 1e-7, 3e-7, 1e-6, 1e-5, 1e-3, 1.0, 7.0, 1e6, 1e30, 1e100]
    rng = np.random.default_rng(nfft + mode)
    x = rng.standard_normal((len(amps), nfft, 2)) * np.asarray(amps)[:, None, None]
    raw = np.ascontiguousarray(x.reshape(-1), np.float64).view(np.uint8)
    ref = co.spectrogram(raw, "cf64_le", 0, nfft, nfft, "rect", len(amps), db_mode=mode)
    got = engine.spectrogram(raw, "cf64_le", nfft, len(amps), hop=nfft, window="rect", out_kind="f64", db_mode=mode)
    assert np.isfinite(got).all()
    assert np.abs(got - ref).max() < 1e-9, np.abs(got - ref).max(axis=1)
    # exact zeros: 20 log10(1e-10) = 10 log10(1e-20) = -200 (literal form in magnitude mode, the table log in power mode)
    assert (got[0] == -200.0).all() if mode == 0 else np.abs(got[0] + 200.0).max() < 1e-11


@pytest.mark.parametrize("dt,header", [("cf32_le", 0), ("ci16_le", 44), ("cu8", 320)])
def test_spectrogram_file_matches_buffer_call(engine, tmp_path, dt, header):
    """sa_spectrogram_file (SigMfHelper.java:59-84: data file, core:header_bytes skipped) reads the capture into the
    pinned ring itself; rows must equal the buffer call on the same bytes, EOF rows included, and a capture limited by
    data_bytes ends where it says."""
    nfft, hop, frames = 1024, 512, 700
    raw = synth.recording((frames - 1) * hop + nfft - 100, dt, seed=11)
    path = tmp_path / "rec.sigmf-data"
    with open(path, "wb") as f:
        f.write(b"\x7f" * header)
        f.write(raw.tobytes())
    ref = engine.spectrogram(raw, dt, nfft, frames, hop=hop, window="hann")
    got = engine.spectrogram_file(str(path), dt, nfft, frames, hop=hop, window="hann", data_offset=header)
    assert (ref[-1] == -150.0).all() and np.array_equal(got, ref)
    half = (raw.size // 2) & ~15
    ref_h = engine.spectrogram(raw[:half], dt, nfft, frames, hop=hop, window="hann")
    got_h = engine.spectrogram_file(str(path), dt, nfft, frames, hop=hop, window="hann", data_offset=header, data_bytes=half)
    assert np.array_equal(got_h, ref_h) and (got_h[-1] == -150.0).all()
    with pytest.raises(EngineError) as e:
        engine.spectrogram_file(str(tmp_path / "missing"), dt, nfft, 1)
    assert e.value.code == 1


def test_spectrogram_file_large_chunks(engine, tmp_path):
    """several pipeline chunks and the parallel pread path (> 4 MiB per chunk)"""
    nfft = 4096
    raw = synth.recording(1 << 22, "ci16_le", seed=12)              # 16 MiB
    path = tmp_path / "rec.sigmf-data"
    raw.tofile(path)
    frames = (1 << 22) // nfft
    import os
    os.environ["SA_CHUNK_MB"] = "4"
    import spectral_analyzer_b200 as sa
    eng = sa.Engine(0)
    del os.environ["SA_CHUNK_MB"]
    try:
        got = eng.spectrogram_file(str(path), "ci16_le", nfft, frames, window="blackman_harris")
        ref = eng.spectrogram(raw, "ci16_le", nfft, frames, window="blackman_harris")
        assert np.array_equal(got, ref)
        assert eng.last_kernel.startswith("spectrogram_r64_kernel<float,4096,ci16")
    finally:
        eng.close()


def test_last_kernel_name_reports_the_selected_variant(engine):
    raw = synth.recording(1024 * 8, "cf32_le", seed=1)
    engine.spectrogram(raw, "cf32_le", 1024, 8, hop=512, window="hann")
    assert engine.last_kernel == "spectrogram_tma_kernel<float,1024,cf32,window>"
    engine.spectrogram(raw, "cf32_le", 1024, 7, hop=513, window="hann")      # odd hop: frames only 8-byte aligned
    assert engine.last_kernel == "spectrogram_kernel<float,1024,cf32,window>"


@pytest.mark.parametrize("dt,prec,kind", [("cf64_le", "f64", "f64"), ("cf64_be", "f64", "f64"), ("cf32_le", "f32", "f32"), ("cf32_be", "f32", "f32")])
def test_four_step_65536_against_oracle(engine, dt, prec, kind):
    """65536 points take the four-step path (large_cols_kernel + large_rows_kernel).  50 % overlap, two trailing EOF
    frames; against the oracle on a sample of frames, then a rect window (FP32 path: no window multiply instantiated)
    and an odd hop (frames only 8-byte aligned)."""
    nfft, hop, frames = 65536, 32768, 61
    raw = synth.recording((frames - 3) * hop + nfft, dt, seed=65)
    got = engine.spectrogram(raw, dt, nfft, frames, hop=hop, window="hann", precision=prec, out_kind=kind)
    assert engine.last_kernel == "large_cols_kernel+large_rows_kernel<%s,256x256,%s,window>" % ("double" if prec == "f64" else "float", dt[:4])
    assert (got[-2:] == -150.0).all()
    pick = [0, 1, 17, 40, frames - 3]
    for f in pick:
        ref = co.spectrogram(raw, dt, f * hop, nfft, hop, "hann", 1)
        if prec == "f64":
            check_db_parity(got[f:f + 1], ref, strong_tol=1e-9, floor_tol=1e-6)
        else:
            check_db_parity(got[f:f + 1], ref)
    if prec == "f32":
        g2 = engine.spectrogram(raw, dt, nfft, 5, precision=prec, out_kind=kind)
        assert engine.last_kernel == "large_cols_kernel+large_rows_kernel<float,256x256,cf32,rect>"
        check_db_parity(g2[:1], co.spectrogram(raw, dt, 0, nfft, nfft, "rect", 1))
        g3 = engine.spectrogram(raw, dt, nfft, 3, hop=nfft + 1, precision=prec, out_kind=kind)
        assert engine.last_kernel == "large_cols_kernel+large_rows_kernel<float,256x256,cf32,rect>"
        check_db_parity(g3[1:2], co.spectrogram(raw, dt, nfft + 1, nfft, nfft, "rect", 1))


@pytest.mark.parametrize("dt", ["cf32_le", "cf32_be", "ci16_le", "ci16_be", "cu8", "ci8"])
@pytest.mark.parametrize("win,hop", [("hann", 1024), ("rect", 2048)])
def test_2048_kernels_against_oracle(engine, dt, win, hop):
    """nfft 2048: the staged small-radix-first kernel on 16-byte aligned frames, the LDG kernel otherwise.  More frames
    than one pass of the grid, two trailing EOF rows; against the oracle, and through the FP64-row epilogue."""
    nfft, frames = 2048, 1500
    raw = synth.recording((frames - 3) * hop + nfft, dt, seed=77)
    got = engine.spectrogram(raw, dt, nfft, frames, hop=hop, window=win)
    assert engine.last_kernel.startswith("spectrogram_mid_kernel(prefetch)<float,2048,")
    assert (got[-2:] == -150.0).all()
    for f in (0, 1, 777, frames - 3):
        check_db_parity(got[f:f + 1], co.spectrogram(raw, dt, f * hop, nfft, hop, win, 1))
    g64 = engine.spectrogram(raw, dt, nfft, 40, hop=hop, window=win, out_kind="f64")
    assert np.array_equal(g64, got[:40].astype(np.float64))
    odd = engine.spectrogram(raw, dt, nfft, 5, hop=hop + 1, window=win)                    # frames not 16-byte aligned
    assert engine.last_kernel.startswith("spectrogram_kernel<float,2048,")
    check_db_parity(odd[:1], co.spectrogram(raw, dt, 0, nfft, hop + 1, win, 1))
