"""Small invocation of every kernel family, for compute-sanitizer (memcheck / racecheck) runs:
    compute-sanitizer --tool memcheck python tests/sanitize_smoke.py
Sizes are tiny (the tools slow kernels down 10-100x); results are still compared with the CPU checker, which is why
this script lives under tests/: only tests, smoke() and the bench's CPU-baseline leg may use oracle/."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import spectral_analyzer_b200 as sa                      # noqa: E402
from spectral_analyzer_b200 import synth                 # noqa: E402
from oracle import c_oracle as co                        # noqa: E402

only = sys.argv[1] if len(sys.argv) > 1 else ""
eng = sa.Engine(0)
n_checked = 0
for nfft in (64, 256, 1024, 2048, 4096, 16384, 65536):
    for dt, win, hop in (("cf32_le", "hann", nfft // 2), ("ci16_le", "rect", nfft), ("cu8", "hann", nfft // 2 + 1)):
        if only and only not in ("spec%d" % nfft):
            continue
        frames = 5
        raw = synth.recording((frames - 2) * hop + nfft + 9, dt, seed=nfft)            # last frame(s) past EOF
        got = eng.spectrogram(raw, dt, nfft, frames, hop=hop, window=win, start_sample=0)
        ref = co.spectrogram(raw, dt, 0, nfft, hop, win, frames)
        strong = ref > ref.max(axis=1, keepdims=True) - 40
        assert np.abs(got - ref)[strong].max() < 1e-3, (nfft, dt)
        n_checked += 1
if not only or only == "f64":
    raw = synth.recording(16384 * 3, "cf64_le", seed=2)
    for nfft in (1024, 16384):
        got = eng.spectrogram(raw, "cf64_le", nfft, 3, window="hann", out_kind="f64")
        ref = co.spectrogram(raw, "cf64_le", 0, nfft, nfft, "hann", 3)
        assert np.abs(got - ref).max() < 1e-6
        n_checked += 1
if not only or only == "analysis":
    raw = synth.recording(40000, "ci16_le", seed=3)
    for down, fast in ((16, False), (5, False), (2, False), (16, True), (600, False)):      # 2: several blocks per thread and tile
        got = eng.downconvert(raw, "ci16_le", 100, 36000, 0.125, down, fast)
        ref = co.downconvert(raw, "ci16_le", 100, 36000, 0.125, down, fast)
        assert np.abs(got - ref).max() / np.abs(ref).max() < 1e-5, (down, fast)
        n_checked += 1
    iq = co.downconvert(raw, "ci16_le", 100, 36000, 0.125, 4, False)
    psd = eng.psd_welch(iq, 250e3, 2048)
    ref = co.psd_welch(iq, 250e3, 2048)
    top = ref[1] > ref[1].max() - 60
    assert np.abs(psd[1] - ref[1])[top].max() < 2e-3
    assert eng.iq_pack(iq, "int16") == co.iq_pack(iq, "int16")
    gm, gf = eng.analysis_series(iq, 250e3, 0.2, 0.05, 1e6)
    rm, rf = co.analysis_series(iq, 250e3, 0.2, 0.05, 1e6)
    assert np.abs(gm - rm).max() < 1e-9 and np.abs(gf[1:] - rf[1:]).max() < 1e-3
    n_checked += 3
if not only or only == "canvas":
    raw = synth.recording(1024 * 40, "cf32_le", seed=5)
    for red in ("nearest", "max", "mean"):
        px = eng.render_canvas(raw, "cf32_le", 1024, 13, 200, 2.4e6, frames_per_column=3, reduce=red, colormap="Heatmap")
        assert px.shape == (200, 13, 4) and (px[..., 3] == 255).all()
        n_checked += 1
if not only or only == "profile":
    # round 2: any-length PSD (direct DFT kernel, FP32 and FP64), FP64 Welch, caller taps / delay / length rules, PSD-only
    # batch, strict decodes, file ingest
    import tempfile
    raw = synth.recording(30000, "ci16_le", seed=8)
    iq = co.downconvert(raw, "ci16_le", 0, 28000, 0.1, 4, False)
    for prec, tol in (("f32", 1e-3), ("f64", 1e-8)):
        eng.set_analysis_config(psd_precision=prec, psd_detrend="constant", psd_scaling="spectrum")
        cfg = co.analysis_cfg(scaling="spectrum", detrend="constant")
        for nf in (777, 1024):
            got = eng.psd_welch(iq, 250e3, nf)
            ref = co.psd_welch(iq, 250e3, nf, cfg=cfg)
            top = ref[1] > ref[1].max() - 40
            assert np.abs(got[1] - ref[1])[top].max() < tol, (prec, nf)
            n_checked += 1
    taps = np.hanning(41) / np.hanning(41).sum()
    eng.set_analysis_config(taps=taps, delay="same", length="ceil")
    got = eng.downconvert(raw, "ci16_le", 7, 20001, -0.2, 8)
    ref = co.downconvert_ex(raw, "ci16_le", 7, 20001, -0.2, 8, False, co.analysis_cfg(taps=taps, delay="same", length="ceil"))
    assert got.shape == ref.shape and np.abs(got - ref).max() < 1e-5
    eng.reset_analysis_config()
    raw32 = synth.recording(8000, "cf32_le", seed=9)            # cf32 at decimation 16 / 8: the row-per-thread kernel, both parities
    for start, down in ((0, 16), (77, 16), (1, 8), (1200, 32)):
        got = eng.downconvert(raw32, "cf32_le", start, 6000, 0.11, down)
        ref = co.downconvert(raw32, "cf32_le", start, 6000, 0.11, down, False)
        assert got.shape == ref.shape and np.abs(got - ref).max() <= 1e-5 * max(np.abs(ref).max(), 0.5)
    eng.set_analysis_config(strict_reference=True)            # an unknown datatype is read as cf32 (strict reference)
    got = eng.downconvert(raw32, "ri16_le", 0, 7000, 0.05, 4)
    ref = co.downconvert_ex(raw32, "ri16_le", 0, 7000, 0.05, 4, False, co.analysis_cfg(strict_reference=True))
    assert np.abs(got - ref).max() <= 1e-5 * max(np.abs(ref).max(), 0.5)
    eng.reset_analysis_config()
    _, psd = eng.downconvert_psd_batch(raw, "ci16_le", 1e6, [(0, 20000, 0.1, 4, False), (100, 900, 0.2, 4, False)], psd_nfft=1024, want_iq=False)
    assert np.isfinite(psd[0]).all() and np.isnan(psd[1][225:]).all()
    with tempfile.NamedTemporaryFile(suffix=".sigmf-data") as f:
        f.write(b"\0" * 44 + raw.tobytes())
        f.flush()
        a = eng.spectrogram_file(f.name, "ci16_le", 1024, 20, hop=512, window="hann", data_offset=44)
    assert np.array_equal(a, eng.spectrogram(raw, "ci16_le", 1024, 20, hop=512, window="hann"))
    n_checked += 4
eng.close()
print("sanitize smoke ok: %d checks" % n_checked)
