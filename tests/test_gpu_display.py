"""GPU parity tests of the rows next to the hot path (SURVEY.md 8f): display canvas (N2), IqData packers and
analysis series (N3), against the oracle restatements of MainController.renderSpectrogram (:1261-1291),
IqData.getInterleavedBinary (IqData.java:160-187) and AnalysisDialogController (:219-290)."""
import os

import numpy as np
import pytest

from oracle import c_oracle as co
from spectral_analyzer_b200 import synth, IqData, EngineError

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def pixel_check(got, ref, n, cmap, max_frac=0.05):
    """channels within one LSB (FP32 dB vs FP64 dB); pixels on a Heatmap breakpoint excluded."""
    got, ref = got.astype(np.int32), ref.astype(np.int32)
    safe = np.ones(n.shape, bool)
    if cmap == "Heatmap":
        safe = (np.abs(n - 0.2) > 1e-4) & (np.abs(n - 0.5) > 1e-4)
    d = np.abs(got - ref)[safe]
    assert d.max() <= 1
    assert (d > 0).mean() < max_frac


@pytest.mark.parametrize("cmap", ["Grayscale", "Heatmap"])
@pytest.mark.parametrize("dt,nfft,W,H", [("cf32_le", 1024, 37, 300), ("ci16_le", 256, 50, 256), ("cu8", 2048, 21, 2500),
                                         ("cf32_le", 64, 19, 100)])
def test_canvas_matches_render_spectrogram(engine, cmap, dt, nfft, W, H):
    """frames_per_column = 1, nearest bin: exactly renderSpectrogram (also H > nfft: rows repeat bins)."""
    fs = 2.4e6
    raw = synth.recording(nfft * (W - 1) + nfft // 2, dt, seed=23)          # the last column runs past EOF (-150 dB row)
    db = co.spectrogram(raw, dt, 0, nfft, nfft, "rect", W)
    conv = 10 * np.log10(fs / nfft) + 20 * np.log10(nfft)
    lo, hi = float(np.percentile(db - conv, 5)), float(db.max() - conv + 3.0)
    ref = co.render_canvas(db, H, fs, lo, hi, cmap)
    got = engine.render_canvas(raw, dt, nfft, W, H, fs, colormap=cmap, min_db=lo, max_db=hi)
    assert got.shape == (H, W, 4) and (got[..., 3] == 255).all()
    bins = (np.arange(H, dtype=np.float64) / H * nfft).astype(np.int64)
    n = np.clip((db[:, bins].T[::-1] - conv - lo) / (hi - lo), 0, 1)             # [H, W], y flipped
    pixel_check(got, ref, n[..., None].repeat(4, -1), cmap)


@pytest.mark.parametrize("reduce", ["max", "mean"])
def test_canvas_pooling_whole_recording(engine, reduce):
    """several frames and bins per pixel, in one host chunk (test_gpu_kernel_matrix.py covers canvases of several
    64 MiB chunks and pooled launches past one wave)."""
    fs, nfft, hop, fpc, W, H = 1.0e6, 512, 256, 5, 41, 96
    raw = synth.recording((W * fpc - 1) * hop + nfft, "ci16_le", seed=29)
    db = co.spectrogram(raw, "ci16_le", 0, nfft, hop, "hann", W * fpc)
    edges = ((np.arange(H + 1, dtype=np.float64)) / H * nfft).astype(np.int64)
    blk = db.reshape(W, fpc, nfft)
    pooled = np.empty((W, H))
    for f in range(H):
        seg = blk[:, :, edges[f]:max(edges[f + 1], edges[f] + 1)]
        pooled[:, f] = seg.max(axis=(1, 2)) if reduce == "max" else 10 * np.log10((10 ** (seg / 10)).mean(axis=(1, 2)))
    conv = 10 * np.log10(fs / nfft) + 20 * np.log10(nfft)
    lo, hi = float(np.percentile(pooled - conv, 5)), float(pooled.max() - conv + 3.0)
    ref = co.render_rgba(pooled.T[::-1].copy() , fs, lo, hi, "Heatmap")          # render of the pooled image
    # render_rgba subtracts conversion for ITS nfft argument (= W here): compensate through min/max instead
    conv_w = 10 * np.log10(fs / W) + 20 * np.log10(W)
    ref = co.render_rgba(pooled.T[::-1].copy(), fs, lo + conv - conv_w, hi + conv - conv_w, "Heatmap")
    got = engine.render_canvas(raw, "ci16_le", nfft, W, H, fs, hop=hop, window="hann", frames_per_column=fpc,
                               reduce=reduce, colormap="Heatmap", min_db=lo, max_db=hi)
    n = np.clip((pooled.T[::-1] - conv - lo) / (hi - lo), 0, 1)
    pixel_check(got, ref, n[..., None].repeat(4, -1), "Heatmap", max_frac=0.08)


_STRICT_ROWS_PATH = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import spectral_analyzer_b200 as sa
e = sa.Engine(0)
raw = np.load(sys.argv[2])
out = {}
for dt, bps in (("cf64_le", 16), ("ri16_le", 8)):
    data = raw[:(9 * 3 - 1) * 1024 * bps + 1024 * bps]
    for reduce in ("max", "mean"):
        out[dt + reduce] = e.render_canvas(data, dt, 1024, 12, 64, 1.0e6, frames_per_column=3, reduce=reduce,
                                           strict_reference=True, min_db=float(sys.argv[4]), max_db=float(sys.argv[5]))
np.savez(sys.argv[3], **out)
"""


def test_strict_reference_pooled_canvas(engine, tmp_path):
    """strict_reference with a datatype the reference cannot decode (cf64, SA_DT_OTHER): every readable frame is
    -200 dB and the pooled MAX / MEAN canvas shows just that, past EOF the -150 dB fill, on the host and the device
    path, identical to the canvas of dB rows (SA_CANVAS_FUSED=0, read once per process: a subprocess)."""
    import subprocess
    import sys
    import ctypes as C
    import torch
    from spectral_analyzer_b200 import _capi
    fs, nfft, W, H, fpc = 1.0e6, 1024, 12, 64, 3
    conv = 10 * np.log10(fs / nfft) + 20 * np.log10(nfft)
    lo, hi = float(-200.0 - conv - 10.0), float(-150.0 - conv + 10.0)
    colour = {v: co.render_rgba(np.full((1, nfft), v), fs, lo, hi, "Grayscale")[0, 0] for v in (-200.0, -150.0)}
    assert not np.array_equal(colour[-200.0], colour[-150.0])
    wr = 9                                                   # the frames of columns 9..11 lie past EOF
    raw = np.random.default_rng(3).integers(0, 256, (wr * fpc - 1) * nfft * 16 + nfft * 16, dtype=np.uint8)
    got = {}
    for dt in ("cf64_le", "ri16_le"):
        bps = 16 if dt == "cf64_le" else 8                   # ri16_le: Global.getBytesPerSample's fallback
        data = raw[:(wr * fpc - 1) * nfft * bps + nfft * bps]
        for reduce in ("max", "mean"):
            g = engine.render_canvas(data, dt, nfft, W, H, fs, frames_per_column=fpc, reduce=reduce,
                                     strict_reference=True, min_db=lo, max_db=hi)
            assert (g[:, :wr] == colour[-200.0]).all() and (g[:, wr:] == colour[-150.0]).all(), (dt, reduce)
            got[dt + reduce] = g
            d_iq = torch.from_numpy(data).cuda()
            d_out = torch.empty(W * H * 4, dtype=torch.uint8, device="cuda")
            p = engine.make_params(dt, nfft, None, "rect", 0, 0, sample_rate=fs, min_db=lo, max_db=hi,
                                   strict_reference=True)
            _capi.check(_capi.lib().sa_render_canvas_device(engine.handle, d_iq.data_ptr(), data.size, C.byref(p), W, H,
                                                            fpc, _capi.REDUCE[reduce], d_out.data_ptr(),
                                                            torch.cuda.current_stream().cuda_stream))
            torch.cuda.synchronize()
            assert np.array_equal(d_out.view(H, W, 4).cpu().numpy(), g), (dt, reduce)
    np.save(tmp_path / "raw.npy", raw)
    script = tmp_path / "rows_path.py"
    script.write_text(_STRICT_ROWS_PATH)
    env = dict(os.environ, SA_CANVAS_FUSED="0")
    subprocess.run([sys.executable, str(script), os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    str(tmp_path / "raw.npy"), str(tmp_path / "rows.npz"), repr(lo), repr(hi)], check=True, env=env)
    rows = np.load(tmp_path / "rows.npz")
    for dt in ("cf64_le", "ri16_le"):
        for reduce in ("max", "mean"):
            assert np.array_equal(rows[dt + reduce], got[dt + reduce]), (dt, reduce)


def test_canvas_argument_errors(engine):
    raw = synth.recording(4096, "cf32_le", seed=1)
    with pytest.raises(EngineError) as ei:
        engine.render_canvas(raw, "cf32_le", 1000, 4, 4, 1e6)            # not a power of two
    assert ei.value.code == 1
    with pytest.raises(EngineError):
        engine.render_canvas(raw, "cf32_le", 1024, 0, 4, 1e6)


def test_iq_pack_bit_exact(engine):
    g = np.load(os.path.join(GOLD, "iqdata_mini.npz"))
    edge = g["edge"]
    assert engine.iq_pack(edge, "float32") == g["edge_f32"].tobytes() == co.iq_pack(edge, "float32")
    assert engine.iq_pack(edge, "int16") == g["edge_i16"].tobytes() == co.iq_pack(edge, "int16")
    a = np.load(os.path.join(GOLD, "analysis_mini.npz"))
    assert engine.iq_pack(a["dc"], "INT16") == g["dc_i16"].tobytes()
    rng = np.random.default_rng(8)
    big = rng.normal(size=(2, 300_001)) * 0.8
    assert engine.iq_pack(big, "float32") == co.iq_pack(big, "float32")
    assert engine.iq_pack(big, "int16") == co.iq_pack(big, "int16")
    d = IqData(big, engine).getDataBuffer()
    assert d["IQ_BUFFER_INT16"] == co.iq_pack(big, "int16") and len(d["IQ_BUFFER_FLOAT32"]) == 8 * 300_001
    with pytest.raises(ValueError):
        engine.iq_pack(big, "int8")                                     # IllegalArgumentException, IqData.java:185


@pytest.mark.parametrize("n", [1, 2, 255, 256, 257, 70_001])
@pytest.mark.parametrize("am,af", [(1.0, 1.0), (0.2, 0.05), (0.01, 0.9)])
def test_analysis_series_matches_oracle(engine, n, am, af):
    rng = np.random.default_rng(n)
    t = np.arange(n)
    z = (0.3 + 0.1 * rng.normal(size=n)) * np.exp(2j * np.pi * (0.07 * t + 0.002 * rng.normal(size=n).cumsum()))
    iq = np.stack([z.real, z.imag])
    rm, rf = co.analysis_series(iq, 250e3, am, af, 915e6)
    gm, gf = engine.analysis_series(iq, 250e3, am, af, 915e6)
    assert np.abs(gm - rm).max() < 1e-9                                  # dB
    assert np.isnan(gf[0])                                               # also for n == 1: the Java loop starts at i = 1
    if n > 1:
        assert np.abs(gf[1:] - rf[1:]).max() < 1e-6 * 250e3 * 1e-3       # Hz (values ~ 9e8)


def test_analysis_series_golden_and_silence(engine):
    g = np.load(os.path.join(GOLD, "iqdata_mini.npz"))
    a = np.load(os.path.join(GOLD, "analysis_mini.npz"))
    gm, gf = engine.analysis_series(a["dc"], 250e3, 0.2, 0.05, 915e6)
    assert np.abs(gm - g["mag"]).max() < 1e-9 and np.abs(gf[1:] - g["frq"][1:]).max() < 1e-3
    zm, _ = engine.analysis_series(np.zeros((2, 100)), 1e6, 0.5, 0.5, 0.0)
    assert np.isneginf(zm).all()                                         # 20 log10(0): the values the Java chart skips


@pytest.mark.parametrize("dt,nfft", [("cf32_le", 1024), ("cu8", 2048)])
def test_canvas_nearest_with_frame_stride_and_sparse_frames(engine, dt, nfft):
    """frames_per_column > 1 with the nearest pick shows frame t*fpc of every column: only those frames are
    transformed and (host path) only their samples are packed and sent.  Also a sparse max-pooled view, and
    columns past the end of the recording (-150 dB rows)."""
    fs, W, H, fpc = 2.4e6, 23, 160, 7
    n = nfft * (fpc * (W - 3)) + 5                                        # the last columns run past EOF
    raw = synth.recording(n, dt, seed=61)
    db = co.spectrogram(raw, dt, 0, nfft, nfft, "rect", W * fpc)
    ref = co.render_canvas(db[::fpc], H, fs, -140.0, -20.0, "Grayscale")
    got = engine.render_canvas(raw, dt, nfft, W, H, fs, frames_per_column=fpc, reduce="nearest", colormap="Grayscale",
                               min_db=-140.0, max_db=-20.0)
    assert np.abs(got.astype(np.int32) - ref.astype(np.int32)).max() <= 1
    assert (got[:, -1, :3] == got[0, -1, :3]).all()                        # EOF column: one colour (-150 dB)
    # sparse hop (3 nfft) with max pooling over 2 frames per column
    hop, fpc2, W2 = 3 * nfft, 2, 11
    raw2 = synth.recording((W2 * fpc2 - 1) * hop + nfft, dt, seed=62)
    db2 = co.spectrogram(raw2, dt, 0, nfft, hop, "hann", W2 * fpc2).reshape(W2, fpc2, nfft)
    edges = (np.arange(H + 1, dtype=np.float64) / H * nfft).astype(np.int64)
    pooled = np.stack([db2[:, :, edges[f]:max(edges[f + 1], edges[f] + 1)].max(axis=(1, 2)) for f in range(H)], axis=1)
    conv = 10 * np.log10(fs / nfft) + 20 * np.log10(nfft)
    n_lvl = np.clip((pooled.T[::-1] - conv + 140.0) / 120.0, 0, 1)
    ref2 = np.floor(n_lvl * 255 + 0.5).astype(np.int32)
    got2 = engine.render_canvas(raw2, dt, nfft, W2, H, fs, hop=hop, window="hann", frames_per_column=fpc2, reduce="max",
                                colormap="Grayscale", min_db=-140.0, max_db=-20.0)
    assert np.abs(got2[..., 0].astype(np.int32) - ref2).max() <= 1
