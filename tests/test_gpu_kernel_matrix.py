"""Every default spectrogram kernel against the FP64 oracle past its first wave, on non-repeating full-band input.

The spectrogram kernels are persistent: the grid is capped at resident CTAs x SMs and each CTA walks frame blocks
with a grid stride; the cp.async-staged mid kernel stages each slot's NEXT frame; the four-step path splits long
requests into workspace chunks addressed through a frame offset.  All of that runs only when a launch has more
frames than one wave (or one chunk), and only white noise makes a wrong frame, a wrong bin or a wrong column
visible in every bin.  So:

  (a) each default in-SM kernel (family x nfft x decode kind x rect/window, aligned and unaligned; FP64 for four
      decode kinds x eight sizes) on 2 W + r frames, W = SMs x (threads per SM / threads per frame) an upper bound
      of the frames one wave holds, every frame checked; the last two frames are EOF rows;
  (b) the power-dB, FP64-row and RGBA epilogues of each family on the same frame counts;
  (c) the four-step kernels over several 512 MiB workspace chunks (sampled frames: both ends of every chunk);
  (d) input offsets past 2^31 and 2^32 bytes of one device buffer, one kernel of each family;
  (e) fused canvas pooling (max / mean) past one wave on the device path and over several host chunks.

Each case asserts the kernel the default dispatch picks (engine.cu launch_spectrogram) against expected_kernel's
table, so that a change of dispatch fails here instead of silently testing another kernel.

Comparator: util.frame_norm_error, E = max_k |A_got - A_ref| / rms_k(A_ref) per frame.  Worst E over this module,
measured on one NVIDIA B200 (power limit 1000 W, max SM clock 1965 MHz), against the bounds util.NORM_TOL_F32 = 1e-5
and util.NORM_TOL_F64 = 1e-12:
  FP32 path  spectrogram_kernel        3.85e-6
             spectrogram_tma_kernel    3.32e-6
             spectrogram_mid_kernel    4.89e-6   (with and without prefetch)
             spectrogram_r64_kernel    4.71e-6
             four-step                 3.38e-6
  FP64 path  spectrogram_kernel        3.12e-13
             four-step                 2.41e-13
The whole module takes about 80 s on that machine.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from spectral_analyzer_b200 import _capi
from util import NORM_TOL_F32, NORM_TOL_F64, frame_norm_error

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BPS = {"cf32": 8, "ci16": 4, "cu8": 2, "ci8": 2, "cf64": 16}
VARIANTS = {"cf32": ("cf32_le", "cf32_be"), "ci16": ("ci16_le", "ci16_be"), "c8": ("cu8", "ci8"),
            "cf64": ("cf64_le", "cf64_be")}
WINDOWS = ["hann", "hamming", "blackman", "blackman_harris"]
# points per thread of the plans (fft_core.cuh Plan<T, N>::P); the mid kernel uses 32, the radix-64 kernel 64
P_F32 = {64: 8, 128: 16, 256: 16, 512: 32, 1024: 32, 2048: 32, 4096: 32, 8192: 32, 16384: 32}
P_F64 = {64: 8, 128: 16, 256: 16, 512: 16, 1024: 16, 2048: 16, 4096: 16, 8192: 16}
SLAB = 1 << 22                       # points per host comparison slab
WORST = {}                           # family -> worst E seen by this module


def dk_name(datatype):
    k = datatype.split("_")[0]
    return "c8" if k in ("cu8", "ci8") else k


def expected_kernel(prec, nfft, datatype, window, aligned, pooled=False):
    """The default dispatch (engine.cu launch_spectrogram / launch_spectrogram_large, spec_inst.cu, large_inst.cu).
    Four-step names carry the n1 x n2 split: only the prefix and the suffix are fixed here."""
    dk = dk_name(datatype)
    if prec == "f64":
        if nfft > 8192:
            return ("large_cols_kernel+large_rows_kernel<double,", ",%s,window>" % dk)
        return ("spectrogram_kernel<double,%d,%s,window>" % (nfft, dk), "")
    w = "rect" if window == "rect" else "window"
    if nfft > 16384:
        return ("large_cols_kernel+large_rows_kernel<float,", ",%s,%s>" % (dk, w))
    if not aligned or nfft <= 512:
        fam = "spectrogram_kernel"
    elif nfft == 1024:
        fam = "spectrogram_tma_kernel"
    elif nfft == 4096 and dk in ("cf32", "ci16") and not pooled:
        fam = "spectrogram_r64_kernel"
    elif nfft == 8192:
        fam = "spectrogram_mid_kernel"
    else:
        fam = "spectrogram_mid_kernel(prefetch)"
    return ("%s<float,%d,%s,%s>" % (fam, nfft, dk, w), "")


def assert_kernel(engine, want):
    name = engine.last_kernel
    pre, suf = want
    if suf:
        assert name.startswith(pre) and name.endswith(suf), (name, want)
    else:
        assert name == pre, (name, want)
    return name


def family(name):
    if name.startswith("large_cols"):
        return ("FP64 " if "<double" in name else "FP32 ") + "four-step"
    return ("FP64 " if "<double" in name else "FP32 ") + name.split("<")[0].replace("(prefetch)", "")


def note_worst(name, e):
    fam = family(name)
    WORST[fam] = max(WORST.get(fam, 0.0), float(e))


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    yield
    print("\nworst frame_norm_error per kernel family:")
    for k in sorted(WORST):
        print("  %-34s %.3e" % (k, WORST[k]))


@pytest.fixture(scope="module")
def device_props():
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, p.max_threads_per_multi_processor


def wave_frames(props, nfft, points_per_thread):
    sms, threads = props
    return sms * (threads // (nfft // points_per_thread))


def device_noise(datatype, n_samples, seed, out=None):
    """White noise of n_samples IQ pairs on the device, seeded: uniformly random bytes for the integer types (every
    byte pattern is a sample), randn for the float types; big-endian variants byte-swapped on the device."""
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    kind = datatype.split("_")[0]
    if kind in ("cf32", "cf64"):
        x = torch.randn(2 * n_samples, dtype=torch.float32 if kind == "cf32" else torch.float64, device=DEV, generator=g)
        x = x.view(torch.uint8)
    else:
        x = torch.randint(0, 256, (n_samples * BPS[kind],), dtype=torch.uint8, device=DEV, generator=g)
    if kind in ("cf32", "ci16", "cf64") and not datatype.endswith("_le"):
        elem = {"cf32": 4, "ci16": 2, "cf64": 8}[kind]
        x = x.view(-1, elem).flip(1).reshape(-1)
    if out is not None:
        out.copy_(x)
        return out
    return x.contiguous()


def run_device(engine, d_iq, iq_bytes, datatype, nfft, hop, window, frames, start, out="f32", **kw):
    obytes = {"f32": 4, "f64": 8, "rgba8": 4}[out]
    d_out = torch.empty(frames * nfft * obytes, dtype=torch.uint8, device=DEV)
    p = engine.make_params(datatype, nfft, hop, window, n_frames=frames, start_sample=start, out=out, **kw)
    engine.spectrogram_device(d_iq.data_ptr(), iq_bytes, p, d_out.data_ptr(), d_out.numel(),
                              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    if out == "rgba8":
        return d_out.view(frames, nfft, 4)
    return d_out.view(torch.float32 if out == "f32" else torch.float64).view(frames, nfft)


def readable(start, hop, nfft, n_samples, idx):
    return start + np.asarray(idx, np.int64) * hop + nfft <= n_samples          # MainController.java:987


def check_rows(got, ref, ok, tol):
    """got / ref: dB rows of the same frames; ok: readable mask.  Returns the worst E of the readable rows."""
    assert (got[~ok] == -150.0).all() and (ref[~ok] == -150.0).all()
    if not ok.any():
        return 0.0
    g = got[ok]
    assert np.isfinite(g).all()
    e = frame_norm_error(g, ref[ok])
    worst = float(e.max())
    assert worst <= tol, "worst E %.3g > %.3g at frame row %d" % (worst, tol, int(np.flatnonzero(ok)[e.argmax()]))
    return worst


def check_all_frames(got_dev, host_raw, datatype, start, nfft, hop, window, frames, tol, db_mode=0):
    n_samples = host_raw.size // BPS[datatype.split("_")[0]]
    step = max(1, SLAB // nfft)
    worst = 0.0
    for f0 in range(0, frames, step):
        f1 = min(frames, f0 + step)
        got = got_dev[f0:f1].cpu().numpy()
        ref = co.spectrogram(host_raw, datatype, start + f0 * hop, nfft, hop, window, f1 - f0, db_mode=db_mode)
        worst = max(worst, check_rows(got, ref, readable(start, hop, nfft, n_samples, np.arange(f0, f1)), tol))
    return worst


# ---------------- (a) every default in-SM kernel ----------------

def insm_cases():
    out = []
    sizes = [64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384]
    for k, nfft in enumerate(sizes):
        for d, dk in enumerate(("cf32", "ci16", "c8")):
            for iw in (0, 1):
                for aligned in (True, False):
                    i = len(out)
                    dt = VARIANTS[dk][(k + iw + int(aligned)) % 2]
                    win = WINDOWS[(k + d) % 4] if iw else "rect"
                    gapped = nfft + nfft // 8
                    if aligned:
                        hop = [nfft, nfft // 2, gapped][(k + d + iw) % 3]
                        if nfft == 4096 and dk != "c8":
                            hop = nfft // 2                  # radix-64 kernel: 32 frames per SM, keep ~20 M samples
                        start = [0, 16, 64][(k + d) % 3]
                    elif (k + d + iw) % 2:
                        hop, start = [nfft, nfft // 2, gapped][(k + d + iw) % 3], 3     # odd start
                    else:
                        hop, start = [nfft - 1, nfft // 2 + 1, gapped + 1][(k + d + iw) % 3], 0   # odd hop
                    out.append(("f32", nfft, dt, win, hop, start, aligned, 3 + 2 * (i % 3)))
    for k, nfft in enumerate([64, 128, 256, 512, 1024, 2048, 4096, 8192]):
        for d, dk in enumerate(("cf64", "cf32", "ci16", "c8")):
            i = len(out)
            dt = VARIANTS[dk][(k + d) % 2]
            win = (["rect"] + WINDOWS)[(k + d) % 5]
            hop = [nfft, nfft // 2, nfft + nfft // 8 + (k % 2)][(k + d) % 3]
            out.append(("f64", nfft, dt, win, hop, [0, 5][(k + d) % 2], True, 3 + 2 * (i % 3)))
    return out


def case_id(c):
    prec, nfft, dt, win, hop, start, aligned, r = c
    return "%s-%d-%s-%s-hop%d-start%d-%s" % (prec, nfft, dt, win, hop, start, "al" if aligned else "unal")


def insm_frames(props, prec, nfft, dt, aligned, r):
    if prec == "f64":
        p = P_F64[nfft]
    elif aligned and nfft == 4096 and dk_name(dt) != "c8":
        p = 64
    else:
        p = P_F32[nfft]
    return 2 * wave_frames(props, nfft, p) + r


@pytest.mark.parametrize("prec,nfft,dt,win,hop,start,aligned,r", insm_cases(), ids=[case_id(c) for c in insm_cases()])
def test_insm_kernel_past_first_wave(engine, device_props, prec, nfft, dt, win, hop, start, aligned, r):
    frames = insm_frames(device_props, prec, nfft, dt, aligned, r)
    n = start + (frames - 3) * hop + nfft + hop // 3               # the last two frames are EOF rows
    d_iq = device_noise(dt, n, seed=nfft * 1000 + hop + start + len(dt))
    out = "f64" if prec == "f64" else "f32"
    got = run_device(engine, d_iq, d_iq.numel(), dt, nfft, hop, win, frames, start, out=out,
                     precision="f64" if prec == "f64" else "auto")
    if prec == "f32":
        assert (start * BPS[dt.split("_")[0]] % 16 == 0 and hop * BPS[dt.split("_")[0]] % 16 == 0) == aligned
    name = assert_kernel(engine, expected_kernel(prec, nfft, dt, win, aligned))
    host = d_iq.cpu().numpy()
    worst = check_all_frames(got, host, dt, start, nfft, hop, win, frames, NORM_TOL_F64 if prec == "f64" else NORM_TOL_F32)
    note_worst(name, worst)


# ---------------- (b) epilogues ----------------

EPI_CASES = [(256, "ci16_le", "hann", 256, 0, True), (1024, "cu8", "blackman", 512, 0, True),
             (2048, "cf32_le", "rect", 2048, 0, True), (4096, "ci16_be", "hann", 2048, 0, True),
             (8192, "ci8", "hamming", 9216, 0, True), (16384, "cf32_be", "blackman_harris", 8192, 0, True),
             (2048, "cu8", "hann", 1025, 0, False)]


@pytest.mark.parametrize("nfft,dt,win,hop,start,aligned", EPI_CASES, ids=["%d-%s-%s" % c[:3] for c in EPI_CASES])
def test_epilogues_past_first_wave(engine, device_props, nfft, dt, win, hop, start, aligned):
    """power dB with FP64 rows, then RGBA (Heatmap), each over 2 W + 1 frames."""
    frames = insm_frames(device_props, "f32", nfft, dt, aligned, 1)
    n = start + (frames - 3) * hop + nfft + 1
    d_iq = device_noise(dt, n, seed=nfft + 17)
    host = d_iq.cpu().numpy()
    got = run_device(engine, d_iq, d_iq.numel(), dt, nfft, hop, win, frames, start, out="f64", db_mode=_capi.DB_POWER)
    name = assert_kernel(engine, expected_kernel("f32", nfft, dt, win, aligned))
    note_worst(name, check_all_frames(got, host, dt, start, nfft, hop, win, frames, NORM_TOL_F32, db_mode=co.DB_POWER))
    del got
    ref = co.spectrogram(host, dt, start, nfft, hop, win, frames)
    ok = readable(start, hop, nfft, n, np.arange(frames))
    fs = 2.4e6
    conv = 10 * np.log10(fs / nfft) + 20 * np.log10(nfft)
    lo, hi = float(ref[ok].min() - conv - 0.5), float(ref[ok].max() - conv + 0.5)       # brackets the image
    rgba = run_device(engine, d_iq, d_iq.numel(), dt, nfft, hop, win, frames, start, out="rgba8", colormap="Heatmap",
                      sample_rate=fs, min_db=lo, max_db=hi)
    assert_kernel(engine, expected_kernel("f32", nfft, dt, win, aligned))
    step = max(1, SLAB // nfft)
    diffs = 0
    for f0 in range(0, frames, step):
        f1 = min(frames, f0 + step)
        g = rgba[f0:f1].cpu().numpy().astype(np.int32)
        r = co.render_rgba(ref[f0:f1], fs, lo, hi, "Heatmap").astype(np.int32)
        lvl = np.clip((ref[f0:f1] - conv - lo) / (hi - lo), 0, 1)[..., None]
        safe = np.broadcast_to((np.abs(lvl - 0.2) > 1e-4) & (np.abs(lvl - 0.5) > 1e-4), g.shape)
        d = np.abs(g - r)[safe]
        assert d.max() <= 1, "frames %d..%d: %d LSB" % (f0, f1, d.max())
        diffs += int((d > 0).sum())
    assert diffs < 0.05 * frames * nfft * 4


# ---------------- (c) four-step chunk boundaries ----------------

def sampled_frames(frames, chunk, n_read, seed):
    idx = set()
    for c0 in range(0, frames, chunk):
        c1 = min(frames, c0 + chunk)
        idx.update([c0, c0 + 1, c1 - 2, c1 - 1])
    idx.update(np.random.default_rng(seed).integers(0, frames, 32).tolist())
    idx.update([n_read - 1, frames - 2, frames - 1])
    return np.array(sorted(i for i in idx if 0 <= i < frames), np.int64)


def check_sampled(d_iq, got_dev, dt, start, nfft, hop, win, n_samples, idx, tol):
    """Oracle check of the frames idx from host copies of only their bytes."""
    bps = BPS[dt.split("_")[0]]
    got = got_dev[torch.from_numpy(idx).to(DEV)].cpu().numpy()
    ok = readable(start, hop, nfft, n_samples, idx)
    ref = np.full(got.shape, -150.0)
    for j in np.flatnonzero(ok):
        s = (start + int(idx[j]) * hop) * bps
        ref[j] = co.spectrogram(d_iq[s:s + nfft * bps].cpu().numpy(), dt, 0, nfft, nfft, win, 1)[0]
    return check_rows(got, ref, ok, tol)


FOUR_STEP = [("f32", 32768, "cu8", "hann", 32768, 0, 2048 + 41),
             ("f32", 65536, "cu8", "blackman_harris", 32768, 0, 2 * 1024 + 23),
             ("f64", 16384, "ci16_le", "hann", 16385, 7, 2048 + 37),
             ("f64", 65536, "ci16_be", "rect", 65536, 0, 2 * 512 + 19)]


@pytest.mark.parametrize("prec,nfft,dt,win,hop,start,frames", FOUR_STEP, ids=["%s-%d-%s" % c[:3] for c in FOUR_STEP])
def test_four_step_chunk_boundaries(engine, prec, nfft, dt, win, hop, start, frames):
    """The default four-step path splits a request into 512 MiB workspace chunks (engine.cu launch_spectrogram_large):
    frames of every chunk, both ends of each, against the oracle."""
    chunk = (512 << 20) // (nfft * (16 if prec == "f64" else 8))
    assert frames > chunk
    n = start + (frames - 3) * hop + nfft + hop // 2
    n_read = (n - start - nfft) // hop + 1
    d_iq = device_noise(dt, n, seed=nfft + frames)
    out = "f64" if prec == "f64" else "f32"
    got = run_device(engine, d_iq, d_iq.numel(), dt, nfft, hop, win, frames, start, out=out, precision=prec)
    name = assert_kernel(engine, expected_kernel(prec, nfft, dt, win, True))
    idx = sampled_frames(frames, chunk, n_read, seed=nfft)
    tol = NORM_TOL_F64 if prec == "f64" else NORM_TOL_F32
    note_worst(name, check_sampled(d_iq, got, dt, start, nfft, hop, win, n, idx, tol))


# ---------------- (d) 64-bit input offsets ----------------

@pytest.fixture(scope="module")
def big_buffer():
    buf = torch.empty((1 << 32) + (1 << 28), dtype=torch.uint8, device=DEV)
    yield buf
    del buf
    torch.cuda.empty_cache()


OFFSET_CASES = [(1024, "cf32_le", "hann", 512), (2048, "cu8", "rect", 2048), (4096, "ci16_le", "blackman", 2048),
                (65536, "cf32_le", "hann", 65536)]


@pytest.mark.parametrize("byte0", [(1 << 31) + (3 << 20), (1 << 32) + (5 << 20)], ids=["past2^31", "past2^32"])
@pytest.mark.parametrize("nfft,dt,win,hop", OFFSET_CASES, ids=["%d-%s" % c[:2] for c in OFFSET_CASES])
def test_input_offsets_past_32_bits(engine, big_buffer, nfft, dt, win, hop, byte0):
    """start_sample points past 2^31 / 2^32 bytes into one device buffer; only the span the request reads holds
    (non-repeating) data."""
    bps = BPS[dt.split("_")[0]]
    frames = 300 if nfft <= 4096 else 120
    start = byte0 // bps
    span = (frames - 3) * hop + nfft + 7
    device_noise(dt, span, seed=nfft + byte0 % 1000, out=big_buffer[byte0:byte0 + span * bps])
    n = start + span
    torch.cuda.synchronize()
    got = run_device(engine, big_buffer, n * bps, dt, nfft, hop, win, frames, start)
    name = assert_kernel(engine, expected_kernel("f32", nfft, dt, win, True))
    idx = sampled_frames(frames, frames, frames - 2, seed=byte0 % 977)
    note_worst(name, check_sampled(big_buffer, got, dt, start, nfft, hop, win, n, idx, NORM_TOL_F32))


# ---------------- (e) fused canvas pooling ----------------

def gain_noise(datatype, n, hop, seed):
    """noise whose level changes by a seeded random gain (+-20 dB) every hop samples: a column's statistics depend on
    exactly which frames it pools"""
    x = device_noise(datatype, n, seed)
    kind = datatype.split("_")[0]
    g = torch.Generator(device=DEV)
    g.manual_seed(seed + 1)
    ft = torch.float32 if kind == "cf32" else torch.float64
    lvl = torch.rand((n + hop - 1) // hop, dtype=ft, device=DEV, generator=g) * 40 - 20
    gain = torch.pow(10.0, lvl / 20).repeat_interleave(hop)[:n]
    z = x.view(ft).view(n, 2)
    z *= gain[:, None]
    return x


def pool_reference(db, W, fpc, H, reduce):
    edges = (np.arange(H + 1, dtype=np.float64) / H * db.shape[1]).astype(np.int64)
    blk = db.reshape(W, fpc, db.shape[1])
    pooled = np.empty((W, H))
    for f in range(H):
        seg = blk[:, :, edges[f]:max(edges[f + 1], edges[f] + 1)]
        pooled[:, f] = seg.max(axis=(1, 2)) if reduce == "max" else 10 * np.log10((10 ** (seg / 10)).mean(axis=(1, 2)))
    return pooled


def check_canvas(got, pooled, nfft, fs, lo, hi, cmap):
    W = pooled.shape[0]
    conv = 10 * np.log10(fs / nfft) + 20 * np.log10(nfft)
    conv_w = 10 * np.log10(fs / W) + 20 * np.log10(W)     # render_rgba subtracts the conversion of ITS row length (W)
    img = pooled.T[::-1].copy()
    ref = co.render_rgba(img, fs, lo + conv - conv_w, hi + conv - conv_w, cmap).astype(np.int32)
    lvl = np.clip((img - conv - lo) / (hi - lo), 0, 1)[..., None]
    safe = np.ones(got.shape, bool)
    if cmap == "Heatmap":
        safe = np.broadcast_to((np.abs(lvl - 0.2) > 1e-4) & (np.abs(lvl - 0.5) > 1e-4), got.shape)
    d = np.abs(got.astype(np.int32) - ref)[safe]
    assert d.max() <= 1, "%d LSB" % d.max()
    assert (d > 0).mean() < 0.05


POOL_CASES = [(256, "cf32_le", "hann"), (1024, "cf32_le", "hann"), (2048, "cf32_le", "blackman"),
              (4096, "cf32_le", "hann"), (8192, "cf32_le", "rect"), (16384, "cf32_le", "hamming"),
              (1024, "cf64_le", "hann")]


@pytest.mark.parametrize("nfft,dt,win", POOL_CASES, ids=["%d-%s" % c[:2] for c in POOL_CASES])
def test_fused_canvas_pooling(engine, device_props, nfft, dt, win):
    """MAX / MEAN canvases: device path (one pooled launch over every frame) and host path (several 64 MiB chunks
    rotating through the three pipeline slots); trailing columns partly and wholly past EOF."""
    prec = "f64" if dt.startswith("cf64") else "f32"
    fs, fpc, H = 1.0e6, 5, 128
    hop = nfft + nfft // 2
    points = (12 << 20) if prec == "f64" else (24 << 20)
    W = points // (nfft * fpc)
    frames = W * fpc
    assert W <= 65535 and frames > wave_frames(device_props, nfft, (P_F64 if prec == "f64" else P_F32)[nfft])
    n_read = frames - 2 * fpc - 2                                    # one partial and two whole EOF columns
    n = (n_read - 1) * hop + nfft
    bps = BPS[dt.split("_")[0]]
    col_bytes = max(fpc * nfft * 4, fpc * hop * bps)
    assert W / ((64 << 20) // col_bytes) > 3                         # host path: more chunks than slots
    d_iq = gain_noise(dt, n, hop, seed=nfft + 3)
    host = d_iq.cpu().numpy()
    db = co.spectrogram(host, dt, 0, nfft, hop, win, frames)
    want = expected_kernel(prec, nfft, dt, win, True, pooled=True)
    for reduce, cmap in (("max", "Heatmap"), ("mean", "Grayscale")):
        pooled = pool_reference(db, W, fpc, H, reduce)
        conv = 10 * np.log10(fs / nfft) + 20 * np.log10(nfft)
        body = pooled[:W - 3] - conv
        lo, hi = float(np.percentile(body, 0.5)), float(body.max() + 1.0)
        p = engine.make_params(dt, nfft, hop, win, 0, 0, colormap=cmap, sample_rate=fs, min_db=lo, max_db=hi)
        d_out = torch.empty(W * H * 4, dtype=torch.uint8, device=DEV)
        _capi.check(_capi.lib().sa_render_canvas_device(engine.handle, d_iq.data_ptr(), n * bps, C.byref(p), W, H, fpc,
                                                        _capi.REDUCE[reduce], d_out.data_ptr(),
                                                        torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert_kernel(engine, want)
        check_canvas(d_out.view(H, W, 4).cpu().numpy(), pooled, nfft, fs, lo, hi, cmap)
        got = engine.render_canvas(host, dt, nfft, W, H, fs, hop=hop, window=win, frames_per_column=fpc, reduce=reduce,
                                   colormap=cmap, min_db=lo, max_db=hi)
        assert_kernel(engine, want)
        check_canvas(got, pooled, nfft, fs, lo, hi, cmap)
