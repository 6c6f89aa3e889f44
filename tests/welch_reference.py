"""Welch PSD test support: segment-identifying input, FP64 references and the launch geometry of the Welch kernels.

Input ("block tones"): sample n of block b = n // B is g_b exp(2 pi i (k_b + d_b) n / nfft) + c_b + white noise, with
a seeded tone bin k_b, a small fractional offset d_b, a gain g_b log-uniform over +-20 dB, an optional DC offset c_b
and noise about 30 dB under the median tone.  With B the hop (or a divisor of it) every segment holds its own tones at
its own levels, so the Welch sum records bin by bin which segments went into it: dropping, repeating, shifting or
substituting one segment moves some bins by a large fraction, where a stationary tone would leave every bin the same.

References: `welch_db` is the C oracle (oracle/sa_oracle.c ora_psd_welch_ex, FP64, agrees with scipy.signal.welch,
tests/test_oracle.py).  `segment_power` / `welch_sum` are the same computation in numpy FP64 one segment at a time, in
slabs, for arbitrary segment lists (the mutants of tests/test_welch_reference.py) and for inputs too long for one
oracle call.  Both are plain FP64 sums; test_welch_reference.py holds them to 1e-12 of each other.

Geometry (restated from the source, like P_F32 / P_F64 in test_gpu_kernel_matrix.py):
  frames per CTA (FPC) and threads per CTA   fft_core.cuh Geo<T, N> (P from Plan<T, N>, SA_CTA_1WPF = SA_CTA_F64 = 512),
                                            spectrogram_mid_kernel.cuh MidGeo<N> (SA_CTA_MID = SA_CTA_MID_4096 = 512)
  kernel per (precision, nfft)              analysis.cu find_welch / welch_prepare (direct kernel: any other length)
  CTAs per signal (nsplit)                  analysis.cu welch_prepare: clamp(ceil(max nseg / (8 FPC)), 1, 64)
  persistent CTAs of the mid kernel         analysis.cu welch_launch: min(n_sig nsplit, SMs x resident CTAs per SM)
"""
import numpy as np

from oracle import c_oracle as co
from util import NORM_TOL_F32, NORM_TOL_F64

WINDOWS = ["rect", "hann", "hamming", "blackman", "blackman_harris"]

# FP32: general plan up to 1024 points, the mid kernel (welch_accum_mid_kernel<N, 512>) from 2048 to 16384
F32_GENERAL_FPC = {64: 64, 128: 64, 256: 32, 512: 32, 1024: 16}
F32_MID_FPC = {2048: 8, 4096: 4, 8192: 2, 16384: 1}
# FP64: general plan, 64 .. 8192 points
F64_FPC = {64: 64, 128: 64, 256: 32, 512: 16, 1024: 2, 2048: 1, 4096: 1, 8192: 1}
F64_CTA = {64: 512, 128: 512, 256: 512, 512: 512, 1024: 128, 2048: 128, 4096: 256, 8192: 512}
MID_CTA = 512
STEPS = 8                # segments per frame slot that welch_prepare aims for
MAX_SPLIT = 64


def kernel_of(prec, nfft):
    """(kernel name as engine.last_kernel reports it, FPC, threads per CTA); FPC None for the direct kernel."""
    t = "double" if prec == "f64" else "float"
    if prec == "f32" and nfft in F32_GENERAL_FPC:
        return "welch_accum_kernel<float,%d>" % nfft, F32_GENERAL_FPC[nfft], 512
    if prec == "f32" and nfft in F32_MID_FPC:
        return "welch_accum_mid_kernel<float,%d>" % nfft, F32_MID_FPC[nfft], MID_CTA
    if prec == "f64" and nfft in F64_FPC:
        return "welch_accum_kernel<double,%d>" % nfft, F64_FPC[nfft], F64_CTA[nfft]
    return "psd_direct_kernel<%s>" % t, None, 256


# Bounds of frame_norm_error per kernel family (derivations and measurements: tests/test_gpu_welch_matrix.py)
MID_F32_TOL = 2.5e-5             # welch_accum_mid_kernel
DIRECT_C = 30.0                  # psd_direct_kernel<float>: C sqrt(nfft) 2^-24


def direct_f32_tol(nfft):
    return max(NORM_TOL_F32, DIRECT_C * np.sqrt(nfft) * 2.0 ** -24)


def tol_of(name, nfft):
    """the bound of the kernel `name` (as kernel_of returns it) at nfft points"""
    if name == "psd_direct_kernel<float>":
        return direct_f32_tol(nfft)
    if name.startswith("welch_accum_mid_kernel"):
        return MID_F32_TOL
    return NORM_TOL_F64 if "<double" in name else NORM_TOL_F32


def family(name):
    """kernel family for the per-family worst-error report"""
    if name.startswith("psd_direct"):
        return name
    return name.split(",")[0] + ">"


def n_segments(n, nfft, hop):
    return 1 + (n - nfft) // hop if n >= nfft else 0


def nsplit_of(max_nseg, fpc):
    return max(1, min(MAX_SPLIT, -(-max_nseg // (STEPS * fpc))))


def iterations(nseg, nsplit, fpc):
    """steps each frame slot takes (the last one ragged when nseg is not a multiple of nsplit FPC)"""
    return -(-nseg // (nsplit * fpc))


def regime(nseg, fpc):
    """1: fewer segments than frame slots; 2: one CTA, several steps; 3: 1 < nsplit < 64, ragged; 4: nsplit = 64 and
    more than 8 steps per slot."""
    ns = nsplit_of(nseg, fpc)
    it = iterations(nseg, ns, fpc)
    if nseg < fpc or (fpc == 1 and nseg == 1):
        return 1
    if ns == 1:
        return 2 if it > 1 else 0
    if ns < MAX_SPLIT:
        return 3 if nseg % (ns * fpc) else 0
    return 4 if it > STEPS else 0


def wave_ctas(sms, max_threads_per_sm, cta):
    """an upper bound of the CTAs of `cta` threads one wave holds"""
    return sms * (max_threads_per_sm // cta)


def regime_nseg(reg, fpc, k):
    if reg == 1:
        return max(1, fpc - 1 - fpc // 4)                     # FPC 1: one segment (a slot cannot be idle)
    if reg == 2:
        return 5 * fpc + fpc // 3 + 1
    if reg == 3:
        return STEPS * fpc * (3 + 4 * (k % 3)) + fpc // 2 + 1  # nsplit 4, 8 or 12
    return MAX_SPLIT * fpc * 9 + fpc // 3 + 2                 # 10 steps per slot, the last one ragged


def matrix_cases():
    """(prec, nfft, regime, nseg, hop, window, scaling, detrend) for every kernel engine.psd_welch reaches with a
    power-of-two nfft, in each of the four regimes; hop < nfft, = nfft, gapped and odd in rotation; detrend always
    with idle slots (regime 1)."""
    sizes = [("f32", n) for n in sorted(F32_GENERAL_FPC)] + [("f32", n) for n in sorted(F32_MID_FPC)] + \
            [("f64", n) for n in sorted(F64_FPC)]
    out = []
    for k, (prec, nfft) in enumerate(sizes):
        fpc = kernel_of(prec, nfft)[1]
        for reg in (1, 2, 3, 4):
            i = k + reg
            hop = [nfft // 2, nfft, nfft + nfft // 8, nfft // 2 + 1 + 2 * (k % 2)][i % 4]
            win = WINDOWS[(k + 2 * reg) % 5]
            scaling = ["density", "spectrum"][i % 2]
            detrend = "constant" if reg == 1 or (i // 2) % 2 else None
            out.append((prec, nfft, reg, regime_nseg(reg, fpc, k), hop, win, scaling, detrend))
    return out


# ---------------- input ----------------

def block_params(n_blocks, nfft, seed, gain_db=20.0, frac=0.2, dc_db=None):
    rng = np.random.default_rng(seed)
    k = rng.integers(0, nfft, n_blocks).astype(np.float64)
    d = rng.uniform(-frac, frac, n_blocks)
    g = np.power(10.0, rng.uniform(-gain_db, gain_db, n_blocks) / 20.0)
    c = np.zeros(n_blocks, np.complex128)
    if dc_db is not None:
        c = np.power(10.0, dc_db / 20.0) * np.exp(2j * np.pi * rng.uniform(0, 1, n_blocks)) * rng.uniform(0.2, 1.0, n_blocks)
    return k + d, g, c, rng


def block_tones(n, nfft, block, seed, noise_db=-30.0, dc_db=None):
    """numpy complex128 [n]: block tones (module docstring); dc_db: per-block DC offsets up to that level."""
    nb = -(-n // block)
    f, g, c, rng = block_params(nb, nfft, seed, dc_db=dc_db)
    idx = np.arange(n, dtype=np.float64)
    b = np.arange(n) // block
    x = g[b] * np.exp(2j * np.pi * (f[b] / nfft) * idx) + c[b]
    s = np.power(10.0, noise_db / 20.0) / np.sqrt(2.0)
    x += s * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return x


def block_tones_device(n, nfft, block, seed, device, noise_db=-30.0):
    """the same construction on the device (torch, FP64 phases), seeded by `seed`; returns complex64 [n]"""
    import torch
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    nb = -(-n // block)
    f = torch.randint(0, nfft, (nb,), device=device, generator=gen).double()
    f += (torch.rand(nb, dtype=torch.float64, device=device, generator=gen) * 2 - 1) * 0.2
    g = torch.pow(10.0, (torch.rand(nb, dtype=torch.float64, device=device, generator=gen) * 40 - 20) / 20)
    out = torch.empty(n, dtype=torch.complex64, device=device)
    s = 10.0 ** (noise_db / 20.0) / np.sqrt(2.0)
    step = 1 << 24
    for a in range(0, n, step):
        idx = torch.arange(a, min(n, a + step), dtype=torch.int64, device=device)
        b = idx // block
        ph = torch.remainder(f[b] * idx.double(), float(nfft)) * (2 * np.pi / nfft)   # exact phase before the scale
        z = torch.polar(g[b], ph)
        z += s * torch.randn(idx.numel(), dtype=torch.complex128, device=device, generator=gen) * np.sqrt(2.0)
        out[a:a + idx.numel()] = z.to(torch.complex64)
    return out


def iq_of(x):
    return np.stack([np.ascontiguousarray(x.real, np.float64), np.ascontiguousarray(x.imag, np.float64)])


# ---------------- references ----------------

def window(name, n, symmetric=False):
    """the periodic windows of ora_window; symmetric=True divides by n - 1 instead (a mutant)"""
    d = (n - 1) if symmetric and n > 1 else n
    x = 2 * np.pi * np.arange(n) / d
    return {"rect": np.ones(n), "hann": 0.5 - 0.5 * np.cos(x), "hamming": 0.54 - 0.46 * np.cos(x),
            "blackman": 0.42 - 0.5 * np.cos(x) + 0.08 * np.cos(2 * x),
            "blackman_harris": 0.35875 - 0.48829 * np.cos(x) + 0.14128 * np.cos(2 * x) - 0.01168 * np.cos(3 * x)}[name]


def welch_db(x, fs, nfft, hop, win, scaling="density", detrend=None):
    """the C oracle's Welch PSD in dB (fft-shifted), x complex [n]"""
    return co.psd_welch(iq_of(x), fs, nfft, hop=hop, window=win, cfg=co.analysis_cfg(scaling=scaling, detrend=detrend))[1]


def segment_power(x, nfft, starts, win, detrend, symmetric=False, slab=1 << 20):
    """FP64 |X|^2 summed over the segments starting at `starts` (samples), numpy, in slabs of about `slab` points.
    Returns the unscaled, unshifted sum [nfft]."""
    w = window(win, nfft, symmetric)
    starts = np.asarray(starts, np.int64)
    acc = np.zeros(nfft)
    per = max(1, slab // nfft)
    off = np.arange(nfft, dtype=np.int64)
    for a in range(0, starts.size, per):
        seg = x[starts[a:a + per, None] + off[None, :]].astype(np.complex128)
        if detrend:
            seg = seg - seg.mean(axis=1, keepdims=True)
        s = np.fft.fft(seg * w, axis=1)
        acc += (s.real * s.real + s.imag * s.imag).sum(axis=0)
    return acc


def to_db(acc, nseg, fs, nfft, win, scaling="density"):
    """scale, dB, fft-shift as welch_finalize_kernel / ora_psd_welch_ex do"""
    w = window(win, nfft)
    den = w.sum() ** 2 if scaling == "spectrum" else fs * (w * w).sum()
    return np.fft.fftshift(10.0 * np.log10(acc / (nseg * den) + 1e-30))


def welch_sum(x, fs, nfft, hop, win, scaling="density", detrend=None):
    """the numpy FP64 Welch PSD in dB (same definition as welch_db), slab-streamed"""
    nseg = n_segments(x.size, nfft, hop)
    return to_db(segment_power(x, nfft, np.arange(nseg) * hop, win, detrend), nseg, fs, nfft, win, scaling)
