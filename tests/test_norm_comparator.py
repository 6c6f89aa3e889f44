"""Self-tests of the norm-wise comparator (util.frame_norm_error) on oracle images of white noise: it accepts an
image that differs from the FP64 reference only by FP32 rounding of the dB values, and rejects each of the
subtle mistakes a spectrogram kernel can make while its output still looks like a spectrogram."""
import numpy as np
import pytest

from oracle import c_oracle as co
from util import NORM_TOL_F32, NORM_TOL_F64, frame_norm_error


def noise(datatype, n, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    if datatype.startswith("cf32"):
        return (rng.standard_normal(2 * n) * scale).astype(np.float32).view(np.uint8)
    bps = co.BYTES_PER_IQ[datatype.split("_")[0]]
    return rng.integers(0, 256, n * bps, dtype=np.uint8)


CASES = [("ci16_le", 256, "hann"), ("cu8", 1024, "rect"), ("cf32_le", 4096, "blackman_harris"), ("ci8", 64, "hamming")]


@pytest.fixture(params=CASES, ids=["%s-%d-%s" % c for c in CASES])
def image(request):
    dt, nfft, win = request.param
    frames = 24
    raw = noise(dt, (frames + 1) * nfft, seed=nfft)
    ref = co.spectrogram(raw, dt, 0, nfft, nfft, win, frames + 1)
    return raw, dt, nfft, win, frames, ref


def test_accepts_fp32_rounded_db(image):
    _raw, _dt, _nfft, _win, frames, ref = image
    e = frame_norm_error(ref[:frames].astype(np.float32), ref[:frames])
    assert e.max() <= NORM_TOL_F32 / 2, e.max()
    assert frame_norm_error(ref, ref).max() == 0.0 < NORM_TOL_F64


def test_rejects_neighbouring_frame(image):
    _raw, _dt, _nfft, _win, frames, ref = image
    assert (frame_norm_error(ref[1:frames + 1], ref[:frames]) > NORM_TOL_F32).all()


def test_rejects_one_sample_shift_of_the_frame_start(image):
    raw, dt, nfft, win, frames, ref = image
    shifted = co.spectrogram(raw, dt, 1, nfft, nfft, win, frames)
    assert (frame_norm_error(shifted, ref[:frames]) > NORM_TOL_F32).all()


def test_rejects_two_swapped_bins(image):
    _raw, _dt, nfft, _win, frames, ref = image
    got = ref[:frames].copy()
    k = nfft // 3
    got[:, [k, k + 1]] = got[:, [k + 1, k]]
    assert frame_norm_error(got, ref[:frames]).max() > NORM_TOL_F32
    # the swap of a frame's strongest bin with its neighbour is rejected in every frame
    got = ref[:frames].copy()
    rows = np.arange(frames)
    top = ref[:frames].argmax(axis=1)
    nb = (top + 1) % nfft
    got[rows, top], got[rows, nb] = ref[rows, nb], ref[rows, top]
    assert (frame_norm_error(got, ref[:frames]) > NORM_TOL_F32).all()


def test_rejects_fftshift_off_by_one(image):
    _raw, _dt, _nfft, _win, frames, ref = image
    assert (frame_norm_error(np.roll(ref[:frames], 1, axis=1), ref[:frames]) > NORM_TOL_F32).all()
    assert (frame_norm_error(np.roll(ref[:frames], -1, axis=1), ref[:frames]) > NORM_TOL_F32).all()


def test_rejects_one_bin_scaled_by_1e4(image):
    _raw, _dt, _nfft, _win, frames, ref = image
    got = ref[:frames].copy()
    rows = np.arange(frames)
    top = ref[:frames].argmax(axis=1)
    got[rows, top] += 20 * np.log10(1 + 1e-4)          # amplitude x (1 + 1e-4)
    assert (frame_norm_error(got, ref[:frames]) > NORM_TOL_F32).all()


def test_rejects_power_db_for_magnitude_db():
    """The two dB modes differ only through their floors, 20 log10(|X| + 1e-10) against 10 log10(|X|^2 + 1e-20):
    a kernel that writes one for the other is wrong where |X| approaches 1e-10, so the noise sits at that level."""
    nfft, frames = 256, 16
    raw = noise("cf32_le", frames * nfft, seed=3, scale=1e-11)
    mag = co.spectrogram(raw, "cf32_le", 0, nfft, nfft, "rect", frames, db_mode=co.DB_MAG_1E10)
    pwr = co.spectrogram(raw, "cf32_le", 0, nfft, nfft, "rect", frames, db_mode=co.DB_POWER)
    assert (frame_norm_error(pwr, mag) > NORM_TOL_F32).all()
    assert (frame_norm_error(mag, pwr) > NORM_TOL_F32).all()
