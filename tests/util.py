"""Tolerances of the parity tests (BASELINE.json north_star):
integer decode and frame indexing bit-exact; FP32 power within 1e-5 relative on signal bins and
within 1e-3 dB on every bin above the noise floor; the FP64 path much tighter."""
import numpy as np

REL_POWER_TOL = 1e-5                     # relative power error on strong bins
DB_OF_REL_POWER = 10 * np.log10(1 + REL_POWER_TOL)   # = 4.34e-5 dB
DB_TOL_ABOVE_FLOOR = 1e-3                # dB, bins above the noise floor
ABOVE_FLOOR_MARGIN_DB = 10.0             # "above the noise floor": at least 10 dB over the frame median
STRONG_BELOW_MAX_DB = 40.0               # "signal" bins: within 40 dB of the frame maximum
# The noise floor of a frame is estimated by its median bin level (the synthetic recordings are
# three tones over white noise, so most bins ARE the floor).  Bins below the floor (Rayleigh dips,
# window-sidelobe nulls) are cancellation residue beyond FP32 dynamic range: those are compared
# in linear amplitude against the frame maximum instead of in dB.


def check_db_parity(got, ref, mode_power=False, strong_tol=DB_OF_REL_POWER, floor_tol=DB_TOL_ABOVE_FLOOR):
    """got: engine dB image, ref: oracle FP64 dB image, same shape [frames, nfft]."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    assert got.shape == ref.shape
    assert np.isfinite(got).all()
    fmax = ref.max(axis=1, keepdims=True)
    diff = np.abs(got - ref)
    strong = ref >= fmax - STRONG_BELOW_MAX_DB
    above = ref >= np.median(ref, axis=1, keepdims=True) + ABOVE_FLOOR_MARGIN_DB
    assert strong.any()
    worst_strong = diff[strong].max()
    worst_above = diff[above].max() if above.any() else 0.0
    assert worst_strong <= strong_tol, "strong bins: %.3g dB > %.3g dB" % (worst_strong, strong_tol)
    assert worst_above <= floor_tol, "bins above floor: %.3g dB > %.3g dB" % (worst_above, floor_tol)
    # far below the floor: compare linear amplitude against the frame maximum instead of dB
    scale = 20.0 if not mode_power else 10.0
    lin_g, lin_r = 10 ** (got / scale), 10 ** (ref / scale)
    lin_max = 10 ** (fmax / scale)
    assert (np.abs(lin_g - lin_r) <= 1e-5 * lin_max).all()
    return worst_strong, worst_above


# Norm-wise bounds of frame_norm_error: 2x and 3x the worst E measured on white noise (tests/test_gpu_kernel_matrix.py)
NORM_TOL_F32 = 1e-5
NORM_TOL_F64 = 1e-12


def frame_norm_error(got, ref):
    """Per frame E = max_k |A_got - A_ref| / rms_k(A_ref), A = 10^(dB/20) the linear magnitude (also in power mode,
    which writes 10 log10 |X|^2).  Unlike check_db_parity it holds EVERY bin of a full-band frame to the same
    absolute scale, so a wrong frame, a shifted bin or a mis-scaled bin shows however weak the bin is.
    got, ref: dB images [frames, nfft]; returns float64 [frames]."""
    a_g = np.power(10.0, np.asarray(got, np.float64) / 20.0)
    a_r = np.power(10.0, np.asarray(ref, np.float64) / 20.0)
    return np.abs(a_g - a_r).max(axis=1) / np.sqrt(np.mean(a_r * a_r, axis=1))
