"""ctypes binding of libsa_engine.so -- the same symbols the Java Panama binding looks up
(include/sa_engine.h).  Thin: argument marshalling and status -> exception mapping only.
There is no CPU fallback: if the CUDA library is missing or no B200 is visible, calls raise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SA_ENGINE_LIB selects another build of the same library (A/B runs of kernel tuning knobs)
LIB_PATH = os.environ.get("SA_ENGINE_LIB") or os.path.join(_HERE, "libsa_engine.so")

SA_OK = 0
ERR_NAMES = {1: "INVALID_ARG", 2: "UNSUPPORTED", 3: "OUT_OF_RANGE", 4: "CUDA", 5: "NO_DEVICE", 6: "OOM",
             7: "SMALL_OUTPUT"}
DTYPE = {"cf32": 0, "ci16": 1, "cu8": 2, "ci8": 3, "cf64": 4}
DT_OTHER = 5          # datatype without a decode branch in the reference; strict_reference only
DELAY = {"causal": 0, "same": 1, "valid": 2}
LENGTH = {"floor": 0, "ceil": 1}
PSD_SCALING = {"density": 0, "spectrum": 1}
DETREND = {None: 0, False: 0, "none": 0, "constant": 1}
WINDOW = {"rect": 0, "hann": 1, "hamming": 2, "blackman": 3, "blackman_harris": 4}
DB_MAG_1E10, DB_POWER = 0, 1
OUT_F32_DB, OUT_F64_DB, OUT_RGBA8 = 0, 1, 2
PREC_AUTO, PREC_F32, PREC_F64 = 0, 1, 2
CMAP = {"Grayscale": 0, "Heatmap": 1}
REDUCE = {"nearest": 0, "max": 1, "mean": 2}
PACK = {"float32": 0, "int16": 1}


class SpectrogramParams(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("dtype", C.c_int32), ("big_endian", C.c_int32),
                ("window", C.c_int32), ("nfft", C.c_uint32), ("db_mode", C.c_int32),
                ("out_kind", C.c_int32), ("precision", C.c_int32), ("start_sample", C.c_uint64),
                ("hop", C.c_uint64), ("n_frames", C.c_uint64), ("eof_fill_db", C.c_double),
                ("colormap", C.c_int32), ("strict_reference", C.c_int32), ("sample_rate", C.c_double),
                ("min_db", C.c_double), ("max_db", C.c_double)]


class AnalysisConfig(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_taps", C.c_uint32), ("taps", C.POINTER(C.c_double)),
                ("delay_mode", C.c_int32), ("length_mode", C.c_int32), ("psd_scaling", C.c_int32),
                ("psd_detrend", C.c_int32), ("psd_precision", C.c_int32), ("strict_reference", C.c_int32)]


class Annotation(C.Structure):
    _fields_ = [("start_sample", C.c_uint64), ("count", C.c_uint64), ("freq_off", C.c_double),
                ("down", C.c_int32), ("fast", C.c_int32)]


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("sa_engine error %d (%s): %s" % (code, ERR_NAMES.get(code, "?"), msg))
        self.code = code


_lib = None


def lib():
    """Loads libsa_engine.so; fails loudly when it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the engine has no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, u64, i32, u32, dbl = C.c_void_p, C.c_uint64, C.c_int32, C.c_uint32, C.c_double
    dp = C.POINTER(C.c_double)
    L.sa_last_error.restype = C.c_char_p
    L.sa_version.restype = C.c_char_p
    L.sa_kernel_launches.restype = u64
    L.sa_kernel_launches.argtypes = [vp]
    L.sa_engine_create.argtypes = [i32, C.POINTER(vp)]
    L.sa_engine_destroy.argtypes = [vp]
    L.sa_engine_destroy.restype = None
    L.sa_bytes_per_iq.argtypes = [i32]
    L.sa_parse_datatype.argtypes = [C.c_char_p, C.POINTER(i32), C.POINTER(i32)]
    L.sa_spectrogram_params_init.argtypes = [C.POINTER(SpectrogramParams)]
    L.sa_spectrogram_params_init.restype = None
    L.sa_register_host.argtypes = [vp, vp, u64, i32]
    L.sa_unregister_host.argtypes = [vp, vp]
    L.sa_spectrogram.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), vp, u64]
    L.sa_spectrogram_device.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), vp, u64, vp]
    L.sa_spectrogram_file.argtypes = [vp, C.c_char_p, u64, u64, C.POINTER(SpectrogramParams), vp, u64]
    L.sa_last_kernel_name.restype = C.c_char_p
    L.sa_last_kernel_name.argtypes = [vp]
    # ablation only (csrc/tc_ablation.cu): not declared in include/sa_engine.h, not part of the drop-in boundary
    L.sa_ablation_tc_spectrogram_device.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), vp, u64, i32, vp]
    L.sa_compute_magnitudes.argtypes = [vp, vp, u64, u64, u32, i32, i32, dp]
    L.sa_downconvert.argtypes = [vp, vp, u64, i32, i32, u64, u64, dbl, i32, i32, dp, dp, C.POINTER(u64)]
    L.sa_lowpass_taps.argtypes = [i32, dp]
    L.sa_analysis_config_init.argtypes = [C.POINTER(AnalysisConfig)]
    L.sa_analysis_config_init.restype = None
    L.sa_set_analysis_config.argtypes = [vp, C.POINTER(AnalysisConfig)]
    L.sa_get_analysis_config.argtypes = [vp, C.POINTER(AnalysisConfig)]
    L.sa_downconvert_length.argtypes = [vp, u64, i32, i32]
    L.sa_downconvert_length.restype = u64
    L.sa_psd_welch.argtypes = [vp, dp, dp, u64, dbl, u32, u64, i32, dp, dp]
    L.sa_downconvert_psd_batch.argtypes = [vp, vp, u64, i32, i32, dbl, C.POINTER(Annotation), u32, u32, u64, i32,
                                           dp, C.POINTER(u64), dp]
    L.sa_downconvert_psd_batch_device.argtypes = [vp, vp, u64, i32, i32, dbl, C.POINTER(Annotation), u32, u32, u64,
                                                  i32, vp, C.POINTER(u64), vp, vp]
    L.sa_render_canvas.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), u32, u32, u64, i32, vp]
    L.sa_render_canvas_device.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), u32, u32, u64, i32, vp, vp]
    L.sa_spectrum_trace.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), u64, vp, vp, vp, u64]
    L.sa_spectrum_trace_device.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), u64, vp, vp, vp, u64, vp]
    L.sa_spectrum_persistence.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), C.c_uint32, C.c_double, C.c_double,
                                          vp, u64]
    L.sa_spectrum_persistence_device.argtypes = [vp, vp, u64, C.POINTER(SpectrogramParams), C.c_uint32, C.c_double,
                                                 C.c_double, vp, u64, vp]
    L.sa_iq_pack.argtypes = [vp, dp, dp, u64, i32, vp]
    L.sa_analysis_series.argtypes = [vp, dp, dp, u64, dbl, dbl, dbl, dbl, dp, dp]
    pu64 = C.POINTER(u64)
    L.sa_iq_pack_batch_device.argtypes = [vp, vp, pu64, pu64, pu64, u32, i32, vp, vp]
    L.sa_analysis_series_batch_device.argtypes = [vp, vp, pu64, pu64, pu64, u32, dbl, dbl, dbl, dbl, vp, vp, vp]
    _lib = L
    return L


def check(rc):
    if rc != SA_OK:
        raise EngineError(rc, lib().sa_last_error().decode("utf-8", "replace"))


def parse_datatype(datatype, strict_reference=False):
    """'ci16_le' -> (dtype id, big_endian) through the library's own rule.  With strict_reference a datatype
    without a decode branch ('ri16_le', ...) maps to DT_OTHER instead of raising."""
    d, be = C.c_int32(), C.c_int32()
    rc = lib().sa_parse_datatype(datatype.encode(), C.byref(d), C.byref(be))
    if rc == 2 and strict_reference:
        return DT_OTHER, (0 if datatype.endswith("_le") else 1)
    check(rc)
    return d.value, be.value


def default_params():
    p = SpectrogramParams()
    lib().sa_spectrogram_params_init(C.byref(p))
    return p
