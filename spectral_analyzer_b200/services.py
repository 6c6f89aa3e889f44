"""Host-side mirror of the reference's DSP service interface, on top of the C-ABI.

Same names, argument meaning and error behaviour as the Java services the engine replaces
(S/ = src/main/java/net/kcundercover/spectral_analyzer/ in the reference):

  SpectralService.computeMagnitudes                S/services/SpectralService.java:33
  ExtractDownConvertService.extractAndDownConvert  S/services/ExtractDownConvertService.java:34,54
  AsyncExtractDownConvertService.extractAndDownConvertAsync   S/services/AsyncExtractDownConvertService.java:48
  PowerSpectralDensity.calculatePsdWelch (JDSP)    call site S/controllers/AnalysisDialogController.java:308-312

plus the batched entry points that replace the per-frame loop of
S/controllers/MainController.java:980-999 and the per-annotation loop of
S/controllers/AnnotationController.java:321-360.  `buffer` is anything exposing the buffer
protocol over the mapped .sigmf-data bytes (numpy array, mmap, bytes) -- the MappedByteBuffer
of S/sigmf/SigMfHelper.java:78-84, position 0 already past core:header_bytes.
"""
import concurrent.futures
import ctypes as C
import os

import numpy as np

from . import _capi
from ._capi import EngineError  # noqa: F401


def _host_view(buffer):
    a = np.frombuffer(buffer, dtype=np.uint8) if not isinstance(buffer, np.ndarray) else buffer
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError("buffer must be contiguous")
    a = a.view(np.uint8).reshape(-1)
    return a, a.ctypes.data, a.size


class Engine:
    """One engine per GPU (sa_engine_create)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        _capi.check(_capi.lib().sa_engine_create(device, C.byref(self._h)))
        self.device = device
        self._strict = False

    def close(self):
        if self._h:
            _capi.lib().sa_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    @property
    def kernel_launches(self):
        return int(_capi.lib().sa_kernel_launches(self._h))

    # ---- analysis profile: the choices JDSP makes inside downConvert / calculatePsdWelch (sa_analysis_config) ----
    def set_analysis_config(self, taps=None, delay="causal", length="floor", psd_scaling="density", psd_detrend=None,
                            psd_precision="f32", strict_reference=False):
        c = _capi.AnalysisConfig()
        _capi.lib().sa_analysis_config_init(C.byref(c))
        keep = None
        if taps is not None:
            keep = np.ascontiguousarray(taps, np.float64)
            c.taps = keep.ctypes.data_as(C.POINTER(C.c_double))
            c.n_taps = keep.size
        c.delay_mode, c.length_mode = _capi.DELAY[delay], _capi.LENGTH[length]
        c.psd_scaling, c.psd_detrend = _capi.PSD_SCALING[psd_scaling], _capi.DETREND[psd_detrend]
        c.psd_precision = {"f32": _capi.PREC_F32, "f64": _capi.PREC_F64}[psd_precision]
        c.strict_reference = int(bool(strict_reference))
        _capi.check(_capi.lib().sa_set_analysis_config(self._h, C.byref(c)))      # the engine copies the taps
        self._strict = bool(strict_reference)

    def reset_analysis_config(self):
        _capi.check(_capi.lib().sa_set_analysis_config(self._h, None))
        self._strict = False

    def analysis_config(self):
        c = _capi.AnalysisConfig()
        _capi.check(_capi.lib().sa_get_analysis_config(self._h, C.byref(c)))
        inv = lambda d, v: [k for k, x in d.items() if x == v and isinstance(k, str)][0]
        return {"taps": None if not c.n_taps else np.array([c.taps[i] for i in range(c.n_taps)]),
                "delay": inv(_capi.DELAY, c.delay_mode), "length": inv(_capi.LENGTH, c.length_mode),
                "psd_scaling": inv(_capi.PSD_SCALING, c.psd_scaling), "psd_detrend": inv(_capi.DETREND, c.psd_detrend),
                "psd_precision": "f64" if c.psd_precision == _capi.PREC_F64 else "f32",
                "strict_reference": bool(c.strict_reference)}

    def downconvert_length(self, count, down, fast=False):
        return int(_capi.lib().sa_downconvert_length(self._h, count, down, int(bool(fast))))

    def register_host(self, buffer, read_only=True):
        _, ptr, n = _host_view(buffer)
        _capi.check(_capi.lib().sa_register_host(self._h, ptr, n, int(read_only)))

    def unregister_host(self, buffer):
        _, ptr, _n = _host_view(buffer)
        _capi.check(_capi.lib().sa_unregister_host(self._h, ptr))

    # ---- spectrogram ----
    def make_params(self, datatype, nfft, hop=None, window="rect", n_frames=0, start_sample=0,
                    db_mode=_capi.DB_MAG_1E10, out="f32", precision="auto", eof_fill_db=-150.0,
                    colormap="Grayscale", sample_rate=1.0, min_db=-160.0, max_db=-30.0, strict_reference=False):
        p = _capi.default_params()
        p.dtype, p.big_endian = _capi.parse_datatype(datatype, strict_reference)
        p.strict_reference = int(bool(strict_reference))
        p.nfft = nfft
        p.hop = nfft if hop is None else hop
        p.window = _capi.WINDOW[window]
        p.n_frames = n_frames
        p.start_sample = start_sample
        p.db_mode = db_mode
        p.out_kind = {"f32": _capi.OUT_F32_DB, "f64": _capi.OUT_F64_DB, "rgba8": _capi.OUT_RGBA8}[out]
        p.precision = {"auto": _capi.PREC_AUTO, "f32": _capi.PREC_F32, "f64": _capi.PREC_F64}[precision]
        p.eof_fill_db = eof_fill_db
        p.colormap = _capi.CMAP[colormap]
        p.sample_rate, p.min_db, p.max_db = sample_rate, min_db, max_db
        return p

    def spectrogram(self, buffer, datatype, nfft, n_frames, hop=None, window="rect", start_sample=0, out=None,
                    **kw):
        """Batched replacement of the updateDisplay frame loop (MainController.java:980-999).
        Host in, host out; returns [n_frames, nfft] float32 / float64, or uint8 [n_frames, nfft, 4]."""
        _, ptr, nbytes = _host_view(buffer)
        kind = kw.get("out_kind", "f32")
        p = self.make_params(datatype, nfft, hop, window, n_frames, start_sample, out=kind,
                             **{k: v for k, v in kw.items() if k != "out_kind"})
        if out is None:
            if kind == "rgba8":
                out = np.empty((n_frames, nfft, 4), np.uint8)
            else:
                out = np.empty((n_frames, nfft), np.float32 if kind == "f32" else np.float64)
        _capi.check(_capi.lib().sa_spectrogram(self._h, ptr, nbytes, C.byref(p), out.ctypes.data, out.nbytes))
        return out

    def spectrogram_file(self, path, datatype, nfft, n_frames, hop=None, window="rect", start_sample=0, out=None,
                         data_offset=0, data_bytes=0, **kw):
        """Same as `spectrogram`, the capture being read from the data file itself (SigMfHelper.java:59-84:
        `data_offset` = core:header_bytes): parallel pread into the engine's pinned ring, no mapped buffer."""
        kind = kw.get("out_kind", "f32")
        p = self.make_params(datatype, nfft, hop, window, n_frames, start_sample, out=kind,
                             **{k: v for k, v in kw.items() if k != "out_kind"})
        if out is None:
            if kind == "rgba8":
                out = np.empty((n_frames, nfft, 4), np.uint8)
            else:
                out = np.empty((n_frames, nfft), np.float32 if kind == "f32" else np.float64)
        _capi.check(_capi.lib().sa_spectrogram_file(self._h, os.fsencode(path), data_offset, data_bytes, C.byref(p),
                                                    out.ctypes.data, out.nbytes))
        return out

    @property
    def last_kernel(self):
        return _capi.lib().sa_last_kernel_name(self._h).decode()

    def spectrogram_device(self, d_iq_ptr, iq_bytes, params, d_out_ptr, out_bytes, stream=0):
        """Device-resident variant (raw device pointers, e.g. torch tensors' data_ptr())."""
        _capi.check(_capi.lib().sa_spectrogram_device(self._h, d_iq_ptr, iq_bytes, C.byref(params), d_out_ptr,
                                                      out_bytes, stream))

    # ---- downconvert / PSD ----
    def downconvert(self, buffer, datatype, start_sample, count, freq_off, down, fast=False):
        _, ptr, nbytes = _host_view(buffer)
        dt, be = _capi.parse_datatype(datatype, self._strict)
        if down < 1:
            raise EngineError(1, "down must be >= 1")
        m = self.downconvert_length(count, down, fast)
        out = np.empty((2, max(m, 1)), np.float64)
        n = C.c_uint64(0)
        dp = C.POINTER(C.c_double)
        _capi.check(_capi.lib().sa_downconvert(self._h, ptr, nbytes, dt, be, start_sample, count, freq_off, down,
                                               int(fast), out[0].ctypes.data_as(dp), out[1].ctypes.data_as(dp),
                                               C.byref(n)))
        return out[:, :n.value]

    def psd_welch(self, iq, fs, nfft, hop=0, window="hann"):
        re = np.ascontiguousarray(iq[0], np.float64)
        im = np.ascontiguousarray(iq[1], np.float64)
        out = np.empty((2, nfft), np.float64)
        dp = C.POINTER(C.c_double)
        _capi.check(_capi.lib().sa_psd_welch(self._h, re.ctypes.data_as(dp), im.ctypes.data_as(dp), re.size, fs, nfft,
                                             hop, _capi.WINDOW[window], out[0].ctypes.data_as(dp),
                                             out[1].ctypes.data_as(dp)))
        return out

    def downconvert_psd_batch(self, buffer, datatype, sample_rate, annotations, psd_nfft=8192, psd_hop=0,
                              psd_window="hann", want_iq=True, want_psd=True):
        """annotations: iterable of (start_sample, count, freq_off, down, fast).
        Returns (list of [2, M_a] float64 arrays or None, [n_ann, psd_nfft] float64 or None)."""
        _, ptr, nbytes = _host_view(buffer)
        dt, be = _capi.parse_datatype(datatype, self._strict)
        anns = (_capi.Annotation * len(annotations))()
        offs = (C.c_uint64 * len(annotations))()
        total = 0
        lens = []
        for i, (s, c, f, d, fast) in enumerate(annotations):
            anns[i] = _capi.Annotation(int(s), int(c), float(f), int(d), int(bool(fast)))
            offs[i] = total
            lens.append(self.downconvert_length(int(c), int(d), fast))
            total += 2 * lens[-1]
        out_iq = np.empty(max(total, 1), np.float64) if want_iq else None
        out_psd = np.empty((len(annotations), psd_nfft), np.float64) if want_psd else None
        dp = C.POINTER(C.c_double)
        _capi.check(_capi.lib().sa_downconvert_psd_batch(
            self._h, ptr, nbytes, dt, be, sample_rate, anns, len(annotations), psd_nfft, psd_hop,
            _capi.WINDOW[psd_window], out_iq.ctypes.data_as(dp) if want_iq else None, offs,
            out_psd.ctypes.data_as(dp) if want_psd else None))
        iq_list = None
        if want_iq:
            iq_list = []
            for i in range(len(annotations)):
                m = lens[i]
                iq_list.append(out_iq[offs[i]:offs[i] + 2 * m].reshape(2, m))
        return iq_list, out_psd


    # ---- rows next to the hot path (SURVEY.md 8f) ----
    def render_canvas(self, buffer, datatype, nfft, canvas_w, canvas_h, sample_rate, hop=None, window="rect",
                      start_sample=0, frames_per_column=1, reduce="nearest", colormap="Grayscale", min_db=-160.0,
                      max_db=-30.0, **kw):
        """MainController.renderSpectrogram (:1261-1291) on the GPU: uint8 [canvas_h, canvas_w, 4], row 0 = top.
        frames_per_column=1 / reduce='nearest' is the reference; 'max' / 'mean' pool frames x bins per pixel."""
        _, ptr, nbytes = _host_view(buffer)
        p = self.make_params(datatype, nfft, hop, window, 0, start_sample, colormap=colormap, sample_rate=sample_rate,
                             min_db=min_db, max_db=max_db, **kw)
        out = np.empty((canvas_h, canvas_w, 4), np.uint8)
        _capi.check(_capi.lib().sa_render_canvas(self._h, ptr, nbytes, C.byref(p), canvas_w, canvas_h,
                                                 frames_per_column, _capi.REDUCE[reduce], out.ctypes.data))
        return out

    TRACE_STATS = ("mean", "max", "min")

    def spectrum_trace(self, buffer, datatype, nfft, n_frames, hop=None, window="rect", start_sample=0,
                       frames_per_row=None, stats=("mean", "max"), out_kind="f32", **kw):
        """Average / peak-hold / minimum-hold spectra of groups of frames_per_row frames of the spectrogram these
        arguments describe (sa_spectrum_trace); frames_per_row=None: one row over all n_frames.  Host in, host out:
        only the rows cross PCIe.  Returns {stat: float32 / float64 [n_rows, nfft]} for the requested stats."""
        _, ptr, nbytes = _host_view(buffer)
        fpr = n_frames if frames_per_row is None else frames_per_row
        p = self.make_params(datatype, nfft, hop, window, n_frames, start_sample, out=out_kind, **kw)
        outs = self._trace_outputs(stats, n_frames, fpr, nfft, out_kind)
        ptrs = [outs[s].ctypes.data if s in outs else None for s in self.TRACE_STATS]
        nb = next(iter(outs.values())).nbytes
        _capi.check(_capi.lib().sa_spectrum_trace(self._h, ptr, nbytes, C.byref(p), fpr, *ptrs, nb))
        return outs

    def _trace_outputs(self, stats, n_frames, fpr, nfft, out_kind):
        stats = (stats,) if isinstance(stats, str) else tuple(stats)
        bad = [s for s in stats if s not in self.TRACE_STATS]
        if bad or not stats:
            raise ValueError("stats must be a non-empty subset of %s, got %r" % (self.TRACE_STATS, stats))
        n_rows = -(-n_frames // fpr) if fpr > 0 and n_frames > 0 else 0
        dt = np.float64 if out_kind == "f64" else np.float32
        return {s: np.empty((n_rows, nfft), dt) for s in self.TRACE_STATS if s in stats}

    def spectrum_trace_device(self, d_iq_ptr, iq_bytes, params, frames_per_row, d_mean=None, d_max=None, d_min=None,
                              out_bytes=0, stream=0):
        """Device-resident variant (raw device pointers; None = statistic not wanted), asynchronous on `stream`."""
        _capi.check(_capi.lib().sa_spectrum_trace_device(self._h, d_iq_ptr, iq_bytes, C.byref(params), frames_per_row,
                                                         d_mean, d_max, d_min, out_bytes, stream))

    def spectrum_persistence(self, buffer, datatype, nfft, n_frames, n_levels, min_db, max_db, hop=None, window="rect",
                             start_sample=0, **kw):
        """Persistence spectrum (sa_spectrum_persistence): per fft-shifted bin, how many of the n_frames frames of the
        spectrogram these arguments describe landed on each of n_levels dB levels of [min_db, max_db) (below: level 0,
        above: the top level).  Host in, host out: only the counts cross PCIe.  Returns uint32 [n_levels, nfft], row 0
        the lowest level; every column sums to n_frames."""
        _, ptr, nbytes = _host_view(buffer)
        p = self.make_params(datatype, nfft, hop, window, n_frames, start_sample, **kw)
        out = np.empty((n_levels, nfft), np.uint32)
        _capi.check(_capi.lib().sa_spectrum_persistence(self._h, ptr, nbytes, C.byref(p), n_levels, min_db, max_db,
                                                        out.ctypes.data, out.nbytes))
        return out

    def spectrum_persistence_device(self, d_iq_ptr, iq_bytes, params, n_levels, min_db, max_db, d_counts, out_bytes,
                                    stream=0):
        """Device-resident variant (raw device pointers; d_counts holds n_levels * nfft uint32), asynchronous on
        `stream`."""
        _capi.check(_capi.lib().sa_spectrum_persistence_device(self._h, d_iq_ptr, iq_bytes, C.byref(params), n_levels,
                                                               min_db, max_db, d_counts, out_bytes, stream))

    def iq_pack(self, iq, fmt):
        """IqData.getInterleavedBinary (IqData.java:160-187): bytes of interleaved LE float32 / int16."""
        if fmt.lower() not in _capi.PACK:
            raise ValueError("Unsupported binary format: " + fmt)       # IllegalArgumentException, :185-186
        re = np.ascontiguousarray(iq[0], np.float64)
        im = np.ascontiguousarray(iq[1], np.float64)
        code = _capi.PACK[fmt.lower()]
        out = np.empty(re.size * (8 if code == 0 else 4), np.uint8)
        dp = C.POINTER(C.c_double)
        _capi.check(_capi.lib().sa_iq_pack(self._h, re.ctypes.data_as(dp), im.ctypes.data_as(dp), re.size, code,
                                           out.ctypes.data))
        return out.tobytes()

    def analysis_series(self, iq, sample_rate, alpha_mag=1.0, alpha_freq=1.0, center_freq=0.0):
        """updateMagnitudeChart / updateFrequencyChart (AnalysisDialogController.java:219-290):
        returns (mag_db[n], inst_freq[n]) with inst_freq[0] = NaN (the Java loop starts at i = 1)."""
        re = np.ascontiguousarray(iq[0], np.float64)
        im = np.ascontiguousarray(iq[1], np.float64)
        mag, frq = np.empty(re.size, np.float64), np.empty(re.size, np.float64)
        dp = C.POINTER(C.c_double)
        _capi.check(_capi.lib().sa_analysis_series(self._h, re.ctypes.data_as(dp), im.ctypes.data_as(dp), re.size,
                                                   sample_rate, alpha_mag, alpha_freq, center_freq,
                                                   mag.ctypes.data_as(dp), frq.ctypes.data_as(dp)))
        return mag, frq


_default_engine = None


def default_engine():
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    return _default_engine


class SpectralService:
    """S/services/SpectralService.java:16-86."""

    def __init__(self, engine=None):
        self.engine = engine or default_engine()

    def computeMagnitudes(self, buffer, startByte, nfft, datatype):
        """double[] computeMagnitudes(MappedByteBuffer, int startByte, int nfft, String datatype)
        (SpectralService.java:33).  Raises EngineError INVALID_ARG for a non power-of-two nfft
        (commons-math3 MathIllegalArgumentException) and OUT_OF_RANGE for reads past the buffer
        (IndexOutOfBoundsException)."""
        _, ptr, nbytes = _host_view(buffer)
        dt, be = _capi.parse_datatype(datatype, self.engine._strict)
        out = np.empty(nfft, np.float64)
        _capi.check(_capi.lib().sa_compute_magnitudes(self.engine.handle, ptr, nbytes, startByte, nfft, dt, be,
                                                      out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def computeWaterfall(self, buffer, currentSampleOffset, canvasW, fftSize, datatype, **kw):
        """The whole `for t in 0..canvasW` loop of MainController.updateDisplay (:980-999) as ONE
        call: waterfall[canvasW][fftSize], EOF rows = -150.0."""
        kw.setdefault("out_kind", "f64")
        return self.engine.spectrogram(buffer, datatype, fftSize, canvasW, start_sample=currentSampleOffset, **kw)


class ExtractDownConvertService:
    """S/services/ExtractDownConvertService.java:17-118."""

    def __init__(self, engine=None):
        self.engine = engine or default_engine()

    def extractAndDownConvert(self, buffer, startSample, count, datatype, freqOff, down, fast=False):
        """double[2][M] extractAndDownConvert(buffer, long startSample, int count, String datatype,
        double freqOff, int down[, boolean fast]) (ExtractDownConvertService.java:34,54)."""
        return self.engine.downconvert(buffer, datatype, startSample, count, freqOff, down, fast)


class AsyncExtractDownConvertService:
    """S/services/AsyncExtractDownConvertService.java:16-57: a worker pool around the sync service.
    The engine serialises calls internally, so the pool only keeps the caller's thread free."""

    def __init__(self, engine=None, workers=None):
        self.syncService = ExtractDownConvertService(engine)
        self.dspExecutor = concurrent.futures.ThreadPoolExecutor(max_workers=workers or os.cpu_count() or 1,
                                                                 thread_name_prefix="DSP-Worker")

    def extractAndDownConvertAsync(self, buffer, startSample, count, datatype, freqOff, down, fast):
        return self.dspExecutor.submit(self.syncService.extractAndDownConvert, buffer, startSample, count, datatype,
                                       freqOff, down, fast)


class PowerSpectralDensity:
    """JDSP net.kcundercover.jdsp.signal.PowerSpectralDensity as called at
    S/controllers/AnalysisDialogController.java:308-312."""

    engine = None

    @classmethod
    def calculatePsdWelch(cls, data, sampleRate, nfft):
        """double[2][K] calculatePsdWelch(double[][] data, double fs, int nfft): row 0 frequency axis
        centred on 0 Hz, row 1 level in dB/Hz."""
        eng = cls.engine or default_engine()
        return eng.psd_welch(data, sampleRate, nfft)


class IqData:
    """S/data/IqData.java: container of the downconverted double[2][N]; only the binary packers
    (getInterleavedBinary, :160-187, and getDataBuffer, :198-208) are mirrored -- they run on the GPU."""

    def __init__(self, iqSamples, engine=None):
        self.iqSamples = np.array(iqSamples, np.float64)          # defensive deep copy, IqData.java:49-52
        self.engine = engine or default_engine()

    def getInterleavedBinary(self, format):
        return self.engine.iq_pack(self.iqSamples, format)

    def getDataBuffer(self):
        return {"IQ_BUFFER_FLOAT32": self.getInterleavedBinary("float32"),
                "IQ_BUFFER_INT16": self.getInterleavedBinary("int16")}
