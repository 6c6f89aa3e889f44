/*
 * sa_engine.h -- C-ABI of the B200 spectral engine (libsa_engine.so).
 *
 * Drop-in boundary for the ONE hot path of GassiusODude/spectral_analyzer: the three Spring
 * @Service bodies and one static JDSP call that today run on the JVM
 * (S/ = src/main/java/net/kcundercover/spectral_analyzer/ in the reference):
 *
 *   SpectralService.computeMagnitudes(MappedByteBuffer,int,int,String)            S/services/SpectralService.java:33
 *   frame loop of MainController.updateDisplay                                    S/controllers/MainController.java:980-999
 *   renderSpectrogram / getColorForMagnitude                                      S/controllers/MainController.java:1261-1291, :926-957
 *   ExtractDownConvertService.extractAndDownConvert(..)                           S/services/ExtractDownConvertService.java:34,54
 *   AsyncExtractDownConvertService.extractAndDownConvertAsync(..)                 S/services/AsyncExtractDownConvertService.java:48
 *   PowerSpectralDensity.calculatePsdWelch(double[][],double,int) [JDSP] call     S/controllers/AnalysisDialogController.java:308-312
 *
 * The reference has no FFI today; these are the symbols a Java 21 Panama (java.lang.foreign)
 * binding would look up (INTEGRATION.md shows that binding).  Plain pointers and sizes only,
 * no callbacks, no global state; every call returns an int32 status (0 = ok) and
 * sa_last_error() returns a thread-local message.  All entry points are re-entrant: calls
 * on one engine serialise on an internal lock, different engines run concurrently.
 * There is NO CPU fallback: without a CUDA device sa_engine_create fails with SA_ERR_NO_DEVICE.
 * The *_device entry points are asynchronous on the caller's stream and use per-engine workspaces:
 * successive device calls on ONE engine must be issued on one stream (or be ordered by the caller),
 * and a host-buffer call on that engine may only follow once the device call's stream has been
 * synchronised (the host-buffer entry points run on the engine's own streams and return when their
 * results are in the caller's memory).  Use one engine per stream for concurrent device work.
 */
#ifndef SA_ENGINE_H
#define SA_ENGINE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SA_API __attribute__((visibility("default")))

typedef struct sa_engine sa_engine;

/* status codes */
enum {
    SA_OK = 0,
    SA_ERR_INVALID_ARG = 1,   /* null pointer, nfft not a power of two (commons-math throws), bad enum */
    SA_ERR_UNSUPPORTED = 2,   /* valid request this build has no kernel for */
    SA_ERR_OUT_OF_RANGE = 3,  /* read past the end of the buffer (IndexOutOfBoundsException in Java) */
    SA_ERR_CUDA = 4,
    SA_ERR_NO_DEVICE = 5,
    SA_ERR_OOM = 6,
    SA_ERR_SMALL_OUTPUT = 7
};

/* SigMF core:datatype families (S/sigmf/Global.java:67-79) */
enum { SA_CF32 = 0, SA_CI16 = 1, SA_CU8 = 2, SA_CI8 = 3, SA_CF64 = 4,
       /* any datatype without a decode branch in the reference (ri16_le, cf16 ...): accepted only with
        * strict_reference, where it decodes as the reference's fall-through branches do (zeros in the
        * spectrogram, SpectralService.java:60-63; cf32 in the downconverter, ExtractDownConvertService.java:93-96) */
       SA_DT_OTHER = 5 };
/* windows, periodic (DFT-even) definitions; the reference spectrogram is SA_WIN_RECT */
enum { SA_WIN_RECT = 0, SA_WIN_HANN = 1, SA_WIN_HAMMING = 2, SA_WIN_BLACKMAN = 3, SA_WIN_BLACKMAN_HARRIS = 4 };
/* dB scaling: MAG_1E10 is the reference, 20*log10(|X| + 1e-10) (SpectralService.java:80-81) */
enum { SA_DB_MAG_1E10 = 0, SA_DB_POWER = 1 /* 10*log10(|X|^2 + 1e-20) */ };
/* output element kinds */
enum { SA_OUT_F32_DB = 0, SA_OUT_F64_DB = 1, SA_OUT_RGBA8 = 2 };
/* arithmetic: F32 kernels (default) or the FP64 path (mandatory for cf64 input) */
enum { SA_PREC_AUTO = 0, SA_PREC_F32 = 1, SA_PREC_F64 = 2 };
/* colormaps of getColorForMagnitude (MainController.java:939-956) */
enum { SA_CMAP_GRAYSCALE = 0, SA_CMAP_HEATMAP = 1 };
/* canvas reduction: NEAREST is renderSpectrogram's nearest-bin pick (MainController.java:1280) */
enum { SA_REDUCE_NEAREST = 0, SA_REDUCE_MAX = 1, SA_REDUCE_MEAN = 2 };
/* IqData.getInterleavedBinary formats (S/data/IqData.java:160-187) */
enum { SA_PACK_F32 = 0, SA_PACK_I16 = 1 };
/* analysis profile (sa_analysis_config) */
enum { SA_DELAY_CAUSAL = 0, SA_DELAY_SAME = 1, SA_DELAY_VALID = 2 };
enum { SA_LEN_FLOOR = 0, SA_LEN_CEIL = 1 };
enum { SA_PSD_DENSITY = 0, SA_PSD_SPECTRUM = 1 };
enum { SA_DETREND_NONE = 0, SA_DETREND_CONSTANT = 1 };

/* Batched spectrogram request: replaces the per-frame loop MainController.java:982-999.
 * Frame t covers samples [start_sample + t*hop, +nfft) of the buffer; a frame that would
 * read past the end of the buffer becomes a row of eof_fill_db (-150.0 in the reference,
 * :994-998).  Row layout: out[t][(k + nfft/2) % nfft] (fft-shifted, SpectralService.java:78).
 * Reference parity mode = {window RECT, hop nfft, db_mode MAG_1E10}. */
typedef struct sa_spectrogram_params {
    uint32_t struct_size;   /* sizeof(sa_spectrogram_params), for forward compatibility */
    int32_t  dtype;         /* SA_CF32.. */
    int32_t  big_endian;    /* 0: "_le" datatypes; 1 otherwise (S/sigmf/SigMfHelper.java:87-91) */
    int32_t  window;        /* SA_WIN_* */
    uint32_t nfft;          /* power of two, 64..65536 (main-scene.fxml:129) */
    int32_t  db_mode;       /* SA_DB_* */
    int32_t  out_kind;      /* SA_OUT_* */
    int32_t  precision;     /* SA_PREC_* */
    uint64_t start_sample;  /* currentSampleOffset (MainController.java:984) */
    uint64_t hop;           /* samples between frame starts; the reference uses nfft */
    uint64_t n_frames;      /* canvasW in the reference */
    double   eof_fill_db;   /* -150.0 (MainController.java:996-997) */
    /* only for SA_OUT_RGBA8: renderSpectrogram's dB/Hz conversion and colour ramp */
    int32_t  colormap;      /* SA_CMAP_* */
    int32_t  strict_reference;  /* 1: decode exactly as SpectralService.java:42-63 does, bugs included: cf64 and
                                 * SA_DT_OTHER have no branch there and decode to zeros (rows of -200 dB); frames are
                                 * addressed with Global.getBytesPerSample (16 for cf64, 8 for unknown datatypes) */
    double   sample_rate;   /* fs: conversion = 10*log10(fs/nfft) + 20*log10(nfft) (:1273-1274) */
    double   min_db;        /* -160 default (main-scene.fxml:143) */
    double   max_db;        /* -30 default  (main-scene.fxml:150) */
} sa_spectrogram_params;

/* One annotation of the batched downconvert(+PSD) call; replaces one iteration of
 * AnnotationController.java:321-360 / one MainController.handleAnalyzeSelection (:684-751). */
typedef struct sa_annotation {
    uint64_t start_sample;  /* targetStart */
    uint64_t count;         /* targetWidth, samples to extract */
    double   freq_off;      /* cycles/sample = (annotation centre - capture fc)/fs (:703,:744) */
    int32_t  down;          /* floor(fs/bw), >= 1 (:721-728) */
    int32_t  fast;          /* 0 conventional (LPF then decimate), 1 polyphase moving average */
} sa_annotation;

/* Analysis profile of an engine: every choice JDSP v1.3.1 (build.gradle:142, NOT vendored in the reference) makes
 * inside Resampler.downConvert / downConvertPolyphase (ExtractDownConvertService.java:106,111-112) and
 * PowerSpectralDensity.calculatePsdWelch (AnalysisDialogController.java:308-312).  The reference pins none of
 * them, so they are parameters here, not constants of the kernels; a maintainer who has JDSP sets them once per
 * engine (INTEGRATION.md maps each field to the JDSP question it answers).  The service entry points keep the
 * reference's signatures: the profile plays the role the JDSP jar plays on the JVM.
 *   conventional:  z[m] = sum_{k<L} h[k] y[m*down + off - k],  y[n] = x[n] exp(-2 pi i freq_off n), y = 0 outside
 *                  [0, count);  off = 0 (CAUSAL), (L-1)/2 (SAME), L-1 (VALID)
 *   fast:          z[m] = (1/down) sum_{k<down} y[m*down + k]          (delay modes do not apply)
 *   outputs:       FLOOR count/down | CEIL ceil(count/down) | VALID (count-L)/down + 1
 *   PSD:           mean over segments of |FFT(w (x - mean))|^2 scaled 1/(fs sum w^2) (DENSITY) or 1/(sum w)^2
 *                  (SPECTRUM), 10 log10, two-sided, fft-shifted; transforms in FP32 or FP64.
 * Defaults (sa_analysis_config_init / engines that never set a profile): built-in taps (sa_lowpass_taps), CAUSAL,
 * FLOOR, DENSITY, no detrend, FP32, strict_reference off. */
typedef struct sa_analysis_config {
    uint32_t struct_size;      /* sizeof(sa_analysis_config) */
    uint32_t n_taps;           /* L; 0 with taps == NULL */
    const double* taps;        /* h[0..L): used for every decimation factor; NULL: Hamming-windowed sinc, 8*down+1 taps */
    int32_t  delay_mode;       /* SA_DELAY_* */
    int32_t  length_mode;      /* SA_LEN_* */
    int32_t  psd_scaling;      /* SA_PSD_* */
    int32_t  psd_detrend;      /* SA_DETREND_* */
    int32_t  psd_precision;    /* SA_PREC_F32 (default) or SA_PREC_F64 (powers of two up to 8192, any length up to ~11000) */
    int32_t  strict_reference; /* 1: the downconverter decodes as ExtractDownConvertService.java:60-67,79-96 does, bugs
                                * included: cf64 is read at an 8-byte stride (re = d[i], im = d[i+1]) and SA_DT_OTHER as cf32 */
} sa_analysis_config;

/* ---- lifecycle ---- */
SA_API int32_t     sa_engine_create(int32_t device_ordinal, sa_engine** out_engine);
SA_API void        sa_engine_destroy(sa_engine* engine);
SA_API const char* sa_last_error(void);                 /* thread-local, never NULL */
SA_API const char* sa_version(void);
/* number of CUDA kernels this engine has launched so far (bench.py's gpu_launches) */
SA_API uint64_t    sa_kernel_launches(const sa_engine* engine);

/* ---- helpers mirroring S/sigmf/Global.java:67-79 and S/sigmf/SigMfHelper.java:87-91 ---- */
SA_API int32_t sa_bytes_per_iq(int32_t dtype);          /* 8,4,2,2,16 ; 0 if unknown */
/* "ci16_le" -> (SA_CI16, 0); prefix match like String.startsWith, order LE iff ends "_le" */
SA_API int32_t sa_parse_datatype(const char* sigmf_datatype, int32_t* dtype, int32_t* big_endian);
SA_API void    sa_spectrogram_params_init(sa_spectrogram_params* p);   /* reference defaults */

/* ---- host memory: the mmapped .sigmf-data MemorySegment (SigMfHelper.java:78-84) ---- */
/* Page-locks [ptr, ptr+bytes) so that the range itself is the DMA source / target.  Optional.
 * Works for anonymous memory (malloc'ed or Arena-allocated segments, heap arrays pinned by the caller).
 * It does NOT work for the file-backed mapping FileChannel.map returns: cudaHostRegister refuses such
 * ranges ("invalid argument", measured on the B200 hosts) and this call then returns SA_ERR_CUDA.
 * Unregistered / pageable memory -- the mapped .sigmf-data buffer included -- is staged by the engine through
 * its own pinned ring with parallel host copies; sa_spectrogram_file reads the file into that ring directly.
 * read_only != 0 for PROT_READ ranges. */
SA_API int32_t sa_register_host(sa_engine* engine, const void* ptr, uint64_t bytes, int32_t read_only);
SA_API int32_t sa_unregister_host(sa_engine* engine, const void* ptr);

/* ---- spectrogram ---- */
/* iq / out are HOST pointers; iq points at sample 0 of the capture (position 0 of the mapped
 * buffer, i.e. already past core:header_bytes, SigMfHelper.java:84) and need only be aligned to
 * its element size.  out holds n_frames*nfft elements of out_kind (4, 8 or 4 bytes each). */
SA_API int32_t sa_spectrogram(sa_engine* engine, const void* iq, uint64_t iq_bytes,
                              const sa_spectrogram_params* params, void* out, uint64_t out_bytes);
/* Same with DEVICE pointers; asynchronous on `cuda_stream` (a cudaStream_t, NULL = the legacy
 * default stream).  d_iq must be aligned to one IQ pair (sa_bytes_per_iq). */
SA_API int32_t sa_spectrogram_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes,
                                     const sa_spectrogram_params* params, void* d_out,
                                     uint64_t out_bytes, void* cuda_stream);
/* Same with the capture read from the data FILE (SigMfHelper.load: S/sigmf/SigMfHelper.java:59-84): sample 0
 * is at byte data_offset of `path` (core:header_bytes), data_bytes limits the capture (0 = to the end of the
 * file; 64-bit, the reference maps at most 2 GiB - 1, :78-82).  The engine preads the frames' bytes straight
 * into its pinned ring with several threads: no mapped buffer, no page-fault + memcpy hop.  out: host. */
SA_API int32_t sa_spectrogram_file(sa_engine* engine, const char* path, uint64_t data_offset, uint64_t data_bytes,
                                   const sa_spectrogram_params* params, void* out, uint64_t out_bytes);
/* name of the kernel family the engine's last launch selected, e.g.
 * "spectrogram_tma_kernel<float,1024,cf32,window>", or for the analysis calls
 * "downconvert_kernel(pipelined)+welch_accum_mid_kernel<float,8192>" (thread-local copy, never NULL) */
SA_API const char* sa_last_kernel_name(sa_engine* engine);
/* SpectralService.computeMagnitudes (SpectralService.java:33-85), kept for API compatibility:
 * one frame at byte offset start_byte, rect window, 20*log10(|X|+1e-10), fft-shifted, FP64 out. */
SA_API int32_t sa_compute_magnitudes(sa_engine* engine, const void* buffer, uint64_t capacity_bytes,
                                     uint64_t start_byte, uint32_t nfft, int32_t dtype,
                                     int32_t big_endian, double* out_magnitudes);

/* ---- analysis profile ---- */
SA_API void     sa_analysis_config_init(sa_analysis_config* config);                 /* the defaults above */
/* copies the configuration (taps included) into the engine; NULL restores the defaults */
SA_API int32_t  sa_set_analysis_config(sa_engine* engine, const sa_analysis_config* config);
/* current profile; out->taps points at the engine's copy (valid until the next sa_set_analysis_config) */
SA_API int32_t  sa_get_analysis_config(sa_engine* engine, sa_analysis_config* out);
/* M, the number of outputs sa_downconvert produces for `count` input samples under the engine's profile */
SA_API uint64_t sa_downconvert_length(sa_engine* engine, uint64_t count, int32_t down, int32_t fast);

/* ---- downconvert (ExtractDownConvertService.java:54-117) ---- */
/* NOT parity-verified against the reference: the arithmetic behind these two calls lives in JDSP, which is not
 * vendored (SURVEY F6); what is verified is the engine against the profile's written spec (oracle/).
 * out_re/out_im: host arrays of at least sa_downconvert_length(count, down, fast) doubles (row 0 / row 1 of the
 * Java double[2][M]); *out_len receives M. */
SA_API int32_t sa_downconvert(sa_engine* engine, const void* iq, uint64_t iq_bytes, int32_t dtype,
                              int32_t big_endian, uint64_t start_sample, uint64_t count,
                              double freq_off, int32_t down, int32_t fast,
                              double* out_re, double* out_im, uint64_t* out_len);
SA_API int32_t sa_lowpass_taps(int32_t down, double* taps /* 8*down+1 */);

/* ---- Welch PSD (JDSP calculatePsdWelch call site, AnalysisDialogController.java:303-313) ---- */
/* NOT parity-verified against the reference (JDSP, see above).  re/im: host FP64 arrays of n samples (rows of
 * double[2][n]).  nfft: ANY length 1 <= nfft <= n -- the caller passes 8192, or n itself for signals shorter than
 * that (AnalysisDialogController.java:303-307); powers of two 64..16384 run on the Stockham kernels, every other
 * length on a direct DFT kernel (up to ~24000 points FP32 / ~11000 FP64).  hop = 0 selects nfft/4 (75 % overlap).
 * out_freq / out_db hold nfft doubles: frequency axis centred on 0 ((k - nfft/2) fs / nfft) and the level in dB,
 * bin i of the transform at (i + nfft/2) % nfft. */
SA_API int32_t sa_psd_welch(sa_engine* engine, const double* re, const double* im, uint64_t n,
                            double fs, uint32_t nfft, uint64_t hop, int32_t window,
                            double* out_freq, double* out_db);

/* ---- batched annotation analysis: downconvert + Welch PSD for many annotations, one call ----
 * iq: HOST pointer to the capture; for annotation a: decimated IQ goes to
 * out_iq + iq_offsets[a] (re block of M_a doubles followed by im block, M_a = sa_downconvert_length) when
 * out_iq != NULL; the PSD (psd_nfft doubles, dB/Hz, fft-shifted; fs' = sample_rate/down) goes to
 * out_psd_db + a*psd_nfft when out_psd_db != NULL.  An annotation with M_a < psd_nfft gets the Java caller's
 * short-signal rule (:304-307): ONE window of M_a points; its M_a bins sit at the start of the row, the rest of
 * the row is NaN.  With out_iq == NULL the decimated IQ never leaves the chip's L2 (PSD-only mode). */
SA_API int32_t sa_downconvert_psd_batch(sa_engine* engine, const void* iq, uint64_t iq_bytes,
                                        int32_t dtype, int32_t big_endian, double sample_rate,
                                        const sa_annotation* anns, uint32_t n_ann,
                                        uint32_t psd_nfft, uint64_t psd_hop, int32_t psd_window,
                                        double* out_iq, const uint64_t* iq_offsets,
                                        double* out_psd_db);
/* device-resident variant used for roofline timing: d_iq device capture, outputs device.
 * (Fast path: an even decimation 4 .. 32 whose rows are whole 16-byte chunks, with a 16-byte aligned d_iq and (start_sample + delay shift) congruent to 0 or -1
 * modulo the samples per 16 bytes -- every start for cf32 -- takes the row-per-thread kernel; everything else the staged
 * kernels.  The host variant above packs each span on a 16-byte boundary itself.  Results do not depend on the path
 * beyond the FP32 tolerance.) */
SA_API int32_t sa_downconvert_psd_batch_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes,
                                               int32_t dtype, int32_t big_endian, double sample_rate,
                                               const sa_annotation* anns, uint32_t n_ann,
                                               uint32_t psd_nfft, uint64_t psd_hop, int32_t psd_window,
                                               double* d_out_iq, const uint64_t* iq_offsets,
                                               double* d_out_psd_db, void* cuda_stream);

/* ---- display canvas (SURVEY.md 8f N2): MainController.renderSpectrogram, :1261-1291 ----
 * Column t of the canvas_w x canvas_h RGBA8 image (row 0 = top = +fs/2, :1288) is built from the
 * frames_per_column frames starting at frame t*frames_per_column of the spectrogram that `params`
 * describes (params->n_frames and out_kind are ignored; hop is the frame stride, the reference uses
 * nfft); pixel row f takes bin (int)(f / canvas_h * nfft) (:1280).  The reference is
 * frames_per_column = 1 with SA_REDUCE_NEAREST; MAX / MEAN reduce the column's frames and the bins
 * [bin(f), bin(f+1)) (MEAN averages linear power).  Colour mapping as SA_OUT_RGBA8.  Only the
 * canvas crosses PCIe on the way back. */
SA_API int32_t sa_render_canvas(sa_engine* engine, const void* iq, uint64_t iq_bytes,
                                const sa_spectrogram_params* params, uint32_t canvas_w, uint32_t canvas_h,
                                uint64_t frames_per_column, int32_t reduce, void* out_rgba);
SA_API int32_t sa_render_canvas_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes,
                                       const sa_spectrogram_params* params, uint32_t canvas_w,
                                       uint32_t canvas_h, uint64_t frames_per_column, int32_t reduce,
                                       void* d_out_rgba, void* cuda_stream);

/* ---- spectrum traces: average, peak-hold and minimum-hold spectra of a capture range ----
 * The frames are those of the spectrogram `params` describes (start_sample, hop, n_frames, window, dtype, byte
 * order, precision, db_mode, eof_fill_db, strict_reference).  Output row r reduces frames [r*F, min((r+1)*F, n_frames)),
 * F = frames_per_row: n_rows = ceil(n_frames / F) rows of nfft bins, fft-shifted as the spectrogram rows.  Per frame t
 * and bin k the power P_t[k] is |X_t[k]|^2 (0 for a strict-reference decode that yields zeros), or for a frame past
 * the end of the buffer the power whose level is eof_fill_db.  MEAN = sum P / count (EOF frames counted; over readable
 * frames this is the Welch PSD of the full band times sum w^2), MAX = max P, MIN = min P, each written as the level
 * 20*log10(sqrt(P) + 1e-10) (SA_DB_MAG_1E10) or 10*log10(P + 1e-20) (SA_DB_POWER) in params->out_kind (F32 or F64).
 * F = 1 gives the spectrogram rows, F = n_frames one trace of the whole range.  Only the rows cross PCIe.
 * out_mean / out_max / out_min: NULL = statistic not wanted (at least one non-NULL); each holds
 * ceil(n_frames / frames_per_row) * nfft elements of params->out_kind; out_bytes is the capacity of each.
 * SA_ERR_INVALID_ARG: frames_per_row == 0, n_frames == 0, all outputs NULL, SA_OUT_RGBA8, misaligned d_iq;
 * SA_ERR_SMALL_OUTPUT: an output is too small.  sa_last_kernel_name names the transform kernel that ran. */
SA_API int32_t sa_spectrum_trace(sa_engine* engine, const void* iq, uint64_t iq_bytes, const sa_spectrogram_params* params,
                                 uint64_t frames_per_row, void* out_mean, void* out_max, void* out_min, uint64_t out_bytes);
/* Same with DEVICE pointers, asynchronous on `cuda_stream`; d_iq aligned to one IQ pair. */
SA_API int32_t sa_spectrum_trace_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes,
                                        const sa_spectrogram_params* params, uint64_t frames_per_row, void* d_mean,
                                        void* d_max, void* d_min, uint64_t out_bytes, void* cuda_stream);

/* ---- persistence spectrum: per-bin histograms of spectrogram levels over a capture range ----
 * The frames are those of the spectrogram `params` describes (start_sample, hop, n_frames, window, dtype, byte order,
 * precision, db_mode, eof_fill_db, strict_reference); params->out_kind, colormap, sample_rate, min_db and max_db are
 * ignored, the level range is [min_db, max_db) of the arguments.  Per frame t and bin k, d[t][k] is the value the
 * spectrogram row holds: the FP32 dB value on FP32 launches, the FP64 value on FP64 launches, eof_fill_db (rounded to
 * the launch's precision) for frames past the end of the buffer, -200 dB for strict-reference zero decodes.  In the
 * launch's precision, each operation rounded on its own (no FMA contraction):
 *   u     = (d - min_db) * s,   s = n_levels / (max_db - min_db)   (min_db and s computed in FP64, then rounded)
 *   level = u >= 1 ? (int)min(u, n_levels - 1) : 0   (below the range and NaN: level 0, above it: n_levels - 1)
 *   counts[level][(k + nfft/2) % nfft] += 1           (bins fft-shifted as the spectrogram rows; level 0 = lowest)
 * Every column sums to n_frames (EOF frames are counted), and the counts are exactly the histogram of the engine's own
 * dB rows for the same request.  Only the counts cross PCIe.
 * out_counts: n_levels * nfft uint32, level-major; out_bytes is its capacity in bytes.
 * SA_ERR_INVALID_ARG: n_levels outside 2..256, min_db / max_db not finite or max_db <= min_db, n_frames == 0,
 * n_frames > 0xFFFFFFFF (counts are uint32), NULL output, misaligned d_iq, or what sa_spectrogram refuses for F32
 * rows of the same request;
 * SA_ERR_SMALL_OUTPUT: the output is too small.  sa_last_kernel_name names the transform and histogram kernels. */
SA_API int32_t sa_spectrum_persistence(sa_engine* engine, const void* iq, uint64_t iq_bytes,
                                       const sa_spectrogram_params* params, uint32_t n_levels, double min_db,
                                       double max_db, uint32_t* out_counts, uint64_t out_bytes);
/* Same with DEVICE pointers, asynchronous on `cuda_stream`; d_iq aligned to one IQ pair. */
SA_API int32_t sa_spectrum_persistence_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes,
                                              const sa_spectrogram_params* params, uint32_t n_levels, double min_db,
                                              double max_db, uint32_t* d_counts, uint64_t out_bytes, void* cuda_stream);

/* ---- downconverter output epilogues (SURVEY.md 8f N3) ----
 * sa_iq_pack: IqData.getInterleavedBinary (S/data/IqData.java:160-187): interleaved little-endian
 * float32 ((float) x) or int16 ((short)(32767 * x), Java narrowing: truncate, saturate to int, keep
 * the low 16 bits; NaN -> 0).  re/im: rows of the Java double[2][n]; out: n*8 or n*4 bytes. */
SA_API int32_t sa_iq_pack(sa_engine* engine, const double* re, const double* im, uint64_t n,
                          int32_t format, void* out);
/* sa_analysis_series: AnalysisDialogController.updateMagnitudeChart / updateFrequencyChart
 * (S/controllers/AnalysisDialogController.java:219-290).  out_mag_db[i] = 20 log10(EMA_i(hypot)),
 * i < n (non-finite values are what the Java loop skips); out_freq[i] = EMA_i(wrapped phase
 * difference / 2 pi * fs) + center_freq for 1 <= i < n (out_freq[0] = NaN, the loop starts at 1).
 * Either output may be NULL. */
SA_API int32_t sa_analysis_series(sa_engine* engine, const double* re, const double* im, uint64_t n,
                                  double sample_rate, double alpha_mag, double alpha_freq,
                                  double center_freq, double* out_mag_db, double* out_freq);
/* Batched device forms on the planar rows sa_downconvert_psd_batch_device wrote: signal a has its
 * re block at d_rows + row_offsets[a], im block lengths[a] doubles later; results start at element
 * out_offsets[a] of the output(s) (elements = IQ pairs for the packer, doubles for the series). */
SA_API int32_t sa_iq_pack_batch_device(sa_engine* engine, const double* d_rows, const uint64_t* row_offsets,
                                       const uint64_t* lengths, const uint64_t* out_offsets, uint32_t n_sig,
                                       int32_t format, void* d_out, void* cuda_stream);
SA_API int32_t sa_analysis_series_batch_device(sa_engine* engine, const double* d_rows,
                                               const uint64_t* row_offsets, const uint64_t* lengths,
                                               const uint64_t* out_offsets, uint32_t n_sig,
                                               double sample_rate, double alpha_mag, double alpha_freq,
                                               double center_freq, double* d_out_mag_db,
                                               double* d_out_freq, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* SA_ENGINE_H */
